"""Flat parameter store: one fp32 master buffer, one fp32 gradient buffer, Adam moments and bf16
tensor-core operand copies for every trainable tensor of a model.

Why: (a) the optimizer (reference train.py:77-78: clip_grad_norm_ + AdamW.step) becomes two passes
over ONE contiguous buffer; (b) DDP buckets are contiguous ranges of the gradient buffer (no
flatten/unflatten copies); (c) conv weights are kept physically in the [Cout][kh*kw][Cin] order the TMA
tensor maps want (one bf16 copy serves fprop and dgrad), while ``nn.Parameter`` objects keep the reference's logical shapes and names
(``state_dict`` / checkpoints interchange with the reference, SURVEY.md 8b).
"""
import weakref

import torch
import torch.nn as nn

from . import kernels as K

_PAD = 8  # elements; keeps bf16 slices 16-byte aligned
_STORE_OF_PARAM = weakref.WeakValueDictionary()


def _kind_of(module, pname):
    if isinstance(module, nn.ConvTranspose2d) and pname == "weight":
        return "convT"
    if isinstance(module, nn.Conv2d) and pname == "weight":
        return "dw" if module.groups > 1 else "conv"
    return "vec"


class Entry:
    __slots__ = ("name", "param", "kind", "offset", "numel", "shape3", "ready_epoch", "pending")

    def __init__(self, name, param, kind, offset):
        self.name, self.param, self.kind, self.offset = name, param, kind, offset
        self.numel = param.numel()
        s = tuple(param.shape)
        if kind == "conv":      # logical [Cout, Cin, kh, kw] -> [N=Cout][T=kh*kw][K=Cin]
            self.shape3 = (s[0], s[2] * s[3], s[1])
        elif kind == "convT":   # logical [Cin, Cout, 2, 2]  -> [N=Cout][T=4][K=Cin]
            self.shape3 = (s[1], s[2] * s[3], s[0])
        elif kind == "dw":      # logical [C, 1, kh, kw]     -> [T=kh*kw][C]
            self.shape3 = (1, s[2] * s[3], s[0])
        else:
            self.shape3 = None
        self.ready_epoch = -1
        self.pending = 0        # forward uses of this tensor whose backward has not run yet (see ParamStore.note_use)

    def logical_view(self, flat):
        """View of flat[offset:offset+numel] with the parameter's logical shape (strided)."""
        sl = flat[self.offset:self.offset + self.numel]
        s = tuple(self.param.shape)
        if self.kind == "conv":
            return sl.view(s[0], s[2], s[3], s[1]).permute(0, 3, 1, 2)
        if self.kind == "convT":
            return sl.view(s[1], s[2], s[3], s[0]).permute(3, 0, 1, 2)
        if self.kind == "dw":
            return sl.view(s[2], s[3], s[1], s[0]).permute(3, 2, 0, 1)
        return sl.view(s)

    def view3(self, flat):
        return flat[self.offset:self.offset + self.numel].view(self.shape3)


class ParamStore:
    def __init__(self, root):
        self.root = weakref.ref(root)
        self.entries = []
        self.by_param = {}
        off = 0
        seen = set()
        for mname, mod in root.named_modules():
            for pname, p in mod.named_parameters(recurse=False):
                if id(p) in seen or not p.requires_grad:
                    continue
                seen.add(id(p))
                e = Entry((mname + "." if mname else "") + pname, p, _kind_of(mod, pname), off)
                self.entries.append(e)
                self.by_param[id(p)] = e
                off += (e.numel + _PAD - 1) // _PAD * _PAD
        self.total = off
        self.flat_p = self.flat_g = self.flat_m = self.flat_v = self.shadow = None
        self.device = None
        self._versions = None
        self.opt_epoch = 0           # bumped by the fused optimizer (it rewrites master + shadow)
        self.grad_epoch = 0          # bumped by zero_grad(); used by DDP bucket bookkeeping
        self.grad_ready_hook = None  # callable(entry) fired right after an entry's gradient is complete
        self.grads_clean = False     # flat_g is known to be all zeros
        for e in self.entries:
            _STORE_OF_PARAM[id(e.param)] = self

    # -- construction / re-attachment ------------------------------------------------------
    def _attached(self, e):
        p = e.param
        return (self.flat_p is not None and p.device == self.flat_p.device and p.dtype == torch.float32
                and p.data_ptr() == self.flat_p.data_ptr() + 4 * e.offset
                and p.stride() == e.logical_view(self.flat_p).stride())

    def ensure(self, device, optimizer_state=True):
        """(Re)build the flat buffers on `device` and point every Parameter at its slice.  optimizer_state=False: masters
        and bf16 operand copies only -- no gradient or Adam-moment buffers (a model that is never trained, e.g. the
        weight average of ema.ModelEMA)."""
        device = torch.device(device)
        if device.type != "cuda" and not getattr(K, "_EMULATED", False):
            raise K._lib.SnnKernelError("parameters must live on a CUDA device (no CPU fallback)")
        if device.type == "cuda" and device.index is None:
            # "cuda" and "cuda:0" must name the same store: a mismatch would silently rebuild the flat buffers (zeroed
            # bf16 operand copies, stale DDP bucket views)
            device = torch.device("cuda", torch.cuda.current_device())
        if self.flat_p is not None and self.device == device and all(self._attached(e) for e in self.entries):
            return self
        old_m, old_v = self.flat_m, self.flat_v
        flat_p = torch.zeros(self.total, device=device, dtype=torch.float32)
        for e in self.entries:
            e.logical_view(flat_p).copy_(e.param.data.to(device=device, dtype=torch.float32))
        self.flat_p = flat_p
        self.grads_clean = True
        if optimizer_state:
            self.flat_g = torch.zeros(self.total, device=device, dtype=torch.float32)
            keep = old_m is not None and old_m.device == device
            self.flat_m = old_m if keep else torch.zeros(self.total, device=device, dtype=torch.float32)
            self.flat_v = old_v if keep else torch.zeros(self.total, device=device, dtype=torch.float32)
        self.shadow = torch.zeros(self.total, device=device, dtype=torch.bfloat16)
        self.device = device
        for e in self.entries:
            e.param.data = e.logical_view(self.flat_p)
            e.param.grad = None
        self._versions = None
        return self

    # -- bf16 operand copies ---------------------------------------------------------------
    def refresh_operands(self):
        """Make `shadow` (bf16 copy of every conv weight, same [Cout][tap][Cin] layout) current.  The fused optimizer
        writes the shadow itself, so this only does work after the masters were changed some other way
        (init, load_state_dict, an external optimizer)."""
        vers = tuple(e.param._version for e in self.entries)
        if vers == self._versions:
            return
        for e in self.entries:
            if e.kind in ("conv", "convT"):
                K.weight_prep(e.view3(self.flat_p), want_fprop=True, want_dgrad=False, wf=e.view3(self.shadow))
        self._versions = vers

    def w_fprop(self, p):
        """bf16 [Cout][taps][Cin] operand of fprop AND dgrad (dgrad reads it MN-major in place)."""
        return self.by_param[id(p)].view3(self.shadow)

    def w_master3(self, p):
        return self.by_param[id(p)].view3(self.flat_p)

    # -- gradients -------------------------------------------------------------------------
    def zero_grad(self):
        """optimizer.zero_grad() of train.py:61.  The fused optimizer leaves the gradient buffer zeroed itself
        (snn_adamw_step(zero_grad=1)); the 481 MB fill only runs when something accumulated since (external optimizer)."""
        if not self.grads_clean:
            self.flat_g.zero_()
        self.grads_clean = True
        self.grad_epoch += 1
        for e in self.entries:
            e.param.grad = e.logical_view(self.flat_g)
            e.pending = 0

    def grad_view(self, p, three_d=False):
        """Gradient slice to accumulate into (PyTorch semantics: a `None` grad means start from zero)."""
        e = self.by_param[id(p)]
        g = p.grad
        self.grads_clean = False
        ours = e.logical_view(self.flat_g)
        if g is None or g.data_ptr() != ours.data_ptr():
            self.flat_g[e.offset:e.offset + e.numel].zero_()
            if g is not None:
                ours.add_(g)
            p.grad = ours
        return e.view3(self.flat_g) if three_d else ours

    def note_use(self, *params):
        """Called by the forward of every autograd op for the parameters it reads: the reference-style per-frame loop
        (`model(frame, hidden)` T times, train.py:62-66) uses each parameter T times, and its gradient is final only
        after the LAST of the T backward calls -- a bucket must not be all-reduced before that.  (Callers check
        ctx.needs_input_grad: grad mode is always off inside Function.forward.)"""
        for p in params:
            if p is not None and p.requires_grad:
                self.by_param[id(p)].pending += 1

    def grad_done(self, p):
        e = self.by_param[id(p)]
        if e.pending > 0:
            e.pending -= 1
        if e.pending == 0 and self.grad_ready_hook is not None:
            self.grad_ready_hook(e)


def store_for(root, device):
    """Store owning `root`'s parameters (shared with an enclosing model if one already claimed them)."""
    st = getattr(root, "_snn_store", None)
    if st is None:
        params = [p for p in root.parameters() if p.requires_grad]
        owner = _STORE_OF_PARAM.get(id(params[0])) if params else None
        if owner is not None and all(_STORE_OF_PARAM.get(id(p)) is owner for p in params):
            st = owner
        else:
            st = ParamStore(root)
        object.__setattr__(root, "_snn_store", st)
    return st.ensure(device)
