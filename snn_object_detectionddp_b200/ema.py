"""Exponential moving average of the weights -- ultralytics' ModelEMA -- updated on the device after every optimizer step.

    ema = ModelEMA(model)                   # model = YOLOTemporalUNet on its device (after the Trainer is built)
    trainer.ema = ema                       # Trainer.optimizer_step now enqueues one update behind the AdamW pass
    ... training steps, graph replays ...
    trainer.validate_step(frames, batch, model=ema.ema)
    evaluate_model(ema.ema, loader, device)
    trainer.ema = None                      # the default step again

Definition (ultralytics/utils/torch_utils.py, ModelEMA, 8.x): after update k (1-based), with
    d(k) = decay * (1 - exp(-k / tau)),
every floating-point entry v of the averaged model's state dict -- parameters (trainable or not) and the BatchNorm
running statistics -- becomes  v *= d;  v += (1 - d) * source.  Integer entries (num_batches_tracked) keep the value copied at creation.
Each tensor is averaged once, also where the state dict names it twice (detection_head.* and its alias model.0.*).

On the device: ``snn_ema_update`` reads row k-1 = {float(d(k)), float(1 - d(k))} of a table computed here once, indexed
by a device update counter that the call advances, so a captured training graph ramps the decay on replay with no host
work.  The table runs until both columns have reached float(decay) and float(1 - decay), so clamping to its last row is
exact for any number of updates.  The result is bit-identical to the two torch lines above on fp32 tensors.

Cost model: 12 B per parameter and update (read the source and the average, write the average), one launch for the flat
master buffer, one for all BatchNorm buffers and frozen parameters, one for the counter.  Memory: fp32 masters and bf16 operand copies of the
averaged model, no gradient or Adam-moment buffers.

Deliberate difference from ultralytics: the frozen feature extractor is SHARED with the live model, not copied.  Its
weights never change; ultralytics averages those constants with themselves, which moves them by up to an ulp per update.
"""
import copy
import math

import numpy as np
import torch

from . import kernels as K
from .params import ParamStore, store_for


def decay_table(decay=0.9999, tau=2000):
    """fp32 [rows, 2]: row k = (float(d(k+1)), float(1 - d(k+1))), d(x) = decay * (1 - exp(-x / tau)) evaluated in double
    precision as ultralytics does; the last row is the first at which both columns equal their limits."""
    _check(decay, tau)
    d_lim, omd_lim = _f32(decay), _f32(1.0 - decay)
    rows, k = [], 0
    while True:
        k += 1
        d = decay * (1 - math.exp(-k / tau))
        rows.append((d, 1 - d))
        if _f32(d) == d_lim and _f32(1 - d) == omd_lim:
            return torch.tensor(rows, dtype=torch.float64).float()


def _f32(x):
    return float(np.float32(x))


def _check(decay, tau):
    if not 0.0 < float(decay) < 1.0:
        raise ValueError(f"decay={decay} must be in (0, 1)")
    if not float(tau) > 0.0:
        raise ValueError(f"tau={tau} must be > 0")


def _segment_tensors(model):
    """[(module name, attribute)] of every floating-point state-dict entry outside the frozen extractor that the flat
    parameter store does not hold -- the BatchNorm running statistics and the frozen parameters (the Detect head's fixed
    DFL projection) -- each module once."""
    skip = {id(m) for m in model.feature_extractor.modules()}
    out = []
    for mname, mod in model.named_modules():
        if id(mod) in skip:
            continue
        for pname, p in mod.named_parameters(recurse=False):
            if not p.requires_grad and p.is_floating_point():
                out.append((mname, pname))
        for bname, b in mod.named_buffers(recurse=False):
            if b is not None and b.is_floating_point() and bname not in mod._non_persistent_buffers_set:
                out.append((mname, bname))
    return out


class ModelEMA:
    """ultralytics' ModelEMA(model, decay, tau, updates) for a YOLOTemporalUNet: `.ema` is the averaged model (eval mode,
    same device), `.updates` the number of updates so far (a host integer; never read from the device)."""

    def __init__(self, model, decay=0.9999, tau=2000, updates=0):
        _check(decay, tau)
        if int(updates) < 0:
            raise ValueError(f"updates={updates} must be >= 0")
        fe = model.feature_extractor
        if any(p.requires_grad for p in fe.parameters()):
            raise ValueError("ModelEMA shares the feature extractor with the model: it must be frozen")
        src = store_for(model, next(p for p in model.parameters() if p.requires_grad).device)
        self.device = src.device
        self.ema = _averaged_copy(model)
        dst = ParamStore(self.ema)
        dst.ensure(self.device, optimizer_state=False)
        # every module of the copy (the shared extractor excepted) names this store, so drop-in forwards of its submodules
        # (ema.ema.temporal_unet(...), ema.ema.detection_head(...)) find it once the parameters below are frozen
        shared = {id(m) for m in self.ema.feature_extractor.modules()}
        for m in self.ema.modules():
            if id(m) not in shared:
                object.__setattr__(m, "_snn_store", dst)
        if [(e.name, e.offset, e.numel) for e in dst.entries] != [(e.name, e.offset, e.numel) for e in src.entries]:
            raise RuntimeError("the averaged copy's parameter layout differs from the model's")
        for p in self.ema.parameters():          # after the store exists: ParamStore collects requires_grad parameters
            p.requires_grad_(False)
        self.ema.eval()
        dst.refresh_operands()
        self._src, self._dst, self._src_flat = src, dst, src.flat_p
        # BatchNorm running statistics and frozen parameters: one (source, destination, length) row per tensor, built once
        live, avg = dict(model.named_modules()), dict(self.ema.named_modules())
        rows, self._bufs = [], []
        for mname, bname in _segment_tensors(model):
            s, d = getattr(live[mname], bname), getattr(avg[mname], bname)
            if s.dtype != torch.float32 or not (s.is_contiguous() and d.is_contiguous()) or s.device != self.device:
                raise ValueError(f"{mname}.{bname}: averaged tensors must be contiguous fp32 on {self.device}")
            rows.append((s.data_ptr(), d.data_ptr(), s.numel()))
            # the table holds addresses: keep the tensors alive with it, and remember where they live to detect replacement
            self._bufs.append((s, d, live[mname], avg[mname], bname))
        self._segments = torch.tensor(rows, dtype=torch.int64).reshape(-1, 3).to(self.device) if rows else None
        self._segment_elems = sum(r[2] for r in rows)
        self.decay, self.tau = float(decay), float(tau)
        self._table = decay_table(self.decay, self.tau).to(self.device)
        self.updates = int(updates)
        self._updates_dev = torch.full((1,), self.updates, device=self.device, dtype=torch.int32)

    def update(self, model=None):
        """One update from the model this average was built from (the argument is accepted for ultralytics' signature).
        One enqueue, no host synchronisation."""
        if model is not None and getattr(model, "_snn_store", None) is not self._src:
            raise ValueError("ModelEMA.update: not the model this average was built from")
        if self._src.flat_p is not self._src_flat:
            raise RuntimeError("the model's parameter buffers were rebuilt (moved to another device?) after ModelEMA was "
                               "created: build a new ModelEMA")
        for s, d, live_m, avg_m, name in self._bufs:
            if getattr(live_m, name).data_ptr() != s.data_ptr() or getattr(avg_m, name).data_ptr() != d.data_ptr():
                raise RuntimeError(f"{name} of a BatchNorm / frozen module was replaced (e.g. load_state_dict(assign=True)) "
                                   "after ModelEMA was created: build a new ModelEMA")
        K.ema_update(self._dst.flat_p, self._src_flat, self._table, self._updates_dev, self._segments, self._segment_elems)
        self.advanced(1)

    def advanced(self, n):
        """Record n updates that ran on the device (update() itself, or replays of a captured graph that contains it; n < 0
        takes back the update a graph capture recorded without running).  The kernel writes the fp32 masters through raw
        pointers, so no Parameter version moves: the next forward of the averaged model must rebuild its bf16 operand
        copies -- once, however many updates came before it."""
        self.updates += n
        self._dst._versions = None

    def state_dict(self):
        """{'state_dict': fp32 CPU state dict of the averaged model (the model's key names), 'updates', 'decay', 'tau'}."""
        return {"state_dict": {k: v.detach().cpu().clone() for k, v in self.ema.state_dict().items()},
                "updates": self.updates, "decay": self.decay, "tau": self.tau}

    def load_state_dict(self, state):
        """Restores what state_dict() returned: weights, BatchNorm statistics, `updates` and the decay ramp."""
        decay, tau = float(state.get("decay", self.decay)), float(state.get("tau", self.tau))
        if (decay, tau) != (self.decay, self.tau):
            _check(decay, tau)
            self._table = decay_table(decay, tau).to(self.device)
            self.decay, self.tau = decay, tau
        # the extractor is shared with the live model and frozen: its keys are never loaded through the average
        sd = {k: v for k, v in state["state_dict"].items() if not k.startswith("feature_extractor.")}
        res = self.ema.load_state_dict(sd, strict=False)
        bad = [k for k in res.missing_keys if not k.startswith("feature_extractor.")] + list(res.unexpected_keys)
        if bad:
            raise RuntimeError(f"ModelEMA.load_state_dict: keys missing or unexpected: {bad[:8]}")
        self.updates = int(state["updates"])
        self._updates_dev.fill_(self.updates)
        self._dst._versions = None


def _averaged_copy(model):
    """Deep copy of `model` without its parameter store and spike statistics, sharing the frozen feature extractor."""
    memo = {id(model.feature_extractor): model.feature_extractor}
    for m in model.modules():
        for attr in ("_snn_store", "spike_stats"):
            v = getattr(m, attr, None)
            if v is not None:
                memo[id(v)] = None
    with torch.no_grad():
        out = copy.deepcopy(model, memo)
    shared = {id(m) for m in model.feature_extractor.modules()}
    for m in out.modules():
        if id(m) not in shared and "_snn_store" in m.__dict__:
            del m.__dict__["_snn_store"]
    return out
