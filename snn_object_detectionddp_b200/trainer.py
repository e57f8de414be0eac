"""Training step of the reference (train.py:48-104, 155-169) on the B200 path.

    zero_grad -> T-step unroll with state carry (fused: one launch sequence per LAYER over the folded T*B batch)
    -> v8DetectionLoss on the LAST step -> backward -> [DDP bucketed all-reduce, overlapped] ->
    clip_grad_norm_(10) + AdamW fused over the flat buffers -> OneCycleLR advance

Nothing in a step reads device memory from the host: the OneCycle schedule (lr and cycled beta1, torch defaults
div_factor 25 / final_div_factor 1e4 / pct_start 0.3 / cos) is tabulated once into a device array the optimizer kernel
indexes, and loss values are returned as device tensors (the caller decides when to ``.item()``; the reference syncs
3-5 times per batch, train.py:81-100).
"""
import math
import os

import torch
import torch.distributed as dist

from . import kernels as K
from .ddp import GradBucketer, broadcast_module_state
from .loss import batch_targets, pad_targets, v8DetectionLoss
from .params import store_for


def one_cycle_table(total_steps, max_lr, weight_decay, pct_start=0.3, div_factor=25.0, final_div_factor=1e4,
                    base_momentum=0.85, max_momentum=0.95, beta2=0.999, eps=1e-8, max_norm=10.0):
    """Row k = hyper-parameters of optimizer step k (0-based): torch.optim.lr_scheduler.OneCycleLR(anneal 'cos',
    cycle_momentum) driving torch.optim.AdamW, as configured at reference train.py:156-169.
    Columns: lr, beta1, beta2, eps, weight_decay, 1-beta1^(k+1), 1-beta2^(k+1), max_norm."""
    initial_lr, min_lr = max_lr / div_factor, max_lr / div_factor / final_div_factor
    end1, end2 = float(pct_start * total_steps) - 1.0, float(total_steps - 1)

    def cos_anneal(start, end, pct):
        return end + (start - end) / 2.0 * (math.cos(math.pi * pct) + 1.0)

    rows = []
    for k in range(total_steps):
        if k <= end1:
            pct = k / end1 if end1 > 0 else 1.0
            lr, b1 = cos_anneal(initial_lr, max_lr, pct), cos_anneal(max_momentum, base_momentum, pct)
        else:
            pct = (k - end1) / (end2 - end1) if end2 > end1 else 1.0
            lr, b1 = cos_anneal(max_lr, min_lr, pct), cos_anneal(base_momentum, max_momentum, pct)
        rows.append([lr, b1, beta2, eps, weight_decay, 1.0 - b1 ** (k + 1), 1.0 - beta2 ** (k + 1), max_norm])
    return torch.tensor(rows, dtype=torch.float64)


class Trainer:
    def __init__(self, model, max_lr=1e-4, weight_decay=5e-4, total_steps=1000, max_norm=10.0, device=None,
                 process_group=None, bucket_mb=32):
        self.model = model
        self.device = torch.device(device if device is not None else "cuda")
        model.to(self.device)
        self.store = store_for(model, self.device)
        self.loss_fn = v8DetectionLoss(model)
        self.hp = one_cycle_table(total_steps, max_lr, weight_decay, max_norm=max_norm).float().to(self.device)
        self.total_steps = total_steps
        self.step_idx = 0
        self._step_dev = torch.zeros(1, device=self.device, dtype=torch.int32)     # device-side schedule cursor
        self._graph = self._graph_key = None
        self._graph_failed = False
        self._eager_calls = 0
        self._sumsq = torch.zeros(1, device=self.device, dtype=torch.float64)
        self.grad_norm = torch.zeros(1, device=self.device, dtype=torch.float32)
        self._ones3 = torch.ones(3, device=self.device, dtype=torch.float32)
        # ema.ModelEMA: while set, every optimizer step also updates this weight average (captured graphs key on it)
        self.ema = None
        # spikes.SpikeRateLoss: while set, every training step also minimises B * its penalty (captured graphs key on it)
        self.spike_reg = None
        self.group = process_group
        self.world = dist.get_world_size(process_group) if dist.is_initialized() else 1
        self.bucketer = None
        if self.world > 1:
            # Dynamic tile scheduling of the persistent conv kernels (work stealing from SMs slowed down by NCCL CTAs) was
            # measured at 8 GPUs: 11.08 ms/step vs 10.75 ms with the static walk (profiles/README.md, negative results):
            # the ring hand-off costs more than the stealing recovers.  Kept selectable, off by default.
            K._lib.lib().snn_set_tile_scheduling(int(os.environ.get("SNN_DYNAMIC_TILES", "0")))
            broadcast_module_state(model, self.store.flat_p, process_group)
            self.store._versions = None       # masters changed under the bf16 operand copies
            spans = [(e.offset, self._padded(e)) for e in self.store.entries]
            self.bucketer = GradBucketer(self.store.flat_g, spans, bucket_mb << 20, process_group)
            index = {id(e): i for i, e in enumerate(self.store.entries)}
            self.store.grad_ready_hook = lambda e: self.bucketer.entry_ready(index[id(e)])

    def _padded(self, e):
        i = self.store.entries.index(e)
        nxt = self.store.entries[i + 1].offset if i + 1 < len(self.store.entries) else self.store.total
        return nxt - e.offset

    # ------------------------------------------------------------------------------------------
    def prepare_batch(self, labels, batch_size, max_boxes=None):
        """Host-side label padding ([M,6] collate layout, train.py:27-37) -> dict accepted by the loss.
        Pass `max_boxes` for a fixed shape (required by train_step_graphed)."""
        return {"padded": pad_targets(labels, batch_size, max_boxes=max_boxes)}

    def train_step(self, frames, batch):
        """frames fp32 [B,T,3,H,W] on the device; batch = {'batch_idx','cls','bboxes'} (train.py:68-72) or
        prepare_batch(...).  Returns (loss*B [3], loss.detach() [3]) as DEVICE tensors.
        With `spike_reg` set, the forward counts into its per-step buffer (zeroed first), its coefficient launch runs before
        the loss, and the LIF backward adds the coefficients to the spike gradients; the return value is unchanged (the
        penalty is in spike_reg.last)."""
        model, st, reg = self.model, self.store, self.spike_reg
        model.train()
        st.zero_grad()
        if self.bucketer is not None:
            self.bucketer.begin_step()
        if reg is not None:
            reg.begin_step()
        det, _ = model.forward_sequence(frames, spike_reg=reg)
        if reg is not None:
            reg.finish_forward(frames.shape[0], frames.shape[1], getattr(model, "spike_stats", None))
        loss, items = self.loss_fn(det, batch)
        # = loss.sum().backward() of train.py:75-76 without the reduction / expand kernels
        torch.autograd.backward((loss,), (self._ones3,))
        if self.bucketer is not None:
            self.bucketer.finish()
        self.optimizer_step()
        return loss.detach(), items

    def optimizer_step(self):
        st = self.store
        K.grad_sumsq(st.flat_g, self._sumsq)
        K.adamw_step(st.flat_p, st.flat_g, st.flat_m, st.flat_v, st.shadow, self.hp, self._sumsq, self.grad_norm,
                     step=self._step_dev, zero_grad=True)
        st.grads_clean = True            # the optimizer pass zeroed the gradient buffer (next step's zero_grad is free)
        if self.ema is not None:
            self.ema.update()
        st.opt_epoch += 1
        self.step_idx += 1

    # ------------------------------------------------------------------------------------------
    def train_step_graphed(self, frames, batch, warmup_calls=2):
        """Same step, replayed from ONE captured CUDA graph (the ~1000 kernel launches of a step cost more host
        time than device time otherwise).  `batch` must be prepare_batch(..., max_boxes=M) so shapes are static.
        The first `warmup_calls` calls run eagerly (they are real steps); the next call captures, then replays.
        Returned tensors are the graph's static outputs: read them before the next call."""
        padded = batch["padded"]
        # attaching / detaching spike statistics (counted LIF forwards), a weight average (one more launch behind the
        # optimizer) or a spike-rate regularizer changes the captured launches: re-capture.  The key holds the objects, so the
        # buffers a captured graph writes live as long as the graph.
        key = (tuple(frames.shape), frames.dtype, tuple(tuple(t.shape) for t in padded), getattr(self.model, "spike_stats", None),
               self.ema, self.spike_reg)
        if self._graph_failed:
            return self.train_step(frames, {"padded": tuple(t.to(self.device) for t in padded)})
        if self._graph is not None and self._graph_key != key:
            self._graph, self._eager_calls = None, max(0, warmup_calls - 1)      # new shapes: one eager step, re-capture
        if self._graph is None:
            if self._eager_calls < warmup_calls:
                self._eager_calls += 1
                return self.train_step(frames, {"padded": tuple(t.to(self.device) for t in padded)})
            self._static_frames = frames.clone()
            self._static_padded = tuple(t.to(self.device).clone() for t in padded)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            try:
                # the bucketed NCCL all-reduces are captured too (side-stream branches of the graph overlapping backward)
                with torch.cuda.graph(g):
                    out = self.train_step(self._static_frames, {"padded": self._static_padded})
            except Exception as e:             # e.g. a collective backend that cannot be captured: stay eager, loudly
                import warnings
                warnings.warn(f"CUDA-graph capture of the training step failed ({type(e).__name__}: {e}); running eagerly")
                torch.cuda.synchronize()
                self._graph_failed = True
                return self.train_step(frames, {"padded": tuple(t.to(self.device) for t in padded)})
            self.step_idx -= 1                 # capture records the launches without running them
            self.store.opt_epoch -= 1
            if self.ema is not None:
                self.ema.advanced(-1)
            self._graph, self._graph_key, self._static_out = g, key, out
        st = self.store
        if tuple(e.param._version for e in st.entries) != st._versions:
            st.refresh_operands()              # masters were modified outside the optimizer (e.g. load_state_dict)
        self._static_frames.copy_(frames, non_blocking=True)
        for s_, t_ in zip(self._static_padded, padded):
            s_.copy_(t_, non_blocking=True)
        self._graph.replay()
        self.step_idx += 1
        st.opt_epoch += 1
        if self.ema is not None:
            self.ema.advanced(1)               # the replay ran the update kernel: the average's bf16 operands are stale
        return self._static_out

    # ------------------------------------------------------------------------------------------
    @torch.no_grad()
    def validate_step(self, frames, batch, metrics=None, conf_thres=0.001, iou_thres=0.6, max_det=300, model=None):
        """validate_one_epoch's inner step (reference train.py:106-131): eval mode (BatchNorm running statistics, state
        reset per window), loss on the last frame, no gradient.  Returns loss.detach() [3] as a DEVICE tensor.
        metrics: a metrics.DetMetrics -- the same forward is also decoded, put through NMS (eval_2.py:108 settings) and
        matched against the batch's targets, without a host synchronisation.
        model: the network to validate (default: the trained one; `self.ema.ema` validates the weight average)."""
        model = self.model if model is None else model
        was_training = model.training
        model.eval()
        try:
            det, _ = model.forward_sequence(frames)
            _, items = self.loss_fn(det, batch)
            if metrics is not None:
                from .infer import decode_head
                from .nms import non_max_suppression_padded
                rows, _, counts = non_max_suppression_padded(decode_head(model, det), conf_thres, iou_thres, max_det=max_det)
                metrics.update(rows, counts, batch_targets(batch, frames.shape[0], frames.device), frames.shape[-2:])
        finally:
            model.train(was_training)
        return items

    # ------------------------------------------------------------------------------------------
    def save_checkpoint(self, path, epoch=0, best_val_loss=float("inf")):
        """The reference's checkpoint dict (train.py:204-209: 'epoch', 'model_state_dict', 'best_val_loss') -- loadable
        by the reference's own `model.load_state_dict(ckpt['model_state_dict'])` for the temporal_unet / detection_head
        keys -- plus what the reference forgets (optimizer moments, schedule position) under 'trainer_state', and with a
        weight average attached its ModelEMA.state_dict() under 'ema' (ultralytics keeps it under 'ema' / 'updates')."""
        st = self.store
        ck = {"epoch": epoch, "model_state_dict": {k: v.detach().cpu().contiguous() for k, v in self.model.state_dict().items()},
              "best_val_loss": best_val_loss,
              "trainer_state": {"step_idx": self.step_idx, "total_steps": self.total_steps,
                                "exp_avg": st.flat_m.cpu(), "exp_avg_sq": st.flat_v.cpu(),
                                "layout": [(e.name, e.offset, e.numel) for e in st.entries]}}
        if self.ema is not None:
            ck["ema"] = self.ema.state_dict()
        torch.save(ck, path)

    def load_checkpoint(self, path, strict=True):
        """Accepts both this class's files and plain reference checkpoints (no 'trainer_state': moments restart at 0).
        The weight average is restored when the file and this trainer both have one; otherwise the file's 'ema' is ignored
        and an attached average is left as it is (ultralytics' resume without 'ema')."""
        ck = torch.load(path, map_location="cpu", weights_only=False)
        self.model.load_state_dict(ck["model_state_dict"], strict=strict)
        st = self.store.ensure(self.device)
        st._versions = None
        st.refresh_operands()
        ts = ck.get("trainer_state")
        if ts is not None and [(e.name, e.offset, e.numel) for e in st.entries] == [tuple(x) for x in ts["layout"]]:
            st.flat_m.copy_(ts["exp_avg"])
            st.flat_v.copy_(ts["exp_avg_sq"])
            self.step_idx = int(ts["step_idx"])
            self._step_dev.fill_(self.step_idx)
        if self.ema is not None and ck.get("ema") is not None:
            self.ema.load_state_dict(ck["ema"])
        self._graph = None                       # captured graphs hold the old buffers' contents only by address: still valid, but re-capture is cheap and safe
        return ck.get("epoch", 0), ck.get("best_val_loss", float("inf"))

    def lr(self):
        return float(self.hp[min(self.step_idx, self.total_steps - 1), 0])
