"""Spike-activity statistics of the LIF layers -- firing rates and synaptic operations -- counted on the device by the
LIF forward kernel itself.

    stats = SpikeStats(model)               # model = YOLOTemporalUNet(neuron='lif') on its device
    model.spike_stats = stats               # every forward / forward_sequence now counts (train and eval mode)
    ... forwards, training steps, graph replays ...
    res = stats.compute()                   # {"spikes/rate": ..., "spikes/synops_fraction": ..., ...}
    stats.reset()
    model.spike_stats = None                # uncounted launches again

Definitions, per LIF layer l (the 16 ConvBlocks of TemporalUNet, by module name):
    S[l][t] = spikes at timestep t, N[l][t] = neurons that ran at t (exact integers, summed over every counted forward);
    rate = S / N;  F[l] = multiply-accumulates one spike-tensor element of l drives in the convs that consume it as
    spikes (TemporalUNet.spike_fanout);  SynOps = sum_l F[l] * sum_t S[l][t];  dense MACs = sum_l F[l] * sum_t N[l][t].
The frozen extractor, the ConvLSTM, the transposed-conv outputs and the SiLU Detect head are not counted.

Cost model: the counting launch (snn_bn_act_fwd_count) adds one popcount per 8 neurons and timestep, a warp and a block
reduction and one 64-bit atomic per block and timestep; the counters live in ONE int64 device buffer [layers][2][max_T]
that is never reallocated, so CUDA graphs captured with the stats attached keep counting on every replay.  Nothing on the
counting path reads the device from the host: ``compute`` is the one read.

SpikeRateLoss is the training-time counterpart: an activity regularizer on the same counts (one training step's), whose
gradient the LIF backward kernel adds to every spike's gradient (see its docstring and DESIGN.md section 3).
"""
import math

import numpy as np
import torch
import torch.distributed as dist

from . import kernels as K

MAX_T = 64          # timesteps one counted launch can tally (kCountMaxT in csrc/neuron.cu)


class _LayerCounters:
    """The LIF layers of a model (the 16 ConvBlocks of TemporalUNet, by module name, in module order), one int64 device
    buffer [layers][2][max_T] of per-timestep spike and neuron-step counts, and the fan-out table recorded by the first
    forward that counts.  Shared by SpikeStats and SpikeRateLoss."""

    def __init__(self, model, max_T=32):
        from .model import ConvBlock
        unet = model.temporal_unet
        self.layers = [n for n, m in unet.named_modules() if isinstance(m, ConvBlock) and m.neuron.kind == "lif"]
        if not self.layers:
            raise ValueError(f"{type(self).__name__} needs a model with LIF layers (this one was built with neuron='silu')")
        if not 1 <= int(max_T) <= MAX_T:
            raise ValueError(f"max_T={max_T} must be in [1, {MAX_T}]")
        self.max_T = int(max_T)
        self._index = {n: i for i, n in enumerate(self.layers)}
        p = next(unet.parameters())
        self.counts = torch.zeros((len(self.layers), 2, self.max_T), device=p.device, dtype=torch.int64)
        self.fanout = None          # {layer: F}, recorded by the first forward that counts; kept by reset()

    def begin_forward(self, unet, T, feature_hw, device):
        """Called by the model before a counted forward launches anything: checks T, the device and the fan-out table."""
        if T > self.max_T:
            raise ValueError(f"a forward over T={T} timesteps does not fit {type(self).__name__}(max_T={self.max_T})")
        if torch.device(device) != self.counts.device:
            raise ValueError(f"forward on {device}, spike counters on {self.counts.device}")
        table = unet.spike_fanout(feature_hw)
        if self.fanout is None:
            self.fanout = table
        elif table != self.fanout:
            raise ValueError("this forward's spike fan-out table differs from the one recorded by earlier counted forwards "
                             "(e.g. frame sizes with and without a resized skip): SynOps would mix two networks; use one "
                             f"{type(self).__name__} per frame size")

    def layer_counts(self, name, T):
        """(spikes [T], steps [T]) int64 views of one layer's counters (what the LIF launch adds into)."""
        i = self._index[name]
        return self.counts[i, 0, :T], self.counts[i, 1, :T]


class SpikeStats(_LayerCounters):
    """Per-layer, per-timestep spike and neuron-step counters of a LIF model.  `max_T`: the longest window counted."""

    def reset(self):
        """Zero the counters in place (no host synchronisation; captured graphs stay valid)."""
        self.counts.zero_()

    def compute(self, process_group=None):
        """Results over everything counted since the last reset.  With a process group the counters of all ranks are
        summed first (one all_reduce); every rank gets the same result.  One device-to-host read."""
        buf = self.counts
        if process_group is not None:
            buf = buf.clone()
            dist.all_reduce(buf, group=process_group)
        return self.results(buf.cpu().numpy())

    def results(self, counts):
        """Host side of compute(): counts = int64 numpy [layers][2][max_T] (spikes, neuron-steps)."""
        spikes, steps = counts[:, 0, :], counts[:, 1, :]
        seen = np.nonzero(steps.any(axis=0))[0]
        T_seen = int(seen[-1]) + 1 if seen.size else 0
        spikes, steps = spikes[:, :T_seen], steps[:, :T_seen]
        s_l = [int(v) for v in spikes.sum(axis=1)]
        n_l = [int(v) for v in steps.sum(axis=1)]
        rate = lambda s, n: s / n if n else float("nan")
        fan = self.fanout or {}
        synops = sum(fan.get(name, 0.0) * s for name, s in zip(self.layers, s_l))
        dense = sum(fan.get(name, 0.0) * n for name, n in zip(self.layers, n_l))
        res = {"spikes/rate": rate(sum(s_l), sum(n_l))}
        for name, s, n in zip(self.layers, s_l, n_l):
            res[f"spikes/rate/{name}"] = rate(s, n)
        res["spikes/synops"] = float(synops)
        res["spikes/dense_macs"] = float(dense)
        res["spikes/synops_fraction"] = rate(synops, dense)
        res["rate_per_t"] = np.where(steps > 0, spikes / np.maximum(steps, 1), np.nan)
        res["spike_counts"] = spikes.astype(np.int64)
        res["neuron_steps"] = steps.astype(np.int64)
        return res


class SpikeRateLoss(_LayerCounters):
    """Activity regularizer of the LIF layers: a penalty on this training step's SynOps fraction (upper bound) and on
    per-layer firing rates (lower bound), trained through the LIF backward kernel.

        reg = SpikeRateLoss(model, synops_weight=1.0, synops_max=0.05, rate_min=0.01, rate_min_weight=0.1)
        trainer.spike_reg = reg                 # train_step / train_step_graphed now minimise loss*B + B*P
        ... steps ...
        reg.read()                              # {"spike_reg/penalty": P, "spike_reg/synops_fraction": phi, ...}
        trainer.spike_reg = None

    Per step (and per rank), over the layers l = 1..L of `layers` (S_l spikes and N_l neuron-steps of this step's forward,
    all T timesteps; F_l the fan-out table of SpikeStats; D = sum_l F_l N_l):
        R_l = S_l / N_l,  phi = sum_l F_l S_l / D   (this step's spikes/synops_fraction)
        P   = synops_weight * max(0, phi - synops_max)^2 + (rate_min_weight / L) * sum_l max(0, rate_min - R_l)^2
    The step minimises loss*B + B*P (B = per-rank batch: the v8DetectionLoss convention, so the weights sit on the scale
    of the box / cls / dfl gains).  The gradient of B*P w.r.t. one spike of layer l is the same for every neuron and
    timestep, c_l = B * dP/dS_l; snn_spike_reg_coef computes it on the device after the counted forward, and
    snn_bn_act_bwd2_ds adds it to dL/ds in fp32 inside the reverse-time surrogate scan (a bf16 add onto the spike
    gradient in autograd would round it away wherever the detection gradient is ~2^9 times larger).  Under DDP the counts
    are the rank's own, like BatchNorm statistics: no extra collective, and the averaged gradient is the mean of the
    per-rank penalties' gradients.

    `coef` (fp32 [L]) and `last` (fp32 [2 + L] = P, phi, R_1..R_L of the latest step) are device tensors written by every
    step (and graph replay); `read()` is the one host read.  No learned state."""

    def __init__(self, model, synops_weight, synops_max=0.0, rate_min=0.0, rate_min_weight=0.0, max_T=32):
        for name, v in (("synops_weight", synops_weight), ("rate_min_weight", rate_min_weight)):
            if not (math.isfinite(float(v)) and float(v) >= 0.0):
                raise ValueError(f"{name}={v} must be a finite number >= 0")
        for name, v in (("synops_max", synops_max), ("rate_min", rate_min)):
            if not 0.0 <= float(v) <= 1.0:
                raise ValueError(f"{name}={v} must be in [0, 1]")
        super().__init__(model, max_T)
        self.synops_weight, self.synops_max = float(synops_weight), float(synops_max)
        self.rate_min, self.rate_min_weight = float(rate_min), float(rate_min_weight)
        dev = self.counts.device
        self.coef = torch.zeros(len(self.layers), device=dev, dtype=torch.float32)
        self.last = torch.zeros(2 + len(self.layers), device=dev, dtype=torch.float32)
        self._fanout_dev = None     # fp64 [L] copy of the fan-out table, made once (before any graph capture)
        self.epoch_mean = None      # mean P of the last epoch run by train.train_one_epoch

    def begin_forward(self, unet, T, feature_hw, device):
        super().begin_forward(unet, T, feature_hw, device)
        if self._fanout_dev is None:
            self._fanout_dev = torch.tensor([self.fanout[n] for n in self.layers], device=self.counts.device,
                                            dtype=torch.float64)

    def layer_grad(self, name):
        """One-element fp32 view of c_l: what the layer's LIF backward adds to every dL/ds."""
        i = self._index[name]
        return self.coef[i:i + 1]

    def begin_step(self):
        """Zero the step's counters (a memset: captured with the step, no host synchronisation)."""
        self.counts.zero_()

    def finish_forward(self, batch_size, T, stats=None):
        """After the step's counted forward: P, phi, R and c from the counts (one launch).  `stats`: an attached SpikeStats
        that also receives the step's counts from the same launch (its forward counting is not repeated)."""
        K.spike_reg_coef(self.counts, self._fanout_dev, self.coef, self.last, self.synops_weight, self.synops_max,
                         self.rate_min, self.rate_min_weight, batch_size, stats=None if stats is None else stats.counts, T=T)

    def read(self):
        """The latest step's penalty, SynOps fraction and per-layer rates (one device-to-host read)."""
        host = self.last.cpu().tolist()
        res = {"spike_reg/penalty": host[0], "spike_reg/synops_fraction": host[1]}
        res.update({f"spike_reg/rate/{n}": host[2 + i] for i, n in enumerate(self.layers)})
        return res
