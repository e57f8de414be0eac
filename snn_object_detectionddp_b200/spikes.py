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
"""
import numpy as np
import torch
import torch.distributed as dist

MAX_T = 64          # timesteps one counted launch can tally (kCountMaxT in csrc/neuron.cu)


class SpikeStats:
    """Per-layer, per-timestep spike and neuron-step counters of a LIF model.  `max_T`: the longest window counted."""

    def __init__(self, model, max_T=32):
        from .model import ConvBlock
        unet = model.temporal_unet
        self.layers = [n for n, m in unet.named_modules() if isinstance(m, ConvBlock) and m.neuron.kind == "lif"]
        if not self.layers:
            raise ValueError("SpikeStats needs a model with LIF layers (this one was built with neuron='silu')")
        if not 1 <= int(max_T) <= MAX_T:
            raise ValueError(f"max_T={max_T} must be in [1, {MAX_T}]")
        self.max_T = int(max_T)
        self._index = {n: i for i, n in enumerate(self.layers)}
        p = next(unet.parameters())
        self.counts = torch.zeros((len(self.layers), 2, self.max_T), device=p.device, dtype=torch.int64)
        self.fanout = None          # {layer: F}, recorded by the first forward that counts; kept by reset()

    def reset(self):
        """Zero the counters in place (no host synchronisation; captured graphs stay valid)."""
        self.counts.zero_()

    def begin_forward(self, unet, T, feature_hw, device):
        """Called by the model before a counted forward launches anything: checks T, the device and the fan-out table."""
        if T > self.max_T:
            raise ValueError(f"a forward over T={T} timesteps does not fit SpikeStats(max_T={self.max_T})")
        if torch.device(device) != self.counts.device:
            raise ValueError(f"forward on {device}, spike counters on {self.counts.device}")
        table = unet.spike_fanout(feature_hw)
        if self.fanout is None:
            self.fanout = table
        elif table != self.fanout:
            raise ValueError("this forward's spike fan-out table differs from the one recorded by earlier counted forwards "
                             "(e.g. frame sizes with and without a resized skip): SynOps would mix two networks; use one "
                             "SpikeStats per frame size")

    def layer_counts(self, name, T):
        """(spikes [T], steps [T]) int64 views of one layer's counters (what the LIF launch adds into)."""
        i = self._index[name]
        return self.counts[i, 0, :T], self.counts[i, 1, :T]

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
