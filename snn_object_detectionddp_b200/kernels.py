"""Functional (non-autograd) wrappers: torch tensors in, libsnnb200 kernels launched on the current stream.

Activations are NHWC tensors ``[NB, H, W, C]`` (NB = T*B folded); a tensor may be a channel slice of
a wider buffer (``stride(2) = ld >= C``).  See include/snn_b200.h for the ABI.
"""
import torch

from . import _lib
from ._lib import (ACT_LIF, ACT_SILU, GEOM_1x1, GEOM_3x3_S1, GEOM_3x3_S2, GEOM_T2x2_S2, GEOM_TAPS, call, ptr,
                   require_cuda, stream_ptr)


def _nhwc_ld(x):
    """Validate an NHWC (channel-slice) view and return its pixel stride."""
    nb, h, w, c = x.shape
    ld = x.stride(2) if w > 1 else (x.stride(1) if h > 1 else (x.stride(0) if nb > 1 else c))
    if x.stride(3) != 1 and c > 1:
        raise ValueError("NHWC view must be channel-contiguous")
    if (w > 1 and x.stride(2) != ld) or (h > 1 and x.stride(1) != w * ld) or (nb > 1 and x.stride(0) != h * w * ld):
        raise ValueError(f"not a dense NHWC pixel grid: shape {tuple(x.shape)} strides {x.stride()}")
    return ld


def out_hw(geom, h, w):
    if geom == GEOM_3x3_S2:
        return h // 2, w // 2
    if geom == GEOM_T2x2_S2:
        return 2 * h, 2 * w
    return h, w


def _conv_flops(geom, nb, h, w, cin, cout):
    """Algorithmic flops of one pass (SURVEY.md 8d): 2 * output pixels * Cout * Cin * taps, padding not counted;
    (h, w) are the conv INPUT dims (transposed conv: every input pixel feeds 4 taps)."""
    ho, wo = out_hw(geom, h, w)
    if geom == GEOM_T2x2_S2:
        return 2.0 * nb * h * w * cout * cin * 4
    return 2.0 * nb * ho * wo * cout * cin * GEOM_TAPS[geom]


def conv_fprop(geom, x0, w_bf16, cout, x1=None, bias=None, out=None, out_dtype=torch.float32, w_coff=0, w_row_off=0,
               accumulate=False):
    """out[NB,Ho,Wo,cout] = conv(cat([x0,x1],C), W[w_row_off:w_row_off+cout, :, w_coff:...]) (+bias)."""
    require_cuda(x0, x1, w_bf16, bias, out)
    nb, h, w, c0 = x0.shape
    ho, wo = out_hw(geom, h, w)
    if out is None:
        out = torch.empty((nb, ho, wo, cout), device=x0.device, dtype=out_dtype)
    assert x0.dtype == torch.bfloat16 and w_bf16.dtype == torch.bfloat16 and w_bf16.is_contiguous()
    assert tuple(out.shape) == (nb, ho, wo, cout)
    rows, taps, wk = w_bf16.shape
    assert taps == GEOM_TAPS[geom]
    c1 = 0 if x1 is None else x1.shape[3]
    if x1 is not None:
        assert x1.dtype == torch.bfloat16 and tuple(x1.shape[:3]) == (nb, h, w)
    assert w_coff + c0 + c1 <= wk and w_row_off + cout <= rows
    call("snn_conv_fprop", geom, nb, h, w, ptr(x0), c0, _nhwc_ld(x0), ptr(x1), c1, 0 if x1 is None else _nhwc_ld(x1),
         ptr(w_bf16), rows, wk, w_coff, cout, w_row_off, ptr(bias), ptr(out), int(out.dtype == torch.float32),
         _nhwc_ld(out), 0, int(accumulate), stream_ptr(), work=("flop", _conv_flops(geom, nb, h, w, c0 + c1, cout), f"g{geom} nb{nb} {h}x{w} {c0 + c1}->{cout}"))
    return out


_STATS_GROUPS = {}


def conv_fprop_partials(geom, x0, w_bf16, cout, T, x1=None):
    """ConvBlock conv whose epilogue also emits the per-(32-pixel group, channel) BatchNorm partial sums.
    Returns (y fp32 [NB,Ho,Wo,cout], partials fp32 [groups][2][cout] | None, groups_per_timestep); partials is None when
    the geometry cannot keep every 128-pixel tile inside one timestep (then the caller runs bn_stats on y)."""
    require_cuda(x0, x1, w_bf16)
    nb, h, w, c0 = x0.shape
    key = (geom, nb, h, w, T)
    if key not in _STATS_GROUPS:
        gpt = _lib.ctypes.c_int(0)
        n = _lib.lib().snn_conv_stats_groups(geom, nb, h, w, nb // T, _lib.ctypes.byref(gpt)) if nb % T == 0 else 0
        _STATS_GROUPS[key] = (int(n), int(gpt.value))
    groups, gpt = _STATS_GROUPS[key]
    if groups == 0:
        return conv_fprop(geom, x0, w_bf16, cout, x1=x1), None, 0
    ho, wo = out_hw(geom, h, w)
    out = torch.empty((nb, ho, wo, cout), device=x0.device, dtype=torch.float32)
    rows, taps, wk = w_bf16.shape
    c1 = 0 if x1 is None else x1.shape[3]
    assert x0.dtype == torch.bfloat16 and w_bf16.dtype == torch.bfloat16 and w_bf16.is_contiguous() and taps == GEOM_TAPS[geom]
    assert c0 + c1 <= wk and cout <= rows
    part = torch.empty((groups, 2, cout), device=x0.device, dtype=torch.float32)
    call("snn_conv_fprop_stats", geom, nb, h, w, ptr(x0), c0, _nhwc_ld(x0), ptr(x1), c1, 0 if x1 is None else _nhwc_ld(x1),
         ptr(w_bf16), rows, wk, 0, cout, 0, ptr(out), nb // T, ptr(part), stream_ptr(),
         work=("flop", _conv_flops(geom, nb, h, w, c0 + c1, cout), f"g{geom} nb{nb} {h}x{w} {c0 + c1}->{cout}"))
    return out, part, gpt


def conv_fprop_stats(geom, x0, w_bf16, cout, T, x1=None):
    """conv_fprop_partials + the fixed-order reduce: returns (y, sums fp64 [T][2][cout] | None)."""
    out, part, gpt = conv_fprop_partials(geom, x0, w_bf16, cout, T, x1=x1)
    if part is None:
        return out, None
    sums = torch.empty((T, 2, cout), device=x0.device, dtype=torch.float64)
    call("snn_bn_stats_from_partials", ptr(part), ptr(sums), T, cout, gpt, stream_ptr(), work=("byte", 4.0 * part.numel()))
    return out, sums


def bn_finalize_partials(part, gpt, gamma, beta, running_mean, running_var, num_batches_tracked, counters, T, C, P, eps, momentum):
    """Partials -> (scale, shift, mean, invstd) [T][C] + the T running-statistics updates + num_batches_tracked += T,
    in one launch.  `counters`: persistent zeroed uint32 [ceil(C/8)] (the kernel leaves it zeroed)."""
    require_cuda(part, gamma, beta, running_mean, running_var, num_batches_tracked, counters)
    dev = part.device
    scale, shift, mean, invstd = (torch.empty((T, C), device=dev, dtype=torch.float32) for _ in range(4))
    sums = torch.empty((T, 2, C), device=dev, dtype=torch.float64)
    ws = torch.empty((int(_lib.lib().snn_bn_finalize_workspace_doubles(T, C, gpt)),), device=dev, dtype=torch.float64)
    assert counters.dtype == torch.int32 and counters.numel() >= (C + 31) // 32
    assert num_batches_tracked is None or num_batches_tracked.dtype == torch.int64
    call("snn_bn_finalize_partials", ptr(part), ptr(sums), ptr(ws), ptr(gamma), ptr(beta), ptr(running_mean), ptr(running_var),
         ptr(num_batches_tracked), ptr(scale), ptr(shift), ptr(mean), ptr(invstd), ptr(counters), T, C, P, gpt, float(eps),
         float(momentum), stream_ptr(), work=("byte", 4.0 * part.numel()))
    return scale, shift, mean, invstd


def conv_dgrad(geom, dy, w_bf16, in_hw, ci, ci_off=0, out=None, out_dtype=torch.bfloat16, accumulate=False):
    """dx[NB,H,W,ci] for the conv-input channel range [ci_off, ci_off+ci); w_bf16 = the fprop weights
    [Cout][taps][Cin_tot], read in place."""
    require_cuda(dy, w_bf16, out)
    nb, hy, wy, cout = dy.shape
    h, w = in_hw
    assert out_hw(geom, h, w) == (hy, wy), (geom, in_hw, dy.shape)
    rows, taps, wk = w_bf16.shape
    assert taps == GEOM_TAPS[geom] and rows == cout and ci_off + ci <= wk
    assert dy.dtype == torch.bfloat16 and w_bf16.dtype == torch.bfloat16 and w_bf16.is_contiguous()
    if out is None:
        out = torch.empty((nb, h, w, ci), device=dy.device, dtype=out_dtype)
    call("snn_conv_dgrad", geom, nb, h, w, ptr(dy), cout, _nhwc_ld(dy), ptr(w_bf16), wk, ci_off, ci, ptr(out),
         int(out.dtype == torch.float32), _nhwc_ld(out), 0, int(accumulate), stream_ptr(),
         work=("flop", _conv_flops(geom, nb, h, w, ci, cout), f"g{geom} nb{nb} {h}x{w} {ci}<-{cout}"))
    return out


def conv_wgrad(geom, x, dy, dw, w_coff=0):
    """dw[Cout][taps][wK] (fp32) += wgrad; x is the conv input NHWC bf16, dy the output gradient NHWC bf16."""
    require_cuda(x, dy, dw)
    nb, h, w, ci = x.shape
    cout = dy.shape[3]
    assert tuple(dy.shape[:3]) == (nb,) + out_hw(geom, h, w)
    rows, taps, wk = dw.shape
    assert rows == cout and taps == GEOM_TAPS[geom] and w_coff + ci <= wk
    assert dw.dtype == torch.float32 and dw.is_contiguous() and x.dtype == torch.bfloat16 and dy.dtype == torch.bfloat16
    call("snn_conv_wgrad", geom, nb, h, w, ptr(x), ci, _nhwc_ld(x), ptr(dy), cout, _nhwc_ld(dy), ptr(dw), wk, w_coff,
         stream_ptr(), work=("flop", _conv_flops(geom, nb, h, w, ci, cout), f"g{geom} nb{nb} {h}x{w} {ci}x{cout}"))
    return dw


PLAN_FIELDS = ("bn", "bh", "bw", "n_tile", "pair", "strip", "hnw", "stages", "stage_bytes", "chunks_per_stage", "ksplit", "items",
               "n_blocks", "ctas", "epi_groups", "small_k", "tma_out", "smem_bytes", "a_bytes", "b_bytes")


def conv_plan(kind, geom, nb, h, w, cin, cout, out_f32=True, frames_per_step=0, accumulate=False):
    """Launch plan of conv_fprop ('fprop') / conv_dgrad ('dgrad') / conv_wgrad ('wgrad') for these shapes, without launching
    (host logic only: works without a GPU).  Returns a dict over PLAN_FIELDS (see snn_conv_plan in include/snn_b200.h)."""
    import ctypes
    out = (ctypes.c_int * 20)()
    rc = _lib.lib().snn_conv_plan({"fprop": 0, "dgrad": 1, "wgrad": 2}[kind], geom, nb, h, w, cin, cout, int(out_f32), frames_per_step,
                             int(accumulate), out)
    if rc:
        raise _lib.SnnKernelError(f"snn_conv_plan failed (rc={rc}): {_lib.lib().snn_last_error().decode()}")
    return dict(zip(PLAN_FIELDS, list(out)))


def weight_prep(w_master, want_fprop=True, want_dgrad=True, wf=None, wt=None):
    """fp32 [N][T][K] -> (bf16 [N][T][K], bf16 [K][T][N])."""
    require_cuda(w_master)
    n, t, k = w_master.shape
    assert w_master.is_contiguous() and w_master.dtype == torch.float32
    if want_fprop and wf is None:
        wf = torch.empty((n, t, k), device=w_master.device, dtype=torch.bfloat16)
    if want_dgrad and wt is None:
        wt = torch.empty((k, t, n), device=w_master.device, dtype=torch.bfloat16)
    call("snn_weight_prep", ptr(w_master), ptr(wf), ptr(wt), n, t, k, stream_ptr())
    return wf, wt


# ---------------------------------------------------------------------------------------------
# neuron layer
# ---------------------------------------------------------------------------------------------
def bn_stats(y, T):
    """y fp32 [T*B, H, W, C] -> sums fp64 [T][2][C]."""
    require_cuda(y)
    c = y.shape[-1]
    p = y.numel() // (T * c)
    sums = torch.empty((T, 2, c), device=y.device, dtype=torch.float64)
    ws = torch.empty((int(_lib.lib().snn_bn_stats_workspace_floats(T, p, c)),), device=y.device, dtype=torch.float32)
    call("snn_bn_stats", ptr(y), ptr(sums), ptr(ws), T, p, c, stream_ptr(), work=("byte", 4.0 * y.numel()))
    return sums


def bn_finalize(sums, gamma, beta, running_mean, running_var, T, C, P, eps, momentum, training):
    require_cuda(sums, gamma, beta, running_mean, running_var)
    dev = gamma.device
    n = T if training else 1
    scale, shift, mean, invstd = (torch.empty((n, C), device=dev, dtype=torch.float32) for _ in range(4))
    call("snn_bn_finalize", ptr(sums), ptr(gamma), ptr(beta), ptr(running_mean), ptr(running_var), ptr(scale), ptr(shift),
         ptr(mean), ptr(invstd), T, C, P, float(eps), float(momentum), int(training), stream_ptr())
    return scale, shift, mean, invstd


def bn_act_fwd(act, y, scale, shift, T, v_init=None, want_mask=True, want_v_final=False, beta=0.5, theta=1.0,
               spike_counts=None):
    """Fused BN affine + LIF scan over T (or SiLU).  y fp32 [T*B,H,W,C] -> bf16 same shape (+mask, +v_final).
    spike_counts: (spikes, steps) int64 device views of >= T elements (LIF only); the launch adds the number of spikes
    of timestep t to spikes[t] and the number of neurons per timestep to steps[t].  Outputs are unchanged."""
    if spike_counts is not None and act != ACT_LIF:
        raise _lib.SnnKernelError("bn_act_fwd: spike counting needs the LIF neuron")
    require_cuda(y, scale, shift, v_init, *(spike_counts or ()))
    c = y.shape[-1]
    n_per_t = y.numel() // T
    out = torch.empty(y.shape, device=y.device, dtype=torch.bfloat16)
    mask = torch.empty((T, n_per_t // 8), device=y.device, dtype=torch.uint8) if (want_mask and act == ACT_LIF) else None
    v_final = torch.empty((n_per_t,), device=y.device, dtype=torch.float32) if want_v_final else None
    ss = c if scale.shape[0] == T and scale.dim() == 2 and scale.shape[0] > 1 else 0
    if scale.dim() == 2 and scale.shape[0] == 1:
        ss = 0
    if T == 1:
        ss = 0
    # algorithmic bytes per neuron-timestep (SURVEY.md 8d): 4 (y fp32) + 2 (spike bf16) + 1/8 (packed mask)
    nbytes = y.numel() * (6.0 + (0.125 if mask is not None else 0.0))
    nbytes += (0 if v_init is None else 4.0 * n_per_t) + (0 if v_final is None else 4.0 * n_per_t)
    if spike_counts is not None:
        spikes, steps = spike_counts
        for t in (spikes, steps):
            if t.dtype != torch.int64 or not t.is_contiguous() or t.numel() < T:
                raise ValueError(f"spike_counts: contiguous int64 views of >= T={T} elements required, got {t.dtype} "
                                 f"{tuple(t.shape)} contiguous={t.is_contiguous()}")
        call("snn_bn_act_fwd_count", ptr(y), ptr(scale), ptr(shift), ptr(v_init), ptr(out), ptr(mask), ptr(v_final), ptr(spikes),
             ptr(steps), T, n_per_t, c, ss, float(beta), float(theta), stream_ptr(), work=("byte", nbytes, f"T{T} n{n_per_t} C{c}"))
        return out, mask, v_final
    call("snn_bn_act_fwd", act, ptr(y), ptr(scale), ptr(shift), ptr(v_init), ptr(out), ptr(mask), ptr(v_final), T, n_per_t,
         c, ss, float(beta), float(theta), stream_ptr(), work=("byte", nbytes, f"T{T} n{n_per_t} C{c}"))
    return out, mask, v_final


def bn_act_bwd(act, training, y, scale, shift, mean, invstd, gs, T, v_init=None, gv_final=None, want_gv_init=False,
               beta=0.5, theta=1.0, alpha=2.0):
    """Returns (gx fp32 | None, dy bf16 | None, gv_init | None, red [T][2][C] | None)."""
    require_cuda(y, scale, shift, mean, invstd, gs, v_init, gv_final)
    c = y.shape[-1]
    p = y.numel() // (T * c)
    dev = y.device
    gx = torch.empty(y.shape, device=dev, dtype=torch.float32) if training else None
    dy = None if training else torch.empty(y.shape, device=dev, dtype=torch.bfloat16)
    red = torch.empty((T, 2, c), device=dev, dtype=torch.float32) if training else None
    gv_init = torch.empty((p * c,), device=dev, dtype=torch.float32) if want_gv_init else None
    ss = 0 if (T == 1 or scale.shape[0] == 1) else c
    assert gs.dtype == torch.bfloat16 and gs.is_contiguous()
    # algorithmic bytes per neuron-timestep: 2 (gs bf16) + 4 (y fp32, membrane recomputed) + 4 (gx fp32) | 2 (dy bf16)
    nbytes = y.numel() * (10.0 if training else 8.0)
    call("snn_bn_act_bwd", act, int(training), ptr(y), ptr(scale), ptr(shift), ptr(mean), ptr(invstd), ptr(v_init), ptr(gs),
         ptr(gv_final), ptr(gx), ptr(dy), ptr(gv_init), ptr(red), T, p, c, ss, float(beta), float(theta), float(alpha),
         stream_ptr(), work=("byte", nbytes))
    return gx, dy, gv_init, red


def bn_act_bwd_train(act, y, scale, shift, mean, invstd, beta_bn, gs, T, dgamma, dbeta, v_init=None, gv_final=None,
                     want_gv_init=False, beta=0.5, theta=1.0, alpha=2.0, ds_add=None):
    """Train-mode (batch-statistics) backward of BN -> LIF|SiLU in two recompute passes (no fp32 gx round trip).
    Returns (dy bf16, gv_init | None, red [T][2][C]); dgamma / dbeta (fp32 [C]) are accumulated into.
    ds_add (LIF only): one-element fp32 device tensor added to every dL/ds in fp32 before the surrogate multiply
    (snn_bn_act_bwd2_ds; the spike-rate regularizer's c_l)."""
    require_cuda(y, scale, shift, mean, invstd, beta_bn, gs, dgamma, dbeta, v_init, gv_final, ds_add)
    if ds_add is not None:
        if act != ACT_LIF:
            raise _lib.SnnKernelError("bn_act_bwd_train: ds_add needs the LIF neuron")
        if ds_add.dtype != torch.float32 or ds_add.numel() != 1:
            raise ValueError(f"ds_add: a one-element fp32 device tensor required, got {ds_add.dtype} {tuple(ds_add.shape)}")
    c = y.shape[-1]
    p = y.numel() // (T * c)
    dev = y.device
    assert gs.dtype == torch.bfloat16 and gs.is_contiguous() and y.is_contiguous()
    assert scale.shape[0] == T and mean.shape[0] == T
    red = torch.empty((T, 2, c), device=dev, dtype=torch.float32)
    dy = torch.empty(y.shape, device=dev, dtype=torch.bfloat16)
    gv_init = torch.empty((p * c,), device=dev, dtype=torch.float32) if want_gv_init else None
    args = (ptr(y), ptr(scale), ptr(shift), ptr(mean), ptr(invstd), ptr(beta_bn), ptr(v_init), ptr(gs), ptr(gv_final), ptr(red),
            ptr(dy), ptr(gv_init), ptr(dgamma), ptr(dbeta), T, p, c, float(beta), float(theta), float(alpha), stream_ptr())
    tag = f"T{T} n{p * c} C{c}"
    if ds_add is not None:      # same bytes: the addend is one broadcast float
        call("snn_bn_act_bwd2_ds", 0, act, *args[:-1], ptr(ds_add), args[-1], work=("byte", 6.0 * y.numel(), "reduce " + tag))
        call("snn_bn_act_bwd2_ds", 1, act, *args[:-1], ptr(ds_add), args[-1], work=("byte", 8.0 * y.numel(), "dx " + tag))
        return dy, gv_init, red
    call("snn_bn_act_bwd2", 0, act, *args, work=("byte", 6.0 * y.numel(), "reduce " + tag))   # reads y fp32 + gs bf16
    call("snn_bn_act_bwd2", 1, act, *args, work=("byte", 8.0 * y.numel(), "dx " + tag))       # reads y + gs, writes dy bf16
    return dy, gv_init, red


def spike_reg_coef(counts, fanout, coef, out, synops_weight, synops_max, rate_min, rate_min_weight, batch_size, stats=None, T=0):
    """Spike-rate regularizer of one step (spikes.SpikeRateLoss), one launch: counts int64 [L][2][max_T] and fanout fp64
    [L] -> coef fp32 [L] (each layer's dL/ds addend) and out fp32 [2 + L] = (P, phi, R_1..R_L).  stats: a SpikeStats
    counts buffer int64 [L][2][stats_max_T] that also receives counts[:, :, :T]."""
    require_cuda(counts, fanout, coef, out, stats)
    if counts.dtype != torch.int64 or counts.dim() != 3 or counts.shape[1] != 2 or not counts.is_contiguous():
        raise ValueError(f"spike_reg_coef: counts must be contiguous int64 [L][2][max_T], got {counts.dtype} {tuple(counts.shape)}")
    L, max_T = counts.shape[0], counts.shape[2]
    for name, t, dt, n in (("fanout", fanout, torch.float64, L), ("coef", coef, torch.float32, L), ("out", out, torch.float32, L + 2)):
        if t is None or t.dtype != dt or t.numel() != n or not t.is_contiguous():
            raise ValueError(f"spike_reg_coef: {name} must be a contiguous {dt} tensor of {n} elements")
    smt = 0
    if stats is not None:
        if stats.dtype != torch.int64 or tuple(stats.shape[:2]) != (L, 2) or stats.dim() != 3 or not stats.is_contiguous():
            raise ValueError(f"spike_reg_coef: stats must be contiguous int64 [{L}][2][max_T], got {stats.dtype} {tuple(stats.shape)}")
        smt = stats.shape[2]
    call("snn_spike_reg_coef", ptr(counts), ptr(fanout), L, max_T, float(synops_weight), float(synops_max), float(rate_min),
         float(rate_min_weight), float(batch_size), ptr(coef), ptr(out), ptr(stats), smt, int(T), stream_ptr(),
         work=("byte", 8.0 * counts.numel() + 8.0 * L + 4.0 * (2 * L + 2) + (16.0 * L * T if stats is not None else 0.0)))


def bn_bwd_dx(red, gamma, gx, y, scale, mean, invstd, dgamma, dbeta, T):
    require_cuda(red, gamma, gx, y, scale, mean, invstd, dgamma, dbeta)
    c = y.shape[-1]
    p = y.numel() // (T * c)
    coef = torch.empty((T, 2, c), device=y.device, dtype=torch.float32)
    dy = torch.empty(y.shape, device=y.device, dtype=torch.bfloat16)
    call("snn_bn_bwd_dx", ptr(red), ptr(gamma), ptr(gx), ptr(y), ptr(scale), ptr(mean), ptr(invstd), ptr(coef), ptr(dgamma),
         ptr(dbeta), ptr(dy), T, p, c, stream_ptr(), work=("byte", 10.0 * y.numel()))
    return dy


# ---------------------------------------------------------------------------------------------
# ConvLSTM gates, layout conversion, optimizer
# ---------------------------------------------------------------------------------------------
def lstm_gates_fwd(gates, c_prev, ch, h_bf16_out=None, c_out=None):
    require_cuda(gates, c_prev, h_bf16_out, c_out)
    p = gates.numel() // (4 * ch)
    shape = gates.shape[:-1] + (ch,)
    c_next = torch.empty(shape, device=gates.device, dtype=torch.float32) if c_out is None else c_out
    h_next = torch.empty(shape, device=gates.device, dtype=torch.float32)
    h_bf16 = torch.empty(shape, device=gates.device, dtype=torch.bfloat16) if h_bf16_out is None else h_bf16_out
    assert gates.is_contiguous() and c_next.is_contiguous() and h_bf16.is_contiguous()
    call("snn_lstm_gates_fwd", ptr(gates), ptr(c_prev), ptr(c_next), ptr(h_next), ptr(h_bf16), p, ch, stream_ptr())
    return h_next, c_next, h_bf16


def lstm_gates_bwd(gates, c_prev, c_next, dh, dc_in, ch, dgates_out=None, dh_bf16=None):
    """dh (fp32 | None) + dh_bf16 (bf16 | None) = total gradient w.r.t. h_t, summed inside the kernel."""
    require_cuda(gates, c_prev, c_next, dh, dh_bf16, dc_in, dgates_out)
    p = gates.numel() // (4 * ch)
    dgates = torch.empty(gates.shape, device=gates.device, dtype=torch.bfloat16) if dgates_out is None else dgates_out
    assert gates.is_contiguous() and dgates.is_contiguous()
    assert dh is None or (dh.is_contiguous() and dh.dtype == torch.float32)
    assert dh_bf16 is None or (dh_bf16.is_contiguous() and dh_bf16.dtype == torch.bfloat16)
    dc_prev = torch.empty(c_next.shape, device=gates.device, dtype=torch.float32)
    call("snn_lstm_gates_bwd", ptr(gates), ptr(c_prev), ptr(c_next), ptr(dh), ptr(dh_bf16), ptr(dc_in), ptr(dgates), ptr(dc_prev), p, ch,
         stream_ptr())
    return dgates, dc_prev


def nchw_to_nhwc(x, dtype=torch.bfloat16, out=None):
    """fp32 NCHW contiguous -> NHWC tensor (bf16 or fp32)."""
    require_cuda(x)
    nb, c, h, w = x.shape
    x = x.contiguous()
    if out is None:
        out = torch.empty((nb, h, w, c), device=x.device, dtype=dtype)
    call("snn_nchw_to_nhwc", ptr(x), ptr(out), int(out.dtype == torch.bfloat16), nb, c, h * w, _nhwc_ld(out), 0, stream_ptr())
    return out


def nhwc_to_nchw(x):
    """NHWC (bf16|fp32, may be a channel slice) -> fp32 NCHW contiguous."""
    require_cuda(x)
    nb, h, w, c = x.shape
    out = torch.empty((nb, c, h, w), device=x.device, dtype=torch.float32)
    call("snn_nhwc_to_nchw", ptr(x), int(x.dtype == torch.bfloat16), ptr(out), nb, c, h * w, _nhwc_ld(x), 0, stream_ptr())
    return out


def bilinear_resize(x, out_hw):
    """bf16 NHWC [NB,Hi,Wi,C] -> [NB,Ho,Wo,C] (F.interpolate bilinear, align_corners=False; reference model.py:43-44)."""
    require_cuda(x)
    nb, hi, wi, c = x.shape
    ho, wo = out_hw
    assert x.is_contiguous() and x.dtype == torch.bfloat16
    y = torch.empty((nb, ho, wo, c), device=x.device, dtype=torch.bfloat16)
    call("snn_bilinear_resize", 0, ptr(x), ptr(y), nb, hi, wi, ho, wo, c, stream_ptr(),
         work=("byte", 2.0 * (x.numel() + y.numel())))
    return y


def bilinear_resize_bwd(gy, in_hw):
    """Gradient of bilinear_resize w.r.t. its input: gy bf16 [NB,Ho,Wo,C] -> bf16 [NB,Hi,Wi,C]."""
    require_cuda(gy)
    nb, ho, wo, c = gy.shape
    hi, wi = in_hw
    assert gy.is_contiguous() and gy.dtype == torch.bfloat16
    gx = torch.empty((nb, hi, wi, c), device=gy.device, dtype=torch.bfloat16)
    call("snn_bilinear_resize", 1, ptr(gy), ptr(gx), nb, hi, wi, ho, wo, c, stream_ptr(),
         work=("byte", 2.0 * (gx.numel() + gy.numel())))
    return gx


def pad_crop(x, out_hw):
    """Bottom/right zero-pad or crop of a contiguous NHWC bf16 tensor to spatial size out_hw."""
    require_cuda(x)
    nb, hs, ws, c = x.shape
    hd, wd = out_hw
    assert x.is_contiguous() and x.dtype == torch.bfloat16
    y = torch.empty((nb, hd, wd, c), device=x.device, dtype=torch.bfloat16)
    call("snn_nhwc_pad_crop", ptr(x), ptr(y), nb, hs, ws, hd, wd, c, stream_ptr(), work=("byte", 2.0 * (x.numel() + y.numel())))
    return y


def colsum_accumulate(dy, acc):
    """acc[c] (fp32) += sum over all pixels of dy[..., c] (bf16)."""
    require_cuda(dy, acc)
    c = dy.shape[-1]
    assert dy.is_contiguous() and dy.dtype == torch.bfloat16 and acc.numel() == c and acc.is_contiguous()
    call("snn_colsum_bf16", ptr(dy), ptr(acc), dy.numel() // c, c, stream_ptr())


def grad_sumsq(g, acc, zero_first=True):
    require_cuda(g, acc)
    call("snn_grad_sumsq", ptr(g), g.numel(), ptr(acc), int(zero_first), stream_ptr(), work=("byte", 4.0 * g.numel()))


def adamw_step(p, g, m, v, shadow, hp, sumsq, gnorm_out=None, step=None, zero_grad=False):
    """hp: one row of 8 floats, or (with `step`, a device int32 scalar) the whole [rows, 8] schedule table.
    zero_grad: leave g zeroed (the next step's optimizer.zero_grad() folded into this pass)."""
    require_cuda(p, g, m, v, shadow, hp, sumsq, gnorm_out, step)
    n_rows = hp.shape[0] if (step is not None and hp.dim() == 2) else 1
    call("snn_adamw_step", ptr(p), ptr(g), ptr(m), ptr(v), ptr(shadow), p.numel(), ptr(hp), ptr(sumsq), ptr(gnorm_out),
         ptr(step), n_rows, int(bool(zero_grad)), stream_ptr(),
         work=("byte", (28.0 + (2.0 if shadow is not None else 0.0)) * p.numel()))


def ema_update(ema, src, decay, updates, segments=None, segment_elems=0):
    """ema = d * ema + (1 - d) * src (fp32, flat, length a multiple of 4), and the same over every (src, dst, n) row of
    `segments` (device int64 [n_seg, 3] of addresses and lengths; `segment_elems` = the sum of the lengths, for the byte
    count).  decay: device fp32 [rows, 2] = {d, 1 - d} per update; updates: device int32 counter picking the row (clamped
    to the last), incremented by the call."""
    require_cuda(ema, src, decay, updates, segments)
    for name, t in (("ema", ema), ("src", src)):
        if t.dtype != torch.float32 or not t.is_contiguous():
            raise ValueError(f"ema_update: {name} must be a contiguous fp32 tensor")
    if ema.numel() != src.numel():
        raise ValueError(f"ema_update: {ema.numel()} averaged elements, {src.numel()} source elements")
    if decay.dtype != torch.float32 or decay.dim() != 2 or decay.shape[1] != 2 or not decay.is_contiguous():
        raise ValueError("ema_update: decay must be a contiguous fp32 [rows, 2] table")
    if updates.dtype != torch.int32 or updates.numel() != 1:
        raise ValueError("ema_update: updates must be a one-element int32 device counter")
    n_seg = 0
    if segments is not None:
        if segments.dtype != torch.int64 or segments.dim() != 2 or segments.shape[1] != 3 or not segments.is_contiguous():
            raise ValueError("ema_update: segments must be a contiguous int64 [n, 3] table")
        n_seg = segments.shape[0]
    call("snn_ema_update", ptr(ema), ptr(src), ema.numel(), ptr(segments), n_seg, ptr(decay), ptr(updates), decay.shape[0],
         stream_ptr(), work=("byte", 12.0 * (ema.numel() + segment_elems)))


# ---------------------------------------------------------------------------------------------
# Detect-head depthwise conv, frame packer
# ---------------------------------------------------------------------------------------------
GEOM_DW3x3 = 4


def dw3x3_fprop(x, w9c, T=0):
    """x bf16 NHWC, w fp32 [9][C] -> y fp32 NHWC.  T > 0: also the per-timestep BatchNorm partial sums of y from the same
    pass -> (y, partials fp32 [T][blocks][2][C], blocks per timestep)."""
    require_cuda(x, w9c)
    nb, h, w, c = x.shape
    assert x.is_contiguous() and x.dtype == torch.bfloat16 and w9c.is_contiguous() and w9c.numel() == 9 * c
    y = torch.empty((nb, h, w, c), device=x.device, dtype=torch.float32)
    nbytes = 6.0 * y.numel()                # algorithmic: read x bf16, write y fp32
    if T and nb % T == 0:
        gpt = int(_lib.lib().snn_dw3x3_stats_blocks(nb // T, w, c))
        part = torch.empty((T, gpt, 2, c), device=x.device, dtype=torch.float32)
        call("snn_dw3x3_fprop_stats", ptr(x), ptr(w9c), ptr(y), nb, h, w, c, T, ptr(part), stream_ptr(),
             work=("byte", nbytes, f"dw fwd+stats nb{nb} {h}x{w} C{c}"))
        return y, part, gpt
    call("snn_dw3x3_fprop", ptr(x), ptr(w9c), ptr(y), nb, h, w, c, stream_ptr(), work=("byte", nbytes, f"dw fwd nb{nb} {h}x{w} C{c}"))
    return (y, None, 0) if T else y


def dw3x3_dgrad(dy, w9c, out=None):
    require_cuda(dy, w9c, out)
    nb, h, w, c = dy.shape
    assert dy.is_contiguous() and dy.dtype == torch.bfloat16
    dx = torch.empty((nb, h, w, c), device=dy.device, dtype=torch.bfloat16) if out is None else out
    assert dx.is_contiguous() and tuple(dx.shape) == (nb, h, w, c) and dx.dtype == torch.bfloat16
    call("snn_dw3x3_dgrad", ptr(dy), ptr(w9c), ptr(dx), nb, h, w, c, stream_ptr(), work=("byte", 4.0 * dy.numel(), f"dw dgrad nb{nb} {h}x{w} C{c}"))
    return dx


def dw3x3_wgrad(x, dy, dw9c):
    require_cuda(x, dy, dw9c)
    nb, h, w, c = x.shape
    assert x.is_contiguous() and dy.is_contiguous() and dw9c.is_contiguous() and dw9c.dtype == torch.float32
    call("snn_dw3x3_wgrad", ptr(x), ptr(dy), ptr(dw9c), nb, h, w, c, stream_ptr(), work=("byte", 4.0 * x.numel(), f"dw wgrad nb{nb} {h}x{w} C{c}"))


def space_to_depth8(frames, B, T):
    """fp32 frames in [0,1] or uint8 frames (divided by 255 on the device) [B,T,3,H,W] (contiguous) -> bf16 NHWC
    [T*B, H/8, W/8, 192] (timestep-major folded batch)."""
    require_cuda(frames)
    assert frames.is_contiguous() and frames.dtype in (torch.float32, torch.uint8)
    h, w = frames.shape[-2:]
    out = torch.empty((T * B, h // 8, w // 8, 192), device=frames.device, dtype=torch.bfloat16)
    name = "snn_space_to_depth8" if frames.dtype == torch.float32 else "snn_space_to_depth8_u8"
    call(name, ptr(frames), ptr(out), B, T, h, w, stream_ptr())
    return out


# ---------------------------------------------------------------------------------------------
# Detect decode + detection-loss tail
# ---------------------------------------------------------------------------------------------
def detect_decode(distri, scores, anchors, stride, xywh, want_probs=True):
    """distri fp32 [B,A,4*reg_max], scores fp32 [B,A,nc] -> boxes [B,A,4] (pixels), probs [B,A,nc] | None."""
    require_cuda(distri, scores, anchors, stride)
    b, a, r4 = distri.shape
    nc = scores.shape[2]
    assert distri.is_contiguous() and scores.is_contiguous() and distri.dtype == torch.float32 and scores.dtype == torch.float32
    boxes = torch.empty((b, a, 4), device=distri.device, dtype=torch.float32)
    probs = torch.empty((b, a, nc), device=distri.device, dtype=torch.float32) if want_probs else None
    call("snn_detect_decode", ptr(distri), ptr(scores), ptr(anchors), ptr(stride), b, a, nc, r4 // 4, int(xywh), ptr(boxes),
         ptr(probs), stream_ptr())
    return boxes, probs


def _a_off_arg(a_off):
    """Row map of scale-major prediction buffers -> (nl, ctypes int array | None); None / () = natural [B][A] rows."""
    if not a_off:
        return 0, None
    arr = (_lib.ctypes.c_int * len(a_off))(*[int(v) for v in a_off])
    return len(a_off) - 1, arr


def detect_assign_loss_fwd(distri, scores, a_off, anchors, stride, gt_cls, gt_box, gt_valid, img_wh, B, A, nc, reg_max, topk,
                           gains, counter):
    """decode -> task-aligned assignment -> fused loss sums -> finalisation, 5 launches (include/snn_b200.h).
    distri [B*A, 4*reg_max] / scores [B*A, nc] fp32 in the row order `a_off` describes.  Returns
    (out6 = loss*B [3] ++ loss [3], coef3, (tbox_px, tscores, fg))."""
    require_cuda(distri, scores, anchors, stride, gt_cls, gt_box, gt_valid, gains, counter)
    dev = distri.device
    M = gt_cls.shape[1]
    assert gt_cls.dtype == torch.int64 and gt_box.dtype == torch.float32 and gt_valid.dtype in (torch.bool, torch.uint8)
    assert gt_cls.is_contiguous() and gt_box.is_contiguous() and gt_valid.is_contiguous() and distri.is_contiguous() and scores.is_contiguous()
    assert tuple(gt_cls.shape) == (B, M) and tuple(gt_box.shape) == (B, M, 4) and distri.numel() == B * A * 4 * reg_max
    assert counter.dtype == torch.int32 and gains.dtype == torch.float32 and gains.numel() == 3
    ws = torch.empty((int(_lib.lib().snn_tal_workspace_bytes(B, A, M)) + 15) // 16 * 4, device=dev, dtype=torch.float32)
    pboxes = torch.empty((B, A, 4), device=dev, dtype=torch.float32)
    probs = torch.empty((B, A, nc), device=dev, dtype=torch.float32)
    tbox = torch.empty((B, A, 4), device=dev, dtype=torch.float32)
    tscores = torch.empty((B, A, nc), device=dev, dtype=torch.float32)
    fg = torch.empty((B, A), device=dev, dtype=torch.uint8)
    sums = torch.empty(3, device=dev, dtype=torch.float64)
    out6 = torch.empty(6, device=dev, dtype=torch.float32)
    coef3 = torch.empty(3, device=dev, dtype=torch.float32)
    nl, arr = _a_off_arg(a_off)
    call("snn_detect_assign_loss_fwd", ptr(distri), ptr(scores), nl, arr, ptr(anchors), ptr(stride), ptr(gt_cls), ptr(gt_box),
         ptr(gt_valid), float(img_wh[0]), float(img_wh[1]), B, A, M, nc, reg_max, int(topk), ptr(gains), ptr(ws), ptr(pboxes),
         ptr(probs), ptr(tbox), ptr(tscores), ptr(fg), ptr(sums), ptr(counter), ptr(out6), ptr(coef3), stream_ptr())
    return out6, coef3, (tbox, tscores, fg)


def tal_assign(probs, pboxes, anchors, stride, gt_cls, gt_box, gt_valid, img_wh, nc, topk=10):
    """The assigner kernels alone: probs [B,A,nc] (sigmoid), pboxes [B,A,4] xyxy px -> (tbox_px, tscores, fg)."""
    require_cuda(probs, pboxes, anchors, stride, gt_cls, gt_box, gt_valid)
    B, A = probs.shape[0], probs.shape[1]
    M = gt_cls.shape[1]
    dev = probs.device
    ws = torch.empty((int(_lib.lib().snn_tal_workspace_bytes(B, A, M)) + 15) // 16 * 4, device=dev, dtype=torch.float32)
    tbox = torch.empty((B, A, 4), device=dev, dtype=torch.float32)
    tscores = torch.empty((B, A, nc), device=dev, dtype=torch.float32)
    fg = torch.empty((B, A), device=dev, dtype=torch.uint8)
    assert probs.is_contiguous() and pboxes.is_contiguous() and gt_cls.dtype == torch.int64
    call("snn_tal_assign", ptr(probs), ptr(pboxes), ptr(anchors), ptr(stride), ptr(gt_cls.contiguous()), ptr(gt_box.contiguous()),
         ptr(gt_valid.contiguous()), float(img_wh[0]), float(img_wh[1]), B, A, M, nc, int(topk), ptr(ws), ptr(tbox), ptr(tscores), ptr(fg),
         stream_ptr())
    return tbox, tscores, fg


def detect_loss_bwd_rows(distri, scores, a_off, anchors, stride, targets, B, A, nc, reg_max, coef3, gout3, bf16):
    """Gradients of sum(gout3 * loss*B) w.r.t. the prediction rows; bf16 (fused head path) or fp32."""
    tbox, tscores, fg = targets
    require_cuda(distri, scores, anchors, stride, tbox, tscores, fg, coef3, gout3)
    dt = torch.bfloat16 if bf16 else torch.float32
    g_distri = torch.empty(distri.shape, device=distri.device, dtype=dt)
    g_scores = torch.empty(scores.shape, device=distri.device, dtype=dt)
    nl, arr = _a_off_arg(a_off)
    assert gout3 is None or (gout3.dtype == torch.float32 and gout3.is_contiguous() and gout3.numel() == 3)
    call("snn_detect_loss_bwd_rows", ptr(distri), ptr(scores), nl, arr, ptr(anchors), ptr(stride), ptr(tbox), ptr(tscores), ptr(fg),
         B, A, nc, reg_max, ptr(coef3), ptr(gout3), ptr(g_distri), ptr(g_scores), int(bf16), stream_ptr())
    return g_distri, g_scores


def detect_loss_fwd(distri, scores, anchors, stride, tbox_px, tscores, fg):
    require_cuda(distri, scores, anchors, stride, tbox_px, tscores, fg)
    b, a, r4 = distri.shape
    sums = torch.empty(3, device=distri.device, dtype=torch.float64)
    for t in (distri, scores, anchors, stride, tbox_px, tscores, fg):
        assert t.is_contiguous()
    assert fg.dtype == torch.uint8 and tscores.dtype == torch.float32 and tbox_px.dtype == torch.float32
    call("snn_detect_loss_fwd", ptr(distri), ptr(scores), ptr(anchors), ptr(stride), ptr(tbox_px), ptr(tscores), ptr(fg), b, a,
         scores.shape[2], r4 // 4, ptr(sums), stream_ptr())
    return sums


def detect_loss_bwd(distri, scores, anchors, stride, tbox_px, tscores, fg, coef):
    require_cuda(distri, scores, anchors, stride, tbox_px, tscores, fg, coef)
    b, a, r4 = distri.shape
    g_distri, g_scores = torch.empty_like(distri), torch.empty_like(scores)
    assert coef.dtype == torch.float32 and coef.is_contiguous() and coef.numel() == 3
    call("snn_detect_loss_bwd", ptr(distri), ptr(scores), ptr(anchors), ptr(stride), ptr(tbox_px), ptr(tscores), ptr(fg), b, a,
         scores.shape[2], r4 // 4, ptr(coef), ptr(g_distri), ptr(g_scores), stream_ptr())
    return g_distri, g_scores
