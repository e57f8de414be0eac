"""-m gpu: the fused train-mode BatchNorm finalize (snn_bn_finalize_partials) against float64 references.

Every ConvBlock of a training step reduces its BatchNorm statistics with this kernel: the conv epilogue (32-pixel
groups) or the depthwise head kernel (one group per thread block) writes fp32 partial rows [T][groups_per_t][2][C];
one launch turns them into the per-timestep scale / shift / mean / invstd, applies the T running-statistics updates in
order and adds T to num_batches_tracked.  It splits the rows of each timestep over S = clamp(groups_per_t / 16, 1, 64)
blocks per 32-channel group; the last block to arrive (atomic ticket on a caller-owned counter, which it resets)
combines the S fp64 partials and walks the timesteps four at a time.

A. Synthetic partials: fp32 y[T][P][C], zero-padded to groups_per_t * 32 rows, summed per 32-row group in fp32 (a
   pairwise tree: error <= 6 * 2^-24 of sum |y|, inside the producers' 1e-6 contract).  Outputs, workspace and the
   sums are pre-filled with NaN, so every (t, c) must be written by the launch; the counter array is longer than
   ceil(C/32) and its tail holds sentinels.
   - sums == the float64 sum of the partials the kernel read, within 1e-13 of sum |partial| (only the fp64 order may
     differ);
   - mean / invstd / scale / shift == the kernel's fp32 formula restated in torch from the kernel's own sums, within
     2 ulp (shift: 2 ulp of |beta| + |mean * scale|; nvcc may contract to FMA, so bit equality is not required);
   - mean / invstd == float64 BatchNorm of y within the bound of B; an all-zero channel gives mean 0 and invstd
     1/sqrt(eps) in float32, a constant channel a variance (implied by invstd) inside the same bound;
   - running statistics == T sequential BatchNorm2d updates restated in float64 with the unbiased variance
     P/(P-1), within (2T + 2) ulp of the largest magnitude in the update chain; num_batches_tracked == 7 + T.

B. The real producers (conv epilogue, depthwise head kernel) at production shapes, through kernels.bn_finalize_partials.
   Reference: float64 BatchNorm statistics of the kernel's own fp32 conv output y.  Derivation of the bound, from the
   partial-sum contract |sum_partials - sum_y| <= k * 1e-6 * sum |y| (and the same for y^2), with k = 1 for the conv
   epilogue (test_gpu_conv.py) and k = 2 for the depthwise kernel (test_gpu_head.py) and for snn_bn_stats
   (test_gpu_bench_shapes.py):
     mean = a / P                    -> |dmean| <= k * 1e-6 * mean|y|                       (+ the fp32 rounding of mean)
     var  = b / P - mean^2           -> |dvar|  <= k * 1e-6 * mean(y^2) + 2 |mean| |dmean|
                                                <= k * 3e-6 * mean(y^2)     (mean|y|^2 <= mean(y^2)) (+ fp32 rounding)
     invstd = 1 / sqrt(var + eps)    -> |invstd / invstd_ref - 1| <= k * 1.5e-6 * mean(y^2) / (var + eps) + 4 * 2^-24
                                                                    (first order; 4 * 2^-24 for the fp32 roundings)
   The variance is E[y^2] - E[y]^2 from fp32 partials, so its error grows with (mean/std)^2: mean(y^2) / var =
   1 + mean^2 / var.  The bound states that growth; the channel-offset case measures it at mean/std = 0, 8 and 32 and
   prints the worst mean^2 / var it saw.  The running statistics are convex combinations of the per-timestep values,
   so they inherit the same bound (times P/(P-1) for the variance) plus the (2T + 2) ulp of A.

C. The fallback (the conv planner declines, ConvBNActFn runs bn_stats + bn_finalize and adds T on the host side) at a
   shape the planner declines: module-level checks as in D, with the snn_bn_stats bound (k = 2).

D. model.ConvBlock in train mode through forward_seq, T = 4, S > 1: LIF 3x3 s1, SiLU 3x3 s2 and the Detect-head
   depthwise block (eps 1e-3, momentum 0.03).  Running statistics vs T float64 updates of the conv output; a second
   forward (reusing bn._snn_counters) == two direct launches bit for bit; one launch captured in a CUDA graph and
   replayed three times == three eager launches bit for bit, counters zero afterwards.
"""
import math

import pytest
import torch

from tests.gpu_util import setup_exact
from tests.test_gpu_conv import _mk, _mkw

pytestmark = pytest.mark.gpu
DEV = "cuda"
G31, G32, G11 = 0, 1, 2
U = 2.0 ** -24                                  # unit roundoff of fp32
SENTINELS = [0x13579BDF, -1, 7, 0x2468ACE]      # counter slots past ceil(C/32): the kernel must not touch them
BN_CFGS = [(1e-5, 0.1), (1e-3, 0.03)]           # U-Net blocks, Detect head


def _pkg():
    from snn_object_detectionddp_b200 import _lib, kernels
    return _lib, kernels


def _splits(gpt):
    return max(1, min(64, gpt // 16))


def _f32(x):
    return float(torch.tensor(x, dtype=torch.float32))


def _ulp(x):
    """ulp of the float32 value(s) x, as float64."""
    x = x.float().abs()
    return (torch.nextafter(x, torch.full_like(x, math.inf)) - x).double()


# ------------------------------------------------------------------------------------------------
# direct launch with buffers the test owns
# ------------------------------------------------------------------------------------------------
def _counters(C):
    ncg = (C + 31) // 32
    return torch.tensor([0] * ncg + SENTINELS, dtype=torch.int32, device=DEV)


def _outputs(T, C, gpt):
    """NaN-filled outputs, sums and workspace: whatever the launch does not write stays NaN."""
    _lib, _ = _pkg()
    nan = lambda *s, dt=torch.float32: torch.full(s, math.nan, device=DEV, dtype=dt)  # noqa: E731
    nws = int(_lib.lib().snn_bn_finalize_workspace_doubles(T, C, gpt))
    return dict(scale=nan(T, C), shift=nan(T, C), mean=nan(T, C), invstd=nan(T, C), sums=nan(T, 2, C, dt=torch.float64),
                ws=nan(nws, dt=torch.float64))


def _launch(part, gpt, T, C, P, eps, momentum, gamma, beta, rm, rv, nbt, counters, out):
    _lib, _ = _pkg()
    p = _lib.ptr
    _lib.require_cuda(part, gamma, beta, rm, rv, nbt, counters, *out.values())
    _lib.call("snn_bn_finalize_partials", p(part), p(out["sums"]), p(out["ws"]), p(gamma), p(beta), p(rm), p(rv), p(nbt),
              p(out["scale"]), p(out["shift"]), p(out["mean"]), p(out["invstd"]), p(counters), T, C, P, gpt, float(eps),
              float(momentum), _lib.stream_ptr())


def _check_counters_and_nan(counters, C, out):
    ncg = (C + 31) // 32
    c = counters.cpu().tolist()
    assert c[:ncg] == [0] * ncg, f"counters not reset: {c[:ncg]}"
    assert c[ncg:] == SENTINELS, f"sentinels past ceil(C/32) changed: {c[ncg:]}"
    for k in ("scale", "shift", "mean", "invstd", "sums"):
        bad = torch.isnan(out[k])
        assert not bool(bad.any()), f"{k}: {int(bad.sum())} entries not written, first at {bad.nonzero()[0].tolist()}"


# ------------------------------------------------------------------------------------------------
# references
# ------------------------------------------------------------------------------------------------
def _f64_stats(y, T, C):
    """float64 BatchNorm statistics of y [T*..., C] per timestep: mean, biased var, mean|y|, mean(y^2) [T][C]."""
    yt = y.reshape(T, -1, C)
    m, v, a, q = [], [], [], []
    for t in range(T):
        d = yt[t].double()
        mt = d.mean(0)
        m.append(mt)
        v.append(((d - mt) ** 2).mean(0))
        a.append(d.abs().mean(0))
        q.append((d * d).mean(0))
    return tuple(torch.stack(s) for s in (m, v, a, q))


def _check_vs_float64(mean, invstd, ref, eps, k, what=""):
    """The bound of B: |dmean| <= k 1e-6 mean|y| (+ fp32 rounding), |invstd/ref - 1| <= k 1.5e-6 mean(y^2)/(var+eps)
    + 4 2^-24."""
    m_ref, v_ref, abs_mean, sq_mean = ref
    dm = (mean.double() - m_ref).abs()
    tol_m = k * 1e-6 * abs_mean + U * m_ref.abs()
    assert bool((dm <= tol_m).all()), f"{what} mean: worst {float((dm / tol_m).max()):.3g} x the bound"
    r = (invstd.double() * torch.sqrt(v_ref + eps) - 1).abs()
    tol_r = k * 1.5e-6 * sq_mean / (v_ref + eps) + 4 * U
    assert bool((r <= tol_r).all()), f"{what} invstd: worst {float((r / tol_r).max()):.3g} x the bound"
    return float((r / tol_r).max())


def _running_ref(rm0, rv0, means, vars_, P, momentum):
    """T sequential BatchNorm2d updates (momentum as the fp32 value the kernel receives) in float64, unbiased variance.
    Also the largest magnitude in each chain (per channel): the scale of the (2T + 2) ulp tolerance."""
    mom = _f32(momentum)
    rm, rv = rm0.double().clone(), rv0.double().clone()
    sm, sv = rm.abs(), rv.abs()
    for t in range(means.shape[0]):
        unb = vars_[t] * (P / (P - 1)) if P > 1 else vars_[t]
        rm = (1 - mom) * rm + mom * means[t]
        rv = (1 - mom) * rv + mom * unb
        sm, sv = torch.maximum(sm, means[t].abs()), torch.maximum(sv, unb.abs())
    return rm, rv, sm, sv


def _check_running_vs_float64(rm, rv, rm0, rv0, ref, P, T, momentum, k, what=""):
    """Running statistics from the kernel vs float64 updates with the true statistics of y: the bound of B (a convex
    combination of per-timestep errors) plus (2T + 2) ulp of arithmetic."""
    m_ref, v_ref, abs_mean, sq_mean = ref
    want_m, want_v, sm, sv = _running_ref(rm0, rv0, m_ref, v_ref, P, momentum)
    tol_m = (k * 1e-6 * abs_mean + U * m_ref.abs()).max(0).values + (2 * T + 2) * _ulp(sm)
    tol_v = (P / max(P - 1, 1)) * (k * 3e-6 * sq_mean + U * v_ref).max(0).values + (2 * T + 2) * _ulp(sv)
    dm, dv = (rm.double() - want_m).abs(), (rv.double() - want_v).abs()
    assert bool((dm <= tol_m).all()), f"{what} running_mean: worst {float((dm / tol_m).max()):.3g} x the bound"
    assert bool((dv <= tol_v).all()), f"{what} running_var: worst {float((dv / tol_v).max()):.3g} x the bound"


# ------------------------------------------------------------------------------------------------
# A. synthetic partials
# ------------------------------------------------------------------------------------------------
# groups_per_t, T, C, P: what the case reaches
SYNTH = [
    (1, 1, 8, 2),             # S = 1; unbiased factor P/(P-1) = 2
    (15, 5, 72, 473),         # second timestep round holds one timestep; C tail of 8 lanes; P not a multiple of 32
    (16, 4, 144, 512),        # last S = 1 case
    (32, 8, 128, 1024),       # S = 2, even chunks
    (33, 3, 1024, 1056),      # S = 2, chunks of 17 and 16
    (1025, 2, 72, 32800),     # S = 64, three empty trailing splits
    (2048, 4, 144, 65536),    # configs[1] enc1 level
    (1100, 16, 40, 35000),    # four timestep rounds at S = 64, two empty trailing splits
]
SYNTH_IDS = [f"g{g}-T{T}-C{C}-P{P}" for g, T, C, P in SYNTH]
ZERO_CH = -1      # all-zero channel (a silent spiking layer)
CONST_CH = 1      # constant, non-zero channel: b/P - md^2 may round below zero and is clamped


def _tree_sum32(v):
    """[T][groups*32][C] -> [T][groups][C]: fp32 pairwise sum of each 32-row group (error <= 5 * 2^-24 of sum |v|)."""
    T, n, C = v.shape
    v = v.view(T, n // 32, 32, C)
    while v.shape[2] > 1:
        h = v.shape[2] // 2
        v = v[:, :, :h] + v[:, :, h:]
    return v[:, :, 0]


def _synthetic(gpt, T, C, P, seed):
    """y [T][P][C] with per-(t, c) means and spreads, one zero and one constant channel; partials [T][gpt][2][C]."""
    assert gpt * 32 >= P       # groups past the map are all zero, as the epilogue writes them for a padded pixel box
    g = torch.Generator(device=DEV).manual_seed(seed)
    mu = torch.randn(T, 1, C, device=DEV, generator=g) * 1.5
    sigma = torch.rand(T, 1, C, device=DEV, generator=g) * 1.5 + 0.25
    y = mu + sigma * torch.randn(T, P, C, device=DEV, generator=g)
    y[:, :, ZERO_CH] = 0.0
    y[:, :, CONST_CH] = (0.7 + 0.45 * torch.arange(T, device=DEV, dtype=torch.float32))[:, None]
    yp = torch.zeros(T, gpt * 32, C, device=DEV)
    yp[:, :P] = y                                   # zero rows past the map, as the epilogue writes them
    part = torch.stack([_tree_sum32(yp), _tree_sum32(yp * yp)], 2).contiguous()
    gamma = torch.rand(C, device=DEV, generator=g) + 0.5
    beta = torch.randn(C, device=DEV, generator=g) * 0.5
    rm0 = torch.randn(C, device=DEV, generator=g) * 0.5
    rv0 = torch.rand(C, device=DEV, generator=g) * 2 + 0.2
    return y, part, gamma, beta, rm0, rv0


def _restate(sums, P, gamma, beta, eps):
    """The kernel's fp32 formula, from its own fp64 sums."""
    a, b = sums[:, 0].double().cpu(), sums[:, 1].double().cpu()
    md = a / P
    vd = (b / P - md * md).clamp_min(0.0)
    m, var = md.float(), vd.float()
    inv = 1.0 / torch.sqrt(var + torch.tensor(eps, dtype=torch.float32))
    sc = gamma.cpu() * inv
    return m, inv, sc, beta.cpu() - m * sc, md, vd


def _run_synthetic(case, eps, momentum, seed=0):
    gpt, T, C, P = case
    y, part, gamma, beta, rm0, rv0 = _synthetic(gpt, T, C, P, seed)
    rm, rv = rm0.clone(), rv0.clone()
    nbt = torch.tensor(7, dtype=torch.int64, device=DEV)
    ctr, out = _counters(C), _outputs(T, C, gpt)
    _launch(part, gpt, T, C, P, eps, momentum, gamma, beta, rm, rv, nbt, ctr, out)
    torch.cuda.synchronize()
    return dict(y=y, part=part, gamma=gamma, beta=beta, rm0=rm0, rv0=rv0, rm=rm, rv=rv, nbt=nbt, ctr=ctr, out=out)


@pytest.mark.parametrize("eps,momentum", BN_CFGS)
@pytest.mark.parametrize("case", SYNTH, ids=SYNTH_IDS)
def test_synthetic_statistics(case, eps, momentum):
    """sums, the restated fp32 formula, float64 BatchNorm of y, the zero / constant channels, counters, no NaN."""
    setup_exact()
    gpt, T, C, P = case
    r = _run_synthetic(case, eps, momentum)
    out = r["out"]
    _check_counters_and_nan(r["ctr"], C, out)
    # sums: the float64 sum of the partials, up to fp64 summation order
    pd = r["part"].double()
    want = pd.sum(1)
    tol = 1e-13 * pd.abs().sum(1)
    d = (out["sums"] - want).abs()
    assert bool((d <= tol).all()), f"sums: worst {float((d / tol.clamp_min(1e-300)).max()):.3g} x 1e-13 sum|partial|"
    # the fp32 formula restated from the kernel's own sums
    m, inv, sc, sh, _, _ = _restate(out["sums"], P, r["gamma"], r["beta"], eps)
    got = {k: out[k].cpu() for k in ("mean", "invstd", "scale", "shift")}
    for name, want_k in (("mean", m), ("invstd", inv), ("scale", sc)):
        dk = (got[name].double() - want_k.double()).abs()
        assert bool((dk <= 2 * _ulp(want_k)).all()), f"{name}: {float((dk / _ulp(want_k)).max()):.3g} ulp from the restated formula"
    tol_sh = 2 * _ulp(r["beta"].cpu().abs() + (m * sc).abs())
    dsh = (got["shift"].double() - sh.double()).abs()
    assert bool((dsh <= tol_sh).all()), f"shift: {float((dsh / tol_sh).max()):.3g} x 2 ulp from the restated formula"
    # independently: float64 BatchNorm of y
    ref = _f64_stats(r["y"], T, C)
    _check_vs_float64(out["mean"], out["invstd"], ref, eps, 1, "synthetic")
    # edge channels
    assert bool((got["mean"][:, ZERO_CH] == 0).all())
    inv_eps = 1.0 / torch.sqrt(torch.tensor(eps, dtype=torch.float32))
    assert bool((got["invstd"][:, ZERO_CH] == inv_eps).all()), (got["invstd"][:, ZERO_CH], inv_eps)
    for k in ("mean", "invstd", "scale", "shift"):
        assert bool(torch.isfinite(got[k][:, [ZERO_CH, CONST_CH]]).all()), k
    var_impl = 1.0 / got["invstd"][:, CONST_CH].double() ** 2 - _f32(eps)
    tol_c = 3e-6 * ref[3][:, CONST_CH].cpu() + 8 * U * _f32(eps)
    assert bool((var_impl.abs() <= tol_c).all()), (var_impl, tol_c)


@pytest.mark.parametrize("eps,momentum", BN_CFGS)
@pytest.mark.parametrize("case", SYNTH, ids=SYNTH_IDS)
def test_synthetic_running_statistics(case, eps, momentum):
    """T sequential updates with the unbiased variance, num_batches_tracked += T; with the running buffers absent
    (NULL) every other output is bit-identical."""
    setup_exact()
    gpt, T, C, P = case
    r = _run_synthetic(case, eps, momentum, seed=1)
    out = r["out"]
    _check_counters_and_nan(r["ctr"], C, out)
    assert int(r["nbt"]) == 7 + T, f"num_batches_tracked {int(r['nbt'])}, want {7 + T}"
    s = out["sums"].double()
    md = s[:, 0] / P
    vd = (s[:, 1] / P - md * md).clamp_min(0.0)
    want_m, want_v, sm, sv = _running_ref(r["rm0"], r["rv0"], md, vd, P, momentum)
    dm, dv = (r["rm"].double() - want_m).abs(), (r["rv"].double() - want_v).abs()
    tol_m, tol_v = (2 * T + 2) * _ulp(sm), (2 * T + 2) * _ulp(sv)
    assert bool((dm <= tol_m).all()), f"running_mean: worst {float((dm / _ulp(sm)).max()):.3g} ulp (tolerance {2 * T + 2})"
    assert bool((dv <= tol_v).all()), f"running_var: worst {float((dv / _ulp(sv)).max()):.3g} ulp (tolerance {2 * T + 2})"
    # no running buffers: same statistics, bit for bit
    ctr2, out2 = _counters(C), _outputs(T, C, gpt)
    _launch(r["part"], gpt, T, C, P, eps, momentum, r["gamma"], r["beta"], None, None, None, ctr2, out2)
    torch.cuda.synchronize()
    _check_counters_and_nan(ctr2, C, out2)
    for k in ("sums", "scale", "shift", "mean", "invstd"):
        assert torch.equal(out[k], out2[k]), k


# ------------------------------------------------------------------------------------------------
# B. the real producers at production shapes
# ------------------------------------------------------------------------------------------------
# geom, T, B, h, w (conv input), C0, C1 (concat source), Cout, expected S, note
CONV_CASES = [
    (G31, 4, 64, 32, 32, 144, 0, 128, 64, "configs[1] enc1"),
    (G31, 4, 64, 32, 32, 128, 128, 128, 64, "configs[1] up3.conv1, two sources"),
    (G32, 4, 64, 32, 32, 128, 0, 256, 32, "configs[1] down1.conv1, 3x3 s2"),
    (G11, 4, 64, 32, 32, 144, 0, 144, 64, "configs[1] head cv3 pointwise, C tail of 16"),
    (G31, 4, 64, 4, 4, 1024, 0, 1024, 2, "configs[1] bottleneck"),
    (G31, 4, 8, 4, 4, 1024, 0, 1024, 1, "bottleneck at B = 8"),
    (G31, 4, 8, 15, 20, 512, 144, 512, 5, "enc3 at the 15x20 P5 level of a 480x640 frame, padded groups"),
]
# T, B, h, w, C, expected S
DW_CASES = [(4, 64, 8, 8, 144, 4), (3, 2, 15, 7, 1024, 1), (4, 64, 32, 32, 144, 18)]


def _producer_check(y, part, gpt, T, C, k, eps=1e-5, momentum=0.1, seed=0, what=""):
    """kernels.bn_finalize_partials on producer partials vs float64 BatchNorm of y; returns the worst mean^2 / var."""
    _, K = _pkg()
    g = torch.Generator(device=DEV).manual_seed(seed)
    gamma = torch.rand(C, device=DEV, generator=g) + 0.5
    beta = torch.randn(C, device=DEV, generator=g) * 0.5
    rm0 = torch.randn(C, device=DEV, generator=g) * 0.5
    rv0 = torch.rand(C, device=DEV, generator=g) * 2 + 0.2
    rm, rv = rm0.clone(), rv0.clone()
    nbt = torch.tensor(7, dtype=torch.int64, device=DEV)
    ctr = torch.zeros((C + 31) // 32, dtype=torch.int32, device=DEV)
    P = y.numel() // (T * C)
    scale, shift, mean, invstd = K.bn_finalize_partials(part, gpt, gamma, beta, rm, rv, nbt, ctr, T, C, P, eps, momentum)
    torch.cuda.synchronize()
    assert bool((ctr == 0).all()) and int(nbt) == 7 + T
    for name, v in (("scale", scale), ("shift", shift), ("mean", mean), ("invstd", invstd)):
        assert bool(torch.isfinite(v).all()), name
    ref = _f64_stats(y, T, C)
    worst = _check_vs_float64(mean, invstd, ref, eps, k, what)
    _check_running_vs_float64(rm, rv, rm0, rv0, ref, P, T, momentum, k, what)
    r2 = ref[0] ** 2 / ref[1].clamp_min(1e-300)
    return float(r2.max()), worst


@pytest.mark.parametrize("geom,T,B,h,w,c0,c1,cout,S,note", CONV_CASES,
                         ids=["enc1", "up3_conv1_concat", "down1_conv1_s2", "cv3_1x1", "bottleneck_b64", "bottleneck_b8",
                              "enc3_15x20"])
def test_conv_epilogue_partials(geom, T, B, h, w, c0, c1, cout, S, note):
    setup_exact()
    _, K = _pkg()
    x0 = _mk(T * B, h, w, c0, 31, spikes=True)
    x1 = _mk(T * B, h, w, c1, 32) if c1 else None
    wgt = _mkw(cout, 1 if geom == G11 else 9, c0 + c1, 33)
    y, part, gpt = K.conv_fprop_partials(geom, x0, wgt, cout, T, x1=x1)
    assert part is not None and _splits(gpt) == S, (gpt, S)
    r2, worst = _producer_check(y, part, gpt, T, cout, 1, what=note)
    print(f"\n[bn finalize] {note}: groups/t {gpt}, S {S}, max mean^2/var {r2:.3g}, worst invstd error {worst:.3g} x bound")


@pytest.mark.parametrize("T,B,h,w,C,S", DW_CASES)
def test_depthwise_partials(T, B, h, w, C, S):
    setup_exact()
    _, K = _pkg()
    x = torch.randn(T * B, h, w, C, device=DEV).to(torch.bfloat16)
    w9 = torch.randn(9, C, device=DEV) * 0.3
    y, part, gpt = K.dw3x3_fprop(x, w9, T=T)
    assert _splits(gpt) == S, (gpt, S)
    _producer_check(y, part, gpt, T, C, 2, eps=1e-3, momentum=0.03, what=f"dw {T}x{B}x{h}x{w}x{C}")


@pytest.mark.parametrize("ratio", [0, 8, 32])
def test_channel_offset_grows_the_variance_error_as_stated(ratio):
    """y = mu + sigma z with mu/sigma = ratio (a 1x1 conv at configs[1] shape whose constant input channel carries the
    offset): the error of E[y^2] - E[y]^2 grows with (mu/sigma)^2, and the bound of B, which scales with
    mean(y^2) / (var + eps), still holds."""
    setup_exact()
    _, K = _pkg()
    T, B, h, w, cin, cout = 4, 64, 32, 32, 144, 144
    x = _mk(T * B, h, w, cin, 41)
    x[..., -1] = 1.0
    wgt = _mkw(cout, 1, cin, 42)
    wgt[:, 0, -1] = float(ratio)                 # every output channel: ratio + (sum over 143 inputs, std ~ 1)
    y, part, gpt = K.conv_fprop_partials(G11, x, wgt, cout, T)
    assert part is not None and _splits(gpt) == 64
    r2, worst = _producer_check(y, part, gpt, T, cout, 1, what=f"mu/sigma {ratio}")
    q = 1 + r2
    print(f"\n[bn finalize] mu/sigma {ratio}: max mean^2/var {r2:.4g} -> invstd bound {1.5e-6 * q + 4 * U:.3g} relative, "
          f"worst error {worst:.3g} x bound")
    if ratio:
        assert r2 > 0.5 * ratio ** 2


# ------------------------------------------------------------------------------------------------
# C + D. model.ConvBlock in train mode, as training runs it
# ------------------------------------------------------------------------------------------------
# name, ConvBlock kwargs, input (T, B, h, w, Cin), producer bound k, expected S (None: the planner declines)
BLOCKS = [
    ("lif_3x3_s1", dict(in_channels=128, out_channels=128, neuron="lif"), (4, 8, 32, 32, 128), 1, 16),
    ("silu_3x3_s2", dict(in_channels=128, out_channels=256, stride=2, neuron="silu"), (4, 8, 64, 64, 128), 1, 16),
    ("detect_dw", dict(in_channels=144, out_channels=144, kernel_size=3, groups=144, neuron="silu", bn_eps=1e-3,
                       bn_momentum=0.03), (4, 64, 8, 8, 144), 2, 4),
    ("fallback_bn_stats", dict(in_channels=128, out_channels=128, neuron="lif"), (4, 3, 8, 8, 128), 2, None),
]


def _block(kw, seed):
    import snn_object_detectionddp_b200.model as M
    from snn_object_detectionddp_b200.params import store_for
    torch.manual_seed(seed)
    blk = M.ConvBlock(**kw).to(DEV).train()
    with torch.no_grad():
        blk.bn.weight.uniform_(0.8, 1.6)
        blk.bn.bias.uniform_(-0.2, 0.5)
        blk.bn.running_mean.uniform_(-0.5, 0.5)
        blk.bn.running_var.uniform_(0.5, 2.0)
        blk.bn.num_batches_tracked.fill_(7)
    st = store_for(blk, DEV)
    st.refresh_operands()
    return M, blk, st


def _forward(M, blk, st, T, x):
    with torch.no_grad():
        blk.forward_seq(M.RunCtx(st, T), x)
    torch.cuda.synchronize()


def _bn_state(blk):
    return blk.bn.running_mean.clone(), blk.bn.running_var.clone(), blk.bn.num_batches_tracked.clone()


@pytest.mark.parametrize("name,kw,shape,k,S", BLOCKS, ids=[b[0] for b in BLOCKS])
def test_convblock_train_forward_running_statistics(name, kw, shape, k, S):
    setup_exact()
    _, K = _pkg()
    M, blk, st = _block(kw, 5)
    T, B, h, w, cin = shape
    x = _mk(T * B, h, w, cin, 51, spikes=True)
    geom, cout = blk.geom, blk.bn.num_features
    # y exactly as the block's producer computes it, from the store's operands
    if geom == K.GEOM_DW3x3:
        y = K.dw3x3_fprop(x, st.w_master3(blk.conv.weight).view(9, cout))
        gpt = int(_pkg()[0].lib().snn_dw3x3_stats_blocks(B, w, cout))
    else:
        y, part, gpt = K.conv_fprop_partials(geom, x, st.w_fprop(blk.conv.weight), cout, T)
        assert (part is None) == (S is None), (name, gpt)
        y_plain = K.conv_fprop(geom, x, st.w_fprop(blk.conv.weight), cout)
        assert torch.equal(y, y_plain)
    if S is not None:
        assert _splits(gpt) == S, (gpt, S)
    rm0, rv0, nbt0 = _bn_state(blk)
    _forward(M, blk, st, T, x)
    P = y.numel() // (T * cout)
    ref = _f64_stats(y, T, cout)
    _check_running_vs_float64(blk.bn.running_mean, blk.bn.running_var, rm0, rv0, ref, P, T, blk.bn.momentum, k, name)
    assert int(blk.bn.num_batches_tracked) == int(nbt0) + T
    # a second forward continues from the first: 2T updates in all
    rm1, rv1, _ = _bn_state(blk)
    _forward(M, blk, st, T, x)
    assert int(blk.bn.num_batches_tracked) == int(nbt0) + 2 * T
    if S is None:
        _check_running_vs_float64(blk.bn.running_mean, blk.bn.running_var, rm1, rv1, ref, P, T, blk.bn.momentum, k, name)
        return
    assert bool((blk.bn._snn_counters == 0).all())
    # the two forwards (reusing bn._snn_counters) == two direct launches on the producer's partials, bit for bit
    if geom == K.GEOM_DW3x3:
        _, part, gpt = K.dw3x3_fprop(x, st.w_master3(blk.conv.weight).view(9, cout), T=T)
    else:
        _, part, gpt = K.conv_fprop_partials(geom, x, st.w_fprop(blk.conv.weight), cout, T)
    rm, rv, nbt = rm0.clone(), rv0.clone(), nbt0.clone()
    ctr = torch.zeros((cout + 31) // 32, dtype=torch.int32, device=DEV)
    for _ in range(2):
        K.bn_finalize_partials(part, gpt, blk.bn.weight, blk.bn.bias, rm, rv, nbt, ctr, T, cout, P, blk.bn.eps, blk.bn.momentum)
    torch.cuda.synchronize()
    assert torch.equal(blk.bn.running_mean, rm) and torch.equal(blk.bn.running_var, rv)
    assert int(blk.bn.num_batches_tracked) == int(nbt)


def test_cuda_graph_replay_equals_eager_launches():
    """One launch captured with persistent buffers (as Trainer.train_step_graphed replays it every step), replayed three
    times == three eager launches, bit for bit; the counters are zero afterwards."""
    setup_exact()
    gpt, T, C, P = 1100, 16, 40, 35000
    eps, momentum = 1e-5, 0.1
    _, part, gamma, beta, rm0, rv0 = _synthetic(gpt, T, C, P, 7)
    runs = {}
    for mode in ("eager", "graph"):
        rm, rv = rm0.clone(), rv0.clone()
        nbt = torch.tensor(7, dtype=torch.int64, device=DEV)
        ctr, out = _counters(C), _outputs(T, C, gpt)
        args = (part, gpt, T, C, P, eps, momentum, gamma, beta, rm, rv, nbt, ctr, out)
        if mode == "eager":
            for _ in range(3):
                _launch(*args)
        else:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                _launch(*args)
            torch.cuda.synchronize()
            assert int(nbt) == 7, "capture must not run the launch"
            for _ in range(3):
                g.replay()
        torch.cuda.synchronize()
        _check_counters_and_nan(ctr, C, out)
        runs[mode] = (rm, rv, nbt, out)
    (rm_e, rv_e, nbt_e, out_e), (rm_g, rv_g, nbt_g, out_g) = runs["eager"], runs["graph"]
    assert int(nbt_e) == int(nbt_g) == 7 + 3 * T
    assert torch.equal(rm_e, rm_g) and torch.equal(rv_e, rv_g)
    for k in ("sums", "scale", "shift", "mean", "invstd"):
        assert torch.equal(out_e[k], out_g[k]), k
