"""-m gpu: the spike-rate regularizer -- snn_spike_reg_coef against the float64 specification, snn_bn_act_bwd2_ds against
snn_bn_act_bwd2 and torch autograd, and spikes.SpikeRateLoss through the training step (counts, gradients, graphs, the
launch sequence, and that the penalty lowers the SynOps fraction)."""
import contextlib

import numpy as np
import pytest
import torch

from oracle import snn_oracle as O
from tests.gpu_util import rel_err, setup_exact
from tests.test_spike_reg_host import FAN, reference, synthetic_counts

pytestmark = pytest.mark.gpu

DEV = "cuda"
HYP = {"box": 7.5, "cls": 1.0, "dfl": 2.5, "reg_max": 16}
LIF = 0


@contextlib.contextmanager
def _deterministic():
    from snn_object_detectionddp_b200 import _lib
    L = _lib.lib()
    before = L.snn_get_deterministic()
    L.snn_set_deterministic(1)
    try:
        yield
    finally:
        L.snn_set_deterministic(before)


def _ulps(got, ref64):
    """|got - fp32(ref)| in units of the fp32 spacing at fp32(ref)."""
    r32 = np.float32(ref64)
    return abs(float(np.float32(got)) - float(r32)) / float(np.spacing(np.abs(r32)) if r32 != 0 else np.float32(1e-45))


# ------------------------------------------------------------------------------------------------------------------
# 1. coefficient kernel
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("params", [(2.0, 0.01, 0.2, 3.0, 64), (0.5, 0.02, 0.0, 0.0, 8), (0.0, 0.0, 0.5, 7.0, 32),
                                    (3.0, 1.0, 0.0, 3.0, 16), (1e3, 0.05, 0.1, 1e2, 64)])
@pytest.mark.parametrize("seed", [0, 1])
def test_coef_kernel_matches_float64_reference(params, seed):
    from snn_object_detectionddp_b200 import kernels as K
    a, phi_max, r_min, b, B = params
    counts = synthetic_counts(seed, T=4, max_T=8, top=1 << 40)
    P, phi, R, c = reference(counts, FAN, a, phi_max, r_min, b, B)
    cd = torch.from_numpy(counts).to(DEV)
    fan = torch.tensor(FAN, dtype=torch.float64, device=DEV)
    coef, out = torch.full((16,), 7.0, device=DEV), torch.full((18,), 7.0, device=DEV)
    stats = torch.arange(16 * 2 * 6, device=DEV, dtype=torch.int64).view(16, 2, 6)
    before = stats.clone()
    K.spike_reg_coef(cd, fan, coef, out, a, phi_max, r_min, b, B, stats=stats, T=4)
    coef, out = coef.cpu().numpy(), out.cpu().numpy()
    for got, ref in [(out[0], P), (out[1], phi)] + list(zip(out[2:], R)) + list(zip(coef, c)):
        assert _ulps(got, ref) <= 1.0, (got, ref)
    assert torch.equal(stats[:, :, :4], before[:, :, :4] + cd[:, :, :4]) and torch.equal(stats[:, :, 4:], before[:, :, 4:])
    out2 = torch.empty(18, device=DEV)
    with pytest.raises(ValueError, match="fanout"):
        K.spike_reg_coef(cd, fan.float(), torch.empty(16, device=DEV), out2, a, phi_max, r_min, b, B)
    with pytest.raises(ValueError, match="counts"):
        K.spike_reg_coef(cd.int(), fan, torch.empty(16, device=DEV), out2, a, phi_max, r_min, b, B)


# ------------------------------------------------------------------------------------------------------------------
# 2./3. backward kernel
# ------------------------------------------------------------------------------------------------------------------
def _bn_inputs(T, B, H, W, C, seed):
    from snn_object_detectionddp_b200 import kernels as K
    g = torch.Generator(device=DEV).manual_seed(seed)
    y = torch.randn(T * B, H, W, C, device=DEV, generator=g) * 1.5 + 0.7
    gamma = torch.rand(C, device=DEV, generator=g) + 0.5
    beta = torch.randn(C, device=DEV, generator=g) * 0.3 + 0.3
    sums = K.bn_stats(y, T)
    scale, shift, mean, invstd = K.bn_finalize(sums, gamma, beta, None, None, T, C, B * H * W, 1e-5, 0.1, True)
    return y, gamma, beta, scale, shift, mean, invstd, g


def _bwd(K, y, scale, shift, mean, invstd, beta, gs, T, v0, gvf, ds_add):
    C = y.shape[-1]
    dg, db = torch.zeros(C, device=DEV), torch.zeros(C, device=DEV)
    dy, gv0, red = K.bn_act_bwd_train(LIF, y, scale, shift, mean, invstd, beta, gs, T, dg, db, v_init=v0, gv_final=gvf,
                                      want_gv_init=v0 is not None, ds_add=ds_add)
    return dy, gv0, red, dg, db


@pytest.mark.parametrize("T", [1, 2, 4, 5, 8, 16])
@pytest.mark.parametrize("C", [64, 144])
def test_zero_addend_is_bit_equal_to_plain_backward(T, C):
    from snn_object_detectionddp_b200 import _lib
    from snn_object_detectionddp_b200 import kernels as K
    B, H, W = 2, 9, 7
    y, gamma, beta, scale, shift, mean, invstd, g = _bn_inputs(T, B, H, W, C, seed=T * 10 + C)
    gs = torch.randn(T * B, H, W, C, device=DEV, generator=g).to(torch.bfloat16)
    zero = torch.zeros(1, device=DEV)
    one_chunk = [False, True] if T == 16 else [False]
    try:
        with _deterministic():
            for oc in one_chunk:
                _lib.lib().snn_debug_set(9, int(oc))
                for with_state in (False, True):
                    v0 = torch.rand(B * H * W * C, device=DEV, generator=g) * 0.5 if with_state else None
                    gvf = torch.randn(B * H * W * C, device=DEV, generator=g) if with_state else None
                    ref = _bwd(K, y, scale, shift, mean, invstd, beta, gs, T, v0, gvf, None)
                    got = _bwd(K, y, scale, shift, mean, invstd, beta, gs, T, v0, gvf, zero)
                    for name, a, b in zip(("dy", "gv_init", "red", "dgamma", "dbeta"), got, ref):
                        assert (a is None and b is None) or torch.equal(a, b), (name, oc, with_state)
    finally:
        _lib.lib().snn_debug_set(9, 0)
    with pytest.raises(_lib.SnnKernelError, match="LIF"):
        K.bn_act_bwd_train(1, y, scale, shift, mean, invstd, beta, gs, T, torch.zeros(C, device=DEV), torch.zeros(C, device=DEV),
                           ds_add=zero)


@pytest.mark.parametrize("case", ["moderate", "gs_dominant", "gs_zero"])
@pytest.mark.parametrize("T,B,H,W,C", [(4, 2, 8, 8, 128), (8, 2, 4, 4, 256), (5, 2, 4, 4, 1024), (16, 1, 4, 4, 64),
                                       (4, 1, 8, 8, 144), (16, 2, 2, 2, 1024), (1, 2, 8, 8, 128), (4, 3, 5, 7, 72)])
def test_addend_matches_autograd(case, T, B, H, W, C):
    """loss = sum gs*s + c*sum s through per-timestep batch-statistics BN + LIF (torch autograd, oracle LIF) vs the kernel.
    gs_dominant: |gs| ~ 2^13 c (a bf16 add of c onto gs would round it away); its contribution is checked on the fp32
    BatchNorm parameter gradients as the difference to the c = 0 run.  gs_zero: the gradient is c's alone."""
    setup_exact()
    from snn_object_detectionddp_b200 import kernels as K
    P = B * H * W
    y, gamma, beta, scale, shift, mean, invstd, g = _bn_inputs(T, B, H, W, C, seed=6)
    c = {"moderate": 0.3, "gs_dominant": 0.01, "gs_zero": 0.4}[case]
    gs = torch.randn(T * B, H, W, C, device=DEV, generator=g) * (80.0 if case == "gs_dominant" else 1.0)
    if case == "gs_zero":
        gs.zero_()
    gs = gs.to(torch.bfloat16)
    v0 = torch.rand(B, H, W, C, device=DEV, generator=g) * 0.5
    gvf = torch.randn(B, H, W, C, device=DEV, generator=g)
    out, _, _ = K.bn_act_fwd(LIF, y, scale, shift, T, v_init=v0)
    cdev = torch.tensor([c], device=DEV)
    dy, gv0, _, dgamma, dbeta = _bwd(K, y, scale, shift, mean, invstd, beta, gs, T, v0, gvf.reshape(-1), cdev)

    def ref(cc):
        yr = y.double().clone().requires_grad_(True)
        g_r, b_r = gamma.double().clone().requires_grad_(True), beta.double().clone().requires_grad_(True)
        yt = yr.reshape(T, P, C)
        m = yt.mean(1, keepdim=True)
        var = yt.var(1, unbiased=False, keepdim=True)
        x = (yt - m) / torch.sqrt(var + 1e-5) * g_r + b_r
        v0r = v0.double().clone().reshape(P, C).requires_grad_(True)
        s, vfin, _ = O.lif_sequence(x, v0r)
        flips = int((s.detach() != out.reshape(s.shape).double()).sum())
        loss = (s * gs.double().reshape(s.shape)).sum() + cc * s.sum() + (vfin * gvf.double().reshape(P, C)).sum()
        return flips, torch.autograd.grad(loss, (yr, g_r, b_r, v0r))

    flips, (gy_ref, gg_ref, gb_ref, gv0_ref) = ref(c)
    if flips:
        pytest.skip(f"{flips} spikes flip between the fp64 reference BN and the kernel's fp32 BN")
    assert rel_err(dy, gy_ref) < 4e-3
    assert rel_err(dgamma, gg_ref) < 2e-4 and rel_err(dbeta, gb_ref) < 2e-4
    assert rel_err(gv0.reshape(P, C), gv0_ref) < 1e-4
    if case == "gs_dominant":
        _, (_, gg0, gb0, _) = ref(0.0)
        _, _, _, dg0, db0 = _bwd(K, y, scale, shift, mean, invstd, beta, gs, T, v0, gvf.reshape(-1), torch.zeros(1, device=DEV))
        # the addend's own share of the parameter gradients: neither lost (0) nor doubled (2x)
        assert rel_err(dbeta - db0, gb_ref - gb0) < 0.05 and rel_err(dgamma - dg0, gg_ref - gg0) < 0.05
        assert float((gb_ref - gb0).norm()) > 0.0


# ------------------------------------------------------------------------------------------------------------------
# 4.-8. model level
# ------------------------------------------------------------------------------------------------------------------
def _small(seed, train=True):
    """A half-width LIF detector (widths 64-512)."""
    from snn_object_detectionddp_b200.model import TemporalUNet, YOLOTemporalUNet
    from snn_object_detectionddp_b200.weight_initialization import initialize_model
    torch.manual_seed(seed)
    net = YOLOTemporalUNet(num_classes=8, hyp=HYP, neuron="lif")
    net.temporal_unet = TemporalUNet([144, 144, 144], neuron="lif", widths=(64, 128, 256, 512))
    initialize_model(net)
    return net.to(DEV).train(train)


def _frames(B, T, H, W, seed):
    from snn_object_detectionddp_b200.data import synthetic_batch
    frames, labels = synthetic_batch(B, T, H, W, seed=seed)
    return frames.to(DEV), labels


def _step_data(tr, B, T, H, seed):
    frames, labels = _frames(B, T, H, H, seed)
    return frames, {"padded": tuple(t.to(DEV) for t in tr.prepare_batch(labels, B, max_boxes=8)["padded"])}


def _sync_state(src, dst):
    for name in ("flat_p", "flat_m", "flat_v", "shadow", "flat_g"):
        getattr(dst.store, name).copy_(getattr(src.store, name))
    for a, b in zip(src.model.buffers(), dst.model.buffers()):
        b.copy_(a)
    dst._step_dev.copy_(src._step_dev)
    dst.step_idx = src.step_idx


def _flat_grad(tr, frames, batch, reg, seed_scale):
    """One forward + backward of the trainer's model (no optimizer step); returns a copy of the flat gradient."""
    st = tr.store
    st.zero_grad()
    if reg is not None:
        reg.begin_step()
    det, _ = tr.model.forward_sequence(frames, spike_reg=reg)
    if reg is not None:
        reg.finish_forward(frames.shape[0], frames.shape[1])
    loss, _ = tr.loss_fn(det, batch)
    torch.autograd.backward((loss,), (torch.full((3,), float(seed_scale), device=DEV),))
    return st.flat_g.clone()


def test_model_counts_coefficients_and_gradient_split():
    from snn_object_detectionddp_b200.spikes import SpikeRateLoss
    from snn_object_detectionddp_b200.trainer import Trainer
    B, T = 2, 4
    with _deterministic():
        tr = Trainer(_small(seed=11), total_steps=10, device=DEV)
        reg = SpikeRateLoss(tr.model, synops_weight=1e5, synops_max=0.0, rate_min=0.2, rate_min_weight=1e3, max_T=8)
        frames, batch = _step_data(tr, B, T, 128, seed=70)
        # counts == count_nonzero of the recorded spikes; coef / last == the float64 specification on those counts
        rec = {}
        reg.begin_step()
        with torch.no_grad():
            tr.model.forward_sequence(frames, record=rec, spike_reg=reg)
        reg.finish_forward(B, T)
        s = torch.stack([torch.count_nonzero(rec[n].view(T, -1), dim=1) for n in reg.layers])
        n = torch.tensor([rec[n].numel() // T for n in reg.layers], device=DEV)
        assert torch.equal(reg.counts[:, 0, :T], s) and torch.equal(reg.counts[:, 1, :T], n[:, None].expand(-1, T))
        assert int(reg.counts[:, :, T:].abs().sum()) == 0
        P, phi, R, c = reference(reg.counts.cpu().numpy(), [reg.fanout[k] for k in reg.layers], 1e5, 0.0, 0.2, 1e3, B)
        last, coef = reg.last.cpu().numpy(), reg.coef.cpu().numpy()
        for got, ref in [(last[0], P), (last[1], phi)] + list(zip(last[2:], R)) + list(zip(coef, c)):
            assert _ulps(got, ref) <= 1.0, (got, ref)
        assert reg.read()["spike_reg/penalty"] == float(last[0]) and P > 0
        # flat gradient with the penalty == detection-only + penalty-only (detection seed 0), to the bf16 rounding of dy
        g_both = _flat_grad(tr, frames, batch, reg, 1.0)
        g_det = _flat_grad(tr, frames, batch, None, 1.0)
        g_pen = _flat_grad(tr, frames, batch, reg, 0.0)
    print(f"flat gradient norms: detection {float(g_det.norm()):.4e}, penalty {float(g_pen.norm()):.4e}")
    assert float(g_pen.norm()) > 0.1 * float(g_det.norm())          # observed 3.2e3 against 4.1e3
    assert rel_err(g_both, g_det + g_pen) < 1e-2, (rel_err(g_both, g_det + g_pen), float(g_pen.norm()), float(g_det.norm()))


def test_zero_weights_attached_are_bit_equal_to_no_regularizer():
    from snn_object_detectionddp_b200.spikes import SpikeRateLoss
    from snn_object_detectionddp_b200.trainer import Trainer
    B, T = 2, 4
    with _deterministic():
        a = Trainer(_small(seed=13), total_steps=10, device=DEV)
        b = Trainer(_small(seed=13), total_steps=10, device=DEV)
        _sync_state(a, b)
        b.spike_reg = SpikeRateLoss(b.model, 0.0, synops_max=0.1, rate_min=0.3, rate_min_weight=0.0)
        for i in range(3):
            frames, batch = _step_data(a, B, T, 128, seed=80 + i)
            la, ia = a.train_step(frames, batch)
            lb, ib = b.train_step(frames, batch)
            assert torch.equal(la, lb) and torch.equal(ia, ib), i
        assert int(b.spike_reg.counts[:, 1].sum()) > 0 and float(b.spike_reg.last[1]) > 0
        assert torch.equal(b.spike_reg.coef, torch.zeros_like(b.spike_reg.coef))
    for name in ("flat_p", "flat_m", "flat_v"):
        assert torch.equal(getattr(a.store, name), getattr(b.store, name)), name


def test_graphed_equals_eager():
    from snn_object_detectionddp_b200.spikes import SpikeRateLoss
    from snn_object_detectionddp_b200.trainer import Trainer
    B, T = 2, 4
    kw = dict(synops_weight=20.0, synops_max=0.02, rate_min=0.05, rate_min_weight=1.0)
    with _deterministic():
        a = Trainer(_small(seed=17), total_steps=20, device=DEV)
        b = Trainer(_small(seed=17), total_steps=20, device=DEV)
        _sync_state(a, b)
        a.spike_reg, b.spike_reg = SpikeRateLoss(a.model, **kw), SpikeRateLoss(b.model, **kw)
        for i in range(5):
            frames, batch = _step_data(a, B, T, 128, seed=90 + i)
            a.train_step(frames, batch)
            b.train_step_graphed(frames, batch)
            assert torch.equal(a.spike_reg.last, b.spike_reg.last), i
        assert b._graph is not None and float(a.spike_reg.last[0]) > 0
    for name in ("flat_p", "flat_m", "flat_v"):
        assert torch.equal(getattr(a.store, name), getattr(b.store, name)), name
    # detaching re-captures without the regularizer
    g = b._graph
    b.spike_reg = None
    for i in range(3):
        b.train_step_graphed(*_step_data(b, B, T, 128, seed=90 + i))
    assert b._graph is not g


def test_launch_sequence_and_co_attached_stats():
    from snn_object_detectionddp_b200 import _lib
    from snn_object_detectionddp_b200.spikes import SpikeRateLoss, SpikeStats
    from snn_object_detectionddp_b200.trainer import Trainer
    B, T = 2, 2
    tr = Trainer(_small(seed=19), total_steps=10, device=DEV)
    frames, batch = _step_data(tr, B, T, 128, seed=40)
    tr.train_step(frames, batch)

    def traced():
        _lib.trace = []
        try:
            tr.train_step(frames, batch)
        finally:
            seq, _lib.trace = _lib.trace, None
        return seq

    plain = traced()
    reg = SpikeRateLoss(tr.model, 1.0, rate_min=0.1, rate_min_weight=1.0)
    assert traced() == plain                                   # exists, not attached
    tr.spike_reg = reg
    try:
        attached = traced()
    finally:
        tr.spike_reg = None
    names = [n for n, _ in attached]
    assert names.count("snn_spike_reg_coef") == 1 and names.count("snn_bn_act_fwd_count") == 16
    assert names.count("snn_bn_act_bwd2_ds") == 32
    assert names.count("snn_bn_act_fwd") == [n for n, _ in plain].count("snn_bn_act_fwd") - 16      # the SiLU head's stay
    i = names.index("snn_spike_reg_coef")
    assert all("loss" not in n for n in names[:i]) and "loss" in names[i + 1]
    assert max(k for k, n in enumerate(names) if n == "snn_bn_act_fwd_count") < i
    mapped = [({"snn_bn_act_fwd_count": "snn_bn_act_fwd", "snn_bn_act_bwd2_ds": "snn_bn_act_bwd2"}.get(n, n), w)
              for n, w in attached if n != "snn_spike_reg_coef"]
    assert mapped == plain
    # co-attached SpikeStats: the same counts as the same steps with the stats alone (the coefficient launch hands them on)
    with _deterministic():
        x = Trainer(_small(seed=21), total_steps=10, device=DEV)
        y = Trainer(_small(seed=21), total_steps=10, device=DEV)
        _sync_state(x, y)
        sx, sy = SpikeStats(x.model), SpikeStats(y.model)
        x.model.spike_stats, y.model.spike_stats = sx, sy
        y.spike_reg = SpikeRateLoss(y.model, 0.0)                  # zero weights: the two runs take the same steps
        for i in range(3):
            f, bt = _step_data(x, B, T, 128, seed=50 + i)
            x.train_step(f, bt)
            y.train_step(f, bt)
    assert int(sx.counts[:, 1].sum()) > 0 and torch.equal(sx.counts, sy.counts)


def test_regularizer_lowers_the_synops_fraction():
    """Seed 23, 40 steps of the same 4 batches (B = 4, T = 4, 128 x 128), max_lr 1e-3: the step SynOps fraction of the run
    with synops_weight = 1e4 ends clearly below that of the plain run (a zero-weight regularizer measures the plain one).
    Observed on a B200: plain 0.1726, regularized 0.1417 (mean of the last 4 steps; each run's 4 values within 0.001)."""
    from snn_object_detectionddp_b200.spikes import SpikeRateLoss
    from snn_object_detectionddp_b200.trainer import Trainer
    B, T = 4, 4
    plain = Trainer(_small(seed=23), max_lr=1e-3, total_steps=40, device=DEV)
    regd = Trainer(_small(seed=23), max_lr=1e-3, total_steps=40, device=DEV)
    _sync_state(plain, regd)
    plain.spike_reg = SpikeRateLoss(plain.model, 0.0)
    regd.spike_reg = SpikeRateLoss(regd.model, 1e4)
    data = [_step_data(plain, B, T, 128, seed=100 + i) for i in range(4)]
    phis = []
    for step in range(40):
        frames, batch = data[step % 4]
        plain.train_step_graphed(frames, batch)
        regd.train_step_graphed(frames, batch)
        if step >= 36:
            phis.append((float(plain.spike_reg.last[1]), float(regd.spike_reg.last[1])))
    phi_plain = sum(p for p, _ in phis) / len(phis)
    phi_reg = sum(r for _, r in phis) / len(phis)
    print(f"step SynOps fraction over the last 4 steps: plain {phi_plain:.5f}, regularized {phi_reg:.5f}")
    assert phi_reg < 0.9 * phi_plain, (phi_plain, phi_reg, phis)


def test_train_loop_logs_the_penalty(tmp_path):
    from snn_object_detectionddp_b200.data import synthetic_batch
    from snn_object_detectionddp_b200.train import train_loop

    class W:
        def __init__(self):
            self.scalars = []

        def add_scalar(self, tag, v, step):
            self.scalars.append((tag, float(v), step))

        def add_scalars(self, tag, d, step):
            pass

    model = _small(seed=29, train=False)
    train = [synthetic_batch(2, 3, 128, 128, seed=110 + i) for i in range(3)]
    val = [synthetic_batch(2, 3, 128, 128, seed=120)]
    config = {"training": {"epochs": 2, "learning_rate": 1e-4, "weight_decay": 5e-4,
                           "spike_reg": {"synops_weight": 10.0, "rate_min": 0.05, "rate_min_weight": 1.0}},
              "dataset": {"train": {"seq_len": 3}}}
    w = W()
    tr = train_loop(model, train, val, config, DEV, tmp_path, writer=w, log_every=2, graphed=True, max_boxes=8)
    assert tr.spike_reg is None
    batch_tags = [(v, s) for t, v, s in w.scalars if t == "Loss/train_spike_reg_batch"]
    epoch_tags = [(v, s) for t, v, s in w.scalars if t == "Loss/train_spike_reg"]
    assert [s for _, s in batch_tags] == list(range(6)) and [s for _, s in epoch_tags] == [0, 1]
    assert all(v > 0 for v, _ in batch_tags)
    for e in (0, 1):
        mean = sum(v for v, s in batch_tags if s // 3 == e) / 3
        assert epoch_tags[e][0] == pytest.approx(mean, rel=1e-5)
    assert {t for t, _, _ in w.scalars} >= {"Loss/train_batch", "Loss/train", "Loss/val"}
