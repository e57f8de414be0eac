"""Host side of the spike-rate regularizer (no GPU): the float64 specification of (P, phi, R, c) from one step's counts, c
against a central finite difference of B * P, argument validation, and the extra column of the training-loop metrics."""
import numpy as np
import pytest
import torch

from tests.test_spike_stats_host import TABLE_256


def reference(counts, fanout, a, phi_max, r_min, b, B):
    """float64 specification (DESIGN.md section 3), evaluated left to right in the order snn_spike_reg_coef uses.
    counts int64 [L][2][max_T], fanout [L] -> (P, phi, R [L], c [L]) as Python floats."""
    counts = np.asarray(counts, dtype=np.int64)
    L = counts.shape[0]
    S = [float(int(v)) for v in counts[:, 0, :].sum(axis=1)]
    N = [float(int(v)) for v in counts[:, 1, :].sum(axis=1)]
    F = [float(v) for v in fanout]
    num = den = pr = 0.0
    for i in range(L):
        num = num + F[i] * S[i]
        den = den + F[i] * N[i]
    R, H = [], []
    for i in range(L):
        r = S[i] / N[i] if N[i] > 0 else 0.0
        h = max(0.0, r_min + -r) if N[i] > 0 else 0.0
        R.append(r)
        H.append(h)
        if N[i] > 0:
            pr = pr + h * h
    phi = num / den if den > 0 else 0.0
    hp = max(0.0, phi + -phi_max)
    P = a * hp * hp + (b / L) * pr
    c = []
    for i in range(L):
        u = 2.0 * a * hp * F[i] / den if den > 0 else 0.0
        v = 2.0 * b / L * H[i] / N[i] if N[i] > 0 else 0.0
        c.append(B * (u + -v))
    return P, phi, R, c


def penalty(S, N, F, a, phi_max, r_min, b):
    """P as a function of real-valued spike totals S (the quantity c differentiates)."""
    L = len(S)
    phi = sum(f * s for f, s in zip(F, S)) / sum(f * n for f, n in zip(F, N))
    return a * max(0.0, phi - phi_max) ** 2 + b / L * sum(max(0.0, r_min - s / n) ** 2 for s, n in zip(S, N))


def synthetic_counts(seed, L=16, T=4, max_T=8, rate_hi=0.3, top=1 << 40):
    rng = np.random.default_rng(seed)
    buf = np.zeros((L, 2, max_T), dtype=np.int64)
    steps = rng.integers(1 << 20, top // T, size=(L, 1)) * np.ones((1, T), dtype=np.int64)
    buf[:, 1, :T] = steps
    buf[:, 0, :T] = (steps * rng.uniform(0.0, rate_hi, size=(L, T))).astype(np.int64)
    return buf


FAN = list(TABLE_256.values())
# (a, phi_max, r_min, b): both hinges active, only the SynOps hinge, only the rate hinge, neither
CASES = [(2.0, 0.01, 0.2, 3.0), (2.0, 0.01, 0.0, 3.0), (2.0, 1.0, 0.2, 3.0), (2.0, 1.0, 0.0, 3.0)]


@pytest.mark.parametrize("a,phi_max,r_min,b", CASES)
def test_coefficient_is_b_times_the_penalty_gradient(a, phi_max, r_min, b):
    B = 16
    counts = synthetic_counts(3, top=1 << 24)
    P, phi, R, c = reference(counts, FAN, a, phi_max, r_min, b, B)
    S = [float(v) for v in counts[:, 0].sum(axis=1)]
    N = [float(v) for v in counts[:, 1].sum(axis=1)]
    assert P == pytest.approx(penalty(S, N, FAN, a, phi_max, r_min, b), rel=1e-12, abs=0.0)
    assert phi == pytest.approx(sum(f * s for f, s in zip(FAN, S)) / sum(f * n for f, n in zip(FAN, N)), rel=1e-15)
    assert R == [s / n for s, n in zip(S, N)]
    active_phi, active_rate = phi > phi_max, any(r < r_min for r in R)
    assert (active_phi, active_rate) == {0: (True, True), 1: (True, False), 2: (False, True), 3: (False, False)}[CASES.index((a, phi_max, r_min, b))]
    if not (active_phi or active_rate):
        assert P == 0.0 and c == [0.0] * len(c)
        return
    for i in range(len(S)):
        h = 1e-3 * N[i] * 1e-3                          # far from every hinge's kink at these counts
        up, dn = list(S), list(S)
        up[i] += h
        dn[i] -= h
        fd = B * (penalty(up, N, FAN, a, phi_max, r_min, b) - penalty(dn, N, FAN, a, phi_max, r_min, b)) / (2 * h)
        assert c[i] == pytest.approx(fd, rel=1e-5, abs=1e-12 * max(abs(x) for x in c)), (i, c[i], fd)
    if active_phi and not active_rate:                  # the SynOps term alone: c proportional to the fan-out
        assert all(ci > 0 for ci in c)
        np.testing.assert_allclose(np.array(c) / np.array(FAN), c[0] / FAN[0], rtol=1e-12)
    if active_rate and not active_phi:                  # the rate term alone: pushes only the layers under the floor up
        assert all((ci < 0) == (r < r_min) and (ci == 0) == (r >= r_min) for ci, r in zip(c, R))


def test_empty_layers_and_zero_weights():
    counts = synthetic_counts(5)
    counts[2] = 0                                       # a layer that did not run: no rate term, R = 0
    P, phi, R, c = reference(counts, FAN, 0.0, 0.0, 0.5, 0.0, 8)
    assert P == 0.0 and c == [0.0] * 16 and R[2] == 0.0 and 0.0 < phi < 1.0
    P, _, _, c = reference(counts, FAN, 0.0, 0.0, 0.5, 1.0, 8)
    assert c[2] == 0.0 and P > 0.0 and all(ci < 0 for i, ci in enumerate(c) if i != 2 and R[i] < 0.5)


@pytest.fixture(scope="module")
def lif_model():
    from snn_object_detectionddp_b200.model import YOLOTemporalUNet
    return YOLOTemporalUNet(num_classes=8, neuron="lif", extractor_backend="standin")


def test_constructor_validates_its_arguments(lif_model):
    from snn_object_detectionddp_b200.model import YOLOTemporalUNet
    from snn_object_detectionddp_b200.spikes import SpikeRateLoss, SpikeStats
    reg = SpikeRateLoss(lif_model, 1.0, synops_max=0.1, rate_min=0.01, rate_min_weight=0.5, max_T=8)
    assert reg.layers == list(TABLE_256) == SpikeStats(lif_model).layers
    assert reg.counts.shape == (16, 2, 8) and reg.counts.dtype == torch.int64
    assert reg.coef.shape == (16,) and reg.last.shape == (18,) and reg.coef.dtype == reg.last.dtype == torch.float32
    assert reg.layer_grad("up2.conv1").data_ptr() == reg.coef[12:13].data_ptr()
    for kw, match in ((dict(synops_weight=-1.0), "synops_weight"), (dict(synops_weight=float("nan")), "synops_weight"),
                      (dict(synops_weight=1.0, rate_min_weight=-0.1), "rate_min_weight"),
                      (dict(synops_weight=1.0, rate_min_weight=float("inf")), "rate_min_weight"),
                      (dict(synops_weight=1.0, synops_max=1.5), "synops_max"), (dict(synops_weight=1.0, synops_max=-0.1), "synops_max"),
                      (dict(synops_weight=1.0, rate_min=2.0), "rate_min"), (dict(synops_weight=1.0, max_T=0), "max_T"),
                      (dict(synops_weight=1.0, max_T=65), "max_T")):
        with pytest.raises(ValueError, match=match):
            SpikeRateLoss(lif_model, **kw)
    with pytest.raises(ValueError, match="SpikeRateLoss needs a model with LIF layers"):
        SpikeRateLoss(YOLOTemporalUNet(num_classes=8, neuron="silu", extractor_backend="standin"), 1.0)
    u = lif_model.temporal_unet
    with pytest.raises(ValueError, match=r"T=9 .*SpikeRateLoss\(max_T=8\)"):
        reg.begin_forward(u, 9, lif_model.feature_extractor.feature_hw(256, 256), reg.counts.device)
    with pytest.raises(ValueError, match="train-mode"):
        lif_model.eval().forward_sequence(torch.zeros(1, 2, 3, 64, 64), spike_reg=reg)
    lif_model.train()


def test_device_metrics_extra_column_and_tags():
    from snn_object_detectionddp_b200.train import DeviceMetrics, _log_batches

    class W:
        def __init__(self):
            self.s = []

        def add_scalar(self, tag, v, step):
            self.s.append((tag, float(v), step))

        def add_scalars(self, tag, d, step):
            pass

    m, w = DeviceMetrics("cpu", every=2, extra=True), W()
    for k in range(3):
        if m.update(torch.tensor([1.0, 2.0, 3.0]), k, 0.1, scale=2.0, extra=torch.tensor([0.25 * k])):
            _log_batches(w, m.flush(), True)
    _log_batches(w, m.flush(), True)
    assert [(t, v, s) for t, v, s in w.s if t == "Loss/train_spike_reg_batch"] == [("Loss/train_spike_reg_batch", 0.25 * k, k)
                                                                                  for k in range(3)]
    assert m.extra_average(3) == pytest.approx(0.25) and m.averages(3)[0] == pytest.approx(12.0)
    plain = DeviceMetrics("cpu", every=2)
    plain.update(torch.tensor([1.0, 2.0, 3.0]), 0, 0.1, scale=2.0)
    assert len(plain.flush()[0]) == 4
