"""-m gpu: exponential moving average of the weights (snn_ema_update, ema.ModelEMA).

The specification is ultralytics' ModelEMA.update on fp32 tensors, run by torch on the same GPU:
    d = decay * (1 - math.exp(-updates / tau));  v *= d;  v += (1 - d) * source
Every comparison is an equality."""
import contextlib
import math
import os
import socket

import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda"
HYP = {"box": 7.5, "cls": 1.0, "dfl": 2.5, "reg_max": 16}


def _d(k, decay, tau):
    return decay * (1 - math.exp(-k / tau))


def _spec(v, s, d):
    """ultralytics' two lines, in place on fp32 tensors."""
    v *= d
    v += (1 - d) * s


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


def _values(n, gen):
    """fp32 values over many magnitudes, with zeros, subnormals and signs."""
    x = torch.randn(n, device=DEV, generator=gen) * torch.exp2(torch.randint(-30, 30, (n,), device=DEV, generator=gen).float())
    x[::97] = 0.0
    x[5::101] = 1e-40
    x[7::103] = -3e-39
    return x


# ------------------------------------------------------------------------------------------------------------------
# 1. kernel vs specification
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("decay,tau", [(0.9999, 2000), (0.999, 100)])
def test_kernel_is_bit_identical_to_torch(decay, tau):
    from snn_object_detectionddp_b200 import kernels as K
    from snn_object_detectionddp_b200.ema import decay_table
    table = decay_table(decay, tau).to(DEV)
    rows = table.shape[0]
    gen = torch.Generator(device=DEV).manual_seed(1)
    seg_lens = (1, 3, 8, 144, 4096)
    pool = _values(2 * sum(seg_lens) + 64, gen)
    full = 120_327_528 // 8 * 8 + 8 * 200
    for n in (8, 12, 1000, 4100, (1 << 20) + 8, full):
        e0, s = _values(n, gen), _values(n, gen)
        # segments at odd offsets of one pool (unaligned addresses), averaged from a second pool
        src_pool = _values(pool.numel(), gen)
        offs, o = [], 1
        for ln in seg_lens:
            offs.append(o)
            o += ln + 1
        for k in ((1, 2, 2000, rows, rows + 5, 10 * rows) if n in (8, full) else (1, 2000, rows + 5)):
            e, p = e0.clone(), pool.clone()
            seg = torch.tensor([(src_pool[a:].data_ptr(), p[a:].data_ptr(), ln) for a, ln in zip(offs, seg_lens)],
                               dtype=torch.int64).to(DEV)
            counter = torch.full((1,), k - 1, device=DEV, dtype=torch.int32)
            K.ema_update(e, s, table, counter, seg, sum(seg_lens))
            ref, pref = e0.clone(), pool.clone()
            d = _d(k, decay, tau)
            _spec(ref, s, d)
            for a, ln in zip(offs, seg_lens):
                _spec(pref[a:a + ln], src_pool[a:a + ln], d)
            assert torch.equal(e, ref), (n, k)
            assert torch.equal(p, pref), (n, k)       # segment tails, and nothing between the segments touched
            assert int(counter) == k
        del e0, s, e, ref


@pytest.mark.parametrize("decay,tau", [(0.9999, 2000), (0.9, 3)])
def test_fifty_consecutive_updates_with_a_changing_source(decay, tau):
    from snn_object_detectionddp_b200 import kernels as K
    from snn_object_detectionddp_b200.ema import decay_table
    table = decay_table(decay, tau).to(DEV)
    gen = torch.Generator(device=DEV).manual_seed(2)
    n = 3 * 1024 + 8
    e, s = _values(n, gen), _values(n, gen)
    bs, be = _values(144, gen), _values(144, gen)
    seg = torch.tensor([(bs.data_ptr(), be.data_ptr(), 144)], dtype=torch.int64).to(DEV)
    ref, bref = e.clone(), be.clone()
    counter = torch.zeros(1, device=DEV, dtype=torch.int32)
    for k in range(1, 51):
        s.add_(_values(n, gen), alpha=0.01)
        bs.mul_(1.001)
        K.ema_update(e, s, table, counter, seg, 144)
        d = _d(k, decay, tau)
        _spec(ref, s, d)
        _spec(bref, bs, d)
        assert torch.equal(e, ref) and torch.equal(be, bref), k
    assert int(counter) == 50


def test_kernel_rejects_bad_arguments():
    from snn_object_detectionddp_b200 import kernels as K
    from snn_object_detectionddp_b200._lib import SnnKernelError
    t, c = torch.ones(4, 2, device=DEV), torch.zeros(1, device=DEV, dtype=torch.int32)
    x = torch.zeros(16, device=DEV)
    with pytest.raises(ValueError):
        K.ema_update(x, torch.zeros(8, device=DEV), t, c)
    with pytest.raises(ValueError):
        K.ema_update(x, x.double(), t, c)
    with pytest.raises(ValueError):
        K.ema_update(x, x, t, c.long())
    with pytest.raises(SnnKernelError):
        K.ema_update(x[:6], x[8:14], t, c)                      # not a multiple of 4
    with pytest.raises(SnnKernelError):
        K.ema_update(x[1:9], x[8:16], t, c)                     # not 16-byte aligned


# ------------------------------------------------------------------------------------------------------------------
# 2./3. through the trainer
# ------------------------------------------------------------------------------------------------------------------
def _model(neuron, seed, widths=(64, 128, 256, 512)):
    from snn_object_detectionddp_b200.model import TemporalUNet, YOLOTemporalUNet
    from snn_object_detectionddp_b200.weight_initialization import initialize_model
    torch.manual_seed(seed)
    net = YOLOTemporalUNet(num_classes=8, hyp=HYP, neuron=neuron, extractor_backend="standin")
    net.temporal_unet = TemporalUNet([144, 144, 144], neuron=neuron, widths=widths)
    initialize_model(net)
    return net.to(DEV)


def _steps(tr, n, seed, B=2, T=3, HW=128):
    from snn_object_detectionddp_b200.data import synthetic_batch
    out = []
    for i in range(n):
        frames, labels = synthetic_batch(B, T, HW, HW, seed=seed + i)
        out.append((frames.to(DEV), {"padded": tuple(t.to(DEV) for t in tr.prepare_batch(labels, B, max_boxes=8)["padded"])}))
    return out


def _sync_state(src, dst):
    for name in ("flat_p", "flat_m", "flat_v", "shadow", "flat_g"):
        getattr(dst.store, name).copy_(getattr(src.store, name))
    for a, b in zip(src.model.buffers(), dst.model.buffers()):
        b.copy_(a)
    dst._step_dev.copy_(src._step_dev)
    dst.step_idx = src.step_idx


class _Replica:
    """ultralytics' ModelEMA on a state dict, each tensor once (the model's state dict names the head twice)."""

    def __init__(self, model, decay=0.9999, tau=2000):
        self.decay, self.tau, self.updates = decay, tau, 0
        sd = model.state_dict()
        self.canon, seen = {}, {}
        for k, v in sd.items():
            key = (v.data_ptr(), tuple(v.shape), v.dtype)
            self.canon[k] = seen.setdefault(key, k)
        self.sd = {k: v.detach().clone() for k, v in sd.items() if self.canon[k] == k}

    def update(self, model):
        self.updates += 1
        d = _d(self.updates, self.decay, self.tau)
        live = model.state_dict()
        for k, v in self.sd.items():
            if v.dtype.is_floating_point:
                _spec(v, live[k].detach(), d)

    def __getitem__(self, k):
        return self.sd[self.canon[k]]


@pytest.mark.parametrize("neuron", ["lif", "silu"])
def test_trainer_ema_equals_ultralytics_replica(neuron):
    from snn_object_detectionddp_b200.ema import ModelEMA
    from snn_object_detectionddp_b200.trainer import Trainer
    tr = Trainer(_model(neuron, seed=3), total_steps=20, device=DEV)
    for frames, batch in _steps(tr, 1, seed=10):          # the BatchNorm statistics have moved off their initial values
        tr.train_step(frames, batch)
    tr.ema = ema = ModelEMA(tr.model)
    rep = _Replica(tr.model)
    nbt0 = {k: v.clone() for k, v in tr.model.state_dict().items() if k.endswith("num_batches_tracked")}
    for frames, batch in _steps(tr, 4, seed=20):
        tr.train_step(frames, batch)
        rep.update(tr.model)
    assert ema.updates == 4 and rep.updates == 4
    sd = ema.ema.state_dict()
    assert list(sd) == list(tr.model.state_dict())
    n_bn = 0
    for k, v in sd.items():
        if v.dtype.is_floating_point:
            assert torch.equal(v, rep[k]), k
            n_bn += k.endswith("running_var")
        else:
            assert torch.equal(v, nbt0[k]), k
    assert n_bn > 10
    # the frozen DFL projection is averaged like every other floating-point entry (ultralytics: it drifts by ulps)
    n_unique_bn = sum(k.endswith("running_var") and not k.startswith("model.0.") for k in sd)
    assert "detection_head.dfl.conv.weight" in sd and len(ema._bufs) == 2 * n_unique_bn + 1
    assert not torch.equal(sd["detection_head.cv2.0.0.bn.running_mean"], tr.model.state_dict()["detection_head.cv2.0.0.bn.running_mean"])
    assert ema.ema.feature_extractor is tr.model.feature_extractor
    live = tr.model.state_dict()
    assert all(torch.equal(v, live[k]) for k, v in sd.items() if k.startswith("feature_extractor."))
    assert ema.ema._snn_store.flat_g is None and ema.ema._snn_store.flat_m is None and not ema.ema.training


def test_training_is_untouched_by_an_attached_ema():
    from snn_object_detectionddp_b200.ema import ModelEMA
    from snn_object_detectionddp_b200.trainer import Trainer
    with _deterministic():
        a = Trainer(_model("lif", seed=5), total_steps=10, device=DEV)
        b = Trainer(_model("lif", seed=5), total_steps=10, device=DEV)
        _sync_state(a, b)
        b.ema = ModelEMA(b.model)
        for frames, batch in _steps(a, 3, seed=30):
            _, ia = a.train_step(frames, batch)
            _, ib = b.train_step(frames, batch)
            assert torch.equal(ia, ib)
        for name in ("flat_p", "flat_m", "flat_v", "shadow"):
            assert torch.equal(getattr(a.store, name), getattr(b.store, name)), name
        assert all(torch.equal(x, y) for x, y in zip(a.model.buffers(), b.model.buffers()))


def test_launch_sequence_with_and_without_ema():
    from snn_object_detectionddp_b200 import _lib
    from snn_object_detectionddp_b200.ema import ModelEMA
    from snn_object_detectionddp_b200.trainer import Trainer
    tr = Trainer(_model("lif", seed=9), total_steps=10, device=DEV)
    (frames, batch), = _steps(tr, 1, seed=40)
    tr.train_step(frames, batch)

    def traced():
        _lib.trace = []
        try:
            tr.train_step(frames, batch)
        finally:
            seq, _lib.trace = _lib.trace, None
        return seq

    plain = traced()
    ema = ModelEMA(tr.model)                         # exists, not attached
    assert traced() == plain
    tr.ema = ema
    with_ema = traced()
    tr.ema = None
    assert traced() == plain
    i = [n for n, _ in plain].index("snn_adamw_step")
    assert [n for n, _ in with_ema] == [n for n, _ in plain[:i + 1]] + ["snn_ema_update"] + [n for n, _ in plain[i + 1:]]
    assert with_ema[:i + 1] == plain[:i + 1] and with_ema[i + 2:] == plain[i + 1:]
    n_el = ema._dst.flat_p.numel() + ema._segment_elems
    assert with_ema[i + 1] == ("snn_ema_update", ("byte", 12.0 * n_el))


# ------------------------------------------------------------------------------------------------------------------
# 4. graphs
# ------------------------------------------------------------------------------------------------------------------
def _ema_state(ema):
    return [ema._dst.flat_p] + [b[1] for b in ema._bufs]


def test_graphed_steps_equal_eager_steps_and_attach_detach_recaptures():
    from snn_object_detectionddp_b200.ema import ModelEMA
    from snn_object_detectionddp_b200.trainer import Trainer
    with _deterministic():
        a = Trainer(_model("lif", seed=7), total_steps=20, device=DEV)
        b = Trainer(_model("lif", seed=7), total_steps=20, device=DEV)
        _sync_state(a, b)
        a.ema, b.ema = ModelEMA(a.model), ModelEMA(b.model)
        steps = _steps(a, 5, seed=50)
        for frames, batch in steps:
            a.train_step(frames, batch)
            b.train_step_graphed(frames, batch)
        assert b._graph is not None
        assert a.ema.updates == b.ema.updates == 5 == b.step_idx
        assert int(b.ema._updates_dev) == 5 and int(b._step_dev) == 5
        assert all(torch.equal(x, y) for x, y in zip(_ema_state(a.ema), _ema_state(b.ema)))
        # update() and replays never read the device
        torch.cuda.synchronize()
        torch.cuda.set_sync_debug_mode("error")
        try:
            b.train_step_graphed(*steps[0])
            b.ema.update()
        finally:
            torch.cuda.set_sync_debug_mode(0)
        assert b.ema.updates == 7 and int(b.ema._updates_dev) == 7
        # detach: re-capture, the average stays as it is
        g_ema, before = b._graph, [t.clone() for t in _ema_state(b.ema)]
        ema_b, b.ema = b.ema, None
        for frames, batch in steps[:3]:
            b.train_step_graphed(frames, batch)
        assert b._graph is not g_ema and all(torch.equal(x, y) for x, y in zip(before, _ema_state(ema_b)))
        assert ema_b.updates == 7
        # attach again: re-capture, the updates resume
        g_plain = b._graph
        b.ema = ema_b
        for frames, batch in steps[:3]:
            b.train_step_graphed(frames, batch)
        assert b._graph is not g_plain and b.ema.updates == 10 and int(b.ema._updates_dev) == 10
        b.ema = None


# ------------------------------------------------------------------------------------------------------------------
# 5. no stale operands
# ------------------------------------------------------------------------------------------------------------------
def _same(r0, r1):
    assert set(r0) == set(r1)
    for k in r0:
        v0, v1 = r0[k], r1[k]
        assert (v0 == v1).all() if hasattr(v0, "shape") else v0 == v1, k


def test_evaluate_model_on_the_average_uses_current_weights():
    from snn_object_detectionddp_b200.data import synthetic_batch
    from snn_object_detectionddp_b200.ema import ModelEMA
    from snn_object_detectionddp_b200.train import evaluate_model
    from snn_object_detectionddp_b200.trainer import Trainer
    loader = [synthetic_batch(4, 3, 128, 128, seed=60 + i) for i in range(2)]
    frames = loader[0][0].to(DEV)
    with _deterministic():
        tr = Trainer(_model("lif", seed=11), total_steps=50, device=DEV)
        tr.ema = ema = ModelEMA(tr.model, decay=0.9, tau=2)       # a fast ramp: the average moves visibly in a few steps
        evaluate_model(ema.ema, loader, DEV)                       # the average has been evaluated before it moves
        for fr, batch in _steps(tr, 4, seed=70):
            tr.train_step(fr, batch)
        tr.store.flat_p.mul_(1.25)                                # a live move the bf16 operand copies cannot round away
        ema.update()
        fresh = _model("lif", seed=99)
        fresh.load_state_dict(ema.state_dict()["state_dict"])
        fresh.eval()
        with torch.no_grad():
            ref = [t.clone() for t in fresh.forward_sequence(frames)[0].flat()]
            got = [t.clone() for t in ema.ema.forward_sequence(frames)[0].flat()]
        assert all(torch.equal(x, y) for x, y in zip(got, ref))
        _same(evaluate_model(ema.ema, loader, DEV), evaluate_model(fresh, loader, DEV))
        # the same check fails when the bf16 operand copies are left as they were before the updates
        tr.store.flat_p.mul_(1.25)
        ema.update()
        st = ema._dst
        st._versions = tuple(e.param._version for e in st.entries)
        fresh.load_state_dict(ema.state_dict()["state_dict"])
        with torch.no_grad():
            ref = [t.clone() for t in fresh.forward_sequence(frames)[0].flat()]
            stale = [t.clone() for t in ema.ema.forward_sequence(frames)[0].flat()]
        assert not all(torch.equal(x, y) for x, y in zip(stale, ref))
        tr.ema = None


def _check_current(ema, frames, features):
    """The average's forward (whole model, and a drop-in submodule forward) equals a fresh model loaded with its state."""
    fresh = _model("lif", seed=99)
    fresh.load_state_dict(ema.state_dict()["state_dict"])
    fresh.eval()
    with torch.no_grad():
        ref = [t.clone() for t in fresh.forward_sequence(frames)[0].flat()]
        got = [t.clone() for t in ema.ema.forward_sequence(frames)[0].flat()]
        ref_u = [t.clone() for t in fresh.temporal_unet(features)[0]]
        got_u = [t.clone() for t in ema.ema.temporal_unet(features)[0]]
    assert all(torch.equal(x, y) for x, y in zip(got, ref))
    assert all(torch.equal(x, y) for x, y in zip(got_u, ref_u))
    return fresh


def test_average_is_current_after_graph_replays():
    from snn_object_detectionddp_b200.data import synthetic_batch
    from snn_object_detectionddp_b200.ema import ModelEMA
    from snn_object_detectionddp_b200.train import evaluate_model
    from snn_object_detectionddp_b200.trainer import Trainer
    loader = [synthetic_batch(4, 3, 128, 128, seed=110 + i) for i in range(2)]
    frames = loader[0][0].to(DEV)
    features = [torch.randn(2, 144, hw, hw, device=DEV) for hw in (16, 8, 4)]
    with _deterministic():
        tr = Trainer(_model("lif", seed=19), total_steps=50, device=DEV)
        tr.ema = ema = ModelEMA(tr.model, decay=0.9, tau=2)
        steps = _steps(tr, 2, seed=120)
        for i in range(4):                                         # eager, eager, capture + replay, replay
            tr.train_step_graphed(*steps[i % 2])
        assert tr._graph is not None and ema.updates == 4
        _check_current(ema, frames, features)                      # operands rebuilt here; replays follow
        for i in range(2):
            tr.store.flat_p.mul_(1.25)                             # a live move the bf16 operand copies cannot round away
            tr.train_step_graphed(*steps[i])
        g = tr._graph
        assert ema.updates == 6 and int(ema._updates_dev) == 6
        fresh = _check_current(ema, frames, features)
        _same(evaluate_model(ema.ema, loader, DEV), evaluate_model(fresh, loader, DEV))
        tr.store.flat_p.mul_(1.25)
        tr.train_step_graphed(*steps[0])
        assert tr._graph is g                                      # replays only, no re-capture in between
        _check_current(ema, frames, features)
        tr.ema = None


def test_replaced_source_buffer_is_an_error():
    from snn_object_detectionddp_b200.ema import ModelEMA
    net = _model("lif", seed=21)
    ema = ModelEMA(net)
    ema.update()
    bn = net.temporal_unet.enc1.bn
    bn.running_mean = bn.running_mean.clone()                     # a new tensor: the segment table still holds the old one
    before = ema._dst.flat_p.clone()
    with pytest.raises(RuntimeError, match="replaced"):
        ema.update()
    assert ema.updates == 1 and torch.equal(ema._dst.flat_p, before)


# ------------------------------------------------------------------------------------------------------------------
# 6. checkpoints
# ------------------------------------------------------------------------------------------------------------------
def test_checkpoint_round_trip(tmp_path):
    from snn_object_detectionddp_b200.ema import ModelEMA
    from snn_object_detectionddp_b200.trainer import Trainer
    with _deterministic():
        a = Trainer(_model("lif", seed=13), total_steps=20, device=DEV)
        a.ema = ModelEMA(a.model)
        steps = _steps(a, 4, seed=80)
        for frames, batch in steps[:2]:
            a.train_step(frames, batch)
        a.save_checkpoint(tmp_path / "with.pt")
        ema_a, a.ema = a.ema, None
        a.save_checkpoint(tmp_path / "without.pt")
        a.ema = ema_a
        ck_w, ck_wo = torch.load(tmp_path / "with.pt", weights_only=False), torch.load(tmp_path / "without.pt", weights_only=False)
        assert "ema" in ck_w and "ema" not in ck_wo
        assert list(ck_w["model_state_dict"]) == list(ck_wo["model_state_dict"])
        assert all(torch.equal(ck_w["model_state_dict"][k], v) for k, v in ck_wo["model_state_dict"].items())
        assert ck_w["ema"]["updates"] == 2 and (ck_w["ema"]["decay"], ck_w["ema"]["tau"]) == (0.9999, 2000)
        assert list(ck_w["ema"]["state_dict"]) == list(ck_w["model_state_dict"])
        assert all(v.device.type == "cpu" for v in ck_w["ema"]["state_dict"].values())

        b = Trainer(_model("lif", seed=14), total_steps=20, device=DEV)
        b.ema = ModelEMA(b.model)
        b.load_checkpoint(tmp_path / "with.pt")
        assert b.ema.updates == 2 and int(b.ema._updates_dev) == 2
        sa, sb = a.ema.ema.state_dict(), b.ema.ema.state_dict()
        assert all(torch.equal(sa[k], sb[k]) for k in sa)
        assert torch.equal(a.ema._dst.flat_p, b.ema._dst.flat_p)
        for frames, batch in steps[2:]:
            a.train_step(frames, batch)
            b.train_step(frames, batch)
        sa, sb = a.ema.ema.state_dict(), b.ema.ema.state_dict()
        assert all(torch.equal(sa[k], sb[k]) for k in sa) and a.ema.updates == b.ema.updates == 4

        # a file without 'ema' leaves a fresh average alone; a trainer without one ignores the file's
        c = Trainer(_model("lif", seed=15), total_steps=20, device=DEV)
        c.ema = ModelEMA(c.model)
        before = {k: v.clone() for k, v in c.ema.ema.state_dict().items()}
        torch.save({"model_state_dict": ck_wo["model_state_dict"]}, tmp_path / "reference.pt")
        c.load_checkpoint(tmp_path / "reference.pt")
        c.load_checkpoint(tmp_path / "without.pt")
        assert c.ema.updates == 0 and all(torch.equal(v, before[k]) for k, v in c.ema.ema.state_dict().items())
        d = Trainer(_model("lif", seed=16), total_steps=20, device=DEV)
        d.load_checkpoint(tmp_path / "with.pt")
        assert d.ema is None and torch.equal(d.store.flat_p, c.store.flat_p)
        a.ema = b.ema = c.ema = None


# ------------------------------------------------------------------------------------------------------------------
# 7. train_loop(ema=True)
# ------------------------------------------------------------------------------------------------------------------
class _Writer:
    def __init__(self):
        self.scalars, self.groups = [], []

    def add_scalar(self, tag, value, step):
        self.scalars.append((tag, float(value), step))

    def add_scalars(self, tag, values, step):
        self.groups.append((tag, dict(values), step))


def test_train_loop_validates_the_average(tmp_path):
    from snn_object_detectionddp_b200.data import synthetic_batch
    from snn_object_detectionddp_b200.metrics import DetMetrics
    from snn_object_detectionddp_b200.train import train_loop, validate_one_epoch
    # 3 batches per epoch: the graph is captured in epoch 0, so epoch 1's validation follows replays only
    train = [synthetic_batch(2, 3, 128, 128, seed=90 + i) for i in range(3)]
    val = [synthetic_batch(4, 3, 128, 128, seed=95 + i) for i in range(2)]
    config = {"training": {"epochs": 2, "learning_rate": 1e-3, "weight_decay": 5e-4}, "dataset": {"train": {"seq_len": 3}}}
    runs = {}
    with _deterministic():
        for use_ema in (False, True):
            w, d = _Writer(), tmp_path / str(use_ema)
            tr = train_loop(_model("lif", seed=17), train, val, config, DEV, d, writer=w, log_every=10, graphed=True, max_boxes=8,
                            eval_map=True, ema=use_ema)
            assert tr.ema is None
            runs[use_ema] = (tr, w, d)
        tr, w, d = runs[True]
        ck = torch.load(d / "latest.pt", weights_only=False)
        assert ck["ema"]["updates"] == 6 == ck["trainer_state"]["step_idx"]
        assert "ema" in torch.load(d / "best.pt", weights_only=False)
        avg = _model("lif", seed=98)
        avg.load_state_dict(ck["ema"]["state_dict"])
        m = DetMetrics(avg.nc, DEV)
        val_loss, _ = validate_one_epoch(tr, val, 3, max_boxes=8, metrics=m, model=avg)
        res = m.compute()
    logged = {(t, e): v for t, v, e in w.scalars}
    assert logged[("Loss/val", 1)] == val_loss
    for tag in ("metrics/precision(B)", "metrics/recall(B)", "metrics/mAP50(B)", "metrics/mAP50-95(B)"):
        assert logged[(tag, 1)] == float(res[tag]), tag
    # ema=False: the same tags and files as before, no 'ema' in the checkpoints
    tr0, w0, d0 = runs[False]
    assert sorted({t for t, _, _ in w0.scalars}) == sorted({t for t, _, _ in w.scalars})
    assert sorted(os.listdir(d0)) == sorted(os.listdir(d))
    assert all("ema" not in torch.load(d0 / f, weights_only=False) for f in ("latest.pt", "best.pt"))


# ------------------------------------------------------------------------------------------------------------------
# 8. two ranks
# ------------------------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _ddp_worker(rank, world, port, out):
    import torch.distributed as dist
    from snn_object_detectionddp_b200.data import synthetic_batch
    from snn_object_detectionddp_b200.ema import ModelEMA
    from snn_object_detectionddp_b200.trainer import Trainer
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    torch.manual_seed(0)
    tr = Trainer(_model("lif", seed=0).to(dev), total_steps=20, device=dev, bucket_mb=1)
    tr.ema = ModelEMA(tr.model)
    for step in range(3):
        frames, labels = synthetic_batch(2, 2, 128, 128, seed=200 + step + 17 * rank)     # different batches per rank
        batch = tr.prepare_batch(labels, 2, max_boxes=8)
        tr.train_step(frames.to(dev), {"padded": tuple(t.to(dev) for t in batch["padded"])})
    flat = tr.ema._dst.flat_p.clone()
    gathered = [torch.zeros_like(flat) for _ in range(world)]
    dist.all_gather(gathered, flat)
    torch.cuda.synchronize()
    if rank == 0:
        out.put((all(torch.equal(gathered[0], g) for g in gathered[1:]), tr.ema.updates))
    dist.barrier()
    os._exit(0)


def test_ema_parameters_stay_identical_across_two_ranks():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import time
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.SimpleQueue()
    port = _free_port()
    procs = [ctx.Process(target=_ddp_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    t0 = time.time()
    try:
        while q.empty():
            if any(p.exitcode not in (None, 0) for p in procs) or time.time() - t0 > 300:
                raise AssertionError(f"worker failed or timed out: exit codes {[p.exitcode for p in procs]}")
            time.sleep(0.2)
        same, updates = q.get()
        for p in procs:
            p.join(60)
    finally:
        for p in procs:
            if p.is_alive():
                p.kill()
                p.join()
    assert same and updates == 3
