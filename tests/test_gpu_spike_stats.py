"""-m gpu: spike-activity statistics counted inside the LIF forward kernel (snn_bn_act_fwd_count, spikes.SpikeStats).

Counts are exact integers, so every comparison here is an equality: against the popcount of the spike mask, against
count_nonzero of the recorded spike tensors (not float sums: fp32 loses exactness past 2^24), against eager runs, and
against the definitions of SynOps and dense MACs over the fan-out table."""
import contextlib
import os
import socket

import pytest
import torch

from tests.test_spike_stats_host import TABLE_256

pytestmark = pytest.mark.gpu

DEV = "cuda"
HYP = {"box": 7.5, "cls": 1.0, "dfl": 2.5, "reg_max": 16}


def _product(neuron, seed=0):
    """The default-width detector (widths 128-1024, 144 feature channels), seeded."""
    from snn_object_detectionddp_b200.model import YOLOTemporalUNet
    from snn_object_detectionddp_b200.weight_initialization import initialize_model
    torch.manual_seed(seed)
    net = YOLOTemporalUNet(num_classes=8, hyp=HYP, neuron=neuron)
    initialize_model(net)
    return net.to(DEV)


def _small(seed):
    """A half-width LIF detector (widths 64-512) in eval mode, for the entry-point tests."""
    from snn_object_detectionddp_b200.model import TemporalUNet, YOLOTemporalUNet
    from snn_object_detectionddp_b200.weight_initialization import initialize_model
    torch.manual_seed(seed)
    net = YOLOTemporalUNet(num_classes=8, hyp=HYP, neuron="lif")
    net.temporal_unet = TemporalUNet([144, 144, 144], neuron="lif", widths=(64, 128, 256, 512))
    initialize_model(net)
    return net.to(DEV).eval()


def _sync_state(src, dst):
    """Copy trainer `src`'s whole training state into `dst` in place."""
    for name in ("flat_p", "flat_m", "flat_v", "shadow", "flat_g"):
        getattr(dst.store, name).copy_(getattr(src.store, name))
    for a, b in zip(src.model.buffers(), dst.model.buffers()):
        b.copy_(a)
    dst._step_dev.copy_(src._step_dev)
    dst.step_idx = src.step_idx

POPCOUNT = torch.tensor([bin(i).count("1") for i in range(256)], dtype=torch.int64)


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


# ------------------------------------------------------------------------------------------------------------------
# 1. kernel
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C", [8, 64, 128, 1024])
@pytest.mark.parametrize("T", [1, 2, 4, 8, 16])
def test_counted_kernel_is_exact_and_bit_identical(T, C):
    from snn_object_detectionddp_b200 import kernels as K
    from snn_object_detectionddp_b200._lib import SnnKernelError
    P = 1001                                          # n_per_t / 8 = P * C / 8 is never a multiple of 256: partial last block
    assert (P * C // 8) % 256 != 0
    g = torch.Generator(device=DEV).manual_seed(T * 1000 + C)
    y = torch.randn(T * P, C, device=DEV, generator=g) * 1.5
    n_per_t = P * C
    for per_t in (True, False):
        rows = T if per_t else 1
        scale = torch.rand(rows, C, device=DEV, generator=g) + 0.5
        shift = torch.rand(rows, C, device=DEV, generator=g) * 0.6
        for v0 in (None, torch.randn(n_per_t, device=DEV, generator=g)):
            kw = dict(v_init=v0, want_mask=True, want_v_final=True)
            out0, mask0, vf0 = K.bn_act_fwd(K.ACT_LIF, y, scale, shift, T, **kw)
            spikes = torch.zeros(T, device=DEV, dtype=torch.int64)
            steps = torch.zeros(T, device=DEV, dtype=torch.int64)
            out, mask, vf = K.bn_act_fwd(K.ACT_LIF, y, scale, shift, T, spike_counts=(spikes, steps), **kw)
            assert torch.equal(out, out0) and torch.equal(mask, mask0) and torch.equal(vf, vf0)
            pop = POPCOUNT.to(DEV)[mask.long()].sum(dim=1)
            nz = torch.count_nonzero(out.view(T, -1), dim=1)
            assert torch.equal(spikes, pop) and torch.equal(spikes, nz), (per_t, v0 is None)
            assert torch.equal(steps, torch.full((T,), n_per_t, device=DEV, dtype=torch.int64))
            assert int(spikes.sum()) > 0
            K.bn_act_fwd(K.ACT_LIF, y, scale, shift, T, spike_counts=(spikes, steps), **kw)
            assert torch.equal(spikes, 2 * pop) and torch.equal(steps, torch.full_like(steps, 2 * n_per_t))
    with pytest.raises(SnnKernelError):
        K.bn_act_fwd(K.ACT_SILU, y, scale, shift, T, spike_counts=(spikes, steps))
    bad_views = [(spikes.int(), steps), (spikes, steps[:T - 1])]
    if T > 1:                                         # a strided view (one element is always contiguous)
        bad_views.append((spikes, torch.zeros(2 * T, device=DEV, dtype=torch.int64)[::2]))
    for bad in bad_views:
        with pytest.raises(ValueError, match="spike_counts"):
            K.bn_act_fwd(K.ACT_LIF, y, scale, shift, T, spike_counts=bad)


# ------------------------------------------------------------------------------------------------------------------
# 2./3. model counts, SynOps
# ------------------------------------------------------------------------------------------------------------------
def _frames(B, T, H, W, seed):
    from snn_object_detectionddp_b200.data import synthetic_batch
    frames, labels = synthetic_batch(B, T, H, W, seed=seed)
    return frames.to(DEV), labels


def _record_counts(rec, names, T):
    """[layers][T] spike counts and [layers] neurons per timestep of record= spike tensors (integer counting)."""
    s = torch.stack([torch.count_nonzero(rec[n].view(T, -1), dim=1) for n in names]).cpu()
    n = torch.tensor([rec[n].numel() // T for n in names])
    return s, n


@pytest.fixture(scope="module")
def net():
    return _product("lif", seed=3)


def test_eval_counts_equal_recorded_spikes_and_outputs_are_unchanged(net):
    from snn_object_detectionddp_b200.spikes import SpikeStats
    B, T = 2, 4
    frames, _ = _frames(B, T, 256, 256, seed=1)
    net.eval()
    with _deterministic(), torch.no_grad():
        det0, _ = net.forward_sequence(frames)
        ref = [t.clone() for t in det0.flat()]
        stats = SpikeStats(net)
        net.spike_stats = stats
        rec = {}
        try:
            det, _ = net.forward_sequence(frames, record=rec)
        finally:
            net.spike_stats = None
    assert all(torch.equal(a, b) for a, b in zip(det.flat(), ref))
    res = stats.compute()
    s, n = _record_counts(rec, stats.layers, T)
    assert torch.equal(torch.from_numpy(res["spike_counts"]), s)
    assert torch.equal(torch.from_numpy(res["neuron_steps"]), n[:, None].expand(-1, T))
    assert int(n.sum()) == 933888 * B and int(res["neuron_steps"].sum()) == 933888 * B * T
    # 3. SynOps / dense MACs: the definitions over the fan-out table
    assert stats.fanout == TABLE_256
    synops = sum(TABLE_256[name] * int(s[i].sum()) for i, name in enumerate(stats.layers))
    dense = sum(TABLE_256[name] * int(n[i]) * T for i, name in enumerate(stats.layers))
    assert res["spikes/synops"] == synops and res["spikes/dense_macs"] == dense
    assert res["spikes/synops_fraction"] == synops / dense and 0 < synops < dense
    assert res["spikes/rate"] == int(s.sum()) / (int(n.sum()) * T)


def test_dense_macs_equal_conv_flops_at_256(net):
    from snn_object_detectionddp_b200 import kernels as K
    from snn_object_detectionddp_b200.spikes import SpikeStats
    B, T = 1, 2
    frames, _ = _frames(B, T, 256, 256, seed=2)
    stats = SpikeStats(net)
    net.eval()
    net.spike_stats = stats
    try:
        with torch.no_grad():
            net.forward_sequence(frames)
    finally:
        net.spike_stats = None
    s1, s2, k1, t2 = K.GEOM_3x3_S1, K.GEOM_3x3_S2, K.GEOM_1x1, K.GEOM_T2x2_S2
    nb = B * T
    # every K-slice that consumes a LIF spike tensor: (geometry, input H = W, input channels, Cout)
    slices = [(s2, 32, 128, 256), (s1, 32, 128, 128), (s1, 16, 256, 256), (s1, 16, 256, 256), (s2, 16, 256, 512),
              (s1, 16, 256, 256), (s1, 8, 512, 512), (s1, 8, 512, 512), (s2, 8, 512, 1024), (s1, 8, 512, 512),
              (s1, 4, 1024, 1024), (s1, 4, 1024, 4096), (t2, 4, 1024, 512), (s1, 8, 512, 512), (t2, 8, 512, 256),
              (k1, 8, 512, 144), (s1, 16, 256, 256), (t2, 16, 256, 128), (k1, 16, 256, 144), (s1, 32, 128, 128),
              (k1, 32, 128, 144)]
    macs = sum(K._conv_flops(g, nb, hw, hw, c, co) / 2 for g, hw, c, co in slices)
    assert stats.compute()["spikes/dense_macs"] == macs


def test_resized_skips_are_not_counted_at_480x640(net):
    from snn_object_detectionddp_b200.spikes import SpikeStats
    B, T = 1, 2
    frames, _ = _frames(B, T, 480, 640, seed=3)
    stats = SpikeStats(net)
    net.eval()
    rec = {}
    net.spike_stats = stats
    try:
        with torch.no_grad():
            net.forward_sequence(frames, record=rec)
    finally:
        net.spike_stats = None
    table = dict(TABLE_256, enc1=576, enc2=1152, enc3=2304)
    assert stats.fanout == table
    res = stats.compute()
    s, n = _record_counts(rec, stats.layers, T)
    assert torch.equal(torch.from_numpy(res["spike_counts"]), s)
    assert res["spikes/synops"] == sum(table[name] * int(s[i].sum()) for i, name in enumerate(stats.layers))
    assert res["spikes/dense_macs"] == sum(table[name] * int(n[i]) * T for i, name in enumerate(stats.layers))


def test_train_mode_losses_bit_equal_with_and_without_stats():
    from snn_object_detectionddp_b200.spikes import SpikeStats
    from snn_object_detectionddp_b200.trainer import Trainer
    B, T = 2, 4
    with _deterministic():
        a = Trainer(_product("lif", seed=5), total_steps=10, device=DEV)
        b = Trainer(_product("lif", seed=5), total_steps=10, device=DEV)
        _sync_state(a, b)
        stats = SpikeStats(b.model)
        b.model.spike_stats = stats
        for step in range(2):
            frames, labels = _frames(B, T, 256, 256, seed=10 + step)
            batch = {"padded": tuple(t.to(DEV) for t in a.prepare_batch(labels, B, max_boxes=8)["padded"])}
            _, ia = a.train_step(frames, batch)
            _, ib = b.train_step(frames, batch)
            assert torch.equal(ia, ib), (step, ia, ib)
        b.model.spike_stats = None
    res = stats.compute()
    assert int(res["neuron_steps"].sum()) == 2 * 933888 * B * T and 0 < res["spikes/rate"] < 1


# ------------------------------------------------------------------------------------------------------------------
# 4./5. graphs, no host synchronisation
# ------------------------------------------------------------------------------------------------------------------
def test_graphed_window_replays_count_like_eager_calls(net):
    from snn_object_detectionddp_b200.infer import GraphedWindowDetector, detect_sequence
    from snn_object_detectionddp_b200.spikes import SpikeStats
    frames, _ = _frames(2, 3, 128, 128, seed=4)
    stats = SpikeStats(net)
    net.spike_stats = stats
    try:
        with _deterministic():
            detect_sequence(net, frames, padded=True)
            one = stats.counts.clone()
            stats.reset()
            det = GraphedWindowDetector(net)
            n = 4
            for i in range(n):
                if i == 1:
                    torch.cuda.synchronize()
                    torch.cuda.set_sync_debug_mode("error")        # replays and reset() never read the device
                det(frames)
            stats.reset()
            det(frames)
            torch.cuda.set_sync_debug_mode(0)
            assert torch.equal(stats.counts, one)
            stats.reset()
            for _ in range(n):
                det(frames)
    finally:
        torch.cuda.set_sync_debug_mode(0)
        net.spike_stats = None
    assert int(one.sum()) > 0 and torch.equal(stats.counts, n * one)


def test_graphed_training_counts_equal_eager_counts_and_attach_detach():
    from snn_object_detectionddp_b200.spikes import SpikeStats
    from snn_object_detectionddp_b200.trainer import Trainer
    B, T = 2, 4
    with _deterministic():
        a = Trainer(_product("lif", seed=7), total_steps=20, device=DEV)
        b = Trainer(_product("lif", seed=7), total_steps=20, device=DEV)
        _sync_state(a, b)
        sa, sb = SpikeStats(a.model), SpikeStats(b.model)
        a.model.spike_stats, b.model.spike_stats = sa, sb
        steps = []
        for i in range(5):
            frames, labels = _frames(B, T, 256, 256, seed=30 + i)
            steps.append((frames, {"padded": tuple(t.to(DEV) for t in a.prepare_batch(labels, B, max_boxes=8)["padded"])}))
        for frames, batch in steps:
            a.train_step(frames, batch)
            b.train_step_graphed(frames, batch)
        assert b._graph is not None
        assert int(sa.counts.sum()) > 0 and torch.equal(sa.counts, sb.counts)
        # replays with stats attached, and reset(), never read the device
        torch.cuda.synchronize()
        torch.cuda.set_sync_debug_mode("error")
        try:
            sb.reset()
            b.train_step_graphed(*steps[0])
        finally:
            torch.cuda.set_sync_debug_mode(0)
        assert int(sb.counts[:, 1].sum()) == 933888 * B * T
        # detach: the next calls re-capture without counting and leave the counts untouched
        b.model.spike_stats = None
        before = sb.counts.clone()
        g_counted = b._graph
        for frames, batch in steps[:3]:
            b.train_step_graphed(frames, batch)
        assert b._graph is not g_counted and torch.equal(sb.counts, before)
        # attach after a capture: re-capture, the counts grow again
        g_plain = b._graph
        sb.reset()
        b.model.spike_stats = sb
        for frames, batch in steps[:3]:
            b.train_step_graphed(frames, batch)
        assert b._graph is not g_plain and int(sb.counts[:, 1].sum()) == 3 * 933888 * B * T and int(sb.counts[:, 0].sum()) > 0
        b.model.spike_stats = a.model.spike_stats = None


# ------------------------------------------------------------------------------------------------------------------
# 6. errors
# ------------------------------------------------------------------------------------------------------------------
def test_errors_raise_before_any_launch(net):
    from snn_object_detectionddp_b200 import _lib
    from snn_object_detectionddp_b200.spikes import SpikeStats
    with pytest.raises(ValueError, match="LIF"):
        SpikeStats(_product("silu", seed=1))
    stats = SpikeStats(net, max_T=2)
    net.spike_stats = stats
    try:
        frames, _ = _frames(1, 3, 128, 128, seed=5)
        n0 = _lib.launch_count
        with pytest.raises(ValueError, match="T=3"), torch.no_grad():
            net.forward_sequence(frames)
        assert _lib.launch_count == n0
        with torch.no_grad():
            net.forward_sequence(frames[:, :2])
            before = stats.counts.clone()
            n0 = _lib.launch_count
            with pytest.raises(ValueError, match="fan-out"):
                net.forward_sequence(_frames(1, 2, 480, 640, seed=6)[0])
        assert _lib.launch_count == n0 and torch.equal(stats.counts, before)
    finally:
        net.spike_stats = None


# ------------------------------------------------------------------------------------------------------------------
# 7. entry points
# ------------------------------------------------------------------------------------------------------------------
def test_evaluate_model_with_spike_stats():
    from snn_object_detectionddp_b200.data import synthetic_batch
    from snn_object_detectionddp_b200.train import evaluate_model
    small = _small(seed=25)
    loader = [synthetic_batch(4, 3, 128, 128, seed=60 + i) for i in range(2)]
    with _deterministic():
        plain = evaluate_model(small, loader, DEV)
        counted = evaluate_model(small, loader, DEV, spike_stats=True)
    assert small.spike_stats is None
    assert {k for k in counted if not k.startswith("spikes/")} == set(plain)
    for k in plain:
        v0, v1 = plain[k], counted[k]
        assert (v0 == v1).all() if hasattr(v0, "shape") else v0 == v1, k
    spk = {k for k in counted if k.startswith("spikes/")}
    assert {"spikes/rate", "spikes/synops", "spikes/dense_macs", "spikes/synops_fraction"} <= spk
    assert len([k for k in spk if k.startswith("spikes/rate/")]) == 16
    assert 0 < counted["spikes/rate"] < 1


class _Writer:
    def __init__(self):
        self.scalars, self.groups = [], []

    def add_scalar(self, tag, value, step):
        self.scalars.append((tag, float(value), step))

    def add_scalars(self, tag, values, step):
        self.groups.append((tag, dict(values), step))


def test_train_loop_logs_spike_tags_every_epoch(tmp_path):
    from snn_object_detectionddp_b200.data import synthetic_batch
    from snn_object_detectionddp_b200.train import train_loop
    small = _small(seed=27)
    train = [synthetic_batch(2, 3, 128, 128, seed=80 + i) for i in range(2)]
    val = [synthetic_batch(4, 3, 128, 128, seed=90 + i) for i in range(2)]
    config = {"training": {"epochs": 2, "learning_rate": 1e-4, "weight_decay": 5e-4}, "dataset": {"train": {"seq_len": 3}}}
    w = _Writer()
    train_loop(small, train, val, config, DEV, tmp_path, writer=w, log_every=10, graphed=True, max_boxes=8, spike_stats=True)
    assert small.spike_stats is None
    tags = ("Spikes/train_rate", "Spikes/train_synops_fraction", "Spikes/val_rate", "Spikes/val_synops_fraction")
    logged = [(t, v, e) for t, v, e in w.scalars if t.startswith("Spikes/")]
    assert sorted((t, e) for t, _, e in logged) == sorted((t, e) for t in tags for e in (0, 1))
    assert all(0.0 <= v <= 1.0 for _, v, _ in logged)
    assert all(v > 0.0 for t, v, _ in logged if t.startswith("Spikes/train"))
    groups = [(t, v, e) for t, v, e in w.groups if t == "Spikes_Val_Rate"]
    assert [e for _, _, e in groups] == [0, 1] and all(len(v) == 16 for _, v, _ in groups)
    assert all(0.0 <= r <= 1.0 for _, v, _ in groups for r in v.values())


def test_off_path_launch_sequence_is_unchanged():
    from snn_object_detectionddp_b200 import _lib
    from snn_object_detectionddp_b200.spikes import SpikeStats
    from snn_object_detectionddp_b200.trainer import Trainer
    B, T = 2, 2
    tr = Trainer(_product("lif", seed=9), total_steps=10, device=DEV)
    frames, labels = _frames(B, T, 128, 128, seed=40)
    batch = {"padded": tuple(t.to(DEV) for t in tr.prepare_batch(labels, B, max_boxes=8)["padded"])}
    tr.train_step(frames, batch)

    def traced():
        _lib.trace = []
        try:
            tr.train_step(frames, batch)
        finally:
            seq, _lib.trace = _lib.trace, None
        return seq

    plain = traced()
    stats = SpikeStats(tr.model)                      # exists, not attached
    unattached = traced()
    assert plain == unattached
    assert not any(name == "snn_bn_act_fwd_count" for name, _ in plain)
    tr.model.spike_stats = stats
    try:
        counted = traced()
    finally:
        tr.model.spike_stats = None
    # attached: the 16 LIF launches become the counting entry point with the same declared bytes, nothing else changes
    assert sum(name == "snn_bn_act_fwd_count" for name, _ in counted) == 16
    assert [("snn_bn_act_fwd" if n == "snn_bn_act_fwd_count" else n, w) for n, w in counted] == plain


# ------------------------------------------------------------------------------------------------------------------
# 7. compute(process_group) over NCCL
# ------------------------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _synthetic_counts(rank, L, max_T):
    g = torch.Generator().manual_seed(100 + rank)
    steps = torch.randint(1 << 20, 1 << 40, (L, 1), generator=g) * torch.ones(1, 3, dtype=torch.int64)
    spikes = torch.randint(0, 1 << 19, (L, 3), generator=g)
    buf = torch.zeros(L, 2, max_T, dtype=torch.int64)
    buf[:, 0, :3], buf[:, 1, :3] = spikes, steps
    return buf


def _small_unet_model(dev):
    from types import SimpleNamespace
    from snn_object_detectionddp_b200.model import TemporalUNet
    return SimpleNamespace(temporal_unet=TemporalUNet([144, 144, 144], neuron="lif", widths=(64, 128, 256, 512)).to(dev))


def _ddp_worker(rank, world, port, out):
    import torch.distributed as dist
    from snn_object_detectionddp_b200.spikes import SpikeStats
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    st = SpikeStats(_small_unet_model(dev), max_T=4)
    st.fanout = dict(TABLE_256)
    st.counts.copy_(_synthetic_counts(rank, len(st.layers), 4))
    res = st.compute(dist.group.WORLD)
    out.put((rank, {k: v for k, v in res.items() if k.startswith("spikes/")}, res["spike_counts"], res["neuron_steps"]))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [1, 2])
def test_compute_over_nccl_sums_the_ranks(world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    import time
    import torch.multiprocessing as mp
    from snn_object_detectionddp_b200.spikes import SpikeStats
    ctx = mp.get_context("spawn")
    q = ctx.SimpleQueue()
    port = _free_port()
    procs = [ctx.Process(target=_ddp_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    got, t0 = {}, time.time()
    try:
        while len(got) < world:
            if not q.empty():
                r, *res = q.get()
                got[r] = res
                continue
            if any(p.exitcode not in (None, 0) for p in procs) or time.time() - t0 > 300:
                raise AssertionError(f"worker failed or timed out: exit codes {[p.exitcode for p in procs]}")
            time.sleep(0.2)
        for p in procs:
            p.join(60)
            assert p.exitcode == 0
    finally:
        for p in procs:
            if p.is_alive():
                p.kill()
                p.join()
    local = SpikeStats(_small_unet_model(DEV), max_T=4)
    local.fanout = dict(TABLE_256)
    ref = local.results(sum(_synthetic_counts(r, len(local.layers), 4) for r in range(world)).numpy())
    for r in range(world):
        scal, sc, ns = got[r]
        assert scal == {k: v for k, v in ref.items() if k.startswith("spikes/")}
        assert (sc == ref["spike_counts"]).all() and (ns == ref["neuron_steps"]).all()
