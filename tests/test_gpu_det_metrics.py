"""-m gpu: detection metrics (csrc/metrics.cu, snn_object_detectionddp_b200/metrics.py) vs the CPU specification
oracle/det_metrics_oracle.py -- TP masks and gt counts bit-exact, metrics within 1e-9 -- and the evaluation / validation
entry points built on them."""
import os
import socket

import numpy as np
import pytest
import torch

from oracle import det_metrics_oracle as S

pytestmark = pytest.mark.gpu
DEV = "cuda"
MAX_DET = 300


def _batch(B, nc, M, seed, H=96, W=128, empty=True):
    """Synthetic NMS output + padded targets: jittered copies of the gts (some exact duplicates, some with the wrong class),
    clutter, boxes on a coarse pixel grid (exact IoU ties), an image without detections and one without gts."""
    g = torch.Generator().manual_seed(seed)
    n_gt = torch.randint(0, M + 1, (B,), generator=g)
    gt_valid = torch.arange(M)[None, :] < n_gt[:, None]
    gt_cls = torch.randint(0, nc, (B, M), generator=g) * gt_valid
    cxcy = torch.rand(B, M, 2, generator=g) * 0.8 + 0.1
    wh = torch.rand(B, M, 2, generator=g) * 0.3 + 0.05
    gt_box = torch.cat((cxcy, wh), 2) * gt_valid[..., None]
    rows = torch.zeros(B, MAX_DET, 6)
    counts = torch.zeros(B, dtype=torch.int32)
    scale = torch.tensor([W, H, W, H], dtype=torch.float32)
    for b in range(B):
        n = int(torch.randint(0, MAX_DET + 1, (1,), generator=g))
        if empty and B > 1 and b == B - 1:
            n = 0
        if empty and B > 2 and b == B - 2:
            gt_valid[b] = False
        k = int(n_gt[b])
        src = torch.randint(0, max(k, 1), (n,), generator=g)
        gx = torch.cat((gt_box[b, :, :2] - gt_box[b, :, 2:] / 2, gt_box[b, :, :2] + gt_box[b, :, 2:] / 2), 1) * scale
        box = gx[src] + torch.randn(n, 4, generator=g) * 4 * (torch.rand(n, 1, generator=g) < 0.7)
        box = box.round()                                                      # integer pixels: exact IoU ties
        clutter = torch.rand(n, generator=g) < (0.3 if k else 1.0)
        rnd = torch.rand(n, 2, generator=g) * torch.tensor([W, H]) * 0.8
        box[clutter] = torch.cat((rnd, rnd + 5 + torch.rand(n, 2, generator=g) * 30), 1)[clutter].round()
        box[:, 2:] = torch.maximum(box[:, 2:], box[:, :2] + 1)
        cls = gt_cls[b][src].clone() if k else torch.zeros(n, dtype=torch.long)
        wrong = torch.rand(n, generator=g) < 0.15
        cls[wrong] = torch.randint(0, nc, (int(wrong.sum()),), generator=g)
        cls[clutter] = torch.randint(0, nc, (int(clutter.sum()),), generator=g)
        conf = (torch.rand(n, generator=g) * 16).floor() / 16 + 0.001            # many equal confidences
        conf, order = torch.sort(conf, descending=True, stable=True)
        rows[b, :n, :4], rows[b, :n, 4], rows[b, :n, 5] = box[order], conf, cls[order].float()
        counts[b] = n
    return rows, counts, (gt_cls, gt_box, gt_valid), (H, W)


def _spec_update(spec, rows, counts, padded, hw):
    spec.update(rows.numpy(), counts.numpy(), padded[0].numpy(), padded[1].numpy(), padded[2].numpy(), hw[1], hw[0])


def _dev(rows, counts, padded):
    return rows.to(DEV), counts.to(DEV), tuple(t.to(DEV) for t in padded)


def _check_results(ours, ref, tol=1e-9):
    for k in S.KEYS:
        assert abs(ours[k] - ref[k]) <= tol, (k, ours[k], ref[k])
    assert list(ours["ap_class_index"]) == list(ref["ap_class_index"])
    np.testing.assert_allclose(ours["ap"], ref["ap"], atol=tol, rtol=0)


@pytest.mark.parametrize("B,nc,M", [(1, 1, 4), (7, 8, 16), (64, 8, 32), (7, 80, 64), (64, 1, 64)])
def test_match_bit_exact_vs_spec(B, nc, M):
    from snn_object_detectionddp_b200.metrics import DetMetrics
    rows, counts, padded, hw = _batch(B, nc, M, seed=B * 100 + nc + M)
    m = DetMetrics(nc, DEV)
    m.update(*_dev(rows, counts, padded), hw)
    conf, cls, tp = (t.cpu().numpy() for t in m.records())
    r_conf, r_cls, r_tp, r_tcls = S.batch_records(rows.numpy(), counts.numpy(), *(t.numpy() for t in padded), hw[1], hw[0])
    assert conf.shape[0] == int(counts.sum()) == r_conf.shape[0]
    np.testing.assert_array_equal(conf, r_conf)
    np.testing.assert_array_equal(cls, r_cls)
    np.testing.assert_array_equal(tp, r_tp)
    assert tp.any() and not tp.all()
    np.testing.assert_array_equal(m.n_gt.cpu().numpy(), np.bincount(r_tcls, minlength=nc))
    _check_results(m.compute(), S.results_dict(r_tp, r_conf, r_cls, r_tcls))


def test_records_are_deterministic_across_batches_and_growth():
    from snn_object_detectionddp_b200.metrics import DetMetrics
    m = DetMetrics(8, DEV, capacity=500)                  # grows during the second batch
    spec = S.SpecMetrics()
    for seed in range(4):
        rows, counts, padded, hw = _batch(7, 8, 16, seed=10 + seed)
        m.update(*_dev(rows, counts, padded), hw)
        _spec_update(spec, rows, counts, padded, hw)
    assert m._cap > 500
    conf, cls, tp = (t.cpu().numpy() for t in m.records())
    np.testing.assert_array_equal(conf, np.concatenate(spec.conf))
    np.testing.assert_array_equal(cls, np.concatenate(spec.cls))
    np.testing.assert_array_equal(tp, np.concatenate(spec.tp))
    _check_results(m.compute(), spec.compute())
    m.reset()
    rows, counts, padded, hw = _batch(7, 8, 16, seed=10)
    m.update(*_dev(rows, counts, padded), hw)
    assert m.records()[0].shape[0] == int(counts.sum())


@pytest.mark.parametrize("nc", [1, 8])
def test_finalize_vs_spec_on_a_million_records(nc):
    """>= 1 M records; with nc = 1 the class segment is > 2000 chunks of the per-class CTA."""
    from snn_object_detectionddp_b200.metrics import DetMetrics
    m = DetMetrics(nc, DEV)
    g = torch.Generator(device=DEV).manual_seed(nc)
    B, M = 64, 32
    for it in range(55):
        rows = torch.zeros(B, MAX_DET, 6, device=DEV)
        xy = torch.rand(B, MAX_DET, 2, device=DEV, generator=g) * 100
        rows[..., :2], rows[..., 2:4] = xy, xy + 4 + torch.rand(B, MAX_DET, 2, device=DEV, generator=g) * 20
        rows[..., 4] = (torch.rand(B, MAX_DET, device=DEV, generator=g) * 4096).floor() / 4096 + 0.001
        rows[..., 5] = torch.randint(0, nc, (B, MAX_DET), device=DEV, generator=g).float()
        counts = torch.full((B,), MAX_DET, device=DEV, dtype=torch.int32)
        gt_cls = torch.randint(0, nc, (B, M), device=DEV, generator=g)
        gt_box = torch.cat((torch.rand(B, M, 2, device=DEV, generator=g) * 0.8 + 0.1,
                            torch.rand(B, M, 2, device=DEV, generator=g) * 0.2 + 0.02), 2)
        hit = torch.cat((gt_box[..., :2] - gt_box[..., 2:] / 2, gt_box[..., :2] + gt_box[..., 2:] / 2), 2) * 128
        rows[:, :M, :4] = hit + torch.randn(B, M, 4, device=DEV, generator=g)   # every gt also detected, roughly
        rows[:, :M, 5] = gt_cls.float()
        m.update(rows, counts, (gt_cls, gt_box, torch.ones(B, M, device=DEV, dtype=torch.bool)), (128, 128))
    conf, cls, tp = (t.cpu().numpy() for t in m.records())
    assert conf.shape[0] >= 1 << 20 and tp[:, 0].sum() > 10000 and not tp[:, 9].all()
    tcls = np.repeat(np.arange(nc), m.n_gt.cpu().numpy())
    _check_results(m.compute(), S.results_dict(tp, conf, cls, tcls))


def test_update_does_not_synchronise():
    from snn_object_detectionddp_b200.metrics import DetMetrics
    m = DetMetrics(8, DEV, capacity=256)
    batches = [_dev(*_batch(7, 8, 16, seed=s)[:3]) for s in range(3)]
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for rows, counts, padded in batches:
            m.update(rows, counts, padded, (96, 128))      # grows at the second batch: still no host read
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert m.records()[0].shape[0] == sum(int(b[1].sum()) for b in batches)


def test_out_of_range_gt_class_raises():
    from snn_object_detectionddp_b200.metrics import DetMetrics
    rows, counts, (gc, gb, gv), hw = _batch(3, 4, 8, seed=5)
    gc[0, 0], gv[0, 0] = 4, True
    m = DetMetrics(4, DEV)
    m.update(*_dev(rows, counts, (gc, gb, gv)), hw)
    with pytest.raises(ValueError, match="outside"):
        m.compute()


def test_evaluate_model_equals_spec_on_product_nms_rows():
    from snn_object_detectionddp_b200.data import synthetic_batch
    from snn_object_detectionddp_b200.infer import detect_sequence
    from snn_object_detectionddp_b200.loss import pad_targets
    from snn_object_detectionddp_b200.train import evaluate_model
    from tests.test_gpu_infer import _models
    from tests.gpu_util import setup_exact
    setup_exact()
    _, net = _models(seed=25)
    loader = [synthetic_batch(4, 3, 128, 128, seed=60 + i) for i in range(3)] + [synthetic_batch(2, 3, 128, 128, seed=63)]
    ours = evaluate_model(net, loader, DEV)
    spec, n_rec = S.SpecMetrics(), 0
    for frames, labels in loader:
        rows, _, counts = detect_sequence(net, frames.to(DEV), conf_thres=0.001, iou_thres=0.6, multi_label=False, padded=True)
        padded = pad_targets(labels, frames.shape[0])
        _spec_update(spec, rows.cpu(), counts.cpu(), padded, (128, 128))
        n_rec += int(counts.sum())
    assert n_rec > 0
    _check_results(ours, spec.compute())


def _deterministic():
    """Context: fixed-order loss sums (snn_set_deterministic), so two validation passes compare bit for bit."""
    import contextlib
    from snn_object_detectionddp_b200 import _lib

    @contextlib.contextmanager
    def ctx():
        L = _lib.lib()
        before = L.snn_get_deterministic()
        L.snn_set_deterministic(1)
        try:
            yield
        finally:
            L.snn_set_deterministic(before)
    return ctx()


def test_validate_one_epoch_with_metrics_keeps_the_loss_and_equals_spec():
    """The hooked validation pass returns bit-equal loss averages, and its metric equals the specification applied to the
    NMS rows of the same eval forwards with the batch's padded targets."""
    from snn_object_detectionddp_b200.data import synthetic_batch
    from snn_object_detectionddp_b200.infer import detect_sequence
    from snn_object_detectionddp_b200.loss import pad_targets
    from snn_object_detectionddp_b200.metrics import DetMetrics
    from snn_object_detectionddp_b200.train import validate_one_epoch
    from snn_object_detectionddp_b200.trainer import Trainer
    from tests.test_gpu_infer import _models
    from tests.gpu_util import setup_exact
    setup_exact()
    _, net = _models(seed=26)
    tr = Trainer(net, total_steps=4, device=DEV)
    loader = [synthetic_batch(4, 3, 128, 128, seed=70 + i) for i in range(3)]
    spec, n_rec = S.SpecMetrics(), 0
    with _deterministic():
        plain = validate_one_epoch(tr, loader, max_boxes=8)
        m = DetMetrics(8, DEV)
        hooked = validate_one_epoch(tr, loader, max_boxes=8, metrics=m)
        for frames, labels in loader:
            rows, _, counts = detect_sequence(net, frames.to(DEV), conf_thres=0.001, iou_thres=0.6, multi_label=False,
                                              padded=True)
            _spec_update(spec, rows.cpu(), counts.cpu(), pad_targets(labels, frames.shape[0], max_boxes=8), (128, 128))
            n_rec += int(counts.sum())
    assert plain[0] == hooked[0] and torch.equal(plain[1], hooked[1])
    assert n_rec > 0 and m.records()[0].shape[0] == n_rec
    _check_results(m.compute(), spec.compute())


class _Writer:
    def __init__(self):
        self.scalars = []

    def add_scalar(self, tag, value, step):
        self.scalars.append((tag, float(value), step))

    def add_scalars(self, tag, values, step):
        pass


def test_train_loop_eval_map_logs_the_validation_metric(tmp_path):
    """train_loop(eval_map=True) logs metrics/{precision,recall,mAP50,mAP50-95}(B) once per epoch; the logged values are
    those of a separate hooked validation pass over the final parameters (eval forwards leave the model unchanged)."""
    from snn_object_detectionddp_b200.data import synthetic_batch
    from snn_object_detectionddp_b200.metrics import KEYS, DetMetrics
    from snn_object_detectionddp_b200.train import train_loop, validate_one_epoch
    from tests.test_gpu_infer import _models
    from tests.gpu_util import setup_exact
    setup_exact()
    _, net = _models(seed=27)
    train = [synthetic_batch(2, 3, 128, 128, seed=80 + i) for i in range(2)]
    val = [synthetic_batch(4, 3, 128, 128, seed=90 + i) for i in range(2)]
    config = {"training": {"epochs": 2, "learning_rate": 1e-4, "weight_decay": 5e-4}, "dataset": {"train": {"seq_len": 3}}}
    w = _Writer()
    tr = train_loop(net, train, val, config, DEV, tmp_path, writer=w, log_every=10, eval_map=True)
    logged = [(t, v, e) for t, v, e in w.scalars if t.startswith("metrics/")]
    assert sorted((t, e) for t, _, e in logged) == sorted((t, e) for t in KEYS[:4] for e in (0, 1))
    assert all(0.0 <= v <= 1.0 for _, v, _ in logged)
    m = DetMetrics(8, DEV)
    validate_one_epoch(tr, val, 3, metrics=m)
    res = m.compute()
    for t, v, e in logged:
        if e == 1:
            assert abs(v - res[t]) <= 1e-12, (t, v, res[t])


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _ddp_worker(rank, world, port, out):
    import torch.distributed as dist
    from snn_object_detectionddp_b200.metrics import DetMetrics
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    m = DetMetrics(8, dev, capacity=512)                  # other ranks may hold more records than this capacity
    for s in range(2 + rank):
        rows, counts, padded, hw = _batch(7, 8, 16, seed=200 + 10 * rank + s)
        m.update(rows.to(dev), counts.to(dev), tuple(t.to(dev) for t in padded), hw)
    res = m.compute(dist.group.WORLD)
    out.put((rank, {k: res[k] for k in S.KEYS}, res["ap"]))
    dist.barrier()
    dist.destroy_process_group()


def _run_ranks(world):
    """Spawns one process per rank; polls, so a crashed rank fails the test instead of hanging it, and kills what is left."""
    import time
    import torch.multiprocessing as mp
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
                r, res, ap = q.get()
                got[r] = (res, ap)
                continue
            if any(p.exitcode not in (None, 0) for p in procs) or time.time() - t0 > 300:
                raise AssertionError(f"metric worker failed or timed out: exit codes {[p.exitcode for p in procs]}")
            time.sleep(0.2)
        for p in procs:
            p.join(60)
            assert p.exitcode == 0
    finally:
        for p in procs:
            if p.is_alive():
                p.kill()
                p.join()
    return got


@pytest.mark.parametrize("world", [1, 2])
def test_ddp_compute_equals_spec_over_rank_major_records(world):
    """compute(process_group) over NCCL: every rank gets the specification's result over the rank-major concatenation of
    all ranks' records.  world = 1 runs the whole gather path (collectives included) on one GPU."""
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    got = _run_ranks(world)
    spec = S.SpecMetrics()
    for rank in range(world):
        for s in range(2 + rank):
            rows, counts, padded, hw = _batch(7, 8, 16, seed=200 + 10 * rank + s)
            _spec_update(spec, rows, counts, padded, hw)
    ref = spec.compute()
    for rank in range(1, world):
        assert got[rank][0] == got[0][0] and np.array_equal(got[rank][1], got[0][1])
    for k in S.KEYS:
        assert abs(got[0][0][k] - ref[k]) <= 1e-9, k
    np.testing.assert_allclose(got[0][1], ref["ap"], atol=1e-9, rtol=0)
