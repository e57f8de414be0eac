"""CPU: host-side logic of the product that needs no GPU -- OneCycle/AdamW hyper-parameter table vs torch's own
scheduler, label padding, the dense (synchronisation-free) task-aligned assigner vs the restated ultralytics
assigner, the synthetic-batch generator, and bucketed gradient all-reduce over gloo with world_size 2."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import detect_oracle as D
from oracle import model_oracle as MO


def test_one_cycle_table_matches_torch_scheduler():
    """Reference train.py:156-169: AdamW(default lr) + OneCycleLR(max_lr=1e-4, pct_start .3, cos), beta1 cycled."""
    from snn_object_detectionddp_b200.trainer import one_cycle_table
    for total in (10, 37, 200):
        p = torch.nn.Parameter(torch.zeros(1))
        opt = torch.optim.AdamW([p], weight_decay=5e-4)
        sch = torch.optim.lr_scheduler.OneCycleLR(opt, max_lr=1e-4, total_steps=total, pct_start=0.3, anneal_strategy="cos")
        tab = one_cycle_table(total, 1e-4, 5e-4)
        for k in range(total):
            g = opt.param_groups[0]
            assert abs(g["lr"] - float(tab[k, 0])) <= 1e-12 + 1e-9 * g["lr"], (total, k)
            assert abs(g["betas"][0] - float(tab[k, 1])) <= 1e-12, (total, k)
            assert float(tab[k, 2]) == g["betas"][1] and float(tab[k, 3]) == g["eps"] and float(tab[k, 4]) == g["weight_decay"]
            assert abs(float(tab[k, 5]) - (1 - g["betas"][0] ** (k + 1))) < 1e-12
            p.grad = torch.ones(1)
            opt.step()
            if k + 1 < total:
                sch.step()


def test_pad_targets_layout_and_empty():
    from snn_object_detectionddp_b200.loss import pad_targets
    lab = torch.tensor([[1, 3, .5, .5, .2, .2], [0, 1, .3, .3, .1, .1], [1, 2, .6, .6, .1, .3]])
    cls, box, valid = pad_targets(lab, 3)
    assert cls.shape == (3, 2) and valid.tolist() == [[True, False], [True, True], [False, False]]
    assert cls[1].tolist() == [3, 2] and torch.allclose(box[1, 1], torch.tensor([.6, .6, .1, .3]))
    cls, box, valid = pad_targets(torch.zeros(0, 6), 2)
    assert cls.shape == (2, 1) and not valid.any()


def test_collate_and_synthetic_batch_match_oracle_generator():
    from snn_object_detectionddp_b200.data import custom_collate_fn, synthetic_batch
    f1, l1 = synthetic_batch(3, 2, 64, 64, seed=7)
    f2, l2 = MO.synthetic_batch(3, 2, 64, 64, seed=7)
    assert torch.equal(f1, f2) and torch.equal(l1, l2)
    assert l1.shape[1] == 6 and float(f1.min()) >= 0 and float(f1.max()) < 1
    imgs, labs = custom_collate_fn([(torch.zeros(2, 3, 8, 8), torch.tensor([[1., .5, .5, .1, .1]])),
                                    (torch.zeros(2, 3, 8, 8), torch.zeros(0, 5))])
    assert imgs.shape == (2, 2, 3, 8, 8) and torch.allclose(labs, torch.tensor([[0, 1, .5, .5, .1, .1]]))
    _, labs = custom_collate_fn([(torch.zeros(1, 3, 8, 8), torch.zeros(0, 5))])
    assert labs.shape == (0, 6)


@pytest.mark.parametrize("seed,B,nmax", [(0, 4, 6), (1, 2, 1), (2, 3, 12)])
def test_dense_assigner_matches_restated_ultralytics(seed, B, nmax):
    from snn_object_detectionddp_b200.loss import task_aligned_assign
    g = torch.Generator().manual_seed(seed)
    nc, strides, hw = 8, (8.0, 16.0, 32.0), 128
    maps = [torch.zeros(B, 1, hw // int(s), hw // int(s)) for s in strides]
    anchors, st = D.make_anchors(maps, strides)
    A = anchors.shape[0]
    pd_scores = torch.rand(B, A, nc, generator=g) * 0.5
    ctr = (anchors * st)[None].expand(B, -1, -1)
    half = torch.rand(B, A, 2, generator=g) * 30 + 4
    jit = (torch.rand(B, A, 2, generator=g) - 0.5) * 6
    pd_bboxes = torch.cat((ctr + jit - half, ctr + jit + half), -1)
    n = torch.randint(0, nmax + 1, (B,), generator=g)
    n[0] = nmax
    gt_labels = torch.randint(0, nc, (B, nmax, 1), generator=g).float()
    c = torch.rand(B, nmax, 2, generator=g) * 90 + 19
    wh = torch.rand(B, nmax, 2, generator=g) * 40 + 8
    gt_bboxes = torch.cat((c - wh / 2, c + wh / 2), -1)
    valid = torch.arange(nmax)[None] < n[:, None]
    gt_bboxes = gt_bboxes * valid[..., None]
    gt_labels = gt_labels * valid[..., None]
    mask_gt = gt_bboxes.sum(2, keepdim=True).gt_(0.0)
    ref = D.TaskAlignedAssigner(topk=10, num_classes=nc)(pd_scores, pd_bboxes, anchors * st, gt_labels, gt_bboxes, mask_gt)
    _, r_boxes, r_scores, r_fg, _ = ref
    t_boxes, t_scores, fg = task_aligned_assign(pd_scores, pd_bboxes, anchors * st, gt_labels.squeeze(-1).long(), gt_bboxes,
                                                mask_gt.squeeze(-1).bool(), nc)
    assert torch.equal(fg.bool(), r_fg)
    assert int(r_fg.sum()) > 0
    assert torch.equal(t_scores, r_scores)
    assert torch.equal(t_boxes[r_fg], r_boxes[r_fg])


# ------------------------------------------------------------------------------------------------
# bucketed all-reduce over gloo, world_size 2
# ------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _ddp_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from snn_object_detectionddp_b200.ddp import GradBucketer, broadcast_module_state
    spans = [(0, 24), (24, 8), (32, 104), (136, 16), (152, 8)]
    flat = torch.arange(160, dtype=torch.float32) * (rank + 1)
    bk = GradBucketer(flat, spans, bucket_bytes=64, group=None)
    assert bk.world == 2 and len(bk.buckets) >= 3
    covered = sorted((lo, hi) for lo, hi, _ in bk.buckets)
    assert covered[0][0] == 0 and covered[-1][1] == 160 and all(a[1] == b[0] for a, b in zip(covered, covered[1:]))
    for step in range(2):
        flat.copy_(torch.arange(160, dtype=torch.float32) * (rank + 1) * (step + 1))
        bk.begin_step()
        for i in (4, 3, 2):          # backward order: last tensors first; tensors 0 and 1 never report (no grad)
            bk.entry_ready(i)
        bk.entry_ready(3)            # duplicate notifications are ignored
        bk.finish()
        expect = torch.arange(160, dtype=torch.float32) * 1.5 * (step + 1)       # mean over ranks of (rank+1)
        assert torch.allclose(flat, expect), (rank, step)
        assert bk.launch_order[0] == bk.bucket_of[4]
    lin = torch.nn.Linear(4, 4)
    torch.manual_seed(rank)
    with torch.no_grad():
        lin.weight.normal_()
    broadcast_module_state(lin)
    ws = [torch.zeros_like(lin.weight) for _ in range(world)]
    dist.all_gather(ws, lin.weight.data)
    assert torch.equal(ws[0], ws[1])
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        q.put("ok")


def test_grad_bucketer_gloo_world2():
    ctx = mp.get_context("spawn")
    q = ctx.SimpleQueue()
    port = _free_port()
    procs = [ctx.Process(target=_ddp_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    assert q.get() == "ok"


# ------------------------------------------------------------------------------------------------
# round 2: metrics, sampler, split, extractor adapter, multi-use gradient readiness
# ------------------------------------------------------------------------------------------------
class _Writer:
    def __init__(self):
        self.scalar, self.scalars = [], []

    def add_scalar(self, tag, value, step):
        self.scalar.append((tag, float(value), int(step)))

    def add_scalars(self, tag, d, step):
        self.scalars.append((tag, {k: float(v) for k, v in d.items()}, int(step)))


def test_device_metrics_emit_reference_tensorboard_tags_with_one_sync_per_n_steps():
    """reference train.py:81-100: per-batch tags and values; here the values are read back once per `every` steps."""
    from snn_object_detectionddp_b200.train import DeviceMetrics, _log_batches
    m, w = DeviceMetrics("cpu", every=3), _Writer()
    rows = [torch.tensor([1.0, 2.0, 3.0]) * (i + 1) for i in range(7)]
    flushes = 0
    for i, it in enumerate(rows):
        if m.update(it, 100 + i, lr=0.01 * i, scale=4.0):
            _log_batches(w, m.flush(), True)
            flushes += 1
    _log_batches(w, m.flush(), True)
    assert flushes == 2
    assert [s for s in w.scalar if s[0] == "Loss/train_batch"] == [("Loss/train_batch", 4.0 * 6.0 * (i + 1), 100 + i) for i in range(7)]
    assert [round(s[1], 6) for s in w.scalar if s[0] == "LearningRate/batch"] == [round(0.01 * i, 6) for i in range(7)]
    assert w.scalars[2] == ("Train_Loss_Components_Batch", {"box_loss_batch": 3.0, "cls_loss_batch": 6.0, "dfl_loss_batch": 9.0}, 102)
    avg, comps = m.averages(7)
    assert abs(avg - 4.0 * 6.0 * 4.0) < 1e-5 and torch.allclose(comps, torch.tensor([4.0, 8.0, 12.0]))
    wv = _Writer()
    _log_batches(wv, [(5, torch.tensor([1.0, 1.0, 1.0]), 0.0, 3.0)], False)
    assert wv.scalar == [("Loss/val_batch", 3.0, 5)] and wv.scalars[0][0] == "Val_Loss_Components_Batch"


def test_sharded_sampler_partitions_like_distributed_sampler():
    from snn_object_detectionddp_b200.train import ShardedSampler
    data = list(range(103))
    for world in (1, 2, 8):
        for drop_last in (False, True):
            per_rank = []
            for r in range(world):
                s = ShardedSampler(data, rank=r, world_size=world, shuffle=True, seed=7, drop_last=drop_last)
                s.set_epoch(3)
                idx = list(s)
                assert len(idx) == len(s)
                per_rank.append(idx)
            assert len({len(p) for p in per_rank}) == 1                       # equal work on every rank
            allidx = [i for p in per_rank for i in p]
            if drop_last:
                assert len(set(allidx)) == len(allidx) == (103 // world) * world
            else:
                assert set(allidx) == set(data) and len(allidx) - 103 < world   # padded by wrap-around only
    a = ShardedSampler(data, 0, 2, seed=7); b = ShardedSampler(data, 0, 2, seed=7)
    a.set_epoch(0); b.set_epoch(1)
    assert list(a) != list(b)                                                  # reshuffled every epoch
    b.set_epoch(0)
    assert list(a) == list(b)                                                  # same permutation on every process
    ref = torch.utils.data.distributed.DistributedSampler(data, num_replicas=2, rank=1, shuffle=False)
    assert list(ShardedSampler(data, 1, 2, shuffle=False)) == list(ref)


def test_sequence_grouped_split_keeps_recordings_apart():
    """reference main.py:16-27: a recording sequence (image directory) lands entirely in train or in validation."""
    from snn_object_detectionddp_b200.train import get_train_val_split

    class DS:
        samples = [(f"/d/seq{ i // 7 }", i, None) for i in range(70)]

        def __len__(self):
            return 70

        def __getitem__(self, i):
            return i

    tr, va = get_train_val_split({}, DS())
    dirs = lambda sub: {DS.samples[i][0] for i in sub.indices}
    assert not (dirs(tr) & dirs(va)) and len(dirs(tr)) == 8 and len(dirs(va)) == 2
    assert sorted(tr.indices + va.indices) == list(range(70))
    tr2, va2 = get_train_val_split({}, DS())
    assert tr2.indices == tr.indices                                           # random_state=42: the reference's split


def test_extractor_uses_real_ultralytics_when_importable(monkeypatch):
    """reference model.py:74-98: YOLO(model_name).model, frozen, always eval, `_, features = model(x)`.  ultralytics is
    not installable here, so a module with the same surface is injected; without it the stand-in pyramid is used."""
    import sys
    import types
    import snn_object_detectionddp_b200.model as M
    assert M.YOLOFeatureExtractor(backend="auto").backend == "standin"
    with pytest.raises(RuntimeError):
        M.YOLOFeatureExtractor(backend="ultralytics")

    class Net(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.c3, self.c4, self.c5 = (torch.nn.Conv2d(3, c, 1, stride=s) for c, s in ((16, 8), (24, 16), (32, 32)))

        def forward(self, x):
            return None, [self.c3(x), self.c4(x), self.c5(x)]

    seen = {}

    class YOLO:
        def __init__(self, name):
            seen["name"] = name
            self.model = Net()

    fake = types.ModuleType("ultralytics")
    fake.YOLO = YOLO
    monkeypatch.setitem(sys.modules, "ultralytics", fake)
    ext = M.YOLOFeatureExtractor("yolo11m.pt")
    assert ext.backend == "ultralytics" and seen["name"] == "yolo11m.pt"
    assert all(not p.requires_grad for p in ext.parameters())
    ext.train()
    assert not ext.model.training                                              # stays in eval (model.py:84-86)
    assert ext.get_feature_channels((1, 3, 64, 64)) == [16, 24, 32]
    f = ext(torch.rand(2, 3, 64, 64))
    assert [tuple(t.shape) for t in f] == [(2, 16, 8, 8), (2, 24, 4, 4), (2, 32, 2, 2)]
    assert any(k.startswith("model.c3") for k in ext.state_dict())            # reference key names: feature_extractor.model.*


def test_gradient_readiness_counts_every_use_of_a_parameter():
    """The reference-style per-frame loop uses each parameter T times: its DDP bucket may be reduced only after the LAST
    backward of those uses (round-1 finding: it was launched after the first)."""
    from snn_object_detectionddp_b200.params import ParamStore
    lin = torch.nn.Conv2d(8, 8, 3, bias=True)
    st = ParamStore(lin)
    ready = []
    st.grad_ready_hook = lambda e: ready.append(e.name)
    for _ in range(3):
        st.note_use(lin.weight, lin.bias)
    st.grad_done(lin.weight); st.grad_done(lin.weight)
    assert ready == []
    st.grad_done(lin.weight)
    assert ready == ["weight"]
    st.grad_done(lin.bias); st.grad_done(lin.bias); st.grad_done(lin.bias)
    assert ready == ["weight", "bias"]
    st.grad_done(lin.bias)                       # a use that was never announced (no_grad forward): fires immediately
    assert ready[-1] == "bias"


def test_bench_comm_overlap_accounting():
    """bench.comm_overlap: exposed communication = NCCL-resident time that no compute kernel overlaps."""
    import bench

    class _TR:
        def __init__(self, a, b):
            self.start, self.end = a, b

    class _EV:
        def __init__(self, n, a, b):
            self.name, self.time_range = n, _TR(a, b)

    evs = [_EV("snn::a", 0, 100), _EV("snn::b", 150, 200), _EV("ncclDevKernel_AllReduce_Sum_f32", 50, 180),
           _EV("ncclDevKernel_AllReduce_Sum_f32", 300, 320)]
    c = bench.comm_overlap(evs, 2)
    assert c["exposed_comm_ms_per_step"] == pytest.approx(0.035) and c["nccl_resident_ms_per_step"] == pytest.approx(0.075)
    assert c["nccl_kernels"]["ncclDevKernel_AllReduce_Sum_f32"]["launches_per_step"] == 1.0
    assert bench.comm_overlap(evs[:2], 1) is None


@pytest.mark.parametrize("record", ["bench_final_default_n1.json", "bench_final_strip_n8.json"])
def test_bench_result_line_stays_compact(record):
    """bench.result_line on full records of this benchmark (one GPU: 21 KB with the 18-row LIF sweep and 40 shapes; eight
    GPUs: 11.6 KB with the NCCL timeline): one strict-JSON line below RESULT_LINE_MAX that keeps the headline, the
    roofline, the per-kernel table and the baselines."""
    import json
    import bench
    path = os.path.join(bench.ROOT, "profiles", "r2", record)
    rec = json.loads(open(path).read().strip().splitlines()[-1])
    assert len(json.dumps(rec)) > bench.RESULT_LINE_MAX
    line = bench.result_line(rec)
    assert len(line.encode()) < bench.RESULT_LINE_MAX and "\n" not in line
    d = json.loads(line)
    assert d["value"] == pytest.approx(rec["value"], rel=1e-5) and d["steps"] == rec["steps"] and d["n_gpus"] == rec["n_gpus"]
    assert d["roofline"]["kernel"] == rec["roofline"]["kernel"] and set(d["kernels"]) == set(rec["kernels"])
    assert d["kernels_by_shape"] == rec["kernels_by_shape"][:8]
    assert (d["comm_timeline"] is None) == (rec["comm_timeline"] is None)
    if rec["lif_microbench"]:
        assert d["cpu_baseline"]["cores"] == rec["cpu_baseline"]["cores"]
        assert d["lif_microbench"]["fwd_frac_min"] == pytest.approx(rec["lif_microbench"]["fwd_frac_min"], rel=1e-5)


def test_bench_dump_outputs(tmp_path):
    """bench.dump_outputs: float32 .npy files of the step's results; the parameters in declaration order, or a sample at
    seeded positions (the same in every run) once there are more than DUMP_PARAM_SAMPLES of them."""
    import numpy as np
    import bench
    torch.manual_seed(0)
    m = torch.nn.Sequential(torch.nn.Linear(64, 32), torch.nn.Linear(32, 3))
    flat = torch.cat([p.detach().reshape(-1) for p in m.parameters()]).numpy()
    args = (torch.arange(3.0), torch.ones(3), torch.tensor([2.5]), m)
    bench.dump_outputs(str(tmp_path / "all"), *args)
    assert sorted(os.listdir(tmp_path / "all")) == ["grad_norm.npy", "loss.npy", "loss_items.npy", "params_sample.npy"]
    for f in os.listdir(tmp_path / "all"):
        assert np.load(tmp_path / "all" / f).dtype == np.float32
    assert np.array_equal(np.load(tmp_path / "all" / "params_sample.npy"), flat)
    assert np.array_equal(np.load(tmp_path / "all" / "loss.npy"), [0.0, 1.0, 2.0])
    old = bench.DUMP_PARAM_SAMPLES
    try:
        bench.DUMP_PARAM_SAMPLES = 500
        bench.dump_outputs(str(tmp_path / "s1"), *args)
        bench.dump_outputs(str(tmp_path / "s2"), *args)
    finally:
        bench.DUMP_PARAM_SAMPLES = old
    s1, s2 = np.load(tmp_path / "s1" / "params_sample.npy"), np.load(tmp_path / "s2" / "params_sample.npy")
    assert s1.shape == (500,) and np.array_equal(s1, s2) and np.isin(s1, flat).all()
