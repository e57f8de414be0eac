"""-m gpu: detection-loss kernels, Detect head, and the whole training step vs the oracle (oracle/detect_oracle.py,
oracle/model_oracle.py).  Head / loss / NMS are PARITY UNPINNED (ultralytics restated, SURVEY.md 8c); the oracle is the
specification.  fp32 kernels: rel 1e-4 (sum order, expf/atanf ulps); anything through bf16 convs: see each test."""
import pytest
import torch

from oracle import detect_oracle as D
from oracle import model_oracle as MO
from tests.gpu_util import rel_err, setup_exact

pytestmark = pytest.mark.gpu
DEV = "cuda"
HYP = {"box": 7.5, "cls": 1.0, "dfl": 2.5, "reg_max": 16}


class _FakeModel:
    """The three attributes v8DetectionLoss(model) reads (reference model.py:178-195)."""

    def __init__(self, nc=8):
        from types import SimpleNamespace
        self.args = SimpleNamespace(**HYP)
        head = SimpleNamespace(stride=torch.tensor([8.0, 16.0, 32.0]), nc=nc, reg_max=16)
        self.model = [head]


def _maps(B, hw, nc, seed):
    g = torch.Generator().manual_seed(seed)
    maps = []
    for s in (8, 16, 32):
        m = torch.randn(B, nc + 64, hw // s, hw // s, generator=g)
        m[:, 64:] -= 3.0                      # low prior class logits
        m[:, :64] *= 2.0
        maps.append(m.to(DEV))
    return maps


@pytest.mark.parametrize("B,hw,seed", [(4, 256, 0), (2, 128, 1), (3, 64, 2)])
def test_detection_loss_matches_oracle(B, hw, seed):
    setup_exact()
    from snn_object_detectionddp_b200.loss import v8DetectionLoss
    nc = 8
    fm = _FakeModel(nc)
    _, labels = MO.synthetic_batch(B, 1, hw, hw, nc=nc, seed=seed + 10)
    labels = labels.to(DEV)
    batch = {"batch_idx": labels[:, 0], "cls": labels[:, 1], "bboxes": labels[:, 2:]}
    maps_r = [m.clone().requires_grad_(True) for m in _maps(B, hw, nc, seed)]
    maps_p = [m.clone().requires_grad_(True) for m in _maps(B, hw, nc, seed)]
    l_ref, it_ref = D.OracleV8DetectionLoss(fm)(maps_r, batch)
    l_ref.sum().backward()
    l_p, it_p = v8DetectionLoss(fm)(maps_p, batch)
    l_p.sum().backward()
    assert float(it_ref[0]) > 0 and float(it_ref[2]) > 0, "degenerate case: no foreground anchors"
    assert torch.allclose(l_p, l_ref, rtol=1e-4, atol=1e-6), (l_p, l_ref)
    assert torch.allclose(it_p, it_ref, rtol=1e-4, atol=1e-6)
    for a, b in zip(maps_p, maps_r):
        assert rel_err(a.grad, b.grad) < 1e-4


def test_detection_loss_no_targets():
    from snn_object_detectionddp_b200.loss import v8DetectionLoss
    fm = _FakeModel(8)
    maps_r = [m.clone().requires_grad_(True) for m in _maps(2, 64, 8, 5)]
    maps_p = [m.clone().requires_grad_(True) for m in _maps(2, 64, 8, 5)]
    empty = torch.zeros(0, 6, device=DEV)
    batch = {"batch_idx": empty[:, 0], "cls": empty[:, 1], "bboxes": empty[:, 2:]}
    l_ref, _ = D.OracleV8DetectionLoss(fm)(maps_r, batch)
    l_p, _ = v8DetectionLoss(fm)(maps_p, batch)
    assert float(l_p[0]) == 0 and float(l_p[2]) == 0
    assert torch.allclose(l_p, l_ref, rtol=1e-4)
    l_ref.sum().backward(); l_p.sum().backward()
    for a, b in zip(maps_p, maps_r):
        assert rel_err(a.grad, b.grad) < 1e-4


def test_decode_matches_oracle():
    from snn_object_detectionddp_b200 import kernels as K
    from snn_object_detectionddp_b200.head import make_anchors
    maps = _maps(3, 128, 8, 7)
    ref = D.decode(maps, torch.tensor([8.0, 16.0, 32.0]), 8, 16)            # [B, 12, A]
    cat = torch.cat([m.reshape(3, 72, -1) for m in maps], 2).permute(0, 2, 1)
    anchors, st = make_anchors([tuple(m.shape[2:]) for m in maps], [8.0, 16.0, 32.0], device=DEV)
    boxes, probs = K.detect_decode(cat[..., :64].contiguous(), cat[..., 64:].contiguous(), anchors.contiguous(),
                                   st.view(-1).contiguous(), xywh=True)
    got = torch.cat((boxes, probs), 2).permute(0, 2, 1)
    assert rel_err(got, ref) < 1e-5


def _models(neuron, widths=(64, 128, 256, 512), seed=0):
    from snn_object_detectionddp_b200.model import YOLOTemporalUNet
    torch.manual_seed(seed)
    orc = MO.OracleYOLOTemporalUNet(num_classes=8, hyp=HYP, neuron=neuron, emulate_bf16=True, widths=widths)
    MO.initialize_model_oracle(orc)
    net = YOLOTemporalUNet(num_classes=8, hyp=HYP, neuron=neuron)
    if widths != (128, 256, 512, 1024):
        from snn_object_detectionddp_b200.model import TemporalUNet
        net.temporal_unet = TemporalUNet([144, 144, 144], neuron=neuron, widths=widths)
    sd = {k: v for k, v in orc.state_dict().items()}
    res = net.load_state_dict(sd, strict=True)        # detection_head.* and temporal_unet.* keys interchange
    assert not res.missing_keys and not res.unexpected_keys
    return orc.to(DEV), net.to(DEV)


def test_feature_extractor_standin_matches_oracle():
    setup_exact()
    orc, net = _models("silu")
    frames, _ = MO.synthetic_batch(2, 2, 128, 128, seed=3)
    frames = frames.to(DEV)
    f_p = net.feature_extractor.forward_seq(frames, 2, 2)
    f_o = orc.feature_extractor(frames.permute(1, 0, 2, 3, 4).reshape(4, 3, 128, 128))
    for a, b in zip(f_p, f_o):
        assert rel_err(a.float().permute(0, 3, 1, 2), b) < 4e-3


def test_detect_head_matches_oracle_train_and_eval():
    setup_exact()
    orc, net = _models("silu")
    g = torch.Generator().manual_seed(4)
    feats = [torch.randn(2, 144, 128 // s, 128 // s, generator=g).to(DEV) for s in (8, 16, 32)]
    orc.train(); net.train()
    m_o = orc.detection_head([f.clone() for f in feats])
    m_p = net.detection_head([f.clone() for f in feats])
    for a, b in zip(m_p, m_o):
        assert a.shape == b.shape and rel_err(a, b) < 2e-2          # bf16 operands + bf16 SiLU outputs, 4 layers deep
    orc.eval(); net.eval()
    with torch.no_grad():
        (y_o, _), (y_p, _) = orc.detection_head(feats), net.detection_head(feats)
    assert y_p.shape == y_o.shape == (2, 12, 336)
    assert rel_err(y_p, y_o) < 2e-2


@pytest.mark.parametrize("neuron", ["silu", "lif"])
def test_training_steps_track_the_oracle(neuron):
    """Three full training steps (fused sequence path, fused loss, fused clip+AdamW with the tabulated OneCycle
    schedule) against the reference step semantics run by the oracle (train.py:58-80): loss items and global grad
    norm per step.  silu: tight; lif: spikes may flip near threshold and the loss is compared loosely.
    Both sides are reproducible -- the oracle runs on the CPU, the product in deterministic mode (snn_set_deterministic:
    no fp32 atomics) -- so which spikes flip, and with it the outcome, is the same on every run instead of depending
    on the order of atomic adds in the steps before."""
    setup_exact()
    from snn_object_detectionddp_b200 import _lib
    from snn_object_detectionddp_b200.trainer import Trainer
    orc, net = _models(neuron, seed=5)
    orc = orc.cpu()
    B, T, HW = 4, 3, 128
    frames, labels = MO.synthetic_batch(B, T, HW, HW, seed=11)
    orc.train()
    loss_fn, opt, sched = MO.make_reference_trainer(orc, total_steps=20)
    L = _lib.lib()
    before = L.snn_get_deterministic()
    L.snn_set_deterministic(1)
    try:
        tr = Trainer(net, total_steps=20, device=DEV)
        labels_d = labels.to(DEV)
        batch = {"batch_idx": labels_d[:, 0], "cls": labels_d[:, 1], "bboxes": labels_d[:, 2:]}
        tol = 3e-2 if neuron == "silu" else 0.25
        for step in range(3):
            _, it_o, gn_o = MO.reference_train_step(orc, loss_fn, opt, sched, frames, labels)
            _, it_p = tr.train_step(frames.to(DEV), batch)
            it_p = it_p.cpu()
            print(neuron, step, it_o.tolist(), it_p.tolist(), float(gn_o), float(tr.grad_norm))
            assert torch.allclose(it_p, it_o, rtol=tol, atol=1e-3), (step, it_p, it_o)
            assert abs(float(tr.grad_norm) - float(gn_o)) < 2 * tol * float(gn_o)
    finally:
        L.snn_set_deterministic(before)
    # parameters moved the same way: AdamW's first steps are +-lr per element, so compare the update direction
    if neuron == "silu":
        po = dict(orc.named_parameters())
        agree = []
        for k, p in net.named_parameters():
            if k.startswith("temporal_unet.enc1.conv"):
                agree.append(rel_err(p.data.cpu(), po[k].data))
        assert max(agree) < 1e-3


def test_skipping_dead_frame_backward_changes_nothing():
    """Only the last frame's predictions reach the loss (train.py:64-74).  Stateless layers (U-Net output convs, Detect
    head) skip the all-zero backward of the earlier frames.  The forward is deterministic (loss and BN buffers must be
    bit-identical); the backward is not (fp32 atomics in the BN reductions and the split-K wgrad), and this tiny
    geometry (2 frames, 2x2 bottleneck) amplifies that noise through ~40 batch-norm backward passes, so the gradients
    are compared (a) tightly on the layers the shortcut touches and (b) against the run-to-run noise elsewhere."""
    setup_exact()
    from snn_object_detectionddp_b200.params import store_for
    from snn_object_detectionddp_b200.loss import v8DetectionLoss
    res = []
    for skip in (True, False, False):
        _, net = _models("lif", seed=7)
        net.skip_dead_backward = skip
        net.train()
        B, T, HW = 2, 3, 128
        frames, labels = MO.synthetic_batch(B, T, HW, HW, seed=13)
        frames, labels = frames.to(DEV), labels.to(DEV)
        st = store_for(net, DEV)
        st.zero_grad()
        det, _ = net.forward_sequence(frames)
        loss, items = v8DetectionLoss(net)(det, {"batch_idx": labels[:, 0], "cls": labels[:, 1], "bboxes": labels[:, 2:]})
        loss.sum().backward()
        torch.cuda.synchronize()
        res.append((items.clone(), st.flat_g.clone(), {k: v.clone() for k, v in net.state_dict().items() if "running" in k}, st))
    (it_a, g_a, bn_a, st), (it_b, g_b, bn_b, _), (it_c, g_c, _, _) = res
    assert torch.equal(it_a, it_b) and torch.equal(it_b, it_c)
    for k in bn_a:
        assert torch.equal(bn_a[k], bn_b[k]), k
    assert float(g_b.abs().max()) > 0
    noise = float(rel_err(g_b, g_c))
    assert float(rel_err(g_a, g_b)) < 3 * noise + 1e-5, (float(rel_err(g_a, g_b)), noise)
    for e in st.entries:
        if e.name.startswith("detection_head.") or ".out_p" in e.name:
            sl = slice(e.offset, e.offset + e.numel)
            # + bf16 rounding of dy (2^-9 per element): bias gradients are sums of as few as 32 such values per channel and
            # cancel heavily, so a handful of rounding flips shows at the percent level; a missing contribution would be O(1)
            assert float(rel_err(g_a[sl], g_b[sl])) < 3 * float(rel_err(g_b[sl], g_c[sl])) + 2e-2, e.name


def test_drop_in_forward_signature_and_eval_outputs():
    """model(frame, hidden) -> (detections, hidden) with the reference's return structure (model.py:197-211):
    train -> list of 3 maps [B, nc+64, h, w]; eval -> (decoded [B, 4+nc, A], maps)."""
    orc, net = _models("lif", seed=6)
    frames, _ = MO.synthetic_batch(2, 2, 128, 128, seed=12)
    frames = frames.to(DEV)
    net.train()
    preds, hid = net(frames[:, 0], None)
    assert isinstance(preds, list) and [tuple(p.shape) for p in preds] == [(2, 72, 16, 16), (2, 72, 8, 8), (2, 72, 4, 4)]
    preds, hid = net(frames[:, 1], hid)
    assert hid[0].shape == (2, 512, 2, 2) and hid[1].shape == (2, 512, 2, 2)
    net.eval()
    with torch.no_grad():
        (dec, maps), hid = net(frames[:, 0], None)
    assert dec.shape == (2, 12, 336) and len(maps) == 3
    assert net.model[0] is net.detection_head and net.nc == 8 and net.args.box == 7.5
    assert torch.equal(net.strides.cpu(), torch.tensor([8.0, 16.0, 32.0]))


def test_checkpoint_roundtrip_and_validation_step(tmp_path):
    """Reference checkpoint format (train.py:204-209) + validation step (train.py:106-131): a reloaded trainer
    reproduces the eval-mode loss exactly and continues with the same optimizer state; a reference-style file that also
    carries frozen-extractor keys loads."""
    setup_exact()
    from snn_object_detectionddp_b200.trainer import Trainer
    _, net = _models("lif", seed=8)
    tr = Trainer(net, total_steps=20, device=DEV)
    frames, labels = MO.synthetic_batch(2, 2, 128, 128, seed=14)
    frames, labels = frames.to(DEV), labels.to(DEV)
    batch = {"batch_idx": labels[:, 0], "cls": labels[:, 1], "bboxes": labels[:, 2:]}
    for _ in range(2):
        tr.train_step(frames, batch)
    v0 = tr.validate_step(frames, batch).clone()
    assert net.training and torch.isfinite(v0).all()
    path = str(tmp_path / "latest.pt")
    tr.save_checkpoint(path, epoch=3, best_val_loss=1.5)
    ck = torch.load(path, map_location="cpu", weights_only=False)
    assert {"epoch", "model_state_dict", "best_val_loss"} <= set(ck) and ck["epoch"] == 3
    assert all(k.startswith(("temporal_unet.", "detection_head.", "model.0.", "feature_extractor.")) for k in ck["model_state_dict"])
    _, net2 = _models("lif", seed=9)                 # different init
    tr2 = Trainer(net2, total_steps=20, device=DEV)
    ck["model_state_dict"]["feature_extractor.model.model.0.conv.weight"] = torch.zeros(3)    # reference files carry these
    torch.save(ck, path)
    epoch, best = tr2.load_checkpoint(path)
    assert (epoch, best) == (3, 1.5) and tr2.step_idx == tr.step_idx
    assert torch.equal(tr2.validate_step(frames, batch), v0)
    assert torch.equal(tr2.store.flat_p, tr.store.flat_p) and torch.equal(tr2.store.flat_m, tr.store.flat_m)
    l1, i1 = tr.train_step(frames, batch)
    l2, i2 = tr2.train_step(frames, batch)
    assert torch.equal(i1, i2)                       # deterministic forward on identical parameters


def test_uint8_frames_equal_host_side_division():
    """uint8 frames divided by 255 on the device (snn_space_to_depth8_u8) == the reference's host-side
    `.float() / 255.0` (dataset.py:152) fed as fp32: bit-identical features, hence identical losses."""
    from snn_object_detectionddp_b200 import kernels as K
    g = torch.Generator().manual_seed(3)
    u8 = torch.randint(0, 256, (3, 2, 3, 64, 128), generator=g, dtype=torch.uint8)
    f32 = u8.float() / 255.0
    a = K.space_to_depth8(u8.to(DEV), 3, 2)
    b = K.space_to_depth8(f32.to(DEV), 3, 2)
    assert torch.equal(a, b)
    _, net = _models("lif", seed=10)
    net.eval()
    with torch.no_grad():
        da, _ = net.forward_sequence(u8.to(DEV))
        db, _ = net.forward_sequence(f32.to(DEV))
    for x, y in zip(da.box + da.cls, db.box + db.cls):
        assert torch.equal(x, y)


def test_reference_training_loop_runs_unchanged_on_the_drop_in_modules():
    """The body of the reference's train_one_epoch (train.py:58-80) verbatim -- per-frame loop threading `hidden`, loss on
    the last predictions, `.sum().backward()`, `clip_grad_norm_(10)`, torch `AdamW` + `OneCycleLR` -- on the drop-in
    modules, next to the fused Trainer path on a twin model: same losses step after step (the fused optimizer and the
    torch optimizer implement the same update; the two forward paths are bit-identical)."""
    setup_exact()
    from snn_object_detectionddp_b200.loss import v8DetectionLoss
    from snn_object_detectionddp_b200.trainer import Trainer
    _, model = _models("lif", seed=12)
    _, twin = _models("lif", seed=12)
    B, T, HW = 2, 3, 128
    image_tensor, labels_tensor = MO.synthetic_batch(B, T, HW, HW, seed=15)
    image_tensor, labels_tensor = image_tensor.to(DEV), labels_tensor.to(DEV)
    total_steps = 10
    # --- reference code path (train.py:155-169 + 58-80) ---
    loss_fn = v8DetectionLoss(model)
    optimizer = torch.optim.AdamW(model.parameters(), lr=1e-4, weight_decay=5e-4)
    scheduler = torch.optim.lr_scheduler.OneCycleLR(optimizer, max_lr=1e-4, total_steps=total_steps)
    tr = Trainer(twin, max_lr=1e-4, weight_decay=5e-4, total_steps=total_steps, device=DEV)
    model.train()
    for step in range(3):
        optimizer.zero_grad()
        hidden_state = None
        for t in range(T):
            frame = image_tensor[:, t, :, :, :]
            preds, hidden_state = model(frame, hidden_state)
        batch_dict = {'batch_idx': labels_tensor[:, 0], 'cls': labels_tensor[:, 1], 'bboxes': labels_tensor[:, 2:]}
        loss, loss_components_detached = loss_fn(preds, batch_dict)
        loss.sum().backward()
        gn = torch.nn.utils.clip_grad_norm_(model.parameters(), 10.0)
        optimizer.step()
        scheduler.step()
        _, items = tr.train_step(image_tensor, batch_dict)
        print(step, loss_components_detached.tolist(), items.tolist(), float(gn), float(tr.grad_norm))
        if step == 0:
            assert torch.equal(items, loss_components_detached)          # identical parameters, deterministic forward
            assert abs(float(gn) - float(tr.grad_norm)) < 2e-2 * float(gn)
        # later steps: the first AdamW updates move every weight by +-lr (sign of a noisy gradient) and this tiny spiking
        # net (2 frames, 2x2 bottleneck) amplifies that: observed 1-13 % apart; the bound only guards against a broken path
        assert torch.isfinite(items).all() and torch.allclose(items, loss_components_detached, rtol=0.5, atol=1e-2)
    assert all(p.grad is not None for p in model.temporal_unet.parameters())


def test_device_prefetcher_pageable_and_pinned_sources():
    """data.DevicePrefetcher: batches arrive intact and in order whether the host tensors are pageable (staged through
    pinned memory) or already pinned, with the copy of batch i+1 queued while batch i is in use."""
    from snn_object_detectionddp_b200.data import DevicePrefetcher
    pf = DevicePrefetcher(DEV)
    g = torch.Generator().manual_seed(4)
    batches = []
    for i in range(5):
        fr = torch.randint(0, 256, (2, 2, 3, 64, 64), generator=g, dtype=torch.uint8)
        pad = (torch.full((2, 8), float(i)), torch.rand(2, 8, 4, generator=g), torch.ones(2, 8, dtype=torch.bool))
        if i % 2:
            fr, pad = fr.pin_memory(), tuple(t.pin_memory() for t in pad)
        batches.append((fr, pad))
    pf.stage(*batches[0])
    for i in range(5):
        fr_d, pad_d = pf.take()
        if i + 1 < 5:
            pf.stage(*batches[i + 1])
        got = (fr_d.clone(), tuple(t.clone() for t in pad_d))
        pf.release()
        torch.cuda.synchronize()
        assert torch.equal(got[0].cpu(), batches[i][0])
        for a, b in zip(got[1], batches[i][1]):
            assert torch.equal(a.cpu(), b)
    assert pf.bytes_per_batch() == sum(t.numel() * t.element_size() for t in (batches[4][0],) + batches[4][1])


# ------------------------------------------------------------------------------------------------
# assigner kernels (csrc/assign.cu) and the fused head -> loss path (scale-major buffers, bf16 gradients)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed,B,nmax,hw", [(0, 4, 6, 128), (1, 2, 1, 128), (2, 3, 12, 256), (3, 64, 8, 256)])
def test_tal_assign_kernels_match_dense_formulation(seed, B, nmax, hw):
    """snn_tal_assign (3 launches) == the dense torch formulation of TaskAlignedAssigner (loss.task_aligned_assign, itself
    pinned to the restated ultralytics assigner on CPU by tests/test_host_logic.py) on the same random predictions.
    Anchors whose alignment metric is exactly 0 may be picked differently among the zero ties of the top-k (torch.topk's
    tie order is unspecified; the kernels take the lower index): they carry target score 0 = no loss weight, so the
    comparison is on the anchors with weight > 0: same foreground set, same boxes, scores to 1e-5."""
    from snn_object_detectionddp_b200 import kernels as K
    from snn_object_detectionddp_b200.head import make_anchors
    from snn_object_detectionddp_b200.loss import task_aligned_assign
    g = torch.Generator().manual_seed(seed)
    nc, strides = 8, (8.0, 16.0, 32.0)
    anchors, st = make_anchors([(hw // int(s), hw // int(s)) for s in strides], strides)
    A = anchors.shape[0]
    probs = torch.rand(B, A, nc, generator=g) * 0.5
    ctr = (anchors * st)[None].expand(B, -1, -1)
    half = torch.rand(B, A, 2, generator=g) * 30 + 4
    jit = (torch.rand(B, A, 2, generator=g) - 0.5) * 6
    pboxes = torch.cat((ctr + jit - half, ctr + jit + half), -1)
    n = torch.randint(0, nmax + 1, (B,), generator=g)
    n[0] = nmax
    cls = torch.randint(0, nc, (B, nmax), generator=g)
    cxy = torch.rand(B, nmax, 2, generator=g) * 0.7 + 0.15
    wh = torch.rand(B, nmax, 2, generator=g) * 0.3 + 0.06
    box = torch.cat((cxy, wh), -1)
    valid = torch.arange(nmax)[None] < n[:, None]
    probs, pboxes, anchors, st, cls, box, valid = (t.to(DEV).contiguous() for t in (probs, pboxes, anchors, st.view(-1), cls, box, valid))
    tb, ts, fg = K.tal_assign(probs, pboxes, anchors, st, cls, box, valid, (float(hw), float(hw)), nc)
    scale = torch.tensor([hw, hw, hw, hw], device=DEV, dtype=torch.float32)
    xy, half_wh = box[..., :2] * scale[:2], box[..., 2:] * scale[2:] / 2
    gt_xyxy = torch.cat((xy - half_wh, xy + half_wh), -1) * valid[..., None]
    mask_gt = valid & (gt_xyxy.sum(-1) > 0)
    r_tb, r_ts, r_fg = task_aligned_assign(probs, pboxes, anchors * st[:, None], cls, gt_xyxy, mask_gt, nc, 10)
    w_k, w_r = ts.sum(-1), r_ts.sum(-1)
    assert int((w_r > 0).sum()) > 0
    assert torch.equal(w_k > 0, w_r > 0), int(((w_k > 0) != (w_r > 0)).sum())
    assert torch.allclose(ts, r_ts, rtol=1e-5, atol=1e-7), float((ts - r_ts).abs().max())
    pos = w_r > 0
    assert bool((fg.bool() | ~pos).all()) and torch.equal(tb[pos], r_tb[pos])
    # foreground flags may differ only on zero-weight anchors
    assert int((fg.bool() != r_fg.bool()).sum()) == int(((fg.bool() != r_fg.bool()) & ~pos).sum())
    tb2, ts2, fg2 = K.tal_assign(probs, pboxes, anchors, st, cls, box, valid, (float(hw), float(hw)), nc)
    assert torch.equal(ts, ts2) and torch.equal(fg, fg2) and torch.equal(tb, tb2)          # deterministic


def test_fused_head_loss_path_equals_list_of_maps_path():
    """`loss_fn(HeadOut)` (scale-major prediction buffers written by the head's closing convs, bf16 gradients handed
    straight to their backward: no torch.cat / split anywhere) == `loss_fn([maps])` (the reference's call with the list
    of [B, nc+64, h, w] maps, train.py:74): same loss values; parameter gradients agree to 1e-2 (the fused path rounds the
    prediction gradients to bf16 once, as every other `dy` on the path)."""
    setup_exact()
    from snn_object_detectionddp_b200.loss import v8DetectionLoss
    from snn_object_detectionddp_b200.params import store_for
    res = []
    for fused in (True, False):
        _, net = _models("lif", seed=21)
        net.train()
        B, T, HW = 4, 2, 128
        frames, labels = MO.synthetic_batch(B, T, HW, HW, seed=22)
        frames, labels = frames.to(DEV), labels.to(DEV)
        batch = {"batch_idx": labels[:, 0], "cls": labels[:, 1], "bboxes": labels[:, 2:]}
        st = store_for(net, DEV)
        st.zero_grad()
        det, _ = net.forward_sequence(frames)
        assert det.flat_box is not None and det.a_off == [0, 256, 320, 336]
        loss, items = v8DetectionLoss(net)(det if fused else det.maps_nchw(), batch)
        loss.sum().backward()
        torch.cuda.synchronize()
        res.append((loss.detach().clone(), items.clone(), st.flat_g.clone(), st))
    (l_f, it_f, g_f, st), (l_m, it_m, g_m, _) = res
    assert torch.allclose(it_f, it_m, rtol=1e-6) and torch.allclose(l_f, l_m, rtol=1e-6), (it_f, it_m)
    assert float(it_f[0]) > 0 and float(g_m.abs().max()) > 0
    worst = []
    for e in st.entries:
        sl = slice(e.offset, e.offset + e.numel)
        if float(g_m[sl].norm()) > 0:
            worst.append((rel_err(g_f[sl], g_m[sl]), e.name))
    print("fused vs list-of-maps, worst parameter-gradient differences:", sorted(worst, reverse=True)[:3])
    assert rel_err(g_f, g_m) < 1e-2
    head = [w for w in worst if w[1].startswith("detection_head.") and (".cv2.0.2." in w[1] or ".cv3.0.2." in w[1])]
    assert head and max(head)[0] < 1e-2, head


def test_dead_frame_shortcut_in_deterministic_mode():
    """Same comparison as test_skipping_dead_frame_backward_changes_nothing with snn_set_deterministic(1): the two full-backward
    runs are now BIT-IDENTICAL (no noise term), and the shortcut differs from them only through the launch shapes of the head /
    output-conv backward (NB = B instead of T*B moves tile and reduction-group boundaries, i.e. fp32 summation order),
    measured 1e-9 relative -- so the percent-level noise band of the default-mode test above is all reordering noise of the
    atomics, not a property of the shortcut.  Bound: 1e-6."""
    setup_exact()
    from snn_object_detectionddp_b200 import _lib
    from snn_object_detectionddp_b200.params import store_for
    from snn_object_detectionddp_b200.loss import v8DetectionLoss
    L = _lib.lib()
    before = L.snn_get_deterministic()
    L.snn_set_deterministic(1)
    try:
        res = []
        for skip in (True, False, False):
            _, net = _models("lif", seed=7)
            net.skip_dead_backward = skip
            net.train()
            B, T, HW = 2, 3, 128
            frames, labels = MO.synthetic_batch(B, T, HW, HW, seed=13)
            frames, labels = frames.to(DEV), labels.to(DEV)
            st = store_for(net, DEV)
            st.zero_grad()
            det, _ = net.forward_sequence(frames)
            loss, items = v8DetectionLoss(net)(det, {"batch_idx": labels[:, 0], "cls": labels[:, 1], "bboxes": labels[:, 2:]})
            loss.sum().backward()
            torch.cuda.synchronize()
            res.append((items.clone(), st.flat_g.clone()))
    finally:
        L.snn_set_deterministic(before)
    (it_a, g_a), (it_b, g_b), (it_c, g_c) = res
    assert torch.equal(it_a, it_b) and torch.equal(it_b, it_c)
    assert float(g_b.abs().max()) > 0 and torch.equal(g_b, g_c)
    e = float(rel_err(g_a, g_b))
    print(f"dead-frame shortcut vs full backward, deterministic mode: rel {e:.2e}")
    assert e < 1e-6, e
