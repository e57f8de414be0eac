"""Detection loss with the call surface of ultralytics' ``v8DetectionLoss`` (built at reference train.py:155 as
``v8DetectionLoss(model)``, called at train.py:74,126 as ``loss_fn(preds, batch) -> (loss*B, loss.detach())``).

PARITY UNPINNED: ultralytics is an un-vendored, unpinned third party (SURVEY.md 8c); its published 8.3.x algorithm is
restated.  Split of the work:

* target assignment (TaskAlignedAssigner, top-k 10, alpha 0.5, beta 6) -- no gradient flows through it; three kernels
  of libsnnb200 (csrc/assign.cu), synchronisation-free.  `task_aligned_assign` below is the same algorithm as dense torch
  ops: the host-checkable formulation the kernels are tested against (tests/test_host_logic.py pins it to the restated
  ultralytics assigner on CPU; tests/test_gpu_train.py pins the kernels to it) -- the product path does not call it;
* everything differentiable (BCE class loss over [B,A,nc], CIoU box loss, DFL, their reductions, the normalisation by the
  target-score sum, the hyp gains and the backward) -- csrc/loss.cu, behind ``DetectLossFn``.
"""
import torch
from torch.autograd import Function

from . import kernels as K


class DetectLossFn(Function):
    """v8DetectionLoss forward + backward on the libsnnb200 kernels (5 + 1 launches, no host synchronisation):
    decode -> task-aligned assignment -> fused BCE / CIoU / DFL sums -> finalisation ; one backward kernel.

    `preds` are either the six per-scale tensors of a HeadOut (views of its scale-major buffers; gradients come back as
    bf16 NHWC views, directly the `dy` operands of the head's closing convs) or (pred_distri [B,A,64], pred_scores
    [B,A,nc]) in natural layout (drop-in list-of-maps path; fp32 gradients).  Returns (loss*B [3], loss [3])."""

    @staticmethod
    def forward(ctx, meta, *preds):
        if meta["a_off"]:
            distri, scores = meta["flat_box"], meta["flat_cls"]
        else:
            distri, scores = preds[0].contiguous(), preds[1].contiguous()
        B, A, nc, reg_max = meta["B"], meta["A"], meta["nc"], meta["reg_max"]
        cls, box, valid = meta["labels"]
        out6, coef3, targets = K.detect_assign_loss_fwd(distri, scores, meta["a_off"], meta["anchors"], meta["stride"], cls, box, valid,
                                                        meta["img_wh"], B, A, nc, reg_max, meta["topk"], meta["gains"], meta["counter"])
        ctx.meta, ctx.saved = meta, (distri, scores, coef3, targets)
        ctx.shapes = [tuple(p.shape) for p in preds]
        loss_b, items = out6[:3], out6[3:]
        ctx.mark_non_differentiable(items)
        return loss_b, items

    @staticmethod
    def backward(ctx, g_loss, _g_items):
        meta = ctx.meta
        distri, scores, coef3, targets = ctx.saved
        gout = g_loss if (g_loss.dtype == torch.float32 and g_loss.is_contiguous()) else g_loss.float().contiguous()
        fused = bool(meta["a_off"])
        gd, gs = K.detect_loss_bwd_rows(distri, scores, meta["a_off"], meta["anchors"], meta["stride"], targets, meta["B"], meta["A"],
                                        meta["nc"], meta["reg_max"], coef3, gout, bf16=fused)
        if not fused:
            return None, gd.view(ctx.shapes[0]), gs.view(ctx.shapes[1])
        B, a_off, nl = meta["B"], meta["a_off"], len(meta["a_off"]) - 1
        grads = [gd[B * a_off[i]:B * a_off[i + 1]].view(ctx.shapes[i]) for i in range(nl)]
        grads += [gs[B * a_off[i]:B * a_off[i + 1]].view(ctx.shapes[nl + i]) for i in range(nl)]
        return (None, *grads)


def _ciou_dense(b1, b2, eps=1e-7):
    """CIoU of broadcastable xyxy boxes [...,4] (assignment metric; no gradient)."""
    x1, y1, x2, y2 = b1.unbind(-1)
    X1, Y1, X2, Y2 = b2.unbind(-1)
    w1, h1, w2, h2 = x2 - x1, y2 - y1 + eps, X2 - X1, Y2 - Y1 + eps
    inter = (torch.minimum(x2, X2) - torch.maximum(x1, X1)).clamp_(0) * (torch.minimum(y2, Y2) - torch.maximum(y1, Y1)).clamp_(0)
    union = w1 * h1 + w2 * h2 - inter + eps
    iou = inter / union
    cw = torch.maximum(x2, X2) - torch.minimum(x1, X1)
    ch = torch.maximum(y2, Y2) - torch.minimum(y1, Y1)
    c2 = cw * cw + ch * ch + eps
    rho2 = ((X1 + X2 - x1 - x2) ** 2 + (Y1 + Y2 - y1 - y2) ** 2) / 4
    v = (4 / torch.pi ** 2) * (torch.atan(w2 / h2) - torch.atan(w1 / h1)) ** 2
    alpha = v / (v - iou + (1 + eps))
    return iou - (rho2 / c2 + v * alpha)


@torch.no_grad()
def task_aligned_assign(pd_scores, pd_bboxes, anc_points, gt_labels, gt_bboxes, mask_gt, nc, topk=10, alpha=0.5, beta=6.0,
                        eps=1e-9):
    """Dense TaskAlignedAssigner.  pd_scores [B,A,nc] (sigmoid), pd_bboxes [B,A,4] xyxy px, anc_points [A,2] px,
    gt_labels [B,M] long, gt_bboxes [B,M,4] xyxy px, mask_gt [B,M] bool (M >= 1).
    Returns target_bboxes [B,A,4], target_scores [B,A,nc], fg uint8 [B,A]."""
    B, A, _ = pd_scores.shape
    M = gt_bboxes.shape[1]
    lt, rb = gt_bboxes[:, :, None, :2], gt_bboxes[:, :, None, 2:]
    deltas = torch.cat((anc_points[None, None] - lt, rb - anc_points[None, None]), -1)             # [B,M,A,4]
    in_gts = deltas.amin(-1) > eps
    valid = in_gts & mask_gt[:, :, None]
    cls_scores = torch.gather(pd_scores.transpose(1, 2), 1, gt_labels.clamp(0, nc - 1)[:, :, None].expand(-1, -1, A))
    zero = pd_scores.new_zeros(())
    bbox_scores = torch.where(valid, cls_scores, zero)
    overlaps = torch.where(valid, _ciou_dense(gt_bboxes[:, :, None, :], pd_bboxes[:, None, :, :]).clamp_(0), zero)
    align = bbox_scores.pow(alpha) * overlaps.pow(beta)
    k = min(topk, A)
    topk_idx = torch.topk(align, k, dim=-1).indices
    topk_idx = torch.where(mask_gt[:, :, None], topk_idx, torch.zeros_like(topk_idx))
    count = torch.zeros((B, M, A), device=align.device, dtype=torch.int32)
    count.scatter_add_(-1, topk_idx, torch.ones_like(topk_idx, dtype=torch.int32))
    mask_pos = ((count == 1) & valid).to(align.dtype)
    # an anchor claimed by several ground truths keeps the one with the largest overlap
    fg_cnt = mask_pos.sum(1)
    is_max = torch.zeros_like(mask_pos).scatter_(1, overlaps.argmax(1, keepdim=True), 1.0)
    mask_pos = torch.where((fg_cnt > 1)[:, None, :].expand(-1, M, -1), is_max, mask_pos)
    fg = mask_pos.sum(1)
    tgt_idx = mask_pos.argmax(1)                                                                    # [B,A]
    t_labels = torch.gather(gt_labels, 1, tgt_idx).clamp_(0)
    t_boxes = torch.gather(gt_bboxes, 1, tgt_idx[:, :, None].expand(-1, -1, 4))
    t_scores = torch.zeros((B, A, nc), device=align.device, dtype=align.dtype).scatter_(2, t_labels[:, :, None], 1.0)
    t_scores = t_scores * (fg > 0)[:, :, None]
    align = align * mask_pos
    pos_align = align.amax(-1, keepdim=True)
    pos_ov = (overlaps * mask_pos).amax(-1, keepdim=True)
    norm = (align * pos_ov / (pos_align + eps)).amax(1)[:, :, None]
    return t_boxes.contiguous(), (t_scores * norm).contiguous(), (fg > 0).to(torch.uint8).contiguous()


def pad_targets(labels, batch_size, device=None, max_boxes=None):
    """[M,6] rows (batch_idx, cls, cx, cy, w, h) (reference train.py:10-44 collate layout) -> dense
    (cls long [B,Mx], xywh fp32 [B,Mx,4], valid bool [B,Mx]); Mx = max boxes per sample, or `max_boxes` if given.  Done where the labels live: call it on the HOST
    tensors of the input pipeline and nothing in the loss has to synchronise."""
    labels = labels.detach()
    idx = labels[:, 0].long()
    counts = torch.bincount(idx, minlength=batch_size) if labels.shape[0] else labels.new_zeros(batch_size, dtype=torch.long)
    mx = max(int(counts.max()) if labels.shape[0] else 0, 1)
    if max_boxes is not None:          # fixed shape (CUDA-graph replay needs static shapes)
        if mx > max_boxes:
            raise ValueError(f"a sample has {mx} boxes > max_boxes={max_boxes}")
        mx = max_boxes
    order = torch.argsort(idx, stable=True)
    sl = labels[order]
    starts = torch.cumsum(counts, 0) - counts
    pos = torch.arange(sl.shape[0], device=labels.device) - starts[idx[order]]
    cls = torch.zeros((batch_size, mx), dtype=torch.long, device=labels.device)
    box = torch.zeros((batch_size, mx, 4), dtype=torch.float32, device=labels.device)
    valid = torch.zeros((batch_size, mx), dtype=torch.bool, device=labels.device)
    cls[idx[order], pos] = sl[:, 1].long()
    box[idx[order], pos] = sl[:, 2:6].float()
    valid[idx[order], pos] = True
    if device is not None:
        cls, box, valid = (t.to(device, non_blocking=True) for t in (cls, box, valid))
    return cls, box, valid


def batch_targets(batch, batch_size, device):
    """The targets of a loss batch -- {'padded': pad_targets(...)} or the collate dict {'batch_idx', 'cls', 'bboxes'}
    (train.py:68-72) -- as device tensors (cls long [B,M], xywh fp32 [B,M,4], valid bool [B,M])."""
    if "padded" in batch:
        cls, box, valid = (t.to(device, non_blocking=True) for t in batch["padded"])
    else:
        lab = torch.cat((batch["batch_idx"].view(-1, 1).float(), batch["cls"].view(-1, 1).float(),
                         batch["bboxes"].view(-1, 4).float()), 1)
        cls, box, valid = pad_targets(lab, batch_size, device)
    return cls.long().contiguous(), box.float().contiguous(), valid.contiguous()


class v8DetectionLoss:
    def __init__(self, model, tal_topk=10):
        m = model.model[-1]                       # the Detect module (reference model.py:195)
        self.hyp = model.args
        self.stride = [float(s) for s in m.stride.tolist()]
        self.nc, self.reg_max = m.nc, m.reg_max
        self.no = m.nc + m.reg_max * 4
        self.topk = tal_topk
        self._gains = None
        self._anchor_cache = {}
        self._scale_cache = {}

    def _anchors(self, shapes, device):
        key = (tuple(shapes), str(device))
        if key not in self._anchor_cache:
            from .head import make_anchors
            pts, st = make_anchors(shapes, self.stride, 0.5, device=device)
            self._anchor_cache[key] = (pts.contiguous(), st.view(-1).contiguous())
        return self._anchor_cache[key]

    def _flatten(self, preds):
        """-> (pred_distri [B,A,4*reg_max], pred_scores [B,A,nc], [(h,w),...])"""
        from .head import HeadOut
        if isinstance(preds, HeadOut):
            d, s = preds.flat()
            return d, s, preds.shapes()
        feats = preds[1] if isinstance(preds, tuple) else preds           # eval-mode (decoded, maps) or list of maps
        b = feats[0].shape[0]
        cat = torch.cat([f.reshape(b, self.no, -1) for f in feats], 2).permute(0, 2, 1)
        return cat[..., :4 * self.reg_max].contiguous(), cat[..., 4 * self.reg_max:].contiguous(), [tuple(f.shape[2:]) for f in feats]

    def _labels(self, batch, B, dev):
        return batch_targets(batch, B, dev)

    def __call__(self, preds, batch):
        from .head import HeadOut
        fused = isinstance(preds, HeadOut) and preds.flat_box is not None
        if fused:
            shapes, dev, B = preds.shapes(), preds.flat_box.device, preds.box[0].shape[0]
            tensors = tuple(preds.box) + tuple(preds.cls)
            a_off, flat_box, flat_cls = tuple(preds.a_off), preds.flat_box, preds.flat_cls
        else:
            distri, scores, shapes = self._flatten(preds)
            tensors = (distri.float(), scores.float())
            dev, B = distri.device, distri.shape[0]
            a_off, flat_box, flat_cls = (), None, None
        anchors, stride = self._anchors(shapes, dev)
        if self._gains is None or self._gains.device != dev:
            self._gains = torch.tensor([self.hyp.box, self.hyp.cls, self.hyp.dfl], device=dev, dtype=torch.float32)
            self._counter = torch.zeros(1, device=dev, dtype=torch.int32)      # ticket of the finalising block (kernel leaves it 0)
        # imgsz = stride-8 map size * stride (ultralytics: feats[0].shape[2:] * stride[0]); (W, H) order for the xywh scaling
        img_wh = (shapes[0][1] * self.stride[0], shapes[0][0] * self.stride[0])
        meta = dict(a_off=a_off, flat_box=flat_box, flat_cls=flat_cls, anchors=anchors, stride=stride, labels=self._labels(batch, B, dev),
                    img_wh=img_wh, B=B, A=anchors.shape[0], nc=self.nc, reg_max=self.reg_max, topk=self.topk, gains=self._gains,
                    counter=self._counter)
        loss_b, items = DetectLossFn.apply(meta, *tensors)
        return loss_b, items
