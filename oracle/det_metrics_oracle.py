"""TEST INFRASTRUCTURE ONLY -- numpy restatement of the ultralytics 8.3 detection metric the reference meant to compute
(eval_2.py:20-130: ``DetectionValidator`` / ``DetMetrics``).

PARITY UNPINNED, like detect_oracle.py: ultralytics is un-vendored and not installable offline, so the published
algorithm is restated here with every tie rule fixed, and the CUDA kernels (csrc/metrics.cu) are compared against it.

* ``DetectionValidator._process_batch`` / ``match_predictions`` (non-scipy branch), stated as
  - ground truth  xywh2xyxy(cx cy w h normalised) * (W, H, W, H) in fp32, predictions = NMS rows x1 y1 x2 y2 conf cls in
    the same input-pixel space (frames are not letterboxed: no scale_boxes);
  - IoU = box_iou in fp32, inter / (area_gt + area_pred - inter + 1e-7) in that order, zeroed across classes;
  - each prediction takes the same-class gt of highest IoU (exact ties: the higher gt index); at threshold t it is a TP
    iff that IoU >= t and it is the lowest NMS row among the predictions whose best gt is that gt with IoU >= t.  A
    prediction whose best gt went to an earlier row is an FP even if another free gt overlaps it (ultralytics does so).
    ``match_predictions_unique_chain`` is the verbatim argsort -> np.unique -> np.unique chain (stable argsort); the
    tests check that both agree.
* ``metrics.ap_per_class`` / ``compute_ap`` / ``smooth`` in float64, with a STABLE sort by confidence (ultralytics uses
  numpy's default, unstable sort: equal confidences keep record order here).
* results = ``DetMetrics.results_dict``: precision, recall, mAP50, mAP50-95 and fitness = 0.1 mAP50 + 0.9 mAP50-95.
"""
import numpy as np
import torch

IOUV = torch.linspace(0.5, 0.95, 10).numpy()           # fp32, as DetectionValidator builds it
EPS_IOU = np.float32(1e-7)
KEYS = ("metrics/precision(B)", "metrics/recall(B)", "metrics/mAP50(B)", "metrics/mAP50-95(B)", "fitness")


def gt_boxes_xyxy(xywh, img_w, img_h):
    """[M, 4] normalised cx cy w h -> fp32 pixel x1 y1 x2 y2: (cx - w/2) * W, ..."""
    b = np.asarray(xywh, np.float32).reshape(-1, 4)
    half = b[:, 2:4] / np.float32(2)
    xyxy = np.concatenate((b[:, :2] - half, b[:, :2] + half), 1)
    return (xyxy * np.array([img_w, img_h, img_w, img_h], np.float32)).astype(np.float32)


def box_iou(gt, pred):
    """fp32 [M, N], operation order of ultralytics.utils.metrics.box_iou(gt, pred)."""
    gt, pred = np.asarray(gt, np.float32).reshape(-1, 4), np.asarray(pred, np.float32).reshape(-1, 4)
    a1, a2 = gt[:, None, :2], gt[:, None, 2:]
    b1, b2 = pred[None, :, :2], pred[None, :, 2:]
    wh = np.clip(np.minimum(a2, b2) - np.maximum(a1, b1), np.float32(0), None)
    inter = wh[..., 0] * wh[..., 1]
    area_a = (a2 - a1)[..., 0] * (a2 - a1)[..., 1]
    area_b = (b2 - b1)[..., 0] * (b2 - b1)[..., 1]
    return (inter / (((area_a + area_b) - inter) + EPS_IOU)).astype(np.float32)


def class_iou(gt_cls, pred_cls, iou):
    return iou * (np.asarray(gt_cls)[:, None] == np.asarray(pred_cls)[None, :])


def match_predictions(pred_cls, gt_cls, iou, iouv=IOUV):
    """-> bool [N, len(iouv)].  iou [M, N] (gt x pred, before the class mask)."""
    iou = class_iou(gt_cls, pred_cls, iou)
    m, n = iou.shape
    correct = np.zeros((n, len(iouv)), bool)
    if m == 0 or n == 0:
        return correct
    best_iou = iou.max(0)
    best_gt = m - 1 - np.argmax(iou[::-1], 0)                # highest IoU, exact ties -> the higher gt index
    for t, thr in enumerate(iouv):
        taken = set()
        for j in range(n):                                   # NMS row order: the lowest row claims the gt
            if best_iou[j] >= thr and best_gt[j] not in taken:
                taken.add(best_gt[j])
                correct[j, t] = True
    return correct


def match_predictions_unique_chain(pred_cls, gt_cls, iou, iouv=IOUV):
    """ultralytics DetectionValidator.match_predictions (use_scipy=False), with a stable argsort."""
    iou = class_iou(gt_cls, pred_cls, iou)
    correct = np.zeros((iou.shape[1], len(iouv)), bool)
    for i, threshold in enumerate(iouv):
        matches = np.nonzero(iou >= threshold)
        matches = np.array(matches).T
        if matches.shape[0]:
            if matches.shape[0] > 1:
                matches = matches[iou[matches[:, 0], matches[:, 1]].argsort(kind="stable")[::-1]]
                matches = matches[np.unique(matches[:, 1], return_index=True)[1]]
                matches = matches[np.unique(matches[:, 0], return_index=True)[1]]
            correct[matches[:, 1].astype(int), i] = True
    return correct


def batch_records(rows, counts, gt_cls, gt_box, gt_valid, img_w, img_h):
    """One batch of NMS output + pad_targets tensors -> (conf fp32 [n], cls int [n], tp bool [n, 10], gt classes [g]).
    rows [B, max_det, 6], counts [B], gt_cls [B, M], gt_box [B, M, 4] (normalised xywh), gt_valid [B, M]."""
    rows, counts = np.asarray(rows, np.float32), np.asarray(counts).astype(int)
    gt_cls, gt_box, gt_valid = np.asarray(gt_cls), np.asarray(gt_box, np.float32), np.asarray(gt_valid).astype(bool)
    confs, clss, tps, tcls = [], [], [], []
    for b in range(rows.shape[0]):
        p = rows[b, :counts[b]]
        v = gt_valid[b]
        gc = gt_cls[b][v]
        tcls.append(gc.astype(np.int64))
        if p.shape[0] == 0:
            continue
        iou = box_iou(gt_boxes_xyxy(gt_box[b][v], img_w, img_h), p[:, :4])
        tps.append(match_predictions(p[:, 5], gc.astype(np.float32), iou))
        confs.append(p[:, 4])
        clss.append(p[:, 5].astype(np.int64))
    cat = lambda xs, shape, dt: np.concatenate(xs) if xs else np.zeros(shape, dt)   # noqa: E731
    return (cat(confs, (0,), np.float32), cat(clss, (0,), np.int64), cat(tps, (0, 10), bool), cat(tcls, (0,), np.int64))


def smooth(y, f=0.05):
    nf = round(len(y) * f * 2) // 2 + 1
    p = np.ones(nf // 2)
    yp = np.concatenate((p * y[0], y, p * y[-1]), 0)
    return np.convolve(yp, np.ones(nf) / nf, mode="valid")


def compute_ap(recall, precision):
    mrec = np.concatenate(([0.0], recall, [1.0]))
    mpre = np.concatenate(([1.0], precision, [0.0]))
    mpre = np.flip(np.maximum.accumulate(np.flip(mpre)))
    x = np.linspace(0, 1, 101)
    return np.trapezoid(np.interp(x, mrec, mpre), x)


def ap_per_class(tp, conf, pred_cls, target_cls, eps=1e-16):
    """-> dict(p, r, f1 [nc_present], ap [nc_present, 10], unique_classes, p_curve, r_curve [nc_present, 1000], index)."""
    tp, conf, pred_cls = np.asarray(tp, bool), np.asarray(conf, np.float32), np.asarray(pred_cls)
    i = np.argsort(-conf, kind="stable")
    tp, conf, pred_cls = tp[i], conf[i], pred_cls[i]
    unique_classes, nt = np.unique(target_cls, return_counts=True)
    nc = unique_classes.shape[0]
    x = np.linspace(0, 1, 1000)
    ap, p_curve, r_curve = np.zeros((nc, tp.shape[1])), np.zeros((nc, 1000)), np.zeros((nc, 1000))
    for ci, c in enumerate(unique_classes):
        i = pred_cls == c
        n_l = nt[ci]
        n_p = i.sum()
        if n_p == 0 or n_l == 0:
            continue
        fpc = (1 - tp[i]).cumsum(0)
        tpc = tp[i].cumsum(0)
        recall = tpc / (n_l + eps)
        r_curve[ci] = np.interp(-x, -conf[i], recall[:, 0], left=0)
        precision = tpc / (tpc + fpc)
        p_curve[ci] = np.interp(-x, -conf[i], precision[:, 0], left=1)
        for j in range(tp.shape[1]):
            ap[ci, j] = compute_ap(recall[:, j], precision[:, j])
    f1 = 2 * p_curve * r_curve / (p_curve + r_curve + eps)
    index = int(smooth(f1.mean(0), 0.1).argmax()) if nc else 0
    return dict(p=p_curve[:, index], r=r_curve[:, index], f1=f1[:, index], ap=ap, unique_classes=unique_classes.astype(int),
                p_curve=p_curve, r_curve=r_curve, index=index)


def results_dict(tp, conf, pred_cls, target_cls):
    """DetMetrics.results_dict (+ per-class AP [n_present, 10] and the class index, as in DetMetrics.ap_class_index)."""
    r = ap_per_class(tp, conf, pred_cls, target_cls)
    ap = r["ap"]
    mp = float(r["p"].mean()) if len(r["p"]) else 0.0
    mr = float(r["r"].mean()) if len(r["r"]) else 0.0
    map50 = float(ap[:, 0].mean()) if len(ap) else 0.0
    map5095 = float(ap.mean()) if len(ap) else 0.0
    fitness = float((np.array([mp, mr, map50, map5095]) * np.array([0.0, 0.0, 0.1, 0.9])).sum())
    out = dict(zip(KEYS, (mp, mr, map50, map5095, fitness)))
    out["ap"] = ap
    out["ap_class_index"] = r["unique_classes"]
    out["index"] = r["index"]
    return out


class SpecMetrics:
    """Accumulates batch_records() over an evaluation, then results_dict() (the stock per-image host route)."""

    def __init__(self):
        self.conf, self.cls, self.tp, self.tcls = [], [], [], []

    def update(self, rows, counts, gt_cls, gt_box, gt_valid, img_w, img_h):
        c, k, t, g = batch_records(rows, counts, gt_cls, gt_box, gt_valid, img_w, img_h)
        self.conf.append(c); self.cls.append(k); self.tp.append(t); self.tcls.append(g)

    def compute(self):
        cat = lambda xs, shape, dt: np.concatenate(xs) if xs else np.zeros(shape, dt)   # noqa: E731
        return results_dict(cat(self.tp, (0, 10), bool), cat(self.conf, (0,), np.float32), cat(self.cls, (0,), np.int64),
                            cat(self.tcls, (0,), np.int64))
