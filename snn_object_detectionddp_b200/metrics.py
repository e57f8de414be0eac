"""Detection quality metrics -- precision, recall, mAP50, mAP50-95 -- with the results of ultralytics' ``DetMetrics``
(what eval_2.py:82-88 meant to report), computed on the device.

    m = DetMetrics(nc, device)
    for each batch:  m.update(rows, counts, padded_targets, (H, W))      # snn_nms output + pad_targets output
    results = m.compute()                                                # {"metrics/mAP50(B)": ..., ...}

PARITY UNPINNED: ultralytics is un-vendored (SURVEY.md 8c); its DetectionValidator matching and ap_per_class are restated
with every tie rule fixed as a CPU specification in the test infrastructure, and the kernels (csrc/metrics.cu) are compared
against it: the TP masks bit for bit, the metrics to 1e-9.  The one deliberate difference: records of equal confidence keep
their order (stable sort; ultralytics sorts unstably).  Boxes stay in the model's input pixels (no scale_boxes: frames are
resized, not letterboxed).

Cost model: ``update`` is one kernel launch per batch and never reads the device from the host (the record buffer grows on
the host-known bound sum(B * max_det), with a stream-ordered device copy); ``compute`` sorts the records once, runs the
finalisation kernels and reads ONE small tensor back.  The stock route copies every image's IoU matrix to numpy.
"""
import torch
import torch.distributed as dist

from ._lib import call, ptr, require_cuda, stream_ptr

KEYS = ("metrics/precision(B)", "metrics/recall(B)", "metrics/mAP50(B)", "metrics/mAP50-95(B)", "fitness")
_SENTINEL = (1 << 63) - 1          # sort key of an unused record slot: past every class
_HEAD = 8                          # out[0..7] = mp, mr, map50, map50-95, fitness, classes present, F1 argmax, errors


class DetMetrics:
    """Accumulates detection records over an evaluation.  `nc` = number of classes of the model; IoU thresholds are
    ultralytics' torch.linspace(0.5, 0.95, 10)."""

    def __init__(self, nc, device="cuda", capacity=1 << 16):
        self.nc, self.device = int(nc), torch.device(device)
        if self.device.type == "cuda" and self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.iouv = torch.linspace(0.5, 0.95, 10).to(self.device)
        self._ticket = torch.zeros(1, device=self.device, dtype=torch.int32)
        self._cap = 0
        self._grow(int(capacity), 0)
        self.reset()

    def _alloc(self, cap):
        d = self.device
        return (torch.empty(cap, device=d, dtype=torch.float32), torch.empty(cap, device=d, dtype=torch.int32),
                torch.zeros(cap, device=d, dtype=torch.int16), torch.full((cap,), _SENTINEL, device=d, dtype=torch.int64))

    def _grow(self, cap, keep):
        new = self._alloc(cap)
        if keep:
            for dst, src in zip(new, (self.conf, self.cls, self.tp, self.key)):
                dst[:keep].copy_(src[:keep])          # device-to-device, stream-ordered: no host read
        self.conf, self.cls, self.tp, self.key = new
        self._cap = cap

    def reset(self):
        self.key.fill_(_SENTINEL)
        self.cursor = torch.zeros(1, device=self.device, dtype=torch.int64)
        self.n_gt = torch.zeros(self.nc, device=self.device, dtype=torch.int64)
        self.err = torch.zeros(1, device=self.device, dtype=torch.int32)
        self.bound = 0                                # host-known upper bound of the records written so far

    def update(self, rows, counts, padded_targets, img_hw):
        """rows fp32 [B, max_det, 6] and counts int32 [B] (``non_max_suppression_padded``), padded_targets =
        ``pad_targets(...)`` = (cls [B, M], xywh [B, M, 4] normalised, valid [B, M]) on the host or the device, img_hw =
        (H, W) of the model input.  One kernel launch, no host synchronisation."""
        require_cuda(rows, counts)
        b, max_det = int(rows.shape[0]), int(rows.shape[1])
        if tuple(rows.shape[2:]) != (6,) or tuple(counts.shape) != (b,):
            raise ValueError(f"rows must be [B, max_det, 6] and counts [B]; got {tuple(rows.shape)}, {tuple(counts.shape)}")
        dev = rows.device
        if dev != self.device:
            raise ValueError(f"detections on {dev}, metrics on {self.device}")
        gcls, gbox, gvalid = padded_targets
        gcls = gcls.to(dev, non_blocking=True).long().contiguous()
        gbox = gbox.to(dev, non_blocking=True).float().contiguous()
        gvalid = gvalid.to(dev, non_blocking=True).to(torch.uint8).contiguous()
        if gcls.shape[0] != b:
            raise ValueError(f"{gcls.shape[0]} target rows for a batch of {b}")
        need = self.bound + b * max_det
        if need > self._cap:
            self._grow(max(need, 2 * self._cap), self.bound)
        h, w = img_hw
        require_cuda(rows, counts, gcls, gbox, gvalid)
        call("snn_det_match", ptr(rows.float().contiguous()), ptr(counts.int().contiguous()), b, max_det, ptr(gcls), ptr(gbox),
             ptr(gvalid), int(gcls.shape[1]), float(w), float(h), ptr(self.iouv), self.nc, ptr(self.conf), ptr(self.cls),
             ptr(self.tp), ptr(self.key), self._cap, ptr(self.cursor), ptr(self._ticket), ptr(self.n_gt), ptr(self.err),
             stream_ptr())
        self.bound = need

    def records(self):
        """(conf, cls, tp [n, 10] bool) of the records so far, in record order (reads the count from the device)."""
        n = int(self.cursor.item())
        bits = self.tp[:n].int()
        tp = ((bits[:, None] >> torch.arange(10, device=self.device)) & 1).bool()
        return self.conf[:n], self.cls[:n], tp

    def _gathered(self, process_group):
        """Every rank's records, concatenated in rank order, and the summed gt histogram / error count (DDP)."""
        world = dist.get_world_size(process_group)
        counts = [torch.zeros(1, device=self.device, dtype=torch.int64) for _ in range(world)]
        dist.all_gather(counts, self.cursor, group=process_group)
        n = [int(c) for c in torch.cat(counts).cpu()]          # the host read of the gather
        pad = max(max(n), 1)
        # TP masks travel as int32: NCCL has no 16-bit integer type
        key = torch.full((pad,), _SENTINEL, device=self.device, dtype=torch.int64)
        tp = torch.zeros(pad, device=self.device, dtype=torch.int32)
        mine = min(pad, self._cap)
        key[:mine].copy_(self.key[:mine])
        tp[:mine].copy_(self.tp[:mine])
        keys = [torch.empty_like(key) for _ in range(world)]
        tps = [torch.empty_like(tp) for _ in range(world)]
        dist.all_gather(keys, key, group=process_group)
        dist.all_gather(tps, tp, group=process_group)
        key = torch.cat([k[:c] for k, c in zip(keys, n)])
        tp = torch.cat([t[:c] for t, c in zip(tps, n)]).to(torch.int16)
        n_gt, err = self.n_gt.clone(), self.err.clone()
        dist.all_reduce(n_gt, group=process_group)
        dist.all_reduce(err, group=process_group)
        return key, tp, n_gt, err

    def compute(self, process_group=None):
        """Results dict of ultralytics DetMetrics (precision, recall, mAP50, mAP50-95 and fitness = 0.1 mAP50 + 0.9
        mAP50-95), plus "ap" [classes with targets, 10] and "ap_class_index".  With a process group every rank gets the
        result over all ranks' records (rank-major order).  A distributed sampler that pads its shards (ShardedSampler,
        DistributedSampler) repeats samples, and the repeats are counted like any other image.
        Without a process group the sort and the finalisation cover the host-known bound sum(B * max_det) of record slots,
        not the device's record count: reading that count first would cost a host synchronisation before the sort.  Unused
        slots hold a sort key past every class, so they land at the end and are never part of a class segment; at a high
        NMS confidence threshold most of the bound is such padding, which costs sort time but changes no result."""
        if process_group is not None:
            key, tp, n_gt, err = self._gathered(process_group)
        else:
            key, tp, n_gt, err = self.key[:max(self.bound, 1)], self.tp, self.n_gt, self.err
        n = int(key.shape[0])
        sorted_key, order = torch.sort(key, stable=True)
        curves = torch.empty((2, self.nc, 1000), device=self.device, dtype=torch.float64)
        out = torch.empty(_HEAD + 11 * self.nc, device=self.device, dtype=torch.float64)
        require_cuda(sorted_key, order, tp, n_gt, err, curves, out)
        call("snn_det_metrics_finalize", ptr(sorted_key), ptr(order), ptr(tp), n, ptr(n_gt), self.nc, ptr(err), ptr(curves),
             ptr(out), stream_ptr())
        host = out.cpu()                                       # the one host read of an evaluation
        if host[7] != 0:
            raise ValueError(f"{int(host[7])} detection records or targets had a class outside [0, {self.nc}) "
                             "(or the record buffer overflowed)")
        res = {k: float(host[i]) for i, k in enumerate(KEYS)}
        present = host[_HEAD + 10 * self.nc:] != 0
        res["ap"] = host[_HEAD:_HEAD + 10 * self.nc].view(self.nc, 10)[present].numpy()
        res["ap_class_index"] = torch.nonzero(present).flatten().numpy()
        return res
