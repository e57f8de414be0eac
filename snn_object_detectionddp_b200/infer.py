"""Inference path of the reference (visualize.py:48-109 batch-1, eval_2.py:96-112 batch-N): T-frame unroll in eval mode,
Detect decode, non-maximum suppression -- on the B200 kernels.

    windowed (what the reference does: state reset per window, visualize.py:66):
        dets = detect_sequence(model, frames[B,T,3,H,W], conf_thres=0.3, iou_thres=0.45, multi_label=True)
    streaming (extension; NOT identical to windowed reset -- membranes and the ConvLSTM state carry over):
        det = StreamingDetector(model, ...);  for chunk in video: dets = det(chunk)
"""
import torch

from . import kernels as K
from .nms import non_max_suppression, non_max_suppression_padded


@torch.no_grad()
def decode_last_step(model, frames, hidden_state=None, return_state=False):
    """Eval-mode fused forward over [B,T,3,H,W]; returns (prediction [B, 4+nc, A] as ultralytics' Detect returns it in
    eval mode, hidden).  The decode is the ``snn_detect_decode`` kernel (DFL expectation, dist2bbox, x stride, sigmoid)."""
    was_training = model.training
    model.eval()
    try:
        det, hidden = model.forward_sequence(frames, hidden_state, return_state=return_state)
    finally:
        model.train(was_training)
    return decode_head(model, det), hidden


@torch.no_grad()
def decode_head(model, det):
    """Detect-head output of an eval-mode forward -> prediction [B, 4+nc, A] (xywh pixels + class scores)."""
    head = model.detection_head
    distri, scores = det.flat()
    from .head import make_anchors
    anchors, strides = make_anchors(det.shapes(), head.stride.tolist(), 0.5, device=distri.device)
    boxes, probs = K.detect_decode(distri.contiguous(), scores.contiguous(), anchors.contiguous(), strides.view(-1).contiguous(),
                                   xywh=True)
    return torch.cat((boxes, probs), 2).permute(0, 2, 1).contiguous()


@torch.no_grad()
def detect_sequence(model, frames, conf_thres=0.3, iou_thres=0.45, multi_label=True, agnostic=False, max_det=300,
                    hidden_state=None, return_state=False, padded=False):
    """One window of frames -> per-image detections [n, 6] (x1, y1, x2, y2, conf, cls) of the LAST frame."""
    pred, hidden = decode_last_step(model, frames, hidden_state, return_state)
    if padded:
        out = non_max_suppression_padded(pred, conf_thres, iou_thres, agnostic, multi_label, max_det)
    else:
        out = non_max_suppression(pred, conf_thres, iou_thres, agnostic=agnostic, multi_label=multi_label, max_det=max_det)
    return (out, hidden) if return_state else out


class StreamingDetector:
    """Carries the ConvLSTM state and the LIF membranes across calls (documented extension: the reference resets the
    state for every window).  `reset()` restores windowed behaviour."""

    def __init__(self, model, conf_thres=0.3, iou_thres=0.45, multi_label=True, agnostic=False, max_det=300):
        self.model, self.kw = model, dict(conf_thres=conf_thres, iou_thres=iou_thres, multi_label=multi_label,
                                          agnostic=agnostic, max_det=max_det)
        self.hidden = None

    def reset(self):
        self.hidden = None

    def __call__(self, frames):
        if frames.dim() == 4:
            frames = frames[:, None]
        out, self.hidden = detect_sequence(self.model, frames, hidden_state=self.hidden, return_state=True, **self.kw)
        return out


class GraphedWindowDetector:
    """`detect_sequence(..., padded=True)` replayed from ONE CUDA graph (static window shape): the ~250 launches of an
    eval window cost ~6 ms of host time eagerly whatever the batch size, a replay is bounded by the GPU.  Returns the
    graph's static (rows [B,max_det,6], kept [B,max_det], counts [B]) device tensors: read them before the next call."""

    def __init__(self, model, conf_thres=0.3, iou_thres=0.45, multi_label=True, agnostic=False, max_det=300, warmup=2):
        self.model, self.warmup = model, warmup
        self.kw = dict(conf_thres=conf_thres, iou_thres=iou_thres, multi_label=multi_label, agnostic=agnostic, max_det=max_det)
        self._graph = self._key = self._in = self._out = None

    @torch.no_grad()
    def __call__(self, frames):
        stats = getattr(self.model, "spike_stats", None)
        key = (tuple(frames.shape), frames.dtype, frames.device, stats)     # holds the stats: its counters outlive the graph
        if self._graph is None or key != self._key:
            saved = None if stats is None else stats.counts.clone()
            for _ in range(self.warmup):
                detect_sequence(self.model, frames, padded=True, **self.kw)
            if saved is not None:
                stats.counts.copy_(saved)          # the warm-up windows are not part of what the caller counts
            self._in = frames.clone()
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._out = detect_sequence(self.model, self._in, padded=True, **self.kw)
            self._graph, self._key = g, key
        self._in.copy_(frames, non_blocking=True)
        self._graph.replay()
        return self._out
