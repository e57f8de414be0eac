"""Host-side mirror of the reference's model.py: same class names, constructor arguments, attribute /
parameter names and forward signatures -- compute is the libsnnb200 CUDA kernels.

    ConvBlock (ref model.py:9-18)      conv -> BN -> {LIF | SiLU}    one fused autograd op over all T steps
    DownBlock (ref model.py:20-30), UpBlock (ref model.py:32-48), ConvLSTM2d (ref model.py:50-71)
    TemporalUNet (ref model.py:100-146), YOLOFeatureExtractor (ref model.py:74-98), YOLOTemporalUNet
    (ref model.py:148-211)

Two entry styles:
  * drop-in, per frame:   ``preds, hidden = model(frame[B,3,H,W], hidden)``  (train.py:64-66 loop works unchanged;
    NCHW fp32 tensors in/out; LIF membranes travel inside the opaque ``hidden``)
  * fused, per sequence:  ``model.forward_sequence(frames[B,T,3,H,W])`` runs layer-by-layer over the folded
    T*B batch (valid because layer l at step t needs only layer l-1 at step t and its own state at t-1;
    SURVEY.md 7.4-2); per-timestep BatchNorm statistics are kept so the numbers equal the per-frame loop.

`neuron='lif'` is the BUILD-DEFINED spiking variant (the reference has no LIF; SURVEY.md section 0);
`neuron='silu'` reproduces the reference network itself.
"""
import math
import os
from types import SimpleNamespace

import torch
import torch.nn as nn

from . import kernels as K
from .ops import BilinearResizeFn, ConvBiasFn, ConvBNActFn, ConvLSTMSeqFn, GradSlot, NeuronCfg, PadEvenFn
from .params import store_for
from ._lib import GEOM_1x1, GEOM_3x3_S1, GEOM_3x3_S2, GEOM_T2x2_S2


class RunCtx:
    """Per-call context handed down the module tree."""

    def __init__(self, store, T, want_state=False, want_mask=False, fp32_outputs=False, live_T=None):
        self.store, self.T, self.want_state, self.want_mask, self.fp32_outputs = store, T, want_state, want_mask, fp32_outputs
        self.record = None      # optional dict: ConvBlock name -> its spike / activation output (tests, spike-rate probes)
        # number of trailing timesteps whose head outputs are consumed (train.py:64-66 keeps only the LAST preds): layers
        # WITHOUT temporal state (U-Net output 1x1 convs, Detect head) still run forward on every frame -- their
        # BatchNorm running statistics advance per frame as in the reference -- but skip the all-zero backward of the
        # dead frames.  None = every timestep is live.
        self.live_T = live_T
        self.spike_stats = None     # spikes.SpikeStats the LIF ConvBlocks count into (None: uncounted launches)


def _to_nhwc_bf16(x):
    """NCHW fp32 (reference layout) -> NHWC bf16, differentiable (drop-in path only)."""
    return x.permute(0, 2, 3, 1).to(torch.bfloat16).contiguous()


def _to_nchw_f32(x):
    return x.float().permute(0, 3, 1, 2)


def make_neuron(neuron):
    if isinstance(neuron, NeuronCfg):
        return neuron
    if neuron is None:
        return NeuronCfg("lif")
    if isinstance(neuron, str):
        return NeuronCfg(neuron)
    d = dict(neuron)
    return NeuronCfg(d.get("type", "lif"), d.get("beta", 0.5), d.get("v_th", 1.0), d.get("alpha", 2.0))


# ----------------------------------------------------------------------------------------------
class ConvBlock(nn.Module):
    """Conv2d(bias=False) -> BatchNorm2d -> neuron.  `conv` / `bn` are parameter containers (same state_dict keys
    as the reference); they are never called."""

    def __init__(self, in_channels, out_channels, kernel_size=3, stride=1, padding=1, neuron=None, groups=1,
                 bn_eps=1e-5, bn_momentum=0.1):
        super().__init__()
        self.conv = nn.Conv2d(in_channels, out_channels, kernel_size, stride, padding, groups=groups, bias=False)
        self.bn = nn.BatchNorm2d(out_channels, eps=bn_eps, momentum=bn_momentum)
        self.neuron = make_neuron(neuron)
        if groups > 1:
            assert groups == in_channels == out_channels and kernel_size == 3 and stride == 1 and padding == 1
            self.geom = K.GEOM_DW3x3
        elif kernel_size == 3 and padding == 1 and stride in (1, 2):
            self.geom = GEOM_3x3_S1 if stride == 1 else GEOM_3x3_S2
        elif kernel_size == 1 and padding == 0 and stride == 1:
            self.geom = GEOM_1x1
        else:
            raise NotImplementedError("ConvBlock supports k3/p1/s{1,2}, k1/p0/s1 and depthwise k3 (the shapes on the path)")
        self.last_mask = None

    def forward_seq(self, rc, x0, x1=None, v_init=None, dead_frames_ok=False, slot_x0=None):
        """dead_frames_ok: the caller guarantees this block's output reaches the loss only through the last rc.live_T
        timesteps and feeds nothing with temporal state (true for the Detect head, NOT for U-Net blocks: the encoder
        feeds the ConvLSTM and LIF blocks carry membranes)."""
        cfg = dict(store=rc.store, geom=self.geom, T=rc.T, bn=self.bn, neuron=self.neuron, training=self.training,
                   want_state=rc.want_state, want_mask=rc.want_mask)
        if dead_frames_ok and rc.live_T is not None and self.neuron.kind == "silu" and rc.live_T < rc.T:
            cfg["live_T"] = rc.live_T
            cfg["dead_grad_unread"] = getattr(rc, "dead_grad_unread", False)
        if slot_x0 is not None:
            cfg["slot_x0"] = slot_x0          # (GradSlot, 'first' | 'last'): see ops.GradSlot
        if rc.spike_stats is not None and self.neuron.kind == "lif":
            cfg["spike_counts"] = rc.spike_stats.layer_counts(self._snn_name, rc.T)
        if self.geom == GEOM_3x3_S2 and ((x0.shape[1] | x0.shape[2]) & 1):
            # odd H or W (e.g. the 15x20 P5 level of a 480x640 frame): zero-pad to even -- the extra row / column is exactly
            # the conv's own padding, so Ho = ceil(H/2) and the values equal nn.Conv2d(k3, s2, p1) on the odd-sized map
            assert x1 is None
            x0 = PadEvenFn.apply(x0)
        out, v = ConvBNActFn.apply(x0, x1, v_init, self.conv.weight, self.bn.weight, self.bn.bias, cfg)
        if rc.want_mask:
            self.last_mask = cfg.get("last_mask")
        if rc.record is not None:
            rc.record[getattr(self, "_snn_name", str(id(self)))] = out.detach()
        return out, v

    def forward(self, x):
        """Drop-in single call on NCHW fp32 (zero initial membrane)."""
        st = store_for(self, x.device)
        st.refresh_operands()
        out, _ = self.forward_seq(RunCtx(st, 1), _to_nhwc_bf16(x))
        return _to_nchw_f32(out)


class DownBlock(nn.Module):
    def __init__(self, in_channels, out_channels, neuron=None):
        super().__init__()
        self.conv1 = ConvBlock(in_channels, out_channels, stride=2, neuron=neuron)
        self.conv2 = ConvBlock(out_channels, out_channels, neuron=neuron)

    def forward_seq(self, rc, x, v=None, slot_x=None):
        v = v or (None, None)
        if slot_x is not None and ((x.shape[1] | x.shape[2]) & 1):
            slot_x = None                       # odd map: the consumer of x is the pad op, not the conv
        x, v1 = self.conv1.forward_seq(rc, x, None, v[0], slot_x0=slot_x)
        x, v2 = self.conv2.forward_seq(rc, x, None, v[1])
        return x, (v1, v2)

    def forward(self, x):
        st = store_for(self, x.device)
        st.refresh_operands()
        out, _ = self.forward_seq(RunCtx(st, 1), _to_nhwc_bf16(x))
        return _to_nchw_f32(out)


class UpBlock(nn.Module):
    def __init__(self, in_channels, skip_channels, out_channels, neuron=None):
        super().__init__()
        self.up = nn.ConvTranspose2d(in_channels, in_channels // 2, kernel_size=2, stride=2)
        self.conv1 = ConvBlock(in_channels // 2 + skip_channels, out_channels, neuron=neuron)
        self.conv2 = ConvBlock(out_channels, out_channels, neuron=neuron)

    def forward_seq(self, rc, x, skip, v=None, slot_x=None, slot_skip=None):
        v = v or (None, None)
        cfg_up = dict(store=rc.store, geom=GEOM_T2x2_S2)
        if slot_x is not None:
            cfg_up["slot_x0"] = slot_x
        up = ConvBiasFn.apply(x, self.up.weight, self.up.bias, cfg_up)
        if up.shape[1:3] != skip.shape[1:3]:
            # reference model.py:43-44: F.interpolate(skip_x, size=x.shape[2:], mode='bilinear', align_corners=False)
            skip = BilinearResizeFn.apply(skip, (up.shape[1], up.shape[2]))
            slot_skip = None                    # the consumer of the skip tensor is the resize op, not the conv
        x, v1 = self.conv1.forward_seq(rc, skip, up, v[0], slot_x0=slot_skip)      # cat([skip_x, x]) order of model.py:45
        x, v2 = self.conv2.forward_seq(rc, x, None, v[1])
        return x, (v1, v2)

    def forward(self, x, skip_x):
        st = store_for(self, x.device)
        st.refresh_operands()
        out, _ = self.forward_seq(RunCtx(st, 1), _to_nhwc_bf16(x), _to_nhwc_bf16(skip_x))
        return _to_nchw_f32(out)


class ConvLSTM2d(nn.Module):
    def __init__(self, in_channels, hidden_channels, kernel_size=3):
        super().__init__()
        assert kernel_size == 3
        self.hidden_channels = hidden_channels
        self.conv = nn.Conv2d(in_channels + hidden_channels, 4 * hidden_channels, kernel_size,
                              padding=kernel_size // 2, bias=True)

    def forward_seq(self, rc, x, state=None):
        """x bf16 [T*B,h,w,Cin]; state = (h, c) fp32 NHWC [B,h,w,Ch] or None. Returns h_all bf16, (h_T, c_T)."""
        h0, c0 = state if state is not None else (None, None)
        cfg = dict(store=rc.store, T=rc.T, bias=self.conv.bias)
        h_all, h_last, c_last = ConvLSTMSeqFn.apply(x, h0, c0, self.conv.weight, self.conv.bias, cfg)
        return h_all, (h_last, c_last)

    def forward(self, x, hidden_state=None):
        st = store_for(self, x.device)
        st.refresh_operands()
        state = None
        if hidden_state is not None:
            state = tuple(s.permute(0, 2, 3, 1).contiguous() for s in hidden_state)
        h_all, (h, c) = self.forward_seq(RunCtx(st, 1), _to_nhwc_bf16(x), state)
        h, c = h.permute(0, 3, 1, 2), c.permute(0, 3, 1, 2)
        return h, (h, c)


# ----------------------------------------------------------------------------------------------
class TemporalUNet(nn.Module):
    """U-Net with ConvLSTM bottleneck (reference model.py:100-146)."""

    def __init__(self, feature_channels, use_conv_lstm=True, neuron=None, widths=(128, 256, 512, 1024)):
        super().__init__()
        if not use_conv_lstm:
            raise NotImplementedError("use_conv_lstm=False (nn.LSTM bottleneck, model.py:114) is outside the B200 hot path")
        ch_p3, ch_p4, ch_p5 = feature_channels
        w1, w2, w3, w4 = widths
        self.use_conv_lstm = use_conv_lstm
        nr = make_neuron(neuron)
        self.neuron = nr
        # fan-out gradients (skips, decoder -> output conv) summed in the second dgrad's epilogue (ops.GradSlot); False = autograd adds
        self.fuse_fanout_grads = os.environ.get("SNN_FUSE_FANOUT_GRADS", "1") != "0"
        self.enc1, self.down1 = ConvBlock(ch_p3, w1, neuron=nr), DownBlock(w1, w2, neuron=nr)
        self.enc2, self.down2 = ConvBlock(w2 + ch_p4, w2, neuron=nr), DownBlock(w2, w3, neuron=nr)
        self.enc3, self.down3 = ConvBlock(w3 + ch_p5, w3, neuron=nr), DownBlock(w3, w4, neuron=nr)
        self.lstm = ConvLSTM2d(w4, w4)
        self.bottleneck_conv = ConvBlock(w4, w4, neuron=nr)
        self.up1, self.up2, self.up3 = UpBlock(w4, w3, w3, neuron=nr), UpBlock(w3, w2, w2, neuron=nr), UpBlock(w2, w1, w1, neuron=nr)
        self.out_p5, self.out_p4, self.out_p3 = nn.Conv2d(w3, ch_p5, 1), nn.Conv2d(w2, ch_p4, 1), nn.Conv2d(w1, ch_p3, 1)
        for name, m in self.named_modules():
            if isinstance(m, ConvBlock):
                m._snn_name = name

    # state = (lstm_state | None, {block name: membrane(s)})
    def forward_seq(self, rc, feats, state=None):
        p3, p4, p5 = feats
        lstm_state, m = state if state is not None else (None, {})
        nm = {}
        # Tensors with two consumers (x1, x2, x3: next encoder stage + decoder skip; d1, d2: next decoder stage + output
        # conv): their two input gradients are summed in the second dgrad's epilogue (ops.GradSlot) instead of by an
        # autograd add kernel.  'first' = the consumer created later in forward = whose backward runs first.
        fuse = torch.is_grad_enabled() and self.training and self.fuse_fanout_grads
        s1, s2, s3, sd1, sd2 = (GradSlot() if fuse else None for _ in range(5))
        role = lambda s_, r_: None if s_ is None else (s_, r_)
        x1, nm["enc1"] = self.enc1.forward_seq(rc, p3, None, m.get("enc1"))
        d, nm["down1"] = self.down1.forward_seq(rc, x1, m.get("down1"), slot_x=role(s1, "last"))
        x2, nm["enc2"] = self.enc2.forward_seq(rc, d, p4, m.get("enc2"))          # cat([down1(x1), p4]) model.py:126
        d, nm["down2"] = self.down2.forward_seq(rc, x2, m.get("down2"), slot_x=role(s2, "last"))
        x3, nm["enc3"] = self.enc3.forward_seq(rc, d, p5, m.get("enc3"))          # model.py:127
        x, nm["down3"] = self.down3.forward_seq(rc, x3, m.get("down3"), slot_x=role(s3, "last"))
        h_all, new_lstm = self.lstm.forward_seq(rc, x, lstm_state)
        x, nm["bottleneck_conv"] = self.bottleneck_conv.forward_seq(rc, h_all, None, m.get("bottleneck_conv"))
        od = torch.float32 if rc.fp32_outputs else torch.bfloat16
        live_n = None if (rc.live_T is None or rc.live_T >= rc.T) else rc.live_T * (p3.shape[0] // rc.T)

        def out_conv(conv, x_, slot):
            cfg = dict(store=rc.store, geom=GEOM_1x1, out_dtype=od, live_n=live_n)
            if slot is not None:
                cfg["slot_x0"] = slot
            return ConvBiasFn.apply(x_, conv.weight, conv.bias, cfg)

        # each output conv is applied right after its decoder level (model.py:146 applies them at the end; the values are the
        # same): it is then created BEFORE the next up-block, its backward runs AFTER it and can add its live-frame gradient
        # into the buffer the up-block's dgrad has written -- no zero-filled full-size gradient for the dead frames.
        d1, nm["up1"] = self.up1.forward_seq(rc, x, x3, m.get("up1"), slot_skip=role(s3, "first"))
        o5 = out_conv(self.out_p5, d1, role(sd1, "last"))
        d2, nm["up2"] = self.up2.forward_seq(rc, d1, x2, m.get("up2"), slot_x=role(sd1, "first"), slot_skip=role(s2, "first"))
        o4 = out_conv(self.out_p4, d2, role(sd2, "last"))
        d3, nm["up3"] = self.up3.forward_seq(rc, d2, x1, m.get("up3"), slot_x=role(sd2, "first"), slot_skip=role(s1, "first"))
        o3 = out_conv(self.out_p3, d3, None)
        return (o3, o4, o5), (new_lstm, nm)

    def spike_fanout(self, feature_hw):
        """{LIF ConvBlock name: F}, F = multiply-accumulates one element of that block's spike output drives, summed over the
        convs that consume it AS SPIKES (borders ignored: the per-element share of the dense MACs).  feature_hw = the (H, W)
        of p3, p4, p5.  Mirrors forward_seq's wiring: the zero pad in front of a stride-2 conv on an odd map adds no spikes
        (its conv still counts); a skip that UpBlock resizes bilinearly is no longer binary (its conv1 K-slice does not
        count); the ConvLSTM h, the transposed-conv outputs and the extractor features are not spikes."""
        if self.neuron.kind != "lif":
            return {}
        half = lambda hw: ((hw[0] + 1) // 2, (hw[1] + 1) // 2)
        hw3, hw4, hw5 = (tuple(int(v) for v in hw) for hw in feature_hw)
        hw_b = half(hw5)                                   # down3 output = ConvLSTM / bottleneck map
        hw_u1 = (2 * hw_b[0], 2 * hw_b[1])
        hw_u2 = (2 * hw_u1[0], 2 * hw_u1[1])
        hw_u3 = (2 * hw_u2[0], 2 * hw_u2[1])
        f = {}

        def edge(src, consumer):
            f[src] = f.get(src, 0.0) + _fanout(consumer)

        edge("enc1", self.down1.conv1.conv)
        edge("down1.conv1", self.down1.conv2.conv)
        edge("down1.conv2", self.enc2.conv)
        edge("enc2", self.down2.conv1.conv)
        edge("down2.conv1", self.down2.conv2.conv)
        edge("down2.conv2", self.enc3.conv)
        edge("enc3", self.down3.conv1.conv)
        edge("down3.conv1", self.down3.conv2.conv)
        edge("down3.conv2", self.lstm.conv)                # the W_x K-slice of the gate conv
        edge("bottleneck_conv", self.up1.up)
        for up, skip, hw_skip, hw_up, out_conv in ((self.up1, "enc3", hw5, hw_u1, self.out_p5),
                                                   (self.up2, "enc2", hw4, hw_u2, self.out_p4),
                                                   (self.up3, "enc1", hw3, hw_u3, self.out_p3)):
            if hw_skip == hw_up:
                edge(skip, up.conv1.conv)
            edge(up.conv1._snn_name, up.conv2.conv)
            edge(up.conv2._snn_name, out_conv)
        edge("up1.conv2", self.up2.up)
        edge("up2.conv2", self.up3.up)
        return f

    def forward(self, features, hidden_state=None):
        """Drop-in: features = 3 NCHW fp32 maps; hidden_state = None | (h, c) | (h, c, membranes)."""
        p3 = features[0]
        st = store_for(self, p3.device)
        st.refresh_operands()
        state = _unpack_hidden(hidden_state)
        rc = RunCtx(st, 1, want_state=True, fp32_outputs=True)
        outs, new_state = self.forward_seq(rc, tuple(_to_nhwc_bf16(f) for f in features), state)
        return tuple(o.permute(0, 3, 1, 2) for o in outs), _pack_hidden(new_state, self.neuron.kind)


def _fanout(conv):
    """Multiply-accumulates one input element of `conv` drives (borders ignored): Cout/groups * kh * kw / (sh * sw) for a
    Conv2d, Cout/groups * kh * kw for a ConvTranspose2d (every input pixel feeds each tap once)."""
    kh, kw = conv.kernel_size
    n = conv.out_channels // conv.groups * kh * kw
    if isinstance(conv, nn.ConvTranspose2d):
        return float(n)
    return n / (conv.stride[0] * conv.stride[1])


def _unpack_hidden(hidden_state):
    if hidden_state is None:
        return None
    h, c = hidden_state[0], hidden_state[1]
    mem = hidden_state[2] if len(hidden_state) > 2 else {}
    return (h.permute(0, 2, 3, 1).contiguous(), c.permute(0, 2, 3, 1).contiguous()), mem


def _pack_hidden(state, kind):
    (h, c), mem = state
    h, c = h.permute(0, 3, 1, 2), c.permute(0, 3, 1, 2)   # NCHW-shaped views, as the reference returns
    return (h, c) if kind == "silu" else (h, c, mem)


# ----------------------------------------------------------------------------------------------
def _load_ultralytics_model(model_name):
    """The reference's backbone (model.py:78: `YOLO(model_name).model`) when the `ultralytics` package AND the weights file
    are obtainable; None otherwise (offline image: neither is)."""
    try:
        from ultralytics import YOLO          # un-vendored third party, see SURVEY.md 8c
    except Exception:
        return None
    try:
        return YOLO(model_name).model
    except Exception as e:                    # package present but weights missing / download impossible
        import warnings
        warnings.warn(f"ultralytics is importable but YOLO({model_name!r}) failed ({type(e).__name__}: {e}); "
                      "using the stand-in feature pyramid")
        return None


class YOLOFeatureExtractor(nn.Module):
    """Frozen multi-scale feature source (reference model.py:74-98).

    backend 'ultralytics' -- what the reference does: `self.model = YOLO(model_name).model`, frozen, always in eval mode,
        `forward(x)` returns the three raw head inputs of `_, features = self.model(x)` (model.py:88-91).  Used whenever
        the package and the weights are importable/loadable (backend='auto', the default).  The frozen third-party net
        runs through its own PyTorch kernels (it is not a kernel target, SURVEY.md 8f-1); its NCHW fp32 maps are repacked
        to the NHWC bf16 layout of the B200 path by one libsnnb200 kernel per level.
    backend 'standin' -- neither the package nor `yolo11m.pt` can exist offline: a deterministic, frozen, randomly
        initialised stride-8/16/32 pyramid with the same interface, run with the tensor-core kernels under no_grad:
        pack 8x8 patches -> 1x1 conv 192->128 + SiLU -> [P3 = 1x1 ->144]
        3x3 s2 128->128 + SiLU -> [P4 = 1x1 ->144];  3x3 s2 + SiLU -> [P5 = 1x1 ->144]
    """
    WIDTH = 128
    OUT = 144

    def __init__(self, model_name="yolo11m.pt", freeze=True, seed=1234, backend="auto"):
        super().__init__()
        assert backend in ("auto", "ultralytics", "standin")
        self.model_name = model_name
        real = _load_ultralytics_model(model_name) if backend in ("auto", "ultralytics") else None
        if backend == "ultralytics" and real is None:
            raise RuntimeError("backend='ultralytics' requested but `ultralytics` / the weights are not available")
        self.backend = "ultralytics" if real is not None else "standin"
        if real is not None:
            self.model = real                              # same attribute name as the reference: state_dict keys match
            if freeze:
                for p in self.model.parameters():
                    p.requires_grad = False
                self.model.eval()
            return
        g = torch.Generator().manual_seed(seed)
        w, o = self.WIDTH, self.OUT

        def mk(rows, taps, k):
            return (torch.randn(rows, taps, k, generator=g) * math.sqrt(2.0 / (taps * k))).to(torch.bfloat16)

        for name, t in (("w_stem", mk(w, 1, 192)), ("w_d4", mk(w, 9, w)), ("w_d5", mk(w, 9, w)),
                        ("w_p3", mk(o, 1, w)), ("w_p4", mk(o, 1, w)), ("w_p5", mk(o, 1, w))):
            self.register_buffer(name, t, persistent=False)
        self.register_buffer("_one", torch.ones(1, w), persistent=False)
        self.register_buffer("_zero", torch.zeros(1, w), persistent=False)

    def train(self, mode=True):          # stays in eval like the reference (model.py:84-86)
        self.training = mode
        if self.backend == "ultralytics":
            self.model.eval()
        return self

    @torch.no_grad()
    def get_feature_channels(self, dummy_input_shape=(1, 3, 640, 640)):
        if self.backend == "standin":
            return [self.OUT] * 3
        dummy = torch.randn(*dummy_input_shape, device=next(self.model.parameters()).device)     # model.py:94-98
        _, features = self.model(dummy)
        return [f.shape[1] for f in features]

    @torch.no_grad()
    def forward_seq(self, frames, B, T):
        """frames fp32 in [0,1] or uint8 [B,T,3,H,W] (or [B,3,H,W] with T=1) contiguous -> (p3, p4, p5) bf16 NHWC [T*B, ...]
        (timestep-major folded batch)."""
        H, W = frames.shape[-2:]
        if self.backend == "ultralytics":
            x = frames.reshape(B, T, 3, H, W).transpose(0, 1).reshape(T * B, 3, H, W)
            x = x.float() / 255.0 if x.dtype == torch.uint8 else x.float()
            _, features = self.model(x)
            return tuple(K.nchw_to_nhwc(f.float()) for f in features)
        if H % 8 or W % 8:
            raise ValueError(f"frame size {H}x{W}: H and W must be multiples of 8 (stride-8 patch packer of the stand-in pyramid)")
        x = K.space_to_depth8(frames.contiguous(), B, T)
        act = lambda y: K.bn_act_fwd(K.ACT_SILU, y, self._one, self._zero, 1)[0]

        def even(f):       # odd level size (e.g. 15x20 at 480x640): the zero row / column is the stride-2 conv's own padding
            h, w = f.shape[1], f.shape[2]
            return K.pad_crop(f, (h + (h & 1), w + (w & 1))) if ((h | w) & 1) else f

        f3 = act(K.conv_fprop(GEOM_1x1, x, self.w_stem, self.WIDTH))
        f4 = act(K.conv_fprop(GEOM_3x3_S2, even(f3), self.w_d4, self.WIDTH))
        f5 = act(K.conv_fprop(GEOM_3x3_S2, even(f4), self.w_d5, self.WIDTH))
        bf = torch.bfloat16
        return (K.conv_fprop(GEOM_1x1, f3, self.w_p3, self.OUT, out_dtype=bf),
                K.conv_fprop(GEOM_1x1, f4, self.w_p4, self.OUT, out_dtype=bf),
                K.conv_fprop(GEOM_1x1, f5, self.w_p5, self.OUT, out_dtype=bf))

    @staticmethod
    def feature_hw(H, W):
        """(H, W) of p3, p4, p5 for an H x W frame: stride 8, 16, 32 with every stride-2 stage rounding up."""
        hw, out = (int(H), int(W)), []
        for k in range(5):
            hw = ((hw[0] + 1) // 2, (hw[1] + 1) // 2)
            if k >= 2:
                out.append(hw)
        return out

    def forward(self, x):
        if self.backend == "ultralytics":      # reference model.py:88-91, verbatim semantics
            with torch.no_grad():
                _, features = self.model(x)
            return tuple(features)
        feats = self.forward_seq(x, x.shape[0], 1)
        return tuple(_to_nchw_f32(f) for f in feats)


# ----------------------------------------------------------------------------------------------
class YOLOTemporalUNet(nn.Module):
    """Reference model.py:148-211: frozen extractor -> TemporalUNet -> Detect head.

    Extra (additive) constructor arguments: `neuron` ('lif' default | 'silu' | dict with type/beta/v_th/alpha) and
    `extractor_backend` ('auto': the real ultralytics YOLO when importable, else the stand-in pyramid), so
    `YOLOTemporalUNet(num_classes, yolo_model_name, use_conv_lstm, hyp)` from main.py:126-131 still works.
    """

    def __init__(self, num_classes=80, yolo_model_name="yolo11m.pt", use_conv_lstm=True,
                 hyp: dict = {"box": 7.5, "cls": 0.5, "dfl": 1.5, "reg_max": 16}, neuron=None, extractor_backend="auto"):
        super().__init__()
        from .head import Detect
        self.args = SimpleNamespace(**hyp)
        self.nc = num_classes
        self.feature_extractor = YOLOFeatureExtractor(model_name=yolo_model_name, freeze=True, backend=extractor_backend)
        feature_channels = self.feature_extractor.get_feature_channels()
        self.temporal_unet = TemporalUNet(feature_channels=feature_channels, use_conv_lstm=use_conv_lstm, neuron=neuron)
        self.detection_head = Detect(nc=num_classes, ch=feature_channels)
        strides = torch.tensor([8.0, 16.0, 32.0])
        self.detection_head.stride = strides
        self.detection_head.reg_max = self.args.reg_max
        self.register_buffer("strides", strides, persistent=False)
        self.model = nn.ModuleList([self.detection_head])
        self.skip_dead_backward = True      # see RunCtx.live_T (False: run the all-zero backward of the dead frames too)
        # spikes.SpikeStats: while set, every forward / forward_sequence counts the LIF layers' spikes into it (a plain
        # attribute: never in state_dict; captured CUDA graphs key on it, see Trainer.train_step_graphed)
        self.spike_stats = None

    def _spike_stats_for(self, frames, T):
        """The attached SpikeStats, checked against this forward (T, device, fan-out table) before anything launches."""
        stats = getattr(self, "spike_stats", None)       # None also for a model pickled before the attribute existed
        if stats is not None:
            stats.begin_forward(self.temporal_unet, T, self.feature_extractor.feature_hw(*frames.shape[-2:]), frames.device)
        return stats

    # ---- fused sequence path -------------------------------------------------------------
    def forward_sequence(self, frames, hidden_state=None, return_state=False, all_steps=False, record=None):
        """frames [B,T,3,H,W] fp32 on the GPU.  Returns (HeadOut of the LAST step as in train.py:64-66, hidden);
        `hidden` is None unless return_state (final LSTM state + LIF membranes, for streaming inference).
        `record`: optional dict that receives every ConvBlock's output (spikes) by module name (flip-rate reports)."""
        B, T = frames.shape[0], frames.shape[1]
        stats = self._spike_stats_for(frames, T)
        st = store_for(self, frames.device)
        st.refresh_operands()
        feats = self.feature_extractor.forward_seq(frames, B, T)
        rc = RunCtx(st, T, want_state=return_state, live_T=None if (all_steps or not self.skip_dead_backward) else 1)
        rc.spike_stats = stats
        # the head's inputs are produced by the U-Net output convs, which slice the dead frames' gradient away themselves:
        # head-internal gradients of the dead frames are never read and need no zero fill
        rc.dead_grad_unread = rc.live_T is not None
        rc.record = record
        outs, new_state = self.temporal_unet.forward_seq(rc, feats, _unpack_hidden(hidden_state))
        det = self.detection_head.forward_seq(rc, outs, B, last_only=not all_steps)
        hidden = _pack_hidden(new_state, self.temporal_unet.neuron.kind) if return_state else None
        return det, hidden

    # ---- drop-in per-frame path (train.py:66, visualize.py:71) ----------------------------
    def forward(self, x, hidden_state=None):
        B = x.shape[0]
        stats = self._spike_stats_for(x, 1)
        st = store_for(self, x.device)
        st.refresh_operands()
        feats = self.feature_extractor.forward_seq(x, B, 1)
        rc = RunCtx(st, 1, want_state=True)
        rc.spike_stats = stats
        outs, new_state = self.temporal_unet.forward_seq(rc, feats, _unpack_hidden(hidden_state))
        det = self.detection_head.forward_seq(rc, outs, B, last_only=True)
        return det.as_reference(self.detection_head), _pack_hidden(new_state, self.temporal_unet.neuron.kind)

    def load_state_dict(self, state_dict, strict=True, assign=False):
        """Reference checkpoints carry the frozen YOLO weights under `feature_extractor.model.*`; the stand-in
        extractor has no persistent state, so those keys are dropped."""
        if self.feature_extractor.backend == "ultralytics":
            return super().load_state_dict(state_dict, strict=strict, assign=assign)
        sd = {k: v for k, v in state_dict.items() if not k.startswith("feature_extractor.")}
        return super().load_state_dict(sd, strict=strict, assign=assign)
