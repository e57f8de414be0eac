"""torch.autograd.Function wrappers around the libsnnb200 kernels.

All activations are NHWC tensors ``[T*B, H, W, C]`` with the timestep-major folded batch; `T` is passed
explicitly.  Weight gradients are accumulated *directly* into the flat gradient buffer of the
ParamStore (params.py) by the backward functions (they return ``None`` for the weight inputs), which is
what lets DDP all-reduce contiguous buckets while backward is still running.
"""
import torch
from torch.autograd import Function

from . import kernels as K
from ._lib import ACT_LIF, ACT_SILU, GEOM_1x1, GEOM_3x3_S1, GEOM_3x3_S2, GEOM_T2x2_S2  # noqa: F401


class NeuronCfg:
    """Build-defined LIF neuron (SURVEY.md 7.2) or the reference's SiLU (model.py:15)."""

    def __init__(self, kind="lif", beta=0.5, v_th=1.0, alpha=2.0):
        assert kind in ("lif", "silu")
        self.kind, self.beta, self.v_th, self.alpha = kind, float(beta), float(v_th), float(alpha)

    @property
    def act(self):
        return ACT_LIF if self.kind == "lif" else ACT_SILU


def _bf16c(g):
    if g is None:
        return None
    if g.dtype != torch.bfloat16:
        g = g.to(torch.bfloat16)
    return g.contiguous()


class GradSlot:
    """Gradient of a tensor with TWO consumers, accumulated in the dgrad epilogue instead of by autograd's add kernel.

    The consumer whose backward runs first ('first': the one created LATER in forward) writes its input gradient into a
    fresh buffer and parks it here; the other ('last') launches its dgrad with accumulate=True into that buffer (bf16 TMA
    reduce-add, same rounding as adding two bf16 tensors) and returns no gradient of its own.  The producer's backward runs
    after both (autograd's dependency count), so it sees the complete sum.  One slot per fan-out tensor per forward."""
    __slots__ = ("buf",)

    def __init__(self):
        self.buf = None


def _dead_padded(x_full, n_live, zero):
    """Full-size input-gradient buffer whose trailing n_live samples the caller fills.  The leading (dead) part is
    zero-filled unless every consumer is known to slice it away (Detect-head internals: cfg['dead_grad_unread'])."""
    alloc = torch.zeros if zero else torch.empty
    g = alloc(x_full.shape, device=x_full.device, dtype=torch.bfloat16)
    return g, g[x_full.shape[0] - n_live:]


class ConvBNActFn(Function):
    """conv(cat[x0,x1]) -> per-timestep BatchNorm -> LIF scan over T (or SiLU).  One ConvBlock (model.py:9-18)."""

    @staticmethod
    def forward(ctx, x0, x1, v_init, weight, gamma, beta, cfg):
        st, geom, T, bn, neuron, training = cfg["store"], cfg["geom"], cfg["T"], cfg["bn"], cfg["neuron"], cfg["training"]
        cout = weight.shape[0]
        sums = part = None
        gpt = 0
        if any(ctx.needs_input_grad):
            st.note_use(weight, *((gamma, beta) if training else ()))
        if geom == K.GEOM_DW3x3:
            if training:        # per-timestep BatchNorm partial sums from the same pass over y
                y, part, gpt = K.dw3x3_fprop(x0, st.w_master3(weight).view(9, cout), T=T)
            else:
                y = K.dw3x3_fprop(x0, st.w_master3(weight).view(9, cout))
        elif training:
            y, part, gpt = K.conv_fprop_partials(geom, x0, st.w_fprop(weight), cout, T, x1=x1)    # BN partial sums from the epilogue
        else:
            y = K.conv_fprop(geom, x0, st.w_fprop(weight), cout, x1=x1)
        nb, ho, wo, _ = y.shape
        P = (nb // T) * ho * wo
        if training and part is not None:
            ctr = getattr(bn, "_snn_counters", None)
            if ctr is None or ctr.device != y.device:
                ctr = torch.zeros(((cout + 7) // 8,), device=y.device, dtype=torch.int32)
                bn._snn_counters = ctr            # plain attribute: not a buffer, never in state_dict
            scale, shift, mean, invstd = K.bn_finalize_partials(part, gpt, gamma, beta, bn.running_mean, bn.running_var,
                                                                bn.num_batches_tracked, ctr, T, cout, P, bn.eps, bn.momentum)
        elif training:
            sums = K.bn_stats(y, T)
            scale, shift, mean, invstd = K.bn_finalize(sums, gamma, beta, bn.running_mean, bn.running_var, T, cout, P,
                                                       bn.eps, bn.momentum, True)
            if bn.num_batches_tracked is not None:
                bn.num_batches_tracked += T
        else:
            scale, shift, mean, invstd = K.bn_finalize(None, gamma, beta, bn.running_mean, bn.running_var, T, cout, P,
                                                       bn.eps, bn.momentum, False)
        want_state = cfg.get("want_state", False) and neuron.kind == "lif"
        out, mask, v_final = K.bn_act_fwd(neuron.act, y, scale, shift, T, v_init=v_init,
                                          want_mask=cfg.get("want_mask", False), want_v_final=want_state,
                                          beta=neuron.beta, theta=neuron.v_th, spike_counts=cfg.get("spike_counts"))
        ctx.cfg = cfg
        ctx.has_x1 = x1 is not None
        ctx.has_v = v_init is not None
        ctx.save_for_backward(x0, x1, v_init, weight, gamma, y, scale, shift, mean, invstd)
        cfg["last_mask"] = mask
        if want_state:
            return out, v_final.view(nb // T, ho, wo, cout)
        return out, None

    @staticmethod
    def backward(ctx, g_out, g_vfinal):
        cfg = ctx.cfg
        st, geom, T, neuron, training = cfg["store"], cfg["geom"], cfg["T"], cfg["neuron"], cfg["training"]
        x0, x1, v_init, weight, gamma, y, scale, shift, mean, invstd = ctx.saved_tensors
        if g_out is None:
            g_out = torch.zeros(y.shape, device=y.device, dtype=torch.bfloat16)
        live_T = cfg.get("live_T")
        x0_full = x0
        if live_T is not None and training and neuron.kind == "silu" and not ctx.has_v and g_vfinal is None:
            # stateless layer, only the last live_T timesteps carry gradient: the per-timestep BatchNorm groups are
            # independent, so the backward of the dead frames (all zeros) is skipped, not computed
            n0 = (y.shape[0] // T) * (T - live_T)
            x0, y, g_out = x0[n0:], y[n0:], g_out[n0:]
            x1 = None if x1 is None else x1[n0:]
            scale, shift, mean, invstd = scale[T - live_T:], shift[T - live_T:], mean[T - live_T:], invstd[T - live_T:]
            T = live_T
        else:
            live_T = None
        gs = _bf16c(g_out)
        gvf = None if g_vfinal is None else g_vfinal.contiguous().view(-1).float()
        want_gv0 = ctx.has_v and ctx.needs_input_grad[2]
        if training:
            dgamma = st.grad_view(cfg["bn"].weight)
            dbeta = st.grad_view(cfg["bn"].bias)
            dy, gv0, _ = K.bn_act_bwd_train(neuron.act, y, scale, shift, mean, invstd, cfg["bn"].bias, gs, T, dgamma, dbeta,
                                            v_init=v_init, gv_final=gvf, want_gv_init=want_gv0, beta=neuron.beta,
                                            theta=neuron.v_th, alpha=neuron.alpha)
            st.grad_done(cfg["bn"].weight)
            st.grad_done(cfg["bn"].bias)
        else:
            _, dy, gv0, _ = K.bn_act_bwd(neuron.act, False, y, scale, shift, mean, invstd, gs, T, v_init=v_init,
                                         gv_final=gvf, want_gv_init=want_gv0, beta=neuron.beta, theta=neuron.v_th,
                                         alpha=neuron.alpha)
        gw3 = st.grad_view(weight, three_d=True)
        if geom == K.GEOM_DW3x3:
            c = weight.shape[0]
            K.dw3x3_wgrad(x0, dy, gw3.view(9, c))
            st.grad_done(weight)
            gx0 = None
            if ctx.needs_input_grad[0]:
                if live_T is None:
                    gx0 = K.dw3x3_dgrad(dy, st.w_master3(weight).view(9, c))
                else:
                    gx0, tail = _dead_padded(x0_full, x0.shape[0], not cfg.get("dead_grad_unread", False))
                    K.dw3x3_dgrad(dy, st.w_master3(weight).view(9, c), out=tail)
            return gx0, None, (None if gv0 is None else gv0.view(v_init.shape)), None, None, None, None
        K.conv_wgrad(geom, x0, dy, gw3, w_coff=0)
        if ctx.has_x1:
            K.conv_wgrad(geom, x1, dy, gw3, w_coff=x0.shape[3])
        st.grad_done(weight)
        gx0 = gx1 = None
        in_hw = (x0.shape[1], x0.shape[2])
        zero = not cfg.get("dead_grad_unread", False)
        if ctx.needs_input_grad[0]:
            slot, role = cfg.get("slot_x0", (None, None))
            if slot is not None and live_T is None and role == "last" and slot.buf is not None:
                # the other consumer of x0 already wrote its gradient: add ours in the epilogue, hand nothing to autograd
                K.conv_dgrad(geom, dy, st.w_fprop(weight), in_hw, x0.shape[3], ci_off=0, out=slot.buf, accumulate=True)
            else:
                tail = None
                if live_T is not None:
                    gx0, tail = _dead_padded(x0_full, x0.shape[0], zero)
                r = K.conv_dgrad(geom, dy, st.w_fprop(weight), in_hw, x0.shape[3], ci_off=0, out=tail)
                gx0 = r if live_T is None else gx0
                if slot is not None and live_T is None and role == "first":
                    slot.buf = gx0
        if ctx.has_x1 and ctx.needs_input_grad[1]:
            tail = None
            if live_T is not None:
                gx1, tail = _dead_padded(ctx.saved_tensors[1], x1.shape[0], zero)
            r = K.conv_dgrad(geom, dy, st.w_fprop(weight), in_hw, x1.shape[3], ci_off=x0.shape[3], out=tail)
            gx1 = r if live_T is None else gx1
        if gv0 is not None:
            gv0 = gv0.view(v_init.shape)
        return gx0, gx1, gv0, None, None, None, None


class BilinearResizeFn(Function):
    """UpBlock skip resize, reference model.py:43-44 (F.interpolate bilinear, align_corners=False), NHWC bf16."""

    @staticmethod
    def forward(ctx, x, out_hw):
        ctx.in_hw = (x.shape[1], x.shape[2])
        return K.bilinear_resize(x.contiguous(), out_hw)

    @staticmethod
    def backward(ctx, gy):
        return K.bilinear_resize_bwd(_bf16c(gy), ctx.in_hw), None


class PadEvenFn(Function):
    """Bottom/right zero-pad to even H, W in front of a stride-2 conv (the pad row/column is the conv's own padding)."""

    @staticmethod
    def forward(ctx, x):
        h, w = x.shape[1], x.shape[2]
        ctx.in_hw = (h, w)
        return K.pad_crop(x.contiguous(), (h + (h & 1), w + (w & 1)))

    @staticmethod
    def backward(ctx, gy):
        return K.pad_crop(_bf16c(gy), ctx.in_hw)


class ConvBiasFn(Function):
    """Plain conv with bias: out_p3/4/5 1x1 convs (model.py:119,146) and UpBlock.up (model.py:36,42)."""

    @staticmethod
    def forward(ctx, x0, weight, bias, cfg):
        st, geom = cfg["store"], cfg["geom"]
        cout = weight.shape[1] if geom == GEOM_T2x2_S2 else weight.shape[0]
        if any(ctx.needs_input_grad):
            st.note_use(weight, bias)
        # cfg["out"]: a caller-provided output view (the Detect head's closing convs write straight into the scale-major
        # prediction buffers the loss kernels read: no torch.cat).  It must NOT stay reachable from ctx: output -> grad_fn ->
        # ctx -> output would be a reference cycle that keeps the whole autograd graph of a step (and its AccumulateGrad
        # nodes, bound to the stream they were created on) alive until the next garbage collection -- a later CUDA-graph
        # capture then fails with "dependency created on uncaptured work in another stream".
        cfg = dict(cfg)
        out = K.conv_fprop(geom, x0, st.w_fprop(weight), cout, bias=bias, out=cfg.pop("out", None),
                           out_dtype=cfg.get("out_dtype", torch.bfloat16))
        ctx.cfg = cfg
        ctx.save_for_backward(x0, weight, bias)
        return out

    @staticmethod
    def backward(ctx, g_out):
        cfg = ctx.cfg
        st, geom = cfg["store"], cfg["geom"]
        x0, weight, bias = ctx.saved_tensors
        live_n = cfg.get("live_n")
        x0_full = x0
        if live_n is not None and live_n < x0.shape[0]:
            n0 = x0.shape[0] - live_n          # only the trailing live_n samples carry gradient (see RunCtx.live_T)
            x0, g_out = x0[n0:], g_out[n0:]
        dy = _bf16c(g_out)
        gw3 = st.grad_view(weight, three_d=True)
        K.conv_wgrad(geom, x0, dy, gw3)
        st.grad_done(weight)
        if bias is not None:
            K.colsum_accumulate(dy, st.grad_view(bias))
            st.grad_done(bias)
        gx0 = None
        if ctx.needs_input_grad[0]:
            slot, role = cfg.get("slot_x0", (None, None))
            hw = (x0.shape[1], x0.shape[2])
            if slot is not None and role == "last" and slot.buf is not None:
                # the other consumer of x0 already wrote the full-size gradient: add ours (live frames only) in the epilogue
                K.conv_dgrad(geom, dy, st.w_fprop(weight), hw, x0.shape[3], out=slot.buf[x0_full.shape[0] - x0.shape[0]:], accumulate=True)
            elif x0 is x0_full:
                gx0 = K.conv_dgrad(geom, dy, st.w_fprop(weight), hw, x0.shape[3])
                if slot is not None and role == "first":
                    slot.buf = gx0
            else:
                gx0 = torch.zeros(x0_full.shape, device=dy.device, dtype=torch.bfloat16)
                K.conv_dgrad(geom, dy, st.w_fprop(weight), hw, x0.shape[3], out=gx0[x0_full.shape[0] - x0.shape[0]:])
                if slot is not None and role == "first":
                    slot.buf = gx0
        return gx0, None, None, None


class ConvLSTMSeqFn(Function):
    """ConvLSTM2d (model.py:50-71) over all T steps.

    gates_t = conv3x3(cat[x_t, h_{t-1}]) + b is split as W_x * x (ONE folded launch over T*B, the x's are the
    spike outputs of down3 and exist for all t up front) + W_h * h_{t-1} (sequential, accumulated into the
    same fp32 buffer).  Returns h for all steps (bf16, operand of bottleneck_conv) and the final (h, c) fp32.
    """

    @staticmethod
    def forward(ctx, x, h0, c0, weight, bias, cfg):
        st, T = cfg["store"], cfg["T"]
        ch = weight.shape[0] // 4
        nb, hh, ww, cx = x.shape
        B = nb // T
        w = st.w_fprop(weight)
        if any(ctx.needs_input_grad):
            st.note_use(weight, bias)
        gates = K.conv_fprop(GEOM_3x3_S1, x, w, 4 * ch, bias=bias, w_coff=0)
        h_all = torch.empty((nb, hh, ww, ch), device=x.device, dtype=torch.bfloat16)
        c_all = torch.empty((nb, hh, ww, ch), device=x.device, dtype=torch.float32)
        h_prev_b = None if h0 is None else h0.to(torch.bfloat16).contiguous()
        c_prev = None if c0 is None else c0.contiguous()
        h_last = None
        for t in range(T):
            g_t = gates[t * B:(t + 1) * B]
            if h_prev_b is not None:
                K.conv_fprop(GEOM_3x3_S1, h_prev_b, w, 4 * ch, out=g_t, w_coff=cx, accumulate=True)
            h_last, c_t, hb = K.lstm_gates_fwd(g_t, c_prev, ch, h_bf16_out=h_all[t * B:(t + 1) * B],
                                               c_out=c_all[t * B:(t + 1) * B])
            h_prev_b, c_prev = hb, c_t
        ctx.cfg = cfg
        ctx.has_state = h0 is not None
        ctx.save_for_backward(x, h0, c0, weight, gates, h_all, c_all)
        return h_all, h_last, c_all[(T - 1) * B:]

    @staticmethod
    def backward(ctx, g_hall, g_hlast, g_clast):
        cfg = ctx.cfg
        st, T = cfg["store"], cfg["T"]
        x, h0, c0, weight, gates, h_all, c_all = ctx.saved_tensors
        ch = weight.shape[0] // 4
        nb, hh, ww, cx = x.shape
        B = nb // T
        wt = st.w_fprop(weight)
        dgates = torch.empty(gates.shape, device=x.device, dtype=torch.bfloat16)
        dh_rec = None if g_hlast is None else g_hlast.contiguous().float()
        dc = None if g_clast is None else g_clast.contiguous().float()
        h0b = None if h0 is None else h0.to(torch.bfloat16).contiguous()
        g_hall = _bf16c(g_hall)
        for t in range(T - 1, -1, -1):
            sl = slice(t * B, (t + 1) * B)
            # dL/dh_t = consumer's gradient (bf16 slice of g_hall) + recurrent gradient (fp32 dgrad of step t+1): summed in-kernel
            c_prev = c_all[(t - 1) * B:t * B] if t > 0 else (None if c0 is None else c0.contiguous())
            _, dc = K.lstm_gates_bwd(gates[sl], c_prev, c_all[sl], dh_rec, dc, ch, dgates_out=dgates[sl],
                                     dh_bf16=None if g_hall is None else g_hall[sl])
            if t > 0 or ctx.has_state:
                dh_rec = K.conv_dgrad(GEOM_3x3_S1, dgates[sl], wt, (hh, ww), ch, ci_off=cx, out_dtype=torch.float32)
            else:
                dh_rec = None
        gw3 = st.grad_view(weight, three_d=True)
        K.conv_wgrad(GEOM_3x3_S1, x, dgates, gw3, w_coff=0)
        if T > 1:
            K.conv_wgrad(GEOM_3x3_S1, h_all[:(T - 1) * B], dgates[B:], gw3, w_coff=cx)
        if h0b is not None:
            K.conv_wgrad(GEOM_3x3_S1, h0b, dgates[:B], gw3, w_coff=cx)
        st.grad_done(weight)
        bias = cfg["bias"]
        if bias is not None:
            K.colsum_accumulate(dgates, st.grad_view(bias))
            st.grad_done(bias)
        gx = None
        if ctx.needs_input_grad[0]:
            gx = K.conv_dgrad(GEOM_3x3_S1, dgates, wt, (hh, ww), cx, ci_off=0)
        gh0 = dh_rec if (ctx.has_state and ctx.needs_input_grad[1]) else None
        gc0 = dc if (ctx.has_state and ctx.needs_input_grad[2]) else None
        return gx, gh0, gc0, None, None, None
