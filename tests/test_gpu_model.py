"""-m gpu: module-level parity of the host-side mirror (snn_object_detectionddp_b200/model.py) against

* the REFERENCE-PINNED golden fixture tests/golden/ref_unet_seq.pt (recorded from the real reference
  TemporalUNet, model.py:100-146, seeded init, T=3 unroll, backward) -- `neuron='silu'` mode, and
* the oracle restatement (oracle/snn_oracle.py) with `emulate_bf16=True` (the numeric contract of the tensor-core
  convs) for the BUILD-DEFINED LIF mode ("parity unpinned": the reference has no spiking neuron).

Tolerances: the product rounds conv operands to bf16 (rel 2^-9 per operand); against an oracle that rounds the
same operands the remaining difference is fp32 summation order (1e-5 per layer, amplified by BatchNorm over tiny
batches) -> 2e-3 on outputs; against the fp32 reference fixture the bf16 rounding itself shows -> 6e-2.
Spikes must agree exactly except where the oracle membrane is within 1e-5 of threshold (flip-rate protocol).
"""
import os

import pytest
import torch

from oracle import snn_oracle as O
from tests.gpu_util import rel_err, sampled_rel_err, setup_exact

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _pkg():
    import snn_object_detectionddp_b200.model as M
    import snn_object_detectionddp_b200.weight_initialization as WI
    from snn_object_detectionddp_b200.params import store_for
    return M, WI, store_for


def _nhwc(x):      # NCHW fp32 -> NHWC bf16
    return x.permute(0, 2, 3, 1).to(torch.bfloat16).contiguous()


def _fold(seq):    # list over t of NCHW [B,...] -> NHWC bf16 [T*B,...]
    return _nhwc(torch.cat(seq, 0))


# ------------------------------------------------------------------------------------------------
# reference-pinned: silu network vs the golden fixture of the real reference
# ------------------------------------------------------------------------------------------------
def _build_seeded(M, WI, neuron):
    torch.manual_seed(42)
    net = M.TemporalUNet([144, 144, 144], use_conv_lstm=True, neuron=neuron)
    net.apply(WI.initialize_weights)
    return net


def test_silu_unet_matches_reference_fixture(golden_dir):
    setup_exact()
    M, WI, store_for = _pkg()
    # geometry of BASELINE.json configs[0] (B=2, T=4, 256x256 frames); the fp32 oracle reproduces this fixture to 1e-4
    # and the bf16-operand oracle deviates from it by 0.8-1.0 % on outputs / 0.3 % on gradient norms (measured on
    # CPU, see DESIGN.md) -> tolerances 3e-2 here.
    fx = torch.load(os.path.join(golden_dir, "ref_unet_seq_256.pt"), weights_only=False)
    net = _build_seeded(M, WI, "silu")
    # same seeded init as the reference (weight_initialization.py:8-56): per-tensor checksums
    for k, v in net.state_dict().items():
        if v.dtype.is_floating_point and k in fx["init_checksums"]:
            s, a = fx["init_checksums"][k]
            assert abs(float(v.double().sum()) - s) <= 1e-6 * max(1.0, a), k
            assert abs(float(v.double().abs().sum()) - a) <= 1e-9 * max(1.0, a), k
    net = net.to(DEV).train()
    B, T = fx["B"], fx["T"]
    g = torch.Generator().manual_seed(fx["feat_seed"])
    feats = [[torch.randn(B, 144, h, h, generator=g).to(DEV) for h in fx["hw"]] for _ in range(T)]
    # drop-in per-frame loop, exactly train.py:62-66
    hid = None
    for fs in feats:
        outs, hid = net(fs, hid)
    loss = sum((o ** 2).mean() for o in outs)
    loss.backward()
    for o, r in zip(outs, fx["outs"]):
        assert sampled_rel_err(o, r, fx["out_stride"]) < 3e-2
    assert rel_err(hid[0].detach().cpu(), fx["h"]) < 3e-2 and rel_err(hid[1].detach().cpu(), fx["c"]) < 3e-2
    assert abs(float(loss) - fx["loss"]) < 1e-2 * fx["loss"]
    assert int(net.enc1.bn.num_batches_tracked) == fx["num_batches_tracked"]
    for k, v in fx["bn_running"].items():
        mine = net.state_dict()[k].cpu()
        assert rel_err(mine, v) < 3e-2, k
    bad = []
    for k, p in net.named_parameters():
        gn = float(p.grad.double().norm())
        if abs(gn - fx["grad_norms"][k]) > 3e-2 * fx["grad_norms"][k] + 1e-7:
            bad.append((k, gn, fx["grad_norms"][k]))
    assert not bad, bad


# ------------------------------------------------------------------------------------------------
# oracle (bf16-operand contract) vs product: narrow network, silu and lif, fused sequence path
# ------------------------------------------------------------------------------------------------
WIDTHS = (64, 128, 256, 512)


def _pair(neuron, seed=0):
    M, WI, store_for = _pkg()
    torch.manual_seed(seed)
    orc = O.OracleTemporalUNet([144, 144, 144], neuron=neuron, emulate_bf16=True, widths=WIDTHS)
    orc.apply(O.initialize_weights_oracle)
    with torch.no_grad():   # non-trivial BN affine so gamma/beta gradients are exercised
        for m in orc.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.weight.uniform_(0.8, 1.6)
                m.bias.uniform_(-0.2, 0.5)
    net = M.TemporalUNet([144, 144, 144], neuron=neuron, widths=WIDTHS)
    missing = net.load_state_dict(orc.state_dict(), strict=True)       # identical key names (SURVEY 8b)
    assert not missing.missing_keys and not missing.unexpected_keys
    return orc.to(DEV), net.to(DEV), store_for


def _feats(B, T, hw, seed=1):
    g = torch.Generator().manual_seed(seed)
    return [[torch.randn(B, 144, hw // s, hw // s, generator=g).to(DEV) for s in (8, 16, 32)] for _ in range(T)]


def _run_product_seq(net, store_for, feats, T, want_state=True):
    from snn_object_detectionddp_b200.model import RunCtx
    st = store_for(net, DEV)
    st.zero_grad()
    st.refresh_operands()
    rc = RunCtx(st, T, want_state=want_state, fp32_outputs=True)
    rc.record = {}
    folded = tuple(_fold([fs[i] for fs in feats]) for i in range(3))
    outs, state = net.forward_seq(rc, folded)
    return outs, state, rc


def test_silu_narrow_unet_fused_sequence_vs_oracle():
    setup_exact()
    orc, net, store_for = _pair("silu")
    B, T = 2, 4
    feats = _feats(B, T, 128)
    orc.train(); net.train()
    o_outs, o_hid = O.run_sequence(orc, feats)
    o_loss = sum((o ** 2).mean() for o in o_outs)
    o_loss.backward()
    outs, ((h, c), _), _ = _run_product_seq(net, store_for, feats, T)
    last = [o[-B:].permute(0, 3, 1, 2) for o in outs]
    # same bf16 operands on both sides; what remains is fp32 summation order / SiLU ulp differences that now and
    # then move an activation across a bf16 rounding boundary (0.4 % on that element) -> 1e-2
    for a, b in zip(last, o_outs):
        assert rel_err(a, b) < 1e-2
    assert rel_err(h.permute(0, 3, 1, 2), o_hid[0]) < 1e-2 and rel_err(c.permute(0, 3, 1, 2), o_hid[1]) < 1e-2
    loss = sum((o ** 2).mean() for o in last)
    loss.backward()
    og = dict(orc.named_parameters())
    worst = max((rel_err(p.grad, og[k].grad), k) for k, p in net.named_parameters())
    assert worst[0] < 3e-2, worst
    # BN running statistics advanced T times, in order
    for k, v in orc.state_dict().items():
        if "running" in k:
            assert rel_err(net.state_dict()[k], v) < 5e-3, k      # near-zero means of deep layers: abs err ~1e-5
        if "num_batches_tracked" in k:
            assert int(net.state_dict()[k]) == int(v)


def test_fused_sequence_equals_per_frame_loop():
    """forward_seq over folded T*B == T drop-in calls threading hidden state (train.py:62-66), LIF mode."""
    setup_exact()
    orc, net, store_for = _pair("lif")
    del orc
    B, T = 2, 3
    feats = _feats(B, T, 128, seed=5)
    net.train()
    sd0 = {k: v.clone() for k, v in net.state_dict().items()}
    outs, ((h, c), mem), _ = _run_product_seq(net, store_for, feats, T)
    net.load_state_dict(sd0)
    hid = None
    for fs in feats:
        o2, hid = net(fs, hid)
    for a, b in zip(outs, o2):
        assert torch.equal(a[-B:].permute(0, 3, 1, 2), b), "fused sequence differs from the per-frame loop"
    assert torch.equal(h.permute(0, 3, 1, 2), hid[0]) and torch.equal(c.permute(0, 3, 1, 2), hid[1])
    # membranes: the per-(t,c) BN statistics are reduced across thread blocks in an order that is not fixed, so the
    # fp32 scale/shift may differ in the last ulp between two launches; spikes (outputs) are compared exactly above
    assert torch.allclose(mem["enc1"], hid[2]["enc1"], rtol=1e-5, atol=1e-6)


def _flip_report(name, s_prod, s_orc, u_orc, theta=1.0):
    flips = s_prod != s_orc
    near = (u_orc - theta).abs() < 1e-5
    return dict(layer=name, n=s_orc.numel(), flips=int(flips.sum()), far=int((flips & ~near).sum()),
                rate=float(s_orc.float().mean()))


def test_lif_convblock_teacher_forced_spikes_and_grads():
    """One spiking ConvBlock, T steps, same input spikes on both sides: spikes exact up to near-threshold flips;
    gradients (surrogate, BN batch statistics, wgrad, dgrad) vs oracle autograd."""
    setup_exact()
    M, WI, store_for = _pkg()
    T, B, H, W, Ci, Co = 4, 2, 16, 16, 128, 128
    torch.manual_seed(3)
    ob = O.OracleConvBlock(Ci, Co, neuron="lif", emulate_bf16=True).to(DEV).train()
    with torch.no_grad():
        ob.bn.weight.uniform_(0.8, 1.6); ob.bn.bias.uniform_(-0.2, 0.5)
    pb = M.ConvBlock(Ci, Co, neuron="lif").to(DEV).train()
    pb.load_state_dict(ob.state_dict())
    xs = [(torch.rand(B, Ci, H, W, device=DEV) < 0.2).float().requires_grad_(True) for _ in range(T)]
    gs = torch.randn(T, B, Co, H, W, device=DEV).to(torch.bfloat16).float()
    v, ss, us = None, [], []
    for t in range(T):
        s, v = ob(xs[t], v)
        ss.append(s); us.append(ob.last_u)
    (torch.stack(ss) * gs).sum().backward()
    st = store_for(pb, DEV)
    st.zero_grad(); st.refresh_operands()
    x = _fold([x.detach() for x in xs]).requires_grad_(True)
    out, _ = pb.forward_seq(M.RunCtx(st, T), x)
    rep = _flip_report("block", out.reshape(T, B, H, W, Co).permute(0, 1, 4, 2, 3).float(), torch.stack(ss).detach(),
                       torch.stack(us))
    assert rep["far"] == 0, rep
    assert rep["flips"] <= 2, rep
    assert 0.03 < rep["rate"] < 0.7, rep
    out.backward(gs.permute(0, 1, 3, 4, 2).reshape(out.shape).to(torch.bfloat16))
    if rep["flips"] == 0:
        gx_ref = torch.cat([x_.grad for x_ in xs], 0).permute(0, 2, 3, 1)
        assert rel_err(x.grad, gx_ref) < 1e-2
        assert rel_err(pb.conv.weight.grad, ob.conv.weight.grad) < 1e-2
        assert rel_err(pb.bn.weight.grad, ob.bn.weight.grad) < 1e-2
        assert rel_err(pb.bn.bias.grad, ob.bn.bias.grad) < 1e-2
    assert rel_err(pb.bn.running_mean, ob.bn.running_mean) < 1e-4
    assert rel_err(pb.bn.running_var, ob.bn.running_var) < 1e-4


def test_lif_unet_flip_rates_end_to_end_and_teacher_forced():
    """Whole spiking U-Net, T=4, per-layer spike agreement with the bf16-operand oracle.

    (1) teacher-forced: every ConvBlock is fed the ORACLE's input of that layer -> spikes must be exact except
        neurons whose oracle membrane is within 1e-5 of threshold (flip-rate protocol, SURVEY 7.2);
    (2) end-to-end: the encoder (9 spiking layers before the ConvLSTM) must still be exact; after the ConvLSTM the
        fp32 hidden state differs by ulps, which now and then moves a bf16 operand rounding of h and from there
        spreads through train-mode BatchNorm statistics -- reported, bounded loosely, never hidden."""
    setup_exact()
    M, _, _ = _pkg()
    orc, net, store_for = _pair("lif", seed=7)
    B, T = 2, 4
    feats = _feats(B, T, 128, seed=9)
    orc.train(); net.train()
    rec_s, rec_u, rec_x = {}, {}, {}
    names = {m: n for n, m in orc.named_modules() if isinstance(m, O.OracleConvBlock)}

    def hook(m, inp, outp):
        rec_x.setdefault(names[m], []).append(inp[0].detach())
        rec_s.setdefault(names[m], []).append(outp[0].detach())
        rec_u.setdefault(names[m], []).append(m.last_u)

    hs = [m.register_forward_hook(hook) for m in names]
    with torch.no_grad():
        o_outs, _ = O.run_sequence(orc, feats)
    for h in hs:
        h.remove()
    with torch.no_grad():
        outs, _, rc = _run_product_seq(net, store_for, feats, T, want_state=False)
    e2e, forced = [], []
    blocks = dict(net.named_modules())
    for name, s_list in rec_s.items():
        s_o, u_o = torch.stack(s_list), torch.stack(rec_u[name])             # [T,B,C,H,W]
        sp = rc.record[name]
        e2e.append(_flip_report(name, sp.reshape(T, B, *sp.shape[1:]).permute(0, 1, 4, 2, 3).float(), s_o, u_o))
        with torch.no_grad():
            st = store_for(net, DEV)
            out, _ = blocks[name].forward_seq(M.RunCtx(st, T), _fold(rec_x[name]))
        forced.append(_flip_report(name, out.reshape(T, B, *out.shape[1:]).permute(0, 1, 4, 2, 3).float(), s_o, u_o))
    print("\nLIF flip report, teacher-forced:", *forced, sep="\n  ")
    print("LIF flip report, end-to-end:", *e2e, sep="\n  ")
    assert sum(r["far"] for r in forced) == 0, forced
    assert sum(r["flips"] for r in forced) <= 4, forced
    pre_lstm = ["enc1", "down1.conv1", "down1.conv2", "enc2", "down2.conv1", "down2.conv2", "enc3", "down3.conv1",
                "down3.conv2"]
    enc = [r for r in e2e if r["layer"] in pre_lstm]
    assert len(enc) == 9 and sum(r["far"] for r in enc) == 0 and sum(r["flips"] for r in enc) <= 4, enc
    total, flips = sum(r["n"] for r in e2e), sum(r["flips"] for r in e2e)
    assert flips / total < 0.1, (flips, total)
    if flips == 0:
        for a, b in zip(outs, o_outs):
            assert rel_err(a[-B:].permute(0, 3, 1, 2), b) < 1e-2


def test_eval_mode_uses_running_stats_and_streams_state():
    """model.eval(): BN running statistics; state threaded through two sequence calls == one long sequence."""
    setup_exact()
    orc, net, store_for = _pair("lif", seed=11)
    B, T = 1, 4
    feats = _feats(B, T, 128, seed=13)
    with torch.no_grad():
        for m in list(orc.modules()):
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.uniform_(-0.2, 0.2); m.running_var.uniform_(0.5, 2.0)
        net.load_state_dict(orc.state_dict())
    orc.eval(); net.eval()
    with torch.no_grad():
        o_outs, _ = O.run_sequence(orc, feats)
        hid = None
        for fs in feats:                                        # drop-in streaming, visualize.py:66-71
            outs, hid = net(fs, hid)
        full, _, _ = _run_product_seq(net, store_for, feats, T)
    for a, b in zip(outs, full):
        assert torch.equal(a, b[-B:].permute(0, 3, 1, 2))
    errs = [rel_err(a, b) for a, b in zip(outs, o_outs)]
    print("eval-mode LIF out errs", errs)
    assert max(errs) < 0.2          # bounded loosely: upstream near-threshold flips propagate (reported above)
