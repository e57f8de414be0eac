"""CPU: the oracle restatement reproduces the golden vectors recorded from the real reference."""
import os

import pytest
import torch

from oracle import snn_oracle as O


def _load(golden_dir, name):
    return torch.load(os.path.join(golden_dir, name), weights_only=False)


def _close(a, b, tol=1e-5):
    assert a.shape == b.shape
    err = (a - b).abs().max().item()
    ref = b.abs().max().item() + 1e-12
    assert err <= tol * max(ref, 1.0), f"max err {err} vs ref scale {ref}"


def _close_ref(a, r, tol, stride):
    """_close against a stored tensor, or against a sampled record (make_golden.sampled): at the stored positions with
    the whole tensor's max |x| as the scale, and on the whole tensor's norm."""
    if torch.is_tensor(r):
        return _close(a, r, tol)
    a = a.detach()
    assert tuple(a.shape) == tuple(r["shape"])
    err = (a.flatten()[::stride] - r["sample"]).abs().max().item()
    assert err <= tol * max(r["absmax"], 1.0), f"max err {err} vs ref scale {r['absmax']}"
    assert abs(float(a.double().norm()) - r["norm"]) <= tol * r["norm"]


@pytest.mark.parametrize("name,stride", [("convblock_s1", 1), ("convblock_s2", 2)])
def test_convblock_matches_reference(golden_dir, name, stride):
    fx = _load(golden_dir, "ref_blocks.pt")[name]
    m = O.OracleConvBlock(16, 32, stride=stride, neuron="silu")
    m.load_state_dict(fx["state"])
    m.train()
    x = fx["x"].clone().requires_grad_(True)
    y, _ = m(x)
    _close(y, fx["y_train"])
    y.backward(fx["gy"])
    _close(x.grad, fx["gx"]); _close(m.conv.weight.grad, fx["gw"])
    _close(m.bn.weight.grad, fx["ggamma"]); _close(m.bn.bias.grad, fx["gbeta"])
    _close(m.bn.running_mean, fx["running_mean"]); _close(m.bn.running_var, fx["running_var"])
    m.eval()
    with torch.no_grad():
        _close(m(fx["x"])[0], fx["y_eval"])


def test_downblock_matches_reference(golden_dir):
    fx = _load(golden_dir, "ref_blocks.pt")["downblock"]
    m = O.OracleDownBlock(16, 32, neuron="silu").train()
    m.load_state_dict(fx["state"])
    x = fx["x"].clone().requires_grad_(True)
    y, _ = m(x)
    _close(y, fx["y"])
    y.backward(fx["gy"])
    _close(x.grad, fx["gx"])
    for k, p in m.named_parameters():
        _close(p.grad, fx["grads"][k], 1e-4)


@pytest.mark.parametrize("name", ["upblock", "upblock_resize"])
def test_upblock_matches_reference(golden_dir, name):
    fx = _load(golden_dir, "ref_blocks.pt")[name]
    m = O.OracleUpBlock(32, 16, 16, neuron="silu").train()
    m.load_state_dict(fx["state"])
    x = fx["x"].clone().requires_grad_(True)
    s = fx["skip"].clone().requires_grad_(True)
    y, _ = m(x, s)
    _close(y, fx["y"])
    y.backward(fx["gy"])
    _close(x.grad, fx["gx"], 1e-4); _close(s.grad, fx["gskip"], 1e-4)
    for k, p in m.named_parameters():
        _close(p.grad, fx["grads"][k], 1e-4)


def test_convlstm_matches_reference(golden_dir):
    fx = _load(golden_dir, "ref_blocks.pt")["convlstm"]
    m = O.OracleConvLSTM2d(16, 16)
    m.load_state_dict(fx["state"])
    xs = [x.clone().requires_grad_(True) for x in fx["xs"]]
    hid, hs = None, []
    for x in xs:
        h, hid = m(x, hid)
        hs.append(h)
    for h, hr in zip(hs, fx["hs"]):
        _close(h, hr)
    _close(hid[1], fx["c_last"])
    ((hs[-1] * fx["gh"]).sum() + (hid[1] * fx["gc"]).sum()).backward()
    for x, gr in zip(xs, fx["gxs"]):
        _close(x.grad, gr, 1e-4)
    for k, p in m.named_parameters():
        _close(p.grad, fx["grads"][k], 1e-4)


@pytest.mark.parametrize("fixture", ["ref_unet_seq.pt", "ref_unet_seq_256.pt"])
def test_unet_sequence_matches_reference(golden_dir, fixture):
    """Seeded init (weight_initialization.py:8-56) + T-step unroll (train.py:62-66) of the full-width net."""
    fx = _load(golden_dir, fixture)
    torch.manual_seed(fx["init_seed"])
    net = O.OracleTemporalUNet([144, 144, 144], neuron="silu")
    net.apply(O.initialize_weights_oracle)
    net.train()
    for k, v in net.state_dict().items():
        if v.dtype.is_floating_point:
            s, a = fx["init_checksums"][k]
            assert abs(float(v.double().sum()) - s) <= 1e-9 * max(1.0, abs(a)), k
            assert abs(float(v.double().abs().sum()) - a) <= 1e-9 * max(1.0, abs(a)), k
    g = torch.Generator().manual_seed(fx["feat_seed"])
    B, T = fx["B"], fx["T"]
    feats = [[torch.randn(B, 144, h, h, generator=g) for h in fx["hw"]] for _ in range(T)]
    outs, hid = O.run_sequence(net, feats)
    so = fx.get("out_stride")
    for o, r in zip(outs, fx["outs"]):
        _close_ref(o, r, 1e-4, so)
    _close(hid[0], fx["h"], 1e-4); _close(hid[1], fx["c"], 1e-4)
    loss = sum((o ** 2).mean() for o in outs)
    assert abs(float(loss) - fx["loss"]) <= 1e-4 * abs(fx["loss"])
    loss.backward()
    for k, p in net.named_parameters():
        r = fx["grad_norms"][k]
        assert abs(float(p.grad.double().norm()) - r) <= 2e-3 * max(r, 1e-6), (k, r)
    sd = net.state_dict()
    for k, v in fx["bn_running"].items():
        _close(sd[k], v, 1e-4)
    assert int(net.enc1.bn.num_batches_tracked) == fx["num_batches_tracked"]
    net.eval()
    with torch.no_grad():
        eo, _ = net(feats[0], None)
    for o, r in zip(eo, fx["eval_outs"]):
        _close_ref(o, r, 1e-4, so)


def test_lif_oracle_hand_case():
    """Build-defined LIF (parity unpinned): hand-computed 1-neuron trace, beta=.5 theta=1."""
    x = torch.tensor([0.6, 0.6, 0.6, 0.1]).reshape(4, 1)
    s, v, u = O.lif_sequence(x)
    # u: .6, .9, 1.05 (spike, reset), .1
    assert s.flatten().tolist() == [0.0, 0.0, 1.0, 0.0]
    assert torch.allclose(u.flatten(), torch.tensor([0.6, 0.9, 1.05, 0.1]))
    assert torch.allclose(v.flatten(), torch.tensor([0.1]))


def test_lif_surrogate_gradcheck_form():
    u = torch.linspace(-1, 3, 9, dtype=torch.float64).requires_grad_(True)
    s = O._ATanSpike.apply(u, 1.0, 2.0)
    s.sum().backward()
    import math
    exp = 1.0 / (1.0 + (math.pi * (u.detach() - 1.0)) ** 2)
    assert torch.allclose(u.grad, exp)


def test_nms_oracle_reproduces_torchvision_fixture(golden_dir):
    """tests/golden/nms_golden.pt was recorded with the REAL torchvision.ops.nms behind the restated ultralytics candidate
    logic (tests/golden/make_golden_nms.py, incl. a torchvision.ops.batched_nms cross-check): the oracle must keep
    reproducing it row for row."""
    from oracle import detect_oracle as D
    fx = torch.load(os.path.join(golden_dir, "nms_golden.pt"), weights_only=False)
    assert len(fx["cases"]) == 3
    for case in fx["cases"]:
        rows = D.non_max_suppression(case["pred"], max_det=300, **case["kwargs"])
        assert len(rows) == len(case["rows"])
        for a, b in zip(rows, case["rows"]):
            assert torch.equal(a, b), case["name"]
        assert sum(r.shape[0] for r in rows) > 0
