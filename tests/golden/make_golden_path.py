"""Generate tests/golden/ref_blocks_path.pt from the UNMODIFIED reference classes (run in the build container):

    python tests/golden/make_golden_path.py

Per-block fixtures at the PATH-TRUE channel counts (reference model.py:9-71 instantiated as TemporalUNet does at
model.py:104-119: 144->128, 128->256 stride 2, UpBlock(256,128,128), ConvLSTM2d) so that the CUDA blocks -- whose
stride-2 / transposed kernels need C % 64 == 0 -- can be compared with the real reference directly (`-m gpu`,
tests/test_gpu_blocks_reference.py), teacher-forced per block.

To make a tight tolerance meaningful for bf16-operand tensor-core kernels, every conv OPERAND the reference sees here is
bf16-representable (inputs and conv weights are rounded to bf16 before the reference runs, in fp32): the reference's
fp32 conv and the tcgen05 bf16 x bf16 -> fp32 conv then multiply identical numbers, and what remains is summation order
(1e-6) plus the bf16 rounding of the product's OUTPUT activations (2^-9).

Weights are not stored (MBs): they are re-created from the recorded seed through the same constructor + the reference's
`initialize_weights` (weight_initialization.py:8-56), which the product mirrors draw for draw; per-tensor checksums pin
that.  Inputs and upstream gradients are not stored either: they are the next draws of the same seeded generator, and
their shapes and checksums are.  Gradients are stored as norms + a 1-in-29 strided sample, output tensors as norm, shape
and a 1-in-7 strided sample (compact(), which keeps the file under 1 MB).
"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle.ref_loader import load_reference  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
STRIDE = 29
OUT_STRIDE = 7
INPUTS = ("x", "skip", "gy", "xs", "gh", "gc")


def bf16r(t):
    return t.to(torch.bfloat16).to(torch.float32)


def sample(t):
    return t.detach().flatten()[::STRIDE].clone()


def prepare(m, wi, g):
    """initialize_weights, then: conv weights -> bf16-representable, BN affine -> non-trivial (so dgamma/dbeta matter)."""
    m.apply(wi.initialize_weights)
    with torch.no_grad():
        for mod in m.modules():
            if isinstance(mod, (torch.nn.Conv2d, torch.nn.ConvTranspose2d)):
                mod.weight.copy_(bf16r(mod.weight))
            if isinstance(mod, torch.nn.BatchNorm2d):
                mod.weight.copy_(torch.rand(mod.weight.shape, generator=g) * 0.8 + 0.8)
                mod.bias.copy_(torch.rand(mod.bias.shape, generator=g) * 0.7 - 0.2)
    return m


def checks(m):
    return {k: (float(v.double().sum()), float(v.double().abs().sum())) for k, v in m.state_dict().items()
            if v.dtype.is_floating_point}


def grads(m):
    return {k: dict(norm=float(p.grad.double().norm()), sample=sample(p.grad)) for k, p in m.named_parameters()}


def compact(fx):
    """In place: every input / upstream gradient -> {shape, sum, abs} (the test draws it again from the generator, in the
    order of INPUTS, and checks the sums), every other tensor of more than 256 elements -> {shape, norm, sample} with an
    OUT_STRIDE strided sample of the flattened tensor."""
    def inp(t):
        assert torch.equal(bf16r(t.float()), t.float())        # bf16-representable by construction
        t = t.double()
        return dict(shape=tuple(t.shape), sum=float(t.sum()), abs=float(t.abs().sum()))

    def out(t):
        return dict(shape=tuple(t.shape), norm=float(t.double().norm()), sample=t.detach().float().flatten()[::OUT_STRIDE].clone())

    fx["out_stride"] = OUT_STRIDE
    for rec in fx.values():
        if not isinstance(rec, dict):
            continue
        for k, v in rec.items():
            if k in INPUTS:
                rec[k] = [inp(t) for t in v] if isinstance(v, list) else inp(v)
            elif isinstance(v, list) and all(torch.is_tensor(t) for t in v):
                rec[k] = [out(t) for t in v]
            elif torch.is_tensor(v) and v.numel() > 256:
                rec[k] = out(v)
    return fx


def main():
    ref, wi = load_reference()
    fx = {"stride": STRIDE}

    def rnd(g, *s):
        return bf16r(torch.randn(*s, generator=g))

    # ---- ConvBlock, stride 1 (enc1: 144 -> 128) and stride 2 (down1.conv1: 128 -> 256), train + eval ----
    for name, (ci, co, stride, seed) in {"convblock_s1": (144, 128, 1, 101), "convblock_s2": (128, 256, 2, 102)}.items():
        g = torch.Generator().manual_seed(seed)
        torch.manual_seed(seed)
        m = prepare(ref.ConvBlock(ci, co, stride=stride), wi, g).train()
        ck = checks(m)
        x = rnd(g, 2, ci, 8, 8).requires_grad_(True)
        y = m(x)
        gy = rnd(g, *y.shape)
        y.backward(gy)
        rec = dict(seed=seed, ci=ci, co=co, stride=stride, checks=ck, x=x.detach().clone(), y_train=y.detach().clone(), gy=gy,
                   gx=x.grad.clone(), grads=grads(m), running_mean=m.bn.running_mean.clone(),
                   running_var=m.bn.running_var.clone(), conv_y=torch.nn.functional.conv2d(x.detach(), m.conv.weight.detach(), None, stride, 1))
        m.eval()
        with torch.no_grad():
            rec["y_eval"] = m(x.detach()).clone()
        fx[name] = rec

    # ---- DownBlock(128, 256) ----
    g = torch.Generator().manual_seed(103)
    torch.manual_seed(103)
    m = prepare(ref.DownBlock(128, 256), wi, g).train()
    ck = checks(m)
    x = rnd(g, 2, 128, 8, 8).requires_grad_(True)
    y = m(x)
    gy = rnd(g, *y.shape)
    y.backward(gy)
    fx["downblock"] = dict(seed=103, checks=ck, x=x.detach().clone(), y=y.detach().clone(), gy=gy, gx=x.grad.clone(), grads=grads(m))

    # ---- UpBlock(256, 128, 128): same-size skip, and the bilinear skip-resize branch (model.py:43-44) ----
    for name, skip_hw, seed in (("upblock", (8, 8), 104), ("upblock_resize", (7, 7), 105), ("upblock_resize_h", (7, 8), 106)):
        g = torch.Generator().manual_seed(seed)
        torch.manual_seed(seed)
        m = prepare(ref.UpBlock(256, 128, 128), wi, g).train()
        ck = checks(m)
        x = rnd(g, 2, 256, 4, 4).requires_grad_(True)
        skip = rnd(g, 2, 128, *skip_hw).requires_grad_(True)
        y = m(x, skip)
        gy = rnd(g, *y.shape)
        y.backward(gy)
        fx[name] = dict(seed=seed, checks=ck, x=x.detach().clone(), skip=skip.detach().clone(), y=y.detach().clone(), gy=gy,
                        gx=x.grad.clone(), gskip=skip.grad.clone(), grads=grads(m))

    # ---- ConvLSTM2d(128, 128): 3 steps with state carry, zero-init state on the first ----
    g = torch.Generator().manual_seed(107)
    torch.manual_seed(107)
    m = prepare(ref.ConvLSTM2d(128, 128), wi, g)
    ck = checks(m)
    xs = [rnd(g, 2, 128, 4, 4).requires_grad_(True) for _ in range(3)]
    hid, hs = None, []
    for x in xs:
        h, hid = m(x, hid)
        hs.append(h)
    gh = rnd(g, *hs[-1].shape)
    gc = rnd(g, *hid[1].shape)
    (hs[-1] * gh).sum().add((hid[1] * gc).sum()).backward()
    fx["convlstm"] = dict(seed=107, checks=ck, xs=[x.detach().clone() for x in xs], hs=[h.detach().clone() for h in hs],
                          c_last=hid[1].detach().clone(), gh=gh, gc=gc, gxs=[x.grad.clone() for x in xs], grads=grads(m))

    compact(fx)
    path = os.path.join(OUT, "ref_blocks_path.pt")
    torch.save(fx, path)
    print("ref_blocks_path.pt", os.path.getsize(path))


if __name__ == "__main__":
    torch.set_num_threads(8)
    main()
