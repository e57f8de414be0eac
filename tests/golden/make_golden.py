"""Generate the committed golden fixtures from the UNMODIFIED reference (run in the build container).

    python tests/golden/make_golden.py

Imports /root/reference/{model,weight_initialization}.py through oracle/ref_loader.py (ultralytics
stubbed) and records inputs/outputs/gradients of the reference's own classes:

* ref_blocks.pt   -- narrow ConvBlock / DownBlock / UpBlock / ConvLSTM2d instances, weights included
                     (reference model.py:9-71), train- and eval-mode BN, forward + backward.
* ref_unet_seq_256.pt -- same as ref_unet_seq.pt at the geometry of BASELINE.json configs[0] (B=2, T=4, feature
                     maps 32/16/8 of a 256x256 frame); BatchNorm groups are >= 32 samples there, so bf16-operand
                     kernels can be compared against it at a meaningful tolerance.  Its output maps are stored as
                     sampled() records (norm, max |x| and a 1-in-7 strided sample), which keeps the file under 1 MB.
* ref_unet_seq.pt -- full-width TemporalUNet([144,144,144]) (model.py:100-146) initialised with
                     initialize_weights (weight_initialization.py:8-56) under torch.manual_seed(42),
                     T=3 unroll with ConvLSTM state carry (train.py:62-66), loss on the last step,
                     backward.  Weights are NOT stored (480 MB): the fixture pins per-parameter
                     checksums of the seeded init, the outputs, the LSTM state, BN running stats and
                     per-parameter gradient norms.

The reference publishes no golden vectors or tests (SURVEY.md section 4); these fixtures are the
"outputs of the reference itself run here" that pin the oracle restatement.
"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle.ref_loader import load_reference  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
OUT_STRIDE = 7


def sampled(t):
    """{shape, norm, absmax, sample}: the whole tensor's shape, norm and max |x|, and an OUT_STRIDE strided sample of it
    flattened."""
    t = t.detach().float()
    return dict(shape=tuple(t.shape), norm=float(t.double().norm()), absmax=float(t.abs().max()),
                sample=t.flatten()[::OUT_STRIDE].clone())


def blocks(ref):
    g = torch.Generator().manual_seed(1234)
    fx = {}

    def rnd(*s):
        return torch.randn(*s, generator=g)

    # ConvBlock stride 1 and 2, train + eval
    for name, stride in (("convblock_s1", 1), ("convblock_s2", 2)):
        torch.manual_seed(7)
        m = ref.ConvBlock(16, 32, stride=stride)
        with torch.no_grad():
            m.bn.weight.copy_(rnd(32) * 0.2 + 1.0)
            m.bn.bias.copy_(rnd(32) * 0.1)
        sd0 = {k: v.clone() for k, v in m.state_dict().items()}
        x = rnd(3, 16, 8, 8).requires_grad_(True)
        m.train()
        y = m(x)
        gy = rnd(*y.shape)
        y.backward(gy)
        rec = dict(state=sd0, x=x.detach().clone(), y_train=y.detach().clone(), gy=gy,
                   gx=x.grad.clone(), gw=m.conv.weight.grad.clone(),
                   ggamma=m.bn.weight.grad.clone(), gbeta=m.bn.bias.grad.clone(),
                   running_mean=m.bn.running_mean.clone(), running_var=m.bn.running_var.clone())
        m.eval()
        with torch.no_grad():
            rec["y_eval"] = m(x.detach()).clone()
        fx[name] = rec

    # DownBlock
    torch.manual_seed(8)
    m = ref.DownBlock(16, 32).train()
    sd0 = {k: v.clone() for k, v in m.state_dict().items()}
    x = rnd(2, 16, 8, 8).requires_grad_(True)
    y = m(x)
    gy = rnd(*y.shape)
    y.backward(gy)
    fx["downblock"] = dict(state=sd0, x=x.detach().clone(), y=y.detach().clone(), gy=gy, gx=x.grad.clone(),
                           grads={k: p.grad.clone() for k, p in m.named_parameters()})

    # UpBlock, same-size skip and odd-size skip (bilinear branch, model.py:43-44)
    for name, skip_hw in (("upblock", (8, 8)), ("upblock_resize", (7, 8))):
        torch.manual_seed(9)
        m = ref.UpBlock(32, 16, 16).train()
        sd0 = {k: v.clone() for k, v in m.state_dict().items()}
        x = rnd(2, 32, 4, 4).requires_grad_(True)
        skip = rnd(2, 16, *skip_hw).requires_grad_(True)
        y = m(x, skip)
        gy = rnd(*y.shape)
        y.backward(gy)
        fx[name] = dict(state=sd0, x=x.detach().clone(), skip=skip.detach().clone(), y=y.detach().clone(),
                        gy=gy, gx=x.grad.clone(), gskip=skip.grad.clone(),
                        grads={k: p.grad.clone() for k, p in m.named_parameters()})

    # ConvLSTM2d: 3 steps with state carry, zero-init state on the first
    torch.manual_seed(10)
    m = ref.ConvLSTM2d(16, 16)
    sd0 = {k: v.clone() for k, v in m.state_dict().items()}
    xs = [rnd(2, 16, 4, 4).requires_grad_(True) for _ in range(3)]
    hid, hs = None, []
    for x in xs:
        h, hid = m(x, hid)
        hs.append(h)
    gh = rnd(*hs[-1].shape)
    gc = rnd(*hid[1].shape)
    (hs[-1] * gh).sum().add((hid[1] * gc).sum()).backward()
    fx["convlstm"] = dict(state=sd0, xs=[x.detach().clone() for x in xs], hs=[h.detach().clone() for h in hs],
                          c_last=hid[1].detach().clone(), gh=gh, gc=gc, gxs=[x.grad.clone() for x in xs],
                          grads={k: p.grad.clone() for k, p in m.named_parameters()})
    torch.save(fx, os.path.join(OUT, "ref_blocks.pt"))
    print("ref_blocks.pt", os.path.getsize(os.path.join(OUT, "ref_blocks.pt")))


def unet_seq(ref, wi, name="ref_unet_seq.pt", B=2, T=3, hw=(8, 4, 2), feat_seed=4242, sample_outs=False):
    torch.manual_seed(42)
    net = ref.TemporalUNet([144, 144, 144], use_conv_lstm=True)
    net.apply(wi.initialize_weights)
    net.train()
    init_ck = {k: (float(v.double().sum()), float(v.double().abs().sum())) for k, v in net.state_dict().items()
               if v.dtype.is_floating_point}
    g = torch.Generator().manual_seed(feat_seed)
    feats = [[torch.randn(B, 144, hw[0], hw[0], generator=g), torch.randn(B, 144, hw[1], hw[1], generator=g),
              torch.randn(B, 144, hw[2], hw[2], generator=g)] for _ in range(T)]
    hid = None
    for f in feats:
        outs, hid = net(f, hid)
    loss = sum((o ** 2).mean() for o in outs)
    loss.backward()
    fx = dict(B=B, T=T, hw=hw, feat_seed=feat_seed, init_seed=42, init_checksums=init_ck, out_stride=OUT_STRIDE,
              outs=[sampled(o) if sample_outs else o.detach().clone() for o in outs], h=hid[0].detach().clone(), c=hid[1].detach().clone(),
              loss=float(loss),
              grad_norms={k: float(p.grad.double().norm()) for k, p in net.named_parameters()},
              bn_running={k: v.clone() for k, v in net.state_dict().items() if "running" in k and v.numel() <= 256},
              num_batches_tracked=int(net.enc1.bn.num_batches_tracked))
    # eval-mode single forward from the post-training-forward buffers
    net.eval()
    with torch.no_grad():
        eo, _ = net(feats[0], None)
    fx["eval_outs"] = [sampled(o) if sample_outs else o.clone() for o in eo]
    torch.save(fx, os.path.join(OUT, name))
    print(name, os.path.getsize(os.path.join(OUT, name)))


if __name__ == "__main__":
    torch.set_num_threads(8)
    ref, wi = load_reference()
    blocks(ref)
    unet_seq(ref, wi)
    # BASELINE.json configs[0] geometry: B=2, T=4, 256x256 frames -> feature maps 32/16/8, bottleneck 4x4
    unet_seq(ref, wi, name="ref_unet_seq_256.pt", B=2, T=4, hw=(32, 16, 8), feat_seed=256256, sample_outs=True)
