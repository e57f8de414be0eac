"""Shared helpers for the -m gpu parity tests (torch fp32 references of single ops, error metrics)."""
import torch
import torch.nn.functional as F

from snn_object_detectionddp_b200 import _lib as L


def setup_exact():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


def rel_err(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / (b.norm() + 1e-30))


def sampled_rel_err(got, ref, stride):
    """rel_err against a fixture tensor stored as {shape, norm, sample} (every stride-th element of the flattened tensor):
    the larger of the error at the stored positions and the error of the whole tensor's norm."""
    got = got.detach().float().cpu()
    assert tuple(got.shape) == tuple(ref["shape"]), (tuple(got.shape), ref["shape"])
    en = abs(float(got.double().norm()) - ref["norm"]) / (ref["norm"] + 1e-30)
    return max(rel_err(got.flatten()[::stride], ref["sample"]), en)


def max_err(a, b):
    return float((a.double() - b.double()).abs().max())


def describe_mismatch(got, ref, tol=1e-2, maxn=8):
    """Human-readable summary of where an NHWC result differs (for blind debugging from logs)."""
    d = (got.double() - ref.double()).abs()
    scale = ref.double().abs().max().item() + 1e-12
    bad = d > tol * scale
    nbad = int(bad.sum())
    msg = [f"shape={tuple(got.shape)} rel={rel_err(got, ref):.3e} max={d.max().item():.3e} scale={scale:.3e} "
           f"bad={nbad}/{bad.numel()} nan={int(torch.isnan(got.float()).sum())}"]
    if nbad:
        idx = bad.nonzero()[:maxn]
        for i in idx:
            t = tuple(int(v) for v in i)
            msg.append(f"  at {t}: got {float(got[t]):.5f} ref {float(ref[t]):.5f}")
        if got.dim() == 4:
            msg.append("  bad per n: " + str(bad.sum((1, 2, 3)).tolist()[:16]))
            msg.append("  bad per h: " + str(bad.sum((0, 2, 3)).tolist()[:16]))
            msg.append("  bad per w: " + str(bad.sum((0, 1, 3)).tolist()[:16]))
            cb = bad.sum((0, 1, 2))
            msg.append("  bad per c (blocks of 8): " + str(cb.reshape(-1, 8).sum(1).tolist()[:40]))
    return "\n".join(msg)


def w_to_torch(geom, w):
    """[rows][taps][K] (fp32/bf16) -> torch conv weight layout."""
    w = w.float()
    rows, taps, k = w.shape
    if geom == L.GEOM_T2x2_S2:   # ConvTranspose2d weight [Cin, Cout, 2, 2]
        return w.reshape(rows, 2, 2, k).permute(3, 0, 1, 2).contiguous()
    ks = 3 if taps == 9 else 1
    return w.reshape(rows, ks, ks, k).permute(0, 3, 1, 2).contiguous()


def w_from_torch(geom, wt):
    """torch conv weight -> [rows][taps][K]."""
    if geom == L.GEOM_T2x2_S2:   # [Cin, Cout, 2, 2] -> [Cout][4][Cin]
        ci, co = wt.shape[:2]
        return wt.permute(1, 2, 3, 0).reshape(co, 4, ci).contiguous()
    co, ci, kh, kw = wt.shape
    return wt.permute(0, 2, 3, 1).reshape(co, kh * kw, ci).contiguous()


def ref_conv(geom, x_nhwc, w, bias=None):
    """fp32 reference of the geometry on NHWC input, weights [rows][taps][K] -> NHWC fp32 output."""
    x = x_nhwc.float().permute(0, 3, 1, 2)
    wt = w_to_torch(geom, w)
    if geom == L.GEOM_3x3_S1:
        y = F.conv2d(x, wt, bias, stride=1, padding=1)
    elif geom == L.GEOM_3x3_S2:
        y = F.conv2d(x, wt, bias, stride=2, padding=1)
    elif geom == L.GEOM_1x1:
        y = F.conv2d(x, wt, bias)
    else:
        y = F.conv_transpose2d(x, wt, bias, stride=2)
    return y.permute(0, 2, 3, 1).contiguous()
