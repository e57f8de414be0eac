"""Times the detection metrics on the GPU (CUDA events, after warm-up) and prints one JSON line:
  * DetMetrics.update per batch: B = 64 images, max_det 300, M = 32 targets, nc = 8, every row kept (conf 0.001 keeps
    nearly all of them);
  * DetMetrics.compute (sort + finalisation + the one host read) at 1 M and 4 M records;
  * the stock route for the same evaluation: per image, rows and targets copied to the host and matched in numpy, then
    ap_per_class (the CPU specification of the test suite), on a smaller sample, reported per batch.
The card's name and power limit are printed beside the numbers.

    python tools/r3/time_det_metrics.py [--out profiles/r3/time_det_metrics.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import det_metrics_oracle as S  # noqa: E402
from snn_object_detectionddp_b200.metrics import DetMetrics  # noqa: E402

B, MAX_DET, M, NC = 64, 300, 32, 8


def batch(g, dev):
    rows = torch.zeros(B, MAX_DET, 6, device=dev)
    xy = torch.rand(B, MAX_DET, 2, device=dev, generator=g) * 600
    rows[..., :2], rows[..., 2:4] = xy, xy + 8 + torch.rand(B, MAX_DET, 2, device=dev, generator=g) * 60
    rows[..., 4] = torch.rand(B, MAX_DET, device=dev, generator=g) + 0.001
    rows[..., 5] = torch.randint(0, NC, (B, MAX_DET), device=dev, generator=g).float()
    gt_cls = torch.randint(0, NC, (B, M), device=dev, generator=g)
    gt_box = torch.cat((torch.rand(B, M, 2, device=dev, generator=g) * 0.8 + 0.1,
                        torch.rand(B, M, 2, device=dev, generator=g) * 0.2 + 0.02), 2)
    hit = torch.cat((gt_box[..., :2] - gt_box[..., 2:] / 2, gt_box[..., :2] + gt_box[..., 2:] / 2), 2) * 640
    rows[:, :M, :4] = hit + torch.randn(B, M, 4, device=dev, generator=g) * 2
    rows[:, :M, 5] = gt_cls.float()
    counts = torch.full((B,), MAX_DET, device=dev, dtype=torch.int32)
    return rows, counts, (gt_cls, gt_box, torch.ones(B, M, device=dev, dtype=torch.bool))


def events_ms(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    rec = {"gpu": smi[0] if smi else torch.cuda.get_device_name(0), "B": B, "max_det": MAX_DET, "M": M, "nc": NC}
    batches = [batch(g, dev) for _ in range(8)]

    # update per batch (buffer preallocated past the timed records: growth is a separate, amortised copy)
    m = DetMetrics(NC, dev, capacity=B * MAX_DET * 1100)
    for bt in batches:
        m.update(*bt, (640, 640))
    torch.cuda.synchronize()
    it = iter(range(1 << 30))
    rec["update_ms_per_batch"] = events_ms(lambda: m.update(*batches[next(it) % 8], (640, 640)), 1000)

    # compute at 1 M and 4 M records
    for n_rec, label in ((1 << 20, "1M"), (1 << 22, "4M")):
        m2 = DetMetrics(NC, dev, capacity=n_rec + B * MAX_DET)
        while m2.bound < n_rec:
            m2.update(*batches[(m2.bound // (B * MAX_DET)) % 8], (640, 640))
        m2.compute()                                      # warm-up (sort workspace, modules)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        reps = 5
        for _ in range(reps):
            m2.compute()                                  # ends in a device-to-host read: host clock is a full-call time
        rec[f"compute_ms_{label}"] = (time.perf_counter() - t0) * 1e3 / reps
        rec[f"records_{label}"] = m2.bound

    # stock route: per-image host copies + numpy matching, 4 batches, then ap_per_class over them
    spec = S.SpecMetrics()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for rows, counts, padded in batches[:4]:
        for b in range(B):
            spec.update(rows[b:b + 1].cpu().numpy(), counts[b:b + 1].cpu().numpy(), padded[0][b:b + 1].cpu().numpy(),
                        padded[1][b:b + 1].cpu().numpy(), padded[2][b:b + 1].cpu().numpy(), 640, 640)
    t1 = time.perf_counter()
    spec.compute()
    t2 = time.perf_counter()
    rec["stock_match_ms_per_batch"] = (t1 - t0) * 1e3 / 4
    rec["stock_ap_per_class_ms_at_records"] = [(t2 - t1) * 1e3, 4 * B * MAX_DET]
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(args.out), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
