"""Times the weight average (snn_ema_update, ema.ModelEMA) on the GPU (CUDA events, after warm-up) and writes one JSON record:
  (a) snn_ema_update alone at the full model size (the flat master buffer of the default-width detector, 120.3 M
      parameters, plus its BatchNorm segment table): 12 B per parameter = 1.44 GB per call, past the 126 MB L2, so every
      call streams from HBM.  Reported as achieved GB/s against the 6555 GB/s measured copy rate (profiles/README.md);
  (b) Trainer.train_step_graphed ms/step at B = 64, T = 4, 256 x 256 with and without a ModelEMA attached, alternating
      blocks of replays (each switch re-captures the graph, outside the timed window).
The card's name, power limit and max SM clock are read in the same run and stored beside the numbers.

    python tools/r5/time_ema.py [--out profiles/r5/time_ema.json] [--quick]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from snn_object_detectionddp_b200 import kernels as K  # noqa: E402

COPY_GBS = 6555.0          # measured device-to-device copy rate of the B200 (profiles/README.md)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def events_ms(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def build(B, T, HW):
    from snn_object_detectionddp_b200.data import synthetic_batch
    from snn_object_detectionddp_b200.model import YOLOTemporalUNet
    from snn_object_detectionddp_b200.trainer import Trainer
    from snn_object_detectionddp_b200.weight_initialization import initialize_model
    torch.manual_seed(0)
    net = YOLOTemporalUNet(num_classes=8, hyp={"box": 7.5, "cls": 1.0, "dfl": 2.5, "reg_max": 16}, neuron="lif")
    initialize_model(net)
    tr = Trainer(net.to("cuda"), total_steps=100000, device="cuda")
    frames, labels = synthetic_batch(B, T, HW, HW, seed=1)
    batch = {"padded": tuple(t.cuda() for t in tr.prepare_batch(labels, B, max_boxes=32)["padded"])}
    return tr, frames.cuda(), batch


def update_row(ema, rounds, reps):
    params = sum(e.numel for e in ema._src.entries)
    n = ema._dst.flat_p.numel() + ema._segment_elems
    for _ in range(3):
        ema.update()
    torch.cuda.synchronize()
    ms = [events_ms(ema.update, reps) for _ in range(rounds)]
    med = statistics.median(ms)
    gbs = 12.0 * n / med / 1e6
    return dict(params=params, flat_elems=ema._dst.flat_p.numel(), segment_elems=ema._segment_elems,
                bn_segments=0 if ema._segments is None else int(ema._segments.shape[0]), bytes_per_call=12.0 * n,
                ms_median=med, ms_min=min(ms), ms_max=max(ms), gbs=gbs, of_copy_rate=gbs / COPY_GBS, rounds=rounds,
                reps=reps)


def train_rows(tr, frames, batch, ema, blocks, steps):
    ms = {"off": [], "on": []}
    for blk in range(2 * blocks):
        mode = "off" if blk % 2 == 0 else "on"
        tr.ema = ema if mode == "on" else None
        for _ in range(4):                     # eager warm-up steps + capture + one replay after the switch
            tr.train_step_graphed(frames, batch)
        torch.cuda.synchronize()
        ms[mode].append(events_ms(lambda: tr.train_step_graphed(frames, batch), steps))
    tr.ema = None
    off, on = statistics.median(ms["off"]), statistics.median(ms["on"])
    return dict(steps_per_block=steps, blocks=blocks, off_ms=off, on_ms=on, overhead_ms=on - off, overhead=on / off - 1.0,
                off_blocks=ms["off"], on_blocks=ms["on"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r5", "time_ema.json"))
    ap.add_argument("--quick", action="store_true", help="fewer rounds (a smoke run of the script)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA GPU")
    from snn_object_detectionddp_b200.ema import ModelEMA
    gpu = gpu_info()
    rounds, reps, blocks, steps = (3, 5, 1, 3) if a.quick else (9, 50, 8, 50)
    B, T, HW = 64, 4, 256
    tr, frames, batch = build(B, T, HW)
    ema = ModelEMA(tr.model)
    upd = update_row(ema, rounds, reps)
    print(json.dumps(upd), flush=True)
    train = dict(B=B, T=T, HW=HW, **train_rows(tr, frames, batch, ema, blocks, steps))
    train["update_share_of_step"] = upd["ms_median"] / train["off_ms"]
    rec = dict(gpu=gpu, device=torch.cuda.get_device_name(), ema_update=upd, train_step_graphed=train)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f)
    print(json.dumps(rec), flush=True)


if __name__ == "__main__":
    main()
