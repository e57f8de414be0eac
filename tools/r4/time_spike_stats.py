"""Times the spike-activity statistics on the GPU (CUDA events, after warm-up) and writes one JSON record:
  (a) the counted LIF forward (snn_bn_act_fwd_count) vs the uncounted one (snn_bn_act_fwd) on the LIF sweep shapes of
      `bench.py --microbench lif` (T = 4, 8, 16; fp32 input >= 1 GiB, past the 126 MB L2), the two run alternately in the
      same process, median of the rounds;
  (b) Trainer.train_step_graphed ms/step at B = 64, T = 4, 256 x 256 with and without a SpikeStats attached, alternating
      blocks of replays (each switch re-captures the graph, outside the timed window);
  (c) SpikeStats.compute() latency (one device-to-host read of the counters + the host arithmetic).
The card's name, power limit and max SM clock are read in the same run and stored beside the numbers.

    python tools/r4/time_spike_stats.py [--out profiles/r4/time_spike_stats.json] [--quick]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from snn_object_detectionddp_b200 import kernels as K  # noqa: E402

SWEEP = ((64, 64), (128, 64), (128, 32), (256, 32), (256, 16), (512, 16))     # (C, H = W), bench.py lif_sweep


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


def lif_rows(rounds, reps):
    rows = []
    for T in (4, 8, 16):
        for C, hw in SWEEP:
            per_img = C * hw * hw
            bn = max(1, (1 << 30) // (4 * T * per_img))
            y = torch.randn(T * bn, hw, hw, C, device="cuda")
            scale, shift = torch.ones(T, C, device="cuda"), torch.full((T, C), 0.2, device="cuda")
            counts = torch.zeros(2, T, device="cuda", dtype=torch.int64)
            plain = lambda: K.bn_act_fwd(K.ACT_LIF, y, scale, shift, T)
            counted = lambda: K.bn_act_fwd(K.ACT_LIF, y, scale, shift, T, spike_counts=(counts[0], counts[1]))
            plain(), counted()
            torch.cuda.synchronize()
            a, b = [], []
            for _ in range(rounds):
                a.append(events_ms(plain, reps))
                b.append(events_ms(counted, reps))
            ma, mb = statistics.median(a), statistics.median(b)
            n = y.numel()
            rows.append(dict(T=T, C=C, HW=hw, B=bn, input_gib=4.0 * n / 2 ** 30, uncounted_ms=ma, counted_ms=mb,
                             overhead=mb / ma - 1.0, uncounted_gbs=n * 6.125 / ma / 1e6, counted_gbs=n * 6.125 / mb / 1e6,
                             spread_uncounted=(min(a), max(a)), spread_counted=(min(b), max(b))))
            print(json.dumps(rows[-1]), flush=True)
            del y
    return rows


def train_rows(B, T, HW, blocks, steps):
    from snn_object_detectionddp_b200.data import synthetic_batch
    from snn_object_detectionddp_b200.model import YOLOTemporalUNet
    from snn_object_detectionddp_b200.spikes import SpikeStats
    from snn_object_detectionddp_b200.trainer import Trainer
    from snn_object_detectionddp_b200.weight_initialization import initialize_model
    torch.manual_seed(0)
    net = YOLOTemporalUNet(num_classes=8, hyp={"box": 7.5, "cls": 1.0, "dfl": 2.5, "reg_max": 16}, neuron="lif")
    initialize_model(net)
    tr = Trainer(net.to("cuda"), total_steps=100000, device="cuda")
    frames, labels = synthetic_batch(B, T, HW, HW, seed=1)
    frames = frames.cuda()
    batch = {"padded": tuple(t.cuda() for t in tr.prepare_batch(labels, B, max_boxes=32)["padded"])}
    stats = SpikeStats(net)
    ms = {"off": [], "on": []}
    for blk in range(2 * blocks):
        mode = "off" if blk % 2 == 0 else "on"
        net.spike_stats = stats if mode == "on" else None
        for _ in range(4):                     # eager warm-up steps + capture + one replay after the switch
            tr.train_step_graphed(frames, batch)
        torch.cuda.synchronize()
        ms[mode].append(events_ms(lambda: tr.train_step_graphed(frames, batch), steps))
    net.spike_stats = stats
    torch.cuda.synchronize()
    lat = []
    for _ in range(20):
        t0 = time.perf_counter()
        res = stats.compute()
        lat.append((time.perf_counter() - t0) * 1e3)
    off, on = statistics.median(ms["off"]), statistics.median(ms["on"])
    return dict(B=B, T=T, HW=HW, steps_per_block=steps, blocks=blocks, off_ms=off, on_ms=on, overhead=on / off - 1.0,
                off_blocks=ms["off"], on_blocks=ms["on"], compute_ms_median=statistics.median(lat), compute_ms_min=min(lat),
                rate=res["spikes/rate"], synops_fraction=res["spikes/synops_fraction"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4", "time_spike_stats.json"))
    ap.add_argument("--quick", action="store_true", help="fewer rounds (a smoke run of the script)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA GPU")
    gpu = gpu_info()
    rounds, reps, blocks, steps = (3, 3, 1, 3) if a.quick else (7, 10, 8, 50)
    lif = lif_rows(rounds, reps)
    train = train_rows(64, 4, 256, blocks, steps)
    rec = dict(gpu=gpu, device=torch.cuda.get_device_name(), lif_forward=lif,
               lif_overhead_max=max(r["overhead"] for r in lif), lif_overhead_median=statistics.median(r["overhead"] for r in lif),
               train_step_graphed=train)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f)
    print(json.dumps({k: v for k, v in rec.items() if k != "lif_forward"}), flush=True)


if __name__ == "__main__":
    main()
