"""Times the spike-rate regularizer on the GPU (CUDA events, after warm-up) and writes one JSON record:
  (a) the LIF backward with the dL/ds addend (snn_bn_act_bwd2_ds) vs without it (snn_bn_act_bwd2), both passes, on the LIF
      sweep shapes of `bench.py --microbench lif` (T = 4, 8, 16; fp32 input >= 1 GiB, past the 126 MB L2); the two run
      alternately in the same process, median of the rounds;
  (b) Trainer.train_step_graphed ms/step at B = 64, T = 4, 256 x 256 with and without a SpikeRateLoss attached, alternating
      blocks of replays (each switch re-captures the graph, outside the timed window).
The card's name, power limit and max SM clock are read in the same run and stored beside the numbers.

    python tools/r6/time_spike_reg.py [--out profiles/r6/time_spike_reg.json] [--quick]
"""
import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from snn_object_detectionddp_b200 import kernels as K  # noqa: E402
from tools.r4.time_spike_stats import SWEEP, events_ms, gpu_info  # noqa: E402


def bwd_rows(rounds, reps):
    rows = []
    for T in (4, 8, 16):
        for C, hw in SWEEP:
            per_img = C * hw * hw
            bn = max(1, (1 << 30) // (4 * T * per_img))
            P = bn * hw * hw
            y = torch.randn(T * bn, hw, hw, C, device="cuda")
            gs = torch.randn(T * bn, hw, hw, C, device="cuda").to(torch.bfloat16)
            gamma, beta = torch.ones(C, device="cuda"), torch.full((C,), 0.2, device="cuda")
            scale, shift = torch.ones(T, C, device="cuda"), torch.full((T, C), 0.2, device="cuda")
            mean, invstd = torch.zeros(T, C, device="cuda"), torch.ones(T, C, device="cuda")
            dg, db = torch.zeros(C, device="cuda"), torch.zeros(C, device="cuda")
            c = torch.full((1,), 1e-3, device="cuda")
            plain = lambda: K.bn_act_bwd_train(K.ACT_LIF, y, scale, shift, mean, invstd, beta, gs, T, dg, db)
            added = lambda: K.bn_act_bwd_train(K.ACT_LIF, y, scale, shift, mean, invstd, beta, gs, T, dg, db, ds_add=c)
            plain(), added()
            torch.cuda.synchronize()
            a, b = [], []
            for _ in range(rounds):
                a.append(events_ms(plain, reps))
                b.append(events_ms(added, reps))
            ma, mb = statistics.median(a), statistics.median(b)
            n = y.numel()
            rows.append(dict(T=T, C=C, HW=hw, B=bn, P=P, input_gib=4.0 * n / 2 ** 30, plain_ms=ma, ds_ms=mb, overhead=mb / ma - 1.0,
                             plain_gbs=n * 14.0 / ma / 1e6, ds_gbs=n * 14.0 / mb / 1e6,
                             spread_plain=(min(a), max(a)), spread_ds=(min(b), max(b))))
            print(json.dumps(rows[-1]), flush=True)
            del y, gs
    return rows


def train_rows(B, T, HW, blocks, steps):
    from snn_object_detectionddp_b200.data import synthetic_batch
    from snn_object_detectionddp_b200.model import YOLOTemporalUNet
    from snn_object_detectionddp_b200.spikes import SpikeRateLoss
    from snn_object_detectionddp_b200.trainer import Trainer
    from snn_object_detectionddp_b200.weight_initialization import initialize_model
    torch.manual_seed(0)
    net = YOLOTemporalUNet(num_classes=8, hyp={"box": 7.5, "cls": 1.0, "dfl": 2.5, "reg_max": 16}, neuron="lif")
    initialize_model(net)
    tr = Trainer(net.to("cuda"), total_steps=100000, device="cuda")
    frames, labels = synthetic_batch(B, T, HW, HW, seed=1)
    frames = frames.cuda()
    batch = {"padded": tuple(t.cuda() for t in tr.prepare_batch(labels, B, max_boxes=32)["padded"])}
    reg = SpikeRateLoss(net, synops_weight=1.0, synops_max=0.05, rate_min=0.01, rate_min_weight=0.1)
    ms = {"off": [], "on": []}
    for blk in range(2 * blocks):
        mode = "off" if blk % 2 == 0 else "on"
        tr.spike_reg = reg if mode == "on" else None
        for _ in range(4):                     # eager warm-up steps + capture + one replay after the switch
            tr.train_step_graphed(frames, batch)
        torch.cuda.synchronize()
        ms[mode].append(events_ms(lambda: tr.train_step_graphed(frames, batch), steps))
    res = reg.read()
    off, on = statistics.median(ms["off"]), statistics.median(ms["on"])
    return dict(B=B, T=T, HW=HW, steps_per_block=steps, blocks=blocks, off_ms=off, on_ms=on, overhead=on / off - 1.0,
                off_blocks=ms["off"], on_blocks=ms["on"], penalty=res["spike_reg/penalty"],
                synops_fraction=res["spike_reg/synops_fraction"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r6", "time_spike_reg.json"))
    ap.add_argument("--quick", action="store_true", help="fewer rounds (a smoke run of the script)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA GPU")
    gpu = gpu_info()
    rounds, reps, blocks, steps = (3, 2, 1, 3) if a.quick else (7, 5, 6, 50)
    bwd = bwd_rows(rounds, reps)
    train = train_rows(64, 4, 256, blocks, steps)
    rec = dict(gpu=gpu, device=torch.cuda.get_device_name(), lif_backward=bwd,
               bwd_overhead_max=max(r["overhead"] for r in bwd), bwd_overhead_median=statistics.median(r["overhead"] for r in bwd),
               train_step_graphed=train)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f)
    print(json.dumps({k: v for k, v in rec.items() if k != "lif_backward"}), flush=True)


if __name__ == "__main__":
    main()
