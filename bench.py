#!/usr/bin/env python
"""Headline benchmark: SNN-detector training throughput (images/s) on B200 through the libsnnb200 hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W]                 # our arm (1 GPU, or under torchrun: N ranks)
    python bench.py --dump-outputs DIR                                  # + the last timed step's results as DIR/*.npy
    python bench.py --impl reference [--steps K] [--warmup W]           # CPU arm: oracle port of the reference path
    python bench.py --impl eager-gpu                                    # GPU comparator: the oracle modules in PyTorch eager
    python bench.py --microbench lif                                    # BASELINE.json configs[3] LIF sweep (GB/s)

A "step" is one training step of the reference (train.py:58-80): T-frame unroll with state carry, detection loss on
the last frame, backward, clip_grad_norm_(10), AdamW, OneCycleLR -- on one synthetic batch.  Workload at every N is
BASELINE.json configs[1] per GPU (default SNN detector, T=4, batch 64, 256x256 frames; weak scaling);
``--config 3`` selects configs[2] (T=8, 512x512).

Prints ONE JSON line (rank 0).  `value` = device-resident throughput (inputs already in HBM), `e2e` = the same metric
through the public API with pinned HOST buffers (H2D of the frames + labels and a D2H read of the loss every step),
`kernels` / `roofline` = per-kernel durations INSIDE the replayed CUDA graph (CUPTI activity records of extra replays
right after the timed region, matched launch by launch to the ABI calls recorded at capture; fallback: CUDA events
around eager launches), `cfg3` = the same measurement on BASELINE.json configs[2] (T=8, 512x512, batch 16/GPU) so that
the scaling runs carry it at every N, `ranks_in_lockstep` = every rank holds bit-identical parameters after the timed
steps, `cpu_baseline` = the oracle port of the reference path on this box's host cores and `gpu_eager_baseline` = the
same oracle modules in PyTorch eager on this GPU (N=1 only), `lif_microbench` = configs[3] sweep with its own clocks
(worst fractions only; `--microbench lif` prints the rows).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

HYP = {"box": 7.5, "cls": 1.0, "dfl": 2.5, "reg_max": 16}      # reference config.yaml:33-37
NUM_CLASSES = 8                                                 # config.yaml:29
MAX_LR, WEIGHT_DECAY = 1e-4, 5e-4                               # config.yaml:23-24


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed training steps of the measured path (the baseline sub-records "
                    "of a single-GPU run use fixed counts: 3 timed + 2 warm-up steps on the GPU, 3 + 1 on the CPU)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "eager-gpu"])
    ap.add_argument("--config", type=int, default=2, choices=[1, 2, 3], help="BASELINE.json configs index + 1")
    ap.add_argument("--batch", type=int, default=None, help="per-GPU batch (default: the config's)")
    ap.add_argument("--neuron", default="lif", choices=["lif", "silu"])
    ap.add_argument("--microbench", default=None, choices=["lif"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-profile", action="store_true", help="skip the per-kernel CUDA-event accounting")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from Python instead of replaying one CUDA graph")
    ap.add_argument("--ref-batch", type=int, default=2, help="sequences per step of the CPU arm (bounded sample)")
    ap.add_argument("--no-cfg3", action="store_true", help="skip the configs[2] (T=8, 512x512) sub-record")
    ap.add_argument("--no-lif", action="store_true", help="skip the configs[3] LIF sweep sub-record")
    ap.add_argument("--no-gpu-eager", action="store_true", help="skip the PyTorch-eager GPU comparator")
    ap.add_argument("--dump-trace", default=None, help="write the ABI call sequence of one training step (name, work, shape tag) as JSON")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write the last one's loss, loss items, gradient norm and a seeded sample of "
                         "the updated parameters as DIR/<name>.npy (float32)")
    return ap.parse_args()


def workload(args, cfg=None):
    cfg = args.config if cfg is None else cfg
    if cfg == 1:
        B, T, HW = 2, 4, 256
    elif cfg == 2:
        B, T, HW = 64, 4, 256
    else:
        B, T, HW = 16, 8, 512
    if args.batch and cfg == args.config:
        B = args.batch
    return B, T, HW


def workload_name(args, B, T, HW, cfg=None):
    cfg = args.config if cfg is None else cfg
    return (f"BASELINE.json configs[{cfg - 1}]: default SNN detector ({args.neuron} neurons), T={T}, batch {B}/GPU, "
            f"synthetic {HW}x{HW} RGB frames, one train step (fwd + loss + bwd + clip + AdamW + OneCycle)")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback (B200_PROFILING.md)")


# ------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons, pw = [], None, set(), []
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1]); pw.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [s for s, p in zip(sm, pw) if p > 250.0] or sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "power_w_max": max(pw) if pw else None, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU arm: oracle port of the reference path (test infrastructure used as the measured baseline)
# ------------------------------------------------------------------------------------------------
def cpu_reference_run(T, HW, batch, steps, warmup, neuron):
    import torch
    from oracle import model_oracle as MO
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(42)
    model = MO.OracleYOLOTemporalUNet(num_classes=NUM_CLASSES, hyp=HYP, neuron=neuron)
    MO.initialize_model_oracle(model)
    model.train()
    loss_fn, opt, sched = MO.make_reference_trainer(model, total_steps=max(1000, steps + warmup + 1), max_lr=MAX_LR,
                                                    weight_decay=WEIGHT_DECAY)
    frames, labels = MO.synthetic_batch(batch, T, HW, HW, nc=NUM_CLASSES, seed=42)
    for _ in range(warmup):
        MO.reference_train_step(model, loss_fn, opt, sched, frames, labels)
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        MO.reference_train_step(model, loss_fn, opt, sched, frames, labels)
        times.append(time.perf_counter() - t0)
    sec = sum(times) / len(times)
    return dict(value=batch / sec, sec_per_step=sec, cores=cores, threads=torch.get_num_threads(),
                sample=f"{steps} timed + {warmup} warm-up training steps of {batch} sequences (T={T}, {HW}x{HW}) = a "
                       f"{batch}-sequence slice of the workload's batch; oracle port (PyTorch fp32 eager, {cores} threads)")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    B, T, HW = workload(args)
    r = cpu_reference_run(T, HW, args.ref_batch, args.steps, args.warmup, args.neuron)
    line = {
        "impl": "reference", "metric": "train images/sec", "value": r["value"], "unit": "images/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["sec_per_step"] * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args, B, T, HW), "per_gpu_batch": B, "T": T, "cpu_sample_batch": args.ref_batch},
        "cpu_baseline": {"value": r["value"], "unit": "images/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]},
        "e2e": {"value": r["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
# ------------------------------------------------------------------------------------------------
# GPU comparator: the same oracle modules (= the reference's classes restated, oracle/) in PyTorch eager on this GPU
# ------------------------------------------------------------------------------------------------
def gpu_eager_run(T, HW, batch, steps, warmup, neuron, dev):
    """Reference step semantics (train.py:58-80) on the GPU through stock PyTorch kernels (cuDNN convs, eager autograd,
    torch.optim.AdamW): fp32 with torch's defaults (TF32 convolutions) and bf16 autocast, channels_last.  Stand-in extractor /
    restated head + loss as in the CPU arm.  Test infrastructure timed as a baseline -- never on the product path."""
    import torch
    from oracle import model_oracle as MO
    out = {}
    frames, labels = MO.synthetic_batch(batch, T, HW, HW, nc=NUM_CLASSES, seed=42)
    frames, labels = frames.to(dev), labels.to(dev)
    for mode in ("fp32", "bf16_autocast"):
        torch.manual_seed(42)
        model = MO.OracleYOLOTemporalUNet(num_classes=NUM_CLASSES, hyp=HYP, neuron=neuron)
        MO.initialize_model_oracle(model)
        model = model.to(dev).to(memory_format=torch.channels_last).train()
        loss_fn, opt, sched = MO.make_reference_trainer(model, total_steps=1000, max_lr=MAX_LR, weight_decay=WEIGHT_DECAY)

        def step():
            if mode == "fp32":
                return MO.reference_train_step(model, loss_fn, opt, sched, frames, labels)
            opt.zero_grad(set_to_none=True)
            with torch.autocast("cuda", dtype=torch.bfloat16):
                hidden = None
                for t in range(frames.shape[1]):
                    preds, hidden = model(frames[:, t], hidden)
            b = {"batch_idx": labels[:, 0], "cls": labels[:, 1], "bboxes": labels[:, 2:]}
            loss, items = loss_fn([p.float() for p in preds], b)
            loss.sum().backward()
            torch.nn.utils.clip_grad_norm_(model.parameters(), max_norm=10.0)
            opt.step()
            sched.step()
            return loss, items, None

        try:
            for _ in range(warmup):
                step()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                step()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out[mode] = {"value": batch / (ms * 1e-3), "ms_per_step": ms}
        except Exception as e:          # e.g. an op without a bf16 autocast path: report, do not hide
            out[mode] = {"error": f"{type(e).__name__}: {e}"[:200]}
        del model, opt, sched, loss_fn
        torch.cuda.empty_cache()
    out.update(unit="images/s", kind="port", batch=batch,
               what=f"oracle modules (reference classes restated) in PyTorch eager on this GPU, channels_last, per-frame loop, torch AdamW; "
                    f"{steps} timed + {warmup} warm-up steps of {batch} sequences (T={T}, {HW}x{HW})")
    return out


def dropin_run(T, HW, batch, steps, warmup, neuron, dev):
    """The reference's own training-loop body (train.py:58-80: per-frame `model(frame, hidden)` loop, `loss_fn(preds, batch)`,
    `.sum().backward()`, `clip_grad_norm_`, torch AdamW + OneCycleLR) running UNCHANGED on the drop-in modules -- the
    "4 import lines" route of INTEGRATION.md section 1.  Every kernel is launched from Python (no CUDA graph, T per-frame
    passes, NCHW<->NHWC conversions at the module boundary): host-bound, reported next to the fused Trainer path."""
    import torch
    from snn_object_detectionddp_b200 import _lib
    from snn_object_detectionddp_b200.data import synthetic_batch
    from snn_object_detectionddp_b200.loss import v8DetectionLoss
    from snn_object_detectionddp_b200.model import YOLOTemporalUNet
    from snn_object_detectionddp_b200.weight_initialization import initialize_model
    torch.manual_seed(42)
    model = YOLOTemporalUNet(num_classes=NUM_CLASSES, yolo_model_name="yolo11m.pt", use_conv_lstm=True, hyp=HYP, neuron=neuron).to(dev)
    initialize_model(model)
    loss_fn = v8DetectionLoss(model)
    optimizer = torch.optim.AdamW(model.parameters(), weight_decay=WEIGHT_DECAY)
    scheduler = torch.optim.lr_scheduler.OneCycleLR(optimizer, max_lr=MAX_LR, total_steps=1000, pct_start=0.3, anneal_strategy="cos")
    frames, labels = synthetic_batch(batch, T, HW, HW, nc=NUM_CLASSES, seed=42)
    image_tensor, labels_tensor = frames.to(dev), labels.to(dev)
    model.train()

    def step():
        optimizer.zero_grad(set_to_none=True)
        hidden_state = None
        for t in range(T):
            preds, hidden_state = model(image_tensor[:, t, :, :, :], hidden_state)
        batch_dict = {"batch_idx": labels_tensor[:, 0], "cls": labels_tensor[:, 1], "bboxes": labels_tensor[:, 2:]}
        loss_components, _ = loss_fn(preds, batch_dict)
        loss_components.sum().backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), max_norm=10.0)
        optimizer.step()
        scheduler.step()

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    l0 = _lib.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    out = {"value": batch / (ms * 1e-3), "unit": "images/s", "ms_per_step": ms, "gpu_launches_per_step": (_lib.launch_count - l0) / steps,
           "what": "reference train.py:58-80 loop body verbatim on the drop-in modules (per-frame calls, list-of-maps loss, torch AdamW/OneCycleLR), eager"}
    del model, optimizer, scheduler, loss_fn
    torch.cuda.empty_cache()
    return out


def run_gpu_eager(args):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    torch.cuda.set_device(0)
    B, T, HW = workload(args)
    r = gpu_eager_run(T, HW, B, args.steps, args.warmup, args.neuron, torch.device("cuda", 0))
    best = max((v for v in (r.get("fp32"), r.get("bf16_autocast")) if v and "value" in v), key=lambda v: v["value"])
    print(json.dumps({"impl": "eager-gpu", "metric": "train images/sec", "value": best["value"], "unit": "images/s", "n_gpus": 1,
                      "steps": args.steps, "warmup": args.warmup, "ms_per_step": best["ms_per_step"], "higher_is_better": True,
                      "scaling": "weak", "vs_baseline": None, "dtype": "f32/bf16", "data": "synthetic",
                      "config": {"workload": workload_name(args, B, T, HW)}, "gpu_eager_baseline": r, "gpu_launches": 0}), flush=True)


# ------------------------------------------------------------------------------------------------
# per-kernel accounting
# ------------------------------------------------------------------------------------------------
# ABI entry point -> substrings of the GPU kernels it launches, in launch order (memsets are not kernels)
EXPECT = {
    "snn_conv_fprop": ["conv_gemm_kernel"], "snn_conv_fprop_stats": ["conv_gemm_kernel"], "snn_conv_dgrad": ["conv_gemm_kernel"],
    "snn_conv_wgrad": ["wgrad_gemm_kernel"], "snn_bn_finalize_partials": ["bn_finalize_partials_kernel"],
    "snn_bn_stats_from_partials": ["bn_stats_from_partials_kernel"], "snn_bn_stats": ["bn_stats_kernel", "bn_stats_from_partials_kernel"],
    "snn_bn_finalize": ["bn_finalize_kernel"], "snn_bn_act_fwd": ["bn_act_fwd_kernel"], "snn_bn_act_bwd2": ["bwd2_kernel"],
    "snn_bn_act_bwd": ["bn_act_bwd_kernel"], "snn_bn_bwd_dx": ["bn_bwd_finalize_kernel", "bn_bwd_dx_kernel"],
    "snn_lstm_gates_fwd": ["lstm_gates_fwd_kernel"], "snn_lstm_gates_bwd": ["lstm_gates_bwd_kernel"],
    "snn_colsum_bf16": ["colsum_bf16_kernel"], "snn_dw3x3_fprop": ["dw3x3_col_kernel"], "snn_dw3x3_fprop_stats": ["dw3x3_col_kernel"],
    "snn_dw3x3_dgrad": ["dw3x3_col_kernel"], "snn_dw3x3_wgrad": ["dw3x3_wgrad_col_kernel"], "snn_space_to_depth8": ["s2d8_kernel"], "snn_space_to_depth8_u8": ["s2d8_u8_kernel"],
    "snn_grad_sumsq": ["sumsq_kernel"], "snn_adamw_step": ["adamw_kernel", "step_advance_kernel"],
    "snn_detect_assign_loss_fwd": ["detect_decode_kernel", "tal_metric_topk_kernel", "tal_resolve_kernel", "tal_targets_kernel",
                                   "detect_loss_fwd_kernel"],
    "snn_detect_loss_bwd_rows": ["detect_loss_bwd_kernel"], "snn_weight_prep": ["weight_prep_kernel"],
    "snn_bilinear_resize": ["bilinear_"], "snn_nhwc_pad_crop": ["pad_crop_kernel"],
}


def cupti_graph_accounting(replay_fn, trace, replays):
    """Kernel durations INSIDE the replayed graph: CUPTI activity records (torch.profiler) of `replays` extra replays,
    matched in launch order to the ABI calls recorded while the graph was captured.  Returns
    (agg {abi name: {ms, calls, flop, byte}}, shapes {(abi name, tag): {...}}, other {kernel name: ms}, total kernel ms)
    or None if CUPTI is unavailable / the sequence cannot be matched."""
    import torch
    try:
        import torch.profiler as tp
        with tp.profile(activities=[tp.ProfilerActivity.CUDA, tp.ProfilerActivity.CPU]) as prof:
            for _ in range(replays):
                replay_fn()
            torch.cuda.synchronize()
        evs = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and not e.name.lower().startswith(("memcpy", "memset"))]
    except Exception as e:
        return None, f"torch.profiler failed: {type(e).__name__}: {e}"[:200]
    if not evs:
        return None, "no CUDA kernel records from torch.profiler (CUPTI unavailable)"
    evs.sort(key=lambda e: e.time_range.start)
    comm = comm_overlap(evs, replays)
    evs = [e for e in evs if not e.name.startswith("nccl")]
    seq = [(name, work, sub, k == 0) for name, work in trace for k, sub in enumerate(EXPECT.get(name, []))]
    agg, shapes, other = {}, {}, {}
    j, total = 0, 0.0
    for _ in range(replays):
        for name, work, sub, first in seq:
            while j < len(evs) and sub not in evs[j].name:
                d = evs[j].time_range.elapsed_us() * 1e-3
                other[evs[j].name[:80]] = other.get(evs[j].name[:80], 0.0) + d
                total += d
                j += 1
            if j >= len(evs):
                return None, f"kernel records ran out while matching {name} ({sub}): capture trace and replay differ"
            d = evs[j].time_range.elapsed_us() * 1e-3
            j += 1
            total += d
            a = agg.setdefault(name, dict(ms=0.0, calls=0, flop=0.0, byte=0.0))
            a["ms"] += d
            if first:
                a["calls"] += 1
                if work:
                    a[work[0]] += work[1]
            if work and len(work) > 2:
                sh = shapes.setdefault((name, work[2]), dict(ms=0.0, calls=0, amount=0.0, kind=work[0]))
                sh["ms"] += d
                if first:
                    sh["calls"] += 1
                    sh["amount"] += work[1]
    while j < len(evs):
        d = evs[j].time_range.elapsed_us() * 1e-3
        other[evs[j].name[:80]] = other.get(evs[j].name[:80], 0.0) + d
        total += d
        j += 1
    if comm:
        other["__comm__"] = comm
    return (agg, shapes, other, total), None


def comm_overlap(evs, replays):
    """Timeline of the gradient exchange inside the replayed graph (N > 1): NCCL kernels by name, the time they are
    resident, and how much of it no compute kernel overlaps (= exposed communication), per step.  From the same CUPTI
    records as the kernel accounting (hardware timestamps), so it needs no separate profiler run."""
    nccl = [(e.time_range.start, e.time_range.end, e.name) for e in evs if e.name.startswith("nccl")]
    if not nccl:
        return None
    comp = sorted((e.time_range.start, e.time_range.end) for e in evs if not e.name.startswith("nccl"))

    def union(iv):
        out = []
        for a, b in sorted(iv):
            if out and a <= out[-1][1]:
                out[-1][1] = max(out[-1][1], b)
            else:
                out.append([a, b])
        return out
    cu, nu = union(comp), union((a, b) for a, b, _ in nccl)
    exposed, j = 0.0, 0
    for a, b in nu:                      # NCCL time minus its intersection with compute time
        covered = 0.0
        while j < len(cu) and cu[j][1] <= a:
            j += 1
        k = j
        while k < len(cu) and cu[k][0] < b:
            covered += max(0.0, min(b, cu[k][1]) - max(a, cu[k][0]))
            k += 1
        exposed += (b - a) - covered
    names = {}
    for a, b, n in nccl:
        d = names.setdefault(n[:90], [0, 0.0])
        d[0] += 1
        d[1] += (b - a) * 1e-3
    return {"nccl_kernels": {n: {"launches_per_step": c / replays, "ms_per_step": round(ms / replays, 4)} for n, (c, ms) in names.items()},
            "nccl_resident_ms_per_step": round(sum(b - a for a, b in nu) * 1e-3 / replays, 4),
            "compute_busy_ms_per_step": round(sum(b - a for a, b in cu) * 1e-3 / replays, 4),
            "exposed_comm_ms_per_step": round(exposed * 1e-3 / replays, 4),
            "how": "CUPTI kernel records of the replayed step graph; exposed = NCCL-resident time with no compute kernel running"}


def events_accounting(records):
    agg, shapes = {}, {}
    for name, work, e0, e1 in records:
        ms = e0.elapsed_time(e1)
        a = agg.setdefault(name, dict(ms=0.0, calls=0, flop=0.0, byte=0.0))
        a["ms"] += ms
        a["calls"] += 1
        if work:
            a[work[0]] += work[1]
        if work and len(work) > 2:
            sh = shapes.setdefault((name, work[2]), dict(ms=0.0, calls=0, amount=0.0, kind=work[0]))
            sh["ms"] += ms; sh["calls"] += 1; sh["amount"] += work[1]
    return agg, shapes


def summarize(agg, shapes, steps, pk):
    by_shape = []
    for (name, tag), a in sorted(shapes.items(), key=lambda kv: -kv[1]["ms"])[:40]:
        rate = a["amount"] / (a["ms"] * 1e-3)
        by_shape.append({"kernel": name, "shape": tag, "ms_per_step": round(a["ms"] / steps, 4), "calls_per_step": a["calls"] / steps,
                         ("tflops" if a["kind"] == "flop" else "gbs"): round(rate / (1e12 if a["kind"] == "flop" else 1e9), 1)})
    out = {}
    for name, a in agg.items():
        d = dict(ms_per_step=a["ms"] / steps, calls_per_step=a["calls"] / steps)
        if a["flop"]:
            d["tflops"] = a["flop"] / (a["ms"] * 1e-3) / 1e12
            d["frac_of_bf16_sustained"] = d["tflops"] / pk["tf_sust"]
            d["frac_of_bf16_burst"] = d["tflops"] / pk["tf_burst"]
        if a["byte"]:
            d["gbs"] = a["byte"] / (a["ms"] * 1e-3) / 1e9
            d["frac_of_hbm"] = d["gbs"] / pk["hbm"]
        out[name] = d
    return out, by_shape


DUMP_PARAM_SAMPLES = 1 << 22          # 16 MB of float32 out of the model's ~120 M parameters


def dump_outputs(out_dir, loss, items, grad_norm, model):
    """What one training step hands back, as float32 .npy files: the loss vector it returns (loss * B and the detached
    box / cls / dfl items), the gradient norm it clipped with, and the parameters its optimizer step wrote.  Parameters
    are taken over model.parameters() in declaration order; above DUMP_PARAM_SAMPLES of them, at positions drawn from a
    fixed seed, so that two builds of the same model are compared at the same weights."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    params = torch.cat([p.detach().reshape(-1).float() for p in model.parameters()])
    if params.numel() > DUMP_PARAM_SAMPLES:
        g = torch.Generator().manual_seed(0)
        idx = torch.randint(0, params.numel(), (DUMP_PARAM_SAMPLES,), generator=g).sort().values
        params = params[idx.to(params.device)]
    arrays = {"loss": loss, "loss_items": items, "grad_norm": grad_norm, "params_sample": params}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


# ------------------------------------------------------------------------------------------------
# our arm: one configuration
# ------------------------------------------------------------------------------------------------
def measure_config(args, cfg_idx, dev, rank, local, world, pk, full):
    """Device-resident throughput, end-to-end throughput, per-kernel accounting of one BASELINE.json config.
    `full`: also e2e + kernel accounting (the main line); the cfg3 sub-record keeps e2e but skips the kernel table."""
    import torch
    import torch.distributed as dist
    from snn_object_detectionddp_b200 import _lib
    from snn_object_detectionddp_b200.data import DevicePrefetcher, synthetic_batch
    from snn_object_detectionddp_b200.model import YOLOTemporalUNet
    from snn_object_detectionddp_b200.trainer import Trainer
    from snn_object_detectionddp_b200.weight_initialization import initialize_model

    B, T, HW = workload(args, cfg_idx)
    torch.manual_seed(42)
    model = YOLOTemporalUNet(num_classes=NUM_CLASSES, yolo_model_name="yolo11m.pt", use_conv_lstm=True, hyp=HYP, neuron=args.neuron)
    initialize_model(model)
    trainer = Trainer(model, max_lr=MAX_LR, weight_decay=WEIGHT_DECAY, total_steps=1000, device=dev,
                      bucket_mb=int(os.environ.get("SNN_BUCKET_MB", "32")))
    frames_cpu, labels_cpu = synthetic_batch(B, T, HW, HW, nc=NUM_CLASSES, seed=42 + rank)
    frames = frames_cpu.to(dev)
    MAXB = 8                                              # synthetic labels: 0-7 boxes per sample (SURVEY 8d)
    batch_dev = {"padded": tuple(t.to(dev) for t in trainer.prepare_batch(labels_cpu, B, max_boxes=MAXB)["padded"])}
    graphed = not args.no_graph
    step_fn = trainer.train_step_graphed if graphed else trainer.train_step

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if args.dump_trace and full and rank == 0:
        trainer.train_step(frames, batch_dev)
        _lib.trace = tr_ = []
        trainer.train_step(frames, batch_dev)
        _lib.trace = None
        json.dump([[n, (list(w) if w else None)] for n, w in tr_], open(args.dump_trace, "w"))

    # ---------------- device-resident throughput ----------------
    trace = None
    for i in range(max(args.warmup, 3)):                  # >= 3: two eager steps, then the graph capture + first replay
        if graphed and i == 2:
            _lib.trace = trace = []                       # the ABI calls recorded INTO the graph = launches of one replay
        step_fn(frames, batch_dev)
        _lib.trace = None
    barrier()
    if graphed and (trainer._graph is None or trainer._graph_failed):
        raise RuntimeError("CUDA-graph capture of the training step failed; rerun with --no-graph to time eager launches")
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    records = None if (args.no_profile or graphed or not full) else []
    _lib.profile = records
    launches0 = _lib.launch_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        loss, items = step_fn(frames, batch_dev)
    ev1.record()
    barrier()
    _lib.profile = None
    launches = len(trace) * args.steps if graphed else _lib.launch_count - launches0
    ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms)
    last_loss = [float(v) for v in items]
    # before the accounting replays below: a graphed step returns the graph's static buffers, which every replay overwrites
    if args.dump_outputs and full and rank == 0:
        dump_outputs(args.dump_outputs, loss, items, trainer.grad_norm, model)

    # ---------------- per-kernel accounting + roofline of the dominant kernel ----------------
    # (done right after the timed region, before the e2e leg re-captures the graph for uint8 host frames)
    res = dict(B=B, T=T, HW=HW, value=world * B * args.steps / (ms_total * 1e-3), ms_per_step=ms_total / args.steps, e2e=None, clocks=None,
               launches=launches, last_loss=last_loss, lockstep=None, graphed=graphed, kernels=None, by_shape=None, roofline=None,
               timing=None, kernel_ms_sum=None, other_kernels=None, comm_timeline=None)
    if full and not args.no_profile:
        acc, timing, kernel_sum, other = None, None, None, None
        if graphed:
            got, why = cupti_graph_accounting(lambda: trainer.train_step_graphed(frames, batch_dev), trace, 3)
            if got is not None:
                agg, shapes, other_d, total = got
                res["comm_timeline"] = other_d.pop("__comm__", None)
                acc, timing, kernel_sum = (agg, shapes, 3), "CUPTI activity records of 3 extra replays of the captured graph, matched to the ABI calls in launch order", total / 3
                other = {k: round(v / 3, 4) for k, v in sorted(other_d.items(), key=lambda kv: -kv[1])[:12]}
            else:
                timing = "fallback to CUDA events around eager launches: " + why
        if acc is None:
            records = records if records else []
            if not records:
                _lib.profile = records
                torch.cuda._sleep(int(1.5e8))            # hold the stream ~75 ms so the launches below queue up back to back
                for _ in range(args.steps):
                    trainer.train_step(frames, batch_dev)
                barrier()
                _lib.profile = None
            agg, shapes = events_accounting(records)
            acc, kernel_sum = (agg, shapes, args.steps), sum(a["ms"] for a in agg.values()) / args.steps
            timing = (timing or "") + " CUDA events around every ABI call of an eager pass"
        agg, shapes, nsteps = acc
        res["kernels"], res["by_shape"] = summarize(agg, shapes, nsteps, pk)
        res["timing"], res["kernel_ms_sum"], res["other_kernels"] = timing, kernel_sum, other
        name, a = max(agg.items(), key=lambda kv: kv[1]["ms"])
        tr_path = os.path.join(ROOT, "profiles", "traffic.json")       # dram bytes per launch from the committed ncu capture
        traffic = json.load(open(tr_path)).get(name) if os.path.isfile(tr_path) else None
        if a["flop"]:
            ach = a["flop"] / (a["ms"] * 1e-3) / 1e12
            res["roofline"] = {"kernel": name, "bound": "tensor", "achieved": ach, "peak": pk["tf_burst"], "unit": "TFLOP/s",
                               "frac": ach / pk["tf_burst"], "frac_of_sustained": ach / pk["tf_sust"], "frac_of_nominal_2250": ach / 2250.0,
                               "traffic": traffic, "peak_source": pk["src"] + ", burst bf16 (the timed region is a fraction of a second at max clocks)",
                               "share_of_step": a["ms"] / nsteps / (ms_total / args.steps), "launches_per_step": a["calls"] / nsteps}
        else:
            ach = a["byte"] / (a["ms"] * 1e-3) / 1e9
            res["roofline"] = {"kernel": name, "bound": "hbm", "achieved": ach, "peak": pk["hbm"], "unit": "GB/s", "frac": ach / pk["hbm"],
                               "frac_of_nominal_8000": ach / 8000.0, "traffic": traffic, "peak_source": pk["src"],
                               "share_of_step": a["ms"] / nsteps / (ms_total / args.steps), "launches_per_step": a["calls"] / nsteps}
    # ---------------- end to end through the public API with host buffers ----------------
    e2e = None
    if not args.no_e2e:
        # host frames as the dataset decodes them: uint8 RGB (reference dataset.py:139-152 converts to fp32 / 255 on the HOST and
        # ships 4x the bytes); the division runs in the frame packer kernel, bit-identical to the host's
        frames_u8 = (frames_cpu * 255.0).round().clamp_(0, 255).to(torch.uint8)
        host_batches = [(frames_u8.clone().pin_memory(),
                         tuple(t.pin_memory() for t in trainer.prepare_batch(labels_cpu, B, max_boxes=MAXB)["padded"])) for _ in range(2)]
        loss_host = torch.zeros(args.steps + args.warmup, 3).pin_memory()
        pf = DevicePrefetcher(dev)

        def e2e_steps(n, base):
            pf.stage(*host_batches[0])
            for i in range(n):
                frames_d, padded_d = pf.take()
                if i + 1 < n:
                    pf.stage(*host_batches[(i + 1) % 2])        # prefetch the next batch while this step computes
                _, it = step_fn(frames_d, {"padded": padded_d})
                pf.release()
                loss_host[base + i].copy_(it, non_blocking=True)     # D2H read of the step's result

        e2e_steps(args.warmup, 0)
        barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        e2e_steps(args.steps, args.warmup)
        t1.record()
        barrier()
        ems = torch.tensor([t0.elapsed_time(t1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ems, op=dist.ReduceOp.MAX)
        e2e = {"value": world * B * args.steps / (float(ems) * 1e-3), "unit": "images/s", "h2d_bytes_per_step": pf.bytes_per_batch(),
               "d2h_bytes_per_step": 12, "ms_per_step": float(ems) / args.steps,
               "api": ("Trainer.train_step_graphed" if graphed else "Trainer.train_step")
                      + " fed by data.DevicePrefetcher: double-buffered pinned host frames (uint8 [B,T,3,H,W], /255 on the device)"
                        " + padded labels, copied on a side stream"}
    clocks = sampler.stop() if rank == 0 else None          # sampled over the timed regions (device-resident, accounting replays, e2e)
    res["e2e"], res["clocks"] = e2e, clocks

    # ---------------- every rank holds the same parameters after the timed steps ----------------
    lockstep = None
    if world > 1:
        st = trainer.store
        chk = torch.stack([st.flat_p.double().sum(), st.flat_p.double().abs().sum(), st.flat_m.double().abs().sum()])
        allc = [torch.zeros_like(chk) for _ in range(world)]
        dist.all_gather(allc, chk)
        lockstep = bool(all(torch.equal(allc[0], c) for c in allc[1:]))
    res["lockstep"] = lockstep

    res["graph_active"] = bool(graphed and trainer._graph is not None and not trainer._graph_failed)
    trainer._graph = None
    del trainer, model
    torch.cuda.empty_cache()
    return res


def run_ours(args):
    import torch
    import torch.distributed as dist
    from snn_object_detectionddp_b200 import _lib

    rank, local, world = (int(os.environ.get(k, d)) for k, d in (("RANK", "0"), ("LOCAL_RANK", "0"), ("WORLD_SIZE", "1")))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.lib()        # fail loudly if libsnnb200.so is missing: there is no fallback
    pk = peaks()
    main = measure_config(args, args.config, dev, rank, local, world, pk, full=True)
    cfg3 = None
    if args.config != 3 and not args.no_cfg3:
        r3 = measure_config(args, 3, dev, rank, local, world, pk, full=False)
        cfg3 = {"workload": workload_name(args, r3["B"], r3["T"], r3["HW"], 3), "value": r3["value"], "unit": "images/s",
                "ms_per_step": r3["ms_per_step"], "per_gpu_batch": r3["B"], "T": r3["T"], "frames_per_s": r3["value"] * r3["T"],
                "e2e": r3["e2e"], "clocks": r3["clocks"], "gpu_launches": r3["launches"], "cuda_graph_active": r3["graph_active"],
                "ranks_in_lockstep": r3["lockstep"], "last_loss_items": r3["last_loss"]}

    def shutdown():
        """Leave without waiting on NCCL teardown: destroy_process_group() was seen to block for minutes on the 2-GPU box
        after the result line was out (captured graphs had referenced the communicator's kernels)."""
        sys.stdout.flush()
        sys.stderr.flush()
        if world > 1:
            torch.cuda.synchronize()
            dist.barrier()
            torch.cuda.synchronize()
            os._exit(0)

    if world > 1:
        dist.barrier()
    if rank != 0:
        shutdown()
        return

    B, T, HW = main["B"], main["T"], main["HW"]
    cpu_baseline = gpu_eager = lif = None
    dropin = None
    if world == 1 and not args.no_gpu_eager:
        gpu_eager = gpu_eager_run(T, HW, B, 3, 2, args.neuron, dev)
        dropin = dropin_run(T, HW, B, 3, 2, args.neuron, dev)
    if world == 1 and not args.no_lif:
        s2 = ClockSampler(local)
        s2.start()
        rows = lif_sweep(pk, quick=True)
        lif = {"config": "BASELINE.json configs[3]: T in {4,8,16} x (C, HxW) in {(64,64^2),(128,64^2),(128,32^2),(256,32^2),(256,16^2),(512,16^2)}, "
                         "tensors >= 1 GiB (L2 is 126 MB), algorithmic bytes: fwd 6.125, bwd 14 (two recompute passes) per neuron-timestep",
               "hbm_peak_gbs": pk["hbm"], "rows": rows, "clocks": s2.stop(),
               "fwd_frac_min": min(r["fwd_frac"] for r in rows), "bwd_frac_min": min(r["bwd_frac"] for r in rows)}
    if world == 1 and not args.no_cpu_baseline:
        r = cpu_reference_run(T, HW, args.ref_batch, 3, 1, args.neuron)
        cpu_baseline = {"value": r["value"], "unit": "images/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]}

    line = {
        "metric": "train images/sec", "value": main["value"], "unit": "images/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": main["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": workload_name(args, B, T, HW),
                   "per_gpu_batch": B, "T": T, "frames_per_s": main["value"] * T,
                   "l2": "per-step working set (240 MB bf16 weights + GBs of activations) exceeds the 126 MB L2; no explicit flush",
                   "parallelism": f"dp{world}", "feature_extractor": "stand-in frozen pyramid (YOLO11m weights unobtainable offline)"},
        "clocks": main["clocks"], "e2e": main["e2e"], "gpu_launches": main["launches"], "roofline": main["roofline"],
        "cpu_baseline": cpu_baseline, "gpu_eager_baseline": gpu_eager, "dropin_eager": dropin, "cfg3": cfg3, "ranks_in_lockstep": main["lockstep"],
        "cuda_graph_active": main["graph_active"], "cuda_graph": main["graphed"],
        "dependent_launch": bool(_lib.lib().snn_get_dependent_launch()),
        "kernel_timing": main["timing"], "kernels": main["kernels"], "kernels_by_shape": main["by_shape"],
        "kernel_ms_sum_per_step": main["kernel_ms_sum"], "other_kernels_ms_per_step": main["other_kernels"],
        "comm_timeline": main["comm_timeline"], "lif_microbench": lif, "last_loss_items": main["last_loss"],
    }
    print(result_line(line), flush=True)
    shutdown()


RESULT_LINE_MAX = 8192       # bytes: readers of the result line keep a bounded tail of stdout (a 21 KB line arrived cut)


def result_line(rec):
    """The one JSON result line of the record: without the per-row LIF sweep (`--microbench lif` prints the rows), the
    per-shape kernel table cut to its 8 costliest entries and floats kept to 6 significant digits, which holds a
    single-GPU record below RESULT_LINE_MAX."""
    def r6(o):
        if isinstance(o, float):
            return float(f"{o:.6g}")
        if isinstance(o, dict):
            return {k: r6(v) for k, v in o.items()}
        if isinstance(o, list):
            return [r6(v) for v in o]
        return o
    rec = dict(rec)
    if rec.get("kernels_by_shape"):
        rec["kernels_by_shape"] = rec["kernels_by_shape"][:8]
    if rec.get("lif_microbench"):
        rec["lif_microbench"] = {k: v for k, v in rec["lif_microbench"].items() if k != "rows"}
    return json.dumps(r6(rec))


# ------------------------------------------------------------------------------------------------
# LIF microbench (BASELINE.json configs[3])
# ------------------------------------------------------------------------------------------------
def lif_sweep(pk, quick=False):
    import torch
    from snn_object_detectionddp_b200 import kernels as K
    from snn_object_detectionddp_b200._lib import call, ptr, stream_ptr
    rows = []
    for T in (4, 8, 16):
        for C, HWs in ((64, 64), (128, 64), (128, 32), (256, 32), (256, 16), (512, 16)):
            per_img = C * HWs * HWs
            Bn = max(1, (1 << 30) // (4 * T * per_img))          # fp32 input tensor >= 1 GiB (L2 is 126 MB)
            y = torch.randn(T * Bn, HWs, HWs, C, device="cuda")
            scale, shift = torch.ones(T, C, device="cuda"), torch.full((T, C), 0.2, device="cuda")
            mean, invstd = torch.zeros(T, C, device="cuda"), torch.ones(T, C, device="cuda")
            gs = torch.randn(T * Bn, HWs, HWs, C, device="cuda").to(torch.bfloat16)
            n = y.numel()

            def timeit(fn, reps=3 if quick else 5):
                fn(); torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(reps):
                    fn()
                e1.record(); torch.cuda.synchronize()
                return e0.elapsed_time(e1) / reps

            bnb = torch.full((C,), 0.2, device="cuda")
            dg, db = torch.zeros(C, device="cuda"), torch.zeros(C, device="cuda")
            red = torch.zeros(T, 2, C, device="cuda")
            dy = torch.empty_like(gs)
            P = n // (T * C)
            a = (ptr(y), ptr(scale), ptr(shift), ptr(mean), ptr(invstd), ptr(bnb), None, ptr(gs), None, ptr(red), ptr(dy), None,
                 ptr(dg), ptr(db), T, P, C, 0.5, 1.0, 2.0)
            K.require_cuda(y)
            f_ms = timeit(lambda: K.bn_act_fwd(0, y, scale, shift, T))
            r_ms = timeit(lambda: call("snn_bn_act_bwd2", 0, 0, *a, stream_ptr()))
            d_ms = timeit(lambda: call("snn_bn_act_bwd2", 1, 0, *a, stream_ptr()))
            be_ms = timeit(lambda: K.bn_act_bwd(0, False, y, scale, shift, mean, invstd, gs, T))
            # algorithmic bytes / neuron-timestep: fwd 4+2+1/8; train bwd pass 1 (reductions) 4+2, pass 2 (dx) 4+2+2;
            # frozen-statistics bwd 4+2+2
            rows.append(dict(T=T, C=C, HW=HWs, B=Bn, fwd_gbs=n * 6.125 / f_ms / 1e6, bwd_reduce_gbs=n * 6.0 / r_ms / 1e6,
                             bwd_dx_gbs=n * 8.0 / d_ms / 1e6, bwd_train_gbs=n * 14.0 / (r_ms + d_ms) / 1e6,
                             bwd_eval_gbs=n * 8.0 / be_ms / 1e6, fwd_ms=f_ms, bwd_reduce_ms=r_ms, bwd_dx_ms=d_ms))
            del y, gs, dy
    for r in rows:
        r["fwd_frac"], r["bwd_frac"] = r["fwd_gbs"] / pk["hbm"], r["bwd_train_gbs"] / pk["hbm"]
        r["fwd_frac_of_nominal_8000"], r["bwd_frac_of_nominal_8000"] = r["fwd_gbs"] / 8000.0, r["bwd_train_gbs"] / 8000.0
    return rows


def run_lif_microbench(args):
    import torch
    pk = peaks()
    torch.cuda.set_device(0)
    s = ClockSampler(0)
    s.start()
    rows = lif_sweep(pk)
    print(json.dumps({"microbench": "lif", "hbm_peak_gbs": pk["hbm"], "peak_source": pk["src"], "rows": rows, "clocks": s.stop()}), flush=True)


if __name__ == "__main__":
    a = parse()
    if a.microbench == "lif":
        run_lif_microbench(a)
    elif a.impl == "reference":
        run_reference(a)
    elif a.impl == "eager-gpu":
        run_gpu_eager(a)
    else:
        run_ours(a)
