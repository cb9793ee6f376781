#!/usr/bin/env python
"""background_bench.py -- `-membrane-background` in the slab drivers on the C4 volume, next to the one-GPU call.

    python profiles/background_bench.py --out DIR [--steps K --warmup W] [--budget-gb 24] [--background-sigma 12]

1. Reads the card's name and power limit (nvidia-smi; nothing is changed).
2. bench.py's C4 volume (2048x2048x1024, seed 0) in pinned host memory, with bench.py's parameters and
   background_sigma = 12 (half-width 31, a slab halo of 20 + 31 planes).
3. Times, alternated, warm-up calls first, each with and without the background:
     one_shot     Context.membrane (visfd_cuda_membrane[_background]) from the host arrays;
     stream_0     Context.membrane_stream with device_bytes = 0;
     stream_B     Context.membrane_stream with a budget of --budget-gb, which takes several slabs;
     multi_4x0    membrane_multi on devices [0, 0, 0, 0];
     multi_all    membrane_multi on every device, when there is more than one.
   The multi calls run after the others: their per-slot contexts keep their cached blocks on the device.
4. Reports wall time, slab count, peak reserved bytes and the gauss / ridge / tv stage times of each call (multi:
   the device time of each slab), and checks that each call's bits_sum_i64 equals the one-shot call's with the same
   background.

Writes DIR/background_bench.json and prints it.  A number is only meaningful with the card it was measured on, which
the file carries.
"""
import argparse
import json
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))
import bench   # the workload's parameters; (importing it points file descriptor 1 at stderr, as bench.py does)
from stream_bench import gpu_info, host_volume

STAGES = ("gauss", "ridge", "select", "compact", "tv")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--budget-gb", type=float, default=24.0)
    ap.add_argument("--background-sigma", type=float, default=12.0)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    res = {"gpu": gpu_info(), "workload": "C4", "shape": list(bench.WORKLOADS["C4"]),
           "background_sigma": args.background_sigma, "budget_bytes": int(args.budget_gb * 1e9),
           "steps": args.steps, "warmup": args.warmup}

    import torch
    import visfd_b200
    dev = torch.device("cuda", 0)
    ctx = visfd_b200.Context(0)
    ctx.set_timing(True)
    ndev = visfd_b200.load_library().visfd_cuda_device_count()
    shape = bench.WORKLOADS["C4"]
    h_src = host_volume(shape, dev)
    h_out = torch.empty(shape, dtype=torch.float32, pin_memory=True)
    src, out = h_src.numpy(), h_out.numpy()
    p = (bench.SIGMA, bench.RATIO, visfd_b200.DECREASING_EIVALS, bench.TV_BEST, True, bench.TV_SIGMA, 4, bench.SQ2)
    budget = int(args.budget_gb * 1e9)

    def one_shot(bg):
        r = ctx.membrane(src, *p, out=out, background_sigma=bg)
        return {"threshold": r["threshold"], "n_slabs": 1}

    def stream(device_bytes):
        def run(bg):
            r = ctx.membrane_stream(src, *p, out=out, device_bytes=device_bytes, background_sigma=bg)
            return {"threshold": r["threshold"], "n_slabs": r["n_slabs"]}
        return run

    def multi(devices):
        def run(bg):
            r = visfd_b200.membrane_multi(devices, src, *p, out=out, background_sigma=bg)
            return {"threshold": r["threshold"], "n_slabs": len(devices), "device_ms": r["device_ms"]}
        return run

    def timed(fn, bg, pooled):
        if pooled:
            ctx.trim()
            ctx.reset_peak_reserved_bytes()
            ctx.reset_stage_ms()
        torch.cuda.synchronize()
        t = time.perf_counter()
        r = fn(bg)
        r["wall_ms"] = (time.perf_counter() - t) * 1e3
        if pooled:
            r["peak_reserved_bytes"] = ctx.peak_reserved_bytes()
            r["stage_ms"] = {k: ctx.stage_ms(k) for k in STAGES}
        r["bits_sum_i64"] = int(h_out.view(torch.int32).sum(dtype=torch.int64).item())
        return r

    # (name, call, uses ctx's pool and stage timers)
    groups = [[("one_shot", one_shot, True), ("stream_0", stream(0), True), ("stream_B", stream(budget), True)],
              [("multi_4x0", multi([0, 0, 0, 0]), False)]]
    if ndev > 1:
        groups[1].append(("multi_all", multi(list(range(ndev))), False))
    runs = {}
    for group in groups:
        ctx.trim()
        for step in range(args.warmup + args.steps):
            for name, fn, pooled in group:
                for bg in (args.background_sigma, 0.0):
                    r = timed(fn, bg, pooled)
                    r["step"] = step
                    key = f"{name}{'_background' if bg > 0 else ''}"
                    print(key, json.dumps(r), file=sys.stderr, flush=True)
                    if step >= args.warmup:
                        runs.setdefault(key, []).append(r)

    summary = {}
    for key, rs in runs.items():
        ref = runs["one_shot_background" if key.endswith("_background") else "one_shot"][0]
        summary[key] = {
            "wall_ms_median": statistics.median(r["wall_ms"] for r in rs),
            "wall_ms": [r["wall_ms"] for r in rs],
            "n_slabs": rs[-1]["n_slabs"],
            "peak_reserved_bytes": rs[-1].get("peak_reserved_bytes"),
            "stage_ms": rs[-1].get("stage_ms"),
            "device_ms": rs[-1].get("device_ms"),
            "threshold": rs[-1]["threshold"],
            "bits_sum_i64": rs[-1]["bits_sum_i64"],
            "matches_one_shot": all(r["bits_sum_i64"] == ref["bits_sum_i64"] and r["threshold"] == ref["threshold"]
                                    for r in rs),
        }
    res["runs"] = summary
    res["all_checksums_equal"] = all(v["matches_one_shot"] for v in summary.values())
    res["gpu_after"] = gpu_info()["nvidia_smi"]
    with open(os.path.join(args.out, "background_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))
    ctx.close()


if __name__ == "__main__":
    main()
