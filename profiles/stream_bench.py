#!/usr/bin/env python
"""stream_bench.py -- visfd_cuda_membrane_stream (Context.membrane_stream) on one B200, next to bench.py.

    python profiles/stream_bench.py --out DIR [--steps K --warmup W] [--c4-budget-gb 24] [--c5-budget-gb 100]
                                           [--no-c4 | --no-c5]

1. Reads the card's name and power limit (nvidia-smi) and the host's memory.
2. C4 (2048x2048x1024, bench.py's parameters): `bench.py --gpus 1 --no-cpu-baseline --no-side-tables`, then the stream
   call on the same seeded volume from pinned host arrays with device_bytes = 0 and with a budget that forces several
   slabs: wall time, slab count, peak reserved bytes, stage times; its output's bits_sum_i64 must equal the bench
   line's checksum.bits_sum_i64.
3. C5 (4096x4096x1024): the stream call with device_bytes = 0 and with a smaller budget, the two checksums compared.
   Source and output need 137 GB of pinned host memory; a host without it records why C5 was not run.

Writes DIR/stream_bench.json and prints it.  A number is only meaningful with the card it was measured on, which the
file carries.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench   # the workload's parameters; (importing it points file descriptor 1 at stderr, as bench.py does)

STAGES = ("gauss", "ridge", "select", "compact", "tv")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,memory.total", "--format=csv,noheader"],
                       capture_output=True, text=True)
    mem = {}
    with open("/proc/meminfo") as f:
        for line in f:
            k, v = line.split(":", 1)
            mem[k] = int(v.split()[0]) * 1024
    return {"nvidia_smi": q.stdout.strip().splitlines(), "host_mem_total": mem.get("MemTotal"),
            "host_mem_available": mem.get("MemAvailable")}


def host_volume(shape, dev):
    """bench.py's seeded volume (synth.tomogram_torch, seed 0) in pinned host memory"""
    import torch
    from visfd_b200 import synth
    h = torch.empty(shape, dtype=torch.float32, pin_memory=True)
    for z in range(0, shape[0], 64):
        h[z:z + 64].copy_(synth.tomogram_torch(shape, dev, seed=0, z0=z, z1=min(shape[0], z + 64)))
    torch.cuda.empty_cache()
    return h


def stream_run(ctx, h_src, h_out, budget):
    import torch
    import visfd_b200
    ctx.trim()
    ctx.reset_peak_reserved_bytes()
    ctx.reset_stage_ms()
    t = time.perf_counter()
    r = ctx.membrane_stream(h_src.numpy(), bench.SIGMA, bench.RATIO, visfd_b200.DECREASING_EIVALS, bench.TV_BEST, True,
                            bench.TV_SIGMA, 4, bench.SQ2, out=h_out.numpy(), device_bytes=budget)
    wall = time.perf_counter() - t
    n = float(np.prod(h_src.shape))
    return {"device_bytes": budget, "wall_ms": wall * 1e3, "Gvoxel_per_s": n / wall / 1e9, "n_slabs": r["n_slabs"],
            "peak_reserved_bytes": ctx.peak_reserved_bytes(), "threshold": r["threshold"],
            "stage_ms": {k: ctx.stage_ms(k) for k in STAGES},
            "bits_sum_i64": int(h_out.view(torch.int32).sum(dtype=torch.int64).item())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--c4-budget-gb", type=float, default=24.0)
    ap.add_argument("--c5-budget-gb", type=float, default=100.0)
    ap.add_argument("--no-c4", action="store_true")
    ap.add_argument("--no-c5", action="store_true")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    res = {"gpu": gpu_info()}

    import torch
    import visfd_b200
    from visfd_b200 import synth
    dev = torch.device("cuda", 0)
    ctx = visfd_b200.Context(0)
    ctx.set_timing(True)
    # first launches load the kernels: a small call before the timed ones
    small = synth.tomogram((128, 128, 128), seed=0)
    ctx.membrane_stream(small, bench.SIGMA, bench.RATIO, visfd_b200.DECREASING_EIVALS, bench.TV_BEST, True,
                        bench.TV_SIGMA, 4, bench.SQ2, device_bytes=0)

    if not args.no_c4:
        cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--no-cpu-baseline", "--no-side-tables",
               "--steps", str(args.steps), "--warmup", str(args.warmup)]
        p = subprocess.run(cmd, capture_output=True, text=True)
        lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
        if p.returncode != 0 or not lines:
            raise SystemExit("bench.py failed:\n" + p.stderr[-4000:])
        b = json.loads(lines[-1])
        res["bench_c4"] = {"cmd": " ".join(cmd[1:]), "ms_per_step": b["ms_per_step"], "e2e": b["e2e"],
                           "stage_ms": b["stage_ms_rank0_last_step"], "checksum": b["checksum"]}

        shape = bench.WORKLOADS["C4"]
        h_src = host_volume(shape, dev)
        h_out = torch.empty(shape, dtype=torch.float32, pin_memory=True)
        runs = []
        for budget in (0, int(args.c4_budget_gb * 1e9)):
            r = stream_run(ctx, h_src, h_out, budget)
            r["matches_bench_checksum"] = r["bits_sum_i64"] == b["checksum"]["bits_sum_i64"]
            runs.append(r)
            print(json.dumps(r), file=sys.stderr, flush=True)
        res["stream_c4"] = runs
        del h_src, h_out
        torch._C._host_emptyCache()   # the pinned C4 buffers go back to the host

    shape = bench.WORKLOADS["C5"]
    need = 2 * 4 * int(np.prod(shape))
    avail = gpu_info()["host_mem_available"]
    if args.no_c5:
        res["stream_c5"] = {"run": False, "why": "--no-c5"}
    elif avail is None or avail < need * 1.05:
        res["stream_c5"] = {"run": False, "why": "source and output need %d bytes of pinned host memory; the host has "
                                                 "%s bytes available" % (need, avail)}
    else:
        h_src = host_volume(shape, dev)
        h_out = torch.empty(shape, dtype=torch.float32, pin_memory=True)
        runs = [stream_run(ctx, h_src, h_out, budget) for budget in (0, int(args.c5_budget_gb * 1e9))]
        res["stream_c5"] = {"run": True, "runs": runs,
                            "checksums_equal": runs[0]["bits_sum_i64"] == runs[1]["bits_sum_i64"],
                            "thresholds_equal": runs[0]["threshold"] == runs[1]["threshold"]}
    res["gpu_after"] = gpu_info()["nvidia_smi"]
    with open(os.path.join(args.out, "stream_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))
    ctx.close()


if __name__ == "__main__":
    main()
