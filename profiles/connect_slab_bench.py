#!/usr/bin/env python
"""connect_slab_bench.py -- the membrane pipeline with `-connect` over Z-slabs (visfd_cuda_membrane_connect_stream /
_multi) next to the one-GPU composition (visfd_cuda_membrane with its tensor, then visfd_cuda_label_connected).

    python profiles/connect_slab_bench.py --out DIR [--steps 2 --warmup 1] [--skip-c4]

1. Reads the card's name and power limit (nvidia-smi; nothing is changed).
2. (a) bench.py's seeded volume (synth.tomogram_torch, seed 0) built at 512x2048x2048, with bench.py's parameters and -connect at the 90th percentile of the positive scores, angle 30.  Times, alternated, after the
   warm-up rounds:
     composition  Context.membrane(want_tensor=True) + Context.label_connected, host arrays (the tensor goes to the
                  host and back);
     stream_0     Context.membrane_connect_stream with device_bytes = 0;
     stream_q     the same under a quarter of the composition's peak pool;
     multi_4x0    membrane_connect_multi on devices [0, 0, 0, 0].
   Each row: wall time, slabs, peak pool bytes (not for multi: its contexts are internal), the host flood's time
   (stage "flood"; multi: not separated), clusters, and whether out and labels equal the composition's.
3. (b) The whole C4 volume (1024x2048x2048): stream at device_bytes = 0 (wall time, slabs, peak pool, clusters, flood
   time), and what the composition does there: its message when it is refused.

Writes DIR/connect_slab_bench.json and prints it.  A number is only meaningful with the card it was measured on, which
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

ANGLE = 30.0


def main():
    def write(res):
        with open(os.path.join(args.out, "connect_slab_bench.json"), "w") as f:
            json.dump(res, f, indent=1)

    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--skip-c4", action="store_true")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    import torch
    import visfd_b200
    dev = torch.device("cuda", 0)
    ctx = visfd_b200.Context(0)
    p = (bench.SIGMA, bench.RATIO, visfd_b200.DECREASING_EIVALS, bench.TV_BEST, True, bench.TV_SIGMA, 4, bench.SQ2)
    res = {"gpu": gpu_info(), "params": list(p), "angle_deg": ANGLE, "steps": args.steps, "warmup": args.warmup}

    def pooled(fn):
        ctx.trim()
        ctx.reset_peak_reserved_bytes()
        ctx.reset_stage_ms()
        t = time.perf_counter()
        r = fn()
        r["wall_ms"] = (time.perf_counter() - t) * 1e3
        r["peak_reserved_bytes"] = ctx.peak_reserved_bytes()
        r["flood_ms"] = ctx.stage_ms("flood")
        return r

    # ---- (a) 512 planes: the composition fits ----
    full = bench.WORKLOADS["C4"]
    shape = (512,) + tuple(full[1:])
    h_src = host_volume(shape, dev)
    src = h_src.numpy()
    r = ctx.membrane(src, *p)
    thr = float(np.quantile(r["out"][r["out"] > 0][::97], 0.9))
    del r
    res["a"] = {"shape": list(shape), "connect_threshold": thr}

    def composition():
        m = ctx.membrane(src, *p, want_tensor=True)
        lc = ctx.label_connected(m["out"], m["tensor"], thr, angle_deg=ANGLE)
        return dict(lc, out=m["out"], n_slabs=1)

    want = pooled(composition)
    res["a"]["composition_peak_reserved_bytes"] = want["peak_reserved_bytes"]
    quarter = want["peak_reserved_bytes"] // 4
    calls = [("composition", lambda: pooled(composition)),
             ("stream_0", lambda: pooled(lambda: ctx.membrane_connect_stream(src, *p, thr, angle_deg=ANGLE))),
             ("stream_q", lambda: pooled(lambda: ctx.membrane_connect_stream(src, *p, thr, angle_deg=ANGLE,
                                                                             device_bytes=quarter)))]

    def multi():
        t = time.perf_counter()
        r = visfd_b200.membrane_connect_multi([0, 0, 0, 0], src, *p, thr, angle_deg=ANGLE)
        r["wall_ms"] = (time.perf_counter() - t) * 1e3
        r["n_slabs"] = 4
        return r
    calls.append(("multi_4x0", multi))   # last: its contexts keep cached blocks on the device
    runs = {}
    for step in range(args.warmup + args.steps):
        for name, fn in calls:
            r = fn()
            row = {k: r.get(k) for k in ("wall_ms", "n_slabs", "peak_reserved_bytes", "flood_ms", "n_clusters",
                                         "device_ms")}
            row["equal_to_composition"] = bool(np.array_equal(r["out"].view(np.int32), want["out"].view(np.int32))
                                               and np.array_equal(r["labels"], want["labels"]))
            print(name, step, json.dumps(row), file=sys.stderr, flush=True)
            if step >= args.warmup:
                runs.setdefault(name, []).append(row)
            del r
    res["a"]["runs"] = {k: dict(v[-1], wall_ms=[x["wall_ms"] for x in v],
                                wall_ms_median=statistics.median(x["wall_ms"] for x in v),
                                flood_ms=[x["flood_ms"] for x in v]) for k, v in runs.items()}
    del src, h_src, want
    # ---- (b) C4 ----
    if not args.skip_c4:
        h_src = host_volume(full, dev)
        src = h_src.numpy()
        rows = []
        for step in range(args.warmup + args.steps):
            r = pooled(lambda: ctx.membrane_connect_stream(src, *p, thr, angle_deg=ANGLE))
            row = {k: r[k] for k in ("wall_ms", "n_slabs", "peak_reserved_bytes", "flood_ms", "n_clusters")}
            print("c4_stream_0", step, json.dumps(row), file=sys.stderr, flush=True)
            if step >= args.warmup:
                rows.append(row)
            del r
        res["b"] = {"shape": list(full), "stream_0": rows}
        write(res)   # (the composition below may exhaust the host)
        # the composition, step by step: the first call that is refused ends it
        ctx.trim()
        step = "visfd_cuda_membrane with the tensor"
        try:
            m = ctx.membrane(src, *p, want_tensor=True)
            step = "visfd_cuda_label_connected"
            ctx.label_connected(m["out"], m["tensor"], thr, angle_deg=ANGLE)
            res["b"]["composition"] = "ran"
        except visfd_b200.VisfdCudaError as e:
            res["b"]["composition"] = f"{step} refused: {e}"
    res["gpu_after"] = gpu_info()["nvidia_smi"]
    write(res)
    print(json.dumps(res, indent=1))
    ctx.close()


if __name__ == "__main__":
    main()
