#!/usr/bin/env python
"""blob_slab_bench.py -- BlobDog through the Z-slab drivers (visfd_cuda_blob_dog_stream / _multi) next to the
one-GPU call, on C3 and on a C5-shaped volume.

    python profiles/blob_slab_bench.py --out DIR [--steps K --warmup W] [--c3-budget-gb 5.5] [--no-c5]

1. Reads the card's name and power limit and the host's memory (nvidia-smi, /proc/meminfo; nothing is changed).
2. C3: bench.py's blob_c3_row input (1024x1024x512, seed 2, 64 dark blobs stamped in, 12 scales sigma = 2 * 4^(n/12),
   `-blob-s minima` thresholds) in pinned host memory.  Times, warm-up calls first:
     one_shot    Context.blob_dog from the host array (visfd_cuda_blob_dog, staged upload);
     stream_0    Context.blob_dog_stream with device_bytes = 0;
     stream_B    Context.blob_dog_stream with --c3-budget-gb, which takes at least 4 slabs;
     multi_4x0   blob_dog_multi on devices [0, 0, 0, 0];
     multi_all   blob_dog_multi on every device, when there is more than one.
   Each call reports its wall time, slab count, and for calls on the context its peak reserved bytes and its
   gauss / blob_scan / h2d stage times; multi reports the device time of each slab.  Every list must equal the
   one-shot lists bit for bit, in order.  upload_ms: CUDA events around one host-to-device copy of the volume.
3. C5 shape (4096x4096x1024, bench.py's seeded volume, 68.7 GB per float volume) with the same scales: the one-shot
   call's refusal, one stream call at device_bytes = 0, and one multi call on every device when there is more than
   one (on one GPU every multi slab would run at once on that device, so it is not attempted); the stream and
   multi lists must be equal.  upload_ms: events around copies of the whole volume, 4 GiB at a time.  A host
   without the memory to pin the volume records why the row was skipped.

Writes DIR/blob_slab_bench.json and prints it.  A number is only meaningful with the card it was measured on, which
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
import bench   # the workloads' shapes; (importing it points file descriptor 1 at stderr, as bench.py does)
from stream_bench import gpu_info, host_volume

STAGES = ("gauss", "blob_scan", "h2d")
SIGMAS = 2.0 * 4.0 ** (np.arange(12) / 12)
RATIO = float(np.sqrt(-2.0 * np.log(0.03)))
# `-blob-s minima` defaults (bin/filter_mrc/settings.cpp:1674-1678, :121-123), as bench.py's C3 row
KW = dict(delta=0.02, truncate_ratio=RATIO, minima_threshold=0.0, maxima_threshold=-np.inf,
          use_threshold_ratios=False)


def c3_host_volume(dev):
    """bench.py blob_c3_row's volume, in pinned host memory"""
    import torch
    from visfd_b200 import synth
    shape = bench.WORKLOADS["C3"]
    vol = synth.tomogram_torch(shape, dev, seed=2, n_shells=0)
    rng = np.random.default_rng(3)
    for _ in range(64):
        bs = rng.uniform(3.0, 6.0)
        c = [rng.uniform(24, d - 24) for d in shape]
        lo = [int(ci - 4 * bs) for ci in c]
        hi = [int(ci + 4 * bs) + 1 for ci in c]
        ax = [torch.arange(a, b, dtype=torch.float32, device=dev) - ci for a, b, ci in zip(lo, hi, c)]
        r2 = ax[0][:, None, None] ** 2 + ax[1][None, :, None] ** 2 + ax[2][None, None, :] ** 2
        vol[lo[0]:hi[0], lo[1]:hi[1], lo[2]:hi[2]] -= 4.0 * torch.exp(-0.5 * r2 / (bs * bs))
    h = torch.empty(shape, dtype=torch.float32, pin_memory=True)
    h.copy_(vol)
    del vol
    torch.cuda.empty_cache()
    return h


def upload_ms(h, dev, chunk_bytes=4 << 30):
    """CUDA events around host-to-device copies of every byte of h, chunk_bytes at a time into one buffer"""
    import torch
    flat = h.view(-1)
    n = min(flat.numel(), chunk_bytes // 4)
    buf = torch.empty(n, dtype=torch.float32, device=dev)
    buf.copy_(flat[:n], non_blocking=True)   # warm-up
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(0, flat.numel(), n):
        k = min(n, flat.numel() - i)
        buf[:k].copy_(flat[i:i + k], non_blocking=True)
    e1.record()
    torch.cuda.synchronize()
    del buf
    torch.cuda.empty_cache()
    return e0.elapsed_time(e1)


def same_lists(a, b):
    return all(x.shape == y.shape and np.array_equal(x.view(np.int32), y.view(np.int32)) for x, y in zip(a, b))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--c3-budget-gb", type=float, default=5.5)
    ap.add_argument("--no-c5", action="store_true")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    res = {"gpu": gpu_info(), "sigmas": [float(s) for s in SIGMAS], "truncate_ratio": RATIO,
           "steps": args.steps, "warmup": args.warmup}

    import torch
    import visfd_b200
    dev = torch.device("cuda", 0)
    ctx = visfd_b200.Context(0)
    ctx.set_timing(True)
    ndev = visfd_b200.load_library().visfd_cuda_device_count()

    def timed(fn, pooled):
        if pooled:
            ctx.trim()
            ctx.reset_peak_reserved_bytes()
            ctx.reset_stage_ms()
        torch.cuda.synchronize()
        t = time.perf_counter()
        r = fn()
        r["wall_ms"] = (time.perf_counter() - t) * 1e3
        if pooled:
            r["peak_reserved_bytes"] = ctx.peak_reserved_bytes()
            r["stage_ms"] = {k: ctx.stage_ms(k) for k in STAGES}
        return r

    def one_shot(src, capacity):
        def run():
            mn, mx = ctx.blob_dog(src, SIGMAS, capacity=capacity, **KW)
            return {"minima": mn, "maxima": mx, "n_slabs": 1}
        return run

    def stream(src, capacity, device_bytes):
        def run():
            return ctx.blob_dog_stream(src, SIGMAS, capacity=capacity, device_bytes=device_bytes, **KW)
        return run

    def multi(src, capacity, devices):
        def run():
            r = visfd_b200.blob_dog_multi(devices, src, SIGMAS, capacity=capacity, **KW)
            r["n_slabs"] = len(devices)
            return r
        return run

    def report(r, ref):
        out = {k: v for k, v in r.items() if k not in ("minima", "maxima")}
        out["n_minima"], out["n_maxima"] = len(r["minima"]), len(r["maxima"])
        out["lists_equal_reference"] = same_lists((r["minima"], r["maxima"]), ref)
        return out

    # ---- C3 ----------------------------------------------------------------------------------------------------
    h3 = c3_host_volume(dev)
    src3, cap3 = h3.numpy(), 1 << 24
    c3 = {"shape": list(bench.WORKLOADS["C3"]), "budget_bytes": int(args.c3_budget_gb * 1e9),
          "upload_ms": upload_ms(h3, dev)}
    calls = [("one_shot", one_shot(src3, cap3), True), ("stream_0", stream(src3, cap3, 0), True),
             ("stream_B", stream(src3, cap3, c3["budget_bytes"]), True),
             ("multi_4x0", multi(src3, cap3, [0, 0, 0, 0]), False)]
    if ndev > 1:
        calls.append(("multi_all", multi(src3, cap3, list(range(ndev))), False))
    ref = one_shot(src3, cap3)()
    ref = (ref["minima"], ref["maxima"])
    runs = {}
    for step in range(args.warmup + args.steps):
        for name, fn, pooled in calls:
            r = report(timed(fn, pooled), ref)
            print("C3", name, json.dumps(r), file=sys.stderr, flush=True)
            if step >= args.warmup:
                runs.setdefault(name, []).append(r)
    c3["runs"] = {name: dict(rs[-1], wall_ms=[r["wall_ms"] for r in rs],
                             wall_ms_median=statistics.median(r["wall_ms"] for r in rs),
                             lists_equal_reference=all(r["lists_equal_reference"] for r in rs))
                  for name, rs in runs.items()}
    c3["all_lists_equal"] = all(v["lists_equal_reference"] for v in c3["runs"].values())
    res["C3"] = c3
    del h3, src3
    ctx.trim()

    # ---- C5 shape --------------------------------------------------------------------------------------------
    shape5 = bench.WORKLOADS["C5"]
    c5 = {"shape": list(shape5)}
    res["C5"] = c5
    vol_bytes = int(np.prod(shape5)) * 4
    avail = gpu_info()["host_mem_available"] or 0
    if args.no_c5:
        c5["skipped"] = "--no-c5"
    elif avail < vol_bytes + (32 << 30):
        c5["skipped"] = f"host memory available {avail} bytes; pinning the volume needs {vol_bytes} + 32 GiB"
    else:
        try:
            h5 = host_volume(shape5, dev)
        except RuntimeError as e:
            h5 = None
            c5["skipped"] = f"pinning {vol_bytes} bytes failed: {e}"
        if h5 is not None:
            src5, cap5 = h5.numpy(), 1 << 28
            c5["upload_ms"] = upload_ms(h5, dev)
            try:
                ctx.blob_dog(src5, SIGMAS, capacity=16, **KW)
                c5["one_shot_refusal"] = None
            except visfd_b200.VisfdCudaError as e:
                c5["one_shot_refusal"] = str(e)
            ctx.trim()
            r = timed(stream(src5, cap5, 0), True)
            ref5 = (r["minima"], r["maxima"])
            c5["runs"] = {"stream_0": report(r, ref5)}
            print("C5 stream_0", json.dumps(c5["runs"]["stream_0"]), file=sys.stderr, flush=True)
            ctx.trim()
            if ndev > 1:
                r = timed(multi(src5, cap5, list(range(ndev))), False)
                c5["runs"]["multi_all"] = report(r, ref5)
                print("C5 multi_all", json.dumps(c5["runs"]["multi_all"]), file=sys.stderr, flush=True)
            else:
                c5["multi_all"] = "not run: one GPU, whose single slab would be the whole volume"
            c5["all_lists_equal"] = all(v["lists_equal_reference"] for v in c5["runs"].values())
            del h5, src5

    res["gpu_after"] = gpu_info()["nvidia_smi"]
    with open(os.path.join(args.out, "blob_slab_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))
    ctx.close()


if __name__ == "__main__":
    main()
