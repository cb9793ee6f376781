#!/usr/bin/env python
"""filter_slab_bench.py -- ApplyGauss / ApplyDog / ApplyLog through the Z-slab drivers (visfd_cuda_filter_stream /
_multi) next to the one-shot host call, on C4 and on a C5-shaped volume.

    python profiles/filter_slab_bench.py --out DIR [--steps K --warmup W] [--no-c5]

1. Reads the card's name and power limit and the host's memory (nvidia-smi, /proc/meminfo; nothing is changed).
2. C5 shape first (4096x4096x1024, bench.py's seeded volume, 68.7 GB per float volume), before any multi call has
   left blocks cached on the device: the Gaussian sigma = 2 (filter_mrc's half-width), in place (out = src) so that
   one pinned array suffices.  The one-shot call's refusal is recorded, then one stream call at device_bytes = 0.  A
   host without the memory to pin the volume records why the row was skipped.
3. C4 (1024x2048x2048, bench.py's seeded volume) in pinned host memory, the result into a second pinned array, for
   the Gaussian sigma = 2 / 4 / 8, DoG sigma 4 / 6.4 (each with the half-width of its own sigma, as filter_mrc's
   -dog) and LoG sigma = 4.  Each round times, per filter:
     one_shot    visfd_cuda_apply_gauss / _dog2 / _log from the host arrays (staged through the device);
     stream_0    Context.filter_stream with device_bytes = 0;
     stream_B    Context.filter_stream with a quarter of the one-shot call's peak pool, which takes >= 4 slabs;
     multi_4x0   filter_multi on devices [0, 0, 0, 0].
   --warmup rounds first, then --steps timed rounds.  Each call reports its wall time, slab count, and for calls on
   the context its peak reserved bytes and its gauss / h2d / d2h stage times; multi reports each slab's device
   time.  Every output's bit-pattern checksum (int64 sum of the int32 patterns) must equal the one-shot call's.

Writes DIR/filter_slab_bench.json and prints it.  A number is only meaningful with the card it was measured on,
which the file carries.
"""
import argparse
import ctypes as C
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

STAGES = ("gauss", "h2d", "d2h")


def filters():
    """name -> FilterParams"""
    from visfd_b200 import FilterParams, gauss_halfwidth
    out = {f"gauss_{s:g}": FilterParams.gauss(s, gauss_halfwidth(s)) for s in (2.0, 4.0, 8.0)}
    out["dog_4_6.4"] = FilterParams.dog(4.0, 6.4, gauss_halfwidth(4.0), hw_b=gauss_halfwidth(6.4))
    out["log_4"] = FilterParams.log(4.0, 0.02, bench.RATIO)
    return out


def one_shot(ctx, p, src, dst):
    """the one-shot C call that FilterParams p stands for (visfd_cuda_apply_gauss / _dog2 / _log), from the host
    array src into the host array dst, as the stream and multi calls write theirs"""
    A, B = C.c_float(), C.c_float()
    nz, ny, nx = src.shape
    head = (ctx.h, C.c_int64(nx), C.c_int64(ny), C.c_int64(nz), C.c_void_p(src.ctypes.data),
            C.c_void_p(dst.ctypes.data), None)
    if p.kind == p.GAUSS:
        rc = ctx.lib.visfd_cuda_apply_gauss(*head, p.sigma_a, p.hw_a, C.c_int(p.normalize), C.byref(A))
    elif p.kind == p.DOG:
        rc = ctx.lib.visfd_cuda_apply_dog2(*head, p.sigma_a, p.sigma_b, p.hw_a, p.hw_b, C.byref(A), C.byref(B))
    else:
        rc = ctx.lib.visfd_cuda_apply_log(*head, p.sigma_a, C.c_float(p.delta), C.c_float(p.truncate_ratio),
                                          C.byref(A), C.byref(B))
    ctx._ck(rc)
    return {"out": dst, "A": A.value, "B": B.value, "n_slabs": 1}


def checksum(a, dev, chunk=1 << 28):
    """int64 sum of the int32 bit patterns of a host array, summed on the GPU a chunk at a time"""
    import torch
    flat = torch.from_numpy(np.ascontiguousarray(a).reshape(-1).view(np.int32))
    total = 0
    for i in range(0, flat.numel(), chunk):
        total += int(flat[i:i + chunk].to(dev, non_blocking=True).sum(dtype=torch.int64).item())
    return total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--no-c5", action="store_true")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    res = {"gpu": gpu_info(), "truncate_ratio": bench.RATIO, "steps": args.steps, "warmup": args.warmup}

    import torch
    import visfd_b200
    dev = torch.device("cuda", 0)
    ctx = visfd_b200.Context(0)
    ctx.set_timing(True)
    flt = filters()

    def timed(fn, pooled):
        if pooled:
            ctx.trim()
            ctx.reset_peak_reserved_bytes()
            ctx.reset_stage_ms()
        torch.cuda.synchronize()
        r = {"device_free_bytes_before": torch.cuda.mem_get_info()[0]}
        t = time.perf_counter()
        r.update(fn())
        r["wall_ms"] = (time.perf_counter() - t) * 1e3
        if pooled:
            r["peak_reserved_bytes"] = ctx.peak_reserved_bytes()
            r["stage_ms"] = {k: ctx.stage_ms(k) for k in STAGES}
        return r

    # ---- C5 shape ------------------------------------------------------------------------------------------------
    shape5 = bench.WORKLOADS["C5"]
    c5 = {"shape": list(shape5), "filter": "gauss_2"}
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
            src5 = h5.numpy()
            params = flt["gauss_2"]
            c5["source_checksum"] = checksum(src5, dev)
            try:
                one_shot(ctx, params, src5, src5)
                c5["one_shot_refusal"] = None
            except visfd_b200.VisfdCudaError as e:
                c5["one_shot_refusal"] = str(e)
            r = timed(lambda: ctx.filter_stream(src5, params, out=src5), True)
            r.pop("out")
            r["checksum"] = checksum(src5, dev)
            c5["stream_0"] = r
            print("C5 stream_0", json.dumps(r), file=sys.stderr, flush=True)
            del h5, src5
    ctx.trim()

    # ---- C4 --------------------------------------------------------------------------------------------------------
    shape4 = bench.WORKLOADS["C4"]
    h4 = host_volume(shape4, dev)
    o4 = torch.empty(shape4, dtype=torch.float32, pin_memory=True)
    src4, out4 = h4.numpy(), o4.numpy()
    c4 = {"shape": list(shape4), "filters": {}}
    res["C4"] = c4
    for name, params in flt.items():
        ref = timed(lambda: one_shot(ctx, params, src4, out4), True)
        ref_sum, budget = checksum(ref.pop("out"), dev), ref["peak_reserved_bytes"] // 4
        calls = [("one_shot", lambda: one_shot(ctx, params, src4, out4), True),
                 ("stream_0", lambda: ctx.filter_stream(src4, params, out=out4), True),
                 ("stream_B", lambda: ctx.filter_stream(src4, params, device_bytes=budget, out=out4), True),
                 ("multi_4x0", lambda: visfd_b200.filter_multi([0, 0, 0, 0], src4, params, out=out4), False)]
        runs = {}
        for step in range(args.warmup + args.steps):
            for call, fn, pooled in calls:
                r = timed(fn, pooled)
                r["checksum"] = checksum(r.pop("out"), dev)
                r["equal_one_shot"] = r["checksum"] == ref_sum and r["A"] == ref["A"] and r["B"] == ref["B"]
                r.setdefault("n_slabs", 4)   # multi_4x0
                print("C4", name, call, json.dumps(r), file=sys.stderr, flush=True)
                if step >= args.warmup:
                    runs.setdefault(call, []).append(r)
        row = {"budget_bytes": budget, "one_shot_checksum": ref_sum,
               "runs": {call: dict(rs[-1], wall_ms=[r["wall_ms"] for r in rs],
                                   wall_ms_median=statistics.median(r["wall_ms"] for r in rs),
                                   equal_one_shot=all(r["equal_one_shot"] for r in rs))
                        for call, rs in runs.items()}}
        row["all_equal"] = all(v["equal_one_shot"] for v in row["runs"].values())
        c4["filters"][name] = row
    c4["all_equal"] = all(v["all_equal"] for v in c4["filters"].values())
    del h4, o4, src4, out4

    res["gpu_after"] = gpu_info()["nvidia_smi"]
    with open(os.path.join(args.out, "filter_slab_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))
    ctx.close()


if __name__ == "__main__":
    main()
