#!/usr/bin/env python
"""bench.py -- the membrane + tensor-voting pipeline of filter_mrc on synthetic tomograms.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N ...            # the reference's CPU path

A "step" is one pass of HandleTV's pipeline (bin/filter_mrc/handlers.cpp:1618-1892:
Gaussian -> Hessian/eigen ridge saliency -> `-tv-best` cut -> TV3D stick voting ->
post-vote planar score) over the workload volume.  Workload = BASELINE.json config 4
(C4): 2048 x 2048 x 1024 float32, membrane sigma 3 voxels (thickness 5.196), `-tv 4.733`
(sigma_tv 14.2, vote radius 20), exponent 4, `-tv-best 0.05`; it fits one B200.  With
N > 1 the SAME volume is split into N Z-slabs (strong scaling); ranks exchange raw-source
halos by NCCL send/recv and all-reduce the cut histograms.

`value`  : voxels of the whole volume / device time of one step, inputs resident in HBM.
`e2e`    : the same through the public call with HOST (pinned) buffers: H2D of the
           source and D2H of the result inside the timed region.
`roofline`: the dominant kernel (tv_gather_kernel): 35 FLOP per (receiver, voter) pair
           (SURVEY.md 8d) x the exact pair count / the kernel's CUDA-event time, against
           the FP32 FMA peak measured in this run (MEASURED_PEAKS.json has no FP32 figure).
`cpu_baseline`: the unmodified reference (oracle/_ref) on a bounded crop, all host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# stdout carries exactly ONE JSON line.  Libraries write there too (NCCL prints its version
# banner on rank 0), so file descriptor 1 is pointed at stderr for the whole run and the result
# goes out through a private duplicate of the original stdout.
RESULT_OUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)

METRIC = "Gvoxel/s of filter_mrc membrane+TV pipeline"
SQ2 = float(np.float32(np.sqrt(2.0)))
# C4 parameters exactly as filter_mrc derives them (settings.cpp:2774, :3535-3540; handlers.cpp:1574)
SIGMA = float(np.float32(np.float32(5.196) / np.sqrt(3.0)))
TV_SIGMA = float(np.float32(np.float32(4.733) * np.float32(SIGMA)))
RATIO = float(np.float32(np.sqrt(np.float32(-2) * np.log(np.float32(0.03)))))
TV_BEST = 0.05
WORKLOADS = {"C4": (1024, 2048, 2048), "C5": (1024, 4096, 4096), "C2": (512, 512, 512), "C3": (512, 1024, 1024),
             "dev": (256, 256, 256)}
CPU_SAMPLE = tuple(int(v) for v in os.environ.get("VISFD_BENCH_CPU_SAMPLE", "128,128,128").split(","))  # override: smoke tests
# dram__bytes_read.sum + dram__bytes_write.sum of the voting kernel, per pipeline pass, from an ncu capture of
# the named workload -- constants of a PROFILED run of the same command, not measured in this run (a number taken
# under a profiler is never a bench value; the traffic of a kernel is).
#   dev: profiles/r02_tv_gather_lut_ncu_full.csv (ncu --set full, tv_gather_lut_kernel, 256^3)
#   C4:  profiles/r02_tv_traffic_c4.csv (ncu --replay-mode application, `bench.py --steps 1 --warmup 0`): the 10.3 GB
#        voter list is re-read ~11 times from DRAM by the layers of receiver tiles it serves (L2 hit rate 99 %);
#        20 GB/s, nowhere near the HBM roofline
NCU_TRAFFIC_BYTES = {"dev": 41.90e6 + 21.66e6, "C4": 115.59e9 + 17.30e9}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--workload", default=os.environ.get("VISFD_BENCH_WORKLOAD", "C4"))
    ap.add_argument("--shape", default=None, help="nz,ny,nx override (development)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-side-tables", action="store_true", help="skip masked / C5 / multi-GPU C3 / C-entry rows")
    ap.add_argument("--no-cpu-big", action="store_true", help="reference arm: skip the extra 256^3 pass")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (CUDA path)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs applies to the CUDA path")
    return args


# voxels of the output volume that --dump-outputs writes: 16 MB of float32 values + 32 MB of float64 indices
DUMP_SAMPLE = 1 << 22


def dump_outputs(path, out, z0, shape, threshold, dist, world, rank, dev):
    """--dump-outputs: what a caller of the timed step receives -- the post-vote score volume and the
    saliency-cut threshold -- as DIR/out_sample.npy, DIR/out_sample_index.npy and DIR/threshold.npy.  The
    volume is written at a fixed, seeded set of voxels (all of them when it has at most DUMP_SAMPLE), with
    their flat z-y-x indices beside the values, so that two builds run with the same arguments can be
    compared output for output.  `out` holds planes [z0, z0 + len(out)) of this rank."""
    import torch
    n = int(np.prod(shape))
    if n <= DUMP_SAMPLE:
        idx = np.arange(n, dtype=np.int64)
    else:
        idx = np.unique(np.random.default_rng(0).integers(0, n, DUMP_SAMPLE, dtype=np.int64))
    lo = z0 * shape[1] * shape[2]
    gidx = torch.from_numpy(idx).to(dev)
    mine = (gidx >= lo) & (gidx < lo + out.numel())
    bits = torch.zeros(len(idx), dtype=torch.int32, device=dev)
    bits[mine] = out.reshape(-1).view(torch.int32)[gidx[mine] - lo]
    if world > 1:
        dist.all_reduce(bits)    # every voxel lies on exactly one rank: its bit pattern plus zeros, exact
    if rank == 0:
        os.makedirs(path, exist_ok=True)
        np.save(os.path.join(path, "out_sample.npy"), bits.view(torch.float32).cpu().numpy())
        np.save(os.path.join(path, "out_sample_index.npy"), idx.astype(np.float64))
        np.save(os.path.join(path, "threshold.npy"), np.array([threshold], np.float64))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); power.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def host_threads():
    """Threads the CPU arm may use: the cores this process is allowed on.  torch.distributed.run
    exports OMP_NUM_THREADS=1 to every rank when nproc > 1, which would silently serialise the
    reference's OpenMP loops, so the count is set explicitly on the OpenMP runtime the reference
    library links (libgomp) after loading it."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    return max(1, n)


def _set_omp_threads(n):
    import ctypes
    os.environ["OMP_NUM_THREADS"] = str(n)
    try:
        gomp = ctypes.CDLL("libgomp.so.1")
        gomp.omp_set_dynamic(0)
        gomp.omp_set_num_threads(int(n))
        return int(gomp.omp_get_max_threads())
    except OSError:
        return n


def cpu_reference_run(shape, seed=0, staged=False):
    """One pass of the UNMODIFIED reference (oracle/_ref, OpenMP on all host cores) over a
    crop of the workload; returns (seconds, threads, kind, per-stage seconds or None).
    staged=True calls the stages of HandleTV one by one (the same reference functions
    ref_membrane chains: CalcHessian, eigen + score loop, cut, TVDenseStick, score loop)."""
    from oracle.pyoracle import Oracle, have
    from visfd_b200 import synth
    kind = "reference" if have("reference") else "port"
    o = Oracle(kind)
    cores = _set_omp_threads(host_threads())
    vol = synth.tomogram(shape, seed=seed)
    stages = None
    t = time.perf_counter()
    if not staged:
        o.membrane(vol, SIGMA, RATIO, 1, TV_BEST, True, TV_SIGMA, 4, SQ2, want_tensor=False)
    else:
        stages = {}
        t0 = time.perf_counter()
        grad, hess = o.calc_hessian(vol, SIGMA, RATIO)[:2]
        stages["gauss_hessian"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        sal, dire, _ = o.hessian_eigen_score(hess, 1, 0)
        del hess
        stages["eigen_score"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        sal, _thr = o.saliency_cut(sal, TV_BEST, True)
        stages["cut"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        ten = o.tv_dense_stick(sal, dire, TV_SIGMA, 4, SQ2)
        stages["tv"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        o.tensor_score(ten, 1, 0)
        stages["post_score"] = time.perf_counter() - t0
    return time.perf_counter() - t, cores, kind, stages


def cpu_sample_text(shape):
    return ("%dx%dx%d crop of the synthetic workload with the same parameters (sigma 3, vote radius 20, "
            "tv-best 0.05): one full pipeline pass of the unmodified reference (OpenMP) per step" % tuple(shape))


def reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path (oracle/_ref: the
    unmodified lib/visfd templates behind HandleTV, handlers.cpp:1618-1892), timed on the host
    cores on a bounded sample of the workload: a CPU_SAMPLE crop with the C4 parameters per step.
    The reference cannot hold C4 itself (int-indexed containers, hours of CPU time); every stage
    is O(voxels) at fixed radii, so the per-voxel rate carries over (a small crop has fewer
    in-image window visits per voxel, which favours the reference).  One extra, untimed-by-the-
    driver 256^3 pass with per-stage seconds is added at N = 1 when the host is fast enough."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    world = int(os.environ.get("WORLD_SIZE", "1"))
    shape = WORKLOADS.get(args.workload, WORKLOADS["C4"])
    t_start = time.perf_counter()
    for _ in range(args.warmup):
        cpu_reference_run(CPU_SAMPLE)
    ts = []
    cores, kind, stages = host_threads(), "reference", None
    for k in range(args.steps):
        dt, cores, kind, st = cpu_reference_run(CPU_SAMPLE, staged=(k == args.steps - 1))
        stages = st or stages
        ts.append(dt)
    dt = float(np.mean(ts))
    val = np.prod(CPU_SAMPLE) / dt / 1e9
    big = None
    spent = time.perf_counter() - t_start
    # a 256^3 pass costs ~8.7 crops (more in-image windows per voxel); only when it fits in ~4 minutes more
    if world == 1 and not args.no_cpu_big and 9.0 * dt < 240.0 and spent + 9.0 * dt < 600.0:
        bshape = (256, 256, 256)
        bdt, _, _, bst = cpu_reference_run(bshape, staged=True)
        big = {"shape_zyx": list(bshape), "seconds": bdt, "value": float(np.prod(bshape)) / bdt / 1e9,
               "unit": "Gvoxel/s", "stage_seconds": bst}
    cfg = workload_config(args.workload, shape)
    cfg["cpu_sample"] = {"shape_zyx": list(CPU_SAMPLE), "note": "the reference arm times this crop, not the full "
                         "volume; value is a per-voxel rate"}
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "Gvoxel/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg,
            "cpu_baseline": {"value": val, "unit": "Gvoxel/s", "cores": cores, "kind": kind,
                             "sample": cpu_sample_text(CPU_SAMPLE), "stage_seconds_last_step": stages,
                             "point_256": big},
            "e2e": {"value": val, "unit": "Gvoxel/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), file=RESULT_OUT, flush=True)
    return 0


def workload_config(name, shape):
    return {"workload": f"{name}: membrane detection (Hessian ridge saliency + TV3D stick voting) on "
                        f"{shape[2]}x{shape[1]}x{shape[0]} float32",
            "shape_zyx": list(shape), "sigma_vox": SIGMA, "gauss_halfwidth": 7, "tv_sigma_vox": TV_SIGMA,
            "tv_halfwidth": 20, "tv_exponent": 4, "tv_best": TV_BEST, "partition": "z-slabs",
            "l2": "inputs (>= 0.5 GB per volume) exceed the 126 MB L2; no flush needed"}


def gauss_c2_table(ctx, dev, hbm_peak, fp32_peak):
    """ApplyGauss and ApplyDog (sigma, 1.6 sigma) on a synthetic 512^3 volume for sigma 2, 4, 8
    (half-widths 5, 10, 21; SURVEY appendix B), device resident, CUDA events, 5 launches after 2
    warm-ups.  Algorithmic bytes: 24 B/voxel per Gaussian, 48 per DoG (SURVEY 8d).  `exact` is the
    default bit-identical arithmetic (un-fused multiply and add per tap), `fast` the FFMA mode.
    Beyond sigma ~ 3 the direct convolution is FP32-bound, so every row also carries the fraction of the FMA
    pipe: (2 hw + 1) taps x 3 sweeps x (2 pipe operations per tap in the exact mode -- a multiply and an add, the
    reference's rounding sequence -- 1 in the FFMA mode) per voxel, against the lane rate behind the FP32 peak
    measured in this run (peak TFLOP/s / 2 FLOP per FMA); `bound` names the larger of the two."""
    import torch
    import visfd_b200
    from visfd_b200 import synth
    shape = WORKLOADS["C2"]
    vol = synth.tomogram_torch(shape, dev, seed=1)
    n = float(np.prod(shape))
    rows = []

    def timed_ms(fn):
        for _ in range(2):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(5):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / 5

    for mode in ("exact", "fast"):
        ctx.set_fast_gauss(mode == "fast")
        for sigma in (2.0, 4.0, 8.0):
            hw = visfd_b200.gauss_halfwidth(sigma)
            hw_dog = visfd_b200.gauss_halfwidth(1.6 * sigma)
            ms_g = timed_ms(lambda: ctx.apply_gauss(vol, [sigma] * 3, [hw] * 3))
            ms_d = timed_ms(lambda: ctx.apply_dog(vol, [sigma] * 3, [1.6 * sigma] * 3, [hw_dog] * 3))
            ops = 2.0 if mode == "exact" else 1.0
            lane_rate = fp32_peak * 1e12 / 2.0
            g_pipe = n * (2 * hw + 1) * 3 * ops / (ms_g * 1e-3) / lane_rate
            d_pipe = n * (2 * hw_dog + 1) * 3 * 2 * ops / (ms_d * 1e-3) / lane_rate
            g_hbm, d_hbm = 24.0 * n / ms_g / 1e6 / hbm_peak, 48.0 * n / ms_d / 1e6 / hbm_peak
            rows.append({"mode": mode, "sigma": sigma, "halfwidth": hw, "gauss_ms": ms_g,
                         "gauss_GBps": 24.0 * n / ms_g / 1e6, "gauss_frac_of_hbm": g_hbm,
                         "gauss_frac_of_fp32_pipe": g_pipe, "gauss_bound": "fp32" if g_pipe > g_hbm else "hbm",
                         "dog_halfwidth": hw_dog, "dog_ms": ms_d, "dog_GBps": 48.0 * n / ms_d / 1e6,
                         "dog_frac_of_hbm": d_hbm, "dog_frac_of_fp32_pipe": d_pipe,
                         "dog_bound": "fp32" if d_pipe > d_hbm else "hbm"})
    ctx.set_fast_gauss(False)
    del vol
    torch.cuda.empty_cache()
    return {"shape_zyx": list(shape), "hbm_peak_GBps": hbm_peak, "rows": rows}


def blob_c3_row(ctx, dev, hbm_peak):
    """BlobDog on BASELINE config 3: 1024x1024x512, `-blob-s minima 2 8 1.14` => 12 scales
    sigma_n = 2 * 4^(n/12), each one ApplyLog with delta 0.02 and the shared half-width
    floor(2.6482 * 1.01 sigma) (SURVEY appendix B), extremum scan over scales 1..10.  Device
    resident input with 64 dark blobs stamped in, one warm-up, two timed calls, CUDA events around the
    whole call (the candidate lists come back to the host inside it).  Algorithmic bytes: 60 B per
    voxel per scale (SURVEY 8d)."""
    import torch
    from visfd_b200 import synth
    shape = WORKLOADS["C3"]
    nz, ny, nx = shape
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
    n_scales = 12
    sigmas = 2.0 * 4.0 ** (np.arange(n_scales) / n_scales)
    ratio = float(np.sqrt(-2.0 * np.log(0.03)))

    def call():
        # `-blob-s minima` defaults (bin/filter_mrc/settings.cpp:1674-1678, :121-123): every minimum with a
        # negative score, absolute thresholds
        return ctx.blob_dog(vol, sigmas, delta=0.02, truncate_ratio=ratio, minima_threshold=0.0,
                            maxima_threshold=-np.inf, use_threshold_ratios=False, capacity=1 << 24)

    minima, maxima = call()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(2):
        call()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 2
    n = float(nz) * ny * nx
    gbps = 60.0 * n * n_scales / ms / 1e6
    del vol
    torch.cuda.empty_cache()
    return {"shape_zyx": list(shape), "scales": n_scales, "sigma_first_last": [float(sigmas[0]), float(sigmas[-1])],
            "ms": ms, "Gvoxel_scales_per_s": n * n_scales / ms / 1e6, "algorithmic_bytes_per_voxel_per_scale": 60,
            "GBps": gbps, "frac_of_hbm": gbps / hbm_peak, "minima": int(len(minima)), "maxima": int(len(maxima)),
            "thresholds": "minima < 0, absolute (the -blob-s minima defaults)"}



def masked_row(ctx, dev):
    """`-mask` is how membrane detection is normally run (the cell, not the whole tomogram): C4 parameters on a
    1024 x 1024 x 512 volume with a centred box mask covering 80 % of it.  Masks route the Gaussian through the masked
    sweeps (denominator volume, no TMA) and add the mask reads to every stage.  Device resident, 1 warm-up + 2 timed."""
    import torch
    import visfd_b200
    from visfd_b200 import synth
    shape = (512, 1024, 1024)
    vol = synth.tomogram_torch(shape, dev, seed=4)
    mask = torch.zeros(shape, dtype=torch.float32, device=dev)
    f = (1 - 0.8 ** (1 / 3)) / 2
    lo = [int(round(s * f)) for s in shape]
    mask[lo[0]:shape[0] - lo[0], lo[1]:shape[1] - lo[1], lo[2]:shape[2] - lo[2]] = 1.0
    out = torch.empty_like(vol)

    def call():
        ctx.reset_stage_ms()
        ctx.membrane(vol, SIGMA, RATIO, visfd_b200.DECREASING_EIVALS, TV_BEST, True, TV_SIGMA, 4, SQ2, mask=mask, out=out)

    call()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(2):
        call()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 2
    n = float(np.prod(shape))
    stage = {k: ctx.stage_ms(k) for k in ("gauss", "ridge", "select", "compact", "tv")}
    row = {"shape_zyx": list(shape), "mask": "centred box, 80 % of the volume", "ms": ms,
           "Gvoxel_per_s": n / ms / 1e6, "masked_fraction": float(1.0 - mask.mean().item()),
           "voters": int(ctx.last_voter_count()), "stage_ms": stage, "tv_kernel": ctx.last_tv_kernel()}
    del vol, mask, out
    torch.cuda.empty_cache()
    return row


def c5_row(ctx, dev, dist, rank, world):
    """BASELINE config 5: 4096 x 4096 x 1024, the full filter_mrc membrane pipeline (blur, eigensolve, voting) and the
    final `-thresh` at the 99th percentile of the post-vote saliency (a second filter_mrc invocation in the
    reference, SURVEY appendix B), sharded as Z-slabs over all ranks.  The percentile is a distributed radix select
    over the result (the same all-reduced histograms as the cut), the threshold map is visfd_cuda_threshold.
    1 warm-up + 2 timed steps, CUDA events, max over ranks."""
    import torch
    import visfd_b200
    from visfd_b200 import synth, MembraneParams
    from visfd_b200.slab import SlabMembrane, distributed_cut_threshold
    shape = WORKLOADS["C5"]
    nz, ny, nx = shape
    params = MembraneParams(SIGMA, RATIO, visfd_b200.DECREASING_EIVALS, TV_BEST, 1, TV_SIGMA, 4, SQ2)
    pipe = SlabMembrane(ctx, shape, params, rank=rank, world=world, dist=dist if world > 1 else None, device=dev)
    z0, z1 = pipe.plan.own
    own = synth.tomogram_torch(shape, dev, seed=0, z0=z0, z1=z1)
    out = torch.empty_like(own)
    maskmap = torch.empty_like(own)
    state = {}

    def step():
        pipe.run(own, out=out)
        # k = floor(n * 0.01)-th largest value = the 99th percentile
        T = distributed_cut_threshold(ctx, out, 0.01, dist=dist, world=world, device=dev)
        ctx.threshold(out, visfd_b200.THRESH_SINGLE, [T], out=maskmap)
        state["T"] = T

    step()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(2):
        step()
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / 2], device=dev, dtype=torch.float64)
    ones = maskmap.sum(dtype=torch.float64).reshape(1)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(ones)
    n = float(nz) * ny * nx
    row = {"shape_zyx": list(shape), "ms_per_step": float(t.item()), "Gvoxel_per_s": n / float(t.item()) / 1e6,
           "threshold_99th_percentile": float(state["T"]), "voxels_above": int(ones.item()),
           "fraction_above": float(ones.item()) / n, "stages": "gauss + ridge + cut + voting + score + percentile + thresh"}
    del pipe, own, out, maskmap
    torch.cuda.empty_cache()
    ctx.trim()
    return row


def blob_c3_multi_row(ctx, dev, dist, rank, world):
    """BASELINE config 3 over Z-slabs (visfd_b200.slab.SlabBlobs): 12 LoG scales + 10 extremum scans on
    1024 x 1024 x 512, halo = widest LoG half-width + 1 planes, candidate lists all-gathered, best scores all-reduced."""
    import torch
    from visfd_b200 import synth
    from visfd_b200.slab import SlabBlobs
    shape = WORKLOADS["C3"]
    n_scales = 12
    sigmas = 2.0 * 4.0 ** (np.arange(n_scales) / n_scales)
    ratio = float(np.sqrt(-2.0 * np.log(0.03)))
    blobs = SlabBlobs(ctx, shape, sigmas, delta=0.02, truncate_ratio=ratio, rank=rank, world=world,
                      dist=dist if world > 1 else None, device=dev)
    z0, z1 = blobs.plan.own
    own = synth.tomogram_torch(shape, dev, seed=2, z0=z0, z1=z1, n_shells=0)

    def call():
        return blobs.run(own, minima_threshold=0.0, maxima_threshold=-np.inf, use_threshold_ratios=False,
                         capacity=1 << 24)

    mn, mx = call()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(2):
        call()
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / 2], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    n = float(np.prod(shape))
    row = {"shape_zyx": list(shape), "scales": n_scales, "ms": float(t.item()),
           "Gvoxel_scales_per_s": n * n_scales / float(t.item()) / 1e6, "minima": int(len(mn)), "maxima": int(len(mx)),
           "halo_planes": blobs.plan.halo, "note": "noise volume without stamped blobs (the lists are all-gathered "
           "through the host: their size is part of the cost)"}
    del own, blobs
    torch.cuda.empty_cache()
    return row


def c_multi_row(dev, dist, rank, world, shape, want_checksum):
    """The same workload through visfd_cuda_membrane_multi: ONE process (rank 0) drives all `world` GPUs of the node
    from pinned host arrays through the C entry a C++ filter_mrc would link; the other ranks have released their
    memory and wait at the barrier.  Upload and download are inside the timed region (it is an end-to-end figure).
    1 warm-up + 1 timed call, wall clock around the call and max of the workers' device times."""
    import torch
    import visfd_b200
    from visfd_b200 import synth
    row = None
    if rank == 0:
        nz, ny, nx = shape
        h_src = torch.empty(shape, dtype=torch.float32, pin_memory=True)
        h_out = torch.empty(shape, dtype=torch.float32, pin_memory=True)
        step = 64
        for z in range(0, nz, step):
            h_src[z:z + step].copy_(synth.tomogram_torch(shape, dev, seed=0, z0=z, z1=min(nz, z + step)))
        torch.cuda.empty_cache()
        src_np, out_np = h_src.numpy(), h_out.numpy()
        devices = list(range(world))
        res = None
        times = []
        for it in range(2):
            t = time.perf_counter()
            res = visfd_b200.membrane_multi(devices, src_np, SIGMA, RATIO, visfd_b200.DECREASING_EIVALS, TV_BEST, True,
                                            TV_SIGMA, 4, SQ2, out=out_np)
            times.append(time.perf_counter() - t)
        n = float(nz) * ny * nx
        bits = int(h_out.view(torch.int32).sum(dtype=torch.int64).item())
        row = {"call": "visfd_cuda_membrane_multi(ndev=%d, host arrays)" % world, "wall_ms": times[-1] * 1e3,
               "device_ms_max": max(res["device_ms"]), "device_ms": res["device_ms"],
               "Gvoxel_per_s": n / times[-1] / 1e9, "h2d_bytes": int(4 * n), "d2h_bytes": int(4 * n),
               "bits_sum_i64": bits, "matches_checksum": bool(bits == want_checksum)}
        del h_src, h_out
    if world > 1:
        # the other ranks wait on the HOST (a key in the rendezvous store), not in an NCCL barrier: a collective
        # kernel spinning on a GPU that rank 0 is driving from another process would have to be time-sliced against it
        import datetime
        store = dist.distributed_c10d._get_default_store()
        if rank == 0:
            store.set("visfd_c_multi_done", "1")
        else:
            store.wait(["visfd_c_multi_done"], datetime.timedelta(minutes=30))
    return row


def main():
    args = parse()
    if args.impl == "reference":
        return reference_arm(args)

    import torch
    import torch.distributed as dist
    import visfd_b200
    from visfd_b200 import synth, MembraneParams
    from visfd_b200.slab import SlabMembrane

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    name = args.workload
    shape = WORKLOADS[name]
    if args.shape:
        shape = tuple(int(v) for v in args.shape.split(","))
        name = "custom"
    nz, ny, nx = shape
    # C4 needs ~100 GB of HBM on one GPU: a device that cannot hold the workload is an error, not
    # a reason to measure something else
    free_b, total_b = torch.cuda.mem_get_info()
    need = 6.5 * 4 * nz * ny * nx / world
    if need > free_b:
        raise SystemExit("bench.py: workload %s needs ~%.0f GB of HBM per GPU at N=%d, %.0f GB free" %
                         (name, need / 1e9, world, free_b / 1e9))

    own = out = d_out = h_src = h_out = src_np = out_np = None
    ctx = visfd_b200.Context(local, stream=torch.cuda.current_stream().cuda_stream)
    params = MembraneParams(SIGMA, RATIO, visfd_b200.DECREASING_EIVALS, TV_BEST, 1, TV_SIGMA, 4, SQ2)
    pipe = SlabMembrane(ctx, shape, params, rank=rank, world=world, dist=dist if world > 1 else None, device=dev)
    z0, z1 = pipe.plan.own
    own = synth.tomogram_torch(shape, dev, seed=0, z0=z0, z1=z1)
    out = torch.empty_like(own)
    n_vox = float(nz) * ny * nx

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    last = {}

    def device_step():
        if world == 1:
            ctx.reset_stage_ms()
            r = ctx.membrane(own, SIGMA, RATIO, visfd_b200.DECREASING_EIVALS, TV_BEST, True, TV_SIGMA, 4, SQ2, out=out)
            last["threshold"] = r["threshold"]
        else:
            pipe.run(own, out=out)
            last["threshold"] = pipe.threshold

    def timed(fn, steps):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        for _ in range(steps):
            fn()
        ev1.record()
        barrier()
        ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) / steps

    # ---- device-resident throughput -----------------------------------------------------
    for _ in range(args.warmup):
        device_step()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = ctx.launch_count()
    ms_step = timed(device_step, args.steps)
    launches = ctx.launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out, z0, shape, last["threshold"], dist, world, rank, dev)
    stage = {k: ctx.stage_ms(k) for k in ("gauss", "ridge", "select", "compact", "tv")}   # last step, this rank
    n_voters = ctx.last_voter_count()
    lt = torch.tensor([launches], device=dev, dtype=torch.int64)
    if world > 1:
        dist.all_reduce(lt)
    launches = int(lt.item())

    # ---- checksum of the result volume: identical at every N if the slabs reproduce one GPU ------
    # exact integer arithmetic on the float bit patterns (associative, so the split does not matter):
    # sum of the bits, and the same weighted by the global plane number (catches misplaced planes)
    plane_bits = torch.stack([out[z].view(torch.int32).sum(dtype=torch.int64) for z in range(out.shape[0])])
    zw = torch.arange(z0 + 1, z1 + 1, device=dev, dtype=torch.int64)
    ck = torch.stack([plane_bits.sum(), (plane_bits * zw).sum()])
    f64 = out.sum(dtype=torch.float64).reshape(1)
    if world > 1:
        dist.all_reduce(ck)
        dist.all_reduce(f64)
    checksum = {"bits_sum_i64": int(ck[0].item()), "plane_weighted_bits_sum_i64": int(ck[1].item()),
                "f64_sum": float(f64.item()),
                "note": "wrapping int64 sums of the float32 bit patterns of the output volume (exact, order "
                        "independent): equal at every N iff the volumes are bit-identical up to permutation "
                        "within a plane"}

    # ---- roofline of the dominant kernel (rank 0's launch) ----------------------------------
    if world == 1:
        r = ctx.membrane(own, SIGMA, RATIO, visfd_b200.DECREASING_EIVALS, TV_BEST, True, 0.0, 4, SQ2)
        sal_after_cut, recv = r["out"], None
        del r
        pairs = ctx.tv_count_pairs(sal_after_cut, -np.inf, 20, recv=recv)
        del sal_after_cut
    else:
        v0, v1 = pipe.plan.vote_local
        o0, o1 = pipe.plan.own_local
        pairs = ctx.tv_count_pairs(pipe.saliency[v0:v1], pipe.threshold, 20, recv=(o0 - v0, o1 - v0))
    fp32_peak = ctx.fp32_peak(300.0)
    fp32_peak_3op = ctx.fp32_peak(300.0, three_operand=True)
    tv_ms = stage["tv"]
    achieved = 35.0 * pairs / (tv_ms * 1e-3) / 1e12
    tv_kernel_name = "tv_gather_lut_kernel" if ctx.last_tv_kernel() else "tv_gather_kernel"
    roofline = {"kernel": tv_kernel_name, "bound": "fp32", "achieved": achieved, "peak": fp32_peak,
                "unit": "TFLOP/s", "frac": achieved / fp32_peak,
                "traffic": NCU_TRAFFIC_BYTES.get(name) if world == 1 else None,
                "peak_source": "measured in this run: register-resident FFMA chains (visfd_cuda_fp32_peak); "
                               "MEASURED_PEAKS.json holds HBM and bf16 tensor peaks only",
                "peak_3_register_operands": fp32_peak_3op, "frac_of_3_operand_peak": achieved / fp32_peak_3op,
                "frac_of_nominal_74.4_TFLOPs": achieved / 74.4,   # 148 SMs x 128 lanes x 2 x 1.965 GHz (SURVEY 8d)
                "algorithmic_flop": 35.0 * pairs, "pairs": int(pairs), "voters": int(n_voters),
                "kernel_ms": tv_ms, "share_of_step": tv_ms / ms_step}

    # ---- Gaussian stage against the HBM roofline (second half of BASELINE's metric) ---------------
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    own_planes = z1 - z0
    n_slab_vox = float(pipe.plan.slab[1] - pipe.plan.slab[0]) * ny * nx
    gauss = {"bound": "hbm", "achieved": 24.0 * n_slab_vox / (stage["gauss"] * 1e-3) / 1e9, "peak": hbm_peak,
             "unit": "GB/s", "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback 6650",
             "algorithmic_bytes_per_voxel": 24, "kernel_ms": stage["gauss"]}
    gauss["frac"] = gauss["achieved"] / hbm_peak
    gauss["frac_of_nominal_8000_GBps"] = gauss["achieved"] / 8000.0        # SURVEY 8d: report both denominators
    ridge = {"bound": "hbm", "achieved": 8.0 * n_slab_vox / (stage["ridge"] * 1e-3) / 1e9, "peak": hbm_peak,
             "unit": "GB/s", "algorithmic_bytes_per_voxel": 8, "kernel_ms": stage["ridge"]}
    ridge["frac"] = ridge["achieved"] / hbm_peak
    ridge["frac_of_nominal_8000_GBps"] = ridge["achieved"] / 8000.0
    # SURVEY 8d counts 20 B/voxel for this pass (4 in, 4 saliency + 12 normal out); the fused pipeline never writes
    # the normals (they are recomputed for the ~5 % of voxels that vote), hence 8.  The pass is bound by the FP64 /
    # conversion pipes, not by HBM: ~58 DFMA-class instructions (64 per clock and SM), 8 float<->double conversions
    # + 3 MUFU (16 per clock and SM) per voxel (DESIGN 4.2)
    ridge["frac_at_survey_20_bytes_per_voxel"] = 20.0 / 8.0 * ridge["frac"]
    ridge["fp64_instructions_per_voxel"] = 58
    ridge["frac_of_fp64_pipe"] = 58.0 * n_slab_vox / (stage["ridge"] * 1e-3) / (64.0 * 148 * 1.965e9)

    # ---- BASELINE config 2: 3-D Gaussian / DoG at sigma 2, 4, 8 on 512^3 (the "Gauss HBM GB/s" half) ---
    gauss_c2 = blob_c3 = None
    if rank == 0 and world == 1:
        gauss_c2 = gauss_c2_table(ctx, dev, hbm_peak, fp32_peak)
        blob_c3 = blob_c3_row(ctx, dev, hbm_peak)

    # ---- end to end: host buffers through the public call ------------------------------------------
    e2e = None
    if not args.no_e2e:
        del out
        torch.cuda.empty_cache()
        h_src = torch.empty((own_planes, ny, nx), dtype=torch.float32, pin_memory=True)
        h_out = torch.empty((own_planes, ny, nx), dtype=torch.float32, pin_memory=True)
        h_src.copy_(own)
        if world == 1:
            del own
            torch.cuda.empty_cache()
            src_np, out_np = h_src.numpy(), h_out.numpy()

            def e2e_step():
                # host pointers: the library stages H2D / D2H itself (the drop-in path)
                ctx.membrane(src_np, SIGMA, RATIO, visfd_b200.DECREASING_EIVALS, TV_BEST, True, TV_SIGMA, 4, SQ2,
                             out=out_np)
        else:
            d_out = torch.empty_like(own)

            def e2e_step():
                own.copy_(h_src, non_blocking=True)
                pipe.run(own, out=d_out, out_host=h_out)   # D2H chunk by chunk behind the voting kernels
                torch.cuda.current_stream().synchronize()
        e2e_step()
        e2e_ms = timed(e2e_step, args.steps)
        e2e = {"value": n_vox / (e2e_ms * 1e-3) / 1e9, "unit": "Gvoxel/s", "ms_per_step": e2e_ms,
               "h2d_bytes_per_step": int(4 * n_vox), "d2h_bytes_per_step": int(4 * n_vox),
               "call": "visfd_cuda_membrane(host pointers)" if world == 1 else
                       "pinned host slab -> H2D -> SlabMembrane.run(out_host=pinned) -> chunked D2H, per rank"}

    # ---- side tables: masked run (N = 1); C5 + multi-GPU C3 + the one-call C entry (N > 1) ---------------
    masked = c5 = blob_multi = c_multi = None
    if not args.no_side_tables:
        own = out = d_out = h_src = h_out = src_np = out_np = e2e_step = device_step = None   # release the C4 buffers
        pipe.smoothed = pipe.saliency = pipe.slab_src = None
        torch.cuda.empty_cache()
        ctx.trim()
        if world == 1:
            masked = masked_row(ctx, dev)
        else:
            blob_multi = blob_c3_multi_row(ctx, dev, dist, rank, world)
            if world == 8:
                c5 = c5_row(ctx, dev, dist, rank, world)
            ctx.trim()
            torch.cuda.empty_cache()
            torch.cuda.synchronize()
            dist.barrier()          # everybody has released its memory and is idle
            torch.cuda.synchronize()
            c_multi = c_multi_row(dev, dist, rank, world, shape, checksum["bits_sum_i64"])

    # ---- CPU baseline (rank 0, N=1 only) ----------------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        dt, cores, kind, st = cpu_reference_run(CPU_SAMPLE, staged=True)
        cpu = {"value": float(np.prod(CPU_SAMPLE)) / dt / 1e9, "unit": "Gvoxel/s", "cores": cores, "kind": kind,
               "seconds": dt, "stage_seconds": st, "sample": cpu_sample_text(CPU_SAMPLE)}

    if rank == 0:
        line = {"metric": METRIC, "value": n_vox / (ms_step * 1e-3) / 1e9, "unit": "Gvoxel/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": workload_config(name, shape), "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
                "checksum": checksum,
                "roofline": roofline, "roofline_gauss": gauss, "roofline_ridge": ridge, "gauss_c2": gauss_c2, "blob_c3": blob_c3,
                "masked_1024": masked, "c5_n8": c5, "blob_c3_multi": blob_multi, "c_entry_multi": c_multi,
                "cpu_baseline": cpu,
                "stage_ms_rank0_last_step": stage, "halo_planes": pipe.plan.halo if world > 1 else 0}
        print(json.dumps(line), file=RESULT_OUT, flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
