"""visfd_cuda_blob_dog_stream (Context.blob_dog_stream) and visfd_cuda_blob_dog_multi (blob_dog_multi): BlobDog in
Z-slabs, on one GPU within a device-memory budget or over several devices.  Their lists must equal
visfd_cuda_blob_dog's row for row, bit for bit and in the same (scale, z, y, x) order, at every slab count, and the
stream call's pool must never hold more than its budget (visfd_cuda_peak_reserved_bytes)."""
import ctypes as C
import re

import numpy as np
import pytest

import visfd_b200
from visfd_b200 import synth
from util import sort_blobs

pytestmark = pytest.mark.gpu

RATIO = 2.6482
SHAPE = (203, 64, 72)   # ragged nz: the last slab's planes are not a multiple of 8
NARROW = (1.0 * 1.25 ** np.arange(6)).astype(np.float32)   # LoG half-widths up to 8: halo 9 planes
WIDE = (2.0 * 1.4 ** np.arange(6)).astype(np.float32)      # up to 28: halo 29 planes, wider than most slabs


def _volume():
    return synth.tomogram(SHAPE, seed=19, n_shells=0, blobs=60, blob_sigma=(1.0, 3.0))


def _cell_mask():
    nz, ny, nx = SHAPE
    z, y, x = np.ogrid[:nz, :ny, :nx]
    inside = ((z - nz / 2) / (0.45 * nz)) ** 2 + ((y - ny / 2) / (0.48 * ny)) ** 2 + ((x - nx / 2) / (0.45 * nx)) ** 2
    return (inside <= 1.0).astype(np.float32)


def _fresh_peak(ctx, fn):
    """fn() with the pool emptied first -> (result, the most the pool held during fn)"""
    ctx.trim()
    ctx.reset_peak_reserved_bytes()
    res = fn()
    return res, ctx.peak_reserved_bytes()


def _same(got, want):
    """row for row, bit for bit, in order"""
    return all(g.shape == w.shape and np.array_equal(g.view(np.int32), w.view(np.int32)) for g, w in zip(got, want))


def _thresholds(ctx, case, vol, sigmas, mask):
    if case == "absolute":   # `-blob-s minima` defaults
        return dict(minima_threshold=0.0, maxima_threshold=-np.inf, use_threshold_ratios=False)
    if case == "ratio":
        return dict(minima_threshold=0.3, maxima_threshold=0.4, use_threshold_ratios=True)
    # finite absolute cuts on both lists, at the median score of each, so that both keep about half
    mn, mx = ctx.blob_dog(vol, sigmas, 0.02, RATIO, mask=mask, minima_threshold=0.0, maxima_threshold=0.0)
    return dict(minima_threshold=float(np.median(mn[:, 4])), maxima_threshold=float(np.median(mx[:, 4])),
                use_threshold_ratios=False)


# (thresholds, sigmas)
CASES = {"absolute": ("absolute", NARROW), "finite": ("finite", NARROW), "ratio": ("ratio", NARROW),
         "wide_halo": ("ratio", WIDE)}


def _inputs(ctx, case, masked):
    thr, sigmas = CASES[case]
    vol = _volume()
    mask = _cell_mask() if masked else None
    return vol, mask, sigmas, _thresholds(ctx, thr, vol, sigmas, mask)


@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("case", sorted(CASES))
def test_stream_equals_one_shot_at_every_slab_count(ctx, case, masked):
    vol, mask, sigmas, kw = _inputs(ctx, case, masked)
    want, one_shot = _fresh_peak(ctx, lambda: ctx.blob_dog(vol, sigmas, 0.02, RATIO, mask=mask, **kw))
    assert len(want[0]) > 0 and (kw["maxima_threshold"] == -np.inf or len(want[1]) > 0)
    # from twice the one-shot peak: a stream slab also holds candidate lists that cannot overflow
    seen = []
    budget = 2 * one_shot
    while not ({1, 2, 3} <= set(seen) and max(seen) >= 6):
        assert budget > one_shot // 50, f"slab counts seen down to {budget} bytes: {seen}"
        got, peak = _fresh_peak(ctx, lambda: ctx.blob_dog_stream(vol, sigmas, 0.02, RATIO, mask=mask,
                                                                 device_bytes=budget, **kw))
        n = got["n_slabs"]
        assert peak <= budget, (n, peak, budget)
        assert _same((got["minima"], got["maxima"]), want), (n, budget)
        seen.append(n)
        budget = budget * 15 // 16


@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("case", sorted(CASES))
def test_multi_equals_one_shot(ctx, case, masked):
    import torch
    vol, mask, sigmas, kw = _inputs(ctx, case, masked)
    want = ctx.blob_dog(vol, sigmas, 0.02, RATIO, mask=mask, **kw)
    n_dev = torch.cuda.device_count()
    device_lists = [[0] * k for k in (1, 2, 3, 4, 8)]
    if n_dev > 1:
        device_lists += [list(range(n_dev)), [d % n_dev for d in range(2 * n_dev)]]
    for devices in device_lists:
        got = visfd_b200.blob_dog_multi(devices, vol, sigmas, 0.02, RATIO, mask=mask, **kw)
        assert _same((got["minima"], got["maxima"]), want), devices
        assert len(got["device_ms"]) == len(devices) and all(t > 0 for t in got["device_ms"]), got["device_ms"]


def _at_smallest_budget(ctx, fn, most=None):
    """fn(device_bytes) at the smallest budget that takes at most `most` slabs (None: that fits at all, so the most
    slabs any budget gives), found by bisection: fewer bytes never take fewer slabs, and the window of budget
    between two slab counts can be narrower than any fixed step"""
    lo, hi = 0, 1 << 31   # lo: more slabs, or refused; hi: at most `most`
    while hi - lo > 1:
        mid = (lo + hi) // 2
        try:
            n = fn(mid)["n_slabs"]
            fits = most is None or n <= most
        except visfd_b200.VisfdCudaError as e:
            assert "needs" in str(e), str(e)
            fits = False
        lo, hi = (lo, mid) if fits else (mid, hi)
    got, peak = _fresh_peak(ctx, lambda: fn(hi))
    assert peak <= hi, (got["n_slabs"], peak, hi)
    return got


def test_reference_fixtures_through_the_slab_drivers(ctx, golden):
    """the reference's blob fixture (tests/test_blob_detection.sh:21; 58 scales, masked, as test_gpu_parity's
    test_reference_blob_fixture_gpu) and the golden blob volume, through stream at 2 slabs and at the most slabs a
    budget gives, and on three multi slots"""
    img, sig, mask = golden["blobfix_img"], golden["blobfix_sigmas"], golden["blobfix_mask"]
    ratio = float(golden["blobfix_ratio"])
    kw = dict(minima_threshold=0.0, maxima_threshold=-np.inf, use_threshold_ratios=False)
    stream = lambda b: ctx.blob_dog_stream(img, sig, 0.02, ratio, mask=mask, device_bytes=b, **kw)
    runs = [_at_smallest_budget(ctx, stream, most) for most in (2, None)]
    assert [r["n_slabs"] for r in runs] == [2, 3]
    runs.append(visfd_b200.blob_dog_multi([0, 0, 0], img, sig, 0.02, ratio, mask=mask, **kw))
    for got in runs:
        assert len(got["minima"]) == 11
        assert np.array_equal(sort_blobs(got["minima"]), sort_blobs(golden["blobfix_minima"]))

    # 28 planes, halo 9: the largest slab of three (all 28 planes, 12 of them its own) is the largest slab of two, so
    # no budget takes three stream slabs; multi runs the three-slab plan
    bvol, bsig = golden["blob_vol"], golden["blob_sigmas"]
    for kw, names in ((dict(minima_threshold=0.0, maxima_threshold=-np.inf, use_threshold_ratios=False),
                       ("blob_minima", "blob_maxima")),
                      (dict(minima_threshold=0.5, maxima_threshold=0.5, use_threshold_ratios=True),
                       ("blob_minima_ratio", "blob_maxima_ratio"))):
        stream = lambda b: ctx.blob_dog_stream(bvol, bsig, 0.02, RATIO, device_bytes=b, **kw)
        runs = [_at_smallest_budget(ctx, stream, most) for most in (2, None)]
        assert [r["n_slabs"] for r in runs] == [2, 2]
        runs.append(visfd_b200.blob_dog_multi([0, 0, 0], bvol, bsig, 0.02, RATIO, **kw))
        for got in runs:
            for rows, name in ((got["minima"], names[0]), (got["maxima"], names[1])):
                assert np.array_equal(sort_blobs(rows), sort_blobs(golden[name])), name


def test_dense_candidates_stay_within_the_budget(ctx):
    """white noise at the smallest scales: extrema everywhere.  The stream's lists are sized so that no scale is
    scanned again into larger lists, and the pool stays within the budget at every slab count down to 3."""
    vol = np.random.default_rng(5).standard_normal((96, 80, 88)).astype(np.float32)
    sigmas = np.array([0.5, 0.6, 0.7, 0.8], np.float32)
    kw = dict(minima_threshold=np.inf, maxima_threshold=-np.inf, use_threshold_ratios=False)
    want, one_shot = _fresh_peak(ctx, lambda: ctx.blob_dog(vol, sigmas, 0.02, RATIO, capacity=1 << 21, **kw))
    print(f"dense: {len(want[0])} minima, {len(want[1])} maxima in {vol.size} voxels")
    assert len(want[0]) + len(want[1]) > vol.size // 200
    budget, n = 2 * one_shot, 0
    while n < 3:
        assert budget > one_shot // 50
        got, peak = _fresh_peak(ctx, lambda: ctx.blob_dog_stream(vol, sigmas, 0.02, RATIO, device_bytes=budget,
                                                                 capacity=1 << 21, **kw))
        n = got["n_slabs"]
        assert peak <= budget, (n, peak, budget)
        assert _same((got["minima"], got["maxima"]), want), budget
        budget = budget * 7 // 8


def _c_call(ctx, fn_name, vol, sigmas, capacity, src_ptr=None, front=(), before_capacity=(), back=()):
    """a blob C entry point with `capacity` rows (absolute thresholds 0 / 0)
    -> (rc, n_minima, n_maxima, stored minima rows, stored maxima rows)"""
    nz, ny, nx = vol.shape
    sg = np.ascontiguousarray(sigmas, np.float32)
    rows = max(capacity, 1)
    bufs = [np.zeros((rows, 3), np.float32), np.zeros(rows, np.float32), np.zeros(rows, np.float32),
            np.zeros((rows, 3), np.float32), np.zeros(rows, np.float32), np.zeros(rows, np.float32)]
    ptrs = [C.c_void_p(b.ctypes.data) for b in bufs]
    nmin, nmax = C.c_int64(), C.c_int64()
    src = C.c_void_p(vol.ctypes.data if src_ptr is None else src_ptr)
    rc = getattr(ctx.lib, fn_name)(*front, C.c_int64(nx), C.c_int64(ny), C.c_int64(nz), src, None,
                                   C.c_void_p(sg.ctypes.data), C.c_int(len(sg)), C.c_float(0.02), C.c_float(RATIO),
                                   C.c_float(0.0), C.c_float(0.0), C.c_int(0), *before_capacity, C.c_int64(capacity),
                                   *ptrs[:3], C.byref(nmin), *ptrs[3:], C.byref(nmax), *back)
    k0, k1 = min(nmin.value, capacity), min(nmax.value, capacity)
    pack = lambda c, s, sc, k: np.concatenate([c[:k], s[:k, None], sc[:k, None]], axis=1)
    return rc, nmin.value, nmax.value, pack(*bufs[:3], k0), pack(*bufs[3:], k1)


def test_errors_leave_the_context_usable(ctx):
    import torch
    vol = _volume()
    kw = dict(minima_threshold=0.0, maxima_threshold=-np.inf, use_threshold_ratios=False)
    want = ctx.blob_dog(vol, NARROW, 0.02, RATIO, **kw)

    def still_works():
        got = ctx.blob_dog_stream(vol, NARROW, 0.02, RATIO, **kw)
        assert got["n_slabs"] == 1 and _same((got["minima"], got["maxima"]), want)
        got = visfd_b200.blob_dog_multi([0, 0], vol, NARROW, 0.02, RATIO, **kw)
        assert _same((got["minima"], got["maxima"]), want)

    # a budget below slabs of 8 planes: the message names the bytes needed
    with pytest.raises(visfd_b200.VisfdCudaError) as e:
        ctx.blob_dog_stream(vol, NARROW, 0.02, RATIO, device_bytes=1 << 20, **kw)
    need = re.search(r"needs (\d+) bytes", str(e.value))
    assert need and int(need.group(1)) > 1 << 20, str(e.value)
    still_works()

    # device pointers are refused by both C entry points
    dev = torch.from_numpy(vol).cuda()
    stream = dict(front=(ctx.h,), before_capacity=(C.c_int64(0),), back=(None,))
    devs = (C.c_int * 2)(0, 0)
    multi = dict(front=(C.c_int(2), devs), back=(None,))
    rc = _c_call(ctx, "visfd_cuda_blob_dog_stream", vol, NARROW, 16, src_ptr=dev.data_ptr(), **stream)[0]
    assert rc != 0 and "HOST arrays" in ctx.lib.visfd_cuda_last_error().decode()
    rc = _c_call(ctx, "visfd_cuda_blob_dog_multi", vol, NARROW, 16, src_ptr=dev.data_ptr(), **multi)[0]
    assert rc != 0 and "HOST arrays" in ctx.lib.visfd_cuda_last_error().decode()
    del dev
    still_works()

    # no device
    with pytest.raises(visfd_b200.VisfdCudaError, match="visfd_cuda_blob_dog_multi: need at least one device"):
        visfd_b200.blob_dog_multi([], vol, NARROW, 0.02, RATIO, **kw)
    still_works()

    # a capacity below the counts: the full counts, the first rows, as visfd_cuda_blob_dog
    full = _c_call(ctx, "visfd_cuda_blob_dog", vol, NARROW, 1 << 16, front=(ctx.h,))
    cut = _c_call(ctx, "visfd_cuda_blob_dog", vol, NARROW, 3, front=(ctx.h,))
    assert full[0] == 0 and cut[0] == 0 and cut[1] == full[1] > 3 and cut[2] == full[2] > 3
    assert _same(cut[3:], (full[3][:3], full[4][:3]))
    for name, args in (("visfd_cuda_blob_dog_stream", stream), ("visfd_cuda_blob_dog_multi", multi)):
        got = _c_call(ctx, name, vol, NARROW, 3, **args)
        assert got[0] == 0 and got[1:3] == cut[1:3], name
        assert _same(got[3:], cut[3:]), name
    with pytest.raises(visfd_b200.VisfdCudaError, match="exceed the capacity"):
        ctx.blob_dog_stream(vol, NARROW, 0.02, RATIO, capacity=3, **kw)
    with pytest.raises(visfd_b200.VisfdCudaError, match="exceed the capacity"):
        visfd_b200.blob_dog_multi([0], vol, NARROW, 0.02, RATIO, capacity=3, **kw)
    still_works()
