"""visfd_cuda_filter_stream (Context.filter_stream) and visfd_cuda_filter_multi (filter_multi): ApplyGauss, ApplyDog
and ApplyLog in Z-slabs, on one GPU within a device-memory budget or over several devices.  The result and the peak
heights must equal the one-shot call's (visfd_cuda_apply_gauss / _dog2 / _log) bit for bit, over the whole volume
(masked-out voxels included), at every slab count and in both arithmetic modes; the stream call's pool must never
hold more than its budget (visfd_cuda_peak_reserved_bytes); dst may be src."""
import ctypes as C
import re

import numpy as np
import pytest

import visfd_b200
from visfd_b200 import FilterParams

pytestmark = pytest.mark.gpu

SHAPES = {"ragged_nz": (203, 64, 72),    # the last slab's planes are not a multiple of 8
          "nx_not_x4": (203, 50, 66)}    # the fall-back X sweeps

# name -> (FilterParams, one-shot call on (ctx, vol, mask) -> (out, A, B))
CASES = {
    "gauss": (FilterParams.gauss(2.0, 5), lambda c, v, m: c.apply_gauss(v, 2.0, 5, mask=m) + (0.0,)),
    "gauss_plain": (FilterParams.gauss(2.0, 5, normalize=False),
                    lambda c, v, m: c.apply_gauss(v, 2.0, 5, mask=m, normalize=False) + (0.0,)),
    "gauss_axes": (FilterParams.gauss((1.0, 2.0, 3.0), (3, 5, 8)),
                   lambda c, v, m: c.apply_gauss(v, (1.0, 2.0, 3.0), (3, 5, 8), mask=m) + (0.0,)),
    # equal half-widths: the fused DoG path at full size (no mask, nx % 4 == 0)
    "dog": (FilterParams.dog(1.5, 2.4, 6), lambda c, v, m: c.apply_dog(v, 1.5, 2.4, 6, mask=m, hw_b=6)),
    "dog_hw_b": (FilterParams.dog(1.5, 2.4, 4, hw_b=6), lambda c, v, m: c.apply_dog(v, 1.5, 2.4, 4, mask=m, hw_b=6)),
    "log": (FilterParams.log(2.0, 0.02, 2.5), lambda c, v, m: c.apply_log(v, 2.0, 0.02, 2.5, mask=m)),
    # halo 31 planes: wider than most slabs of a 203-plane volume cut into 6 or more
    "wide_halo": (FilterParams.gauss(8.0, 30), lambda c, v, m: c.apply_gauss(v, 8.0, 30, mask=m) + (0.0,)),
}


def _volume(shape, seed=23):
    return np.random.default_rng(seed).standard_normal(shape).astype(np.float32)


def _cell_mask(shape):
    nz, ny, nx = shape
    z, y, x = np.ogrid[:nz, :ny, :nx]
    inside = ((z - nz / 2) / (0.45 * nz)) ** 2 + ((y - ny / 2) / (0.48 * ny)) ** 2 + ((x - nx / 2) / (0.45 * nx)) ** 2
    return (inside <= 1.0).astype(np.float32)


def _fresh_peak(ctx, fn):
    """fn() with the pool emptied first -> (result, the most the pool held during fn)"""
    ctx.trim()
    ctx.reset_peak_reserved_bytes()
    res = fn()
    return res, ctx.peak_reserved_bytes()


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.int32)


def _same(got, want):
    """the whole volume and both peak heights, bit for bit"""
    out, A, B = want
    return (np.array_equal(_bits(got["out"]), _bits(out)) and _bits(np.float32(got["A"])) == _bits(np.float32(A)) and
            _bits(np.float32(got["B"])) == _bits(np.float32(B)))


def _stream_down(ctx, one_shot_peak, run, check, most=6):
    """run(device_bytes) from twice the one-shot peak down, 1/32 at a time (with the wide halo, 3 slabs fit in a
    window of budgets 6 % wide), until 1, 2, 3 and >= `most` slabs have run; check(result) on each, and the pool
    within the budget -> the slab counts seen"""
    seen, budget = [], 2 * one_shot_peak
    while not ({1, 2, 3} <= set(seen) and max(seen) >= most):
        assert budget > one_shot_peak // 50, f"slab counts seen down to {budget} bytes: {seen}"
        got, peak = _fresh_peak(ctx, lambda: run(budget))
        n = got["n_slabs"]
        assert peak <= budget, (n, peak, budget)
        check(got, n, budget)
        seen.append(n)
        budget = budget * 31 // 32
    return seen


@pytest.mark.parametrize("fast", [False, True])
@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("shape", sorted(SHAPES))
@pytest.mark.parametrize("case", sorted(CASES))
def test_stream_equals_one_shot_at_every_slab_count(ctx, case, shape, masked, fast):
    params, one_shot = CASES[case]
    vol = _volume(SHAPES[shape])
    mask = _cell_mask(vol.shape) if masked else None
    ctx.set_fast_gauss(fast)
    try:
        want, peak = _fresh_peak(ctx, lambda: one_shot(ctx, vol, mask))

        def check(got, n, budget):
            assert _same(got, want), (n, budget)

        _stream_down(ctx, peak, lambda b: ctx.filter_stream(vol, params, mask=mask, device_bytes=b), check)
    finally:
        ctx.set_fast_gauss(False)


@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("shape", sorted(SHAPES))
@pytest.mark.parametrize("case", sorted(CASES))
def test_multi_equals_one_shot(ctx, case, shape, masked):
    import torch
    params, one_shot = CASES[case]
    vol = _volume(SHAPES[shape])
    mask = _cell_mask(vol.shape) if masked else None
    want = one_shot(ctx, vol, mask)
    n_dev = torch.cuda.device_count()
    device_lists = [[0] * k for k in (1, 2, 3, 4, 8)]
    if n_dev > 1:
        device_lists += [list(range(n_dev)), [d % n_dev for d in range(2 * n_dev)]]
    for devices in device_lists:
        got = visfd_b200.filter_multi(devices, vol, params, mask=mask)
        assert _same(got, want), devices
        assert len(got["device_ms"]) == len(devices) and all(t > 0 for t in got["device_ms"]), got["device_ms"]


@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("case", ["wide_halo", "dog_hw_b"])
def test_dst_may_be_src(ctx, case, masked):
    """out=src: a slab's delivery overwrites raw planes that later slabs read as halo, over several slabs with the
    wide halo"""
    params, one_shot = CASES[case]
    vol = _volume(SHAPES["ragged_nz"])
    mask = _cell_mask(vol.shape) if masked else None
    want, peak = _fresh_peak(ctx, lambda: one_shot(ctx, vol, mask))

    def run(budget):
        a = vol.copy()
        got = ctx.filter_stream(a, params, mask=mask, device_bytes=budget, out=a)
        assert got["out"] is a
        return got

    def check(got, n, budget):
        assert _same(got, want), (n, budget)

    _stream_down(ctx, peak, run, check)
    a = vol.copy()
    got = visfd_b200.filter_multi([0] * 8, a, params, mask=mask, out=a)
    assert got["out"] is a and _same(got, want)


def test_default_budget_takes_slabs_when_memory_is_short(ctx):
    """device_bytes = 0 (the shim's path) while a torch allocation leaves little free: several slabs, the same bits"""
    import torch
    shape = (256, 512, 512)   # 256 MiB per volume
    vol = _volume(shape, seed=3)
    params, one_shot = CASES["dog"]
    want = one_shot(ctx, vol, None)
    ctx.trim()
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info()
    target = 2 << 30   # the stream keeps 1 GiB free: about 1 GiB for the slabs, one slab needs 1.25 GiB
    hog = torch.empty(max(0, free - target), dtype=torch.uint8, device="cuda")
    try:
        free_now, _ = torch.cuda.mem_get_info()
        assert free_now < (4 << 30), free_now
        got = ctx.filter_stream(vol, params)
    finally:
        del hog
        torch.cuda.empty_cache()
    assert got["n_slabs"] > 1 and _same(got, want), got["n_slabs"]


def test_errors_leave_the_context_usable(ctx):
    import torch
    vol = _volume(SHAPES["ragged_nz"])
    params, one_shot = CASES["log"]
    want = one_shot(ctx, vol, None)

    def still_works():
        got = ctx.filter_stream(vol, params)
        assert got["n_slabs"] == 1 and _same(got, want)
        assert _same(visfd_b200.filter_multi([0, 0], vol, params), want)

    # a budget below slabs of 8 planes: the message names the bytes needed
    with pytest.raises(visfd_b200.VisfdCudaError) as e:
        ctx.filter_stream(vol, params, device_bytes=1 << 20)
    need = re.search(r"visfd_cuda_filter_stream: the filter needs (\d+) bytes", str(e.value))
    assert need and int(need.group(1)) > 1 << 20, str(e.value)
    still_works()

    # device pointers are refused by both C entry points, torch tensors by the binding
    dev = torch.from_numpy(vol).cuda()
    out = np.empty_like(vol)
    nz, ny, nx = vol.shape
    dims = (C.c_int64(nx), C.c_int64(ny), C.c_int64(nz))
    rc = ctx.lib.visfd_cuda_filter_stream(ctx.h, *dims, C.c_void_p(dev.data_ptr()), None, C.byref(params),
                                          C.c_int64(0), C.c_void_p(out.ctypes.data), None, None, None)
    assert rc != 0 and "visfd_cuda_filter_stream takes HOST arrays" in ctx.lib.visfd_cuda_last_error().decode()
    devs = (C.c_int * 2)(0, 0)
    rc = ctx.lib.visfd_cuda_filter_multi(C.c_int(2), devs, *dims, C.c_void_p(out.ctypes.data), None, C.byref(params),
                                         C.c_void_p(dev.data_ptr()), None, None, None)
    assert rc != 0 and "visfd_cuda_filter_multi takes HOST arrays" in ctx.lib.visfd_cuda_last_error().decode()
    with pytest.raises(visfd_b200.VisfdCudaError, match="visfd_cuda_filter_stream takes numpy"):
        ctx.filter_stream(dev, params)
    del dev
    still_works()

    # no device, an unknown kind
    with pytest.raises(visfd_b200.VisfdCudaError, match="visfd_cuda_filter_multi: need at least one device"):
        visfd_b200.filter_multi([], vol, params)
    with pytest.raises(visfd_b200.VisfdCudaError, match="visfd_cuda_filter_stream: unknown filter kind"):
        ctx.filter_stream(vol, FilterParams(kind=7))
    still_works()
