"""visfd_cuda_membrane_stream_background and visfd_cuda_membrane_multi_background (Context.membrane_stream and
membrane_multi with background_sigma > 0): `-membrane-background` in the Z-slab drivers.  Their result and threshold
must equal visfd_cuda_membrane_background bit for bit at every slab count, with and without a mask and with either
normalisation, and stream must stay within its budget (visfd_cuda_peak_reserved_bytes)."""
import ctypes as C
import re

import numpy as np
import pytest

import visfd_b200
from visfd_b200 import synth

SQ2 = float(np.float32(np.sqrt(2.0)))
RATIO = float(np.float32(np.sqrt(np.float32(-2) * np.log(np.float32(0.03)))))   # Gaussian half-width 3 at sigma 1.2
SHAPE = (203, 64, 72)   # ragged nz: the last slab's planes are not a multiple of 8
ORDER = visfd_b200.DECREASING_EIVALS


def _volume():
    return synth.tomogram(SHAPE, seed=11, n_shells=4)


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


def _same_bits(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.int32), b.view(np.int32))


def _same_threshold(a, b):
    return np.float32(a).view(np.int32) == np.float32(b).view(np.int32)


def _devices(k):
    n = visfd_b200.load_library().visfd_cuda_device_count()
    return [i % n for i in range(k)]


# (cut: a fraction, or "abs" / "below_zero" for an absolute cut from the data, tv_sigma, exponent, background_sigma,
#  normalize, VISFD_CUDA_CHUNK_WAVES=0, voting kernel: 0 MUFU or None)
# background_sigma 3 -> background half-width 7 > 1 + 3, the halo is wider than without it; 1 -> half-width 2
CASES = {
    "fraction_wide_halo": (0.05, 4.0, 4, 3.0, True, True, None),
    "fraction_narrow_halo": (0.05, 4.0, 4, 1.0, True, False, None),
    "absolute_mufu": ("abs", 5.0, 2, 3.0, True, False, 0),
    "no_normalize": (0.05, 4.0, 4, 3.0, False, True, None),
    "no_vote": (0.1, 0.0, 4, 3.0, True, False, None),
    "below_zero": ("below_zero", 4.0, 4, 3.0, True, False, 0),
}


def _case_args(ctx, case, vol, mask):
    """-> (args of Context.membrane, background keyword arguments)"""
    cut, tv_sigma, exponent, sigma_b, normalize, _, _ = CASES[case]
    bg = dict(background_sigma=sigma_b, normalize=normalize)
    is_fraction = not isinstance(cut, str)
    if not is_fraction:
        # the cut that keeps about a fifth of the voxels; below zero: its negative, so that voxels whose peak height
        # is negative, and with it their saliency, vote as well
        t = ctx.membrane(vol, 1.2, RATIO, ORDER, 0.2, True, 0.0, 4, SQ2, mask=mask, **bg)["threshold"]
        assert t > 0
        cut = -t if cut == "below_zero" else t
    return (1.2, RATIO, ORDER, cut, is_fraction, tv_sigma, exponent, SQ2), bg


@pytest.mark.gpu
@pytest.mark.parametrize("masked", [False, True], ids=["nomask", "mask"])
@pytest.mark.parametrize("case", sorted(CASES))
def test_stream_background_equals_one_shot_at_every_slab_count(ctx, monkeypatch, case, masked):
    chunked, kernel = CASES[case][5], CASES[case][6]
    if chunked:   # many small chunks in the overlapped download (slabs of >= 64 own planes: 1 to 3 slabs here)
        monkeypatch.setenv("VISFD_CUDA_CHUNK_WAVES", "0")
    vol = _volume()
    mask = _cell_mask() if masked else None
    args, bg = _case_args(ctx, case, vol, mask)
    want, one_shot = _fresh_peak(ctx, lambda: ctx.membrane(vol, *args, mask=mask, **bg))
    if kernel is not None:
        assert ctx.last_tv_kernel() == kernel
    seen = []
    budget = one_shot
    while not ({1, 2, 3} <= set(seen) and max(seen) >= 6):
        assert budget > one_shot // 50, f"slab counts seen down to {budget} bytes: {seen}"
        got, peak = _fresh_peak(ctx, lambda: ctx.membrane_stream(vol, *args, mask=mask, device_bytes=budget, **bg))
        n = got["n_slabs"]
        assert peak <= budget, (n, peak, budget)
        assert _same_bits(got["out"], want["out"]), (n, budget)
        assert _same_threshold(got["threshold"], want["threshold"]), (n, got["threshold"], want["threshold"])
        if kernel is not None:
            assert ctx.last_tv_kernel() == kernel
        seen.append(n)
        budget = budget * 15 // 16


@pytest.mark.gpu
@pytest.mark.parametrize("masked", [False, True], ids=["nomask", "mask"])
@pytest.mark.parametrize("case", sorted(CASES))
def test_multi_background_equals_one_shot(ctx, monkeypatch, case, masked):
    if CASES[case][5]:
        monkeypatch.setenv("VISFD_CUDA_CHUNK_WAVES", "0")
    vol = _volume()
    mask = _cell_mask() if masked else None
    args, bg = _case_args(ctx, case, vol, mask)
    want = ctx.membrane(vol, *args, mask=mask, **bg)
    for k in (1, 2, 3, 4, 8):
        got = visfd_b200.membrane_multi(_devices(k), vol, *args, mask=mask, **bg)
        assert _same_bits(got["out"], want["out"]), k
        assert _same_threshold(got["threshold"], want["threshold"]), (k, got["threshold"], want["threshold"])


def _stream_background_c(ctx, vol, p, sigma_b, budget, src=None, out=None):
    """the C entry point itself -> (rc, out, threshold, n_slabs)"""
    res = np.empty(SHAPE, np.float32)
    thr, n = C.c_float(), C.c_int64()
    nz, ny, nx = SHAPE
    rc = ctx.lib.visfd_cuda_membrane_stream_background(
        ctx.h, C.c_int64(nx), C.c_int64(ny), C.c_int64(nz), C.c_void_p(src if src else vol.ctypes.data), None,
        C.byref(p), C.c_float(sigma_b), C.c_int(1), C.c_int64(budget), C.c_void_p(out if out else res.ctypes.data),
        C.byref(thr), C.byref(n))
    return rc, res, thr.value, n.value


def _multi_background_c(vol, p, sigma_b, devices):
    lib = visfd_b200.load_library()
    res = np.empty(SHAPE, np.float32)
    thr = C.c_float()
    nz, ny, nx = SHAPE
    devs = (C.c_int * len(devices))(*devices)
    rc = lib.visfd_cuda_membrane_multi_background(len(devices), devs, C.c_int64(nx), C.c_int64(ny), C.c_int64(nz),
                                                  C.c_void_p(vol.ctypes.data), None, C.byref(p), C.c_float(sigma_b),
                                                  C.c_int(1), C.c_void_p(res.ctypes.data), C.byref(thr), None)
    return rc, res, thr.value


@pytest.mark.gpu
def test_background_sigma_zero_is_the_plain_call(ctx):
    vol = _volume()
    args = (1.2, RATIO, ORDER, 0.05, True, 4.0, 4, SQ2)
    p = visfd_b200.MembraneParams(*args[:4], 1, *args[5:])
    want, one_shot = _fresh_peak(ctx, lambda: ctx.membrane(vol, *args))
    # budgets from the free memory down to one the plain call refuses: the same slab counts, then the same refusal
    seen = []
    for budget in [0] + [int(one_shot * 0.875 ** k) for k in range(100)]:
        rc, out, thr, n = _stream_background_c(ctx, vol, p, 0.0, budget)
        err = ctx.lib.visfd_cuda_last_error().decode()
        try:
            plain = ctx.membrane_stream(vol, *args, device_bytes=budget)
        except visfd_b200.VisfdCudaError as e:
            need = re.search(r"needs (\d+) bytes", str(e))
            assert rc != 0 and need, (budget, rc, str(e))
            assert re.search(r"needs (\d+) bytes", err).group(1) == need.group(1), (err, str(e))
            break
        assert rc == 0, (budget, err)
        assert n == plain["n_slabs"], (budget, n, plain["n_slabs"])
        assert _same_bits(out, plain["out"]) and _same_bits(out, want["out"])
        assert _same_threshold(thr, plain["threshold"])
        seen.append(n)
    else:
        pytest.fail(f"no budget was refused: {seen}")
    assert len(set(seen)) >= 3, seen
    for k in (1, 3):
        rc, out, thr = _multi_background_c(vol, p, 0.0, _devices(k))
        assert rc == 0, visfd_b200.load_library().visfd_cuda_last_error().decode()
        assert _same_bits(out, want["out"]) and _same_threshold(thr, want["threshold"])


@pytest.mark.gpu
def test_stream_background_c4_parameters_in_a_third_of_the_one_shot_memory(ctx):
    import torch
    shape = (512, 512, 512)
    vol = synth.tomogram_torch(shape, torch.device("cuda", 0), seed=3).cpu().numpy()
    torch.cuda.empty_cache()
    sigma = float(np.float32(np.float32(5.196) / np.sqrt(3.0)))
    tv_sigma = float(np.float32(np.float32(4.733) * np.float32(sigma)))
    assert visfd_b200.tv_halfwidth(tv_sigma, SQ2) == 20
    assert int(np.floor(np.float32(12.0) * np.float32(RATIO))) == 31   # halo 20 + 31
    args = (sigma, RATIO, ORDER, 0.05, True, tv_sigma, 4, SQ2)
    want, one_shot = _fresh_peak(ctx, lambda: ctx.membrane(vol, *args, background_sigma=12.0))
    budget = one_shot // 3
    got, peak = _fresh_peak(ctx, lambda: ctx.membrane_stream(vol, *args, device_bytes=budget, background_sigma=12.0))
    print(f"512^3, background 12: one shot {one_shot / 2**20:.0f} MiB; stream {peak / 2**20:.0f} MiB "
          f"in {got['n_slabs']} slabs")
    assert peak <= budget and got["n_slabs"] > 1
    assert _same_threshold(got["threshold"], want["threshold"])
    assert _same_bits(got["out"], want["out"])


@pytest.mark.gpu
def test_background_errors_leave_the_context_usable(ctx):
    import torch
    vol = _volume()
    args = (1.2, RATIO, ORDER, 0.05, True, 4.0, 4, SQ2)
    p = visfd_b200.MembraneParams(*args[:4], 1, *args[5:])
    want = ctx.membrane(vol, *args, background_sigma=3.0)
    lib = visfd_b200.load_library()

    def still_works():
        got = ctx.membrane_stream(vol, *args, device_bytes=0, background_sigma=3.0)
        assert got["n_slabs"] == 1 and _same_bits(got["out"], want["out"])
        got = visfd_b200.membrane_multi(_devices(3), vol, *args, background_sigma=3.0)
        assert _same_bits(got["out"], want["out"])

    # a negative or NaN background width
    for sigma_b in (-1.0, float("nan")):
        rc, _, _, _ = _stream_background_c(ctx, vol, p, sigma_b, 0)
        assert rc != 0 and "negative background width" in ctx.lib.visfd_cuda_last_error().decode()
        rc, _, _ = _multi_background_c(vol, p, sigma_b, _devices(2))
        assert rc != 0 and "negative background width" in lib.visfd_cuda_last_error().decode()
        still_works()

    # a budget below one slab of 8 planes: the message names the bytes needed, more than without the background
    def need(**bg):
        with pytest.raises(visfd_b200.VisfdCudaError) as e:
            ctx.membrane_stream(vol, *args, device_bytes=1 << 20, **bg)
        m = re.search(r"needs (\d+) bytes", str(e.value))
        assert m, str(e.value)
        return int(m.group(1))
    assert need(background_sigma=3.0) > need() > 1 << 20
    still_works()

    # device pointers are refused
    dev = torch.from_numpy(vol).cuda()
    out = torch.empty_like(dev)
    rc, _, _, _ = _stream_background_c(ctx, vol, p, 3.0, 0, src=dev.data_ptr(), out=out.data_ptr())
    assert rc != 0 and "HOST arrays" in ctx.lib.visfd_cuda_last_error().decode()
    nz, ny, nx = SHAPE
    devs = (C.c_int * 2)(*_devices(2))
    rc = lib.visfd_cuda_membrane_multi_background(2, devs, C.c_int64(nx), C.c_int64(ny), C.c_int64(nz),
                                                  C.c_void_p(dev.data_ptr()), None, C.byref(p), C.c_float(3.0),
                                                  C.c_int(1), C.c_void_p(out.data_ptr()), None, None)
    assert rc != 0 and "HOST arrays" in lib.visfd_cuda_last_error().decode()
    del dev, out
    still_works()
