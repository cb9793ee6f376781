"""visfd_cuda_membrane_stream (Context.membrane_stream): the membrane pipeline on one GPU in Z-slabs run one after
another within a device-memory budget.  Its result must equal visfd_cuda_membrane bit for bit at every slab count,
and the context's pool must never hold more than the budget (visfd_cuda_peak_reserved_bytes)."""
import ctypes as C
import re

import numpy as np
import pytest

import visfd_b200
from visfd_b200 import synth
from visfd_b200.slab import partition

SQ2 = float(np.float32(np.sqrt(2.0)))
RATIO = float(np.float32(np.sqrt(np.float32(-2) * np.log(np.float32(0.03)))))   # Gaussian half-width 3 at sigma 1.2
SHAPE = (203, 64, 72)   # ragged nz: the last slab's planes are not a multiple of 8


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


def _absolute_cut(ctx, vol, mask):
    """an absolute cut that keeps about a fifth of the voxels"""
    r = ctx.membrane(vol, 1.2, RATIO, visfd_b200.DECREASING_EIVALS, 0.2, True, 0.0, 4, SQ2, mask=mask)
    return r["threshold"]


# (cut, cut_is_fraction, tv_sigma, exponent, masked, voting kernel of the last slab: 1 table, 0 MUFU)
CASES = {
    "fraction": (0.05, True, 4.0, 4, False, 1),
    "fraction_mask": (0.3, True, 5.0, 4, True, 1),
    "absolute_mufu": (None, False, 5.0, 2, False, 0),
    "absolute_mask": (None, False, 4.0, 4, True, 1),
    "no_vote": (0.1, True, 0.0, 4, True, None),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(CASES))
def test_stream_equals_one_shot_at_every_slab_count(ctx, case):
    cut, is_fraction, tv_sigma, exponent, masked, kernel = CASES[case]
    vol = _volume()
    mask = _cell_mask() if masked else None
    if cut is None:
        cut = _absolute_cut(ctx, vol, mask)
    args = (1.2, RATIO, visfd_b200.DECREASING_EIVALS, cut, is_fraction, tv_sigma, exponent, SQ2)
    want, one_shot = _fresh_peak(ctx, lambda: ctx.membrane(vol, *args, mask=mask))
    seen = []
    budget = one_shot
    while not ({1, 2, 3} <= set(seen) and max(seen) >= 6):
        assert budget > one_shot // 50, f"slab counts seen down to {budget} bytes: {seen}"
        got, peak = _fresh_peak(ctx, lambda: ctx.membrane_stream(vol, *args, mask=mask, device_bytes=budget))
        n = got["n_slabs"]
        assert peak <= budget, (n, peak, budget)
        assert _same_bits(got["out"], want["out"]), (n, budget)
        assert np.float32(got["threshold"]).view(np.int32) == np.float32(want["threshold"]).view(np.int32)
        if kernel is not None:
            assert ctx.last_tv_kernel() == kernel
        seen.append(n)
        budget = budget * 15 // 16
    # among them a plan whose last slab is thinner than every other one
    def last_is_thinnest(n):
        own = [z1 - z0 for z0, z1 in partition(SHAPE[0], n)]
        return n > 1 and own[-1] < min(own[:-1])
    assert any(last_is_thinnest(n) for n in seen), seen


@pytest.mark.gpu
def test_stream_c4_parameters_in_a_third_of_the_one_shot_memory(ctx):
    import torch
    shape = (512, 512, 512)
    vol = synth.tomogram_torch(shape, torch.device("cuda", 0), seed=3).cpu().numpy()
    torch.cuda.empty_cache()
    sigma = float(np.float32(np.float32(5.196) / np.sqrt(3.0)))
    tv_sigma = float(np.float32(np.float32(4.733) * np.float32(sigma)))
    assert visfd_b200.tv_halfwidth(tv_sigma, SQ2) == 20
    args = (sigma, RATIO, visfd_b200.DECREASING_EIVALS, 0.05, True, tv_sigma, 4, SQ2)
    want, one_shot = _fresh_peak(ctx, lambda: ctx.membrane(vol, *args))
    budget = one_shot // 3
    got, peak = _fresh_peak(ctx, lambda: ctx.membrane_stream(vol, *args, device_bytes=budget))
    print(f"512^3: one shot {one_shot / 2**20:.0f} MiB; stream {peak / 2**20:.0f} MiB in {got['n_slabs']} slabs")
    assert peak <= budget and got["n_slabs"] > 1
    assert got["threshold"] == want["threshold"]
    assert _same_bits(got["out"], want["out"])


@pytest.mark.gpu
def test_stream_errors_leave_the_context_usable(ctx):
    import torch
    vol = _volume()
    args = (1.2, RATIO, visfd_b200.DECREASING_EIVALS, 0.05, True, 4.0, 4, SQ2)
    want = ctx.membrane(vol, *args)

    def still_works():
        got = ctx.membrane_stream(vol, *args, device_bytes=0)
        assert got["n_slabs"] == 1 and _same_bits(got["out"], want["out"])

    # a budget below one slab of 8 planes: the message names the bytes needed
    with pytest.raises(visfd_b200.VisfdCudaError) as e:
        ctx.membrane_stream(vol, *args, device_bytes=1 << 20)
    need = re.search(r"needs (\d+) bytes", str(e.value))
    assert need and int(need.group(1)) > 1 << 20, str(e.value)
    still_works()

    # device pointers are refused by the C entry point
    dev = torch.from_numpy(vol).cuda()
    out = torch.empty_like(dev)
    p = visfd_b200.MembraneParams(*args[:4], 1, *args[5:])
    nz, ny, nx = SHAPE
    rc = ctx.lib.visfd_cuda_membrane_stream(ctx.h, C.c_int64(nx), C.c_int64(ny), C.c_int64(nz),
                                            C.c_void_p(dev.data_ptr()), None, C.byref(p), C.c_int64(0),
                                            C.c_void_p(out.data_ptr()), None, None)
    assert rc != 0 and "HOST arrays" in ctx.lib.visfd_cuda_last_error().decode()
    del dev, out
    still_works()

    # nothing left to cut
    with pytest.raises(visfd_b200.VisfdCudaError, match="no un-masked voxels"):
        ctx.membrane_stream(vol, *args, mask=np.zeros(SHAPE, np.float32))
    still_works()
