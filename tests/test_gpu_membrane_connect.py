"""visfd_cuda_membrane_connect_stream and visfd_cuda_membrane_connect_multi (Context.membrane_connect_stream,
membrane_connect_multi): the membrane pipeline and `-connect` over Z-slabs with the vote tensor kept on the GPU.
Their out, threshold, labels, cluster counts, maxima and directions must equal, bit for bit and at every slab count,
Context.membrane(..., want_tensor=True) followed by Context.label_connected on its out and tensor (what HandleTV does,
handlers.cpp:1932-1970), and stream must stay within its budget (visfd_cuda_peak_reserved_bytes).  The coverage
assertions make sure that a pass has exercised the seams: for one of the slab plans a test runs, accepted voxels on
both planes next to a slab boundary and a cluster that spans two slabs; and accepted voxels on the first and last
planes, where the stencil is clamped."""
import re

import numpy as np
import pytest

import visfd_b200
from visfd_b200 import synth
from visfd_b200.slab import partition

pytestmark = pytest.mark.gpu
SQ2 = float(np.float32(np.sqrt(2.0)))
RATIO = float(np.float32(np.sqrt(np.float32(-2) * np.log(np.float32(0.03)))))   # Gaussian half-width 3 at sigma 1.2
SHAPE = (203, 64, 72)   # ragged nz: the last slab's planes are not a multiple of 8
ORDER = visfd_b200.DECREASING_EIVALS
ANGLE = 30.0
QUANTILE = 0.5   # clustering threshold: this quantile of the positive scores


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


def _devices(k):
    n = visfd_b200.load_library().visfd_cuda_device_count()
    return [i % n for i in range(k)]


# (masked, background_sigma, consider_dot_product_sign, want_direction)
CASES = {
    "plain": (False, 0.0, False, True),
    "mask_background": (True, 3.0, False, False),
    "mask_signed": (True, 0.0, True, True),
    "background_signed": (False, 1.5, True, False),
}
ARGS = (1.2, RATIO, ORDER, 0.05, True, 4.0, 4, SQ2)


def _composition(ctx, case):
    """-> (volume, mask, keyword arguments of the slab drivers, the composition's result, its peak pool bytes)"""
    masked, sigma_b, signed, want_dir = CASES[case]
    vol = _volume()
    mask = _cell_mask() if masked else None
    bg = dict(background_sigma=sigma_b, normalize=True)

    def run():
        r = ctx.membrane(vol, *ARGS, mask=mask, want_tensor=True, **bg)
        thr = float(np.quantile(r["out"][r["out"] > 0], QUANTILE))
        lc = ctx.label_connected(r["out"], r["tensor"], thr, angle_deg=ANGLE, order=ORDER, mask=mask,
                                 want_direction=want_dir, consider_dot_product_sign=signed)
        return dict(lc, out=r["out"], threshold=r["threshold"], connect=thr)

    want, peak = _fresh_peak(ctx, run)
    kw = dict(mask=mask, want_direction=want_dir, consider_dot_product_sign=signed, **bg)
    assert want["n_clusters"] > 1
    if not masked:   # (the cell mask leaves out the first and last planes)
        accepted = _accepted(want)
        assert accepted[0].any() and accepted[-1].any(), "no accepted voxel on the first or last plane"
    return vol, kw, want, peak


def _accepted(res):
    """voxels in a cluster (outside the mask the labels keep the marker n_maxima + 1)"""
    return (res["labels"] >= 1) & (res["labels"] <= res["n_clusters"])


def _check(got, want, what):
    assert _same_bits(got["out"], want["out"]), what
    assert np.float32(got["threshold"]).view(np.int32) == np.float32(want["threshold"]).view(np.int32), what
    assert got["n_clusters"] == want["n_clusters"] and got["n_maxima"] == want["n_maxima"], what
    assert np.array_equal(got["labels"], want["labels"]), what
    assert _same_bits(got["maxima"], want["maxima"]), what
    if want["direction"] is None:
        assert got["direction"] is None
    else:
        assert _same_bits(got["direction"], want["direction"]), what


def _seams_exercised(res, n):
    """accepted voxels on both planes of some slab boundary, and a cluster on both sides of one"""
    labels, accepted = res["labels"], _accepted(res)
    bounds = [z0 for z0, _ in partition(SHAPE[0], n)[1:]]
    both = [b for b in bounds if accepted[b - 1].any() and accepted[b].any()]
    spanning = [b for b in both if set(np.unique(labels[b - 1][accepted[b - 1]])) &
                set(np.unique(labels[b][accepted[b]]))]
    return bool(both) and bool(spanning)


@pytest.mark.parametrize("case", sorted(CASES))
def test_stream_equals_composition_at_every_slab_count(ctx, case):
    vol, kw, want, one_shot = _composition(ctx, case)
    got = ctx.membrane_connect_stream(vol, *ARGS, want["connect"], angle_deg=ANGLE, device_bytes=0, **kw)
    _check(got, want, "device_bytes=0")
    seen = [got["n_slabs"]]
    budget = one_shot
    while not ({1, 2, 3} <= set(seen) and max(seen) >= 6):
        assert budget > one_shot // 50, f"slab counts seen down to {budget} bytes: {seen}"
        got, peak = _fresh_peak(ctx, lambda: ctx.membrane_connect_stream(vol, *ARGS, want["connect"], angle_deg=ANGLE,
                                                                         device_bytes=budget, **kw))
        n = got["n_slabs"]
        assert peak <= budget, (n, peak, budget)
        _check(got, want, (n, budget))
        seen.append(n)
        budget = budget * 15 // 16
    assert any(_seams_exercised(want, n) for n in set(seen) if n > 1), seen


@pytest.mark.parametrize("case", sorted(CASES))
def test_multi_equals_composition(ctx, case):
    vol, kw, want, _ = _composition(ctx, case)
    ks = (1, 2, 3, 4, 8)
    for k in ks:
        got = visfd_b200.membrane_connect_multi(_devices(k), vol, *ARGS, want["connect"], angle_deg=ANGLE, **kw)
        _check(got, want, k)
    assert any(_seams_exercised(want, k) for k in ks if k > 1)


def test_direction_does_not_change_the_labels(ctx):
    vol, kw, want, _ = _composition(ctx, "plain")
    kw["want_direction"] = False
    got = visfd_b200.membrane_connect_multi(_devices(3), vol, *ARGS, want["connect"], angle_deg=ANGLE, **kw)
    assert got["direction"] is None and np.array_equal(got["labels"], want["labels"])


def test_c1_pass2_through_the_slab_drivers(ctx, golden):
    """BASELINE config 1, pass 2 (-connect 1e+09 -connect-angle 30 on the output of pass 1) through the new calls: the
    stock binary's label image, 1 cluster of 69 voxels (as test_gpu_connect.py::test_c1_pass2_through_the_gpu_path)."""
    sigma, ratio, tv_sigma, expo, cutoff, best = [float(v) for v in golden["c1_params"]]
    args = (sigma, ratio, ORDER, best, True, tv_sigma, int(expo), cutoff, 1e9)
    cli = golden["c1_connect_labels"]
    for res in (ctx.membrane_connect_stream(golden["c1_in_binned"], *args, angle_deg=30.0),
                visfd_b200.membrane_connect_multi(_devices(2), golden["c1_in_binned"], *args, angle_deg=30.0)):
        assert res["n_clusters"] == int(golden["c1_connect_n_clusters"][0]) == 1
        assert np.array_equal(res["labels"] == 1, cli == 1) and int((res["labels"] == 1).sum()) == 69
        assert np.array_equal(res["labels"] == -1, cli == 2)


def test_budget_too_small_fails_and_the_context_stays_usable(ctx):
    vol = _volume()
    with pytest.raises(visfd_b200.VisfdCudaError) as e:
        ctx.membrane_connect_stream(vol, *ARGS, 1.0, angle_deg=ANGLE, device_bytes=1 << 20)
    msg = str(e.value)
    need = re.search(r"needs (\d+) bytes", msg)
    assert "visfd_cuda_membrane_connect_stream" in msg and need and int(need.group(1)) > 1 << 20, msg
    got = ctx.membrane_connect_stream(vol, *ARGS, 1.0, angle_deg=ANGLE, device_bytes=0)
    assert got["n_slabs"] == 1 and (got["out"] > 0).any()
