"""GPU parity: every C-ABI entry point of libvisfd_cuda.so against the CPU oracle on the
same seeded inputs, and against the committed reference vectors.

Tolerances (BASELINE.json:north_star): 1e-5 relative for Gaussian/DoG/LoG outputs,
1e-4 for saliency and vote outputs, normals up to sign, masks / blob lists / index work
bit-exact.  "Relative" is util.rel_err: per-voxel |a-b| / max(|b|, 1e-3 * max|b|).

The separable filters are held to a stricter bar than north_star asks: in their default
(EXACT) arithmetic mode the Gaussian / DoG / LoG / CalcHessian outputs must be
BIT-IDENTICAL to the reference; the 1e-5 tolerance is only used for the opt-in FFMA mode.
"""
import numpy as np
import pytest

from util import (TOL_GAUSS, TOL_SALIENCY, rel_err, tensor_rel_err, direction_err, sort_blobs,
                  vote_score_err)
from visfd_b200 import synth
import visfd_b200 as vb

pytestmark = pytest.mark.gpu
SQ2 = float(np.float32(np.sqrt(2.0)))


def test_library_is_the_cuda_one(ctx):
    import ctypes
    assert ctx.lib.visfd_cuda_version() >= 1
    n0 = ctx.launch_count()
    ctx.apply_gauss(np.ones((4, 4, 4), np.float32), 1.0, 1)
    assert ctx.launch_count() - n0 == 3  # Z, Y, X sweeps


def test_no_fallback_error_paths(ctx):
    with pytest.raises(vb.VisfdCudaError):
        ctx.calc_hessian(np.zeros((2, 5, 5), np.float32), 1.0, 2.5)   # feature.hpp:1260-1264
    with pytest.raises(vb.VisfdCudaError):
        ctx.tv_dense_stick(np.zeros((4, 4, 4), np.float32), np.zeros((4, 4, 4, 3), np.float32), -1.0, 4, SQ2)


# ---- taps (host code of the library) -------------------------------------------------------
def test_taps_bit_exact(golden, oracle):
    for k, (s, hw) in enumerate(golden["taps_cases"]):
        assert np.array_equal(vb.gen_gauss1d(float(s), int(hw)), golden[f"taps_{k}"])
    for s in (0.5, 1.7, 3.0, 7.13, 10.0, 10.5):
        hw = vb.gauss_halfwidth(s, -1.0, 0.03)
        assert np.array_equal(vb.gen_gauss1d(s, hw), oracle.gen_gauss1d(s, hw))


# ---- separable filters -----------------------------------------------------------------------
def test_gauss_golden(ctx, golden):
    vol, mask = golden["vol"], golden["mask"]
    d, A = ctx.apply_gauss(vol, 1.3, 3)
    assert np.array_equal(d, golden["gauss_s1.3_hw3"])
    assert np.float32(A) == golden["gauss_A"]
    assert np.array_equal(ctx.apply_gauss(vol, 1.3, 3, normalize=False)[0], golden["gauss_s1.3_hw3_nonorm"])
    assert np.array_equal(ctx.apply_gauss(vol, (1.0, 2.0, 0.7), (2, 5, 1))[0], golden["gauss_aniso"])
    assert np.array_equal(ctx.apply_gauss(vol, 1.3, 3, mask=mask)[0], golden["gauss_masked"])
    assert np.array_equal(ctx.apply_gauss(vol, 1.3, 3, mask=mask, normalize=False)[0],
                          golden["gauss_masked_nonorm"])
    assert np.array_equal(ctx.apply_gauss(vol, 4.0, 10)[0], golden["gauss_wide"])
    d, a, b = ctx.apply_dog(vol, 1.2, 1.92, 5)
    assert np.array_equal(d, golden["dog"])
    assert np.array_equal(np.array([a, b], np.float32), golden["dog_AB"])
    d, a, b = ctx.apply_log(vol, 1.5, 0.02, 2.6482)
    assert np.array_equal(d, golden["log"])
    assert np.array_equal(np.array([a, b], np.float32), golden["log_AB"])
    assert np.array_equal(ctx.apply_log(vol, 1.5, 0.02, 2.6482, mask=mask)[0], golden["log_masked"])


@pytest.mark.parametrize("shape", [(1, 1, 1), (3, 1, 2), (5, 7, 130), (70, 9, 33), (9, 140, 7), (64, 64, 128),
                                   (67, 65, 131)])
@pytest.mark.parametrize("sigma,hw", [(1.0, 2), (3.0, 7), (8.0, 21)])
def test_gauss_shapes(ctx, oracle, shape, sigma, hw):
    """ragged / degenerate shapes, half-widths beyond the image, unaligned x (scalar tail path)"""
    vol = synth.tomogram(shape, seed=1) if min(shape) > 1 else np.random.default_rng(0).standard_normal(
        shape).astype(np.float32)
    want, A0 = oracle.apply_gauss(vol, sigma, hw)
    got, A1 = ctx.apply_gauss(vol, sigma, hw)
    assert np.array_equal(got, want)
    assert np.float32(A0) == np.float32(A1)


def test_gauss_fast_mode_tolerance(ctx, oracle):
    """opt-in FFMA sweeps: |a-b| <= 1e-5 * max(|b|, 1% of the volume's max)"""
    vol = synth.tomogram((48, 56, 72), seed=21)
    ctx.set_fast_gauss(True)
    try:
        for sigma, hw in ((1.0, 2), (3.0, 7), (8.0, 21)):
            want, _ = oracle.apply_gauss(vol, sigma, hw)
            got, _ = ctx.apply_gauss(vol, sigma, hw)
            assert rel_err(got, want, floor_frac=1e-2) <= TOL_GAUSS
            assert np.abs(got - want).max() <= 4e-7 * np.abs(want).max()
        # several CTAs per column, ragged ends
        vol = synth.tomogram((150, 139, 64), seed=22)
        for sigma, hw in ((3.0, 8), (5.0, 15), (8.0, 21)):
            want, _ = oracle.apply_gauss(vol, sigma, hw)
            got, _ = ctx.apply_gauss(vol, sigma, hw)
            assert np.abs(got - want).max() <= 4e-7 * np.abs(want).max(), (sigma, hw)
    finally:
        ctx.set_fast_gauss(False)


def test_gauss_masked_and_device_path(ctx, oracle):
    import torch
    vol = synth.tomogram((40, 50, 72), seed=2)
    rng = np.random.default_rng(3)
    mask = (rng.random(vol.shape) > 0.3).astype(np.float32)
    mask[rng.random(vol.shape) > 0.9] = 0.5
    for normalize in (True, False):
        want, _ = oracle.apply_gauss(vol, 2.0, 5, mask=mask, normalize=normalize)
        got, _ = ctx.apply_gauss(vol, 2.0, 5, mask=mask, normalize=normalize)
        assert np.array_equal(got, want)
        # device-resident path: same kernels, no staging
        got_d, _ = ctx.apply_gauss(torch.from_numpy(vol).cuda(), 2.0, 5, mask=torch.from_numpy(mask).cuda(),
                                   normalize=normalize)
        assert np.array_equal(got_d.cpu().numpy(), got)
    # explicit taps (ApplySeparable)
    tx, ty, tz = (vb.gen_gauss1d(s, h) for s, h in ((1.0, 3), (2.5, 6), (0.7, 2)))
    want, _ = oracle.apply_gauss(vol, (1.0, 2.5, 0.7), (3, 6, 2))
    got, _ = ctx.apply_separable(vol, (tx, ty, tz))
    assert np.array_equal(got, want)


def test_dog_log(ctx, oracle):
    vol = synth.tomogram((48, 40, 56), seed=4)
    want, a0, b0 = oracle.apply_dog(vol, 2.0, 3.2, 8)
    got, a1, b1 = ctx.apply_dog(vol, 2.0, 3.2, 8)
    assert np.array_equal(got, want)
    assert (np.float32(a0), np.float32(b0)) == (np.float32(a1), np.float32(b1))
    # ApplyLog: a difference of two Gaussians 2 % apart in sigma times 1/delta^2 = 2500 --
    # only bit-exact Gaussians make this reproducible
    vol = synth.tomogram((40, 44, 48), seed=6, blobs=4)
    want, _, _ = oracle.apply_log(vol, 2.0, 0.02, 2.6482)
    got, _, _ = ctx.apply_log(vol, 2.0, 0.02, 2.6482)
    assert np.array_equal(got, want)


def test_dog_shared_z_sweep_with_unequal_halfwidths(ctx, oracle):
    """The pair of Gaussians of a DoG shares one Z sweep (the shorter filter zero-padded and centred in the
    longer one's tap array) whenever that costs no extra group of 8 taps: half-widths 5 and 7 qualify, 5 and 12
    take the separate sweeps.  Either way: the two oracle Gaussians, subtracted, bit for bit."""
    vol = synth.tomogram((44, 36, 64), seed=12)
    for hw_a, hw_b in ((5, 7), (7, 5), (5, 12), (0, 3)):
        ga, _ = oracle.apply_gauss(vol, 2.0, hw_a)
        gb, _ = oracle.apply_gauss(vol, 2.9, hw_b)
        got, _, _ = ctx.apply_dog(vol, 2.0, 2.9, hw_a, hw_b=hw_b)
        assert np.array_equal(got, ga - gb), (hw_a, hw_b)
    # the FFMA mode shares the sweep up to one extra group of taps (5 / 8); equal half-widths share the X sweep too
    ctx.set_fast_gauss(True)
    try:
        for hw_a, hw_b in ((5, 8), (8, 8), (5, 16)):
            ga, _ = oracle.apply_gauss(vol, 2.0, hw_a)
            gb, _ = oracle.apply_gauss(vol, 2.9, hw_b)
            got, _, _ = ctx.apply_dog(vol, 2.0, 2.9, hw_a, hw_b=hw_b)
            assert np.abs(got - (ga - gb)).max() <= 8e-7 * np.abs(vol).max(), (hw_a, hw_b)
    finally:
        ctx.set_fast_gauss(False)


def test_separable_filters_seeded_sweep_of_shapes(ctx, oracle):
    """120 seeded cases over ragged and degenerate shapes (one plane, one row, nx not a multiple of 4, several CTAs
    per column), widths and half-widths (0 included): ApplyGauss, ApplyDog with equal and with unequal half-widths,
    ApplyLog -- each bit for bit the oracle's."""
    rng = np.random.default_rng(2024)
    for it in range(120):
        nx = int(rng.choice([4, 8, 12, 20, 64, 132, 260, 7, 33]))
        ny = int(rng.choice([1, 2, 3, 5, 33, 70, 130]))
        nz = int(rng.choice([1, 2, 7, 40, 100, 140]))
        vol = rng.standard_normal((nz, ny, nx)).astype(np.float32)
        sa = float(rng.uniform(0.5, 6.0))
        sb = sa * float(rng.uniform(1.01, 1.8))
        ratio = float(rng.uniform(1.5, 3.0))
        hw = max(1, int(ratio * sb)) if rng.random() < 0.9 else 0
        kind = ("gauss", "dog", "dog2", "log")[int(rng.integers(0, 4))]
        if kind == "gauss":
            want, _ = oracle.apply_gauss(vol, sa, hw)
            got, _ = ctx.apply_gauss(vol, sa, hw)
        elif kind == "dog":
            want, _, _ = oracle.apply_dog(vol, sa, sb, hw)
            got, _, _ = ctx.apply_dog(vol, sa, sb, hw)
        elif kind == "dog2":
            hwa = max(0, hw - int(rng.integers(0, 6)))
            ga, _ = oracle.apply_gauss(vol, sa, hwa)
            gb, _ = oracle.apply_gauss(vol, sb, hw)
            want = ga - gb
            got, _, _ = ctx.apply_dog(vol, sa, sb, hwa, hw_b=hw)
        else:
            want, _, _ = oracle.apply_log(vol, sa, 0.02, ratio)
            got, _, _ = ctx.apply_log(vol, sa, 0.02, ratio)
        assert np.array_equal(got, want), (it, kind, vol.shape, sa, sb, hw)


def test_gauss_linearity_and_constant(ctx):
    """size-independent properties at a larger size: linearity; a constant image stays
    constant under the normalised filter (borders included)."""
    shape = (96, 160, 256)
    a = synth.tomogram(shape, seed=7)
    b = synth.tomogram(shape, seed=8)
    ga, _ = ctx.apply_gauss(a, 3.0, 7)
    gb, _ = ctx.apply_gauss(b, 3.0, 7)
    gab, _ = ctx.apply_gauss(a + 2 * b, 3.0, 7)
    assert rel_err(gab, ga + 2 * gb, floor_frac=1e-2) <= 2e-5
    gc, _ = ctx.apply_gauss(np.full(shape, 3.25, np.float32), 3.0, 7)
    assert np.abs(gc - 3.25).max() <= 3.25 * 1e-6


def test_gauss_slab_equals_whole(ctx):
    import torch
    shape = (60, 40, 72)
    vol = synth.tomogram(shape, seed=9)
    whole, _ = ctx.apply_gauss(vol, 2.0, 5)
    z0, z1, halo = 20, 41, 5
    lo, hi = z0 - halo, z1 + halo
    slab, _ = ctx.apply_gauss(vol[lo:hi].copy(), 2.0, 5, z_offset=lo, nz_global=shape[0])
    assert np.array_equal(slab[halo:halo + (z1 - z0)], whole[z0:z1])
    # a slab touching the global border reproduces the border normalisation
    slab0, _ = ctx.apply_gauss(vol[:30].copy(), 2.0, 5, z_offset=0, nz_global=shape[0])
    assert np.array_equal(slab0[:25], whole[:25])


# ---- Hessian / eigen / saliency ------------------------------------------------------------------
def test_calc_hessian(ctx, oracle, golden):
    vol, mask = golden["vol"], golden["mask"]
    g, h = ctx.calc_hessian(vol, 1.1, 2.6482)
    assert np.array_equal(g, golden["hess_grad"])
    assert np.array_equal(h, golden["hess_hess"])
    g, h = ctx.calc_hessian(vol, 1.1, 2.6482, mask=mask)
    assert np.array_equal(g, golden["hess_grad_masked"])
    assert np.array_equal(h, golden["hess_hess_masked"])
    assert np.all(h[mask == 0] == 0)


def test_tensor_score_matches_reference_eigen(ctx, oracle, golden):
    """the eigensolver alone, on the reference's own Hessians: float eigenvalues and scores"""
    h = golden["hess_hess"]
    for order in (0, 1):
        sal, ev, dire = ctx.tensor_score(h, order=order, score_kind=vb.SCORE_PLANAR, is_vote_tensor=False,
                                         want_eivals=True, want_direction=True)
        assert rel_err(ev, golden[f"ridge_ev_o{order}"]) <= 1e-6
        assert rel_err(sal, golden[f"ridge_sal_o{order}"]) <= 1e-5
        # normals only where the top eigenvalue is separated (degenerate voxels have none)
        evr = golden[f"ridge_ev_o{order}"].astype(np.float64)
        gap = np.abs(evr[..., 0] - evr[..., 1]) / np.abs(evr).max()
        assert direction_err(dire, golden[f"ridge_dir_o{order}"], weight=gap > 1e-3) <= 1e-5
    sal, _, _ = ctx.tensor_score(h, order=1, score_kind=vb.SCORE_LINEAR, is_vote_tensor=False)
    assert rel_err(sal, golden["ridge_sal_linear"]) <= 1e-5
    sc, _, _ = ctx.tensor_score(golden["mem_tensor"], order=1, score_kind=vb.SCORE_PLANAR, is_vote_tensor=True)
    assert rel_err(sc, golden["tv_score_planar"]) <= 1e-5


def test_newton_eigenvalues_match_closed_form(ctx):
    """sym3_eigenvalues_newton (eigen3.cuh: Newton step on the characteristic polynomial, no transcendental
    functions) against LAPACK in float64 on float32 matrices: generic, nearly double and triple eigenvalues at
    either end of the spectrum, rank one, diagonal, identity multiples, zero, and scales from 1e-12 to 1e12."""
    rng = np.random.default_rng(5)
    mats = []

    def from_spectrum(lam, n):
        q, _ = np.linalg.qr(rng.standard_normal((n, 3, 3)))
        return np.einsum("nij,nj,nkj->nik", q, np.broadcast_to(lam, (n, 3)) if np.ndim(lam) == 1 else lam, q)

    n = 20000
    mats.append(from_spectrum(rng.standard_normal((n, 3)), n))
    for eps in (1e-1, 1e-3, 1e-5, 1e-7, 0.0):
        lam = rng.standard_normal((n // 4, 3))
        lam[:, 1] = lam[:, 0] * (1 + eps * rng.standard_normal(n // 4))          # a nearly double pair
        mats.append(from_spectrum(lam, n // 4))
        lam = 1 + eps * rng.standard_normal((n // 4, 3))                           # nearly triple
        mats.append(from_spectrum(lam, n // 4) * rng.choice([-1.0, 1.0], (n // 4, 1, 1)))
    v = rng.standard_normal((n // 4, 3))
    mats.append(np.einsum("ni,nj->nij", v, v))                                     # rank one (membrane-like)
    d = np.zeros((n // 4, 3, 3))
    d[:, [0, 1, 2], [0, 1, 2]] = rng.standard_normal((n // 4, 3))
    mats.append(d)
    mats.append(np.eye(3)[None] * rng.standard_normal((64, 1, 1)))
    mats.append(np.zeros((8, 3, 3)))
    a = np.concatenate(mats)
    a = a * 10.0 ** rng.integers(-12, 13, (len(a), 1, 1))
    a = 0.5 * (a + np.swapaxes(a, 1, 2))
    flat = np.stack([a[:, 0, 0], a[:, 1, 1], a[:, 2, 2], a[:, 0, 1], a[:, 1, 2], a[:, 0, 2]], -1).astype(np.float32)
    a64 = np.zeros((len(flat), 3, 3))
    for k, (i, j) in enumerate([(0, 0), (1, 1), (2, 2), (0, 1), (1, 2), (0, 2)]):
        a64[:, i, j] = a64[:, j, i] = flat[:, k].astype(np.float64)
    want = np.linalg.eigvalsh(a64)                                                 # ascending
    scale = np.abs(want).max(axis=1, keepdims=True) + 1e-300
    for order in (0, 1):
        _, ev, _ = ctx.tensor_score(flat.reshape(-1, 1, 1, 6), order=order, score_kind=vb.SCORE_PLANAR,
                                    is_vote_tensor=False, want_eivals=True)
        ev = ev.reshape(-1, 3).astype(np.float64)
        w = want.copy()
        if order == 1:        # decreasing = first and last exchanged (eigen3_simple.hpp:252-264)
            w[:, [0, 2]] = w[:, [2, 0]]
        err = np.abs(ev - w) / scale
        # float32 output: half an ulp of the scale, plus the ~1e-8 of a nearly double root (as the reference)
        assert err.max() <= 1.0e-7, (order, err.max(), flat[np.argmax(err.max(axis=1))])


@pytest.mark.parametrize("order", [0, 1])
def test_hessian_ridge(ctx, oracle, order):
    vol = synth.tomogram((36, 44, 52), seed=10)
    if order == 0:
        vol = -vol
    g, h = oracle.calc_hessian(vol, 2.0, 2.6482)
    want_sal, want_dir, want_ev = oracle.hessian_eigen_score(h, order=order)
    sal, dire = ctx.hessian_ridge(vol, 2.0, 2.6482, order=order)
    assert rel_err(sal, want_sal) <= TOL_SALIENCY
    strong = want_sal > 1e-3 * want_sal.max()
    assert direction_err(dire, want_dir, weight=strong) <= 1e-4


def test_ridge_march_kernel_edges(ctx, oracle):
    """The saliency-only kernel (ridge_march_kernel: z-marching register windows) at the shapes where its plane
    bookkeeping can go wrong: 3 planes (every plane uses the stencil of plane 1), chunks of 32 planes that end one
    plane before / on / after the volume, both eigenvalue orders, the linear score, a mask, and slab-local plane
    ranges with a global offset; against the kernel that writes normals too (one thread per voxel) and the oracle."""
    rng = np.random.default_rng(21)
    for shape in ((3, 3, 3), (3, 7, 5), (4, 9, 66), (31, 5, 6), (32, 4, 130), (33, 6, 7), (65, 5, 9)):
        vol = rng.standard_normal(shape).astype(np.float32)
        for order in (0, 1):
            for kind in (vb.SCORE_PLANAR, vb.SCORE_LINEAR):
                a, _ = ctx.hessian_ridge(vol, 1.2, 2.6482, order=order, score_kind=kind, want_direction=False)
                b, _ = ctx.hessian_ridge(vol, 1.2, 2.6482, order=order, score_kind=kind, want_direction=True)
                assert rel_err(a, b) <= 1e-5, (shape, order, kind)
        g, h = oracle.calc_hessian(vol, 1.2, 2.6482)
        want, _, _ = oracle.hessian_eigen_score(h, order=1)
        got, _ = ctx.hessian_ridge(vol, 1.2, 2.6482, order=1, want_direction=False)
        assert rel_err(got, want) <= TOL_SALIENCY, shape
        mask = (rng.random(shape) > 0.3).astype(np.float32)
        g, h = oracle.calc_hessian(vol, 1.2, 2.6482, mask=mask)
        want, _, _ = oracle.hessian_eigen_score(h, order=1, mask=mask)
        got, _ = ctx.hessian_ridge(vol, 1.2, 2.6482, order=1, mask=mask, want_direction=False)
        assert rel_err(got, want) <= TOL_SALIENCY and np.all(got[mask == 0] == 0), shape
    # slab stage: planes [z_offset, z_offset + n) of a taller volume; the planes next to an internal face are not
    # produced (zero), every other plane equals the whole-volume result bit for bit
    import torch
    vol = rng.standard_normal((70, 12, 20)).astype(np.float32)
    whole, _ = ctx.hessian_ridge(vol, 1.2, 2.6482, order=1, want_direction=False)
    hw = 3   # floor(1.2 * 2.6482)
    for (lo, hi) in ((0, 40), (17, 70), (20, 55), (33, 66)):
        dev = torch.from_numpy(np.ascontiguousarray(vol[lo:hi])).cuda()
        sm, sal = ctx.ridge_saliency_slab(dev, lo, vol.shape[0], 1.2, 2.6482, order=1)
        sal = sal.cpu().numpy()
        a = 0 if lo == 0 else hw + 1
        b = hi - lo if hi == vol.shape[0] else hi - lo - hw - 1
        assert np.array_equal(sal[a:b], whole[lo + a:lo + b]), (lo, hi)


def test_hessian_ridge_masked(ctx, oracle):
    vol = synth.tomogram((30, 34, 40), seed=12)
    mask = np.ones(vol.shape, np.float32)
    mask[:, :, :9] = 0
    mask[10:20, 10:20, 20:30] = 0
    g, h = oracle.calc_hessian(vol, 1.5, 2.6482, mask=mask)
    want_sal, want_dir, _ = oracle.hessian_eigen_score(h, order=1, mask=mask)
    sal, dire = ctx.hessian_ridge(vol, 1.5, 2.6482, order=1, mask=mask)
    assert rel_err(sal, want_sal) <= TOL_SALIENCY
    assert np.all(sal[mask == 0] == 0)


# ---- saliency cut ----------------------------------------------------------------------------------
def test_saliency_cut_bit_exact(ctx, oracle, golden):
    sal = golden["ridge_sal_o1"]
    out, thr = ctx.saliency_cut(sal, 0.1, True)
    assert np.float32(thr) == golden["cut_frac0.1_thr"] and np.array_equal(out, golden["cut_frac0.1"])
    out, thr = ctx.saliency_cut(sal, 0.25, True, mask=golden["mask"])
    assert np.float32(thr) == golden["cut_frac0.25_masked_thr"]
    assert np.array_equal(out, golden["cut_frac0.25_masked"])
    out, thr = ctx.saliency_cut(sal, float(golden["cut_frac0.1_thr"]), False)
    assert np.array_equal(out, golden["cut_frac0.1"])


@pytest.mark.parametrize("n,frac", [(1, 0.05), (37, 0.5), (37, 1.0), (1000, 0.0), (100003, 0.05),
                                    (1 << 20, 0.013), (300007, 0.999)])
def test_radix_select_matches_sort(ctx, oracle, n, frac):
    rng = np.random.default_rng(n)
    v = (rng.standard_normal(n) ** 2 * 1e9).astype(np.float32)
    v[rng.random(n) < 0.1] = 0.0                         # ties
    v[rng.random(n) < 0.05] = v[0]
    if n > 100:
        v[:50] = -v[:50]                                 # negative keys too
    want, thr0 = oracle.saliency_cut(v, frac, True)
    got, thr1 = ctx.saliency_cut(v, frac, True)
    assert np.float32(thr0) == np.float32(thr1)
    assert np.array_equal(got, want)
    again, _ = ctx.saliency_cut(got, thr1, False)        # idempotent
    assert np.array_equal(again, got)


# ---- tensor voting -------------------------------------------------------------------------------------
def test_tv_golden(ctx, golden):
    sal, dire = golden["mem_hess_saliency"], golden["mem_direction"]
    assert tensor_rel_err(ctx.tv_dense_stick(sal, dire, 2.4, 4, SQ2), golden["mem_tensor"]) <= TOL_SALIENCY
    assert tensor_rel_err(ctx.tv_dense_stick(sal, dire, 2.4, 2, SQ2), golden["tv_e2"]) <= TOL_SALIENCY
    assert tensor_rel_err(ctx.tv_dense_stick(sal, dire, 2.4, 3, SQ2), golden["tv_e3"]) <= TOL_SALIENCY
    assert tensor_rel_err(ctx.tv_dense_stick(sal, dire, 2.4, 4, SQ2, curves=True),
                          golden["tv_e4_curves"]) <= TOL_SALIENCY
    tm = golden["tv_mask"]
    got = ctx.tv_dense_stick(sal, dire, 2.4, 4, SQ2, mask_src=tm, mask_dst=tm)
    assert tensor_rel_err(got, golden["tv_e4_masked"]) <= TOL_SALIENCY
    assert np.all(got[tm == 0] == 0)


# The voting kernel each radius of test_tv_radii takes (exponent 4, positive weights): the table kernel up to
# radius 24, with the full table (1) while it fits in the B200's 227 KB of shared memory beside the voter rings
# (radius <= 20), else the table clamped at the support (2); the MUFU kernel (0) beyond.
TV_RADII_KERNEL = {2.9: 1, 7.08: 1, 14.2: 1, 15.6: 2, 18.5: 0}


@pytest.mark.parametrize("sigma_tv,shape", [(2.9, (20, 24, 28)), (7.08, (30, 33, 41)), (14.2, (44, 48, 50)),
                                            (15.6, (32, 36, 40)), (18.5, (32, 36, 40))])
def test_tv_radii(ctx, oracle, sigma_tv, shape):
    """vote radii 4, 10, 20, 22 and 26 (hw = floor(sigma*sqrt2)); includes the lattice points that
    sit exactly on the support shell r^2 == hw^2"""
    vol = synth.tomogram(shape, seed=13)
    m = oracle.membrane(vol, 1.5, 2.6482, 1, 0.05, True, 0.0, 4, SQ2)
    sal, dire = m["hess_saliency"], m["direction"]
    want = oracle.tv_dense_stick(sal, dire, sigma_tv, 4, SQ2)
    got = ctx.tv_dense_stick(sal, dire, sigma_tv, 4, SQ2)
    assert ctx.last_tv_kernel() == TV_RADII_KERNEL[sigma_tv]
    assert tensor_rel_err(got, want) <= TOL_SALIENCY
    hw = vb.tv_halfwidth(sigma_tv, SQ2)
    pairs = ctx.tv_count_pairs(sal, -np.inf, hw)
    assert pairs > 0


def test_tv_nonpositive_weights_and_no_voters(ctx, oracle):
    """a voter with negative saliency (thr = -inf) leaves the table kernel for the MUFU kernel without
    the sqrt(weight) form; no voters at all: MUFU kernel, all-zero tensor"""
    vol = synth.tomogram((20, 24, 28), seed=13)
    m = oracle.membrane(vol, 1.5, 2.6482, 1, 0.05, True, 0.0, 4, SQ2)
    sal, dire = m["hess_saliency"].copy(), m["direction"]
    # negative voters at x < 10, positive ones at x >= 18: the radius is 4, so no receiver adds votes of
    # both signs (a cancelling sum would be judged against its own small size)
    sal[:, :, :10] *= -1.0
    sal[:, :, 10:18] = 0.0
    assert (sal < 0).any() and (sal > 0).any()
    want = oracle.tv_dense_stick(sal, dire, 2.9, 4, SQ2)
    got = ctx.tv_dense_stick(sal, dire, 2.9, 4, SQ2)
    assert ctx.last_tv_kernel() == 0
    assert tensor_rel_err(got, want) <= TOL_SALIENCY
    got = ctx.tv_dense_stick(np.zeros_like(sal), dire, 2.9, 4, SQ2)
    assert ctx.last_voter_count() == 0 and ctx.last_tv_kernel() == 0
    assert not got.any()


def test_tv_single_voter_support(ctx, oracle):
    """one voter: the support is exactly the reference's truncated table (shell included)"""
    for sigma_tv in (2.9, 3.6, 5.0, 7.08):
        hw = vb.tv_halfwidth(sigma_tv, SQ2)
        n = 2 * hw + 5
        sal = np.zeros((n, n, n), np.float32)
        dire = np.zeros((n, n, n, 3), np.float32)
        c = n // 2
        sal[c, c, c] = 2.0
        dire[c, c, c] = (0.6, 0.0, 0.8)
        want = oracle.tv_dense_stick(sal, dire, sigma_tv, 4, SQ2)
        got = ctx.tv_dense_stick(sal, dire, sigma_tv, 4, SQ2)
        tw, tg = np.abs(want).sum(-1), np.abs(got).sum(-1)
        # same support: every voxel the reference votes on (above rounding dust: votes along
        # the stick axis are exactly 0 there, ~1e-14 here) and nothing outside its table
        assert np.all(tg[tw > 1e-6 * tw.max()] > 0)
        assert np.all(tg[tw == 0] <= 1e-9 * tw.max())
        assert tensor_rel_err(got, want) <= TOL_SALIENCY


def test_membrane_golden_and_c1(ctx, golden):
    tvol = golden["tv_vol"]
    m = ctx.membrane(tvol, 1.0, 2.6482, 1, 0.12, True, 2.4, 4, SQ2, want_saliency=True, want_direction=True,
                     want_tensor=True)
    assert np.float32(m["threshold"]) == golden["mem_thr"] or rel_err(m["threshold"], golden["mem_thr"]) <= 1e-5
    kept_ref = golden["mem_hess_saliency"] != 0
    assert np.array_equal(m["hess_saliency"] != 0, kept_ref)       # same survivors
    assert rel_err(m["hess_saliency"], golden["mem_hess_saliency"]) <= TOL_SALIENCY
    assert direction_err(m["direction"], golden["mem_direction"], weight=kept_ref) <= 1e-4
    assert tensor_rel_err(m["tensor"], golden["mem_tensor"]) <= TOL_SALIENCY
    assert rel_err(m["out"], golden["mem_out"]) <= TOL_SALIENCY
    # same call without the optional outputs takes the recompute-directions path
    m2 = ctx.membrane(tvol, 1.0, 2.6482, 1, 0.12, True, 2.4, 4, SQ2)
    assert rel_err(m2["out"], golden["mem_out"]) <= TOL_SALIENCY
    mm = ctx.membrane(tvol, 1.0, 2.6482, 1, 0.12, True, 2.4, 4, SQ2, mask=golden["tv_mask"])
    assert rel_err(mm["out"], golden["mem_masked_out"]) <= TOL_SALIENCY
    mx = ctx.membrane(-tvol, 1.0, 2.6482, 0, 0.12, True, 2.4, 4, SQ2)
    assert rel_err(mx["out"], golden["mem_maxima_out"]) <= TOL_SALIENCY
    # BASELINE config 1 (the reference's own test, output of the stock filter_mrc binary)
    sigma, ratio, tv_sigma, expo, tv_ratio, frac = [float(v) for v in golden["c1_params"]]
    c1 = ctx.membrane(golden["c1_in_binned"], sigma, ratio, 1, frac, True, tv_sigma, int(expo), tv_ratio)
    assert rel_err(c1["out"], golden["c1_out"]) <= TOL_SALIENCY
    assert (c1["out"] != 0).sum() == 419
    assert abs(c1["out"].sum(dtype=np.float64) / 4.141152e11 - 1) < 1e-5
    c1n = ctx.membrane(golden["c1_in_binned"], sigma, ratio, 1, frac, True, 0.0, int(expo), tv_ratio)
    assert rel_err(c1n["out"], golden["c1_out_notv"]) <= TOL_SALIENCY
    assert (c1n["out"] != 0).sum() == 27


def test_membrane_pipeline_vs_oracle(ctx, oracle):
    """the C4 parameter set (sigma 3, hw_gauss 7, sigma_tv 14.2, hw_tv 20, exponent 4,
    -tv-best 0.05) on a volume the oracle finishes in seconds"""
    vol = synth.tomogram((56, 60, 64), seed=14, n_shells=2)
    sigma, ratio, tv_sigma = 2.99991, 2.6482, 14.1986
    want = oracle.membrane(vol, sigma, ratio, 1, 0.05, True, tv_sigma, 4, SQ2, want_tensor=True)
    got = ctx.membrane(vol, sigma, ratio, 1, 0.05, True, tv_sigma, 4, SQ2, want_saliency=True, want_tensor=True)
    # Gaussian + finite differences are bit-exact and the eigenvalues agree to double
    # rounding, so the cut threshold and the set of surviving voxels are IDENTICAL
    assert np.float32(got["threshold"]) == np.float32(want["threshold"])
    assert np.array_equal(got["hess_saliency"] != 0, want["hess_saliency"] != 0)
    assert rel_err(got["hess_saliency"], want["hess_saliency"], floor_frac=1e-6) <= TOL_SALIENCY
    assert tensor_rel_err(got["tensor"], want["tensor"]) <= TOL_SALIENCY
    assert vote_score_err(got["out"], want["out"], want["tensor"]) <= TOL_SALIENCY
    # thresholded mask of the result (-thresh at the 99th percentile): bit-exact except
    # voxels within tolerance of the threshold
    T = float(np.quantile(want["out"], 0.99))
    ma = ctx.threshold(got["out"], vb.THRESH_SINGLE, [T])
    mb = oracle.threshold1(want["out"], T)
    differ = ma != mb
    assert np.all(np.abs(want["out"][differ] - T) <= TOL_SALIENCY * T)


def test_c4_full_size_crops_match_oracle(ctx, oracle):
    """BASELINE config 4 at its full size (2048 x 2048 x 1024, the bench workload and seed): the oracle
    cannot run 4.3 Gvoxel, but a crop with a margin of hw_tv + 1 + hw_gauss = 28 voxels reproduces the
    interior exactly when it is given the full run's cut as an ABSOLUTE threshold (SURVEY 8d).  38 interiors: three
    16^3 ones (on the membrane shell in the middle of the volume; the first and last image corners, where the crop's
    border is the image border), 32 seeded random 8^3 ones and three across the planes z = 128 k."""
    import torch
    shape = (1024, 2048, 2048)
    sigma = float(np.float32(np.float32(5.196) / np.sqrt(3.0)))
    tv_sigma = float(np.float32(np.float32(4.733) * np.float32(sigma)))
    ratio = float(np.sqrt(-2.0 * np.log(0.03)))
    vol = synth.tomogram_torch(shape, "cuda", seed=0)
    out = torch.empty_like(vol)
    r = ctx.membrane(vol, sigma, ratio, 1, 0.05, True, tv_sigma, 4, SQ2, out=out)
    n = float(np.prod(shape))
    assert abs(ctx.last_voter_count() / n - 0.05) < 1e-6
    assert float(out.min().item()) >= 0.0 and bool(torch.isfinite(out).all().item())
    margin = 28
    # (the first interior straddles linear voxel index 2^31, the third one ends at index 2^32 - 1)
    boxes = [((504, 1016, 1322), 16), ((0, 0, 0), 16), ((1008, 2032, 2032), 16)]
    # 32 seeded random 8^3 interiors, half of them pulled onto the membrane shell (radius 0.3 * 1024 around the
    # volume centre), plus interiors that straddle the planes where an 8-GPU run cuts the volume (z = 128 k)
    rng = np.random.default_rng(2024)
    for k in range(32):
        if k % 2:
            d = rng.standard_normal(3)
            c = np.array([512.0, 1024.0, 1024.0]) + 307.2 * d / np.linalg.norm(d)
        else:
            c = rng.uniform(0, 1, 3) * np.array(shape)
        corner = tuple(int(min(max(v - 4, 0), s - 8)) for v, s in zip(c, shape))
        boxes.append((corner, 8))
    for k in (1, 4, 7):
        boxes.append(((128 * k - 4, 1024 - 4 + 37 * k, 1024 + 300), 8))
    strict = []
    n_live = 0
    for corner, side in boxes:
        lo = [max(c - margin, 0) for c in corner]
        hi = [min(c + side + margin, s) for c, s in zip(corner, shape)]
        crop = vol[lo[0]:hi[0], lo[1]:hi[1], lo[2]:hi[2]].contiguous().cpu().numpy()
        want = oracle.membrane(crop, sigma, ratio, 1, r["threshold"], False, tv_sigma, 4, SQ2, want_tensor=True)
        inner = tuple(slice(c - l, c - l + side) for c, l in zip(corner, lo))
        got = out[corner[0]:corner[0] + side, corner[1]:corner[1] + side, corner[2]:corner[2] + side].cpu().numpy()
        w = want["out"][inner]
        n_live += int(w.max() > 0)
        assert vote_score_err(got, w, want["tensor"][inner]) <= TOL_SALIENCY, (corner, side)
        nz = w > 1e-3 * max(float(w.max()), 1e-30)
        strict.append(np.abs(got[nz] - w[nz]) / w[nz])
    assert n_live >= 20, "too few interiors see any vote"
    # the PLAIN relative error of the post-vote score lambda1 - lambda2 (no trace floor), over the voxels whose score
    # exceeds 1e-3 of their interior's maximum: what vote_score_err's floor (10 % of the trace) is there to absorb
    strict = np.concatenate(strict)
    p50, p99, pmax = [float(v) for v in (np.quantile(strict, 0.5), np.quantile(strict, 0.99), strict.max())]
    print("C4 post-vote score, strict relative error over %d voxels: p50 %.2e p99 %.2e max %.2e" %
          (strict.size, p50, p99, pmax))
    assert p50 <= 2e-6 and p99 <= 1e-4, (p50, p99, pmax)
    # the Gaussian alone at the same size (hw 7), and the 99th-percentile threshold map of the result
    # (BASELINE config 5's last stage): bit-exact on the same three interiors
    del out
    smooth, _ = ctx.apply_gauss(vol, sigma, 7)
    for corner in ((504, 1016, 1322), (0, 0, 0), (1008, 2032, 2032)):
        lo = [max(c - 7, 0) for c in corner]
        hi = [min(c + side + 7, s) for c, s in zip(corner, shape)]
        crop = vol[lo[0]:hi[0], lo[1]:hi[1], lo[2]:hi[2]].contiguous().cpu().numpy()
        want = oracle.apply_gauss(crop, sigma, 7)[0]
        inner = tuple(slice(c - l, c - l + side) for c, l in zip(corner, lo))
        got = smooth[corner[0]:corner[0] + side, corner[1]:corner[1] + side, corner[2]:corner[2] + side].cpu().numpy()
        assert np.array_equal(got, want[inner])
    m = ctx.threshold(smooth, vb.THRESH_SINGLE, [-0.01])
    for corner in ((504, 1016, 1322), (0, 0, 0), (1008, 2032, 2032)):
        box = tuple(slice(c, c + side) for c in corner)
        assert np.array_equal(m[box].cpu().numpy(), oracle.threshold1(smooth[box].contiguous().cpu().numpy(), -0.01))
    ones = int((m == 1.0).sum().item())
    assert ones + int((m == 0.0).sum().item()) == m.numel() and 0 < ones < m.numel()
    del vol, smooth, m
    torch.cuda.empty_cache()


def test_membrane_masked_c4_parameters(ctx, oracle):
    """`-mask` is the normal way membrane detection is run: the C4 parameter set (sigma 3, vote radius 20, tv-best 0.05)
    on a 192^3 volume with a centred box mask covering 80 % of it, plus a weighted rim (mask value 0.5) one voxel
    thick inside the box -- masks route the Gaussian through the masked sweeps and disable the chunked upload."""
    shape = (192, 192, 192)
    sigma = float(np.float32(np.float32(5.196) / np.sqrt(3.0)))
    tv_sigma = float(np.float32(np.float32(4.733) * np.float32(sigma)))
    ratio = float(np.sqrt(-2.0 * np.log(0.03)))
    vol = synth.tomogram(shape, seed=5)
    mask = np.zeros(shape, np.float32)
    lo = int(round(192 * (1 - 0.8 ** (1 / 3)) / 2))
    mask[lo:192 - lo, lo:192 - lo, lo:192 - lo] = 0.5
    mask[lo + 1:191 - lo, lo + 1:191 - lo, lo + 1:191 - lo] = 1.0
    want = oracle.membrane(vol, sigma, ratio, 1, 0.05, True, tv_sigma, 4, SQ2, mask=mask, want_tensor=True)
    got = ctx.membrane(vol, sigma, ratio, 1, 0.05, True, tv_sigma, 4, SQ2, mask=mask, want_saliency=True,
                       want_tensor=True)
    assert np.float32(got["threshold"]) == np.float32(want["threshold"])
    assert np.array_equal(got["hess_saliency"] != 0, want["hess_saliency"] != 0)
    assert np.all(got["out"][mask == 0] == 0)
    assert tensor_rel_err(got["tensor"], want["tensor"]) <= TOL_SALIENCY
    assert vote_score_err(got["out"], want["out"], want["tensor"]) <= TOL_SALIENCY


def test_membrane_device_path_identical(ctx):
    import torch
    vol = synth.tomogram((40, 40, 48), seed=15)
    a = ctx.membrane(vol, 2.0, 2.6482, 1, 0.05, True, 5.0, 4, SQ2)
    b = ctx.membrane(torch.from_numpy(vol).cuda(), 2.0, 2.6482, 1, 0.05, True, 5.0, 4, SQ2)
    assert np.array_equal(a["out"], b["out"].cpu().numpy())
    assert ctx.last_voter_count() > 0


def test_membrane_host_path_chunked_d2h(ctx, monkeypatch):
    """>= 64 planes: with host arrays the voting runs in z-chunks whose results are copied back
    behind the kernels; it must equal the single-launch device path bit for bit.  The library keeps
    chunks large enough to fill the GPU for many waves, so a small test volume is only chunked when
    VISFD_CUDA_CHUNK_WAVES lowers that bound: 70 planes -> 9 chunks of 8 planes, the last one ragged."""
    import torch
    vol = synth.tomogram((70, 24, 40), seed=16)
    b = ctx.membrane(torch.from_numpy(vol).cuda(), 1.5, 2.6482, 1, 0.08, True, 4.3, 4, SQ2)
    launches = {}
    for waves in ("0", None):
        if waves is None:
            monkeypatch.delenv("VISFD_CUDA_CHUNK_WAVES", raising=False)
        else:
            monkeypatch.setenv("VISFD_CUDA_CHUNK_WAVES", waves)
        before = ctx.launch_count()
        a = ctx.membrane(vol, 1.5, 2.6482, 1, 0.08, True, 4.3, 4, SQ2)
        launches[waves] = ctx.launch_count() - before
        assert np.array_equal(a["out"], b["out"].cpu().numpy())
        assert np.count_nonzero(a["out"]) > 0
    assert launches["0"] - launches[None] == 8     # nine voting launches instead of one


def test_membrane_host_path_chunked_upload(ctx, monkeypatch):
    """host source without a mask: upload, smoothing and ridge saliency run as a pipeline over z-chunks
    (each a z-slab with hw+1 halo planes, uploaded behind the previous chunk's kernels).  Forced onto a
    small volume with VISFD_CUDA_UPLOAD_CHUNK, every output must equal the single-pass device path
    bit for bit: chunks of 8 planes (9 chunks, the last ragged), of 5 (not a multiple of anything),
    and one larger than the halo allows to overlap (37: two chunks)."""
    import torch
    vol = synth.tomogram((70, 24, 40), seed=18, n_shells=2)
    args = (1.5, 2.6482, 1, 0.08, True, 4.3, 4, SQ2)
    want = ctx.membrane(torch.from_numpy(vol).cuda(), *args, want_saliency=True, want_direction=True, want_tensor=True)
    for chunk in ("8", "5", "37"):
        monkeypatch.setenv("VISFD_CUDA_UPLOAD_CHUNK", chunk)
        before = ctx.launch_count()
        got = ctx.membrane(vol, *args, want_saliency=True, want_direction=True, want_tensor=True)
        n_chunks = -(-70 // int(chunk))
        assert ctx.launch_count() - before >= 4 * n_chunks      # 3 sweeps + ridge per chunk
        assert np.float32(got["threshold"]) == np.float32(want["threshold"])
        for k in ("out", "hess_saliency", "direction", "tensor"):
            assert np.array_equal(got[k], want[k].cpu().numpy()), (chunk, k)
        # and without voting (the saliency lands in `out`)
        a = ctx.membrane(vol, 1.5, 2.6482, 1, 0.08, True, 0.0, 4, SQ2)
        monkeypatch.delenv("VISFD_CUDA_UPLOAD_CHUNK")
        b = ctx.membrane(vol, 1.5, 2.6482, 1, 0.08, True, 0.0, 4, SQ2)
        assert np.array_equal(a["out"], b["out"])


# ---- thresholds -----------------------------------------------------------------------------------------
def test_thresholds_bit_exact(ctx, oracle, golden):
    x = golden["thr_x"]
    assert np.array_equal(ctx.threshold(x, vb.THRESH_SINGLE, [0.5]), golden["thr1"])
    assert np.array_equal(ctx.threshold(x, vb.THRESH_2, [0.2, 1.4]), golden["thr2_up"])
    assert np.array_equal(ctx.threshold(x, vb.THRESH_2, [1.4, 0.2], -1.0, 2.0), golden["thr2_down"])
    assert np.array_equal(ctx.threshold(x, vb.THRESH_4, [-1.0, -0.5, 1.5, 2.0]), golden["thr4"])
    assert np.array_equal(ctx.threshold(x, vb.THRESH_4, [2.0, 1.5, -0.5, -1.0]), golden["thr4_rev"])
    rng = np.random.default_rng(5)
    v = rng.standard_normal(100001).astype(np.float32)
    mask = (rng.random(v.size) > 0.5).astype(np.float32)
    want = oracle.threshold2(v, -0.3, 0.8, 0.0, 1.0)
    got = ctx.threshold(v, vb.THRESH_2, [-0.3, 0.8], mask=mask, masked_value=-7.0)
    assert np.array_equal(got[mask != 0], want[mask != 0]) and np.all(got[mask == 0] == -7.0)
    r = ctx.threshold(None, vb.RESCALE, [2.0, 1.0], out=v.copy())
    assert np.array_equal(r, v * np.float32(2.0) + np.float32(1.0))
    empty = ctx.threshold(np.zeros(0, np.float32), vb.THRESH_SINGLE, [0.0])
    assert empty.size == 0


def test_mean_stddev(ctx, golden):
    vol, mask = golden["vol"], golden["mask"]
    m, s = ctx.mean_stddev(vol)
    mw, sw = ctx.mean_stddev(vol, mask)
    np.testing.assert_allclose([m, s, mw, sw], golden["mean_std"], rtol=2e-6)
    # the same numbers from per-slab partial sums (what the ranks all-reduce for -cl)
    import torch
    from visfd_b200.slab import distributed_mean_stddev, partition

    class TwoRanks:                      # stands in for torch.distributed: sums over two emulated ranks
        def __init__(self, parts):
            self.parts, self.calls = parts, 0

        def moment_sums(self, own, w, center, squared):
            tot = [0.0, 0.0]
            for a, ww in self.parts:
                s = ctx.moment_sums(a, ww, center, squared)
                tot = [tot[0] + s[0], tot[1] + s[1]]
            return tuple(tot)

    (a0, a1), (b0, b1) = partition(vol.shape[0], 2)
    dv, dm = torch.from_numpy(vol).cuda(), torch.from_numpy(mask).cuda()
    be = TwoRanks([(dv[a0:a1].contiguous(), None), (dv[b0:b1].contiguous(), None)])
    assert distributed_mean_stddev(be, None) == (m, s)
    be = TwoRanks([(dv[a0:a1].contiguous(), dm[a0:a1].contiguous()), (dv[b0:b1].contiguous(), dm[b0:b1].contiguous())])
    np.testing.assert_allclose(distributed_mean_stddev(be, None), (mw, sw), rtol=1e-6)


# ---- blobs ---------------------------------------------------------------------------------------------------
def test_blob_dog_lists_exact(ctx, oracle, golden):
    bvol, sig = golden["blob_vol"], golden["blob_sigmas"]
    for kw, names in ((dict(minima_threshold=0.0, maxima_threshold=-np.inf, use_threshold_ratios=False),
                       ("blob_minima", "blob_maxima")),
                      (dict(minima_threshold=0.5, maxima_threshold=0.5, use_threshold_ratios=True),
                       ("blob_minima_ratio", "blob_maxima_ratio"))):
        mn, mx = ctx.blob_dog(bvol, sig, 0.02, 2.6482, **kw)
        for got, name in ((mn, names[0]), (mx, names[1])):
            want = sort_blobs(golden[name])
            got = sort_blobs(got)
            assert got.shape == want.shape
            assert np.array_equal(got, want)      # positions, scales AND scores: bit-exact


def test_blob_dog_masked_vs_oracle(ctx, oracle):
    vol = synth.tomogram((30, 34, 38), seed=16, blobs=12, noise=0.1, n_shells=0, blob_sigma=(1.5, 2.5))
    mask = np.ones(vol.shape, np.float32)
    mask[:, :8, :] = 0
    sig = 1.0 * 1.25 ** np.arange(6)
    want = oracle.blob_dog(vol, sig, 0.02, 2.6482, mask=mask, minima_threshold=0.0, maxima_threshold=-np.inf,
                           use_threshold_ratios=False)
    got = ctx.blob_dog(vol, sig, 0.02, 2.6482, mask=mask, minima_threshold=0.0, maxima_threshold=-np.inf,
                       use_threshold_ratios=False)
    for g, w in zip(got, want):
        g, w = sort_blobs(g), sort_blobs(w)
        assert g.shape == w.shape and np.array_equal(g, w)


# ---- Z-slab stages (multi-GPU building blocks, emulated on one GPU) -----------------------------------
@pytest.mark.parametrize("world", [2, 3])
def test_slab_stages_reproduce_whole_volume(ctx, world):
    """each emulated rank runs SlabMembrane's stages on its slab (own planes + raw-source
    halo); stitched together the result equals the single-volume pipeline bit for bit: the ridge
    saliency, the global cut and the post-vote score"""
    import torch
    from visfd_b200.slab import make_plan, distributed_cut_threshold
    shape = (60, 40, 48)
    vol = synth.tomogram(shape, seed=17, n_shells=2)
    sigma, ratio, tv_sigma = 1.5, 2.6482, 4.3
    whole = ctx.membrane(vol, sigma, ratio, 1, 0.08, True, tv_sigma, 4, SQ2, want_saliency=True)
    p = vb.MembraneParams(sigma, ratio, 1, 0.08, 1, tv_sigma, 4, SQ2)
    gauss_hw = int(np.floor(np.float32(sigma) * np.float32(ratio)))
    tv_hw = vb.tv_halfwidth(tv_sigma, SQ2)
    dvol = torch.from_numpy(vol).cuda()
    plans = [make_plan(shape[0], world, r, gauss_hw, tv_hw) for r in range(world)]
    stage1 = []
    for pl in plans:
        sm, sal = ctx.ridge_saliency_slab(dvol[pl.slab[0]:pl.slab[1]].contiguous(), pl.slab[0], shape[0], sigma, ratio)
        stage1.append((sm, sal))
    # the global cut over the union of the ranks' OWN planes (what the all-reduce computes)
    own_sal = torch.cat([stage1[r][1][plans[r].own_local[0]:plans[r].own_local[1]] for r in range(world)])
    assert np.array_equal(own_sal.cpu().numpy() >= whole["threshold"], whole["hess_saliency"] != 0)
    thr = distributed_cut_threshold(ctx, own_sal, 0.08)
    assert np.float32(thr) == np.float32(whole["threshold"])
    out = np.zeros(shape, np.float32)
    for pl, (sm, sal) in zip(plans, stage1):
        res, _ = ctx.vote_slab(sal, sm, pl.slab[0], shape[0], pl.own_local, pl.vote_local, thr, p)
        out[pl.own[0]:pl.own[1]] = res.cpu().numpy()
    assert rel_err(out, whole["out"], floor_frac=1e-2) <= 1e-5
    # slabs and voter planes start on multiples of 8 planes (visfd_b200/slab.py, visfd_cuda_vote_slab), so
    # every receiver meets its voters in the order of the undivided volume: identical float sums
    assert all(pl.own[0] % 8 == 0 and pl.slab[0] % 8 == 0 for pl in plans)
    assert np.array_equal(out, whole["out"])


@pytest.mark.parametrize("world", [2, 3])
def test_blob_slabs_reproduce_whole_volume(ctx, oracle, world):
    """visfd_cuda_blob_dog_slab on each emulated rank's slab (own planes + LoG halo), lists concatenated per
    scale in rank order, best scores reduced, visfd_cuda_blob_finalize == BlobDog on the whole volume (and the
    oracle), rows and order, for ratio and absolute thresholds"""
    import torch
    from visfd_b200.slab import make_plan, log_halfwidth, _concat_by_scale
    shape = (61, 40, 52)
    vol = synth.tomogram(shape, seed=19, n_shells=0, blobs=30, blob_sigma=(1.0, 3.0))
    dvol = torch.from_numpy(vol).cuda()
    sigmas = (1.0 * 1.25 ** np.arange(6)).astype(np.float32)
    hw = max(log_halfwidth(s, 0.02, 2.6482) for s in sigmas)
    plans = [make_plan(shape[0], world, r, hw, 0) for r in range(world)]
    for kw in (dict(minima_threshold=0.3, maxima_threshold=0.3, use_threshold_ratios=True),
               dict(minima_threshold=0.0, maxima_threshold=-np.inf, use_threshold_ratios=False)):
        whole = ctx.blob_dog(dvol, sigmas, 0.02, 2.6482, **kw)
        want = oracle.blob_dog(vol, sigmas, 0.02, 2.6482, **kw)
        parts = [ctx.blob_dog_slab(dvol[pl.slab[0]:pl.slab[1]].contiguous(), pl.slab[0], shape[0], pl.own_local, sigmas,
                                   0.02, 2.6482, **kw) for pl in plans]
        best = (min(p[2][0] for p in parts), max(p[2][1] for p in parts))
        got = ctx.blob_finalize(_concat_by_scale([p[0] for p in parts], sigmas),
                                _concat_by_scale([p[1] for p in parts], sigmas), best, **kw)
        for k in (0, 1):
            assert np.array_equal(got[k], whole[k]) and np.array_equal(got[k], want[k])
        assert len(got[0]) > 0
    # a slab without the halo is refused, not silently wrong
    pl = plans[1]
    with pytest.raises(vb.VisfdCudaError):
        ctx.blob_dog_slab(dvol[pl.own[0]:pl.own[1]].contiguous(), pl.own[0], shape[0], (0, pl.own[1] - pl.own[0]), sigmas,
                          0.02, 2.6482)


def test_vote_slab_host_delivery(ctx, monkeypatch):
    """visfd_cuda_vote_slab_host: the host copy (chunked D2H behind the kernels when the slab owns
    >= 64 planes, one plain copy otherwise) equals the device result"""
    import torch
    from visfd_b200.slab import make_plan
    for shape, world in (((80, 24, 40), 1), ((60, 24, 40), 2)):
        vol = synth.tomogram(shape, seed=21, n_shells=2)
        sigma, ratio, tv_sigma = 1.5, 2.6482, 4.3
        p = vb.MembraneParams(sigma, ratio, 1, 0.08, 1, tv_sigma, 4, SQ2)
        gauss_hw = int(np.floor(np.float32(sigma) * np.float32(ratio)))
        pl = make_plan(shape[0], world, 0, gauss_hw, vb.tv_halfwidth(tv_sigma, SQ2))
        dvol = torch.from_numpy(vol).cuda()
        sm, sal = ctx.ridge_saliency_slab(dvol[pl.slab[0]:pl.slab[1]].contiguous(), pl.slab[0], shape[0], sigma, ratio)
        thr = float(np.quantile(sal.cpu().numpy(), 0.92))
        host = np.full((pl.own[1] - pl.own[0],) + shape[1:], -1.0, np.float32)
        for waves in ("0", "64"):
            monkeypatch.setenv("VISFD_CUDA_CHUNK_WAVES", waves)
            host[:] = -1.0
            res, _ = ctx.vote_slab(sal, sm, pl.slab[0], shape[0], pl.own_local, pl.vote_local, thr, p, out_host=host)
            assert np.array_equal(host, res.cpu().numpy())
            assert np.count_nonzero(host) > 0


# ---- binning (SURVEY 8f rank 3) ------------------------------------------------------------------------
def test_binning_bit_exact(ctx, oracle, golden):
    """BinArray3D / UnbinArray3D (lib/visfd/resample.hpp:53-166) against the reference's vectors,
    host and device pointers, ragged sizes, shifted windows, and the reference's argument check"""
    import torch
    src = golden["bin_src"]
    assert np.array_equal(ctx.bin3d(src, bin_size=2), golden["bin_2"])
    assert np.array_equal(ctx.bin3d(src, bin_size=3), golden["bin_3"])
    assert np.array_equal(ctx.bin3d(src, dst_shape=(4, 5, 7), offset=(1, 2, 0)), golden["bin_aniso_off"])
    assert np.array_equal(ctx.unbin3d(golden["bin_2"], (13, 17, 22)), golden["unbin_2"])
    assert np.array_equal(ctx.unbin3d(golden["bin_2"], (13, 17, 22), offset=(1, 0, 1)), golden["unbin_2_off"])
    d = ctx.bin3d(torch.from_numpy(src).cuda(), bin_size=2)
    assert d.is_cuda and np.array_equal(d.cpu().numpy(), golden["bin_2"])
    with pytest.raises(vb.VisfdCudaError):
        ctx.bin3d(src, bin_size=2, offset=(2, 0, 0))
    with pytest.raises(vb.VisfdCudaError):
        ctx.bin3d(src, dst_shape=(14, 17, 22))
    rng = np.random.default_rng(5)
    big = rng.standard_normal((70, 131, 259)).astype(np.float32)   # more than one CTA in every direction
    for b in (2, 4, 5):
        got = ctx.bin3d(big, bin_size=b)
        assert np.array_equal(got, oracle.bin3d(big, bin_size=b))
        assert np.array_equal(ctx.unbin3d(got, big.shape), oracle.unbin3d(got, big.shape))


def test_c1_from_the_raw_fixture(ctx, golden):
    """BASELINE config 1 end to end as filter_mrc runs it: -bin 2 (BinArray3D) of the 16^3 fixture,
    then the membrane pipeline; compared with the stock binary's output"""
    binned = ctx.bin3d(golden["c1_in_raw"], bin_size=2)
    assert np.array_equal(binned, golden["c1_in_binned"])
    sigma, ratio, tv_sigma, expo, tv_ratio, frac = [float(v) for v in golden["c1_params"]]
    c1 = ctx.membrane(binned, sigma, ratio, 1, frac, True, tv_sigma, int(expo), tv_ratio)
    assert rel_err(c1["out"], golden["c1_out"]) <= TOL_SALIENCY


def test_draw_regions_bit_exact(ctx, oracle, golden):
    """DrawRegions (lib/visfd/draw.hpp:90-237) against the reference's own outputs, then random region
    lists against the oracle, host and device images alike."""
    import torch
    from util import draw_cases
    for name, (img, mask, regions, subtract) in draw_cases().items():
        got = ctx.draw_regions(img, regions, mask=mask, negative_means_subtract=subtract)
        assert np.array_equal(got, golden["draw_" + name]), name
    rng = np.random.default_rng(6)
    shape = (33, 70, 131)
    for trial in range(12):
        regions = []
        for _ in range(int(rng.integers(1, 9))):
            v = float(rng.choice([-1.0, 1.0, 2.5, 0.0]))
            if rng.random() < 0.5:
                regions.append(("sphere", float(rng.uniform(-5, 140)), float(rng.uniform(-5, 75)),
                                float(rng.uniform(-5, 38)), float(rng.uniform(0, 30)), v))
            else:
                lo = rng.uniform(-6, 100, 3)
                hi = lo + rng.uniform(-1, 60, 3)
                regions.append(("rect", lo[0], hi[0], lo[1], hi[1], lo[2], hi[2], v))
        img = np.zeros(shape, np.float32) if trial % 2 else rng.standard_normal(shape).astype(np.float32)
        mask = None if trial % 3 else (rng.random(shape) > 0.4).astype(np.float32)
        for subtract in (False, True):
            want = oracle.draw_regions(img, regions, mask=mask, negative_means_subtract=subtract)
            assert np.array_equal(ctx.draw_regions(img, regions, mask=mask, negative_means_subtract=subtract), want)
            d = torch.from_numpy(img).cuda()
            dm = None if mask is None else torch.from_numpy(mask).cuda()
            r = ctx.draw_regions(d, regions, mask=dm, negative_means_subtract=subtract)
            assert r.data_ptr() == d.data_ptr() and np.array_equal(d.cpu().numpy(), want)   # in place
    with pytest.raises(vb.VisfdCudaError):
        ctx.draw_regions(img, [("cone", 1, 2, 3)])


def test_draw_regions_properties_large(ctx):
    """at a bench-like size: the voxel count of a sphere painted into zeros equals the lattice count,
    painting is idempotent, and add-then-subtract of the same region leaves nothing"""
    import torch
    shape = (256, 384, 512)
    a = torch.zeros(shape, device="cuda")
    R = 100.3
    ctx.draw_regions(a, [("sphere", 250.0, 190.0, 128.0, R, 1.0)])
    ax = [np.arange(n) for n in shape]
    jz, jy = ax[0][:, None] - 128, ax[1][None, :] - 190
    descr = np.float32(R) * np.float32(R) - (jy * jy + jz * jz).astype(np.float32)
    xr = np.floor(np.sqrt(np.maximum(descr, 0))).astype(np.int64)
    count = np.where(descr >= 0, np.minimum(250 + xr, 511) - np.maximum(250 - xr, 0) + 1, 0)
    count = np.where((np.abs(jz) <= 100) & (np.abs(jy) <= 100), count, 0).sum()
    assert int(a.sum().item()) == int(count)
    b = a.clone()
    ctx.draw_regions(b, [("sphere", 250.0, 190.0, 128.0, R, 1.0)])
    assert torch.equal(a, b)
    ctx.draw_regions(b, [("sphere", 250.0, 190.0, 128.0, R, -1.0)], negative_means_subtract=True)
    assert float(b.abs().max().item()) == 0.0


def test_binning_properties_large(ctx):
    """size-independent properties at a bench-like size: a constant image stays constant, binning
    commutes with a scaling by 2, and un-binning replicates every voxel over its bin"""
    import torch
    g = torch.Generator(device="cuda").manual_seed(3)
    a = torch.randn((256, 512, 512), device="cuda", generator=g)
    c = torch.full_like(a, 1.25)
    assert torch.all(ctx.bin3d(c, bin_size=2) == 1.25)
    b = ctx.bin3d(a, bin_size=2)
    assert b.shape == (128, 256, 256)
    assert torch.equal(ctx.bin3d(a * 2.0, bin_size=2), b * 2.0)
    u = ctx.unbin3d(b, a.shape)
    assert torch.equal(u[::2, ::2, ::2], b) and torch.equal(u[1::2, 1::2, 1::2], b) and torch.equal(u[1::2, ::2, 1::2], b)


def test_reference_blob_fixture_gpu(ctx, golden):
    """the reference's own blob fixture (tests/test_blob_detection.sh:21; 58 scales, masked): the
    11 minima the stock binary finds, position / scale / score bit for bit"""
    mn, _ = ctx.blob_dog(golden["blobfix_img"], golden["blobfix_sigmas"], 0.02, float(golden["blobfix_ratio"]),
                         mask=golden["blobfix_mask"], minima_threshold=0.0, maxima_threshold=-np.inf,
                         use_threshold_ratios=False)
    assert len(mn) == 11
    assert np.array_equal(sort_blobs(mn), sort_blobs(golden["blobfix_minima"]))
