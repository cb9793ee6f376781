"""Pins the CPU oracle (oracle/visfd_oracle.cpp, our restatement) to the reference:
against tests/golden/reference_vectors.npz (outputs of the unmodified reference, see
tests/golden/make_golden.py) everywhere, and against oracle/_ref itself where it has
been built.  Same compiler + libm => the restatement is expected to be BIT-identical.
"""
import numpy as np
import pytest

from util import sort_blobs

SQ2 = float(np.float32(np.sqrt(2.0)))


def eq(a, b):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape
    assert np.array_equal(a, b), f"max |diff| = {np.abs(a.astype(np.float64) - b).max()}"


def test_taps(oracle, golden):
    for k, (s, hw) in enumerate(golden["taps_cases"]):
        eq(oracle.gen_gauss1d(float(s), int(hw)), golden[f"taps_{k}"])
    # SURVEY.md 8c bootstrap value: GenFilterGauss1D(2.0, 5)
    t = oracle.gen_gauss1d(2.0, 5)
    np.testing.assert_allclose(t[:6], [0.00931539, 0.0261393, 0.0615941, 0.11853, 0.180124, 0.208593], rtol=1e-5)
    assert abs(t.sum() - 1.0) < 1e-6 and np.array_equal(t, t[::-1])


def test_separable(oracle, golden):
    vol, mask = golden["vol"], golden["mask"]
    d, A = oracle.apply_gauss(vol, 1.3, 3)
    eq(d, golden["gauss_s1.3_hw3"])
    assert np.float32(A) == golden["gauss_A"]
    eq(oracle.apply_gauss(vol, 1.3, 3, normalize=False)[0], golden["gauss_s1.3_hw3_nonorm"])
    eq(oracle.apply_gauss(vol, (1.0, 2.0, 0.7), (2, 5, 1))[0], golden["gauss_aniso"])
    eq(oracle.apply_gauss(vol, 1.3, 3, mask=mask)[0], golden["gauss_masked"])
    eq(oracle.apply_gauss(vol, 1.3, 3, mask=mask, normalize=False)[0], golden["gauss_masked_nonorm"])
    eq(oracle.apply_gauss(vol, 4.0, 10)[0], golden["gauss_wide"])
    d, a, b = oracle.apply_dog(vol, 1.2, 1.92, 5)
    eq(d, golden["dog"])
    eq(np.array([a, b], np.float32), golden["dog_AB"])
    d, a, b = oracle.apply_log(vol, 1.5, 0.02, 2.6482)
    eq(d, golden["log"])
    eq(np.array([a, b], np.float32), golden["log_AB"])
    eq(oracle.apply_log(vol, 1.5, 0.02, 2.6482, mask=mask)[0], golden["log_masked"])


def test_hessian_eigen_cut(oracle, golden):
    vol, mask = golden["vol"], golden["mask"]
    g, h = oracle.calc_hessian(vol, 1.1, 2.6482)
    eq(g, golden["hess_grad"])
    eq(h, golden["hess_hess"])
    g, h2 = oracle.calc_hessian(vol, 1.1, 2.6482, mask=mask)
    eq(g, golden["hess_grad_masked"])
    eq(h2, golden["hess_hess_masked"])
    for order in (0, 1):
        sal, dire, ev = oracle.hessian_eigen_score(h, order=order, score_kind=0)
        eq(sal, golden[f"ridge_sal_o{order}"])
        eq(dire, golden[f"ridge_dir_o{order}"])
        eq(ev, golden[f"ridge_ev_o{order}"])
    eq(oracle.hessian_eigen_score(h, order=1, score_kind=1)[0], golden["ridge_sal_linear"])
    cut, thr = oracle.saliency_cut(golden["ridge_sal_o1"], 0.1, True)
    eq(cut, golden["cut_frac0.1"])
    assert np.float32(thr) == golden["cut_frac0.1_thr"]
    cut, thr = oracle.saliency_cut(golden["ridge_sal_o1"], 0.25, True, mask=mask)
    eq(cut, golden["cut_frac0.25_masked"])
    assert np.float32(thr) == golden["cut_frac0.25_masked_thr"]
    with pytest.raises(ValueError):
        oracle.calc_hessian(np.zeros((2, 5, 5), np.float32), 1.0, 2.5)


def test_tensor_voting(oracle, golden):
    hw, decay, disp = oracle.tv_tables(2.4, np.sqrt(2.0))
    assert hw == int(golden["tv_tables_hw"])
    eq(decay, golden["tv_decay"])
    eq(disp, golden["tv_disp"])
    tvol = golden["tv_vol"]
    m = oracle.membrane(tvol, 1.0, 2.6482, 1, 0.12, True, 2.4, 4, SQ2)
    for k in ("hess_saliency", "direction", "tensor", "out"):
        eq(m[k], golden["mem_" + k])
    assert np.float32(m["threshold"]) == golden["mem_thr"]
    sal, dire = golden["mem_hess_saliency"], golden["mem_direction"]
    eq(oracle.tv_dense_stick(sal, dire, 2.4, 2, SQ2), golden["tv_e2"])
    eq(oracle.tv_dense_stick(sal, dire, 2.4, 3, SQ2), golden["tv_e3"])
    eq(oracle.tv_dense_stick(sal, dire, 2.4, 4, SQ2, curves=True), golden["tv_e4_curves"])
    tm = golden["tv_mask"]
    eq(oracle.tv_dense_stick(sal, dire, 2.4, 4, SQ2, mask_src=tm, mask_dst=tm), golden["tv_e4_masked"])
    eq(oracle.tensor_score(golden["mem_tensor"], order=1, score_kind=0), golden["tv_score_planar"])
    mm = oracle.membrane(tvol, 1.0, 2.6482, 1, 0.12, True, 2.4, 4, SQ2, mask=tm)
    eq(mm["out"], golden["mem_masked_out"])
    mx = oracle.membrane(-tvol, 1.0, 2.6482, 0, 0.12, True, 2.4, 4, SQ2)
    eq(mx["out"], golden["mem_maxima_out"])


def test_thresholds(oracle, golden):
    x = golden["thr_x"]
    eq(oracle.threshold1(x, 0.5, 0.0, 1.0), golden["thr1"])
    eq(oracle.threshold2(x, 0.2, 1.4, 0.0, 1.0), golden["thr2_up"])
    eq(oracle.threshold2(x, 1.4, 0.2, -1.0, 2.0), golden["thr2_down"])
    eq(oracle.threshold4(x, -1.0, -0.5, 1.5, 2.0, 0.0, 1.0), golden["thr4"])
    eq(oracle.threshold4(x, 2.0, 1.5, -0.5, -1.0, 0.0, 1.0), golden["thr4_rev"])
    vol, mask = golden["vol"], golden["mask"]
    ms = np.array([oracle.average(vol), oracle.stddev(vol), oracle.average(vol, mask), oracle.stddev(vol, mask)],
                  np.float32)
    eq(ms, golden["mean_std"])


def test_blobs(oracle, golden):
    bvol, sig = golden["blob_vol"], golden["blob_sigmas"]
    mn, mx = oracle.blob_dog(bvol, sig, 0.02, 2.6482, minima_threshold=0.0, maxima_threshold=-np.inf,
                             use_threshold_ratios=False)
    eq(sort_blobs(mn), sort_blobs(golden["blob_minima"]))
    eq(sort_blobs(mx), sort_blobs(golden["blob_maxima"]))
    assert len(mn) > 0
    mn, mx = oracle.blob_dog(bvol, sig, 0.02, 2.6482, minima_threshold=0.5, maxima_threshold=0.5,
                             use_threshold_ratios=True)
    eq(sort_blobs(mn), sort_blobs(golden["blob_minima_ratio"]))
    eq(sort_blobs(mx), sort_blobs(golden["blob_maxima_ratio"]))


def test_c1_reference_fixture(oracle, golden):
    """BASELINE config 1: tests/test_membrane_detection.sh on test_image_membrane.rec, as run
    by the stock filter_mrc binary (SURVEY.md 8c known answers)."""
    if "c1_out" not in golden.files:
        pytest.skip("C1 fixture not generated")
    sigma, ratio, tv_sigma, expo, tv_ratio, frac = [float(v) for v in golden["c1_params"]]
    m = oracle.membrane(golden["c1_in_binned"], sigma, ratio, 1, frac, True, tv_sigma, int(expo), tv_ratio)
    eq(m["out"], golden["c1_out"])
    c1 = golden["c1_out"]
    assert abs(c1.sum(dtype=np.float64) / 4.141152e11 - 1) < 1e-6
    assert abs(c1.max() / 6.827661e9 - 1) < 1e-6 and np.unravel_index(c1.argmax(), c1.shape) == (2, 3, 2)
    assert (c1 != 0).sum() == 419
    m0 = oracle.membrane(golden["c1_in_binned"], sigma, ratio, 1, frac, True, 0.0, int(expo), tv_ratio)
    eq(m0["out"], golden["c1_out_notv"])
    assert (m0["out"] != 0).sum() == 27


def port_live_outputs(o):
    """Every stage of the path on a seeded 15 x 18 x 21 tomogram with a random mask, through checker `o`:
    name -> array"""
    from visfd_b200 import synth
    vol = synth.tomogram((15, 18, 21), seed=11)
    rng = np.random.default_rng(2)
    mask = (rng.random(vol.shape) > 0.2).astype(np.float32)
    out = {}
    for name, kw in (("gauss", dict()), ("gauss_masked", dict(mask=mask)), ("gauss_nonorm", dict(normalize=False))):
        out[name] = o.apply_gauss(vol, 1.7, 4, **kw)[0]
    out["log"] = o.apply_log(vol, 2.0, 0.02, 2.6482)[0]
    m = o.membrane(vol, 1.2, 2.6482, 1, 0.1, True, 3.0, 4, SQ2, mask=mask)
    for k in ("hess_saliency", "direction", "tensor", "out"):
        out["membrane_" + k] = m[k]
    out["membrane_threshold"] = np.float32(m["threshold"])
    return out


def test_port_matches_reference_live(oracle, golden):
    """Fresh seeded inputs, every stage, bit for bit: against the reference's outputs stored in
    tests/golden/reference_vectors_live.npz (tests/golden/README.md), and against oracle/_ref itself where it
    has been built."""
    from oracle.pyoracle import Oracle, have
    got = port_live_outputs(oracle)
    for k, v in got.items():
        eq(v, golden["live_port_" + k])
    if have("reference"):
        for k, v in port_live_outputs(Oracle("reference")).items():
            eq(got[k], v)


def test_binning_matches_reference(golden, oracle):
    """BinArray3D / UnbinArray3D (lib/visfd/resample.hpp:53-166): the restatement is bit-identical"""
    src = golden["bin_src"]
    assert np.array_equal(oracle.bin3d(src, bin_size=2), golden["bin_2"])
    assert np.array_equal(oracle.bin3d(src, bin_size=3), golden["bin_3"])
    assert np.array_equal(oracle.bin3d(src, dst_shape=(4, 5, 7), offset=(1, 2, 0)), golden["bin_aniso_off"])
    assert np.array_equal(oracle.unbin3d(golden["bin_2"], (13, 17, 22)), golden["unbin_2"])
    assert np.array_equal(oracle.unbin3d(golden["bin_2"], (13, 17, 22), offset=(1, 0, 1)), golden["unbin_2_off"])
    assert np.array_equal(oracle.bin3d(golden["c1_in_raw"], bin_size=2), golden["c1_in_binned"])
    with pytest.raises(ValueError):
        oracle.bin3d(src, bin_size=2, offset=(2, 0, 0))


def test_reference_blob_fixture(oracle, golden):
    """the reference's own blob test (tests/test_blob_detection.sh:21): 58 scales, 11 minima
    (SURVEY.md 8c), list produced by the stock filter_mrc binary"""
    if "blobfix_minima" not in golden.files:
        pytest.skip("blob fixture not generated")
    mn, _ = oracle.blob_dog(golden["blobfix_img"], golden["blobfix_sigmas"], 0.02, float(golden["blobfix_ratio"]),
                            mask=golden["blobfix_mask"], minima_threshold=0.0, maxima_threshold=-np.inf,
                            use_threshold_ratios=False)
    assert len(golden["blobfix_sigmas"]) == 58 and len(mn) == 11
    eq(sort_blobs(mn), sort_blobs(golden["blobfix_minima"]))
    # ... and the two blobs the reference's test expects after non-max suppression are among them
    # (known answers of SURVEY 8c: `235.2 392 313.6 177.915 -140.018`, `254.8 98 274.4 177.915 -109.148`)
    cli = golden["blobfix_cli"]
    for want in ((235.2, 392.0, 313.6, 177.915, -140.018), (254.8, 98.0, 274.4, 177.915, -109.148)):
        assert np.any(np.all(np.isclose(cli, want, rtol=1e-5), axis=1)), want


def test_draw_regions(oracle, golden):
    """DrawRegions (lib/visfd/draw.hpp:90-237): painting order, subtraction, the all-zero special case,
    masks, fractional centres and radii, boxes clipped by the image."""
    from util import draw_cases
    for name, (img, mask, regions, subtract) in draw_cases().items():
        eq(oracle.draw_regions(img, regions, mask=mask, negative_means_subtract=subtract), golden["draw_" + name])
    # the fixture exercises what it claims to
    g = golden["draw_add_sub"]
    assert set(np.unique(g)) == {0.0, 0.5, 1.0, 2.0, 3.0}
    assert golden["draw_from_ones"].min() == 0.0 and golden["draw_from_ones"][0, 23, 27] == 1.0
    assert np.array_equal(golden["draw_empty"], draw_cases()["empty"][0])


def random_draw_cases():
    """20 random sets of 1 to 6 spheres and boxes, half of them on a zero image, a third of them masked
    -> (trial, image, mask, regions)"""
    rng = np.random.default_rng(5)
    shape = (17, 19, 23)
    for trial in range(20):
        regions = []
        for _ in range(int(rng.integers(1, 7))):
            v = float(rng.choice([-1.0, 1.0, 2.5, 0.0]))
            if rng.random() < 0.5:
                regions.append(("sphere", *rng.uniform(-3, 25, 3).tolist(), float(rng.uniform(0, 9)), v))
            else:
                lo = rng.uniform(-4, 20, 3)
                hi = lo + rng.uniform(-1, 12, 3)
                regions.append(("rect", lo[0], hi[0], lo[1], hi[1], lo[2], hi[2], v))
        img = np.zeros(shape, np.float32) if trial % 2 else rng.standard_normal(shape).astype(np.float32)
        mask = None if trial % 3 else (rng.random(shape) > 0.4).astype(np.float32)
        yield trial, img, mask, regions


def test_draw_regions_vs_reference(oracle, golden):
    """random_draw_cases: the reference's images, stored as the voxels it changed, NaN elsewhere
    (tests/golden/reference_vectors_live.npz, tests/golden/README.md)"""
    for trial, img, mask, regions in random_draw_cases():
        for subtract in (False, True):
            changed = golden["live_draw_%d_%d" % (trial, subtract)]
            eq(oracle.draw_regions(img, regions, mask=mask, negative_means_subtract=subtract),
               np.where(np.isnan(changed), img, changed))


def test_c1_pass2_known_answer(golden):
    """tests/test_membrane_detection.sh pass 2 (-connect 1e+09 -connect-angle 30 -select-cluster 1), run by
    the stock binary when the fixtures were made: 1 cluster of 69 voxels (SURVEY 8c), all of them above the
    saliency threshold of the post-vote image.  This pins the known answer of SURVEY 8f rank 1
    (LabelConnected), which round 1 has not built; nothing in the product is compared here."""
    labels, sal = golden["c1_connect_labels"], golden["c1_out"]
    assert golden["c1_connect_n_clusters"].tolist() == [1]
    assert labels.shape == sal.shape == (8, 8, 8)
    assert int((labels == 1).sum()) == 69
    assert np.all(sal[labels == 1] >= 1e9)


def test_label_connected_hook_reproduces_the_cli(ref_oracle, golden):
    """oracle/ref_shim.cpp::ref_label_connected (the unmodified LabelConnected behind the arguments HandleTV
    passes) on the C1 pipeline output == the stock binary's pass 2: test infrastructure for SURVEY 8f rank 1."""
    sigma, ratio, tv_sigma, expo, cutoff, best = [float(v) for v in golden["c1_params"]]
    r = ref_oracle.membrane(golden["c1_in_binned"], sigma, ratio, 1, best, True, tv_sigma, int(expo), cutoff)
    assert np.array_equal(r["out"], golden["c1_out"])
    labels, n = ref_oracle.label_connected(r["out"], r["tensor"], 1e9, angle_deg=30.0)
    assert n == int(golden["c1_connect_n_clusters"][0]) == 1
    cli = golden["c1_connect_labels"]
    assert np.array_equal(labels == 1, cli == 1) and int((labels == 1).sum()) == 69
    assert np.array_equal(labels == -1, cli == 2)          # undefined voxels: max label + 1 in the file


def _random_connect_case(oracle, seed, shape=(18, 20, 22)):
    rng = np.random.default_rng(500 + seed)
    smooth = lambda a: oracle.apply_gauss(a.astype(np.float32), 1.5, 4)[0]
    sal = smooth(rng.standard_normal(shape))
    sal = (sal - sal.min()).astype(np.float32)
    if seed % 3 == 2:                       # plateaus
        sal = np.round(sal / sal.max() * 10.0).astype(np.float32)
    n = np.stack([smooth(rng.standard_normal(shape)) for _ in range(3)], axis=-1)
    n /= np.linalg.norm(n, axis=-1, keepdims=True) + 1e-12
    T = np.stack([n[..., 0] ** 2, n[..., 1] ** 2, n[..., 2] ** 2, n[..., 0] * n[..., 1], n[..., 1] * n[..., 2],
                  n[..., 0] * n[..., 2]], axis=-1) * rng.uniform(0.5, 2.0, shape)[..., None]
    T[..., :3] += 0.05 + 0.02 * rng.standard_normal(shape + (3,))
    mask = (rng.random(shape) > 0.15).astype(np.float32) if seed % 2 else None
    return sal, T.astype(np.float32), mask, float(np.quantile(sal, 0.6))


def restatement_connect_calls(o, golden):
    """The LabelConnected calls of test_label_connected_restatement_is_the_reference: (name, args, kwargs) for the C1
    pipeline output of checker `o`, random fields with masks, plateaus, rejected seeds and merges, and one field
    with the direction thresholds disabled"""
    sigma, ratio, tv_sigma, expo, cutoff, best = [float(v) for v in golden["c1_params"]]
    r = o.membrane(golden["c1_in_binned"], sigma, ratio, 1, best, True, tv_sigma, int(expo), cutoff)
    yield "c1", (r["out"], r["tensor"], 1e9), dict(angle_deg=30.0, want_direction=True)
    for seed in range(6):
        sal, T, mask, thr = _random_connect_case(o, seed)
        for angle in (25.0, 60.0):
            yield "random_%d_%g" % (seed, angle), (sal, T, thr), dict(angle_deg=angle, mask=mask, want_direction=True)
    sal, T, mask, thr = _random_connect_case(o, 2)
    yield "thresholds_disabled", (sal, T, 6.0), dict(thresholds=(-np.inf,) * 4)


def test_label_connected_restatement_is_the_reference(oracle, golden):
    """oracle/visfd_oracle.cpp::vo_label_connected == the unmodified LabelConnected (lib/visfd/connect.hpp:171) behind
    HandleTV's arguments, label for label and direction for direction (bit-identical: same compiler, same libm), on
    restatement_connect_calls: against the reference's labels, stored directions of the clustered voxels and a SHA-256
    of the whole direction field (tests/golden/reference_vectors_live.npz, tests/golden/README.md), and against
    oracle/_ref itself where it has been built."""
    from oracle.pyoracle import Oracle, have
    from util import sha256_of
    ref = Oracle("reference") if have("reference") else None
    total = 0
    for name, args, kw in restatement_connect_calls(oracle, golden):
        key = "live_connect_%s_" % name
        a = oracle.label_connected(*args, **kw)
        assert a[1] == int(golden[key + "n_clusters"]), name
        assert np.array_equal(a[0], golden[key + "labels"]), name
        if kw.get("want_direction"):
            eq(a[2][a[0] >= 1], golden[key + "direction_inside"])
            assert sha256_of(a[2]) == str(golden[key + "direction_sha256"]), name
        if ref is not None:
            b = ref.label_connected(*args, **kw)
            assert a[1] == b[1] and np.array_equal(a[0], b[0]), name
            if kw.get("want_direction"):
                assert np.array_equal(a[2], b[2]), name
        total += a[1] if name.startswith("random") else 0
    assert int(golden["live_connect_c1_n_clusters"]) == 1
    assert total > 20 and int(golden["live_connect_thresholds_disabled_n_clusters"]) > 1


def test_label_connected_restatement_c1_known_answer(oracle, golden):
    """Without the reference tree: the restatement on the C1 pipeline (restated too) gives the stock binary's pass 2."""
    sigma, ratio, tv_sigma, expo, cutoff, best = [float(v) for v in golden["c1_params"]]
    r = oracle.membrane(golden["c1_in_binned"], sigma, ratio, 1, best, True, tv_sigma, int(expo), cutoff)
    labels, n = oracle.label_connected(r["out"], r["tensor"], 1e9, angle_deg=30.0)
    cli = golden["c1_connect_labels"]
    assert n == 1 and np.array_equal(labels == 1, cli == 1) and np.array_equal(labels == -1, cli == 2)
