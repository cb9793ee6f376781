"""Blob list post-processing (include/visfd_blobs.h, SURVEY 8f rank 4) against the reference:
SortBlobs / DiscardMaskedBlobs / DiscardOverlappingBlobs on the reference's own blob fixture
(tests/test_blob_detection.sh: 11 minima -> the 2 blobs its test expects) and on a synthetic
list of 600 blobs.  Host code: no GPU needed."""
import numpy as np
import pytest

from visfd_b200 import blobs as vblobs


@pytest.fixture(scope="module")
def lists():
    return vblobs.open_library()


def test_reference_fixture_nms_known_answer(lists, golden):
    """HandleBlobsNonmaxSuppression (bin/filter_mrc/handlers.cpp:428-640) step by step"""
    if "blobnms_in" not in golden.files:
        pytest.skip("blob fixture not generated")
    b = golden["blobnms_in"]
    assert len(b) == 11
    kept = lists.filter(b, score_upper=-90.0)                       # -minima-threshold -90
    kept = lists.discard_masked(kept, golden["blobfix_mask"])
    out = lists.discard_overlapping(kept, 1.1)                      # -blob-separation 1.1
    assert np.array_equal(out, golden["blobnms_out"])
    assert len(out) == 2                                            # what the reference's test asserts
    # the two lines of SURVEY 8c, as the stock binary printed them (physical units, -w 19.6)
    phys = out.astype(np.float64) * np.array([19.6, 19.6, 19.6, 19.6, 1.0], np.float32)
    assert np.allclose(phys, golden["blobnms_cli"], rtol=2e-5)
    for want in ((235.2, 392.0, 313.6, 177.915, -140.018), (254.8, 98.0, 274.4, 177.915, -109.148)):
        assert np.any(np.all(np.isclose(phys, want, rtol=1e-5), axis=1)), want


def test_list_functions_match_reference(lists, golden):
    big = golden["bloblist_in"]
    assert np.array_equal(lists.sort(big, vblobs.SORT_DECREASING_MAGNITUDE, False), golden["bloblist_sorted_mag"])
    assert np.array_equal(lists.sort(big, vblobs.SORT_INCREASING, True), golden["bloblist_sorted_inc"])
    assert np.array_equal(lists.discard_overlapping(big, 1.0), golden["bloblist_nms_sep"])
    assert np.array_equal(lists.discard_overlapping(big, 0.0, 0.3, 0.6), golden["bloblist_nms_vol"])
    assert np.array_equal(lists.discard_overlapping(big, 0.8, np.inf, np.inf, vblobs.SORT_INCREASING),
                          golden["bloblist_nms_inc"])
    assert np.array_equal(lists.sort(big, vblobs.DO_NOT_SORT), big)
    # empty lists, bad criteria
    assert lists.discard_overlapping(np.zeros((0, 5), np.float32), 1.0).shape == (0, 5)
    with pytest.raises(ValueError):
        lists.sort(big, 9)


def test_nms_properties(lists):
    """idempotence and priority order; surviving pairs respect the separation rule except near the
    upper faces of the bounding box, where the reference's occupancy table (size = extent / 6,
    truncated; lib/visfd/feature.hpp:773-774) has no cell and the search skips them"""
    g = np.random.default_rng(5)
    n = 3000
    b = np.stack([g.uniform(0, 300, n), g.uniform(0, 300, n), g.uniform(0, 120, n), g.uniform(6, 24, n),
                  -np.abs(g.standard_normal(n)) * 30], axis=1).astype(np.float32)
    out = lists.discard_overlapping(b, 1.0)
    assert 0 < len(out) < n
    again = lists.discard_overlapping(out, 1.0)       # (tied scores swap places: sort(rbegin, rend) of (score, index))
    assert np.array_equal(again[np.lexsort(again.T)], out[np.lexsort(out.T)])
    assert np.all(np.diff(np.abs(out[:, 4])) <= 0)                   # priority order: decreasing |score|
    inner = out[np.all(out[:, :3] + out[:, 3:4] < np.array([300, 300, 120]) - 12, axis=1)]
    d = np.linalg.norm(inner[:, None, :3].astype(np.float64) - inner[None, :, :3], axis=2)
    rsum = (inner[:, None, 3] + inner[None, :, 3]) / 2.0
    np.fill_diagonal(d, np.inf)
    assert len(inner) > 100 and np.all(d >= rsum * (1 - 1e-6))


# DiscardOverlappingBlobs arguments of live_cases: separation, large and small overlap ratios, sort criterion
LIVE_OVERLAP_ARGS = ((1.0, np.inf, np.inf, 3), (0.5, 0.2, 0.9, 3), (0.0, 0.5, 0.5, 1), (1.3, np.inf, np.inf, 4))


def live_cases():
    """random lists of 1, 7 and 400 blobs -> (n, blobs, blobs clipped to a 150 x 150 x 60 image, a random mask)"""
    g = np.random.default_rng(11)
    for n in (1, 7, 400):
        b = np.stack([g.uniform(0, 150, n), g.uniform(0, 150, n), g.uniform(0, 60, n), g.uniform(3, 40, n),
                      g.standard_normal(n) * 10], axis=1).astype(np.float32)
        mask = (g.uniform(size=(60, 150, 150)) > 0.3).astype(np.float32)
        bb = b.copy()
        bb[:, :3] = np.clip(bb[:, :3], 0, [149, 149, 59])
        yield n, b, bb, mask


def test_live_against_reference_build(lists, golden):
    """live_cases through DiscardOverlappingBlobs and DiscardMaskedBlobs: the blobs the reference kept, in its order
    (stored as row numbers of the input; tests/golden/README.md)"""
    for n, b, bb, mask in live_cases():
        for k, (sep, large, small, crit) in enumerate(LIVE_OVERLAP_ARGS):
            want = b[golden["live_blobs_%d_overlap%d" % (n, k)]]
            assert np.array_equal(lists.discard_overlapping(b, sep, large, small, crit), want), (n, sep, large, small, crit)
        assert np.array_equal(lists.discard_masked(bb, mask), bb[golden["live_blobs_%d_masked" % n]])
