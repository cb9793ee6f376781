"""LabelConnected on the GPU path (visfd_cuda_label_connected: device predicates + ordered host flood) against the
UNMODIFIED reference (lib/visfd/connect.hpp:171 behind the arguments HandleTV passes,
bin/filter_mrc/handlers.cpp:1963-1993): its labels and directions for the inputs built here are stored in
tests/golden/connect_labels.npz (tests/golden/README.md).  Labels are compared exactly, voxel for voxel:
cluster numbering included."""
import os

import numpy as np
import pytest

import visfd_b200
from visfd_b200 import synth
from util import sha256_of

pytestmark = pytest.mark.gpu
SQ2 = float(np.float32(np.sqrt(2.0)))
MEMBRANE_CASES = [(0, (40, 44, 48), 30.0, 0.90), (1, (32, 32, 32), 15.0, 0.85), (2, (48, 40, 36), 45.0, 0.95),
                  (3, (36, 36, 60), 20.0, 0.80)]
RANDOM_FIELD_ANGLES = (25.0, 60.0)
PLATEAU_THRESHOLD = 7.0


@pytest.fixture(scope="module")
def want():
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "connect_labels.npz"))


def test_c1_pass2_through_the_gpu_path(ctx, golden):
    """BASELINE config 1, pass 2 (tests/test_membrane_detection.sh:9): -connect 1e+09 -connect-angle 30 on the output
    of pass 1 -> the stock binary's label image: 1 cluster of 69 voxels, everything else undefined."""
    sigma, ratio, tv_sigma, expo, cutoff, best = [float(v) for v in golden["c1_params"]]
    r = ctx.membrane(golden["c1_in_binned"], sigma, ratio, 1, best, True, tv_sigma, int(expo), cutoff, want_tensor=True)
    res = ctx.label_connected(np.asarray(r["out"]), np.asarray(r["tensor"]), 1e9, angle_deg=30.0)
    cli = golden["c1_connect_labels"]
    assert res["n_clusters"] == int(golden["c1_connect_n_clusters"][0]) == 1
    assert np.array_equal(res["labels"] == 1, cli == 1) and int((res["labels"] == 1).sum()) == 69
    assert np.array_equal(res["labels"] == -1, cli == 2)      # undefined voxels: max label + 1 in the file


def membrane_case(oracle, seed, shape, quant):
    """Synthetic tomogram (noise + dark shells) -> membrane pipeline of the CPU restatement (so that the stored labels
    do not hang on the rounding of the GPU's votes) -> (saliency, tensor, threshold)"""
    vol = synth.tomogram(shape, seed=seed, n_shells=2)
    ratio = float(np.float32(np.sqrt(np.float32(-2) * np.log(np.float32(0.03)))))
    r = oracle.membrane(vol, 1.2, ratio, visfd_b200.DECREASING_EIVALS, 0.1, True, 4.0, 4, SQ2)
    out, tensor = r["out"], r["tensor"]
    thr = float(np.quantile(out[out > 0], quant)) if np.any(out > 0) else 1.0
    return out, tensor, thr


def _check_inputs(want, key, *arrays):
    assert sha256_of(*arrays) == str(want[key + "inputs_sha256"]), \
        "the inputs are not those the stored labels were made from: regenerate with tests/golden/make_connect_golden.py"


@pytest.mark.parametrize("seed,shape,angle,quant", MEMBRANE_CASES)
def test_membrane_output_clusters_like_the_reference(ctx, oracle, want, seed, shape, angle, quant):
    """Synthetic tomogram (noise + dark shells) -> membrane pipeline -> LabelConnected, against the reference fed
    the SAME saliency and tensor arrays: identical label images (numbering by size included) and standardised
    directions."""
    out, tensor, thr = membrane_case(oracle, seed, shape, quant)
    key = "membrane_%d_" % seed
    _check_inputs(want, key, out, tensor, np.float32(thr))
    labels_want, n_want = want[key + "labels"], int(want[key + "n_clusters"])
    res = ctx.label_connected(out, tensor, thr, angle_deg=angle, want_direction=True)
    assert n_want > 0, "test volume yields no cluster: pick other parameters"
    assert res["n_clusters"] == n_want
    assert np.array_equal(res["labels"], labels_want)
    inside = labels_want >= 1
    dots = np.sum(res["direction"][inside] * want[key + "direction_inside"], axis=-1)
    assert np.all(np.abs(dots) > 0.999), "standardised directions differ in value"
    # the sign is fixed by the flood and the centre-of-mass rule -- except in a cluster of ONE voxel, where that rule
    # sees a zero sum (connect.hpp:1270-1284) and the eigenvector keeps the arbitrary sign of its solver
    sizes = np.bincount(labels_want[inside])
    big = sizes[labels_want[inside]] >= 2
    assert np.all(dots[big] > 0.999), "standardised directions differ in sign"


def random_field_case(oracle, seed):
    """Smooth random saliency, tensors built from a smooth random direction field plus noise, random mask on odd
    seeds -> (saliency, tensor, mask, threshold)"""
    rng = np.random.default_rng(100 + seed)
    shape = (28, 30, 34)
    smooth = lambda a: oracle.apply_gauss(a.astype(np.float32), 1.5, 4)[0]
    sal = smooth(rng.standard_normal(shape))
    sal = (sal - sal.min()).astype(np.float32)
    n = np.stack([smooth(rng.standard_normal(shape)) for _ in range(3)], axis=-1)
    n /= np.linalg.norm(n, axis=-1, keepdims=True) + 1e-12
    lam = rng.uniform(0.5, 2.0, shape)[..., None]
    # T = lam * n n^T + small isotropic part + noise on the diagonal (flat order xx,yy,zz,xy,yz,xz)
    T = np.stack([n[..., 0] ** 2, n[..., 1] ** 2, n[..., 2] ** 2, n[..., 0] * n[..., 1], n[..., 1] * n[..., 2],
                  n[..., 0] * n[..., 2]], axis=-1) * lam
    T[..., :3] += 0.05 + 0.02 * rng.standard_normal(shape + (3,))
    T = T.astype(np.float32)
    mask = (rng.random(shape) > 0.15).astype(np.float32) if seed % 2 else None
    return sal, T, mask, float(np.quantile(sal, 0.6))


@pytest.mark.parametrize("seed", range(6))
def test_random_fields_cluster_like_the_reference(ctx, oracle, want, seed):
    """random_field_case: many small clusters, rejected voxels, rejected seeds and merges.  Exact label equality."""
    sal, T, mask, thr = random_field_case(oracle, seed)
    _check_inputs(want, "random_%d_" % seed, sal, T, mask, np.float32(thr))
    for angle in RANDOM_FIELD_ANGLES:
        key = "random_%d_%g_" % (seed, angle)
        labels_want, n_want = want[key + "labels"], int(want[key + "n_clusters"])
        res = ctx.label_connected(sal, T, thr, angle_deg=angle, mask=mask)
        assert res["n_clusters"] == n_want
        if mask is not None:   # voxels outside the mask keep the reference's internal marker
            assert np.array_equal(res["labels"][mask == 0], labels_want[mask == 0])
        assert np.array_equal(res["labels"], labels_want)


def plateau_case(oracle):
    """Quantised smooth noise as saliency, random tensors -> (saliency, tensor)"""
    rng = np.random.default_rng(7)
    shape = (20, 24, 26)
    sal = oracle.apply_gauss(rng.standard_normal(shape).astype(np.float32), 2.0, 5)[0]
    sal = np.round((sal - sal.min()) / (sal.max() - sal.min()) * 12.0).astype(np.float32)
    return sal, rng.standard_normal(shape + (6,)).astype(np.float32)


def test_plateaus_and_thresholds_disabled(ctx, oracle, want):
    """Quantised saliency (plateaus of equal values, among them maxima) and all four direction thresholds disabled
    (-inf, as settings.cpp:3645-3646 does for two of them): plain thresholded connected components from plateau
    seeds, numbering by size with ties."""
    sal, T = plateau_case(oracle)
    _check_inputs(want, "plateau_", sal, T)
    ninf = -np.inf
    labels_want, n_want = want["plateau_labels"], int(want["plateau_n_clusters"])
    res = ctx.label_connected(sal, T, PLATEAU_THRESHOLD, thresholds=(ninf, ninf, ninf, ninf))
    assert n_want > 1
    assert res["n_clusters"] == n_want and np.array_equal(res["labels"], labels_want)


def test_device_resident_inputs(ctx, golden):
    import torch
    sigma, ratio, tv_sigma, expo, cutoff, best = [float(v) for v in golden["c1_params"]]
    r = ctx.membrane(golden["c1_in_binned"], sigma, ratio, 1, best, True, tv_sigma, int(expo), cutoff, want_tensor=True)
    host = ctx.label_connected(np.asarray(r["out"]), np.asarray(r["tensor"]), 1e9, angle_deg=30.0, want_direction=True)
    dev = ctx.label_connected(torch.from_numpy(np.asarray(r["out"])).cuda(), torch.from_numpy(np.asarray(r["tensor"])).cuda(),
                              1e9, angle_deg=30.0, want_direction=True)
    assert np.array_equal(host["labels"], dev["labels"])
    assert np.array_equal(host["direction"], dev["direction"].cpu().numpy())
