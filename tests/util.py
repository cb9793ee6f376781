"""Parity metrics shared by the tests (tolerances from BASELINE.json:north_star)."""
import hashlib

import numpy as np

TOL_GAUSS = 1e-5      # Gaussian / DoG / LoG outputs
TOL_SALIENCY = 1e-4   # ridge saliency, vote tensors, post-vote score


def rel_err(a, b, floor_frac=1e-3):
    """max |a-b| / max(|b|, floor) with floor = floor_frac * max|b| over the volume.

    A per-voxel relative error with a floor: voxels whose reference value is a
    cancellation residue (e.g. a Gaussian-blurred noise value near a zero crossing, or
    lambda1^2 ~ lambda2^2) are judged against the scale of the volume instead of
    their own ~0 magnitude."""
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    scale = np.abs(b).max() if b.size else 0.0
    if scale == 0.0:
        return float(np.abs(a).max()) if a.size else 0.0
    den = np.maximum(np.abs(b), floor_frac * scale)
    return float((np.abs(a - b) / den).max())


def tensor_rel_err(a, b):
    """Per-voxel Frobenius error of 6-component tensors relative to the tensor norm
    (off-diagonal components cancel, so they are judged against the whole tensor)."""
    a = np.asarray(a, np.float64).reshape(-1, 6)
    b = np.asarray(b, np.float64).reshape(-1, 6)
    w = np.array([1, 1, 1, 2, 2, 2], np.float64)
    nb = np.sqrt((b * b * w).sum(1))
    d = np.sqrt(((a - b) ** 2 * w).sum(1))
    scale = nb.max() if nb.size else 0.0
    if scale == 0.0:
        return float(d.max()) if d.size else 0.0
    return float((d / np.maximum(nb, 1e-3 * scale)).max())


def direction_err(a, b, weight=None):
    """max over voxels of 1 - |cos| between unit vectors (normals are sign-free)."""
    a = np.asarray(a, np.float64).reshape(-1, 3)
    b = np.asarray(b, np.float64).reshape(-1, 3)
    c = np.abs((a * b).sum(1)) / np.maximum(np.linalg.norm(a, axis=1) * np.linalg.norm(b, axis=1), 1e-30)
    e = 1.0 - c
    if weight is not None:
        e = e[np.asarray(weight).reshape(-1) != 0]
    return float(e.max()) if e.size else 0.0


def sort_blobs(t):
    """canonical order: (sigma, z, y, x)"""
    t = np.asarray(t)
    if len(t) == 0:
        return t.reshape(0, 5)
    idx = np.lexsort((t[:, 0], t[:, 1], t[:, 2], t[:, 3]))
    return t[idx]


def vote_score_err(a, b, tensor_ref):
    """Error of the post-vote score lambda1 - lambda2 (ScoreTensorPlanar).  The score is a
    DIFFERENCE of eigenvalues of a float32-accumulated tensor: where the tensor is nearly
    isotropic (inside a closed membrane) the score is orders of magnitude smaller than the
    tensor itself and carries the tensor's absolute rounding noise, the reference's own
    included.  It is therefore judged against max(|b|, 10 % of trace(T_ref)), floored at
    1e-3 of the volume's maximum."""
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    t = np.asarray(tensor_ref, np.float64)
    tr = t[..., 0] + t[..., 1] + t[..., 2]
    den = np.maximum(np.maximum(np.abs(b), 0.1 * tr), 1e-3 * np.abs(b).max())
    return float((np.abs(a - b) / den).max())


def draw_cases():
    """name -> (image, mask, regions, negative_means_subtract); shared with the tests (imported from here)."""
    shape = (20, 24, 28)
    rng = np.random.default_rng(31)
    zeros = np.zeros(shape, np.float32)
    noisy = rng.standard_normal(shape).astype(np.float32)
    mask = (rng.random(shape) > 0.3).astype(np.float32)
    add_sub = [("rect", 2.0, 20.4, 3.0, 18.0, 1.0, 15.0, 1.0), ("sphere", 12.0, 10.0, 8.0, 5.0, -1.0),
               ("sphere", 13.2, 11.7, 8.4, 2.6, 3.0), ("rect", 22.0, 40.0, -5.0, 6.49, 15.5, 30.0, 0.5),
               ("sphere", 27.0, 23.0, 19.0, 3.5, 2.0)]
    return {
        "add_sub": (zeros, None, add_sub, True),
        "from_ones": (zeros, None, [("sphere", 14.0, 12.0, 10.0, 6.3, -1.0), ("rect", 0.0, 5.0, 0.0, 5.0, 0.0, 5.0, -1.0),
                                    ("sphere", 14.0, 12.0, 10.0, 2.0, 1.0)], True),
        "from_ones_masked": (zeros, mask, [("rect", 3.0, 9.0, 3.0, 9.0, 3.0, 9.0, -2.0)], True),
        "no_subtract": (noisy, None, [("sphere", 10.5, 10.5, 10.5, 4.3, -1.0), ("sphere", 5.0, 6.0, 7.0, 0.0, 9.0),
                                      ("sphere", 20.0, 6.0, 7.0, 0.4, 8.0), ("rect", 1.5, 2.5, 0.0, 30.0, 4.0, 4.0, 7.0)], False),
        "masked": (noisy, mask, add_sub, True),
        "negative_first_nonzero": (noisy, None, [("sphere", 9.0, 9.0, 9.0, 5.0, -1.0)], True),
        "empty": (noisy, None, [], True),
    }


def sha256_of(*arrays):
    """SHA-256 (hex) of the bytes, shapes and dtypes of the arrays, None skipped: a stored check that the inputs or
    outputs of a test are, bit for bit, those some stored vectors were made from."""
    h = hashlib.sha256()
    for a in arrays:
        if a is not None:
            a = np.ascontiguousarray(a)
            h.update(("%s%s" % (a.dtype.str, a.shape)).encode())
            h.update(a.tobytes())
    return h.hexdigest()
