"""The membrane + -connect Z-slab drivers (visfd_cuda_membrane_connect_multi / _stream) without a GPU: both are
exported, and every bad argument ends in a VisfdCudaError that names the C entry point, never in a crash
(tests/test_gpu_membrane_connect.py runs them on the GPU).  The arguments are checked before any device is touched, so
a stream call with a NULL context still reports the argument it refuses."""
import ctypes as C

import numpy as np
import pytest

import visfd_b200

SHAPE = (16, 12, 10)
SQ2 = float(np.float32(np.sqrt(2.0)))
MULTI = "visfd_cuda_membrane_connect_multi"
STREAM = "visfd_cuda_membrane_connect_stream"


def _params(tv_sigma=4.0):
    return visfd_b200.MembraneParams(1.2, 2.6, visfd_b200.DECREASING_EIVALS, 0.05, 1, tv_sigma, 4, SQ2)


def _call(stream, shape=SHAPE, p=None, background_sigma=0.0, labels=True, out=True, capacity=16, device_bytes=0,
          devices=(0,)):
    """the C entry point (stream: with a NULL context) -> its error message"""
    lib = visfd_b200.load_library()
    src = np.zeros(shape, np.float32)
    res = np.zeros(shape, np.float32)
    lab = np.zeros(shape, np.int64)
    p = _params() if p is None else p
    c = visfd_b200.ConnectParams(1.0, 0.9, 0.9, 0.9, 0.9, 0)
    maxima = np.zeros((max(capacity, 1), 3), np.float32)
    nz, ny, nx = shape
    head = [C.c_int64(nx), C.c_int64(ny), C.c_int64(nz), C.c_void_p(src.ctypes.data), None, C.byref(p),
            C.c_float(background_sigma), C.c_int(1), C.byref(c)]
    outs = [C.c_void_p(res.ctypes.data) if out else None, None, C.c_void_p(lab.ctypes.data) if labels else None, None,
            None, C.c_void_p(maxima.ctypes.data), C.c_int64(capacity), None]
    if stream:
        rc = lib.visfd_cuda_membrane_connect_stream(None, *head, C.c_int64(device_bytes), *outs, None)
    else:
        devs = (C.c_int * len(devices))(*devices)
        rc = lib.visfd_cuda_membrane_connect_multi(C.c_int(len(devices)), devs, *head, *outs, None)
    assert rc != 0
    return lib.visfd_cuda_last_error().decode()


def test_both_entry_points_are_exported():
    lib = visfd_b200.load_library()
    assert hasattr(lib, MULTI) and hasattr(lib, STREAM)


BAD = {   # id -> (keyword arguments of _call, message)
    "null_labels": (dict(labels=False), "bad arguments"),
    "null_out": (dict(out=False), "bad arguments"),
    "negative_capacity": (dict(capacity=-1), "bad arguments"),
    "no_vote": (dict(p=_params(0.0)), "-connect clusters the vote tensor: tv_sigma must be positive"),
    "negative_vote": (dict(p=_params(-1.0)), "-connect clusters the vote tensor: tv_sigma must be positive"),
    "negative_background": (dict(background_sigma=-1.0), "negative background width"),
    "nan_background": (dict(background_sigma=float("nan")), "negative background width"),
    "thin_x": (dict(shape=(16, 12, 2)), "LabelConnected needs an image at least 3 voxels wide"),
    "thin_z": (dict(shape=(2, 12, 10)), "LabelConnected needs an image at least 3 voxels wide"),
}


@pytest.mark.parametrize("case", sorted(BAD))
def test_bad_arguments_are_refused(case):
    kw, msg = BAD[case]
    assert f"{MULTI}: {msg}" in _call(False, **kw)
    assert f"{STREAM}: {msg}" in _call(True, **kw)


def test_negative_budget_and_null_context():
    assert f"{STREAM}: negative device_bytes" in _call(True, device_bytes=-1)
    assert f"{STREAM}: context is NULL" in _call(True)


def test_multi_needs_a_device():
    assert f"{MULTI}: need at least one device" in _call(False, devices=())
    if visfd_b200.load_library().visfd_cuda_device_count() > 0:
        pytest.skip("a CUDA device is present: the GPU tests run the call")
    assert MULTI in _call(False)


def test_wrappers_take_numpy_arrays():
    torch = pytest.importorskip("torch")
    args = (1.2, 2.6, visfd_b200.DECREASING_EIVALS, 0.05, True, 4.0, 4, SQ2, 1.0)
    with pytest.raises(visfd_b200.VisfdCudaError, match=f"{MULTI} takes numpy"):
        visfd_b200.membrane_connect_multi([0], torch.zeros(SHAPE), *args)
    # (no context can be made without a GPU; the refusal comes before the context is used)
    ctx = object.__new__(visfd_b200.Context)
    with pytest.raises(visfd_b200.VisfdCudaError, match=f"{STREAM} takes numpy"):
        ctx.membrane_connect_stream(np.zeros(SHAPE, np.float32), *args, mask=torch.ones(SHAPE))


def test_params_follow_label_connected():
    """angle_deg sets all four cosines as Context.label_connected does; thresholds override them"""
    from visfd_b200.capi import _connect_args
    src = np.zeros(SHAPE, np.float32)
    _, _, out, labels, direction, p, _ = _connect_args("x", src, None, 2.5, 30.0, None, True, True)
    c = np.float32(np.cos(np.pi / 6))
    assert p.threshold_saliency == 2.5 and p.consider_dot_product_sign == 1
    assert p.threshold_vector_saliency == p.threshold_vector_neighbor == p.threshold_tensor_saliency == \
        p.threshold_tensor_neighbor == c
    assert out.shape == SHAPE and labels.dtype == np.int64 and direction.shape == SHAPE + (3,)
    _, _, _, _, direction, p, _ = _connect_args("x", src, None, 1.0, 30.0, (0.1, 0.2, 0.3, 0.4), False, False)
    assert direction is None and np.isclose(p.threshold_tensor_neighbor, 0.4) and p.consider_dot_product_sign == 0
