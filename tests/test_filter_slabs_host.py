"""The filter Z-slab drivers (visfd_cuda_filter_multi / visfd_cuda_filter_stream) without a GPU: both are exported,
and every bad argument ends in a VisfdCudaError that names the C entry point, never in a crash
(tests/test_gpu_filter_slabs.py runs them on the GPU).  The arguments are checked before any device is touched, so a
stream call with a NULL context still reports the argument it refuses."""
import ctypes as C

import numpy as np
import pytest

import visfd_b200
from visfd_b200 import FilterParams

SHAPE = (16, 12, 10)


def _multi(params, src=None, mask=None, out=None, devices=(0,)):
    src = np.zeros(SHAPE, np.float32) if src is None else src
    return visfd_b200.filter_multi(list(devices), src, params, mask=mask, out=out)


def _stream(params, mask=None, out=None, device_bytes=0):
    """the C entry point with a NULL context -> its error message"""
    lib = visfd_b200.load_library()
    src = np.zeros(SHAPE, np.float32)
    dst = np.zeros(SHAPE, np.float32) if out is None else out
    nz, ny, nx = SHAPE
    ptr = lambda a: None if a is None else C.c_void_p(a.ctypes.data)
    rc = lib.visfd_cuda_filter_stream(None, C.c_int64(nx), C.c_int64(ny), C.c_int64(nz), ptr(src), ptr(mask),
                                      C.byref(params), C.c_int64(device_bytes), ptr(dst), None, None, None)
    assert rc != 0
    return lib.visfd_cuda_last_error().decode()


def test_both_entry_points_are_exported():
    lib = visfd_b200.load_library()
    assert hasattr(lib, "visfd_cuda_filter_multi") and hasattr(lib, "visfd_cuda_filter_stream")


def test_params_mirror_the_one_shot_arguments():
    p = FilterParams.dog((1.0, 2.0, 3.0), 1.6, 4)
    assert p.kind == FilterParams.DOG and list(p.sigma_a) == [1.0, 2.0, 3.0]
    assert list(p.sigma_b) == [np.float32(1.6)] * 3
    assert list(p.hw_a) == list(p.hw_b) == [4, 4, 4]
    assert list(FilterParams.dog(1.0, 1.6, 3, hw_b=5).hw_b) == [5, 5, 5]
    g = FilterParams.gauss(2.0, (5, 6, 7), normalize=False)
    assert g.kind == FilterParams.GAUSS and list(g.hw_a) == [5, 6, 7] and g.normalize == 0
    lg = FilterParams.log(4.0, 0.05, 3.0)
    assert lg.kind == FilterParams.LOG and np.isclose(lg.delta, 0.05) and lg.truncate_ratio == 3.0


def test_multi_needs_a_device():
    g = FilterParams.gauss(1.0, 2)
    with pytest.raises(visfd_b200.VisfdCudaError, match="visfd_cuda_filter_multi: need at least one device"):
        _multi(g, devices=())
    if visfd_b200.load_library().visfd_cuda_device_count() > 0:
        pytest.skip("a CUDA device is present: the GPU tests run the call")
    with pytest.raises(visfd_b200.VisfdCudaError, match="visfd_cuda_filter_multi"):
        _multi(g)


def test_drivers_take_numpy_arrays():
    torch = pytest.importorskip("torch")
    g = FilterParams.gauss(1.0, 2)
    with pytest.raises(visfd_b200.VisfdCudaError, match="visfd_cuda_filter_multi takes numpy"):
        _multi(g, src=torch.zeros(SHAPE))
    # (no context can be made without a GPU; the refusal comes before the context is used)
    ctx = object.__new__(visfd_b200.Context)
    with pytest.raises(visfd_b200.VisfdCudaError, match="visfd_cuda_filter_stream takes numpy"):
        ctx.filter_stream(np.zeros(SHAPE, np.float32), g, mask=torch.ones(SHAPE))


BAD_PARAMS = [   # (id, params, message)
    ("kind", FilterParams(kind=3), "unknown filter kind 3"),
    ("sigma", FilterParams.gauss(-1.0, 2), "negative sigma or half-width"),
    ("hw", FilterParams.gauss(1.0, (2, -1, 2)), "negative sigma or half-width"),
    ("nan_sigma_b", FilterParams.dog(1.0, float("nan"), 2), "negative sigma or half-width"),
    ("hw_b", FilterParams.dog(1.0, 1.6, 2, hw_b=(2, 2, -3)), "negative sigma or half-width"),
    ("log_ratio", FilterParams.log(2.0, 0.02, -1.0), "negative sigma or half-width"),   # hw from the ratio
]


@pytest.mark.parametrize("params,msg", [c[1:] for c in BAD_PARAMS], ids=[c[0] for c in BAD_PARAMS])
def test_bad_params_are_refused(params, msg):
    with pytest.raises(visfd_b200.VisfdCudaError, match=f"visfd_cuda_filter_multi: {msg}"):
        _multi(params)
    assert f"visfd_cuda_filter_stream: {msg}" in _stream(params)


def test_negative_budget_and_null_context():
    g = FilterParams.gauss(1.0, 2)
    assert "visfd_cuda_filter_stream: negative device_bytes" in _stream(g, device_bytes=-1)
    assert "visfd_cuda_filter_stream: context is NULL" in _stream(g)


def test_mask_sharing_dst_is_refused():
    g = FilterParams.gauss(1.0, 2, normalize=True)
    mask = np.ones(SHAPE, np.float32)
    with pytest.raises(visfd_b200.VisfdCudaError, match="visfd_cuda_filter_multi: the mask must not share memory"):
        _multi(g, mask=mask, out=mask)
    assert "visfd_cuda_filter_stream: the mask must not share memory" in _stream(g, mask=mask, out=mask)
