"""The blob Z-slab drivers without a GPU: their argument checks and a missing device end in a VisfdCudaError that
names the C entry point, never in a crash (tests/test_gpu_blob_slabs.py runs them on the GPU)."""
import numpy as np
import pytest

import visfd_b200

SIGMAS = (1.0, 1.25, 1.5625)


def test_blob_dog_multi_needs_a_device():
    vol = np.zeros((16, 12, 10), np.float32)
    with pytest.raises(visfd_b200.VisfdCudaError, match="visfd_cuda_blob_dog_multi: need at least one device"):
        visfd_b200.blob_dog_multi([], vol, SIGMAS)
    if visfd_b200.load_library().visfd_cuda_device_count() > 0:
        pytest.skip("a CUDA device is present: the GPU tests run the call")
    with pytest.raises(visfd_b200.VisfdCudaError, match="visfd_cuda_blob_dog_multi"):
        visfd_b200.blob_dog_multi([0], vol, SIGMAS)


def test_blob_slab_drivers_take_numpy_arrays():
    torch = pytest.importorskip("torch")
    with pytest.raises(visfd_b200.VisfdCudaError, match="numpy"):
        visfd_b200.blob_dog_multi([0], torch.zeros((16, 12, 10)), SIGMAS)
