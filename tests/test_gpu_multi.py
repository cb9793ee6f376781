"""Real multi-GPU run of the Z-slab pipeline (NCCL) against the single-GPU result; needs >= 2 GPUs
(the gloo tests in test_slab_gloo.py cover the host logic everywhere else)."""
import os
import subprocess
import sys
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_multi_device_c_entry_equals_one_gpu():
    """visfd_cuda_membrane_multi (one C call, one worker thread per device; tests/cpp/multi_check.cpp) == the one-GPU
    result bit for bit for 1, 2, 3, 4 and 8 workers and for two calls made at once -- on as many devices as the box has
    (a one-GPU box lists the same device several times, which runs the same slab logic).  Calls that fail (no
    un-masked voxel, a voting radius above the maximum, a missing device) return their error."""
    exe = os.path.join(ROOT, "tests", "cpp", "multi_check")
    if not os.path.exists(exe):
        subprocess.check_call(["make", "-s", "-C", os.path.dirname(exe)])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=900)
    print(r.stdout[-4000:], r.stderr[-2000:])
    assert r.returncode == 0 and "OK (0 failures)" in r.stdout


@pytest.mark.gpu
def test_slab_pipeline_over_nccl_equals_one_gpu():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("one GPU on this box")
    n = 2 if n < 4 else (4 if n < 8 else 8)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
           "--master-addr", "127.0.0.1", "--master-port", "29517", os.path.join(ROOT, "tests", "multi_gpu_check.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    print(r.stdout[-3000:], r.stderr[-3000:])
    assert r.returncode == 0 and "MULTI_GPU_CHECK OK" in r.stdout
