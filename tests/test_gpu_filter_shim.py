"""The shim's ApplyGauss / ApplyDog / ApplyLog (visfd_b200/csrc/visfd_cuda_shim.hpp), which run through
visfd_cuda_filter_stream, driven with the reference's and filter_mrc's overloads on float*** tables, in place too
(tests/cpp/filter_check.cpp): every result equals the one-shot C call bit for bit.  The checker is compiled into a
temporary directory against the in-tree library."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _build(out_dir):
    exe = os.path.join(str(out_dir), "filter_check")
    lib_dir = os.path.join(ROOT, "visfd_b200")
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O2", "-Wall", "-Werror",
                           os.path.join(ROOT, "tests", "cpp", "filter_check.cpp"), "-o", exe,
                           "-L" + lib_dir, "-lvisfd_cuda", "-Wl,-rpath," + lib_dir])
    return exe


def test_cpp_filter_check_compiles(tmp_path):
    _build(tmp_path)


@pytest.mark.gpu
def test_cpp_shim_filters_equal_the_one_shot_calls(tmp_path):
    r = subprocess.run([_build(tmp_path)], capture_output=True, text=True, timeout=600)
    print(r.stdout, r.stderr)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "OK (0 failures)" in r.stdout
