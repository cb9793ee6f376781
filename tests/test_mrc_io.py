"""MRC/REC file I/O (include/visfd_mrc.h, SURVEY 8f rank 2) against the reference's MrcSimple:
golden files in every mode, what MrcSimple::Read made of them, the bytes MrcSimple::Write
produced (tests/golden/make_golden.py).  Host code: no GPU needed."""
import numpy as np
import pytest

from visfd_b200 import mrc as vmrc


@pytest.fixture(scope="module")
def io():
    return vmrc.open_library()


def _cases(golden):
    return [str(n) for n in golden["mrc_names"]]


def test_read_and_write_match_the_reference(io, golden, tmp_path):
    for name in _cases(golden):
        key = name.replace(".", "_")
        src = tmp_path / name                      # the suffix matters (.rec => unsigned bytes)
        src.write_bytes(golden["mrc_in_" + key].tobytes())
        hdr, vox = io.read(src)
        assert np.array_equal(vox, golden["mrc_vox_" + key]), name
        hdr_only = io.read_header(src)
        assert hdr_only.as_bytes() == hdr.as_bytes(), name
        dst = tmp_path / ("out_" + name)
        io.write(dst, hdr, vox)
        assert dst.read_bytes() == golden["mrc_out_" + key].tobytes(), name          # byte-identical file
        assert hdr.as_bytes() == golden["mrc_hdr_" + key].tobytes(), name            # header incl. new dmin/dmax/dmean
        # what was written reads back as the same image, now mode 2
        hdr2, vox2 = io.read(dst)
        assert hdr2.mode == 2 and np.array_equal(vox2, vox), name


def live_case(io):
    """a header from visfd_mrc_header_init with a shape and a cell set, random float voxels"""
    rng = np.random.default_rng(9)
    vox = rng.standard_normal((9, 4, 11)).astype(np.float32)
    h = vmrc.MrcHeader()
    io.lib.visfd_mrc_header_init(ctypes_byref(h))
    h.nvoxels[:] = (11, 4, 9)
    h.mvoxels[:] = (11, 4, 9)
    h.cellA[:] = (22.0, 8.0, 18.0)
    return h, vox


def test_live_against_reference_build(io, golden, tmp_path):
    """live_case written and read back: the bytes the reference's MrcSimple::Write produced for it and the header
    its MrcSimple::Read made of the file (tests/golden/README.md)"""
    h, vox = live_case(io)
    ours = tmp_path / "a.mrc"
    io.write(ours, h, vox)
    assert ours.read_bytes() == golden["live_mrc_out"].tobytes()
    ho, vo = io.read(ours)
    assert ho.as_bytes() == golden["live_mrc_hdr"].tobytes() and np.array_equal(vo, vox)


def ctypes_byref(x):
    import ctypes
    return ctypes.byref(x)


def test_errors(io, tmp_path):
    with pytest.raises(vmrc.MrcError, match="Unable to open"):
        io.read(tmp_path / "missing.mrc")
    short = tmp_path / "short.mrc"
    short.write_bytes(b"\0" * 100)
    with pytest.raises(vmrc.MrcError):
        io.read(short)
    bad = tmp_path / "mode4.mrc"
    hdr = np.zeros(256, np.int32)
    hdr[0:3], hdr[3], hdr[16:19] = (2, 2, 2), 4, (1, 2, 3)
    bad.write_bytes(hdr.tobytes() + b"\0" * 64)
    with pytest.raises(vmrc.MrcError, match="UNSUPPORTED MODE"):
        io.read(bad)
    trunc = tmp_path / "trunc.mrc"
    hdr[3] = 2
    trunc.write_bytes(hdr.tobytes() + b"\0" * 16)            # 8 voxels announced, 4 present
    with pytest.raises(vmrc.MrcError, match="ends before"):
        io.read(trunc)


def test_large_volume_round_trip_and_speed(io, tmp_path):
    """64-bit sizes and bulk I/O: a 96 MB volume goes out and comes back unchanged at memory-copy-like
    speed (the reference moves one voxel per stream call, 13 Mvoxel/s per SURVEY 6)"""
    import time
    rng = np.random.default_rng(4)
    vox = rng.standard_normal((96, 512, 512), dtype=np.float32)
    h = vmrc.MrcHeader()
    io.lib.visfd_mrc_header_init(ctypes_byref(h))
    h.nvoxels[:] = (512, 512, 96)
    h.mvoxels[:] = (512, 512, 96)
    p = tmp_path / "big.mrc"
    dt = np.inf
    for _ in range(3):        # best of three: the machine running the suite may be busy compiling
        t = time.perf_counter()
        io.write(p, h, vox)
        hb, back = io.read(p, capacity=vox.size)
        dt = min(dt, time.perf_counter() - t)
        if vox.size / dt > 50e6:
            break
    assert np.array_equal(back, vox)
    assert abs(hb.dmean - vox.mean(dtype=np.float64)) < 1e-6 and hb.dmin == vox.min() and hb.dmax == vox.max()
    assert vox.size / dt > 25e6, f"{vox.size / dt / 1e6:.0f} Mvoxel/s"
