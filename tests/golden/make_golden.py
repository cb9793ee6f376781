#!/usr/bin/env python
"""Generate tests/golden/*.npz from the UNMODIFIED reference (oracle/_ref).

Run in the development container, where /root/reference exists:

    make -C oracle ref && python tests/golden/make_golden.py

Every array written here is an output of the reference's own code (the header-only
library instantiated by oracle/ref_shim.cpp, or the stock filter_mrc binary) on small
seeded inputs.  The fixtures travel with the repo, so that on machines without
/root/reference (the GPU box) the oracle port and the CUDA path are still pinned to
the reference.  The inputs are stored too: nothing has to be regenerated to check.
"""
import os
import subprocess
import sys
import tempfile
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle.pyoracle import Oracle, have  # noqa: E402
from visfd_b200 import synth  # noqa: E402
sys.path.insert(0, os.path.join(ROOT, "tests"))
from util import draw_cases  # noqa: E402

REFERENCE = os.environ.get("VISFD_REFERENCE", "/root/reference")


def read_mrc(path):
    """Minimal reader of the mrc_simple wire format (SURVEY.md appendix A)."""
    raw = open(path, "rb").read()
    h = np.frombuffer(raw[:1024], np.int32)
    nx, ny, nz, mode = int(h[0]), int(h[1]), int(h[2]), int(h[3])
    dt = {0: np.uint8, 1: np.int16, 2: np.float32, 6: np.uint16}[mode]
    a = np.frombuffer(raw[1024:1024 + nx * ny * nz * np.dtype(dt).itemsize], dt)
    return a.reshape(nz, ny, nx).astype(np.float32)


def mrc_file_bytes(mode, nvox, data, mapcrs=(1, 2, 3), imod=None, nsymbt=0):
    """A synthetic MRC file: every header word set to something recognisable (SURVEY appendix A)."""
    hdr = np.zeros(256, np.int32)
    hdr[0:3] = nvox
    hdr[3] = mode
    hdr[4:7] = (1, 2, 3)
    hdr[7:10] = (9, 9, 9)
    hdr[10:13] = np.array([10.5, 21.25, 33.75], np.float32).view(np.int32)
    hdr[13:16] = np.array([90, 90, 90], np.float32).view(np.int32)
    hdr[16:19] = mapcrs
    hdr[19:22] = np.array([-1.5, 2.5, 0.25], np.float32).view(np.int32)
    hdr[22], hdr[23] = 1, nsymbt
    hdr[24:49] = np.arange(25) * 7 + 3
    hdr[52:256] = np.arange(204) * 11 + 5
    if imod is not None:
        hdr[38], hdr[39] = 1146047817, imod
    hdr[49:52] = np.array([1.5, -2.5, 3.5], np.float32).view(np.int32)
    return hdr.tobytes() + data.tobytes()



def main():
    if not have("reference"):
        raise SystemExit("oracle/_ref/libvisfd_ref.so missing: run `make -C oracle ref` first")
    ref = Oracle("reference")
    out = {}

    # ---- Gaussian taps (GenFilterGauss1D) -------------------------------------------------
    taps_cases = [(2.0, 5), (0.8269, 2), (3.0, 7), (8.0, 21), (9.5, 25), (12.8, 33), (1.0, 1), (0.0, 2)]
    out["taps_cases"] = np.array(taps_cases, np.float64)
    for k, (s, hw) in enumerate(taps_cases):
        out[f"taps_{k}"] = ref.gen_gauss1d(s, hw)

    # ---- separable filters on a ragged little volume --------------------------------------
    shape = (11, 13, 17)
    rng = np.random.default_rng(1)
    vol = synth.tomogram(shape, seed=3) + rng.standard_normal(shape).astype(np.float32) * 0.1
    mask = np.ones(shape, np.float32)
    mask[:, :3, :] = 0.0
    mask[4:7, 5:9, 6:12] = 0.0
    mask[8:, 9:, 2:5] = 0.5          # weights, not just 0/1
    out["vol"], out["mask"] = vol, mask
    out["gauss_s1.3_hw3"], A = ref.apply_gauss(vol, 1.3, 3)
    out["gauss_A"] = np.float32(A)
    out["gauss_s1.3_hw3_nonorm"], _ = ref.apply_gauss(vol, 1.3, 3, normalize=False)
    out["gauss_aniso"], _ = ref.apply_gauss(vol, (1.0, 2.0, 0.7), (2, 5, 1))
    out["gauss_masked"], _ = ref.apply_gauss(vol, 1.3, 3, mask=mask)
    out["gauss_masked_nonorm"], _ = ref.apply_gauss(vol, 1.3, 3, mask=mask, normalize=False)
    out["gauss_wide"], _ = ref.apply_gauss(vol, 4.0, 10)   # half-width >= the image in z
    out["dog"], a, b = ref.apply_dog(vol, 1.2, 1.92, 5)
    out["dog_AB"] = np.array([a, b], np.float32)
    out["log"], a, b = ref.apply_log(vol, 1.5, 0.02, 2.6482)
    out["log_AB"] = np.array([a, b], np.float32)
    out["log_masked"], _, _ = ref.apply_log(vol, 1.5, 0.02, 2.6482, mask=mask)

    # ---- Hessian / eigen / cut -------------------------------------------------------------
    g, h = ref.calc_hessian(vol, 1.1, 2.6482)
    out["hess_grad"], out["hess_hess"] = g, h
    gm, hm = ref.calc_hessian(vol, 1.1, 2.6482, mask=mask)
    out["hess_grad_masked"], out["hess_hess_masked"] = gm, hm
    for order in (0, 1):
        sal, dire, ev = ref.hessian_eigen_score(h, order=order, score_kind=0)
        out[f"ridge_sal_o{order}"], out[f"ridge_dir_o{order}"], out[f"ridge_ev_o{order}"] = sal, dire, ev
    sal_lin, _, _ = ref.hessian_eigen_score(h, order=1, score_kind=1)
    out["ridge_sal_linear"] = sal_lin
    cut, thr = ref.saliency_cut(out["ridge_sal_o1"], 0.1, True)
    out["cut_frac0.1"], out["cut_frac0.1_thr"] = cut, np.float32(thr)
    cutm, thrm = ref.saliency_cut(out["ridge_sal_o1"], 0.25, True, mask=mask)
    out["cut_frac0.25_masked"], out["cut_frac0.25_masked_thr"] = cutm, np.float32(thrm)

    # ---- tensor voting -----------------------------------------------------------------------
    hw, decay, disp = ref.tv_tables(2.4, np.sqrt(2.0))
    out["tv_tables_hw"], out["tv_decay"], out["tv_disp"] = np.int32(hw), decay, disp
    tshape = (14, 12, 16)
    tvol = synth.tomogram(tshape, seed=5)
    out["tv_vol"] = tvol
    m = ref.membrane(tvol, 1.0, 2.6482, 1, 0.12, True, 2.4, 4, float(np.float32(np.sqrt(2.0))))
    for k in ("hess_saliency", "direction", "tensor", "out"):
        out["mem_" + k] = m[k]
    out["mem_thr"] = np.float32(m["threshold"])
    # explicit TVDenseStick with exponent 2 / generic exponent 3 / curves, and with masks
    sal, dire = m["hess_saliency"], m["direction"]
    out["tv_e2"] = ref.tv_dense_stick(sal, dire, 2.4, 2, float(np.float32(np.sqrt(2.0))))
    out["tv_e3"] = ref.tv_dense_stick(sal, dire, 2.4, 3, float(np.float32(np.sqrt(2.0))))
    out["tv_e4_curves"] = ref.tv_dense_stick(sal, dire, 2.4, 4, float(np.float32(np.sqrt(2.0))), curves=True)
    tmask = np.ones(tshape, np.float32)
    tmask[:, :, :3] = 0.0
    tmask[5:9, 4:8, 8:12] = 0.0
    out["tv_mask"] = tmask
    out["tv_e4_masked"] = ref.tv_dense_stick(sal, dire, 2.4, 4, float(np.float32(np.sqrt(2.0))),
                                             mask_src=tmask, mask_dst=tmask)
    out["tv_score_planar"] = ref.tensor_score(m["tensor"], order=1, score_kind=0)
    mm = ref.membrane(tvol, 1.0, 2.6482, 1, 0.12, True, 2.4, 4, float(np.float32(np.sqrt(2.0))), mask=tmask)
    out["mem_masked_out"], out["mem_masked_thr"] = mm["out"], np.float32(mm["threshold"])
    mx = ref.membrane(-tvol, 1.0, 2.6482, 0, 0.12, True, 2.4, 4, float(np.float32(np.sqrt(2.0))))
    out["mem_maxima_out"] = mx["out"]

    # ---- thresholds ------------------------------------------------------------------------------
    x = np.linspace(-2, 3, 101).astype(np.float32)
    out["thr_x"] = x
    out["thr1"] = ref.threshold1(x, 0.5, 0.0, 1.0)
    out["thr2_up"] = ref.threshold2(x, 0.2, 1.4, 0.0, 1.0)
    out["thr2_down"] = ref.threshold2(x, 1.4, 0.2, -1.0, 2.0)
    out["thr4"] = ref.threshold4(x, -1.0, -0.5, 1.5, 2.0, 0.0, 1.0)
    out["thr4_rev"] = ref.threshold4(x, 2.0, 1.5, -0.5, -1.0, 0.0, 1.0)
    out["mean_std"] = np.array([ref.average(vol), ref.stddev(vol), ref.average(vol, mask), ref.stddev(vol, mask)],
                               np.float32)

    # ---- blobs --------------------------------------------------------------------------------------
    bshape = (28, 30, 32)
    bvol = synth.tomogram(bshape, seed=9, blobs=10, noise=0.1, n_shells=0, blob_sigma=(1.5, 2.5))
    out["blob_vol"] = bvol
    sig = 1.0 * (1.25 ** np.arange(6))
    out["blob_sigmas"] = sig.astype(np.float32)
    mn, mx_ = ref.blob_dog(bvol, sig, 0.02, 2.6482, minima_threshold=0.0, maxima_threshold=-np.inf,
                           use_threshold_ratios=False)
    out["blob_minima"], out["blob_maxima"] = mn, mx_
    mn2, mx2 = ref.blob_dog(bvol, sig, 0.02, 2.6482, minima_threshold=0.5, maxima_threshold=0.5,
                            use_threshold_ratios=True)
    out["blob_minima_ratio"], out["blob_maxima_ratio"] = mn2, mx2

    # ---- binning (lib/visfd/resample.hpp) -------------------------------------------------------------
    bsrc = np.random.default_rng(23).standard_normal((13, 17, 22)).astype(np.float32)
    out["bin_src"] = bsrc
    out["bin_2"] = ref.bin3d(bsrc, bin_size=2)
    out["bin_3"] = ref.bin3d(bsrc, bin_size=3)
    out["bin_aniso_off"] = ref.bin3d(bsrc, dst_shape=(4, 5, 7), offset=(1, 2, 0))
    out["unbin_2"] = ref.unbin3d(out["bin_2"], (13, 17, 22))
    out["unbin_2_off"] = ref.unbin3d(out["bin_2"], (13, 17, 22), offset=(1, 0, 1))

    # ---- mask rasterisation (lib/visfd/draw.hpp:90-237) ----------------------------------------------
    for name, (img, mask, regions, subtract) in draw_cases().items():
        out["draw_" + name] = ref.draw_regions(img, regions, mask=mask, negative_means_subtract=subtract)

    # ---- MRC files (lib/mrc_simple): small files in every mode the reference reads, what its
    # MrcSimple::Read makes of them and the bytes its MrcSimple::Write produces ----------------------
    import ctypes
    from visfd_b200.mrc import MrcIO
    ref_mrc = MrcIO(ctypes.CDLL(os.path.join(ROOT, "oracle", "_ref", "libvisfd_ref.so")), "ref_mrc_")
    rng = np.random.default_rng(31)
    nvox, N = (5, 6, 7), 5 * 6 * 7
    mrc_cases = [
        ("m0u.rec", 0, rng.integers(0, 256, N).astype(np.uint8), {}),                  # .rec => unsigned bytes
        ("m0s.mrc", 0, rng.integers(0, 256, N).astype(np.uint8), {}),                  # default: signed bytes
        ("m0imod0.mrc", 0, rng.integers(0, 256, N).astype(np.uint8), dict(imod=0)),    # IMOD flag: unsigned
        ("m0imod1.rec", 0, rng.integers(0, 256, N).astype(np.uint8), dict(imod=1)),    # IMOD flag beats .rec
        ("m1.mrc", 1, rng.integers(-30000, 30000, N).astype(np.int16), {}),
        ("m6.mrc", 6, rng.integers(0, 65535, N).astype(np.uint16), {}),
        ("m2.mrc", 2, rng.standard_normal(N).astype(np.float32), dict(nsymbt=80)),     # nsymbt is ignored
        ("m2_213.mrc", 2, rng.standard_normal(N).astype(np.float32), dict(mapcrs=(2, 1, 3))),
        ("m1_132.rec", 1, rng.integers(-300, 300, N).astype(np.int16), dict(mapcrs=(1, 3, 2))),
        ("m2_321.mrc", 2, rng.standard_normal(N).astype(np.float32), dict(mapcrs=(3, 2, 1))),
    ]
    names = []
    with tempfile.TemporaryDirectory() as td:
        for name, mode, data, kw in mrc_cases:
            raw = mrc_file_bytes(mode, nvox, data, **kw)
            pth = os.path.join(td, name)
            open(pth, "wb").write(raw)
            hdr, vox = ref_mrc.read(pth)
            outp = os.path.join(td, "out_" + name)
            ref_mrc.write(outp, hdr, vox)
            key = name.replace(".", "_")
            names.append(name)
            out["mrc_in_" + key] = np.frombuffer(raw, np.uint8)
            out["mrc_vox_" + key] = vox
            out["mrc_hdr_" + key] = np.frombuffer(hdr.as_bytes(), np.uint8)     # after Write: with dmin/dmax/dmean
            out["mrc_out_" + key] = np.frombuffer(open(outp, "rb").read(), np.uint8)
    out["mrc_names"] = np.array(names)

    # ---- C1: the reference's own membrane test, run by the stock filter_mrc binary -----------------
    fm = os.path.join(ROOT, "oracle", "_ref", "filter_mrc")
    fixture = os.path.join(REFERENCE, "tests", "test_image_membrane.rec")
    if os.path.exists(fm) and os.path.exists(fixture):
        raw = read_mrc(fixture)
        binned = raw.reshape(8, 2, 8, 2, 8, 2).sum(axis=(1, 3, 5), dtype=np.float32) / np.float32(8)
        with tempfile.TemporaryDirectory() as td:
            o = os.path.join(td, "out.rec")
            # tests/test_membrane_detection.sh:8 without -save-progress
            subprocess.run([fm, "-w", "19.2", "-in", fixture, "-out", o, "-membrane", "minima", "55", "-tv", "4",
                            "-tv-angle-exponent", "4", "-bin", "2"], check=True, stdout=subprocess.DEVNULL,
                           stderr=subprocess.DEVNULL)
            c1 = read_mrc(o)
            o2 = os.path.join(td, "out_notv.rec")
            subprocess.run([fm, "-w", "19.2", "-in", fixture, "-out", o2, "-membrane", "minima", "55", "-bin", "2"],
                           check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            c1n = read_mrc(o2)
            # pass 2 of the same test (tests/test_membrane_detection.sh:9, in one invocation): the connected
            # surfaces -- the known answer for SURVEY 8f rank 1 (LabelConnected), not yet built
            o3 = os.path.join(td, "out_clusters.rec")
            log = subprocess.run([fm, "-w", "19.2", "-in", fixture, "-out", o3, "-membrane", "minima", "55", "-tv", "4",
                                  "-tv-angle-exponent", "4", "-bin", "2", "-connect", "1e+09", "-connect-angle", "30",
                                  "-select-cluster", "1"], check=True, stdout=subprocess.DEVNULL,
                                 stderr=subprocess.PIPE, text=True).stderr
            c1c = read_mrc(o3)
            n_clusters = [int(line.split()[4]) for line in log.splitlines() if "Number of clusters found:" in line]
        out["c1_connect_labels"] = c1c
        out["c1_connect_n_clusters"] = np.array(n_clusters, np.int64)
        print("C1 pass 2: clusters", n_clusters, "voxels in cluster 1:", int((c1c == 1).sum()))
        # parameters exactly as settings.cpp / filter_mrc.cpp derive them (float arithmetic)
        vw = np.float32(19.2) * np.float32(2)
        sigma = np.float32(np.float32(55.0) / np.sqrt(3.0))
        tv_sigma = np.float32(np.float32(4.0) * sigma)
        sigma = np.float32(sigma / vw)
        tv_sigma = np.float32(tv_sigma / vw)
        ratio = np.float32(np.sqrt(np.float32(-2) * np.log(np.float32(0.03))))
        assert np.array_equal(ref.bin3d(raw, bin_size=2), binned)
        out["c1_in_raw"] = raw
        out["c1_in_binned"] = binned
        out["c1_params"] = np.array([sigma, ratio, tv_sigma, 4, np.float32(np.sqrt(2.0)), 0.05], np.float32)
        out["c1_out"] = c1
        out["c1_out_notv"] = c1n
        # cross-check: the library path with these parameters reproduces the CLI bit for bit
        chk = ref.membrane(binned, float(sigma), float(ratio), 1, 0.05, True, float(tv_sigma), 4,
                           float(np.float32(np.sqrt(2.0))))
        assert np.array_equal(chk["out"], c1), "C1: library replay differs from filter_mrc output"
        print("C1: sum=%.6e max=%.6e nonzero=%d" % (c1.sum(dtype=np.float64), c1.max(), (c1 != 0).sum()))

    # ---- the reference's own blob test (tests/test_blob_detection.sh:21): `-blob minima f 160 280 1.01`
    # with -w 19.6 and a mask, run by the stock binary; the library replay with the parameters
    # filter_mrc derives (settings.cpp:1702-1743, filter_mrc.cpp:330-333, feature.hpp:469-471) ------------
    bfix = os.path.join(REFERENCE, "tests", "test_blob_detect.rec")
    bmask = os.path.join(REFERENCE, "tests", "test_blob_detect_mask.rec")
    if os.path.exists(fm) and os.path.exists(bfix):
        img, msk = read_mrc(bfix), read_mrc(bmask)
        with tempfile.TemporaryDirectory() as td:
            lst = os.path.join(td, "blobs.txt")
            subprocess.run([fm, "-w", "19.6", "-mask", bmask, "-in", bfix, "-blob", "minima", lst, "160.0", "280.0",
                            "1.01"], check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            cli = np.loadtxt(lst, ndmin=2)
        wmin, wmax, growth = np.float32(160.0), np.float32(280.0), np.float32(1.01)
        nsc = 1 + int(np.ceil(np.log(np.float64(wmax / wmin)) / np.log(np.float64(growth))))
        growth = np.float32(np.power(np.float64(wmax / wmin), 1.0 / nsc))
        diam = [np.float32(wmin)]
        for _ in range(1, nsc):
            diam.append(np.float32(diam[-1] * growth))
        vw = np.float32(19.6)
        diam = np.array([np.float32(d / vw) for d in diam], np.float32)
        sig = np.array([np.float32(np.float64(d) / (2.0 * np.sqrt(3.0))) for d in diam], np.float32)
        ratio_b = float(np.float32(np.sqrt(-2 * np.log(np.float32(0.03)))))
        mn_b, _ = ref.blob_dog(img, sig, 0.02, ratio_b, mask=msk, minima_threshold=0.0, maxima_threshold=-np.inf,
                               use_threshold_ratios=False)
        # the CLI prints x y z diameter score in physical units with 6 significant digits, best score first
        order = np.argsort(mn_b[:, 4], kind="stable")
        phys = np.stack([mn_b[order, 0] * vw, mn_b[order, 1] * vw, mn_b[order, 2] * vw,
                         np.float32(mn_b[order, 3] * np.float32(2.0 * np.sqrt(3.0))) * vw, mn_b[order, 4]], axis=1)
        assert cli.shape == phys.shape, (cli.shape, phys.shape)
        assert np.allclose(np.sort(cli, axis=0), np.sort(phys, axis=0), rtol=2e-5), "blob fixture: replay differs from filter_mrc"
        out["blobfix_img"], out["blobfix_mask"], out["blobfix_sigmas"] = img, msk, sig
        out["blobfix_ratio"] = np.float32(ratio_b)
        out["blobfix_minima"] = mn_b
        out["blobfix_cli"] = cli
        print("blob fixture: %d scales, %d minima" % (nsc, len(mn_b)))

        # ---- ... and its non-max suppression step (tests/test_blob_detection.sh:25): `-discard-blobs
        # in out -blob-separation 1.1 -minima-threshold -90`; known answer: 2 blobs (SURVEY 8c).
        # Replay of HandleBlobsNonmaxSuppression (handlers.cpp:428-640) with the reference's functions.
        from visfd_b200.blobs import BlobLists, SORT_DECREASING_MAGNITUDE
        rb = BlobLists(ctypes.CDLL(os.path.join(ROOT, "oracle", "_ref", "libvisfd_ref.so")), "ref_blobs_")
        with tempfile.TemporaryDirectory() as td:
            lst, lst2 = os.path.join(td, "blobs.txt"), os.path.join(td, "nms.txt")
            subprocess.run([fm, "-w", "19.6", "-mask", bmask, "-in", bfix, "-blob", "minima", lst, "160.0", "280.0",
                            "1.01"], check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            subprocess.run([fm, "-w", "19.6", "-mask", bmask, "-in", bfix, "-discard-blobs", lst, lst2,
                            "-blob-separation", "1.1", "-minima-threshold", "-90"], check=True,
                           stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            txt_in = np.loadtxt(lst, ndmin=2).astype(np.float32)
            cli2 = np.loadtxt(lst2, ndmin=2)
        # what the CLI reads back from its own text file (6 significant digits), in voxels
        nms_in = txt_in.copy()
        nms_in[:, :3] = np.floor(txt_in[:, :3] / vw + np.float32(0.5))
        nms_in[:, 3] = txt_in[:, 3] / vw
        kept = nms_in[(nms_in[:, 4] >= -np.inf) & (nms_in[:, 4] <= np.float32(-90.0))]
        kept = rb.discard_masked(kept, msk)
        nms_out = rb.discard_overlapping(kept, 1.1, np.inf, np.inf, SORT_DECREASING_MAGNITUDE)
        phys2 = nms_out.astype(np.float64) * np.array([vw, vw, vw, vw, 1.0])
        assert cli2.shape == phys2.shape == (2, 5), (cli2.shape, phys2.shape)
        assert np.allclose(cli2, phys2, rtol=2e-5), "blob NMS: replay differs from filter_mrc"
        out["blobnms_in"], out["blobnms_out"], out["blobnms_cli"] = nms_in, nms_out, cli2
        # a larger synthetic list for the list functions on their own
        g = np.random.default_rng(77)
        big = np.stack([g.uniform(0, 200, 600), g.uniform(0, 180, 600), g.uniform(0, 90, 600),
                        g.uniform(4, 30, 600), g.standard_normal(600) * 50], axis=1).astype(np.float32)
        big[::50, 4] = big[1::50, 4][:len(big[::50])]          # some tied scores
        out["bloblist_in"] = big
        out["bloblist_sorted_mag"] = rb.sort(big, SORT_DECREASING_MAGNITUDE, False)
        out["bloblist_sorted_inc"] = rb.sort(big, 2, True)
        out["bloblist_nms_sep"] = rb.discard_overlapping(big, 1.0)
        out["bloblist_nms_vol"] = rb.discard_overlapping(big, 0.0, 0.3, 0.6)
        out["bloblist_nms_inc"] = rb.discard_overlapping(big, 0.8, np.inf, np.inf, 2)
        print("blob NMS: %d -> %d (CLI %d); synthetic 600 -> %d / %d / %d" % (
            len(nms_in), len(nms_out), len(cli2), len(out["bloblist_nms_sep"]), len(out["bloblist_nms_vol"]),
            len(out["bloblist_nms_inc"])))

    # ---- reference_vectors_live.npz: the reference's results for the inputs of the tests that also compare with
    # oracle/_ref directly (test_*_live, test_*_vs_reference, test_*_is_the_reference, test_live_*); README.md in
    # this directory says where the committed values came from ------------------------------------------------------
    import test_blob_lists
    import test_mrc_io
    from visfd_b200.blobs import BlobLists
    from visfd_b200.mrc import open_library
    h, vox = test_mrc_io.live_case(open_library())
    with tempfile.TemporaryDirectory() as td:
        pth = os.path.join(td, "a.mrc")
        ref_mrc.write(pth, h, vox)
        out["live_mrc_out"] = np.frombuffer(open(pth, "rb").read(), np.uint8)
        out["live_mrc_hdr"] = np.frombuffer(ref_mrc.read(pth)[0].as_bytes(), np.uint8)
    ref_lists = BlobLists(ctypes.CDLL(os.path.join(ROOT, "oracle", "_ref", "libvisfd_ref.so")), "ref_blobs_")

    def rows(src, kept):
        """row numbers in src of the blobs kept, in their order"""
        return np.array([np.flatnonzero(np.all(src == r, axis=1))[0] for r in kept], np.int64)

    for n, b, bb, mask in test_blob_lists.live_cases():
        for k, args in enumerate(test_blob_lists.LIVE_OVERLAP_ARGS):
            out["live_blobs_%d_overlap%d" % (n, k)] = rows(b, ref_lists.discard_overlapping(b, *args))
        out["live_blobs_%d_masked" % n] = rows(bb, ref_lists.discard_masked(bb, mask))

    import test_oracle_golden
    for trial, img, mask, regions in test_oracle_golden.random_draw_cases():
        for subtract in (False, True):
            d = ref.draw_regions(img, regions, mask=mask, negative_means_subtract=subtract)
            out["live_draw_%d_%d" % (trial, subtract)] = np.where(d != img, d, np.float32(np.nan)).astype(np.float32)
    for k, v in test_oracle_golden.port_live_outputs(ref).items():
        out["live_port_" + k] = v
    from util import sha256_of
    for name, args, kw in test_oracle_golden.restatement_connect_calls(ref, out):
        res = ref.label_connected(*args, **kw)
        key = "live_connect_%s_" % name
        out[key + "labels"], out[key + "n_clusters"] = res[0].astype(np.int16), np.int64(res[1])
        if kw.get("want_direction"):
            out[key + "direction_inside"] = res[2][res[0] >= 1]
            out[key + "direction_sha256"] = np.array(sha256_of(res[2]))

    # files of less than 1 MB each; tests/conftest.py merges them
    lists = ("bloblist_", "blobfix_", "blobnms_")
    parts = {"reference_vectors_blob_lists.npz": {k: v for k, v in out.items() if k.startswith(lists)},
             "reference_vectors_live.npz": {k: v for k, v in out.items() if k.startswith("live_")},
             "reference_vectors.npz": {k: v for k, v in out.items() if not k.startswith(lists + ("live_",))}}
    for name, arrays in parts.items():
        path = os.path.join(HERE, name)
        np.savez_compressed(path, **arrays)
        print("wrote", path, "%.1f KiB" % (os.path.getsize(path) / 1024), len(arrays), "arrays")


if __name__ == "__main__":
    main()
