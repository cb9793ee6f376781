"""ctypes binding of the C ABI in include/visfd_cuda.h (visfd_b200/libvisfd_cuda.so).

This is plumbing for tests, bench.py and the multi-GPU slab driver: every array may be
a C-contiguous float32 numpy array (HOST path: the library stages it through device
memory, exactly what the reference-side C++ shim does with Alloc3D memory) or a
contiguous float32 torch CUDA tensor (DEVICE path: no copies).  Volumes are indexed
[z][y][x] like the reference's ``aaafI[iz][iy][ix]``.

There is no CPU fallback: importing works without a GPU (so that the symbol table can
be checked), creating a Context without a usable B200 raises.
"""
import ctypes as C
import os
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libvisfd_cuda.so")

INCREASING_EIVALS = 0
DECREASING_EIVALS = 1
SCORE_PLANAR = 0
SCORE_LINEAR = 1
THRESH_SINGLE, THRESH_2, THRESH_4, THRESH_GAUSS, RESCALE = 1, 2, 4, 5, 6

_f, _i, _i64, _p, _d = C.c_float, C.c_int, C.c_int64, C.c_void_p, C.c_double


class VisfdCudaError(RuntimeError):
    """Mirror of VisfdErr (lib/visfd/err_visfd.hpp:15-22) for the Python host side."""


class MembraneParams(C.Structure):
    _fields_ = [("sigma", _f), ("truncate_ratio", _f), ("eival_order", _i), ("cut", _f),
                ("cut_is_fraction", _i), ("tv_sigma", _f), ("tv_exponent", _i),
                ("tv_cutoff_ratio", _f)]


_lib = None


def load_library():
    """Load the CUDA library; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise VisfdCudaError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(make -C visfd_b200/csrc). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    lib.visfd_cuda_last_error.restype = C.c_char_p
    lib.visfd_cuda_launch_count.restype = _i64
    lib.visfd_cuda_peak_reserved_bytes.restype = _i64
    lib.visfd_cuda_reset_peak_reserved_bytes.restype = None
    lib.visfd_cuda_last_voter_count.restype = _i64
    lib.visfd_cuda_last_tv_kernel.restype = C.c_int
    lib.visfd_cuda_stage_ms.restype = _d
    lib.visfd_cuda_key_to_float.restype = _f
    lib.visfd_cuda_set_timing.restype = None
    lib.visfd_cuda_set_fast_gauss.restype = None
    lib.visfd_cuda_reset_stage_ms.restype = None
    lib.visfd_cuda_destroy.restype = None
    lib.visfd_cuda_gen_gauss1d.restype = None
    _lib = lib
    return lib


def _is_torch(x):
    return type(x).__module__.startswith("torch")


def _ptr(x):
    if x is None:
        return None
    if _is_torch(x):
        assert x.is_cuda and x.is_contiguous() and x.dtype.is_floating_point and x.element_size() == 4
        # The library runs on its own non-blocking stream and every entry point is synchronous
        # (SURVEY 8b), so the only ordering the caller owes it is that whatever torch (or NCCL, through
        # torch's stream) still has in flight for this tensor is finished before the call reads it.
        import torch
        torch.cuda.current_stream(x.device).synchronize()
        return _p(x.data_ptr())
    assert isinstance(x, np.ndarray) and x.dtype == np.float32 and x.flags.c_contiguous
    return _p(x.ctypes.data)


REGION_DTYPE = np.dtype([("type", np.int32), ("p", np.float32, 6), ("value", np.float32)])  # struct visfd_region


def pack_regions(regions):
    """("rect", xmin, xmax, ymin, ymax, zmin, zmax, value) / ("sphere", x0, y0, z0, r, value) tuples ->
    an array of `visfd_region` records (include/visfd_cuda.h; visfd::SimpleRegion<float>, draw.hpp:41-87)."""
    rec = np.zeros(len(regions), REGION_DTYPE)
    for i, r in enumerate(regions):
        if r[0] == "sphere" and len(r) == 6:
            rec[i] = (1, tuple(r[1:5]) + (0.0, 0.0), r[5])
        elif r[0] == "rect" and len(r) == 8:
            rec[i] = (0, tuple(r[1:7]), r[7])
        else:
            raise VisfdCudaError("bad region %r" % (r,))
    return rec


def _pack_blobs(c, s, sc, n):
    return np.concatenate([c[:n], s[:n, None], sc[:n, None]], axis=1)


def blob_finalize(minima, maxima, best, minima_threshold=np.inf, maxima_threshold=-np.inf,
                  use_threshold_ratios=False, lib=None):
    """The final score filter of BlobDog on (n, 5) candidate rows x,y,z,sigma,score (host only, no GPU)."""
    lib = lib or load_library()
    out, cols, counts = [], [], []
    for rows in (minima, maxima):
        rows = np.ascontiguousarray(rows, np.float32).reshape(-1, 5)
        c = np.ascontiguousarray(rows[:, :3])
        sg = np.ascontiguousarray(rows[:, 3])
        sc = np.ascontiguousarray(rows[:, 4])
        cols.append((c, sg, sc))
        counts.append(_i64(len(rows)))
    rc = lib.visfd_cuda_blob_finalize(_f(minima_threshold), _f(maxima_threshold), _i(int(use_threshold_ratios)),
                                      _f(best[0]), _f(best[1]), _ptr(cols[0][0]), _ptr(cols[0][1]), _ptr(cols[0][2]),
                                      C.byref(counts[0]), _ptr(cols[1][0]), _ptr(cols[1][1]), _ptr(cols[1][2]),
                                      C.byref(counts[1]))
    if rc != 0:
        raise VisfdCudaError(lib.visfd_cuda_last_error().decode())
    for (c, sg, sc), n in zip(cols, counts):
        out.append(_pack_blobs(c, sg, sc, n.value))
    return out[0], out[1]


def _prep(x):
    """float32, contiguous; numpy stays numpy, torch stays torch."""
    if x is None:
        return None
    if _is_torch(x):
        import torch
        if not x.is_cuda:
            raise VisfdCudaError("torch tensors must live on the GPU (use numpy for host arrays)")
        return x.contiguous().to(torch.float32)
    return np.ascontiguousarray(x, dtype=np.float32)


def _empty(like, shape):
    if _is_torch(like):
        import torch
        return torch.empty(shape, dtype=torch.float32, device=like.device)
    return np.empty(shape, np.float32)


def _zeros(like, shape):
    if _is_torch(like):
        import torch
        return torch.zeros(shape, dtype=torch.float32, device=like.device)
    return np.zeros(shape, np.float32)


def _f3(v):
    v = [v] * 3 if np.isscalar(v) else list(v)
    return (_f * 3)(*v)


def _i3(v):
    v = [v] * 3 if np.isscalar(v) else list(v)
    return (_i * 3)(*[int(t) for t in v])


def gen_gauss1d(sigma, hw):
    """GenFilterGauss1D<float>(sigma, hw) (lib/visfd/filter1d.hpp:411-460); host only."""
    t = np.zeros(2 * hw + 1, np.float32)
    load_library().visfd_cuda_gen_gauss1d(_f(sigma), _i(hw), _ptr(t))
    return t


def gauss_halfwidth(sigma, truncate_ratio=-1.0, truncate_threshold=0.03):
    return load_library().visfd_cuda_gauss_halfwidth(_f(sigma), _f(truncate_ratio), _f(truncate_threshold))


def tv_halfwidth(sigma, cutoff_ratio):
    return load_library().visfd_cuda_tv_halfwidth(_f(sigma), _f(cutoff_ratio))


def membrane_multi(devices, src, sigma, truncate_ratio, order, cut, cut_is_fraction, tv_sigma, tv_exponent,
                   tv_cutoff_ratio, mask=None, out=None, lib=None, background_sigma=0.0, normalize=True):
    """visfd_cuda_membrane_multi: the fused pipeline of HandleTV on several GPUs of this node behind one C call
    (one worker thread per device, Z-slabs, host arrays in and out).  devices: list of CUDA device indices (a device
    may appear more than once).  background_sigma > 0: `-membrane-background`
    (visfd_cuda_membrane_multi_background).  -> dict(out, threshold, device_ms).  numpy (host) arrays only."""
    lib = lib or load_library()
    src = np.ascontiguousarray(src, np.float32)
    mask = None if mask is None else np.ascontiguousarray(mask, np.float32)
    res = out if out is not None else np.empty(src.shape, np.float32)
    assert isinstance(res, np.ndarray) and res.dtype == np.float32 and res.flags.c_contiguous and res.shape == src.shape
    p = MembraneParams(sigma, truncate_ratio, order, cut, int(cut_is_fraction), tv_sigma, tv_exponent, tv_cutoff_ratio)
    devs = (C.c_int * len(devices))(*[int(d) for d in devices])
    ms = (C.c_double * len(devices))()
    thr = _f()
    nz, ny, nx = src.shape
    if background_sigma > 0.0:
        rc = lib.visfd_cuda_membrane_multi_background(_i(len(devices)), devs, _i64(nx), _i64(ny), _i64(nz), _ptr(src),
                                                      _ptr(mask), C.byref(p), _f(background_sigma),
                                                      _i(int(normalize)), _ptr(res), C.byref(thr), ms)
    else:
        rc = lib.visfd_cuda_membrane_multi(_i(len(devices)), devs, _i64(nx), _i64(ny), _i64(nz), _ptr(src),
                                           _ptr(mask), C.byref(p), _ptr(res), C.byref(thr), ms)
    if rc != 0:
        raise VisfdCudaError(lib.visfd_cuda_last_error().decode())
    return dict(out=res, threshold=thr.value, device_ms=list(ms))


class Context:
    """One context per GPU (visfd_cuda_init)."""

    def __init__(self, device=-1, stream=None):
        self.lib = load_library()
        self.h = _p()
        rc = self.lib.visfd_cuda_init(_i(device), C.byref(self.h))
        if rc != 0:
            self.h = None
            raise VisfdCudaError(self.lib.visfd_cuda_last_error().decode())
        if stream is not None:
            self._ck(self.lib.visfd_cuda_set_stream(self.h, _p(stream)))

    def close(self):
        if getattr(self, "h", None):
            self.lib.visfd_cuda_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            raise VisfdCudaError(self.lib.visfd_cuda_last_error().decode())

    @staticmethod
    def _dims(shape):
        nz, ny, nx = shape
        return _i64(nx), _i64(ny), _i64(nz)

    # ---- bookkeeping -----------------------------------------------------------------
    def launch_count(self):
        return self.lib.visfd_cuda_launch_count(self.h)

    def peak_reserved_bytes(self):
        """Highest number of bytes the context's pool has held from cudaMalloc (live + cached) since creation or
        the last reset_peak_reserved_bytes()."""
        return self.lib.visfd_cuda_peak_reserved_bytes(self.h)

    def reset_peak_reserved_bytes(self):
        """Restart the peak from what the pool holds now (trim() first to start from zero)."""
        self.lib.visfd_cuda_reset_peak_reserved_bytes(self.h)

    def stage_ms(self, stage):
        return self.lib.visfd_cuda_stage_ms(self.h, stage.encode())

    def reset_stage_ms(self):
        self.lib.visfd_cuda_reset_stage_ms(self.h)

    @staticmethod
    def tv_halfwidth(sigma, cutoff_ratio):
        return tv_halfwidth(sigma, cutoff_ratio)

    def set_timing(self, enabled):
        self.lib.visfd_cuda_set_timing(self.h, _i(int(enabled)))

    def set_fast_gauss(self, enabled):
        """FFMA sweeps (fast) instead of the default bit-exact mul+add sweeps."""
        self.lib.visfd_cuda_set_fast_gauss(self.h, _i(int(enabled)))

    def trim(self):
        self._ck(self.lib.visfd_cuda_trim(self.h))

    def last_voter_count(self):
        return self.lib.visfd_cuda_last_voter_count(self.h)

    def last_tv_kernel(self):
        """Voting kernel of the last call: 0 = MUFU decay, 1 = r^2 table, 2 = r^2 table with clamped index."""
        return self.lib.visfd_cuda_last_tv_kernel(self.h)

    def fp32_peak(self, ms=200.0, packed=False, three_operand=False):
        t = _d()
        fn = self.lib.visfd_cuda_fp32_peak_packed if packed else self.lib.visfd_cuda_fp32_peak
        if three_operand:
            fn = self.lib.visfd_cuda_fp32_peak_3op
        self._ck(fn(self.h, _d(ms), C.byref(t)))
        return t.value

    def tv_count_pairs(self, saliency, threshold, halfwidth, mask_src=None, mask_dst=None, recv=None):
        s = _prep(saliency)
        n = _i64()
        r0, r1 = (0, s.shape[0]) if recv is None else recv
        self._ck(self.lib.visfd_cuda_tv_count_pairs(self.h, *self._dims(s.shape), _ptr(s), _f(threshold),
                                                    _ptr(_prep(mask_src)), _ptr(_prep(mask_dst)),
                                                    _i(halfwidth), _i64(r0), _i64(r1), C.byref(n)))
        return n.value

    # ---- separable filters --------------------------------------------------------------
    def apply_separable(self, src, taps, mask=None, normalize=True):
        """ApplySeparable (lib/visfd/filter3d.hpp:688-1050); taps = (tx, ty, tz) numpy arrays."""
        src, mask = _prep(src), _prep(mask)
        dst = _empty(src, src.shape)
        t = [np.ascontiguousarray(a, np.float32) for a in taps]
        hw = _i3([(len(a) - 1) // 2 for a in t])
        tp = (_p * 3)(*[a.ctypes.data for a in t])
        A = _f()
        self._ck(self.lib.visfd_cuda_apply_separable(self.h, *self._dims(src.shape), _ptr(src), _ptr(dst),
                                                     _ptr(mask), tp, hw, _i(int(normalize)), C.byref(A)))
        return dst, A.value

    def apply_gauss(self, src, sigma, hw, mask=None, normalize=True, z_offset=0, nz_global=None):
        """ApplyGauss (lib/visfd/filter3d.hpp:1088-1124); slab form when z_offset/nz_global are given."""
        src, mask = _prep(src), _prep(mask)
        dst = _empty(src, src.shape)
        A = _f()
        nzg = src.shape[0] if nz_global is None else nz_global
        self._ck(self.lib.visfd_cuda_apply_gauss_slab(self.h, *self._dims(src.shape), _i64(z_offset), _i64(nzg),
                                                      _ptr(src), _ptr(dst), _ptr(mask), _f3(sigma), _i3(hw),
                                                      _i(int(normalize)), C.byref(A)))
        return dst, A.value

    def apply_dog(self, src, sigma_a, sigma_b, hw, mask=None, hw_b=None):
        """ApplyDog (lib/visfd/filter3d.hpp:1340-1402); hw_b: the second Gaussian's own half-width, as
        filter_mrc's -dog gives each Gaussian (bin/filter_mrc/handlers.cpp:HandleDog)."""
        src, mask = _prep(src), _prep(mask)
        dst = _empty(src, src.shape)
        A, B = _f(), _f()
        if hw_b is None:
            self._ck(self.lib.visfd_cuda_apply_dog(self.h, *self._dims(src.shape), _ptr(src), _ptr(dst), _ptr(mask),
                                                   _f3(sigma_a), _f3(sigma_b), _i3(hw), C.byref(A), C.byref(B)))
        else:
            self._ck(self.lib.visfd_cuda_apply_dog2(self.h, *self._dims(src.shape), _ptr(src), _ptr(dst), _ptr(mask),
                                                    _f3(sigma_a), _f3(sigma_b), _i3(hw), _i3(hw_b), C.byref(A),
                                                    C.byref(B)))
        return dst, A.value, B.value

    def apply_log(self, src, sigma, delta=0.02, truncate_ratio=2.5, mask=None, z_offset=0, nz_global=None):
        """ApplyLog (lib/visfd/filter3d.hpp:1430-1507)."""
        src, mask = _prep(src), _prep(mask)
        dst = _empty(src, src.shape)
        A, B = _f(), _f()
        nzg = src.shape[0] if nz_global is None else nz_global
        self._ck(self.lib.visfd_cuda_apply_log_slab(self.h, *self._dims(src.shape), _i64(z_offset), _i64(nzg),
                                                    _ptr(src), _ptr(dst), _ptr(mask), _f3(sigma), _f(delta),
                                                    _f(truncate_ratio), C.byref(A), C.byref(B)))
        return dst, A.value, B.value

    # ---- Hessian / eigen --------------------------------------------------------------------
    def calc_hessian(self, src, sigma, truncate_ratio, mask=None):
        """CalcHessian (lib/visfd/feature.hpp:1210-1348) -> (gradient[...,3], hessian[...,6])."""
        src, mask = _prep(src), _prep(mask)
        grad = _zeros(src, tuple(src.shape) + (3,))
        hess = _zeros(src, tuple(src.shape) + (6,))
        self._ck(self.lib.visfd_cuda_calc_hessian(self.h, *self._dims(src.shape), _ptr(src), _ptr(mask), _f(sigma),
                                                  _f(truncate_ratio), _ptr(grad), _ptr(hess)))
        return grad, hess

    def hessian_ridge(self, src, sigma, truncate_ratio, order=DECREASING_EIVALS, score_kind=SCORE_PLANAR,
                      mask=None, want_direction=True):
        """CalcHessian + the eigen/score loop of HandleTV (handlers.cpp:1645-1746), fused."""
        src, mask = _prep(src), _prep(mask)
        sal = _empty(src, src.shape)
        dire = _zeros(src, tuple(src.shape) + (3,)) if want_direction else None
        self._ck(self.lib.visfd_cuda_hessian_ridge(self.h, *self._dims(src.shape), _ptr(src), _ptr(mask), _f(sigma),
                                                   _f(truncate_ratio), _i(order), _i(score_kind), _ptr(sal),
                                                   _ptr(dire)))
        return sal, dire

    def tensor_score(self, tensor, order=DECREASING_EIVALS, score_kind=SCORE_PLANAR, is_vote_tensor=True,
                     mask=None, out=None, want_eivals=False, want_direction=False):
        tensor, mask = _prep(tensor), _prep(mask)
        shape = tuple(tensor.shape[:-1])
        n = int(np.prod(shape))
        score = _zeros(tensor, shape) if out is None else _prep(out)
        ev = _zeros(tensor, shape + (3,)) if want_eivals else None
        dr = _zeros(tensor, shape + (3,)) if want_direction else None
        self._ck(self.lib.visfd_cuda_tensor_score(self.h, _i64(n), _ptr(tensor), _ptr(mask), _i(order),
                                                  _i(score_kind), _i(int(is_vote_tensor)), _ptr(score), _ptr(ev),
                                                  _ptr(dr)))
        return score, ev, dr

    def surface_points(self, saliency, direction, labels=None, mask=None, select_cluster=1, voxel_width=(1.0, 1.0, 1.0),
                       curve_ds=0.2, find_ridge=True, max_distance=1.3, capacity=None):
        """The oriented point cloud of `-normals-file` (handlers.cpp:2039-2309) -> (rows [n, 6] numpy, n_found);
        labels: float image (tomo_out after LabelConnected) or None for every un-masked voxel."""
        direction = _prep(direction)
        saliency, labels, mask = _prep(saliency), _prep(labels), _prep(mask)
        shape = tuple(direction.shape[:-1])
        nz, ny, nx = shape
        cap = int(capacity if capacity is not None else nz * ny * nx)
        rows = np.zeros((max(cap, 1), 6), np.float32)
        n = C.c_int64(0)
        vw = (C.c_float * 3)(*[float(v) for v in voxel_width])
        self._ck(self.lib.visfd_cuda_surface_points(self.h, _i64(nx), _i64(ny), _i64(nz), _ptr(saliency), _ptr(direction),
                                                    _ptr(labels), _ptr(mask), _i(int(select_cluster)), vw,
                                                    C.c_float(curve_ds), _i(int(find_ridge)), C.c_float(max_distance),
                                                    rows.ctypes.data_as(C.c_void_p), _i64(cap), C.byref(n)))
        return rows[:min(n.value, cap)], int(n.value)

    # ---- clustering --------------------------------------------------------------------------------
    def label_connected(self, saliency, tensor, threshold_saliency, angle_deg=15.0, order=DECREASING_EIVALS,
                        mask=None, direction=None, want_direction=False, consider_dot_product_sign=False,
                        thresholds=None):
        """LabelConnected as HandleTV calls it (connect.hpp:171, handlers.cpp:1927-2034; `-connect T -connect-angle A`).
        -> dict(labels int64 [-1 undefined, clusters from 1 by decreasing size], n_clusters, n_maxima, maxima (n, 3),
        direction (standardised; only if want_direction or direction was given)).  Arrays: numpy (host) only for
        `labels`; inputs numpy or torch.  thresholds: (vector_saliency, vector_neighbor, tensor_saliency,
        tensor_neighbor) cosines overriding angle_deg (settings.cpp:3075-3086 sets all four to cos(angle))."""
        saliency, tensor, mask = _prep(saliency), _prep(tensor), _prep(mask)
        shape = tuple(saliency.shape)
        nz, ny, nx = shape
        n = nz * ny * nx
        c = float(np.float32(np.cos(angle_deg * np.pi / 180.0)))
        tvs, tvn, tts, ttn = thresholds if thresholds is not None else (c, c, c, c)
        from_tensor = 0
        if direction is not None:
            direction = _prep(direction)
            if _is_torch(direction):
                direction = direction.clone()
            else:
                direction = np.array(direction, dtype=np.float32, copy=True, order="C")
        elif want_direction:
            if tensor is None:
                raise VisfdCudaError("want_direction needs a tensor or a direction field")
            direction = _zeros(saliency, shape + (3,))
            from_tensor = 1
        labels = np.zeros(shape, np.int64)
        ncl, nmax = _i64(), _i64()
        cap = 1 << 16
        maxima = np.zeros((cap, 3), np.float32)
        self._ck(self.lib.visfd_cuda_label_connected(
            self.h, _i64(nx), _i64(ny), _i64(nz), _ptr(saliency), _ptr(mask), _ptr(tensor), _ptr(direction),
            _i(from_tensor), _i(order), _i(int(consider_dot_product_sign)), _f(threshold_saliency), _f(tvs), _f(tvn),
            _f(tts), _f(ttn), labels.ctypes.data_as(C.c_void_p), C.byref(ncl), _ptr(maxima), _i64(cap), C.byref(nmax)))
        return dict(labels=labels, n_clusters=ncl.value, n_maxima=nmax.value,
                    maxima=maxima[:min(ncl.value, cap)].copy(), direction=direction)

    # ---- saliency cut ----------------------------------------------------------------------------
    def saliency_cut(self, sal, cut, is_fraction, mask=None):
        """handlers.cpp:1751-1797 -> (saliency after the cut, threshold)."""
        mask = _prep(mask)
        if _is_torch(sal):
            out = _prep(sal).clone()
        else:
            out = np.array(sal, dtype=np.float32, copy=True, order="C")
        thr = _f()
        self._ck(self.lib.visfd_cuda_saliency_cut(self.h, _i64(out.size if not _is_torch(out) else out.numel()),
                                                  _ptr(out), _ptr(mask), _f(cut), _i(int(is_fraction)),
                                                  C.byref(thr)))
        return out, thr.value

    def select_hist(self, sal, prefix, prefix_bits, mask=None):
        sal, mask = _prep(sal), _prep(mask)
        n = sal.numel() if _is_torch(sal) else sal.size
        hist = np.zeros(2048, np.uint64)
        self._ck(self.lib.visfd_cuda_select_hist(self.h, _i64(n), _ptr(sal), _ptr(mask), C.c_uint32(prefix),
                                                 _i(prefix_bits), hist.ctypes.data_as(_p)))
        return hist

    def select_step(self, hist, prefix, prefix_bits, rank):
        hist = np.ascontiguousarray(hist, np.uint64)
        p, b, r = C.c_uint32(prefix), _i(prefix_bits), C.c_uint64(rank)
        rc = self.lib.visfd_cuda_select_step(hist.ctypes.data_as(_p), C.byref(p), C.byref(b), C.byref(r))
        if rc != 0:
            raise VisfdCudaError("saliency cut: rank outside the population")
        return p.value, b.value, r.value

    def key_to_float(self, key):
        return self.lib.visfd_cuda_key_to_float(C.c_uint32(key))

    # ---- tensor voting -------------------------------------------------------------------------------
    def tv_dense_stick(self, sal, direction, sigma, exponent, cutoff_ratio, mask_src=None, mask_dst=None,
                       curves=False):
        """TV3D(sigma, exponent, cutoff_ratio).TVDenseStick (lib/visfd/feature.hpp:1712-2037)."""
        sal, direction = _prep(sal), _prep(direction)
        tensor = _zeros(sal, tuple(sal.shape) + (6,))
        self._ck(self.lib.visfd_cuda_tv_dense_stick(self.h, *self._dims(sal.shape), _ptr(sal), _ptr(direction),
                                                    _ptr(_prep(mask_src)), _ptr(_prep(mask_dst)), _f(sigma),
                                                    _i(exponent), _f(cutoff_ratio), _i(int(curves)), _i(0), _i(0),
                                                    _ptr(tensor)))
        return tensor

    def membrane(self, src, sigma, truncate_ratio, order, cut, cut_is_fraction, tv_sigma, tv_exponent,
                 tv_cutoff_ratio, mask=None, want_saliency=False, want_direction=False, want_tensor=False,
                 out=None, background_sigma=0.0, normalize=True):
        """The fused HandleTV pipeline (bin/filter_mrc/handlers.cpp:1618-1892); background_sigma > 0:
        `-membrane-background` (:1577-1592)."""
        src, mask = _prep(src), _prep(mask)
        p = MembraneParams(sigma, truncate_ratio, order, cut, int(cut_is_fraction), tv_sigma, tv_exponent,
                           tv_cutoff_ratio)
        res = out if out is not None else _empty(src, src.shape)
        sal = _empty(src, src.shape) if want_saliency else None
        dire = _zeros(src, tuple(src.shape) + (3,)) if want_direction else None
        tensor = _empty(src, tuple(src.shape) + (6,)) if want_tensor else None
        thr = _f()
        if background_sigma > 0.0:
            self._ck(self.lib.visfd_cuda_membrane_background(self.h, *self._dims(src.shape), _ptr(src), _ptr(mask),
                                                             C.byref(p), _f(background_sigma), _i(int(normalize)),
                                                             _ptr(res), _ptr(sal), _ptr(dire), _ptr(tensor), C.byref(thr)))
        else:
            self._ck(self.lib.visfd_cuda_membrane(self.h, *self._dims(src.shape), _ptr(src), _ptr(mask), C.byref(p),
                                                  _ptr(res), _ptr(sal), _ptr(dire), _ptr(tensor), C.byref(thr)))
        return dict(out=res, hess_saliency=sal, direction=dire, tensor=tensor, threshold=thr.value)

    def membrane_stream(self, src, sigma, truncate_ratio, order, cut, cut_is_fraction, tv_sigma, tv_exponent,
                        tv_cutoff_ratio, mask=None, out=None, device_bytes=0, background_sigma=0.0, normalize=True):
        """visfd_cuda_membrane_stream: the fused pipeline on this context's GPU in Z-slabs run one after another,
        for volumes whose working set does not fit on it; the device memory the call reserves stays within
        device_bytes (0: the free memory at entry, less a margin).  background_sigma > 0: `-membrane-background`
        (visfd_cuda_membrane_stream_background).  -> dict(out, threshold, n_slabs).  numpy (host) arrays only; the
        result is bit-identical to membrane() with the same arguments."""
        src = np.ascontiguousarray(src, np.float32)
        mask = None if mask is None else np.ascontiguousarray(mask, np.float32)
        res = out if out is not None else np.empty(src.shape, np.float32)
        assert isinstance(res, np.ndarray) and res.dtype == np.float32 and res.flags.c_contiguous and res.shape == src.shape
        p = MembraneParams(sigma, truncate_ratio, order, cut, int(cut_is_fraction), tv_sigma, tv_exponent,
                           tv_cutoff_ratio)
        thr, n_slabs = _f(), _i64()
        if background_sigma > 0.0:
            self._ck(self.lib.visfd_cuda_membrane_stream_background(
                self.h, *self._dims(src.shape), _ptr(src), _ptr(mask), C.byref(p), _f(background_sigma),
                _i(int(normalize)), _i64(int(device_bytes)), _ptr(res), C.byref(thr), C.byref(n_slabs)))
        else:
            self._ck(self.lib.visfd_cuda_membrane_stream(self.h, *self._dims(src.shape), _ptr(src), _ptr(mask),
                                                         C.byref(p), _i64(int(device_bytes)), _ptr(res), C.byref(thr),
                                                         C.byref(n_slabs)))
        return dict(out=res, threshold=thr.value, n_slabs=n_slabs.value)

    # ---- slab stages (device tensors only) -----------------------------------------------------------------
    def ridge_saliency_slab(self, src, z_offset, nz_global, sigma, truncate_ratio, order=DECREASING_EIVALS,
                            score_kind=SCORE_PLANAR, mask=None, smoothed=None, saliency=None):
        src, mask = _prep(src), _prep(mask)
        smoothed = _empty(src, src.shape) if smoothed is None else smoothed
        saliency = _empty(src, src.shape) if saliency is None else saliency
        self._ck(self.lib.visfd_cuda_ridge_saliency_slab(self.h, *self._dims(src.shape), _i64(z_offset),
                                                         _i64(nz_global), _ptr(src), _ptr(mask), _f(sigma),
                                                         _f(truncate_ratio), _i(order), _i(score_kind),
                                                         _ptr(smoothed), _ptr(saliency)))
        return smoothed, saliency

    def vote_slab(self, saliency, smoothed, z_offset, nz_global, own, vote, threshold, params, mask=None,
                  want_tensor=False, out=None, out_host=None):
        """out_host (optional, host array of the own planes): filled chunk by chunk behind the kernels."""
        if out_host is not None and _is_torch(out_host):
            assert not out_host.is_cuda
            out_host = out_host.numpy()
        shape = tuple(saliency.shape)
        n_own = own[1] - own[0]
        res = out if out is not None else _empty(saliency, (n_own,) + shape[1:])
        tensor = _empty(saliency, (n_own,) + shape[1:] + (6,)) if want_tensor else None
        self._ck(self.lib.visfd_cuda_vote_slab_host(self.h, *self._dims(shape), _i64(z_offset), _i64(nz_global),
                                                    _i64(own[0]), _i64(own[1]), _i64(vote[0]), _i64(vote[1]),
                                                    _ptr(saliency), _ptr(smoothed), _ptr(_prep(mask)),
                                                    _f(threshold), C.byref(params), _ptr(res), _ptr(tensor),
                                                    _ptr(out_host)))
        return res, tensor

    # ---- thresholds -----------------------------------------------------------------------------------------------
    def threshold(self, a, kind, t, outA=0.0, outB=1.0, mask=None, masked_value=None, out=None):
        """HandleThresholds inner loop (handlers.cpp:1037-1080) + mask fill (filter_mrc.cpp:771-776)."""
        a, mask = _prep(a), _prep(mask)
        res = _empty(a, a.shape) if out is None else _prep(out)
        t4 = (_f * 4)(*(list(t) + [0.0] * (4 - len(t))))
        n = res.numel() if _is_torch(res) else res.size
        self._ck(self.lib.visfd_cuda_threshold(self.h, _i64(n), _ptr(a), _ptr(res), _i(kind), t4, _f(outA), _f(outB),
                                               _ptr(mask), _i(int(masked_value is not None)),
                                               _f(0.0 if masked_value is None else masked_value)))
        return res

    def moment_sums(self, a, weights=None, center=0.0, squared=False):
        """visfd_cuda_moment_sums -> (sum w*h or sum w*(h-center)^2, sum w) as Python floats (double)."""
        a, weights = _prep(a), _prep(weights)
        n = a.numel() if _is_torch(a) else a.size
        out = (_d * 2)()
        self._ck(self.lib.visfd_cuda_moment_sums(self.h, _i64(n), _ptr(a), _ptr(weights), _d(center), _i(int(squared)), out))
        return out[0], out[1]

    def mean_stddev(self, a, weights=None):
        a, weights = _prep(a), _prep(weights)
        n = a.numel() if _is_torch(a) else a.size
        m, s = _f(), _f()
        self._ck(self.lib.visfd_cuda_mean_stddev(self.h, _i64(n), _ptr(a), _ptr(weights), C.byref(m), C.byref(s)))
        return m.value, s.value

    # ---- binning ---------------------------------------------------------------------------------------------------
    def _resample(self, fn, a, dst_shape, offset):
        a = _prep(a)
        res = _empty(a, tuple(dst_shape))
        ss = (_i64 * 3)(a.shape[2], a.shape[1], a.shape[0])
        ds = (_i64 * 3)(dst_shape[2], dst_shape[1], dst_shape[0])
        off = None if offset is None else (_i * 3)(*[int(v) for v in offset])
        self._ck(fn(self.h, ss, ds, _ptr(a), _ptr(res), off))
        return res

    def bin3d(self, a, bin_size=None, dst_shape=None, offset=None):
        """BinArray3D (lib/visfd/resample.hpp:53-104).  a: [nz][ny][nx]; give bin_size (HandleBinning's
        rule: destination = source // bin_size per axis) or an explicit dst_shape (nz, ny, nx);
        offset = (ox, oy, oz)."""
        if dst_shape is None:
            dst_shape = tuple(int(n) // int(bin_size) for n in a.shape)
        return self._resample(self.lib.visfd_cuda_bin3d, a, dst_shape, offset)

    def unbin3d(self, a, dst_shape, offset=None):
        """UnbinArray3D (lib/visfd/resample.hpp:106-166): nearest-voxel expansion to dst_shape (nz, ny, nx)."""
        return self._resample(self.lib.visfd_cuda_unbin3d, a, dst_shape, offset)

    # ---- mask rasterisation ----------------------------------------------------------------------------------------
    def draw_regions(self, image, regions, mask=None, negative_means_subtract=False):
        """DrawRegions (lib/visfd/draw.hpp:90-237; caller bin/filter_mrc/filter_mrc.cpp:280-284).
        regions, in painting order and in voxels: ("rect", xmin, xmax, ymin, ymax, zmin, zmax, value) or
        ("sphere", x0, y0, z0, r, value).  A numpy image is copied and the painted copy returned; a CUDA
        tensor is painted in place (and returned)."""
        img = _prep(image)
        if not _is_torch(img):
            img = np.array(img, np.float32, order="C", copy=True)
        mask = _prep(mask)
        rec = pack_regions(regions)
        self._ck(self.lib.visfd_cuda_draw_regions(self.h, *self._dims(img.shape), _ptr(img), _ptr(mask),
                                                  rec.ctypes.data_as(C.c_void_p), _i(len(rec)),
                                                  _i(int(negative_means_subtract))))
        if _is_torch(image) and img.data_ptr() != image.data_ptr():
            image.copy_(img)
            return image
        return img

    # ---- blobs -----------------------------------------------------------------------------------------------------
    def blob_dog(self, src, sigmas, delta=0.02, truncate_ratio=2.5, mask=None, minima_threshold=np.inf,
                 maxima_threshold=-np.inf, use_threshold_ratios=False, capacity=1 << 20):
        """BlobDog (lib/visfd/feature.hpp:56-427) -> (minima, maxima) rows of x,y,z,sigma,score."""
        src, mask = _prep(src), _prep(mask)
        sg = np.ascontiguousarray(np.asarray(sigmas), np.float32)
        bufs = [np.zeros((capacity, 3), np.float32), np.zeros(capacity, np.float32), np.zeros(capacity, np.float32),
                np.zeros((capacity, 3), np.float32), np.zeros(capacity, np.float32), np.zeros(capacity, np.float32)]
        nmin, nmax = _i64(), _i64()
        self._ck(self.lib.visfd_cuda_blob_dog(self.h, *self._dims(src.shape), _ptr(src), _ptr(mask), _ptr(sg),
                                              _i(len(sg)), _f(delta), _f(truncate_ratio), _f(minima_threshold),
                                              _f(maxima_threshold), _i(int(use_threshold_ratios)), _i64(capacity),
                                              _ptr(bufs[0]), _ptr(bufs[1]), _ptr(bufs[2]), C.byref(nmin),
                                              _ptr(bufs[3]), _ptr(bufs[4]), _ptr(bufs[5]), C.byref(nmax)))
        if nmin.value > capacity or nmax.value > capacity:
            raise VisfdCudaError("blob_dog: %d minima / %d maxima exceed the capacity of %d rows; call again with a "
                                 "larger capacity" % (nmin.value, nmax.value, capacity))
        return (_pack_blobs(bufs[0], bufs[1], bufs[2], nmin.value),
                _pack_blobs(bufs[3], bufs[4], bufs[5], nmax.value))

    def blob_dog_slab(self, src, z_offset, nz_global, own, sigmas, delta=0.02, truncate_ratio=2.5, mask=None,
                      minima_threshold=np.inf, maxima_threshold=-np.inf, use_threshold_ratios=False,
                      capacity=1 << 20):
        """visfd_cuda_blob_dog_slab: BlobDog on a z-slab (device tensor; own = slab-local receiver planes).
        -> (minima, maxima, (best_min, best_max)): candidate rows x,y,z(image),sigma,score BEFORE the final
        filter, and this slab's best scores (see blob_finalize)."""
        src, mask = _prep(src), _prep(mask)
        sg = np.ascontiguousarray(np.asarray(sigmas), np.float32)
        bufs = [np.zeros((capacity, 3), np.float32), np.zeros(capacity, np.float32), np.zeros(capacity, np.float32),
                np.zeros((capacity, 3), np.float32), np.zeros(capacity, np.float32), np.zeros(capacity, np.float32)]
        nmin, nmax = _i64(), _i64()
        best = (_f * 2)()
        self._ck(self.lib.visfd_cuda_blob_dog_slab(self.h, *self._dims(src.shape), _i64(z_offset), _i64(nz_global),
                                                   _i64(own[0]), _i64(own[1]), _ptr(src), _ptr(mask), _ptr(sg),
                                                   _i(len(sg)), _f(delta), _f(truncate_ratio), _f(minima_threshold),
                                                   _f(maxima_threshold), _i(int(use_threshold_ratios)),
                                                   _i64(capacity), _ptr(bufs[0]), _ptr(bufs[1]), _ptr(bufs[2]),
                                                   C.byref(nmin), _ptr(bufs[3]), _ptr(bufs[4]), _ptr(bufs[5]),
                                                   C.byref(nmax), best))
        if nmin.value > capacity or nmax.value > capacity:
            raise VisfdCudaError("blob candidate lists exceed the capacity given")
        return (_pack_blobs(bufs[0], bufs[1], bufs[2], nmin.value), _pack_blobs(bufs[3], bufs[4], bufs[5], nmax.value),
                (best[0], best[1]))

    def blob_finalize(self, minima, maxima, best, minima_threshold=np.inf, maxima_threshold=-np.inf,
                      use_threshold_ratios=False):
        """visfd_cuda_blob_finalize: the final score filter (feature.hpp:362-417) on gathered candidate rows,
        given the best scores of the whole image."""
        return blob_finalize(minima, maxima, best, minima_threshold, maxima_threshold, use_threshold_ratios, self.lib)
