// visfd_cuda_shim.hpp -- C++ host-side mirror of the reference's `namespace visfd`
// entry points for the membrane / blob hot path, forwarding to the C ABI of
// include/visfd_cuda.h (libvisfd_cuda.so, sm_100a).
//
// Same names, argument order, argument meaning and error behaviour as the reference
// templates instantiated with Scalar=float, Integer=int, VectorContainer=array<float,3>,
// TensorContainer=float* -- the only instantiation filter_mrc uses
// (bin/filter_mrc/handlers.cpp:1556-1565, :1821-1836) -- so a call site switches by
// changing the namespace:   visfd::ApplyGauss(...)  ->  visfd_cuda::ApplyGauss(...)
// (INTEGRATION.md shows the patch).  Errors surface as visfd_cuda::VisfdErr, the mirror
// of lib/visfd/err_visfd.hpp:15-22 (derive it from the reference's class when building
// inside the reference tree: define VISFD_CUDA_ERR_BASE before including this file).
//
// Arrays keep the reference's pointer-table layout (float***, array<float,3>***,
// float****).  Alloc3D memory is one contiguous block (lib/visfd/alloc3d.hpp:56-62) and
// is handed over without a copy; anything else (non-contiguous tables, the per-voxel
// float**** of CompactMultiChannelImage3D, lib/visfd/multichannel_image3d.hpp:93-142)
// is gathered / scattered through a dense host buffer.
//
// There is no CPU fallback: a failed CUDA call throws.
#pragma once
#include <algorithm>
#include <array>
#include <cmath>
#include <cstdint>
#include <exception>
#include <limits>
#include <ostream>
#include <string>
#include <vector>

#include "../../include/visfd_cuda.h"

namespace visfd_cuda {

#ifdef VISFD_CUDA_ERR_BASE
typedef VISFD_CUDA_ERR_BASE VisfdErr;
#else
class VisfdErr : public std::exception {
  std::string msg;
 public:
  explicit VisfdErr(const std::string &m) : msg(m) {}
  const char *what() const noexcept override { return msg.c_str(); }
};
#endif

// ---- process-wide context (filter_mrc is single-threaded, SURVEY 8b) ------------------
inline visfd_ctx *Context() {
  static visfd_ctx *ctx = nullptr;
  if (!ctx) {
    if (visfd_cuda_init(-1, &ctx) != 0)
      throw VisfdErr(std::string("Error: ") + visfd_cuda_last_error() + "\n");
  }
  return ctx;
}
inline void Check(int rc) {
  if (rc != 0) throw VisfdErr(std::string("Error: ") + visfd_cuda_last_error() + "\n");
}

// ---- pointer-table <-> dense views --------------------------------------------------------
// Dense [nz][ny][nx][C] view of a T*** table (C scalars per entry).  Contiguous tables
// are used in place; others are gathered (and scattered back on commit()).
template <typename Entry, int C>
class Dense3 {
  std::vector<float> buf;
  Entry ***tab = nullptr;
  float *ptr = nullptr;
  size_t nx, ny, nz;
  bool writable = false;
 public:
  Dense3(const int size[3], Entry const *const *const *table, bool will_write)
      : tab(const_cast<Entry ***>(table)), nx(size[0]), ny(size[1]), nz(size[2]), writable(will_write) {
    static_assert(sizeof(Entry) == C * sizeof(float), "entry must be C packed floats");
    if (!tab) return;
    bool contiguous = true;
    const Entry *base = tab[0][0];
    for (size_t iz = 0; iz < nz && contiguous; iz++)
      for (size_t iy = 0; iy < ny; iy++)
        if (tab[iz][iy] != base + (iz * ny + iy) * nx) { contiguous = false; break; }
    if (contiguous) {
      ptr = reinterpret_cast<float *>(const_cast<Entry *>(base));
    } else {
      buf.resize(nx * ny * nz * C);
      for (size_t iz = 0; iz < nz; iz++)
        for (size_t iy = 0; iy < ny; iy++) {
          const float *row = reinterpret_cast<const float *>(tab[iz][iy]);
          std::copy(row, row + nx * C, buf.begin() + (iz * ny + iy) * nx * C);
        }
      ptr = buf.data();
    }
  }
  float *data() { return ptr; }
  void commit() {
    if (!tab || buf.empty() || !writable) return;
    for (size_t iz = 0; iz < nz; iz++)
      for (size_t iy = 0; iy < ny; iy++) {
        float *row = reinterpret_cast<float *>(tab[iz][iy]);
        std::copy(buf.begin() + (iz * ny + iy) * nx * C, buf.begin() + (iz * ny + iy + 1) * nx * C, row);
      }
  }
};

// Dense [N][C] buffer behind a float**** (per-voxel pointer, nullptr where masked out).
class DenseTensor {
  std::vector<float> buf;
  float ****tab;
  size_t nx, ny, nz;
  int C;
 public:
  DenseTensor(const int size[3], float ****table, int channels, bool load)
      : tab(table), nx(size[0]), ny(size[1]), nz(size[2]), C(channels) {
    if (!tab) return;
    buf.assign(nx * ny * nz * C, 0.0f);
    if (load)
      for (size_t iz = 0; iz < nz; iz++)
        for (size_t iy = 0; iy < ny; iy++)
          for (size_t ix = 0; ix < nx; ix++)
            if (const float *p = tab[iz][iy][ix])
              std::copy(p, p + C, buf.begin() + ((iz * ny + iy) * nx + ix) * C);
  }
  float *data() { return tab ? buf.data() : nullptr; }
  void commit() {
    if (!tab) return;
    for (size_t iz = 0; iz < nz; iz++)
      for (size_t iy = 0; iy < ny; iy++)
        for (size_t ix = 0; ix < nx; ix++)
          if (float *p = tab[iz][iy][ix])
            std::copy(buf.begin() + ((iz * ny + iy) * nx + ix) * C, buf.begin() + ((iz * ny + iy) * nx + ix + 1) * C, p);
  }
};

// ---- separable filters (lib/visfd/filter3d.hpp) ---------------------------------------------
// Every filter runs in Z-slabs within the GPU's free memory: one slab, and the one-shot call's bits, when the volume
// fits; several slabs, and still the same bits, when it does not.  aaafDest may be aaafSource.
inline void RunFilter(const int image_size[3], float const *const *const *aaafSource, float ***aaafDest,
                   float const *const *const *aaafMask, const visfd_filter_params &p, float *pA, float *pB) {
  Dense3<float, 1> s(image_size, aaafSource, false), m(image_size, aaafMask, false), d(image_size, aaafDest, true);
  Check(visfd_cuda_filter_stream(Context(), image_size[0], image_size[1], image_size[2], s.data(), m.data(), &p, 0,
                                 d.data(), pA, pB, nullptr));
  d.commit();
}
inline visfd_filter_params DogParams(const float sigma_a[3], const float sigma_b[3], const int hw_a[3],
                                     const int hw_b[3]) {
  visfd_filter_params p{};
  p.kind = VISFD_FILTER_DOG;
  std::copy(sigma_a, sigma_a + 3, p.sigma_a);
  std::copy(sigma_b, sigma_b + 3, p.sigma_b);
  std::copy(hw_a, hw_a + 3, p.hw_a);
  std::copy(hw_b, hw_b + 3, p.hw_b);
  return p;
}

// ApplyGauss(sigma[3], truncate_halfwidth[3]): filter3d.hpp:1088-1124
inline float ApplyGauss(const int image_size[3], float const *const *const *aaafSource, float ***aaafDest,
                        float const *const *const *aaafMask, float const sigma[3],
                        const int truncate_halfwidth[3], bool normalize = true,
                        std::ostream *pReportProgress = nullptr) {
  visfd_filter_params p{};
  p.kind = VISFD_FILTER_GAUSS;
  std::copy(sigma, sigma + 3, p.sigma_a);
  std::copy(truncate_halfwidth, truncate_halfwidth + 3, p.hw_a);
  p.normalize = normalize ? 1 : 0;
  float A = 0;
  RunFilter(image_size, aaafSource, aaafDest, aaafMask, p, &A, nullptr);
  if (pReportProgress) *pReportProgress << " -- Gaussian filter applied on the GPU --\n";
  return A;
}
// ApplyGauss(sigma, truncate_halfwidth): filter3d.hpp:1163-1187
inline float ApplyGauss(const int image_size[3], float const *const *const *aaafSource, float ***aaafDest,
                        float const *const *const *aaafMask, float sigma, int truncate_halfwidth,
                        bool normalize = true, std::ostream *pReportProgress = nullptr) {
  float afSigma[3] = {sigma, sigma, sigma};
  int hw[3] = {truncate_halfwidth, truncate_halfwidth, truncate_halfwidth};
  return ApplyGauss(image_size, aaafSource, aaafDest, aaafMask, afSigma, hw, normalize, pReportProgress);
}
// ApplyGauss(sigma[3], truncate_ratio): filter3d.hpp:1228-1258 (hw = max(1, floor(sigma*ratio)))
inline float ApplyGauss(const int image_size[3], float const *const *const *aaafSource, float ***aaafDest,
                        float const *const *const *aaafMask, const float sigma[3], float truncate_ratio = 2.5,
                        bool normalize = true, std::ostream *pReportProgress = nullptr) {
  int hw[3];
  for (int d = 0; d < 3; d++) hw[d] = visfd_cuda_gauss_halfwidth(sigma[d], truncate_ratio, 1.0f);
  return ApplyGauss(image_size, aaafSource, aaafDest, aaafMask, sigma, hw, normalize, pReportProgress);
}
// filter_mrc's variant with (truncate_ratio, truncate_threshold): bin/filter_mrc/filter3d_variants.hpp:500-528
inline float ApplyGauss(const int image_size[3], float const *const *const *aaafSource, float ***aaafDest,
                        float const *const *const *aaafMask, const float sigma[3], float truncate_ratio,
                        float truncate_threshold, bool normalize, std::ostream *pReportProgress = nullptr) {
  int hw[3];
  for (int d = 0; d < 3; d++) hw[d] = visfd_cuda_gauss_halfwidth(sigma[d], truncate_ratio, truncate_threshold);
  return ApplyGauss(image_size, aaafSource, aaafDest, aaafMask, sigma, hw, normalize, pReportProgress);
}

// ApplyDog: filter3d.hpp:1340-1402
inline void ApplyDog(const int image_size[3], float const *const *const *aaafSource, float ***aaafDest,
                     float const *const *const *aaafMask, float const sigma_a[3], float const sigma_b[3],
                     const int truncate_halfwidth[3], float *pA = nullptr, float *pB = nullptr,
                     std::ostream *pReportProgress = nullptr) {
  (void)pReportProgress;
  RunFilter(image_size, aaafSource, aaafDest, aaafMask,
            DogParams(sigma_a, sigma_b, truncate_halfwidth, truncate_halfwidth), pA, pB);
}

// ApplyLog: filter3d.hpp:1430-1507
inline void ApplyLog(const int image_size[3], float const *const *const *aaafSource, float ***aaafDest,
                     float const *const *const *aaafMask, const float sigma[3],
                     float delta_sigma_over_sigma = 0.02, float truncate_ratio = 2.5, float *pA = nullptr,
                     float *pB = nullptr, std::ostream *pReportProgress = nullptr) {
  (void)pReportProgress;
  visfd_filter_params p{};
  p.kind = VISFD_FILTER_LOG;
  std::copy(sigma, sigma + 3, p.sigma_a);
  p.delta = delta_sigma_over_sigma;
  p.truncate_ratio = truncate_ratio;
  RunFilter(image_size, aaafSource, aaafDest, aaafMask, p, pA, pB);
}


// filter_mrc's variants with (truncate_ratio, truncate_threshold): bin/filter_mrc/filter3d_variants.hpp:542-597, :603-634
inline void ApplyDog(const int image_size[3], float const *const *const *aaafSource, float ***aaafDest,
                     float const *const *const *aaafMask, const float sigma_a[3], const float sigma_b[3],
                     float filter_truncate_ratio, float filter_truncate_threshold, float *pA = nullptr,
                     float *pB = nullptr, std::ostream *pReportProgress = nullptr) {
  (void)pReportProgress;
  int hwa[3], hwb[3];   // each Gaussian keeps the half-width of its own sigma (two ApplyGauss calls in the reference)
  for (int d = 0; d < 3; d++) {
    hwa[d] = visfd_cuda_gauss_halfwidth(sigma_a[d], filter_truncate_ratio, filter_truncate_threshold);
    hwb[d] = visfd_cuda_gauss_halfwidth(sigma_b[d], filter_truncate_ratio, filter_truncate_threshold);
  }
  RunFilter(image_size, aaafSource, aaafDest, aaafMask, DogParams(sigma_a, sigma_b, hwa, hwb), pA, pB);
}
inline void ApplyLog(const int image_size[3], float const *const *const *aaafSource, float ***aaafDest,
                     float const *const *const *aaafMask, const float sigma[3], float delta_sigma_over_sigma,
                     float filter_truncate_ratio, float filter_truncate_threshold, float *pA = nullptr,
                     float *pB = nullptr, std::ostream *pReportProgress = nullptr) {
  if (filter_truncate_ratio < 0) filter_truncate_ratio = std::sqrt(-2 * std::log(filter_truncate_threshold));
  ApplyLog(image_size, aaafSource, aaafDest, aaafMask, sigma, delta_sigma_over_sigma, filter_truncate_ratio, pA, pB,
           pReportProgress);
}

// ---- features (lib/visfd/feature.hpp) ---------------------------------------------------------
// CalcHessian<float, array<float,3>, float*>: feature.hpp:1210-1348
inline void CalcHessian(int const image_size[3], float const *const *const *aaafSource,
                        std::array<float, 3> ***aaaafGradient, float ****aaaafHessian,
                        float const *const *const *aaafMask, float sigma, float truncate_ratio = 2.5,
                        std::ostream *pReportProgress = nullptr) {
  (void)pReportProgress;
  Dense3<float, 1> s(image_size, aaafSource, false), m(image_size, aaafMask, false);
  Dense3<std::array<float, 3>, 3> g(image_size, aaaafGradient, true);
  DenseTensor h(image_size, aaaafHessian, 6, aaafMask != nullptr);
  Check(visfd_cuda_calc_hessian(Context(), image_size[0], image_size[1], image_size[2], s.data(), m.data(), sigma,
                                truncate_ratio, g.data(), h.data()));
  g.commit();
  h.commit();
}

// BlobDog<float>: feature.hpp:56-427 (isotropic blobs; filter_mrc's aspect ratio is 1,1,1)
inline void BlobDog(int const image_size[3], float const *const *const *aaafSource,
                    float const *const *const *aaafMask, const std::vector<float> &blob_sigma,
                    std::vector<std::array<float, 3> > *pva_minima_crds = nullptr,
                    std::vector<std::array<float, 3> > *pva_maxima_crds = nullptr,
                    std::vector<float> *pv_minima_sigma = nullptr, std::vector<float> *pv_maxima_sigma = nullptr,
                    std::vector<float> *pv_minima_scores = nullptr, std::vector<float> *pv_maxima_scores = nullptr,
                    const float aspect_ratio[3] = nullptr, float delta_sigma_over_sigma = 0.02,
                    float truncate_ratio = 2.5, float minima_threshold = std::numeric_limits<float>::infinity(),
                    float maxima_threshold = -std::numeric_limits<float>::infinity(),
                    bool use_threshold_ratios = true, std::ostream *pReportProgress = nullptr,
                    float ****aaaafI = nullptr) {
  (void)pReportProgress;
  (void)aaaafI;  // scratch volumes live on the device
  if (aspect_ratio && (aspect_ratio[0] != 1.0f || aspect_ratio[1] != 1.0f || aspect_ratio[2] != 1.0f))
    throw VisfdErr("Error: the CUDA BlobDog supports isotropic blobs only (aspect ratio 1,1,1)\n");
  Dense3<float, 1> s(image_size, aaafSource, false), m(image_size, aaafMask, false);
  int64_t capacity = 1 << 16, nmin = 0, nmax = 0;
  std::vector<float> mc, ms, msc, xc, xs, xsc;
  for (int attempt = 0; attempt < 2; attempt++) {
    mc.resize(3 * capacity); ms.resize(capacity); msc.resize(capacity);
    xc.resize(3 * capacity); xs.resize(capacity); xsc.resize(capacity);
    // in Z-slabs within the GPU's free memory: one slab, and the one-GPU lists, when the volume fits; several
    // slabs, and still the same lists, when it does not
    Check(visfd_cuda_blob_dog_stream(Context(), image_size[0], image_size[1], image_size[2], s.data(), m.data(),
                                     blob_sigma.data(), (int)blob_sigma.size(), delta_sigma_over_sigma,
                                     truncate_ratio, minima_threshold, maxima_threshold, use_threshold_ratios ? 1 : 0,
                                     0, capacity, mc.data(), ms.data(), msc.data(), &nmin, xc.data(), xs.data(),
                                     xsc.data(), &nmax, nullptr));
    if (nmin <= capacity && nmax <= capacity) break;
    capacity = std::max(nmin, nmax);
  }
  auto emit = [](int64_t n, const std::vector<float> &c, const std::vector<float> &sg, const std::vector<float> &sc,
                 std::vector<std::array<float, 3> > *pc, std::vector<float> *ps, std::vector<float> *pscore) {
    if (pc) pc->clear();
    if (ps) ps->clear();
    if (pscore) pscore->clear();
    for (int64_t i = 0; i < n; i++) {
      if (pc) pc->push_back({c[3 * i], c[3 * i + 1], c[3 * i + 2]});
      if (ps) ps->push_back(sg[i]);
      if (pscore) pscore->push_back(sc[i]);
    }
  };
  emit(nmin, mc, ms, msc, pva_minima_crds, pv_minima_sigma, pv_minima_scores);
  emit(nmax, xc, xs, xsc, pva_maxima_crds, pv_maxima_sigma, pv_maxima_scores);
}


// BlobDogD<float>: feature.hpp:449-512 (diameters instead of sigmas: sigma = diameter / (2 sqrt 3))
inline void BlobDogD(int const image_size[3], float const *const *const *aaafSource,
                     float const *const *const *aaafMask, const std::vector<float> &blob_diameters,
                     std::vector<std::array<float, 3> > *pva_minima_crds = nullptr,
                     std::vector<std::array<float, 3> > *pva_maxima_crds = nullptr,
                     std::vector<float> *pv_minima_diameters = nullptr, std::vector<float> *pv_maxima_diameters = nullptr,
                     std::vector<float> *pv_minima_scores = nullptr, std::vector<float> *pv_maxima_scores = nullptr,
                     const float aspect_ratio[3] = nullptr, float delta_sigma_over_sigma = 0.02,
                     float truncate_ratio = 2.5, float minima_threshold = std::numeric_limits<float>::infinity(),
                     float maxima_threshold = -std::numeric_limits<float>::infinity(),
                     bool use_threshold_ratios = false, std::ostream *pReportProgress = nullptr,
                     float ****aaaafI = nullptr) {
  std::vector<float> minima_sigma, maxima_sigma, blob_sigma(blob_diameters.size());
  for (size_t i = 0; i < blob_diameters.size(); i++) blob_sigma[i] = blob_diameters[i] / (2.0 * std::sqrt(3));
  BlobDog(image_size, aaafSource, aaafMask, blob_sigma, pva_minima_crds, pva_maxima_crds, &minima_sigma, &maxima_sigma,
          pv_minima_scores, pv_maxima_scores, aspect_ratio, delta_sigma_over_sigma, truncate_ratio, minima_threshold,
          maxima_threshold, use_threshold_ratios, pReportProgress, aaaafI);
  if (pv_minima_diameters) {
    pv_minima_diameters->resize(minima_sigma.size());
    for (size_t i = 0; i < minima_sigma.size(); i++) (*pv_minima_diameters)[i] = minima_sigma[i] * 2.0 * std::sqrt(3);
  }
  if (pv_maxima_diameters) {
    pv_maxima_diameters->resize(maxima_sigma.size());
    for (size_t i = 0; i < maxima_sigma.size(); i++) (*pv_maxima_diameters)[i] = maxima_sigma[i] * 2.0 * std::sqrt(3);
  }
}

// LabelConnected<float, ptrdiff_t, float, array<float,3>, float*>: lib/visfd/connect.hpp:171-1432 with the argument
// list of the reference (the values HandleTV and HandleLabelConnected pass, handlers.cpp:1963-1993, :1438-1470).
// Supported: connectivity 1, clusters grown from maxima, sorted by size, no voxel weights, no must-link
// constraints; aaaafVectorStandardized must be nullptr or alias aaaafVector (as in HandleTV).  Anything else throws.
inline size_t LabelConnected(const int image_size[3], float const *const *const *aaafSaliency, ptrdiff_t ***aaaiDest,
                             float const *const *const *aaafMask,
                             float threshold_saliency = -std::numeric_limits<float>::infinity(),
                             std::array<float, 3> const *const *const *aaaafVector = nullptr,
                             float threshold_vector_saliency = -std::numeric_limits<float>::infinity(),
                             float threshold_vector_neighbor = -std::numeric_limits<float>::infinity(),
                             bool consider_dot_product_sign = true, float *const *const *const *aaaafSymmetricTensor = nullptr,
                             float threshold_tensor_saliency = -std::numeric_limits<float>::infinity(),
                             float threshold_tensor_neighbor = -std::numeric_limits<float>::infinity(),
                             bool tensor_is_positive_definite_near_target = true, int connectivity = 1,
                             ptrdiff_t label_undefined = -1,
                             std::vector<std::array<float, 3> > *pv_cluster_maxima = nullptr,
                             std::vector<float> *pv_cluster_sizes = nullptr,
                             std::vector<float> *pv_cluster_saliencies = nullptr, int sort_criteria = 1 /*SORT_BY_SIZE*/,
                             float const *const *const *aaafVoxelWeights = nullptr,
                             std::array<float, 3> ***aaaafVectorStandardized = nullptr,
                             const void *pMustLinkConstraints = nullptr, const void *pMustLinkDirections = nullptr,
                             bool start_from_saliency_maxima = true, std::ostream *pReportProgress = nullptr) {
  if (connectivity != 1 || !tensor_is_positive_definite_near_target || !start_from_saliency_maxima ||
      sort_criteria != 1 || aaafVoxelWeights || pMustLinkConstraints)
    throw VisfdErr("Error: the CUDA LabelConnected supports connectivity 1, maxima seeds, size ordering, no weights and "
                   "no must-link constraints\n");
  (void)pMustLinkDirections;   // only read together with the constraints (connect.hpp:946-961); HandleTV passes an empty list
  if (aaaafVectorStandardized && (std::array<float, 3> const *const *const *)aaaafVectorStandardized != aaaafVector)
    throw VisfdErr("Error: the CUDA LabelConnected standardises the direction array in place\n");
  if (aaaafSymmetricTensor && !aaaafVector)
    throw VisfdErr("Error: LabelConnected with tensors needs the direction array as well (connect.hpp:648-676)\n");
  Dense3<float, 1> sal(image_size, aaafSaliency, false), m(image_size, aaafMask, false);
  Dense3<std::array<float, 3>, 3> v(image_size, aaaafVector, aaaafVectorStandardized != nullptr);
  DenseTensor t(image_size, const_cast<float ****>(aaaafSymmetricTensor), 6, true);
  const size_t N = (size_t)image_size[0] * image_size[1] * image_size[2];
  std::vector<int64_t> lab(N);
  int64_t n_clusters = 0, n_maxima = 0;
  std::vector<float> maxima(3 * (size_t)(1 << 20));
  // a caller that does not want standardised directions must not see its array change: work on a copy
  std::vector<float> vcopy;
  float *vptr = v.data();
  if (vptr && !aaaafVectorStandardized) {
    vcopy.assign(vptr, vptr + 3 * N);
    vptr = vcopy.data();
  }
  Check(visfd_cuda_label_connected(Context(), image_size[0], image_size[1], image_size[2], sal.data(), m.data(), t.data(),
                                   vptr, 0, VISFD_DECREASING_EIVALS, consider_dot_product_sign ? 1 : 0,
                                   threshold_saliency, threshold_vector_saliency, threshold_vector_neighbor,
                                   threshold_tensor_saliency, threshold_tensor_neighbor, lab.data(), &n_clusters,
                                   maxima.data(), (int64_t)(maxima.size() / 3), &n_maxima));
  v.commit();
  const size_t nx = image_size[0], ny = image_size[1], nz = image_size[2];
  for (size_t iz = 0; iz < nz; iz++)
    for (size_t iy = 0; iy < ny; iy++)
      for (size_t ix = 0; ix < nx; ix++) {
        const int64_t l = lab[(iz * ny + iy) * nx + ix];
        aaaiDest[iz][iy][ix] = (l == -1) ? label_undefined : (ptrdiff_t)l;
      }
  if (pv_cluster_maxima) {
    pv_cluster_maxima->resize((size_t)n_clusters);
    for (size_t c = 0; c < (size_t)n_clusters && 3 * c + 2 < maxima.size(); c++)
      (*pv_cluster_maxima)[c] = {maxima[3 * c], maxima[3 * c + 1], maxima[3 * c + 2]};
  }
  if (pv_cluster_sizes) pv_cluster_sizes->clear();            // not reported (HandleTV does not read them)
  if (pv_cluster_saliencies) pv_cluster_saliencies->clear();
  if (pReportProgress) *pReportProgress << "Number of clusters found: " << n_clusters << "\n";
  return (size_t)n_clusters;
}

// ---- oriented point cloud (`-normals-file`) -----------------------------------------------------
// The loop of HandleTV that fills `crds` / `norms` for WriteOrientedPointCloudPLY (bin/filter_mrc/handlers.cpp:2039-2309;
// the reference has no function for it, so the name is ours and the arguments are the variables of that block):
// aaafVoxel2Cluster = tomo_out.aaafI after LabelConnected, or nullptr when the voxels were not clustered.
inline void SurfacePointCloud(const int image_size[3], float const *const *const *aaafSaliency,
                              std::array<float, 3> const *const *const *aaaafDirection,
                              float const *const *const *aaafVoxel2Cluster, float const *const *const *aaafMask,
                              int select_cluster, const float voxel_width[3], float surface_normal_curve_ds,
                              bool surface_find_ridge, float max_distance_to_feature,
                              std::vector<std::array<float, 3> > &crds, std::vector<std::array<float, 3> > &norms) {
  Dense3<float, 1> sal(image_size, aaafSaliency, false), lab(image_size, aaafVoxel2Cluster, false), m(image_size, aaafMask, false);
  Dense3<std::array<float, 3>, 3> dir(image_size, aaaafDirection, false);
  const int64_t N = (int64_t)image_size[0] * image_size[1] * image_size[2];
  int64_t n = 0, cap = 1 << 16;
  std::vector<float> rows;
  for (;;) {
    rows.resize(6 * (size_t)cap);
    Check(visfd_cuda_surface_points(Context(), image_size[0], image_size[1], image_size[2], sal.data(), dir.data(), lab.data(),
                                    m.data(), select_cluster, voxel_width, surface_normal_curve_ds, surface_find_ridge ? 1 : 0,
                                    max_distance_to_feature, rows.data(), cap, &n));
    if (n <= cap) break;
    cap = std::min<int64_t>(n, N);
  }
  crds.resize((size_t)n);
  norms.resize((size_t)n);
  for (size_t i = 0; i < (size_t)n; i++) {
    crds[i] = {rows[6 * i], rows[6 * i + 1], rows[6 * i + 2]};
    norms[i] = {rows[6 * i + 3], rows[6 * i + 4], rows[6 * i + 5]};
  }
}

// TV3D<float, int, array<float,3>, float*>: feature.hpp:1631-2483
class TV3D {
  float sigma = 0.0f;
  int exponent = 4;
  float cutoff_ratio = 2.5f;
 public:
  TV3D() {}
  TV3D(float set_sigma, int set_exponent, float filter_cutoff_ratio = 2.5)
      : sigma(set_sigma), exponent(set_exponent), cutoff_ratio(filter_cutoff_ratio) {}
  void SetExponent(int set_exponent) { exponent = set_exponent; }
  void SetSigma(float set_sigma, float filter_cutoff_ratio = 2.5) {
    sigma = set_sigma;
    cutoff_ratio = filter_cutoff_ratio;
  }
  // feature.hpp:1712-1901
  void TVDenseStick(int const image_size[3], float const *const *const *aaafSaliency,
                    std::array<float, 3> const *const *const *aaaafV, float ****aaaafDest,
                    float const *const *const *aaafMaskSource = nullptr,
                    float const *const *const *aaafMaskDest = nullptr, bool detect_curves_not_surfaces = false,
                    bool normalize = true, bool diagonalize_dest = false,
                    std::ostream *pReportProgress = nullptr) {
    if (pReportProgress) *pReportProgress << "---- Begin Tensor Voting (dense, stick, CUDA) ----\n";
    Dense3<float, 1> sal(image_size, aaafSaliency, false), ms(image_size, aaafMaskSource, false),
        md(image_size, aaafMaskDest, false);
    Dense3<std::array<float, 3>, 3> v(image_size, aaaafV, false);
    DenseTensor t(image_size, aaaafDest, 6, false);
    Check(visfd_cuda_tv_dense_stick(Context(), image_size[0], image_size[1], image_size[2], sal.data(), v.data(),
                                    ms.data(), md.data(), sigma, exponent, cutoff_ratio,
                                    detect_curves_not_surfaces ? 1 : 0, normalize ? 1 : 0, diagonalize_dest ? 1 : 0,
                                    t.data()));
    t.commit();
  }
};

// ---- the fused pipeline that replaces bin/filter_mrc/handlers.cpp:1618-1892 --------------------
// tomo_in -> tomo_out (post-vote planar saliency, or the ridge saliency after the cut when
// tv_sigma <= 0).  Optional: aaaafDirection (eivects[0], handlers.cpp:1738-1740) and
// aaaafVoteTensor (for -save-progress, handlers.cpp:1897-1922).
inline float MembranePipeline(int const image_size[3], float const *const *const *aaafSource, float ***aaafDest,
                              float const *const *const *aaafMask, const visfd_membrane_params &p,
                              std::array<float, 3> ***aaaafDirection = nullptr,
                              float ****aaaafVoteTensor = nullptr, float background_sigma = 0.0f /* settings.width_b[0] */,
                              bool normalize_near_boundaries = true) {
  Dense3<float, 1> s(image_size, aaafSource, false), m(image_size, aaafMask, false), d(image_size, aaafDest, true);
  Dense3<std::array<float, 3>, 3> dir(image_size, aaaafDirection, true);
  DenseTensor t(image_size, aaaafVoteTensor, 6, false);
  float thr = 0;
  Check(visfd_cuda_membrane_background(Context(), image_size[0], image_size[1], image_size[2], s.data(), m.data(), &p,
                                       background_sigma > 0.0f ? background_sigma : 0.0f, normalize_near_boundaries ? 1 : 0,
                                       d.data(), nullptr, dir.data(), t.data(), &thr));
  d.commit();
  dir.commit();
  t.commit();
  return thr;
}

// ---- binning (lib/visfd/resample.hpp:53-166; callers handlers.cpp:2361-2425, :2321-2355) ---------
inline void BinArray3D(int const size_source[3], int const size_dest[3], float const *const *const *aaafSource,
                       float ***aaafDest, int const *offset = nullptr) {
  Dense3<float, 1> s(size_source, aaafSource, false), d(size_dest, aaafDest, true);
  const int64_t ss[3] = {size_source[0], size_source[1], size_source[2]}, ds[3] = {size_dest[0], size_dest[1], size_dest[2]};
  Check(visfd_cuda_bin3d(Context(), ss, ds, s.data(), d.data(), offset));
  d.commit();
}
inline void UnbinArray3D(int const size_source[3], int const size_dest[3], float const *const *const *aaafSource,
                         float ***aaafDest, int const *offset = nullptr) {
  Dense3<float, 1> s(size_source, aaafSource, false), d(size_dest, aaafDest, true);
  const int64_t ss[3] = {size_source[0], size_source[1], size_source[2]}, ds[3] = {size_dest[0], size_dest[1], size_dest[2]};
  Check(visfd_cuda_unbin3d(Context(), ss, ds, s.data(), d.data(), offset));
  d.commit();
}

// ---- mask rasterisation (lib/visfd/draw.hpp:90-237; caller bin/filter_mrc/filter_mrc.cpp:280-284) ----
// Region is visfd::SimpleRegion<float> (draw.hpp:41-87) or any type with the same members.
template <typename Region>
inline void DrawRegions(int const image_size[3], float ***aaafDest, float const *const *const *aaafMask,
                        const std::vector<Region> &vRegions, bool negative_means_subtract = false) {
  std::vector<visfd_region> flat(vRegions.size());
  for (size_t i = 0; i < vRegions.size(); i++) {
    const Region &r = vRegions[i];
    visfd_region &f = flat[i];
    f.value = r.value;
    for (int k = 0; k < 6; k++) f.p[k] = 0.0f;
    if (r.type == Region::SPHERE) {
      f.type = VISFD_REGION_SPHERE;
      f.p[0] = r.data.sphere.x0; f.p[1] = r.data.sphere.y0; f.p[2] = r.data.sphere.z0; f.p[3] = r.data.sphere.r;
    } else {
      f.type = VISFD_REGION_RECT;
      f.p[0] = r.data.rect.xmin; f.p[1] = r.data.rect.xmax; f.p[2] = r.data.rect.ymin;
      f.p[3] = r.data.rect.ymax; f.p[4] = r.data.rect.zmin; f.p[5] = r.data.rect.zmax;
    }
  }
  Dense3<float, 1> d(image_size, aaafDest, true), m(image_size, aaafMask, false);
  Check(visfd_cuda_draw_regions(Context(), image_size[0], image_size[1], image_size[2], d.data(), m.data(),
                                flat.data(), (int)flat.size(), negative_means_subtract ? 1 : 0));
  d.commit();
}

// ---- thresholds (lib/threshold/threshold.hpp; bin/filter_mrc/handlers.cpp:1037-1080) ------------
inline void ThresholdImage(int const image_size[3], float const *const *const *aaafIn, float ***aaafOut, int kind,
                           const float t[4], float outA, float outB, float const *const *const *aaafMask = nullptr,
                           bool use_masked_value = false, float masked_value = 0.0f) {
  Dense3<float, 1> in(image_size, aaafIn, false), m(image_size, aaafMask, false);
  Dense3<float, 1> out(image_size, aaafOut, true);
  int64_t n = (int64_t)image_size[0] * image_size[1] * image_size[2];
  Check(visfd_cuda_threshold(Context(), n, in.data(), out.data(), kind, t, outA, outB, m.data(),
                             use_masked_value ? 1 : 0, masked_value));
  out.commit();
}

}  // namespace visfd_cuda
