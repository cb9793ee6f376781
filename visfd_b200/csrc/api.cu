// api.cu -- the extern "C" entry points declared in include/visfd_cuda.h: argument
// checks, host<->device staging for the drop-in (host pointer) path, error mapping.
// All compute is in the other translation units; nothing here runs on the CPU except
// parameter generation (taps, half-widths), which the reference also does on the host.
#include <cstdlib>

#include "common.cuh"
#include "kernels.cuh"
#include <cmath>
#include <algorithm>

using namespace visfd_cuda;

#define API_BEGIN(ctx)                                         \
  try {                                                        \
    VREQUIRE((ctx) != nullptr, "context is NULL");             \
    VCK(cudaSetDevice((ctx)->device));                         \
    drop_pending_stage_events(ctx);

#define API_END(ctx)                                           \
    VCK(cudaStreamSynchronize((ctx)->stream));                 \
    resolve_stage_times(ctx);                                  \
    return 0;                                                  \
  } catch (const std::exception &ex) {                         \
    set_last_error(ex.what());                                 \
    if (ctx) { cudaStreamSynchronize((ctx)->stream); cudaGetLastError(); } \
    return 1;                                                  \
  }

static void check_dims(int64_t nx, int64_t ny, int64_t nz) {
  VREQUIRE(nx > 0 && ny > 0 && nz > 0, "image dimensions must be positive");
  VREQUIRE(nx < (1LL << 31) && ny < (1LL << 31) && nz < (1LL << 31), "image dimension too large");
}

static bool on_host(const void *p) { return p != nullptr && !is_device_pointer(p); }

void visfd_cuda::emit_blob_list(const BlobList &l, int64_t capacity, float *crds, float *sg, float *sc, int64_t *cnt) {
  int64_t n = (int64_t)l.score.size();
  if (cnt) *cnt = n;
  int64_t k = std::min(n, capacity);
  if (crds && k) memcpy(crds, l.crds.data(), 3 * k * sizeof(float));
  if (sg && k) memcpy(sg, l.sigma.data(), k * sizeof(float));
  if (sc && k) memcpy(sc, l.score.data(), k * sizeof(float));
}

extern "C" {

// ---- host-side parameter helpers ---------------------------------------------------------
void visfd_cuda_gen_gauss1d(float sigma, int hw, float *taps) { gen_gauss1d(sigma, hw, taps); }

int visfd_cuda_gauss_halfwidth(float sigma, float truncate_ratio, float truncate_threshold) {
  // bin/filter_mrc/filter3d_variants.hpp:516-518, lib/visfd/filter3d.hpp:1241-1246
  if (truncate_ratio <= 0) truncate_ratio = sqrtf(-2 * logf(truncate_threshold));  // float overloads, as in the reference
  int hw = (int)floorf(sigma * truncate_ratio);
  if (hw < 1) hw = 1;
  return hw;
}

int visfd_cuda_tv_halfwidth(float sigma, float cutoff_ratio) { return tv_halfwidth(sigma, cutoff_ratio); }

// ---- separable filters ---------------------------------------------------------------------
int visfd_cuda_apply_separable(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, const float *src,
                               float *dst, const float *mask, const float *const taps[3],
                               const int hw[3], int normalize, float *A_out) {
  API_BEGIN(ctx)
  check_dims(nx, ny, nz);
  VREQUIRE(src && dst && taps && hw, "NULL argument");
  const size_t N = (size_t)nx * ny * nz;
  const bool host = on_host(src);
  Staged<float> s(ctx, src, N, Dir::In, host), m(ctx, mask, N, Dir::In, host), d(ctx, dst, N, Dir::Out, host);
  float A = separable_device(ctx, nx, ny, nz, 0, nz, s.get(), d.get(), m.get(), taps, hw, normalize != 0,
                             nullptr, 1.0f);
  d.finish();
  if (A_out) *A_out = A;
  API_END(ctx)
}

int visfd_cuda_apply_gauss_slab(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz_local, int64_t z_offset,
                                int64_t nz_global, const float *src, float *dst, const float *mask,
                                const float sigma[3], const int hw[3], int normalize, float *A_out) {
  API_BEGIN(ctx)
  check_dims(nx, ny, nz_local);
  VREQUIRE(src && dst && sigma && hw, "NULL argument");
  const size_t N = (size_t)nx * ny * nz_local;
  const bool host = on_host(src);
  Staged<float> s(ctx, src, N, Dir::In, host), m(ctx, mask, N, Dir::In, host), d(ctx, dst, N, Dir::Out, host);
  float A = gauss_device(ctx, nx, ny, nz_local, z_offset, nz_global, s.get(), d.get(), m.get(), sigma, hw,
                         normalize != 0, nullptr, 1.0f);
  d.finish();
  if (A_out) *A_out = A;
  API_END(ctx)
}

int visfd_cuda_apply_gauss(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, const float *src, float *dst,
                           const float *mask, const float sigma[3], const int hw[3], int normalize,
                           float *A_out) {
  return visfd_cuda_apply_gauss_slab(ctx, nx, ny, nz, 0, nz, src, dst, mask, sigma, hw, normalize, A_out);
}

int visfd_cuda_apply_dog(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, const float *src, float *dst,
                         const float *mask, const float sigma_a[3], const float sigma_b[3], const int hw[3],
                         float *A_out, float *B_out) {
  API_BEGIN(ctx)
  check_dims(nx, ny, nz);
  VREQUIRE(src && dst && sigma_a && sigma_b && hw, "NULL argument");
  const size_t N = (size_t)nx * ny * nz;
  const bool host = on_host(src);
  Staged<float> s(ctx, src, N, Dir::In, host), m(ctx, mask, N, Dir::In, host), d(ctx, dst, N, Dir::Out, host);
  dog_device(ctx, nx, ny, nz, 0, nz, s.get(), d.get(), m.get(), sigma_a, sigma_b, hw, 1.0f, A_out, B_out);
  d.finish();
  API_END(ctx)
}

int visfd_cuda_apply_dog2(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, const float *src, float *dst,
                          const float *mask, const float sigma_a[3], const float sigma_b[3], const int hw_a[3],
                          const int hw_b[3], float *A_out, float *B_out) {
  API_BEGIN(ctx)
  check_dims(nx, ny, nz);
  VREQUIRE(src && dst && sigma_a && sigma_b && hw_a && hw_b, "NULL argument");
  const size_t N = (size_t)nx * ny * nz;
  const bool host = on_host(src);
  Staged<float> s(ctx, src, N, Dir::In, host), m(ctx, mask, N, Dir::In, host), d(ctx, dst, N, Dir::Out, host);
  dog_device(ctx, nx, ny, nz, 0, nz, s.get(), d.get(), m.get(), sigma_a, sigma_b, hw_a, 1.0f, A_out, B_out, hw_b);
  d.finish();
  API_END(ctx)
}

int visfd_cuda_apply_log_slab(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz_local, int64_t z_offset,
                              int64_t nz_global, const float *src, float *dst, const float *mask,
                              const float sigma[3], float delta, float truncate_ratio, float *A_out,
                              float *B_out) {
  API_BEGIN(ctx)
  check_dims(nx, ny, nz_local);
  VREQUIRE(src && dst && sigma, "NULL argument");
  const size_t N = (size_t)nx * ny * nz_local;
  const bool host = on_host(src);
  float sa[3], sb[3], scale, A = 0, B = 0;
  int hw[3];
  log_params(sigma, delta, truncate_ratio, sa, sb, hw, &scale);
  Staged<float> s(ctx, src, N, Dir::In, host), m(ctx, mask, N, Dir::In, host), d(ctx, dst, N, Dir::Out, host);
  dog_device(ctx, nx, ny, nz_local, z_offset, nz_global, s.get(), d.get(), m.get(), sa, sb, hw, scale, &A, &B);
  d.finish();
  // lib/visfd/filter3d.hpp:1500-1504: the reported peak heights are scaled as well
  if (A_out) *A_out = A * scale;
  if (B_out) *B_out = B * scale;
  API_END(ctx)
}

int visfd_cuda_apply_log(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, const float *src, float *dst,
                         const float *mask, const float sigma[3], float delta, float truncate_ratio,
                         float *A_out, float *B_out) {
  return visfd_cuda_apply_log_slab(ctx, nx, ny, nz, 0, nz, src, dst, mask, sigma, delta, truncate_ratio,
                                   A_out, B_out);
}

// ---- Hessian / eigen -------------------------------------------------------------------------
static void smooth_for_hessian(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz_local, int64_t z_offset,
                               int64_t nz_global, const float *src, const float *mask, float sigma,
                               float truncate_ratio, float *smoothed) {
  // CalcHessian, lib/visfd/feature.hpp:1223, :1248-1255: hw = floor(sigma*ratio), normalised
  int h = (int)floor(sigma * truncate_ratio);
  VREQUIRE(h >= 0, "negative Gaussian half-width");
  float sg[3] = {sigma, sigma, sigma};
  int hw[3] = {h, h, h};
  gauss_device(ctx, nx, ny, nz_local, z_offset, nz_global, src, smoothed, mask, sg, hw, true, nullptr, 1.0f);
}

int visfd_cuda_calc_hessian(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, const float *src,
                            const float *mask, float sigma, float truncate_ratio, float *gradient,
                            float *hessian) {
  API_BEGIN(ctx)
  check_dims(nx, ny, nz);
  VREQUIRE(src && (gradient || hessian), "NULL argument");
  const size_t N = (size_t)nx * ny * nz;
  const bool host = on_host(src);
  Staged<float> s(ctx, src, N, Dir::In, host), m(ctx, mask, N, Dir::In, host);
  // entries of masked voxels are left untouched => outputs are read-modify-write when masked
  Dir od = mask ? Dir::InOut : Dir::Out;
  Staged<float> g(ctx, gradient, 3 * N, od, host), h(ctx, hessian, 6 * N, od, host);
  Scratch<float> sm(ctx, N);
  smooth_for_hessian(ctx, nx, ny, nz, 0, nz, s.get(), m.get(), sigma, truncate_ratio, sm.get());
  hessian_fd_device(ctx, nx, ny, nz, 0, nz, sm.get(), m.get(), sigma, g.get(), h.get());
  g.finish();
  h.finish();
  API_END(ctx)
}

int visfd_cuda_hessian_ridge(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, const float *src,
                             const float *mask, float sigma, float truncate_ratio, int eival_order,
                             int score_kind, float *saliency, float *direction) {
  API_BEGIN(ctx)
  check_dims(nx, ny, nz);
  VREQUIRE(src && saliency, "NULL argument");
  const size_t N = (size_t)nx * ny * nz;
  const bool host = on_host(src);
  Staged<float> s(ctx, src, N, Dir::In, host), m(ctx, mask, N, Dir::In, host);
  Staged<float> sal(ctx, saliency, N, Dir::Out, host);
  Staged<float> dir(ctx, direction, 3 * N, mask ? Dir::InOut : Dir::Out, host);
  Scratch<float> sm(ctx, N);
  smooth_for_hessian(ctx, nx, ny, nz, 0, nz, s.get(), m.get(), sigma, truncate_ratio, sm.get());
  ridge_device(ctx, nx, ny, nz, 0, nz, 0, nz, sm.get(), m.get(), sigma, eival_order, score_kind, sal.get(),
               dir.get());
  sal.finish();
  dir.finish();
  API_END(ctx)
}

int visfd_cuda_tensor_score(visfd_ctx *ctx, int64_t n, const float *tensor, const float *mask,
                            int eival_order, int score_kind, int kind_is_vote_tensor, float *score,
                            float *eivals, float *direction) {
  API_BEGIN(ctx)
  VREQUIRE(n >= 0 && tensor, "bad arguments");
  const bool host = on_host(tensor);
  Staged<float> t(ctx, tensor, 6 * (size_t)n, Dir::In, host), m(ctx, mask, n, Dir::In, host);
  Dir od = mask ? Dir::InOut : Dir::Out;
  Staged<float> sc(ctx, score, n, od, host), ev(ctx, eivals, 3 * (size_t)n, od, host),
      dr(ctx, direction, 3 * (size_t)n, od, host);
  tensor_score_device(ctx, n, t.get(), m.get(), eival_order, score_kind, kind_is_vote_tensor, sc.get(),
                      ev.get(), dr.get());
  sc.finish();
  ev.finish();
  dr.finish();
  API_END(ctx)
}

// ---- saliency cut -------------------------------------------------------------------------------
int visfd_cuda_saliency_cut(visfd_ctx *ctx, int64_t n, float *saliency, const float *mask, float cut,
                            int is_fraction, float *threshold_out) {
  API_BEGIN(ctx)
  VREQUIRE(n > 0 && saliency, "bad arguments");
  const bool host = on_host(saliency);
  Staged<float> s(ctx, saliency, n, Dir::InOut, host), m(ctx, mask, n, Dir::In, host);
  float thr = cut;
  if (is_fraction) thr = select_threshold_device(ctx, n, s.get(), m.get(), cut);
  apply_cut_device(ctx, n, s.get(), thr);
  s.finish();
  if (threshold_out) *threshold_out = thr;
  API_END(ctx)
}

int visfd_cuda_select_hist(visfd_ctx *ctx, int64_t n, const float *saliency, const float *mask,
                           uint32_t prefix, int prefix_bits, uint64_t *hist) {
  API_BEGIN(ctx)
  VREQUIRE(n >= 0 && hist && (n == 0 || saliency), "bad arguments");
  const bool host = on_host(saliency);
  Staged<float> s(ctx, saliency, n, Dir::In, host), m(ctx, mask, n, Dir::In, host);
  select_hist_device(ctx, n, s.get(), m.get(), prefix, prefix_bits, hist);
  API_END(ctx)
}

int visfd_cuda_select_step(const uint64_t *hist, uint32_t *prefix, int *prefix_bits, uint64_t *rank) {
  if (!hist || !prefix || !prefix_bits || !rank) return 1;
  return select_step_host(hist, prefix, prefix_bits, rank);
}

float visfd_cuda_key_to_float(uint32_t key) { return key_to_float(key); }

// ---- tensor voting -------------------------------------------------------------------------------
int visfd_cuda_tv_dense_stick(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, const float *saliency,
                              const float *direction, const float *mask_src, const float *mask_dst,
                              float sigma, int exponent, float cutoff_ratio, int curves, int normalize,
                              int diagonalize_dest, float *tensor) {
  API_BEGIN(ctx)
  check_dims(nx, ny, nz);
  VREQUIRE(saliency && direction && tensor, "NULL argument");
  VREQUIRE(!normalize && !diagonalize_dest,
           "TVDenseStick: normalize / diagonalize_dest are not supported (filter_mrc passes false for both)");
  const size_t N = (size_t)nx * ny * nz;
  const bool host = on_host(saliency);
  Staged<float> s(ctx, saliency, N, Dir::In, host), d(ctx, direction, 3 * N, Dir::In, host),
      ms(ctx, mask_src, N, Dir::In, host), md(ctx, mask_dst, N, Dir::In, host),
      t(ctx, tensor, 6 * N, Dir::Out, host);
  TVParams p{sigma, exponent, cutoff_ratio, curves};
  tv_device(ctx, nx, ny, nz, 0, nz, 0, nz, s.get(), -INFINITY, d.get(), nullptr, 0.0f, 0, 0, ms.get(),
            md.get(), p, t.get(), nullptr);
  t.finish();
  API_END(ctx)
}

// ---- fused membrane pipeline ------------------------------------------------------------------------
// Host-resident source, no mask: upload + smoothing + ridge saliency as a pipeline over z-chunks, so
// that only the first chunk's upload is exposed (the chunk's planes plus hw+1 halo planes travel on the
// copy stream into one of two staging slabs while the previous chunk is smoothed and scored) and the
// source never has to be resident as a whole.  Every chunk is a z-slab in the sense of the header
// (global borders only at the global ends), so smoothed/saliency/direction are bit-identical to the
// single-pass result.  Returns false (nothing done) when the volume is too small to be worth it.
static bool upload_smooth_ridge_chunked(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, const float *src_host,
                                        const visfd_membrane_params *p, float *smoothed, float *saliency,
                                        float *direction) {
  const int h = (int)floor(p->sigma * p->truncate_ratio);
  VREQUIRE(h >= 0, "negative Gaussian half-width");
  const int64_t halo = h + 1;
  const char *env = getenv("VISFD_CUDA_UPLOAD_CHUNK");       // planes per chunk (tests: small chunks)
  int64_t cz = env ? std::max(1, atoi(env)) : std::max<int64_t>(64, ((nz + 15) / 16 + 7) / 8 * 8);
  if (!env && (nz < 2 * cz || nx * ny < (1 << 16))) return false;
  if (nz < 3 || cz >= nz) return false;
  const size_t plane = (size_t)nx * (size_t)ny;
  const int64_t slab_max = std::min<int64_t>(nz, cz + 2 * halo);
  Scratch<float> stage0(ctx, (size_t)slab_max * plane), stage1(ctx, (size_t)slab_max * plane);
  Scratch<float> slab_sm(ctx, (size_t)slab_max * plane);
  float *stage[2] = {stage0.get(), stage1.get()};
  if (!ctx->copy_stream) VCK(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
  const int n_chunks = (int)((nz + cz - 1) / cz);
  EventList events(ctx);   // declared after the staging slabs: drained and destroyed before they return to the pool
  std::vector<cudaEvent_t> uploaded((size_t)n_chunks), consumed((size_t)n_chunks);
  for (int c = 0; c < n_chunks; c++) {
    uploaded[(size_t)c] = events.add();
    consumed[(size_t)c] = events.add();
  }
  const float sg[3] = {p->sigma, p->sigma, p->sigma};
  const int hw[3] = {h, h, h};
  // the staging slabs come from the stream-ordered pool: whatever used them last ran on ctx->stream
  cudaEvent_t start = events.add();
  VCK(cudaEventRecord(start, ctx->stream));
  VCK(cudaStreamWaitEvent(ctx->copy_stream, start, 0));
  for (int c = 0; c < n_chunks; c++) {
    const int64_t c0 = (int64_t)c * cz, c1 = std::min(nz, c0 + cz);
    const int64_t lo = std::max<int64_t>(0, c0 - halo), hi = std::min(nz, c1 + halo);
    float *buf = stage[c & 1];
    if (c >= 2) VCK(cudaStreamWaitEvent(ctx->copy_stream, consumed[(size_t)c - 2], 0));
    VCK(cudaMemcpyAsync(buf, src_host + (size_t)lo * plane, (size_t)(hi - lo) * plane * sizeof(float),
                        cudaMemcpyHostToDevice, ctx->copy_stream));
    VCK(cudaEventRecord(uploaded[(size_t)c], ctx->copy_stream));
    VCK(cudaStreamWaitEvent(ctx->stream, uploaded[(size_t)c], 0));
    gauss_device(ctx, nx, ny, hi - lo, lo, nz, buf, slab_sm.get(), nullptr, sg, hw, true, nullptr, 1.0f);
    VCK(cudaEventRecord(consumed[(size_t)c], ctx->stream));
    VCK(cudaMemcpyAsync(smoothed + (size_t)c0 * plane, slab_sm.get() + (size_t)(c0 - lo) * plane,
                        (size_t)(c1 - c0) * plane * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream));
    // slab-local planes [c0-lo, c1-lo) of a saliency / direction array whose plane 0 is global plane lo
    ridge_device(ctx, nx, ny, hi - lo, lo, nz, c0 - lo, c1 - lo, slab_sm.get(), nullptr, p->sigma, p->eival_order,
                 VISFD_SCORE_PLANAR, saliency + (size_t)lo * plane, direction ? direction + 3 * (size_t)lo * plane : nullptr);
  }
  VCK(cudaStreamSynchronize(ctx->copy_stream));
  VCK(cudaStreamSynchronize(ctx->stream));   // before the staging slabs go back to the pool
  return true;
}

// background_sigma > 0: `-membrane-background` (handlers.cpp:1577-1592): both scores are multiplied by
// peak_height = source - Gauss(source, background_sigma) (:1698-1702, :1883-1887)
static void membrane_impl(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, const float *src, const float *mask,
                          const visfd_membrane_params *p, float background_sigma, int normalize, float *out,
                          float *hess_saliency, float *direction, float *tensor, float *threshold_out) {
  check_dims(nx, ny, nz);
  VREQUIRE(src && p && out, "NULL argument");
  const size_t N = (size_t)nx * ny * nz;
  const bool host = on_host(src);
  const bool peak = background_sigma > 0.0f;
  Staged<float> m(ctx, mask, N, Dir::In, host);
  Staged<float> o(ctx, out, N, Dir::Out, host);
  Staged<float> hs(ctx, hess_saliency, N, Dir::Out, host);
  Staged<float> dir(ctx, direction, 3 * N, mask ? Dir::InOut : Dir::Out, host);
  Staged<float> tn(ctx, tensor, 6 * N, Dir::Out, host);
  const bool vote = p->tv_sigma > 0.0f;

  Scratch<float> sm(ctx, N);
  // saliency lives in `out` when there is no voting, else in hess_saliency's buffer or scratch
  Scratch<float> sal_scratch;
  float *sal = nullptr;
  if (!vote) sal = o.get();
  else if (hs.get()) sal = hs.get();
  else { sal_scratch.reset(ctx, N); sal = sal_scratch.get(); }
  Staged<float> s_all;          // the whole source on the device: only when the peak height needs it
  Scratch<float> bg;
  if (peak) {
    s_all.init(ctx, const_cast<float *>(src), N, Dir::In, host);
    bg.reset(ctx, N);
    const float sg[3] = {background_sigma, background_sigma, background_sigma};
    const int h = (int)floorf(background_sigma * p->truncate_ratio);   // handlers.cpp:1582-1583
    const int hw[3] = {h, h, h};
    // tomo_background = tomo_in (:1580), then the blur: voxels outside the mask are never read back
    gauss_device(ctx, nx, ny, nz, 0, nz, s_all.get(), bg.get(), m.get(), sg, hw, normalize != 0, nullptr, 1.0f);
  }
  if (peak || !(host && !mask && upload_smooth_ridge_chunked(ctx, nx, ny, nz, src, p, sm.get(), sal, dir.get()))) {
    Staged<float> s_tmp;
    if (!peak) s_tmp.init(ctx, const_cast<float *>(src), N, Dir::In, host);
    const float *s = peak ? s_all.get() : s_tmp.get();
    smooth_for_hessian(ctx, nx, ny, nz, 0, nz, s, m.get(), p->sigma, p->truncate_ratio, sm.get());
    ridge_device(ctx, nx, ny, nz, 0, nz, 0, nz, sm.get(), m.get(), p->sigma, p->eival_order,
                 VISFD_SCORE_PLANAR, sal, dir.get());
    // (the pool is stream-ordered: the staged source may be recycled once the work above is queued)
  }
  if (peak) scale_by_peak_device(ctx, (i64)N, sal, s_all.get(), bg.get(), m.get());
  float thr = p->cut;
  if (p->cut_is_fraction) thr = select_threshold_device(ctx, N, sal, m.get(), p->cut);
  if (threshold_out) *threshold_out = thr;
  if (vote) {
    TVParams tp{p->tv_sigma, p->tv_exponent, p->tv_cutoff_ratio, 0};
    // voters' directions: the stored field if the caller asked for it, else recomputed
    // for the surviving ~5 % only
    // with a host `out` the result travels back chunk by chunk behind the voting kernels (not when the peak height
    // still has to multiply it)
    o.delivered = tv_device(ctx, nx, ny, nz, 0, nz, 0, nz, sal, thr, dir.get(), sm.get(), p->sigma, p->eival_order,
                            VISFD_SCORE_PLANAR, m.get(), m.get(), tp, tn.get(), o.get(), (host && !peak) ? out : nullptr);
    if (peak) scale_by_peak_device(ctx, (i64)N, o.get(), s_all.get(), bg.get(), m.get());
    if (hs.get()) apply_cut_device(ctx, N, hs.get(), thr);
  } else {
    apply_cut_device(ctx, N, sal, thr);
    if (hs.get()) VCK(cudaMemcpyAsync(hs.get(), sal, N * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream));
    VREQUIRE(!tensor, "tensor output requested without voting");
  }
  o.finish();
  hs.finish();
  dir.finish();
  tn.finish();
}

int visfd_cuda_membrane(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, const float *src,
                        const float *mask, const visfd_membrane_params *p, float *out,
                        float *hess_saliency, float *direction, float *tensor, float *threshold_out) {
  API_BEGIN(ctx)
  membrane_impl(ctx, nx, ny, nz, src, mask, p, 0.0f, 1, out, hess_saliency, direction, tensor, threshold_out);
  API_END(ctx)
}

int visfd_cuda_membrane_background(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, const float *src,
                                   const float *mask, const visfd_membrane_params *p, float background_sigma,
                                   int normalize_near_boundaries, float *out, float *hess_saliency, float *direction,
                                   float *tensor, float *threshold_out) {
  API_BEGIN(ctx)
  VREQUIRE(background_sigma >= 0.0f, "negative background width");
  membrane_impl(ctx, nx, ny, nz, src, mask, p, background_sigma, normalize_near_boundaries, out, hess_saliency, direction,
                tensor, threshold_out);
  API_END(ctx)
}

int visfd_cuda_ridge_saliency_slab(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz_local, int64_t z_offset,
                                   int64_t nz_global, const float *src, const float *mask, float sigma,
                                   float truncate_ratio, int eival_order, int score_kind, float *smoothed,
                                   float *saliency) {
  API_BEGIN(ctx)
  check_dims(nx, ny, nz_local);
  VREQUIRE(src && smoothed && saliency, "NULL argument");
  VREQUIRE(is_device_pointer(src) && is_device_pointer(smoothed) && is_device_pointer(saliency) &&
               (!mask || is_device_pointer(mask)),
           "slab entry points take device pointers only");
  smooth_for_hessian(ctx, nx, ny, nz_local, z_offset, nz_global, src, mask, sigma, truncate_ratio, smoothed);
  // planes whose +-1 neighbours exist in the slab (or are clamped at the global border)
  int64_t z0 = (z_offset == 0) ? 0 : 1;
  int64_t z1 = (z_offset + nz_local == nz_global) ? nz_local : nz_local - 1;
  const size_t plane = (size_t)nx * ny;
  if (z0 > 0) VCK(cudaMemsetAsync(saliency, 0, plane * sizeof(float), ctx->stream));
  if (z1 < nz_local) VCK(cudaMemsetAsync(saliency + (size_t)z1 * plane, 0, plane * sizeof(float), ctx->stream));
  if (z1 > z0)
    ridge_device(ctx, nx, ny, nz_local, z_offset, nz_global, z0, z1, smoothed, mask, sigma, eival_order,
                 score_kind, saliency, nullptr);
  API_END(ctx)
}

}  // extern "C"

namespace visfd_cuda {
void vote_slab_device(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz_local, int64_t z_offset, int64_t nz_global,
                      int64_t own_z0, int64_t own_z1, int64_t vote_z0, int64_t vote_z1, const float *saliency,
                      const float *smoothed, const float *mask, float threshold, const visfd_membrane_params *p,
                      float *out, float *tensor, float *out_host, const float *peak) {
  VREQUIRE(!out_host || !is_device_pointer(out_host), "out_host must be a host pointer");
  check_dims(nx, ny, nz_local);
  VREQUIRE(saliency && smoothed && p && out, "NULL argument");
  VREQUIRE(is_device_pointer(saliency) && is_device_pointer(smoothed) && is_device_pointer(out),
           "slab entry points take device pointers only");
  VREQUIRE(0 <= vote_z0 && vote_z0 <= own_z0 && own_z0 <= own_z1 && own_z1 <= vote_z1 && vote_z1 <= nz_local,
           "plane ranges must nest: 0 <= vote_z0 <= own_z0 <= own_z1 <= vote_z1 <= nz_local");
  const size_t plane = (size_t)nx * ny;
  const size_t n_own = plane * (size_t)(own_z1 - own_z0);
  bool delivered = false;
  if (p->tv_sigma > 0.0f) {
    // direction recompute reads smoothed planes vote_z0-1 .. vote_z1 (clamped at the global border)
    VREQUIRE((vote_z0 >= 1 || z_offset == 0) && (vote_z1 <= nz_local - 1 || z_offset + nz_local == nz_global),
             "slab lacks the 1-plane halo around the voter planes");
    TVParams tp{p->tv_sigma, p->tv_exponent, p->tv_cutoff_ratio, 0};
    // The voter list is ordered by 4^3 brick and float sums depend on the order, so the voter planes
    // start on a GLOBAL multiple of 8 whenever the slab has the planes for it (the extra ones are out of
    // every receiver's reach): with receiver planes that start on a multiple of 4 as well, a slab then
    // reproduces the undivided volume bit for bit.
    int64_t v0 = vote_z0 - (z_offset + vote_z0) % 8;
    if (v0 < 0 || (v0 < 1 && z_offset != 0)) v0 = vote_z0;
    const size_t o = plane * (size_t)v0;
    if (tv_device(ctx, nx, ny, vote_z1 - v0, z_offset + v0, nz_global, own_z0 - v0,
              own_z1 - v0, saliency + o, threshold, nullptr, smoothed + o, p->sigma, p->eival_order,
              VISFD_SCORE_PLANAR, mask ? mask + o : nullptr, mask ? mask + o : nullptr, tp, tensor, out, out_host,
              peak ? peak + o : nullptr))
      delivered = true;
  } else {
    VCK(cudaMemcpyAsync(out, saliency + plane * (size_t)own_z0, n_own * sizeof(float), cudaMemcpyDeviceToDevice,
                        ctx->stream));
    apply_cut_device(ctx, n_own, out, threshold);
  }
  if (out_host && !delivered) {
    VCK(cudaMemcpyAsync(out_host, out, n_own * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    VCK(cudaStreamSynchronize(ctx->stream));
  }
}
}  // namespace visfd_cuda

extern "C" {

int visfd_cuda_vote_slab_host(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz_local, int64_t z_offset,
                              int64_t nz_global, int64_t own_z0, int64_t own_z1, int64_t vote_z0, int64_t vote_z1,
                              const float *saliency, const float *smoothed, const float *mask, float threshold,
                              const visfd_membrane_params *p, float *out, float *tensor, float *out_host) {
  API_BEGIN(ctx)
  vote_slab_device(ctx, nx, ny, nz_local, z_offset, nz_global, own_z0, own_z1, vote_z0, vote_z1, saliency, smoothed,
                   mask, threshold, p, out, tensor, out_host, nullptr);
  API_END(ctx)
}

int visfd_cuda_vote_slab(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz_local, int64_t z_offset,
                         int64_t nz_global, int64_t own_z0, int64_t own_z1, int64_t vote_z0, int64_t vote_z1,
                         const float *saliency, const float *smoothed, const float *mask, float threshold,
                         const visfd_membrane_params *p, float *out, float *tensor) {
  return visfd_cuda_vote_slab_host(ctx, nx, ny, nz_local, z_offset, nz_global, own_z0, own_z1, vote_z0, vote_z1,
                                   saliency, smoothed, mask, threshold, p, out, tensor, nullptr);
}

// ---- threshold / mask maps --------------------------------------------------------------------------
int visfd_cuda_threshold(visfd_ctx *ctx, int64_t n, const float *in, float *out, int kind, const float t[4],
                         float outA, float outB, const float *mask, int use_masked_value, float masked_value) {
  API_BEGIN(ctx)
  VREQUIRE(n >= 0 && out && (in || kind == VISFD_RESCALE), "bad arguments");
  const bool host = on_host(out);
  Staged<float> i(ctx, in, n, Dir::In, host), m(ctx, mask, n, Dir::In, host);
  Staged<float> o(ctx, out, n, kind == VISFD_RESCALE ? Dir::InOut : Dir::Out, host);
  threshold_device(ctx, n, i.get(), o.get(), kind, t, outA, outB, m.get(), use_masked_value, masked_value);
  o.finish();
  API_END(ctx)
}

int visfd_cuda_bin3d(visfd_ctx *ctx, const int64_t size_src[3], const int64_t size_dst[3], const float *src,
                     float *dst, const int *offset) {
  API_BEGIN(ctx)
  VREQUIRE(size_src && size_dst && src && dst, "NULL argument");
  const size_t ns = (size_t)size_src[0] * size_src[1] * size_src[2], nd = (size_t)size_dst[0] * size_dst[1] * size_dst[2];
  const bool host = on_host(src);
  Staged<float> s(ctx, src, ns, Dir::In, host);
  Staged<float> d(ctx, dst, nd, Dir::Out, host);
  bin3d_device(ctx, size_src, size_dst, s.get(), d.get(), offset);
  d.finish();
  API_END(ctx)
}

int visfd_cuda_unbin3d(visfd_ctx *ctx, const int64_t size_src[3], const int64_t size_dst[3], const float *src,
                       float *dst, const int *offset) {
  API_BEGIN(ctx)
  VREQUIRE(size_src && size_dst && src && dst, "NULL argument");
  const size_t ns = (size_t)size_src[0] * size_src[1] * size_src[2], nd = (size_t)size_dst[0] * size_dst[1] * size_dst[2];
  const bool host = on_host(src);
  Staged<float> s(ctx, src, ns, Dir::In, host);
  Staged<float> d(ctx, dst, nd, Dir::Out, host);
  unbin3d_device(ctx, size_src, size_dst, s.get(), d.get(), offset);
  d.finish();
  API_END(ctx)
}

int visfd_cuda_draw_regions(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, float *image, const float *mask,
                            const visfd_region *regions, int n_regions, int negative_means_subtract) {
  API_BEGIN(ctx)
  check_dims(nx, ny, nz);
  VREQUIRE(image && (regions || n_regions == 0) && n_regions >= 0, "bad argument");
  const size_t N = (size_t)nx * ny * nz;
  const bool host = on_host(image);
  Staged<float> img(ctx, image, N, Dir::InOut, host), m(ctx, mask, N, Dir::In, host);
  draw_regions_device(ctx, nx, ny, nz, img.get(), m.get(), regions, n_regions, negative_means_subtract != 0);
  img.finish();
  API_END(ctx)
}

int visfd_cuda_moment_sums(visfd_ctx *ctx, int64_t n, const float *in, const float *weights, double center,
                           int squared, double sums[2]) {
  API_BEGIN(ctx)
  VREQUIRE(n >= 0 && (in || n == 0) && sums, "bad arguments");
  const bool host = on_host(in);
  Staged<float> i(ctx, in, n, Dir::In, host), w(ctx, weights, n, Dir::In, host);
  moment_sums_device(ctx, n, i.get(), w.get(), center, squared != 0, sums);
  API_END(ctx)
}

int visfd_cuda_mean_stddev(visfd_ctx *ctx, int64_t n, const float *in, const float *weights, float *mean_out,
                           float *stddev_out) {
  API_BEGIN(ctx)
  VREQUIRE(n > 0 && in, "bad arguments");
  const bool host = on_host(in);
  Staged<float> i(ctx, in, n, Dir::In, host), w(ctx, weights, n, Dir::In, host);
  mean_stddev_device(ctx, n, i.get(), w.get(), mean_out, stddev_out);
  API_END(ctx)
}

// ---- blob detection ------------------------------------------------------------------------------------
int visfd_cuda_blob_dog(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, const float *src, const float *mask,
                        const float *sigmas, int n_sigmas, float delta, float truncate_ratio,
                        float minima_threshold, float maxima_threshold, int use_threshold_ratios,
                        int64_t capacity, float *min_crds, float *min_sigma, float *min_score,
                        int64_t *n_minima, float *max_crds, float *max_sigma, float *max_score,
                        int64_t *n_maxima) {
  API_BEGIN(ctx)
  check_dims(nx, ny, nz);
  VREQUIRE(src && sigmas && n_sigmas >= 0 && capacity >= 0, "bad arguments");
  const size_t N = (size_t)nx * ny * nz;
  const bool host = on_host(src);
  Staged<float> s(ctx, src, N, Dir::In, host), m(ctx, mask, N, Dir::In, host);
  BlobList mins, maxs;
  blob_dog_device(ctx, nx, ny, nz, 0, nz, 0, nz, s.get(), m.get(), sigmas, n_sigmas, delta, truncate_ratio,
                  minima_threshold, maxima_threshold, use_threshold_ratios, mins, maxs, true, nullptr);
  emit_blob_list(mins, capacity, min_crds, min_sigma, min_score, n_minima);
  emit_blob_list(maxs, capacity, max_crds, max_sigma, max_score, n_maxima);
  API_END(ctx)
}

int visfd_cuda_blob_dog_slab(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz_local, int64_t z_offset,
                             int64_t nz_global, int64_t own_z0, int64_t own_z1, const float *src, const float *mask,
                             const float *sigmas, int n_sigmas, float delta, float truncate_ratio,
                             float minima_threshold, float maxima_threshold, int use_threshold_ratios,
                             int64_t capacity, float *min_crds, float *min_sigma, float *min_score,
                             int64_t *n_minima, float *max_crds, float *max_sigma, float *max_score,
                             int64_t *n_maxima, float *best_scores) {
  API_BEGIN(ctx)
  check_dims(nx, ny, nz_local);
  VREQUIRE(src && sigmas && n_sigmas >= 0 && capacity >= 0 && best_scores, "bad arguments");
  VREQUIRE(is_device_pointer(src) && (!mask || is_device_pointer(mask)), "slab entry points take device pointers only");
  BlobList mins, maxs;
  blob_dog_device(ctx, nx, ny, nz_local, z_offset, nz_global, own_z0, own_z1, src, mask, sigmas, n_sigmas, delta,
                  truncate_ratio, minima_threshold, maxima_threshold, use_threshold_ratios, mins, maxs, false,
                  best_scores);
  emit_blob_list(mins, capacity, min_crds, min_sigma, min_score, n_minima);
  emit_blob_list(maxs, capacity, max_crds, max_sigma, max_score, n_maxima);
  API_END(ctx)
}

int visfd_cuda_blob_finalize(float minima_threshold, float maxima_threshold, int use_threshold_ratios,
                             float best_min_score, float best_max_score, float *min_crds, float *min_sigma,
                             float *min_score, int64_t *n_minima, float *max_crds, float *max_sigma,
                             float *max_score, int64_t *n_maxima) {
  try {
    VREQUIRE(n_minima && n_maxima && *n_minima >= 0 && *n_maxima >= 0, "bad arguments");
    auto load = [](const float *crds, const float *sg, const float *sc, int64_t n) {
      BlobList l;
      VREQUIRE(n == 0 || (crds && sg && sc), "NULL list");
      l.crds.assign(crds, crds + 3 * n);
      l.sigma.assign(sg, sg + n);
      l.score.assign(sc, sc + n);
      return l;
    };
    BlobList mins = load(min_crds, min_sigma, min_score, *n_minima), maxs = load(max_crds, max_sigma, max_score, *n_maxima);
    blob_final_filter(mins, maxs, minima_threshold, maxima_threshold, use_threshold_ratios, best_min_score,
                      best_max_score);
    emit_blob_list(mins, *n_minima, min_crds, min_sigma, min_score, n_minima);
    emit_blob_list(maxs, *n_maxima, max_crds, max_sigma, max_score, n_maxima);
    return 0;
  } catch (const std::exception &ex) {
    set_last_error(ex.what());
    return 1;
  }
}

// ---- bookkeeping -------------------------------------------------------------------------------------------
int64_t visfd_cuda_last_voter_count(visfd_ctx *ctx) { return ctx ? ctx->last_voters : -1; }
int visfd_cuda_last_tv_kernel(visfd_ctx *ctx) { return ctx ? ctx->last_tv_kernel : -1; }

int visfd_cuda_tv_count_pairs(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, const float *saliency,
                              float threshold, const float *mask_src, const float *mask_dst, int halfwidth,
                              int64_t recv_z0, int64_t recv_z1, int64_t *pairs) {
  API_BEGIN(ctx)
  check_dims(nx, ny, nz);
  VREQUIRE(saliency && pairs, "NULL argument");
  const size_t N = (size_t)nx * ny * nz;
  const bool host = on_host(saliency);
  Staged<float> s(ctx, saliency, N, Dir::In, host), ms(ctx, mask_src, N, Dir::In, host),
      md(ctx, mask_dst, N, Dir::In, host);
  VREQUIRE(0 <= recv_z0 && recv_z0 <= recv_z1 && recv_z1 <= nz, "receiver planes outside the volume");
  *pairs = tv_count_pairs_device(ctx, nx, ny, nz, s.get(), threshold, ms.get(), md.get(), halfwidth,
                                 (int)recv_z0, (int)recv_z1);
  API_END(ctx)
}

int visfd_cuda_fp32_peak(visfd_ctx *ctx, double ms, double *tflops) {
  API_BEGIN(ctx)
  VREQUIRE(tflops, "NULL argument");
  *tflops = fp32_peak_device(ctx, ms, 0);
  API_END(ctx)
}

int visfd_cuda_fp32_peak_packed(visfd_ctx *ctx, double ms, double *tflops) {
  API_BEGIN(ctx)
  VREQUIRE(tflops, "NULL argument");
  *tflops = fp32_peak_device(ctx, ms, 1);
  API_END(ctx)
}

int visfd_cuda_fp32_peak_3op(visfd_ctx *ctx, double ms, double *tflops) {
  API_BEGIN(ctx)
  VREQUIRE(tflops, "NULL argument");
  *tflops = fp32_peak_device(ctx, ms, 2);
  API_END(ctx)
}

}  // extern "C"
