// kernels.cuh -- internal (device-pointer level) interface between the .cu files.
// Everything here works on DEVICE memory of ctx's GPU and enqueues on ctx->stream;
// the extern "C" layer in api.cu adds host staging, argument checks and timing.
#pragma once
#include <functional>

#include "common.cuh"

namespace visfd_cuda {

// ---- gauss.cu ---------------------------------------------------------------------
void gen_gauss1d(float sigma, int hw, float *taps);
float separable_device(visfd_ctx *ctx, i64 nx, i64 ny, i64 nz_local, i64 z_offset, i64 nz_global,
                       const float *src, float *dst, const float *mask, const float *const taps[3],
                       const int hw[3], bool normalize, const float *combine_minuend,
                       float combine_scale, bool z_swept = false /* dst already holds the Z sweep (dog_device) */);
// Device bytes separable_device (and gauss_device) takes from the pool for a slab of nz_local planes.
size_t separable_workspace_bytes(i64 nx, i64 ny, i64 nz_local, const int hw[3], bool masked, bool normalize);
float gauss_device(visfd_ctx *ctx, i64 nx, i64 ny, i64 nz_local, i64 z_offset, i64 nz_global,
                   const float *src, float *dst, const float *mask, const float sigma[3],
                   const int hw[3], bool normalize, const float *combine_minuend,
                   float combine_scale, bool z_swept = false);
void dog_device(visfd_ctx *ctx, i64 nx, i64 ny, i64 nz_local, i64 z_offset, i64 nz_global,
                const float *src, float *dst, const float *mask, const float sigma_a[3],
                const float sigma_b[3], const int hw[3], float scale, float *A, float *B,
                const int *hw_b = nullptr /* half-width of the second Gaussian if it differs (filter_mrc's -dog) */);
void log_params(const float sigma[3], float delta, float truncate_ratio, float sigma_a[3],
                float sigma_b[3], int hw[3], float *scale);
void fill_device(visfd_ctx *ctx, float *p, float v, i64 n);

// ---- ridge.cu ---------------------------------------------------------------------
// Finite-difference gradient / Hessian of a smoothed slab (CalcHessian's second half).
void hessian_fd_device(visfd_ctx *ctx, i64 nx, i64 ny, i64 nz_local, i64 z_offset, i64 nz_global,
                       const float *smoothed, const float *mask, float sigma, float *gradient,
                       float *hessian);
// Fused finite-difference Hessian + eigen + score on planes [z0,z1) of a smoothed slab.
// saliency/direction/eivals are indexed like the slab (plane z at offset z*ny*nx);
// direction and eivals may be NULL.
void ridge_device(visfd_ctx *ctx, i64 nx, i64 ny, i64 nz_local, i64 z_offset, i64 nz_global,
                  i64 z0, i64 z1, const float *smoothed, const float *mask, float sigma,
                  int eival_order, int score_kind, float *saliency, float *direction);
// Per-voxel eigen + score of a stored tensor image (N*6).
void tensor_score_device(visfd_ctx *ctx, i64 n, const float *tensor, const float *mask,
                         int eival_order, int score_kind, int is_vote_tensor, float *score,
                         float *eivals, float *direction);

// ---- select.cu --------------------------------------------------------------------
constexpr int HIST_BINS = 2048;
void select_hist_device(visfd_ctx *ctx, i64 n, const float *sal, const float *mask,
                        uint32_t prefix, int prefix_bits, uint64_t *hist_host /*HIST_BINS*/);
int select_step_host(const uint64_t *hist, uint32_t *prefix, int *prefix_bits, uint64_t *rank);
uint32_t float_to_key(float f);
float key_to_float(uint32_t k);
// count of un-masked voxels
i64 count_unmasked_device(visfd_ctx *ctx, i64 n, const float *mask);
// Threshold such that the reference's cut (handlers.cpp:1751-1797) is reproduced, by a radix select over
// histograms that summed_hist fills: the HIST_BINS-bin histogram of the keys that match the prefix, summed
// over every part of the volume (select_hist_device on each part).  *n_at_or_above (if given): the number of
// un-masked voxels whose saliency is at or above the threshold, ties included.
float select_threshold(float fraction,
                       const std::function<void(uint32_t prefix, int prefix_bits, uint64_t *hist)> &summed_hist,
                       uint64_t *n_at_or_above = nullptr);
float select_threshold_device(visfd_ctx *ctx, i64 n, const float *sal, const float *mask,
                              float fraction);
void apply_cut_device(visfd_ctx *ctx, i64 n, float *sal, float thr);
// score *= src - background where mask != 0 (mask may be NULL); background == NULL: src is the peak height itself
void scale_by_peak_device(visfd_ctx *ctx, i64 n, float *score, const float *src, const float *background, const float *mask);

// ---- tv.cu ------------------------------------------------------------------------
struct TVParams {
  float sigma;
  int exponent;
  float cutoff_ratio;
  int curves;
};
// Dense stick voting on a slab.  Voters: every slab voxel with saliency >= thr,
// saliency != 0 and mask_src != 0.  Receivers: planes [own_z0, own_z1) of the slab with
// mask_dst != 0.  direction: N*3 (slab) or NULL, in which case the voters' directions
// are recomputed from `smoothed` (fused pipeline: finite-difference Hessian + eigenvector
// with ridge_sigma / eival_order).  tensor (optional): (own_z1-own_z0)*ny*nx*6.
// score (optional): (own_z1-own_z0)*ny*nx floats = ScoreTensorPlanar/Linear of the vote
// tensor diagonalised with eival_order.  score_host (optional, HOST pointer of the same
// size): the receiver planes are voted in up to 8 chunks and every finished chunk of
// `score` is copied to score_host on a second stream while the next chunk is computed;
// returns true if score_host has been filled that way.  peak (optional, N floats indexed like the slab): the score
// of every receiver with mask_dst != 0 is multiplied by its peak height (`-membrane-background`), chunk by chunk
// before the chunk's copy to score_host.
bool tv_device(visfd_ctx *ctx, i64 nx, i64 ny, i64 nz_local, i64 z_offset, i64 nz_global,
               i64 own_z0, i64 own_z1, const float *saliency, float thr, const float *direction,
               const float *smoothed, float ridge_sigma, int eival_order, int score_kind,
               const float *mask_src, const float *mask_dst, const TVParams &p, float *tensor,
               float *score, float *score_host = nullptr, const float *peak = nullptr);
// Upper bound of the device bytes tv_device takes from the pool for a slab of nz_local voter planes, own_planes
// receiver planes and at most n_voters voters: the voter list (48 B per voter), its brick offsets and the rest.
size_t tv_workspace_bytes(i64 nx, i64 ny, i64 nz_local, i64 own_planes, uint64_t n_voters);
int tv_halfwidth(float sigma, float cutoff_ratio);

// ---- api.cu -----------------------------------------------------------------------
// visfd_cuda_vote_slab_host without its API frame (the slab drivers of multi.cu).  peak (optional, nz_local*ny*nx
// floats like saliency): the voted score is multiplied by the peak height (tv_device); without voting the saliency
// is expected to carry it already.
void vote_slab_device(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz_local, int64_t z_offset, int64_t nz_global,
                      int64_t own_z0, int64_t own_z1, int64_t vote_z0, int64_t vote_z1, const float *saliency,
                      const float *smoothed, const float *mask, float threshold, const visfd_membrane_params *p,
                      float *out, float *tensor, float *out_host, const float *peak);

// ---- threshold.cu -----------------------------------------------------------------
void threshold_device(visfd_ctx *ctx, i64 n, const float *in, float *out, int kind,
                      const float t[4], float outA, float outB, const float *mask,
                      int use_masked_value, float masked_value);
void mean_stddev_device(visfd_ctx *ctx, i64 n, const float *in, const float *w, float *mean,
                        float *stddev);
void moment_sums_device(visfd_ctx *ctx, i64 n, const float *in, const float *w, double center, bool squared,
                        double sums[2]);

// ---- resample.cu ------------------------------------------------------------------
// BinArray3D / UnbinArray3D (lib/visfd/resample.hpp:53-166); sizes are {nx, ny, nz}.
void bin3d_device(visfd_ctx *ctx, const i64 size_src[3], const i64 size_dst[3], const float *src, float *dst,
                  const int *offset);
void unbin3d_device(visfd_ctx *ctx, const i64 size_src[3], const i64 size_dst[3], const float *src, float *dst,
                    const int *offset);

// ---- draw.cu ----------------------------------------------------------------------
// DrawRegions (lib/visfd/draw.hpp:90-237), in place on a device image; `regions` is a host array.
void draw_regions_device(visfd_ctx *ctx, i64 nx, i64 ny, i64 nz, float *img, const float *mask,
                         const visfd_region *regions, int n_regions, bool negative_means_subtract);

// ---- blob.cu ----------------------------------------------------------------------
struct BlobList {
  std::vector<float> crds, sigma, score;  // crds: 3 per entry (x,y,z)
};
// slab form (whole image: z_offset 0, nz_global = nz, own planes [0, nz), finalize true); best: NULL or 2 floats
void blob_dog_device(visfd_ctx *ctx, i64 nx, i64 ny, i64 nz, i64 z_offset, i64 nz_global, i64 own_z0, i64 own_z1,
                     const float *src, const float *mask,
                     const float *sigmas, int n_sigmas, float delta, float truncate_ratio,
                     float minima_threshold, float maxima_threshold, int use_threshold_ratios,
                     BlobList &minima, BlobList &maxima, bool finalize, float best[2]);
void blob_final_filter(BlobList &minima, BlobList &maxima, float minima_threshold, float maxima_threshold,
                       int use_threshold_ratios, float gmin, float gmax);

// ---- util.cu ----------------------------------------------------------------------
i64 tv_count_pairs_device(visfd_ctx *ctx, i64 nx, i64 ny, i64 nz, const float *sal, float thr,
                          const float *mask_src, const float *mask_dst, int hw, int recv_z0, int recv_z1);
double fp32_peak_device(visfd_ctx *ctx, double ms_target, int mode);  // 0 FFMA chains, 1 packed FFMA2, 2 three register operands

}  // namespace visfd_cuda
