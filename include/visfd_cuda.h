/* visfd_cuda.h -- C ABI of the B200 (sm_100a) implementation of visfd's
 * filter_mrc membrane / blob hot path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++ or torch types.
 * Every entry point names the reference interface it replaces (paths are into
 * the jewettaij/visfd tree).  The C++ mirror of the reference's `namespace visfd`
 * template API that forwards to these symbols is visfd_b200/csrc/visfd_cuda_shim.hpp;
 * INTEGRATION.md shows the reference-side patch.
 *
 * Conventions
 *  - Volumes are dense row-major float32 [nz][ny][nx] (x fastest), exactly the
 *    contiguous block behind Alloc3D<float> (lib/visfd/alloc3d.hpp:25-67).
 *  - Vector fields are AoS float[N][3] (array<float,3>***), tensors AoS
 *    float[N][6] in flat order xx,yy,zz,xy,yz,xz (lib/visfd/lin3_utils.hpp:400-406).
 *  - Masks are float volumes: 0 = ignore, anything else = weight
 *    (lib/visfd/filter1d.hpp:273-275).  NULL = no mask.
 *  - Every array argument may be a HOST pointer (the library stages it through
 *    device memory: this is the drop-in path) or a DEVICE pointer on the
 *    context's GPU (no copies: the resident path used by the multi-GPU driver
 *    and the benchmark).  All arrays of one call must be of the same kind.
 *  - All sizes are 64-bit; the reference's `int` limits (alloc3d.hpp:33-35,
 *    multichannel_image3d.hpp:126-133) do not apply.
 *  - DEVICE arrays: the library works on its own non-blocking stream (or the one
 *    given to visfd_cuda_set_stream), so work the caller still has in flight on
 *    OTHER streams that produces an input must be finished (stream or event
 *    synchronised) before the call; outputs are complete on return.
 *  - Calls are synchronous (results are complete on return) and return 0 on
 *    success, non-zero on failure with a message in visfd_cuda_last_error().
 *    The C++ shim rethrows it as VisfdErr (lib/visfd/err_visfd.hpp:15-22).
 *  - There is no CPU fallback: without a usable CUDA device every call fails.
 *
 * Z-slab form.  Entry points ending in _slab operate on a slab of nz_local
 * planes that represents global planes [z_offset, z_offset+nz_local) of a volume
 * with nz_global planes: image-border behaviour (zero extension + renormalisation,
 * clamped finite-difference stencils) is applied at the GLOBAL borders only, so a
 * slab carrying a halo of at least the stencil radius reproduces the single-volume
 * result on its interior planes.  The non-slab forms are the slab forms with
 * z_offset = 0 and nz_global = nz.
 */
#ifndef VISFD_CUDA_H
#define VISFD_CUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct visfd_ctx visfd_ctx;

#define VISFD_INCREASING_EIVALS 0 /* selfadjoint_eigen3::INCREASING_EIVALS, eigen3_simple.hpp:36-43 */
#define VISFD_DECREASING_EIVALS 1 /* selfadjoint_eigen3::DECREASING_EIVALS */

#define VISFD_SCORE_PLANAR 0 /* ScoreHessianPlanar / ScoreTensorPlanar, feature.hpp:1529, 1593 */
#define VISFD_SCORE_LINEAR 1 /* ScoreHessianLinear / ScoreTensorLinear, feature.hpp:1572, 1610 */

/* ---- context -------------------------------------------------------------- */
int visfd_cuda_version(void);
/* Number of CUDA devices this process can see (0 if none / no driver). */
int visfd_cuda_device_count(void);
/* One context per GPU.  device < 0 selects the current device. */
int visfd_cuda_init(int device, visfd_ctx **ctx);
void visfd_cuda_destroy(visfd_ctx *ctx);
const char *visfd_cuda_last_error(void);
/* Use an existing stream (cudaStream_t passed as void*) for all work of ctx. */
int visfd_cuda_set_stream(visfd_ctx *ctx, void *cuda_stream);
/* Separable-filter arithmetic.  0 (default): every tap is a separate IEEE multiply and
 * add in the reference's accumulation order, so Gaussian / DoG / LoG outputs are
 * bit-identical to the reference's x86-64 build.  1: one fused multiply-add per tap
 * (half the FP32 instructions; differences ~1e-7 of the image scale).  The environment
 * variable VISFD_CUDA_FAST_GAUSS=1 sets the initial value. */
void visfd_cuda_set_fast_gauss(visfd_ctx *ctx, int enabled);
/* Release cached device workspace. */
int visfd_cuda_trim(visfd_ctx *ctx);
/* Number of kernel launches issued by ctx since creation (bench bookkeeping). */
int64_t visfd_cuda_launch_count(visfd_ctx *ctx);
/* Device milliseconds spent in a named stage since the last visfd_cuda_reset_stage_ms,
 * measured with CUDA events on the context's stream around the stage's kernels:
 * "gauss", "ridge", "select", "compact", "tv", "threshold", "blob_scan", "h2d", "d2h".
 * Returns -1 for a stage that has not run. */
double visfd_cuda_stage_ms(visfd_ctx *ctx, const char *stage);
void visfd_cuda_reset_stage_ms(visfd_ctx *ctx);

/* ---- host-side parameter helpers (no GPU work) ----------------------------- */
/* GenFilterGauss1D<float>(sigma, halfwidth): lib/visfd/filter1d.hpp:411-460.
 * taps[i+hw], i = -hw..hw. */
void visfd_cuda_gen_gauss1d(float sigma, int hw, float *taps);
/* Halfwidth rules: max(1,floor(sigma*ratio)) (lib/visfd/filter3d.hpp:1241-1246);
 * ratio <= 0 means ratio = sqrt(-2 ln threshold)
 * (bin/filter_mrc/filter3d_variants.hpp:500-528). */
int visfd_cuda_gauss_halfwidth(float sigma, float truncate_ratio, float truncate_threshold);
/* TV3D::SetSigma: hw = floor(sigma*cutoff_ratio), lib/visfd/feature.hpp:1669-1675 */
int visfd_cuda_tv_halfwidth(float sigma, float cutoff_ratio);

/* ---- separable filters ----------------------------------------------------- */
/* ApplySeparable<float>: lib/visfd/filter3d.hpp:688-1050.
 * taps[d] -> 2*hw[d]+1 floats (host memory), d = 0:x 1:y 2:z.  *A_out (may be
 * NULL) receives the returned peak height. */
int visfd_cuda_apply_separable(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz,
                               const float *src, float *dst, const float *mask,
                               const float *const taps[3], const int hw[3],
                               int normalize, float *A_out);
/* ApplyGauss<float>(sigma[3], truncate_halfwidth[3]): lib/visfd/filter3d.hpp:1088-1124
 * (the other three overloads, :1163, :1228, :1299, and the filter_mrc variant,
 * filter3d_variants.hpp:500-528, are argument adapters over this one). */
int visfd_cuda_apply_gauss(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz,
                           const float *src, float *dst, const float *mask,
                           const float sigma[3], const int hw[3], int normalize,
                           float *A_out);
int visfd_cuda_apply_gauss_slab(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz_local,
                                int64_t z_offset, int64_t nz_global, const float *src,
                                float *dst, const float *mask, const float sigma[3],
                                const int hw[3], int normalize, float *A_out);
/* (All separable filters: with DEVICE pointers dst must not alias src or mask -- the call fails otherwise;
 * host arrays are staged through separate device buffers and may alias as in the reference.) */
/* ApplyDog<float>: lib/visfd/filter3d.hpp:1340-1402 */
int visfd_cuda_apply_dog(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz,
                         const float *src, float *dst, const float *mask,
                         const float sigma_a[3], const float sigma_b[3], const int hw[3],
                         float *A_out, float *B_out);
/* filter_mrc's own ApplyDog (bin/filter_mrc/filter3d_variants.hpp:542-597, caller HandleDog handlers.cpp:309-320):
 * each Gaussian with the half-width derived from its OWN sigma. */
int visfd_cuda_apply_dog2(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz,
                          const float *src, float *dst, const float *mask,
                          const float sigma_a[3], const float sigma_b[3], const int hw_a[3],
                          const int hw_b[3], float *A_out, float *B_out);
/* ApplyLog<float>: lib/visfd/filter3d.hpp:1430-1507 */
int visfd_cuda_apply_log(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz,
                         const float *src, float *dst, const float *mask,
                         const float sigma[3], float delta_sigma_over_sigma,
                         float truncate_ratio, float *A_out, float *B_out);
int visfd_cuda_apply_log_slab(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz_local,
                              int64_t z_offset, int64_t nz_global, const float *src,
                              float *dst, const float *mask, const float sigma[3],
                              float delta_sigma_over_sigma, float truncate_ratio,
                              float *A_out, float *B_out);

/* ---- Hessian, eigensolve, ridge saliency ------------------------------------ */
/* CalcHessian<float, array<float,3>, float*>: lib/visfd/feature.hpp:1210-1348.
 * gradient (N*3) and hessian (N*6) may each be NULL.  Entries of voxels whose
 * mask is 0 are left untouched. */
int visfd_cuda_calc_hessian(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz,
                            const float *src, const float *mask, float sigma,
                            float truncate_ratio, float *gradient, float *hessian);
/* The per-voxel loop of HandleTV, bin/filter_mrc/handlers.cpp:1645-1746, fused
 * with CalcHessian: smooth, finite-difference Hessian, ConvertFlatSym2Evects3
 * (lib/visfd/eigen3_simple.hpp:392) and ScoreHessianPlanar/Linear, without
 * writing the 6-component tensor.  saliency: N floats (0 where mask==0);
 * direction: N*3 floats = eivects[0] (may be NULL; untouched where mask==0). */
int visfd_cuda_hessian_ridge(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz,
                             const float *src, const float *mask, float sigma,
                             float truncate_ratio, int eival_order, int score_kind,
                             float *saliency, float *direction);
/* Per-voxel eigen-decomposition + score of an existing N*6 tensor image:
 * ConvertFlatSym2Evects3 + ScoreHessian* (kind_is_vote_tensor = 0) as in
 * handlers.cpp:1656-1704, or DiagonalizeFlatSym3 + ScoreTensor* (= 1) as in
 * handlers.cpp:1870-1892.  eivals (N*3) and direction (N*3) may be NULL.
 * Voxels with mask==0 keep their previous score. */
int visfd_cuda_tensor_score(visfd_ctx *ctx, int64_t n_voxels, const float *tensor,
                            const float *mask, int eival_order, int score_kind,
                            int kind_is_vote_tensor, float *score, float *eivals,
                            float *direction);

/* ---- saliency cut ------------------------------------------------------------ */
/* bin/filter_mrc/handlers.cpp:1751-1797.  is_fraction: threshold = element
 * floor(n*cut) of the un-masked saliencies sorted in decreasing order; then
 * every voxel with saliency < threshold is set to 0 in place. */
int visfd_cuda_saliency_cut(visfd_ctx *ctx, int64_t n_voxels, float *saliency,
                            const float *mask, float cut, int is_fraction,
                            float *threshold_out);
/* Building block of the cut for multi-GPU drivers: 2048-bin histogram of the
 * order-preserving 32-bit keys of saliency[i] (mask[i]!=0) whose top
 * `prefix_bits` bits equal `prefix`; bin = next 11 (or the remaining) bits.
 * hist: 2048 uint64 on the HOST.  Ranks all-reduce hist and call
 * visfd_cuda_select_step to narrow the prefix. */
int visfd_cuda_select_hist(visfd_ctx *ctx, int64_t n_voxels, const float *saliency,
                           const float *mask, uint32_t prefix, int prefix_bits,
                           uint64_t *hist);
/* Given a (globally reduced) histogram and the rank still to skip (number of
 * keys greater than the current prefix range already accounted for), returns
 * the new prefix/prefix_bits and the updated rank.  Pure host code. */
int visfd_cuda_select_step(const uint64_t *hist, uint32_t *prefix, int *prefix_bits,
                           uint64_t *rank);
/* key <-> float helpers for drivers */
float visfd_cuda_key_to_float(uint32_t key);

/* ---- tensor voting -------------------------------------------------------------- */
/* TV3D<float,int,array<float,3>,float*>(sigma, exponent, cutoff_ratio) followed by
 * TVDenseStick(...): lib/visfd/feature.hpp:1645-1651, 1712-1901, 2218-2384.
 * tensor: N*6 floats (voxels with mask_dst==0 are left untouched).  normalize and
 * diagonalize_dest must be 0 (filter_mrc passes false for both,
 * bin/filter_mrc/handlers.cpp:1834-1835). */
int visfd_cuda_tv_dense_stick(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz,
                              const float *saliency, const float *direction,
                              const float *mask_src, const float *mask_dst, float sigma,
                              int exponent, float cutoff_ratio,
                              int detect_curves_not_surfaces, int normalize,
                              int diagonalize_dest, float *tensor);

/* ---- fused membrane pipeline --------------------------------------------------- */
/* What HandleTV computes between bin/filter_mrc/handlers.cpp:1618 and :1892 when no
 * background subtraction is requested: CalcHessian -> eigen + planar score ->
 * saliency cut -> TVDenseStick -> DiagonalizeFlatSym3 + ScoreTensorPlanar.
 * out: N floats (tomo_out).  Optional outputs (NULL to skip):
 *   hess_saliency: N floats, ridge saliency after the cut
 *   direction    : N*3 floats, eivects[0] (only voxels that survive the cut are
 *                  guaranteed to be filled)
 *   tensor       : N*6 floats, vote tensor (-save-progress, handlers.cpp:1897-1922)
 *   threshold_out: the cut threshold used.
 * tv_sigma <= 0 skips voting (out = saliency after the cut). */
typedef struct visfd_membrane_params {
  float sigma;            /* settings.width_a[0] in voxels                       */
  float truncate_ratio;   /* filter_truncate_ratio (after the threshold rule)    */
  int eival_order;        /* VISFD_DECREASING_EIVALS for -membrane minima        */
  float cut;              /* settings.hessian_score_threshold                    */
  int cut_is_fraction;    /* settings.hessian_score_threshold_is_a_fraction      */
  float tv_sigma;         /* settings.tv_sigma in voxels                         */
  int tv_exponent;        /* settings.tv_exponent                                */
  float tv_cutoff_ratio;  /* settings.tv_truncate_ratio                          */
} visfd_membrane_params;

int visfd_cuda_membrane(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz,
                        const float *src, const float *mask,
                        const visfd_membrane_params *p, float *out, float *hess_saliency,
                        float *direction, float *tensor, float *threshold_out);

/* The same with `-membrane-background` (settings.width_b > 0; handlers.cpp:1577-1592): both the ridge score
 * (before the cut; :1698-1702) and the post-vote score (:1883-1887) are multiplied by peak_height =
 * source - ApplyGauss(source, background_sigma, halfwidth floor(background_sigma * truncate_ratio), mask,
 * normalize_near_boundaries).  background_sigma == 0: identical to visfd_cuda_membrane. */
int visfd_cuda_membrane_background(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, const float *src,
                                   const float *mask, const visfd_membrane_params *p, float background_sigma,
                                   int normalize_near_boundaries, float *out, float *hess_saliency, float *direction,
                                   float *tensor, float *threshold_out);

/* Slab stages of the same pipeline for the multi-GPU driver (DEVICE pointers only).
 * A rank owns global planes [z_offset+own_z0, z_offset+own_z1) and holds a slab that
 * extends them by a halo of RAW SOURCE planes (exchanged once, before stage 1):
 *   halo >= tv_halfwidth + 1 + gauss_halfwidth   (clipped at the global borders)
 * so that every later stage is slab-local and the only collective left is the
 * all-reduce of the cut histograms (visfd_cuda_select_hist / _select_step).
 * Stage 1: Gaussian + ridge saliency on every plane of the slab; planes closer than
 *   gauss_halfwidth+1 to an INTERNAL slab face hold incomplete values and must not be
 *   used (they are exactly the planes outside [vote_z0, vote_z1) below).
 *   smoothed, saliency: nz_local*ny*nx floats each.
 * Stage 2 (after the global cut threshold is known): receivers are planes
 *   [own_z0, own_z1), voters come from planes [vote_z0, vote_z1) (slab-local indices,
 *   vote range = own range widened by tv_halfwidth, clipped to the volume).
 *   out: (own_z1-own_z0)*ny*nx floats; tensor (optional): the same region * 6.
 *   With p->tv_sigma <= 0, out = saliency after the cut. */
int visfd_cuda_ridge_saliency_slab(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz_local,
                                   int64_t z_offset, int64_t nz_global, const float *src,
                                   const float *mask, float sigma, float truncate_ratio,
                                   int eival_order, int score_kind, float *smoothed,
                                   float *saliency);
int visfd_cuda_vote_slab(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz_local,
                         int64_t z_offset, int64_t nz_global, int64_t own_z0, int64_t own_z1,
                         int64_t vote_z0, int64_t vote_z1, const float *saliency,
                         const float *smoothed, const float *mask, float threshold,
                         const visfd_membrane_params *p, float *out, float *tensor);
/* The same, and the result also delivered to the HOST array out_host ((own_z1-own_z0)*ny*nx
 * floats): the receiver planes are voted in chunks and each finished chunk is copied back on
 * a second stream while the next one is computed (the slab counterpart of what
 * visfd_cuda_membrane does for a host `out`). */
int visfd_cuda_vote_slab_host(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz_local,
                              int64_t z_offset, int64_t nz_global, int64_t own_z0, int64_t own_z1,
                              int64_t vote_z0, int64_t vote_z1, const float *saliency,
                              const float *smoothed, const float *mask, float threshold,
                              const visfd_membrane_params *p, float *out, float *tensor,
                              float *out_host);

/* ---- the same pipeline on several GPUs of one node, one call (SURVEY 8b / 8e) ------------------ */
/* visfd_cuda_membrane with HOST arrays, spread over `ndev` devices as Z-slabs (one host thread per device, no
 * process per GPU, no MPI): the drop-in a C++ host such as filter_mrc links.  devices[] may name a device more than
 * once.  Each device uploads its slab (own planes + halo of raw source, halo = tv_halfwidth + 1 + gauss_halfwidth)
 * straight from src_host; the `-tv-best` cut is a global radix select (histograms summed on the host, handlers.cpp:
 * 1766-1782); every device writes its planes of the result into out_host behind its voting kernels.  The result is
 * bit-identical to visfd_cuda_membrane on one GPU.  mask_host may be NULL.  device_ms (ndev doubles or NULL): device
 * time of each worker, first upload to last download.  The call keeps one context per entry of devices[], created
 * on first use and kept for later calls; concurrent calls are therefore serialised (one runs at a time). */
int visfd_cuda_membrane_multi(int ndev, const int *devices, int64_t nx, int64_t ny, int64_t nz,
                              const float *src_host, const float *mask_host, const visfd_membrane_params *p,
                              float *out_host, float *threshold_out, double *device_ms);

/* ---- clustering: LabelConnected ------------------------------------------------------ */
/* lib/visfd/connect.hpp:171-1432 with the arguments HandleTV passes (bin/filter_mrc/handlers.cpp:1927-2034;
 * `-connect`, SURVEY 8f rank 1): connectivity 1, clusters grown from the saliency MAXIMA, the tensor positive
 * definite near the target, clusters numbered from 1 by decreasing size, no must-link constraints, no voxel weights.
 *   saliency  N floats; mask N floats or NULL (0 = ignore);
 *   tensor    N*6 floats (flat xx,yy,zz,xy,yz,xz) or NULL (aaaafSymmetricTensor);
 *   direction N*3 floats or NULL (aaaafVector AND aaaafVectorStandardized, which HandleTV aliases, :1985): read as the
 *             voxels' directions unless direction_from_tensor != 0, in which case it is first filled with the principal
 *             eigenvector of each tensor (handlers.cpp:1933-1950, eival_order); on return, with unsigned dot products,
 *             it holds the sign-standardised directions (connect.hpp:698-722, :1080-1300).  NULL with a tensor: the
 *             eigenvectors are computed internally and not returned.
 *   thresholds as LabelConnected's arguments (cosines; -connect-angle, settings.cpp:175-178, :3075-3086).
 *   labels    N int64: cluster number from 1, -1 = undefined; voxels outside the mask keep the reference's internal
 *             marker n_maxima + 1 (connect.hpp:1398-1401 skips them; n_maxima is returned for that purpose).
 *   cluster_maxima  optional, 3 floats (x,y,z) per cluster in label order, at most maxima_capacity clusters.
 * Per-voxel tests and the six directed neighbour tests run on the GPU in one pass (16 flag bits per voxel); the
 * priority-queue flood that assigns basins and merges clusters runs on the host in the reference's pop order over
 * those flags (the basin numbering, the polarity of the standardised directions and the cut of non-orientable loops
 * depend on that order).  The whole image must fit on one GPU (saliency 4 + tensor 24 + direction 12 + flags 2 B/voxel).
 * DEVICE or HOST pointers (all image arrays on the same side; `labels` may be on either side). */
int visfd_cuda_label_connected(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, const float *saliency,
                               const float *mask, const float *tensor, float *direction, int direction_from_tensor,
                               int eival_order, int consider_dot_product_sign, float threshold_saliency,
                               float threshold_vector_saliency, float threshold_vector_neighbor,
                               float threshold_tensor_saliency, float threshold_tensor_neighbor, int64_t *labels,
                               int64_t *n_clusters, float *cluster_maxima, int64_t maxima_capacity, int64_t *n_maxima);

/* ---- oriented point cloud of a detected surface ---------------------------------------
 * The block of HandleTV that runs when `-normals-file` is given (bin/filter_mrc/handlers.cpp:2039-2309; the
 * reference has no function for it).  For every un-masked voxel whose label equals select_cluster (`labels` =
 * tomo_out after LabelConnected, a float image as in the reference; `-select-cluster`, settings.cpp:3171):
 * follow the unit surface normal (`direction`, N*3) in both directions in steps of curve_ds
 * (`settings.surface_normal_curve_ds`, 0.2) while inside the cluster, take the saliency-weighted mean position
 * (:2097-2215), then move it onto the ridge of the saliency along the eigenvector of the saliency's
 * finite-difference Hessian with the largest |eigenvalue| (`surface_find_ridge`, :2224-2295), dropping points
 * further than max_distance voxels from the ridge (`max_distance_to_feature`, 1.3; <= 0 disables the test).
 * labels == NULL: every un-masked voxel with its position times voxel_width and its direction (:2053-2066).
 * rows: capacity x {x, y, z, nx, ny, nz} in the reference's order (raster order of the source voxel), positions
 * times voxel_width when the ridge step ran (:2283-2285) and in voxels otherwise, normals scaled by the saliency
 * of the source voxel; *n_points = number found (rows beyond capacity are not stored): the columns of the PLY
 * file WriteOrientedPointCloudPLY writes (bin/filter_mrc/file_io.hpp:501-527).  A walk over a zero direction,
 * endless in the reference, stops after 4 (nx+ny+nz) / curve_ds steps.  DEVICE or HOST pointers. */
int visfd_cuda_surface_points(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, const float *saliency,
                              const float *direction, const float *labels, const float *mask, int select_cluster,
                              const float voxel_width[3], float curve_ds, int find_ridge, float max_distance,
                              float *rows, int64_t capacity, int64_t *n_points);

/* ---- bookkeeping for benchmarks (no reference counterpart) ------------------------- */
/* Enable/disable the per-stage CUDA-event timing behind visfd_cuda_stage_ms. */
void visfd_cuda_set_timing(visfd_ctx *ctx, int enabled);
/* Voters (saliency != 0 after the cut, mask != 0) seen by the most recent voting call. */
int64_t visfd_cuda_last_voter_count(visfd_ctx *ctx);
/* Which voting kernel the most recent voting call ran: 0 = tv_gather_kernel (radial decay by MUFU; every
 * parameter set), 1 / 2 = tv_gather_lut_kernel (decay and 1/r^2 from a shared-memory table indexed by the integer
 * r^2; exponent 4, positive weights, radius <= 24; 2 = the table ends at the support and the index is clamped).
 * Environment switches read by the voting call, for tests and tuning only: VISFD_CUDA_NO_LUT=1 forces kernel 0,
 * VISFD_CUDA_LUT_MODE=2 forces the clamped table, VISFD_CUDA_CHUNK_WAVES=n sets the smallest receiver chunk of the
 * overlapped download (default 64 waves of CTAs); visfd_cuda_membrane also reads VISFD_CUDA_UPLOAD_CHUNK=planes. */
int visfd_cuda_last_tv_kernel(visfd_ctx *ctx);
/* Number of (receiver, voter) pairs the reference's TVReceiveStickVotes would evaluate
 * past its skip tests (feature.hpp:2251-2270) for this input: voters as above, receivers
 * = voxels of planes [recv_z0, recv_z1) with mask_dst != 0 at squared distance <= hw^2.
 * The roofline's FLOP count is 35 * pairs.  DEVICE or HOST pointers. */
int visfd_cuda_tv_count_pairs(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz,
                              const float *saliency, float threshold, const float *mask_src,
                              const float *mask_dst, int halfwidth, int64_t recv_z0,
                              int64_t recv_z1, int64_t *pairs);
/* Sustained FP32 FMA throughput of the device in TFLOP/s (register-resident FFMA chains,
 * `ms` milliseconds of work): the measured denominator of the voting roofline. */
int visfd_cuda_fp32_peak(visfd_ctx *ctx, double ms, double *tflops);
/* The same with packed FFMA2 (fma.rn.f32x2) chains. */
int visfd_cuda_fp32_peak_packed(visfd_ctx *ctx, double ms, double *tflops);
/* FFMA with three distinct register operands (acc += x*y): register-file bandwidth (two
 * 32-bit operands per lane per clock) holds this form to ~2/3 of the chain peak. */
int visfd_cuda_fp32_peak_3op(visfd_ctx *ctx, double ms, double *tflops);

/* ---- threshold / mask maps -------------------------------------------------------- */
#define VISFD_THRESH_SINGLE 1 /* in > a ? outB : outA           handlers.cpp:1049-1053 */
#define VISFD_THRESH_2      2 /* Threshold2, lib/threshold/threshold.hpp:52-77         */
#define VISFD_THRESH_4      4 /* Threshold4, lib/threshold/threshold.hpp:117-169       */
#define VISFD_THRESH_GAUSS  5 /* SelectIntensityRangeGauss, threshold.hpp:248-258      */
#define VISFD_RESCALE       6 /* out = out*t[0] + t[1],      handlers.cpp:1040-1043    */
/* HandleThresholds inner loop (bin/filter_mrc/handlers.cpp:1037-1080) fused with the
 * mask fill of bin/filter_mrc/filter_mrc.cpp:771-776 (applied when mask != NULL and
 * use_masked_value != 0).  t[4]: thresholds (unused entries ignored). */
int visfd_cuda_threshold(visfd_ctx *ctx, int64_t n_voxels, const float *in, float *out,
                         int kind, const float t[4], float outA, float outB,
                         const float *mask, int use_masked_value, float masked_value);
/* AverageArr / StdDevArr (lib/visfd/visfd_utils.hpp:685-790), needed by -cl. */
int visfd_cuda_mean_stddev(visfd_ctx *ctx, int64_t n_voxels, const float *in,
                           const float *weights, float *mean_out, float *stddev_out);
/* The two sums behind them, for a multi-GPU caller (SURVEY 8e: "-cl needs mean + stddev => allreduce"):
 * sums[0] = sum w*h, or sum w*(h - center)^2 when squared != 0; sums[1] = sum w (w = 1 without
 * weights); both in double.  All-reduce (sum) over the ranks, then mean = s0/s1 and, after a second
 * call with center = (float)mean, stddev = sqrt(s0/s1). */
int visfd_cuda_moment_sums(visfd_ctx *ctx, int64_t n_voxels, const float *in, const float *weights,
                           double center, int squared, double sums[2]);

/* ---- binning (SURVEY 8f rank 3: the resampling filter_mrc wraps around the path) ------ */
/* BinArray3D<float,int>: lib/visfd/resample.hpp:53-104 (caller HandleBinning,
 * bin/filter_mrc/handlers.cpp:2361-2425).  size_* = {nx, ny, nz}; bin size per axis =
 * size_src / size_dst (integer division; trailing source voxels are discarded); every
 * destination voxel is the float mean of its bin, summed in the reference's order.
 * offset: NULL or 3 shifts in [0, bin size).  HOST or DEVICE pointers (both alike). */
int visfd_cuda_bin3d(visfd_ctx *ctx, const int64_t size_src[3], const int64_t size_dst[3],
                     const float *src, float *dst, const int *offset);
/* UnbinArray3D<float,int>: lib/visfd/resample.hpp:106-166 (caller handlers.cpp:2321-2355):
 * dst[Z][Y][X] = src[clamp((Z-oz)/bz)][clamp((Y-oy)/by)][clamp((X-ox)/bx)], bin size =
 * size_dst / size_src. */
int visfd_cuda_unbin3d(visfd_ctx *ctx, const int64_t size_src[3], const int64_t size_dst[3],
                       const float *src, float *dst, const int *offset);

/* ---- mask rasterisation (SURVEY 8f rank 3) ------------------------------------------- */
/* One primitive of the list DrawRegions paints: mirrors visfd::SimpleRegion<float>
 * (lib/visfd/draw.hpp:41-87).  RECT: p = {xmin, xmax, ymin, ymax, zmin, zmax};
 * SPHERE: p = {x0, y0, z0, r, -, -}; all in voxels (the caller has already divided
 * by the voxel width, bin/filter_mrc/filter_mrc.cpp:225-270). */
enum { VISFD_REGION_RECT = 0, VISFD_REGION_SPHERE = 1 };
typedef struct visfd_region {
  int32_t type;
  float p[6];
  float value;
} visfd_region;
/* DrawRegions<float>: lib/visfd/draw.hpp:90-237 (caller filter_mrc.cpp:280-284, which passes
 * no mask and negative_means_subtract = true).  image: nz*ny*nx floats, updated IN PLACE
 * (HOST or DEVICE pointer, mask alike); regions: HOST array.  Regions are applied in list
 * order; voxels where mask == 0 are never touched; with negative_means_subtract a region of
 * negative value clears the positive voxels it covers, and an all-zero image whose FIRST
 * region is negative starts from ones (draw.hpp:98-134). */
int visfd_cuda_draw_regions(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, float *image,
                            const float *mask, const visfd_region *regions, int n_regions,
                            int negative_means_subtract);

/* ---- scale-space blob detection ----------------------------------------------------- */
/* BlobDog<float>: lib/visfd/feature.hpp:56-427.  Results are written to caller
 * (HOST) buffers of `capacity` entries each: crds (capacity*3, voxel x,y,z),
 * sigma, score; *n_minima / *n_maxima receive the full counts (which may exceed
 * capacity).  Lists are ordered by (scale, z, y, x). */
int visfd_cuda_blob_dog(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz,
                        const float *src, const float *mask, const float *sigmas,
                        int n_sigmas, float delta_sigma_over_sigma, float truncate_ratio,
                        float minima_threshold, float maxima_threshold,
                        int use_threshold_ratios, int64_t capacity, float *min_crds,
                        float *min_sigma, float *min_score, int64_t *n_minima,
                        float *max_crds, float *max_sigma, float *max_score,
                        int64_t *n_maxima);
/* Z-slab form for the multi-GPU driver (SURVEY 8e, row K6).  The slab holds image planes
 * [z_offset, z_offset + nz_local) and must carry, around the receiver planes [own_z0, own_z1)
 * (slab-local), a halo of (largest LoG half-width + 1) planes wherever the slab does not end at the
 * image border.  Candidates are reported for the receiver planes only, z as the IMAGE plane index,
 * ordered by (scale, z, y, x), after the absolute thresholds but BEFORE the ratio thresholds, which
 * need the best scores of the whole image (feature.hpp:341-344, :369-372): best_scores[0] /
 * best_scores[1] receive this slab's best minimum / maximum score (1 / -1 if none).  The caller
 * all-reduces them (min / max), concatenates the ranks' lists per scale in rank order and finishes
 * with visfd_cuda_blob_finalize.  src / mask: DEVICE pointers; lists: HOST buffers. */
int visfd_cuda_blob_dog_slab(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz_local, int64_t z_offset,
                             int64_t nz_global, int64_t own_z0, int64_t own_z1, const float *src,
                             const float *mask, const float *sigmas, int n_sigmas, float delta,
                             float truncate_ratio, float minima_threshold, float maxima_threshold,
                             int use_threshold_ratios, int64_t capacity, float *min_crds,
                             float *min_sigma, float *min_score, int64_t *n_minima, float *max_crds,
                             float *max_sigma, float *max_score, int64_t *n_maxima, float *best_scores);
/* The final score filter of BlobDog (feature.hpp:362-417) on gathered HOST lists, in place;
 * *n_minima / *n_maxima: lengths in, lengths out. */
int visfd_cuda_blob_finalize(float minima_threshold, float maxima_threshold, int use_threshold_ratios,
                             float best_min_score, float best_max_score, float *min_crds,
                             float *min_sigma, float *min_score, int64_t *n_minima, float *max_crds,
                             float *max_sigma, float *max_score, int64_t *n_maxima);

#ifdef __cplusplus
}
#endif
#endif /* VISFD_CUDA_H */
