// multi.cu -- the membrane pipeline over Z-slabs behind ONE C call, for host arrays (SURVEY 8b/8e): a C++ host such
// as filter_mrc hands over its host arrays and gets the result back, with no MPI, no Python and no process per GPU.
//
//   visfd_cuda_membrane_multi(ndev, devices, nx, ny, nz, src_host, mask_host, params, out_host, &threshold)
//     one slab per device, all slabs at once: every GPU of the node on one volume;
//   visfd_cuda_membrane_stream(ctx, nx, ny, nz, src_host, mask_host, params, device_bytes, out_host, &threshold)
//     one device, the slabs one after another within a device-memory budget: volumes whose working set does not fit.
// Their _background forms add `-membrane-background`: both scores multiplied by the peak height
// source - Gauss(source, background_sigma), as visfd_cuda_membrane_background does on one GPU.
// visfd_cuda_blob_dog_multi / visfd_cuda_blob_dog_stream do the same for BlobDog, in one pass (see below), and
// visfd_cuda_filter_multi / visfd_cuda_filter_stream for ApplyGauss, ApplyDog and ApplyLog.
// visfd_cuda_membrane_connect_multi / visfd_cuda_membrane_connect_stream add `-connect` (LabelConnected) to the
// membrane drivers, with the vote tensor kept on the device (see "-connect over Z-slabs" below).
//
// The volume is cut into Z-slabs exactly as visfd_b200/slab.py does for the process-per-GPU driver (rank boundaries
// on multiples of 8 planes, slabs widened by a halo of RAW SOURCE planes, halo = tv_halfwidth + 1 + gauss_halfwidth,
// slab start rounded down to a multiple of 8), so every stage is slab-local and the result is bit-identical to the
// one-GPU result for any number of slabs.  With the background the raw-source part of the halo is
// max(1 + gauss_halfwidth, background_halfwidth): the peak height must be exact on every voter plane.  Because the source lives in host memory, each slab uploads its planes --
// halo included -- straight from the caller's array: there is no device-to-device halo traffic at all.
//
// A slab always runs the same steps: (1) upload + ridge saliency; (2) for the `-tv-best` cut, per round of the radix
// select (select_threshold), a histogram of its own planes into 2048 bins, which the calling thread sums (the cut
// must be a GLOBAL order statistic, bin/filter_mrc/handlers.cpp:1766-1782); (3) voting, delivering its planes of the
// result into the caller's array chunk by chunk behind the voting kernels (visfd_cuda_vote_slab_host).
//
// visfd_cuda_membrane_multi runs them in phases.  A phase runs every slab at once (slab 0 on the calling thread, the
// others on threads of their own) and is joined on the host before the next one starts, so a slab that fails cannot
// leave the others waiting for it.  The same device may be listed several times (two slabs on one GPU): that is how
// the one-GPU test box exercises the slab logic.
//
// visfd_cuda_membrane_stream runs passes: in each pass the slabs take their turn, and every slab repeats step (1)
// before the step of the pass, since nothing stays on the device from one slab to the next (Gaussian + ridge are
// under 1 % of a C4 step).  Its slab count is the smallest whose slabs fit the budget by slab_bytes.
#include <algorithm>
#include <chrono>
#include <memory>
#include <mutex>
#include <thread>

#include "common.cuh"
#include "kernels.cuh"

using namespace visfd_cuda;

namespace {

struct SlabPlan {
  int64_t own0, own1;     // global planes this worker delivers
  int64_t slab0, slab1;   // global planes it holds
  int64_t vote0, vote1;   // global voter planes
};

// visfd_b200/slab.py: partition() + make_plan().  bg_hw: the half-width of the background Gaussian, 0 without one.
std::vector<SlabPlan> make_plans(int64_t nz, int world, int gauss_hw, int tv_hw, int bg_hw) {
  const int64_t unit = (nz / 8 >= world) ? 8 : 1;
  const int64_t base = (nz / unit) / world, rem = (nz / unit) % world;
  // the smoothed volume is exact 1 + gauss_hw planes inside the slab, the peak height bg_hw planes inside
  const int64_t raw = std::max(1 + gauss_hw, bg_hw);
  const int64_t halo = tv_hw > 0 ? tv_hw + raw : raw;
  std::vector<SlabPlan> plans((size_t)world);
  int64_t z = 0;
  for (int r = 0; r < world; r++) {
    const int64_t n = (base + (r < rem ? 1 : 0)) * unit;
    SlabPlan &p = plans[(size_t)r];
    p.own0 = z;
    p.own1 = (r == world - 1) ? nz : z + n;
    z += n;
    p.slab0 = std::max<int64_t>(0, p.own0 - halo) / 8 * 8;
    p.slab1 = std::min(nz, p.own1 + halo);
    p.vote0 = std::max<int64_t>(0, p.own0 - std::max(tv_hw, 0));
    p.vote1 = std::min(nz, p.own1 + std::max(tv_hw, 0));
  }
  return plans;
}

int max_slabs(int64_t nz) { return (int)std::max<int64_t>(1, nz / 8); }   // at least 8 planes per slab

// `-membrane-background`: sigma > 0 multiplies both scores by the peak height source - Gauss(source, sigma)
struct Background {
  float sigma = 0.0f;
  int hw = 0;               // floor(sigma * truncate_ratio), handlers.cpp:1582-1583
  bool normalize = true;
  bool on() const { return sigma > 0.0f; }
};

// One call at a time: the contexts are kept between calls, one per (slot, device), and a call uses them throughout.
std::mutex g_call_mutex;
std::vector<std::pair<int, visfd_ctx *> > g_ctx;   // index = slot

visfd_ctx *context_for(const char *name, int slot, int device) {
  if ((int)g_ctx.size() <= slot) g_ctx.resize((size_t)slot + 1, {-1, nullptr});
  auto &e = g_ctx[(size_t)slot];
  if (e.second && e.first != device) {
    visfd_cuda_destroy(e.second);
    e.second = nullptr;
  }
  if (!e.second) {
    visfd_ctx *c = nullptr;
    if (visfd_cuda_init(device, &c) != 0) throw Error(std::string(name) + ": " + visfd_cuda_last_error());
    e = {device, c};
  }
  return e.second;
}

// The device time of a multi worker, first upload to last download.
struct DeviceClock {
  cudaEvent_t start = nullptr, stop = nullptr;
  double ms = 0.0;
  void begin(cudaStream_t s) {
    VCK(cudaEventCreate(&start));
    VCK(cudaEventCreate(&stop));
    VCK(cudaEventRecord(start, s));
  }
  void end(cudaStream_t s) {
    VCK(cudaEventRecord(stop, s));
    VCK(cudaEventSynchronize(stop));
    float t = 0;
    VCK(cudaEventElapsedTime(&t, start, stop));
    ms = t;
  }
  ~DeviceClock() {
    if (start) cudaEventDestroy(start);
    if (stop) cudaEventDestroy(stop);
  }
};

// What a slab keeps on its device from one step to the next.
struct Slab {
  visfd_ctx *ctx = nullptr;
  SlabPlan plan;
  Scratch<float> mask, smoothed, saliency;
  Scratch<float> peak;   // with the background: the peak height of every plane of the slab, until the vote ends
  DeviceClock clock;
  uint64_t hist[HIST_BINS];
  std::vector<float> tensor_lo, tensor_hi;   // -connect: the vote tensor of the first / last two own planes (seams)
};

void make_slabs(std::vector<Slab> &slabs, const std::vector<SlabPlan> &plans, visfd_ctx *ctx) {
  for (size_t r = 0; r < plans.size(); r++) {
    slabs[r].ctx = ctx;
    slabs[r].plan = plans[r];
  }
}

// Step (1): upload the slab, halo included, and compute its ridge saliency (times the peak height with the
// background).
void upload_and_ridge(Slab &s, int64_t nx, int64_t ny, int64_t nz, const float *src_host, const float *mask_host,
                      const visfd_membrane_params *p, const Background &bg) {
  const SlabPlan &pl = s.plan;
  const size_t plane = (size_t)nx * (size_t)ny;
  const size_t n = (size_t)(pl.slab1 - pl.slab0) * plane;
  Scratch<float> src(s.ctx, n);   // the raw slab is not needed after this step
  s.smoothed.reset(s.ctx, n);
  s.saliency.reset(s.ctx, n);
  VCK(cudaMemcpyAsync(src.get(), src_host + (size_t)pl.slab0 * plane, n * sizeof(float), cudaMemcpyHostToDevice,
                      s.ctx->stream));
  if (mask_host) {
    s.mask.reset(s.ctx, n);
    VCK(cudaMemcpyAsync(s.mask.get(), mask_host + (size_t)pl.slab0 * plane, n * sizeof(float), cudaMemcpyHostToDevice,
                        s.ctx->stream));
  }
  if (bg.on()) {
    // source - Gauss(source) in one volume, through the filter's minuend epilogue: (src - G(src)) * 1 has the bits
    // of the one-GPU path's __fsub_rn(src, bg)
    s.peak.reset(s.ctx, n);
    const float sg[3] = {bg.sigma, bg.sigma, bg.sigma};
    const int hw[3] = {bg.hw, bg.hw, bg.hw};
    gauss_device(s.ctx, nx, ny, pl.slab1 - pl.slab0, pl.slab0, nz, src.get(), s.peak.get(), s.mask.get(), sg, hw,
                 bg.normalize, src.get(), 1.0f);
    VCK(cudaStreamSynchronize(s.ctx->stream));
    resolve_stage_times(s.ctx);   // (the entry point below drops the stage events it finds pending)
  }
  if (visfd_cuda_ridge_saliency_slab(s.ctx, nx, ny, pl.slab1 - pl.slab0, pl.slab0, nz, src.get(), s.mask.get(),
                                     p->sigma, p->truncate_ratio, p->eival_order, VISFD_SCORE_PLANAR, s.smoothed.get(),
                                     s.saliency.get()) != 0)
    throw Error(visfd_cuda_last_error());
  // before any histogram: the cut ranks the scaled score (handlers.cpp:1698-1702)
  if (bg.on()) scale_by_peak_device(s.ctx, (i64)n, s.saliency.get(), s.peak.get(), nullptr, s.mask.get());
}

// Step (2): the histogram of the slabs' own planes, summed into hist.  run(step) runs step(slab) on every slab.
template <typename Run>
void summed_own_hist(std::vector<Slab> &slabs, const Run &run, size_t plane, bool masked, uint32_t prefix,
                     int prefix_bits, uint64_t *hist) {
  run([&](Slab &s) {
    const size_t own = (size_t)(s.plan.own0 - s.plan.slab0) * plane;
    select_hist_device(s.ctx, (i64)((size_t)(s.plan.own1 - s.plan.own0) * plane), s.saliency.get() + own,
                       masked ? s.mask.get() + own : nullptr, prefix, prefix_bits, s.hist);
    resolve_stage_times(s.ctx);   // (select_hist_device has synchronised the stream)
  });
  std::fill(hist, hist + HIST_BINS, 0);
  for (const Slab &s : slabs)
    for (int b = 0; b < HIST_BINS; b++) hist[b] += s.hist[b];
}

// Step (3): voting on the own planes, delivered into the caller's array (each chunk times its peak height with the
// background).
void vote_to_host(Slab &s, int64_t nx, int64_t ny, int64_t nz, float threshold, const visfd_membrane_params *p,
                  float *out_host) {
  const SlabPlan &pl = s.plan;
  const size_t plane = (size_t)nx * (size_t)ny;
  Scratch<float> out(s.ctx, (size_t)(pl.own1 - pl.own0) * plane);
  vote_slab_device(s.ctx, nx, ny, pl.slab1 - pl.slab0, pl.slab0, nz, pl.own0 - pl.slab0, pl.own1 - pl.slab0,
                   pl.vote0 - pl.slab0, pl.vote1 - pl.slab0, s.saliency.get(), s.smoothed.get(), s.mask.get(),
                   threshold, p, out.get(), nullptr, out_host + (size_t)pl.own0 * plane, s.peak.get());
  VCK(cudaStreamSynchronize(s.ctx->stream));
  resolve_stage_times(s.ctx);
}

// Runs fn(slab) for every slab at once, slab 0 on the calling thread and the others on threads of their own, each
// on its slab's device.  Returns when all of them have finished, and then throws the error of the first slab that
// failed.
template <typename S, typename Fn>
void for_each_slab(const char *name, std::vector<S> &slabs, const Fn &fn) {
  std::vector<std::string> errors(slabs.size());
  auto run = [&](size_t r) {
    try {
      VCK(cudaSetDevice(slabs[r].ctx->device));
      fn(slabs[r]);
    } catch (const std::exception &ex) {
      errors[r] = ex.what();
    }
  };
  std::vector<std::thread> threads;
  for (size_t r = 1; r < slabs.size(); r++) {
    try {
      threads.emplace_back(run, r);
    } catch (const std::exception &ex) {   // no thread for this slab; the others still run and are joined
      errors[r] = ex.what();
    }
  }
  run(0);
  for (std::thread &t : threads) t.join();
  for (size_t r = 0; r < slabs.size(); r++)
    if (!errors[r].empty())
      throw Error(std::string(name) + ", slab " + std::to_string(r) + " on device " +
                  std::to_string(slabs[r].ctx->device) + ": " + errors[r]);
}

// The device bytes the pool holds at most while one slab of visfd_cuda_membrane_stream takes its turn, in the blocks
// visfd_ctx::alloc takes.  Step (1) holds the uploaded source, the mask, the smoothed volume, the saliency and the
// Gaussian's scratch; a cut or count pass (vote == false) adds the select's histogram.  The vote pass releases the
// step's scratch before step (3), which holds the mask, the smoothed volume and the saliency, the own-plane output
// and the voting workspace for at most `voters` voters in the whole volume.
// With the background both steps also hold the slab's whole peak height.  In step (1) the background Gaussian runs
// first, beside the same volumes; its scratch goes back to the pool, where the smoothing's scratch, which has at least
// as many volumes, takes them again, so only its block of taps may stay cached next to the smoothing's.
// With -connect (vote_and_flag) the vote also holds the own planes' tensor; then everything but the mask, the output
// and the tensor goes back to the device, and the flags step adds the own planes' directions and flags.  A seam step
// holds the same blocks for 4 planes: never more than a slab of at least 8 own planes.
size_t slab_bytes(const SlabPlan &pl, int64_t nx, int64_t ny, bool masked, const visfd_membrane_params *p,
                  int gauss_hw, const Background &bg, bool vote, uint64_t voters, bool connect) {
  const size_t plane = (size_t)nx * (size_t)ny;
  const int64_t slab = pl.slab1 - pl.slab0;
  const size_t vol = visfd_ctx::block_bytes((size_t)slab * plane * sizeof(float));
  const int hw[3] = {gauss_hw, gauss_hw, gauss_hw}, hw_bg[3] = {bg.hw, bg.hw, bg.hw};
  const size_t peak = bg.on() ? vol : 0;
  const size_t bg_taps = bg.on() ? separable_workspace_bytes(nx, ny, slab, hw_bg, false, false) - vol : 0;
  const size_t ridge = (masked ? 4 : 3) * vol + peak + separable_workspace_bytes(nx, ny, slab, hw, masked, true) + bg_taps;
  if (!vote) return ridge + visfd_ctx::block_bytes(HIST_BINS * sizeof(uint64_t));
  const size_t own = (size_t)(pl.own1 - pl.own0) * plane;
  const size_t out = visfd_ctx::block_bytes(own * sizeof(float));
  const size_t tensor = connect ? visfd_ctx::block_bytes(own * 6 * sizeof(float)) : 0;
  size_t voting = (masked ? 3 : 2) * vol + peak + out + tensor;
  if (p->tv_sigma > 0.0f) {
    // visfd_cuda_vote_slab_host widens the voter planes down to a global multiple of 8: up to 7 more planes, whose
    // saliency may be incomplete, so they may add up to 7 planes of voters to the count of the whole volume
    const int64_t vplanes = std::min(pl.vote1 - pl.vote0 + 7, slab);
    const uint64_t vox = (uint64_t)vplanes * plane;
    const uint64_t n = voters < vox ? std::min(vox, voters + 7 * (uint64_t)plane) : vox;
    voting += tv_workspace_bytes(nx, ny, vplanes, pl.own1 - pl.own0, n);
  }
  const size_t flags = connect ? (masked ? vol : 0) + out + tensor + visfd_ctx::block_bytes(own * 3 * sizeof(float)) +
                                     visfd_ctx::block_bytes(own * sizeof(uint16_t))
                               : 0;
  return std::max({ridge, voting, flags});
}

// The ridge step's scratch and every block a finished slab leaves behind go back to the device, so that the next
// step or slab allocates afresh rather than next to cached blocks it cannot reuse.
void release_cache(visfd_ctx *ctx) {
  VCK(cudaStreamSynchronize(ctx->stream));
  ctx->trim();
}

// The budget of a stream call: device_bytes, or for 0 the free memory at entry less a margin.  Releases the cache
// first: blocks cached by earlier calls count against the budget.
int64_t stream_budget(visfd_ctx *ctx, int64_t device_bytes) {
  VCK(cudaSetDevice(ctx->device));
  drop_pending_stage_events(ctx);
  release_cache(ctx);
  if (device_bytes != 0) return device_bytes;
  // the margin covers what the call needs outside the pool: the allocation granularity of cudaMalloc, code of
  // kernels loaded on first use, local memory
  size_t free_b = 0, total_b = 0;
  VCK(cudaMemGetInfo(&free_b, &total_b));
  return (int64_t)free_b - (int64_t)(1u << 30);
}

// The fewest slabs whose every slab fits the budget, 0 if none does; *need: the bytes of the largest slab of the last
// plan tried.  bytes(plan) is what one slab holds at most.
template <typename Bytes>
int fewest_slabs(int64_t nz, int gauss_hw, int tv_hw, int bg_hw, int64_t budget, const Bytes &bytes, size_t *need) {
  for (int world = 1; world <= max_slabs(nz); world++) {
    *need = 0;
    for (const SlabPlan &pl : make_plans(nz, world, gauss_hw, tv_hw, bg_hw)) *need = std::max(*need, bytes(pl));
    if (*need <= (size_t)std::max<int64_t>(budget, 0)) return world;
  }
  return 0;
}

Error too_small(const std::string &who, const char *what, size_t need, int64_t budget) {
  return Error(who + ": " + what + " needs " + std::to_string(need) +
               " bytes of device memory in slabs of 8 planes; the budget is " + std::to_string(budget) + " bytes");
}

// After a failed stream call: nothing of it stays on the device, and the context takes the next call.
void reset_after_failure(visfd_ctx *ctx) {
  if (!ctx) return;
  cudaStreamSynchronize(ctx->stream);
  cudaGetLastError();
  ctx->trim();
}

// The background of a _background entry point, checked; sigma 0: none (the plain entry points).
Background background(const std::string &who, const visfd_membrane_params *p, float sigma, int normalize) {
  VREQUIRE(sigma >= 0.0f, who + ": negative background width");   // (NaN fails too)
  Background bg;
  bg.sigma = sigma;
  bg.hw = sigma > 0.0f ? (int)floorf(sigma * p->truncate_ratio) : 0;   // as visfd_cuda_membrane_background
  bg.normalize = normalize != 0;
  return bg;
}

// ---- -connect over Z-slabs -------------------------------------------------------------------------------------
// LabelConnected's per-voxel predicates read the post-vote score, the vote tensor, its first eigenvector and the mask
// within +-1 plane only (2 planes at the global ends, where the stencil is clamped), and the host flood reads only the
// 16-bit flags, the score and the directions.  So a slab computes, right after its vote, the flags of every own plane
// whose neighbours it holds, and sends 2 B per voxel home instead of the 24 B of the tensor.  Slab boundaries lie on
// multiples of 8 planes with at least 8 own planes per slab, so the two planes next to an internal boundary b are
// inner planes of the volume: a seam step computes their flags from planes b-2 .. b+1 (score and mask from the
// caller's arrays, the two tensor planes each side kept on the host by the slabs).  Receivers are not voted again:
// a receiver is bit-exact only inside whole 4-plane patches of its slab.

// The arguments and outputs of a connect call; flags: the whole image's, filled by the slabs and the seams.
struct Connect {
  visfd_connect_params c;   // thresholds as LabelConnected takes them (negative vector cosines clamped)
  int64_t *labels = nullptr;
  float *direction = nullptr;
  int64_t *n_clusters = nullptr, *n_maxima = nullptr;
  float *maxima = nullptr;
  int64_t capacity = 0;
  std::unique_ptr<uint16_t[]> flags;
};

Connect connect_args(const std::string &who, int64_t nx, int64_t ny, int64_t nz, const float *src_host,
                     const visfd_membrane_params *p, float background_sigma, const visfd_connect_params *c,
                     float *out_host, int64_t *labels, float *direction, int64_t capacity) {
  VREQUIRE(src_host && p && c && out_host && labels && capacity >= 0, who + ": bad arguments");
  VREQUIRE(p->tv_sigma > 0.0f, who + ": -connect clusters the vote tensor: tv_sigma must be positive");
  VREQUIRE(background_sigma >= 0.0f, who + ": negative background width");   // (NaN fails too)
  VREQUIRE(nx >= 3 && ny >= 3 && nz >= 3, who + ": LabelConnected needs an image at least 3 voxels wide");
  VREQUIRE(nx < (1LL << 31) && ny < (1LL << 31) && nz < (1LL << 31), who + ": bad image dimensions");
  VREQUIRE(!is_device_pointer(labels) && !is_device_pointer(direction), who + " takes HOST arrays");
  Connect cn;
  cn.c = *c;
  if (!c->consider_dot_product_sign) {   // connect.hpp:190-205, as visfd_cuda_label_connected
    cn.c.threshold_vector_saliency = std::max(cn.c.threshold_vector_saliency, 0.0f);
    cn.c.threshold_vector_neighbor = std::max(cn.c.threshold_vector_neighbor, 0.0f);
  }
  cn.labels = labels;
  cn.direction = direction;
  cn.capacity = capacity;
  return cn;
}

// Flags of `planes` planes [z0, z1) of arrays that start at global plane z_offset, into cn.flags.
void flag_planes(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, int64_t planes, int64_t z_offset, int64_t z0,
                 int64_t z1, const float *score, const float *mask, const float *tensor,
                 const visfd_membrane_params *p, Connect &cn, float *direction_host) {
  const size_t plane = (size_t)nx * (size_t)ny, n = (size_t)planes * plane;
  Scratch<float> dir(ctx, 3 * n);
  Scratch<uint16_t> state(ctx, n);
  first_eigenvectors_device(ctx, (i64)n, tensor, mask, p->eival_order, dir.get());
  const visfd_connect_params &c = cn.c;
  // the Hessian of the score is diagonalised with DECREASING eigenvalues, as visfd_cuda_label_connected does
  connect_predicates_device(ctx, nx, ny, planes, z_offset, nz, z0, z1, score, mask, tensor, dir.get(), 1,
                            c.consider_dot_product_sign != 0, c.threshold_saliency, c.threshold_vector_saliency,
                            c.threshold_vector_neighbor, c.threshold_tensor_saliency, c.threshold_tensor_neighbor,
                            state.get());
  {
    StageTimer t(ctx, "d2h");
    VCK(cudaMemcpyAsync(cn.flags.get() + (size_t)(z_offset + z0) * plane, state.get() + (size_t)z0 * plane,
                        (size_t)(z1 - z0) * plane * sizeof(uint16_t), cudaMemcpyDeviceToHost, ctx->stream));
    if (direction_host)
      VCK(cudaMemcpyAsync(direction_host, dir.get(), 3 * n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  }
  VCK(cudaStreamSynchronize(ctx->stream));
}

// Step (3) with -connect: voting on the own planes, delivered into the caller's array, with their tensor kept on the
// device; then the flags of the own planes whose neighbours the slab holds, the directions, and the tensor planes the
// seams need.
void vote_and_flag(Slab &s, int64_t nx, int64_t ny, int64_t nz, float threshold, const visfd_membrane_params *p,
                   float *out_host, Connect &cn) {
  const SlabPlan &pl = s.plan;
  const size_t plane = (size_t)nx * (size_t)ny;
  const int64_t own = pl.own1 - pl.own0;
  Scratch<float> out(s.ctx, (size_t)own * plane), tensor(s.ctx, (size_t)own * plane * 6);
  vote_slab_device(s.ctx, nx, ny, pl.slab1 - pl.slab0, pl.slab0, nz, pl.own0 - pl.slab0, pl.own1 - pl.slab0,
                   pl.vote0 - pl.slab0, pl.vote1 - pl.slab0, s.saliency.get(), s.smoothed.get(), s.mask.get(),
                   threshold, p, out.get(), tensor.get(), out_host + (size_t)pl.own0 * plane, s.peak.get());
  // the voting workspace and the volumes only the vote read go back to the device
  s.smoothed.free();
  s.saliency.free();
  s.peak.free();
  release_cache(s.ctx);
  const float *mask = s.mask.get() ? s.mask.get() + (size_t)(pl.own0 - pl.slab0) * plane : nullptr;
  flag_planes(s.ctx, nx, ny, nz, own, pl.own0, pl.own0 > 0 ? 1 : 0, pl.own1 < nz ? own - 1 : own, out.get(), mask,
              tensor.get(), p, cn, cn.direction ? cn.direction + 3 * (size_t)pl.own0 * plane : nullptr);
  const size_t two = 2 * plane * 6;
  if (pl.own0 > 0) {
    s.tensor_lo.resize(two);
    VCK(cudaMemcpyAsync(s.tensor_lo.data(), tensor.get(), two * sizeof(float), cudaMemcpyDeviceToHost, s.ctx->stream));
  }
  if (pl.own1 < nz) {
    s.tensor_hi.resize(two);
    VCK(cudaMemcpyAsync(s.tensor_hi.data(), tensor.get() + (size_t)(own - 2) * plane * 6, two * sizeof(float),
                        cudaMemcpyDeviceToHost, s.ctx->stream));
  }
  VCK(cudaStreamSynchronize(s.ctx->stream));
  resolve_stage_times(s.ctx);
}

// The boundary between two slabs: planes b-2, b-1 belong to the slab below, b, b+1 to the one above.
struct Seam {
  visfd_ctx *ctx = nullptr;
  int64_t b = 0;
  const float *tensor_below = nullptr, *tensor_above = nullptr;   // two planes each
};

std::vector<Seam> seams_of(const std::vector<Slab> &slabs) {
  std::vector<Seam> seams(slabs.size() - 1);
  for (size_t r = 0; r + 1 < slabs.size(); r++)
    seams[r] = {slabs[r].ctx, slabs[r].plan.own1, slabs[r].tensor_hi.data(), slabs[r + 1].tensor_lo.data()};
  return seams;
}

// The flags of planes b-1 and b, from the result already in the caller's array.
void seam_flags(const Seam &sm, int64_t nx, int64_t ny, int64_t nz, const float *out_host, const float *mask_host,
                const visfd_membrane_params *p, Connect &cn) {
  const size_t plane = (size_t)nx * (size_t)ny, n = 4 * plane, first = (size_t)(sm.b - 2) * plane;
  Scratch<float> score(sm.ctx, n), mask, tensor(sm.ctx, 6 * n);
  {
    StageTimer t(sm.ctx, "h2d");
    VCK(cudaMemcpyAsync(score.get(), out_host + first, n * sizeof(float), cudaMemcpyHostToDevice, sm.ctx->stream));
    if (mask_host) {
      mask.reset(sm.ctx, n);
      VCK(cudaMemcpyAsync(mask.get(), mask_host + first, n * sizeof(float), cudaMemcpyHostToDevice, sm.ctx->stream));
    }
    VCK(cudaMemcpyAsync(tensor.get(), sm.tensor_below, 3 * n * sizeof(float), cudaMemcpyHostToDevice,
                        sm.ctx->stream));
    VCK(cudaMemcpyAsync(tensor.get() + 3 * n, sm.tensor_above, 3 * n * sizeof(float), cudaMemcpyHostToDevice,
                        sm.ctx->stream));
  }
  flag_planes(sm.ctx, nx, ny, nz, 4, sm.b - 2, 1, 3, score.get(), mask.get(), tensor.get(), p, cn, nullptr);
  resolve_stage_times(sm.ctx);
}

// The ordered flood over the flags of the whole image, on the calling thread, and the outputs of the call.  Its host
// time goes to ctx's stage "flood".
void connect_flood(Connect &cn, visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, const float *out_host) {
  std::vector<float> maxima;
  i64 n_max = 0;
  const auto t0 = std::chrono::steady_clock::now();
  const i64 nc = connect_flood_host(nx, ny, nz, out_host, cn.flags.get(), cn.direction,
                                    cn.c.consider_dot_product_sign == 0, cn.c.threshold_saliency, cn.labels, &maxima,
                                    &n_max);
  ctx->stage_ms["flood"] += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  if (cn.n_clusters) *cn.n_clusters = nc;
  if (cn.n_maxima) *cn.n_maxima = n_max;
  if (cn.maxima && cn.capacity > 0)
    std::copy(maxima.begin(), maxima.begin() + 3 * std::min<i64>(nc, cn.capacity), cn.maxima);
}

// cn: -connect, or NULL for the membrane pipeline alone.
int membrane_multi(const char *name, int ndev, const int *devices, int64_t nx, int64_t ny, int64_t nz,
                   const float *src_host, const float *mask_host, const visfd_membrane_params *p,
                   float background_sigma, int normalize, float *out_host, float *threshold_out,
                   double *device_ms, Connect *cn = nullptr) {
  try {
    const std::string who(name);
    VREQUIRE(ndev >= 1 && devices, who + ": need at least one device");
    VREQUIRE(nx > 0 && ny > 0 && nz > 0 && src_host && p && out_host, who + ": bad arguments");
    VREQUIRE(!is_device_pointer(src_host) && !is_device_pointer(out_host) && !is_device_pointer(mask_host),
             who + " takes HOST arrays (use the slab entry points for device-resident data)");
    const Background bg = background(who, p, background_sigma, normalize);
    const int gauss_hw = (int)floor(p->sigma * p->truncate_ratio);
    const int tv_hw = p->tv_sigma > 0.0f ? tv_halfwidth(p->tv_sigma, p->tv_cutoff_ratio) : 0;
    const int world = std::min(ndev, max_slabs(nz));
    const std::vector<SlabPlan> plans = make_plans(nz, world, gauss_hw, tv_hw, bg.hw);
    const size_t plane = (size_t)nx * (size_t)ny;

    std::lock_guard<std::mutex> lock(g_call_mutex);
    std::vector<Slab> slabs((size_t)world);
    make_slabs(slabs, plans, nullptr);
    for (int r = 0; r < world; r++) slabs[(size_t)r].ctx = context_for(name, r, devices[r]);
    auto concurrently = [&](const auto &step) { for_each_slab(name, slabs, step); };

    for_each_slab(name, slabs, [&](Slab &s) {
      s.clock.begin(s.ctx->stream);
      upload_and_ridge(s, nx, ny, nz, src_host, mask_host, p, bg);
    });

    float threshold = p->cut;
    if (p->cut_is_fraction)
      threshold = select_threshold(p->cut, [&](uint32_t prefix, int prefix_bits, uint64_t *hist) {
        summed_own_hist(slabs, concurrently, plane, mask_host != nullptr, prefix, prefix_bits, hist);
      });

    if (cn) cn->flags.reset(new uint16_t[plane * (size_t)nz]);
    for_each_slab(name, slabs, [&](Slab &s) {
      if (cn) vote_and_flag(s, nx, ny, nz, threshold, p, out_host, *cn);
      else vote_to_host(s, nx, ny, nz, threshold, p, out_host);
      s.clock.end(s.ctx->stream);
    });
    if (cn) {
      std::vector<Seam> seams = seams_of(slabs);
      if (!seams.empty())
        for_each_slab(name, seams, [&](Seam &sm) { seam_flags(sm, nx, ny, nz, out_host, mask_host, p, *cn); });
      connect_flood(*cn, slabs[0].ctx, nx, ny, nz, out_host);
    }

    if (threshold_out) *threshold_out = threshold;
    if (device_ms)
      for (int r = 0; r < ndev; r++) device_ms[r] = r < world ? slabs[(size_t)r].clock.ms : 0.0;
    return 0;
  } catch (const std::exception &ex) {
    set_last_error(ex.what());
    return 1;
  }
}

int membrane_stream(const char *name, visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, const float *src_host,
                    const float *mask_host, const visfd_membrane_params *p, float background_sigma, int normalize,
                    int64_t device_bytes, float *out_host, float *threshold_out, int64_t *n_slabs_out,
                    Connect *cn = nullptr) {
  try {
    const std::string who(name);
    VREQUIRE(ctx != nullptr, who + ": context is NULL");
    VREQUIRE(nx > 0 && ny > 0 && nz > 0 && src_host && p && out_host && device_bytes >= 0, who + ": bad arguments");
    VREQUIRE(!is_device_pointer(src_host) && !is_device_pointer(out_host) && !is_device_pointer(mask_host),
             who + " takes HOST arrays (use visfd_cuda_membrane for device-resident data)");
    const Background bg = background(who, p, background_sigma, normalize);
    const int64_t budget = stream_budget(ctx, device_bytes);
    const int gauss_hw = (int)floor(p->sigma * p->truncate_ratio);
    const int tv_hw = p->tv_sigma > 0.0f ? tv_halfwidth(p->tv_sigma, p->tv_cutoff_ratio) : 0;
    const size_t plane = (size_t)nx * (size_t)ny;
    const bool masked = mask_host != nullptr, vote = p->tv_sigma > 0.0f;

    auto fewest = [&](bool vote_pass, uint64_t voters, size_t *need) {
      return fewest_slabs(nz, gauss_hw, tv_hw, bg.hw, budget, [&](const SlabPlan &pl) {
        return slab_bytes(pl, nx, ny, masked, p, gauss_hw, bg, vote_pass, voters, cn && vote_pass);
      }, need);
    };
    // Runs step(slab) on every slab in turn, each after step (1) and each released before the next.
    auto one_by_one = [&](std::vector<Slab> &slabs, const auto &step) {
      for (size_t r = 0; r < slabs.size(); r++) {
        Slab &s = slabs[r];
        try {
          upload_and_ridge(s, nx, ny, nz, src_host, mask_host, p, bg);
          step(s);
        } catch (const std::exception &ex) {
          throw Error(who + ", slab " + std::to_string(r) + " of " + std::to_string(slabs.size()) + ": " + ex.what());
        }
        s.mask.free();
        s.smoothed.free();
        s.saliency.free();
        s.peak.free();
        release_cache(ctx);
      }
    };

    // The passes before the vote: the cut's rounds, or for an absolute cut one count of the voters when the vote
    // pass would otherwise need more slabs than these passes.  Their slabs are sized without voters.
    size_t need = 0;
    const int n_cut = fewest(false, 0, &need);
    if (n_cut == 0) throw too_small(who, "the upload and ridge step", need, budget);
    float threshold = p->cut;
    uint64_t voters = UINT64_MAX;   // unknown: every voxel of a slab's voter planes may vote
    if (p->cut_is_fraction || (vote && fewest(true, voters, &need) != n_cut)) {
      std::vector<Slab> slabs((size_t)n_cut);
      make_slabs(slabs, make_plans(nz, n_cut, gauss_hw, tv_hw, bg.hw), ctx);
      auto in_turn = [&](const auto &step) { one_by_one(slabs, step); };
      if (p->cut_is_fraction) {
        threshold = select_threshold(p->cut, [&](uint32_t prefix, int prefix_bits, uint64_t *hist) {
          summed_own_hist(slabs, in_turn, plane, masked, prefix, prefix_bits, hist);
        }, &voters);
      } else {
        // voters have a saliency at or above the cut: at most the keys of its first-round bin and those above
        uint64_t hist[HIST_BINS];
        summed_own_hist(slabs, in_turn, plane, masked, 0, 0, hist);
        voters = 0;
        for (uint32_t b = float_to_key(threshold) >> 21; b < HIST_BINS; b++) voters += hist[b];
      }
    }

    const int n_vote = fewest(true, voters, &need);
    if (n_vote == 0) throw too_small(who, "the vote pass", need, budget);
    std::vector<Slab> slabs((size_t)n_vote);
    make_slabs(slabs, make_plans(nz, n_vote, gauss_hw, tv_hw, bg.hw), ctx);
    if (cn) cn->flags.reset(new uint16_t[plane * (size_t)nz]);
    one_by_one(slabs, [&](Slab &s) {
      release_cache(ctx);   // the ridge step's scratch
      if (cn) vote_and_flag(s, nx, ny, nz, threshold, p, out_host, *cn);
      else vote_to_host(s, nx, ny, nz, threshold, p, out_host);
    });
    if (cn) {
      for (const Seam &sm : seams_of(slabs)) {
        seam_flags(sm, nx, ny, nz, out_host, mask_host, p, *cn);
        release_cache(ctx);
      }
      connect_flood(*cn, ctx, nx, ny, nz, out_host);
    }

    if (threshold_out) *threshold_out = threshold;
    if (n_slabs_out) *n_slabs_out = n_vote;
    return 0;
  } catch (const std::exception &ex) {
    set_last_error(ex.what());
    reset_after_failure(ctx);
    return 1;
  }
}

// ---- BlobDog over Z-slabs ------------------------------------------------------------------------------------
// A slab needs no collective before the end: it scans its own planes at every scale (blob_dog_device, slab form)
// and keeps its lists and best scores on the host.  The lists are then concatenated per scale in slab order -- the
// one-GPU (scale, z, y, x) order -- and the final filter runs once on the best scores of the whole image
// (feature.hpp:341-344, :369-372).  In ratio mode a slab pre-filters on the device against the best scores of its
// own earlier scales, a threshold never stricter than the global one, so the final filter decides.

struct BlobArgs {
  const float *sigmas;
  int n_sigmas;
  float delta, truncate_ratio, minima_threshold, maxima_threshold;
  int use_threshold_ratios;
};

// The widest LoG half-width over the scales (log_params' arithmetic, as blob_dog_device checks the halo against):
// a slab's halo is this + 1 planes of raw source.
int blob_halfwidth(const BlobArgs &a) {
  int widest = 0;
  for (int i = 0; i < a.n_sigmas; i++) {
    const float s3[3] = {a.sigmas[i], a.sigmas[i], a.sigmas[i]};
    float sa[3], sb[3], scale;
    int hw[3];
    log_params(s3, a.delta, a.truncate_ratio, sa, sb, hw, &scale);
    widest = std::max(widest, hw[2]);
  }
  return widest;
}

// Rows a candidate list of a slab with `own` planes needs for one scale: a strict extremum of its 26 neighbours
// excludes every one of them, so at most one voxel of each 2x2x2 block is listed.  Lists this long cannot overflow,
// so blob_dog_device never scans a scale again into larger lists, which would grow the pool past its plan.
i64 blob_rows(int64_t nx, int64_t ny, int64_t own) { return ((nx + 1) / 2) * ((ny + 1) / 2) * ((own + 1) / 2); }

struct BlobSlab {
  visfd_ctx *ctx = nullptr;
  SlabPlan plan;
  BlobList minima, maxima;
  float best[2] = {1.0f, -1.0f};
  DeviceClock clock;
};

// Uploads the slab's planes, halo included, straight from the caller's arrays and scans its own planes.
void blob_slab(BlobSlab &s, int64_t nx, int64_t ny, int64_t nz, const float *src_host, const float *mask_host,
               const BlobArgs &a) {
  const SlabPlan &pl = s.plan;
  const size_t plane = (size_t)nx * (size_t)ny;
  const size_t n = (size_t)(pl.slab1 - pl.slab0) * plane;
  Scratch<float> src(s.ctx, n), mask;
  {
    StageTimer t(s.ctx, "h2d");
    VCK(cudaMemcpyAsync(src.get(), src_host + (size_t)pl.slab0 * plane, n * sizeof(float), cudaMemcpyHostToDevice,
                        s.ctx->stream));
    if (mask_host) {
      mask.reset(s.ctx, n);
      VCK(cudaMemcpyAsync(mask.get(), mask_host + (size_t)pl.slab0 * plane, n * sizeof(float),
                          cudaMemcpyHostToDevice, s.ctx->stream));
    }
  }
  blob_dog_device(s.ctx, nx, ny, pl.slab1 - pl.slab0, pl.slab0, nz, pl.own0 - pl.slab0, pl.own1 - pl.slab0,
                  src.get(), mask.get(), a.sigmas, a.n_sigmas, a.delta, a.truncate_ratio, a.minima_threshold,
                  a.maxima_threshold, a.use_threshold_ratios, s.minima, s.maxima, false, s.best,
                  blob_rows(nx, ny, pl.own1 - pl.own0));
  VCK(cudaStreamSynchronize(s.ctx->stream));
  resolve_stage_times(s.ctx);
}

// The device bytes the pool holds at most while a slab of visfd_cuda_blob_dog_stream runs, in the blocks
// visfd_ctx::alloc takes.  For the whole scan: the uploaded source and mask, the three LoG volumes, the two
// candidate lists (blob_rows) and their counters.  At every scale dog_device adds the first Gaussian's volume and
// the separable filter's scratch volume (with a mask also the two volumes of its normalisation), plus one small block
// of taps and edge profiles at a time.  These come from the cache once the first scale has put them there, except
// the small blocks: they grow with sigma, so each scale may add up to two new ones (the shared Z sweep's taps and
// the filter's constants), and a small request that takes a cached volume (visfd_ctx::reuses: tiny volumes) makes
// the next volume request a new block.
size_t blob_slab_bytes(const SlabPlan &pl, int64_t nx, int64_t ny, bool masked, int log_hw, int n_sigmas) {
  const int64_t slab = pl.slab1 - pl.slab0;
  const size_t vol = visfd_ctx::block_bytes((size_t)slab * (size_t)nx * (size_t)ny * sizeof(float));
  const size_t lists = 2 * visfd_ctx::block_bytes((size_t)blob_rows(nx, ny, pl.own1 - pl.own0) * 4 * sizeof(float)) +
                       visfd_ctx::block_bytes(2 * sizeof(unsigned long long));
  // dog_device's largest small request: both Gaussians' taps and edge profiles
  const size_t small = visfd_ctx::block_bytes(2 * (size_t)(3 * (2 * log_hw + 1) + nx + ny + slab) * sizeof(float));
  const size_t scan = (masked ? 5 : 4) * vol + lists;
  const size_t dog = (masked ? 4 : 2) * vol + 2 * (size_t)n_sigmas * small +
                     (visfd_ctx::reuses(vol, small) ? vol : 0);
  return scan + dog;
}

void check_blob_args(const std::string &who, int64_t nx, int64_t ny, int64_t nz, const float *src_host,
                     const float *mask_host, const BlobArgs &a, int64_t capacity,
                     const std::vector<const float *> &outputs) {
  VREQUIRE(nx > 0 && ny > 0 && nz > 0 && src_host && (a.sigmas || a.n_sigmas == 0) && a.n_sigmas >= 0 &&
               capacity >= 0,
           who + ": bad arguments");
  bool host = !is_device_pointer(src_host) && !is_device_pointer(mask_host);
  for (const float *o : outputs) host = host && !is_device_pointer(o);
  VREQUIRE(host, who + " takes HOST arrays (use visfd_cuda_blob_dog_slab for device-resident data)");
}

// The slabs' lists per scale in slab order, the best scores of the whole image, the final filter, and the first
// `capacity` rows into the caller's buffers.
void finish_blobs(const std::vector<BlobSlab> &slabs, const BlobArgs &a, int64_t capacity, float *min_crds,
                  float *min_sigma, float *min_score, int64_t *n_minima, float *max_crds, float *max_sigma,
                  float *max_score, int64_t *n_maxima) {
  auto concat = [&](BlobList BlobSlab::*list) {
    BlobList out;
    std::vector<size_t> at(slabs.size(), 0);   // next row of each slab
    for (int i = 0; i < a.n_sigmas; i++)
      for (size_t r = 0; r < slabs.size(); r++) {
        const BlobList &l = slabs[r].*list;
        const size_t k0 = at[r], k1 = k0 + (size_t)l.scale_rows[(size_t)i];
        out.crds.insert(out.crds.end(), l.crds.begin() + 3 * k0, l.crds.begin() + 3 * k1);
        out.sigma.insert(out.sigma.end(), l.sigma.begin() + k0, l.sigma.begin() + k1);
        out.score.insert(out.score.end(), l.score.begin() + k0, l.score.begin() + k1);
        at[r] = k1;
      }
    return out;
  };
  BlobList minima = concat(&BlobSlab::minima), maxima = concat(&BlobSlab::maxima);
  float gmin = 1.0f, gmax = -1.0f;   // feature.hpp:122-123
  for (const BlobSlab &s : slabs) {
    gmin = std::min(gmin, s.best[0]);
    gmax = std::max(gmax, s.best[1]);
  }
  blob_final_filter(minima, maxima, a.minima_threshold, a.maxima_threshold, a.use_threshold_ratios, gmin, gmax);
  emit_blob_list(minima, capacity, min_crds, min_sigma, min_score, n_minima);
  emit_blob_list(maxima, capacity, max_crds, max_sigma, max_score, n_maxima);
}

int blob_multi(const char *name, int ndev, const int *devices, int64_t nx, int64_t ny, int64_t nz,
               const float *src_host, const float *mask_host, const BlobArgs &a, int64_t capacity, float *min_crds,
               float *min_sigma, float *min_score, int64_t *n_minima, float *max_crds, float *max_sigma,
               float *max_score, int64_t *n_maxima, double *device_ms) {
  try {
    const std::string who(name);
    VREQUIRE(ndev >= 1 && devices, who + ": need at least one device");
    check_blob_args(who, nx, ny, nz, src_host, mask_host, a, capacity,
                    {min_crds, min_sigma, min_score, max_crds, max_sigma, max_score});
    const int world = std::min(ndev, max_slabs(nz));
    const std::vector<SlabPlan> plans = make_plans(nz, world, blob_halfwidth(a), 0, 0);

    std::lock_guard<std::mutex> lock(g_call_mutex);
    std::vector<BlobSlab> slabs((size_t)world);
    for (int r = 0; r < world; r++) {
      slabs[(size_t)r].plan = plans[(size_t)r];
      slabs[(size_t)r].ctx = context_for(name, r, devices[r]);
    }
    for_each_slab(name, slabs, [&](BlobSlab &s) {
      drop_pending_stage_events(s.ctx);
      s.clock.begin(s.ctx->stream);
      blob_slab(s, nx, ny, nz, src_host, mask_host, a);
      s.clock.end(s.ctx->stream);
    });
    finish_blobs(slabs, a, capacity, min_crds, min_sigma, min_score, n_minima, max_crds, max_sigma, max_score,
                 n_maxima);
    if (device_ms)
      for (int r = 0; r < ndev; r++) device_ms[r] = r < world ? slabs[(size_t)r].clock.ms : 0.0;
    return 0;
  } catch (const std::exception &ex) {
    set_last_error(ex.what());
    return 1;
  }
}

int blob_stream(const char *name, visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, const float *src_host,
                const float *mask_host, const BlobArgs &a, int64_t device_bytes, int64_t capacity, float *min_crds,
                float *min_sigma, float *min_score, int64_t *n_minima, float *max_crds, float *max_sigma,
                float *max_score, int64_t *n_maxima, int64_t *n_slabs_out) {
  try {
    const std::string who(name);
    VREQUIRE(ctx != nullptr, who + ": context is NULL");
    VREQUIRE(device_bytes >= 0, who + ": bad arguments");
    check_blob_args(who, nx, ny, nz, src_host, mask_host, a, capacity,
                    {min_crds, min_sigma, min_score, max_crds, max_sigma, max_score});
    const int64_t budget = stream_budget(ctx, device_bytes);
    const int log_hw = blob_halfwidth(a);
    size_t need = 0;
    const int n = fewest_slabs(nz, log_hw, 0, 0, budget, [&](const SlabPlan &pl) {
      return blob_slab_bytes(pl, nx, ny, mask_host != nullptr, log_hw, a.n_sigmas);
    }, &need);
    if (n == 0) throw too_small(who, "blob detection", need, budget);
    const std::vector<SlabPlan> plans = make_plans(nz, n, log_hw, 0, 0);
    std::vector<BlobSlab> slabs((size_t)n);
    for (size_t r = 0; r < slabs.size(); r++) {
      slabs[r].ctx = ctx;
      slabs[r].plan = plans[r];
      try {
        blob_slab(slabs[r], nx, ny, nz, src_host, mask_host, a);
      } catch (const std::exception &ex) {
        throw Error(who + ", slab " + std::to_string(r) + " of " + std::to_string(n) + ": " + ex.what());
      }
      release_cache(ctx);
    }
    finish_blobs(slabs, a, capacity, min_crds, min_sigma, min_score, n_minima, max_crds, max_sigma, max_score,
                 n_maxima);
    if (n_slabs_out) *n_slabs_out = n;
    return 0;
  } catch (const std::exception &ex) {
    set_last_error(ex.what());
    reset_after_failure(ctx);
    return 1;
  }
}

// ---- ApplyGauss / ApplyDog / ApplyLog over Z-slabs -----------------------------------------------------------
// A slab uploads its planes, halo included, runs the slab form of gauss_device / dog_device (z_offset = its first
// plane, nz_global = nz: zero taps, edge profiles and masked denominators are those of the whole volume) and
// delivers its own planes into the caller's array.  The halo is the filter's Z half-width.
// dst_host may be src_host, as for the one-shot host call: delivering a slab overwrites raw planes that later slabs
// read as their lower halo, so multi delivers only once every slab has uploaded, and stream keeps those planes in
// a host buffer (the carry) before it delivers.

// A checked visfd_filter_params: both Gaussians' sigmas and half-widths (a Gaussian alone: the same one twice).
struct Filter {
  int kind = VISFD_FILTER_GAUSS;
  float sa[3], sb[3];
  int hwa[3], hwb[3];
  bool normalize = true;
  float scale = 1.0f;   // LoG: 1 / delta^2
  int z_halfwidth() const { return std::max(hwa[2], hwb[2]); }
};

Filter filter_args(const std::string &who, const visfd_filter_params *p) {
  VREQUIRE(p != nullptr, who + ": params is NULL");
  VREQUIRE(p->kind == VISFD_FILTER_GAUSS || p->kind == VISFD_FILTER_DOG || p->kind == VISFD_FILTER_LOG,
           who + ": unknown filter kind " + std::to_string(p->kind));
  Filter f;
  f.kind = p->kind;
  f.normalize = p->normalize != 0;
  const bool dog = p->kind == VISFD_FILTER_DOG;
  if (p->kind == VISFD_FILTER_LOG) {
    log_params(p->sigma_a, p->delta, p->truncate_ratio, f.sa, f.sb, f.hwa, &f.scale);   // as visfd_cuda_apply_log
    std::copy(f.hwa, f.hwa + 3, f.hwb);
  } else {
    std::copy(p->sigma_a, p->sigma_a + 3, f.sa);
    std::copy(p->hw_a, p->hw_a + 3, f.hwa);
    std::copy(dog ? p->sigma_b : p->sigma_a, (dog ? p->sigma_b : p->sigma_a) + 3, f.sb);
    std::copy(dog ? p->hw_b : p->hw_a, (dog ? p->hw_b : p->hw_a) + 3, f.hwb);
  }
  for (int d = 0; d < 3; d++)   // (NaN fails too)
    VREQUIRE(f.sa[d] >= 0.0f && f.sb[d] >= 0.0f && f.hwa[d] >= 0 && f.hwb[d] >= 0,
             who + ": negative sigma or half-width");
  return f;
}

bool overlap(const float *a, const float *b, size_t n) {
  const uintptr_t x = (uintptr_t)a, y = (uintptr_t)b, bytes = n * sizeof(float);
  return x < y + bytes && y < x + bytes;
}

void check_filter_args(const std::string &who, int64_t nx, int64_t ny, int64_t nz, const float *src_host,
                       const float *mask_host, const float *dst_host) {
  VREQUIRE(nx > 0 && ny > 0 && nz > 0 && nx < (1LL << 31) && ny < (1LL << 31) && nz < (1LL << 31) && src_host &&
               dst_host,
           who + ": bad arguments");
  VREQUIRE(!is_device_pointer(src_host) && !is_device_pointer(mask_host) && !is_device_pointer(dst_host),
           who + " takes HOST arrays (use visfd_cuda_apply_gauss / _dog2 / _log for device-resident data)");
  const size_t n = (size_t)nx * (size_t)ny * (size_t)nz;
  VREQUIRE(!mask_host || !overlap(mask_host, dst_host, n), who + ": the mask must not share memory with dst");
  VREQUIRE(dst_host == src_host || !overlap(src_host, dst_host, n), who + ": dst must be src or apart from it");
}

struct FilterSlab {
  visfd_ctx *ctx = nullptr;
  SlabPlan plan;
  Scratch<float> out;   // every plane of the slab, filtered
  float A = 0.0f, B = 0.0f;
  DeviceClock clock;
};

// Uploads the slab's planes, halo included, and filters them into s.out.  carry (may be NULL): raw source planes
// from global plane carry0 up to the slab's own0, which the upload takes instead of the caller's array.
void filter_slab(FilterSlab &s, const Filter &f, int64_t nx, int64_t ny, int64_t nz, const float *src_host,
                 const float *mask_host, const float *carry, int64_t carry0) {
  const SlabPlan &pl = s.plan;
  const size_t plane = (size_t)nx * (size_t)ny;
  const int64_t nzl = pl.slab1 - pl.slab0;
  const size_t n = (size_t)nzl * plane;
  const int64_t split = carry ? pl.own0 : pl.slab0;   // the planes below it come from the carry
  Scratch<float> src(s.ctx, n), mask;
  s.out.reset(s.ctx, n);
  {
    StageTimer t(s.ctx, "h2d");
    if (split > pl.slab0)
      VCK(cudaMemcpyAsync(src.get(), carry + (size_t)(pl.slab0 - carry0) * plane,
                          (size_t)(split - pl.slab0) * plane * sizeof(float), cudaMemcpyHostToDevice, s.ctx->stream));
    VCK(cudaMemcpyAsync(src.get() + (size_t)(split - pl.slab0) * plane, src_host + (size_t)split * plane,
                        (size_t)(pl.slab1 - split) * plane * sizeof(float), cudaMemcpyHostToDevice, s.ctx->stream));
    if (mask_host) {
      mask.reset(s.ctx, n);
      VCK(cudaMemcpyAsync(mask.get(), mask_host + (size_t)pl.slab0 * plane, n * sizeof(float),
                          cudaMemcpyHostToDevice, s.ctx->stream));
    }
  }
  if (f.kind == VISFD_FILTER_GAUSS) {
    s.A = gauss_device(s.ctx, nx, ny, nzl, pl.slab0, nz, src.get(), s.out.get(), mask.get(), f.sa, f.hwa, f.normalize,
                       nullptr, 1.0f);
  } else {
    dog_device(s.ctx, nx, ny, nzl, pl.slab0, nz, src.get(), s.out.get(), mask.get(), f.sa, f.sb, f.hwa, f.scale, &s.A,
               &s.B, f.hwb);
    if (f.kind == VISFD_FILTER_LOG) {   // as visfd_cuda_apply_log_slab: the peak heights are scaled as well
      s.A *= f.scale;
      s.B *= f.scale;
    }
  }
  // the upload has read the caller's planes once this returns: a delivery may overwrite them
  VCK(cudaStreamSynchronize(s.ctx->stream));
  resolve_stage_times(s.ctx);
}

// Copies the slab's own planes into the caller's array.
void deliver_slab(FilterSlab &s, int64_t nx, int64_t ny, float *dst_host) {
  const SlabPlan &pl = s.plan;
  const size_t plane = (size_t)nx * (size_t)ny;
  {
    StageTimer t(s.ctx, "d2h");
    VCK(cudaMemcpyAsync(dst_host + (size_t)pl.own0 * plane, s.out.get() + (size_t)(pl.own0 - pl.slab0) * plane,
                        (size_t)(pl.own1 - pl.own0) * plane * sizeof(float), cudaMemcpyDeviceToHost, s.ctx->stream));
  }
  VCK(cudaStreamSynchronize(s.ctx->stream));
  resolve_stage_times(s.ctx);
}

// The device bytes the pool holds at most while a slab of visfd_cuda_filter_stream runs, in the blocks
// visfd_ctx::alloc takes: the source (+ mask) and the filtered slab, plus the filter's workspace.  After the trim
// that precedes every slab the pool cannot hold more than the sum of the filter's requests.  A Gaussian's
// requests are separable_workspace_bytes.  DoG and LoG add the first Gaussian's volume to one of dog_device's two
// paths, chosen from the slab's shape (x2_qualifies on ny times its planes), so both are counted: the fused path's
// block of both filters' taps and edge profiles plus one scratch volume, or the shared Z sweep's taps plus both
// Gaussians' separable workspaces.
size_t filter_slab_bytes(const SlabPlan &pl, int64_t nx, int64_t ny, bool masked, const Filter &f) {
  const int64_t slab = pl.slab1 - pl.slab0;
  const size_t vol = visfd_ctx::block_bytes((size_t)slab * (size_t)nx * (size_t)ny * sizeof(float));
  const size_t held = (masked ? 3 : 2) * vol;
  if (f.kind == VISFD_FILTER_GAUSS) return held + separable_workspace_bytes(nx, ny, slab, f.hwa, masked, f.normalize);
  const size_t per = (size_t)(2 * f.hwa[0] + 1 + 2 * f.hwa[1] + 1 + 2 * f.hwa[2] + 1 + nx + ny + slab);
  const size_t fused = visfd_ctx::block_bytes(2 * per * sizeof(float)) + vol;
  const size_t two_calls = visfd_ctx::block_bytes(2 * (size_t)(2 * f.z_halfwidth() + 1) * sizeof(float)) +
                           separable_workspace_bytes(nx, ny, slab, f.hwa, masked, true) +
                           separable_workspace_bytes(nx, ny, slab, f.hwb, masked, true);
  return held + vol + std::max(fused, two_calls);
}

int filter_multi(const char *name, int ndev, const int *devices, int64_t nx, int64_t ny, int64_t nz,
                 const float *src_host, const float *mask_host, const visfd_filter_params *p, float *dst_host,
                 float *A_out, float *B_out, double *device_ms) {
  try {
    const std::string who(name);
    VREQUIRE(ndev >= 1 && devices, who + ": need at least one device");
    check_filter_args(who, nx, ny, nz, src_host, mask_host, dst_host);
    const Filter f = filter_args(who, p);
    const int world = std::min(ndev, max_slabs(nz));
    const std::vector<SlabPlan> plans = make_plans(nz, world, f.z_halfwidth(), 0, 0);

    std::lock_guard<std::mutex> lock(g_call_mutex);
    std::vector<FilterSlab> slabs((size_t)world);
    for (int r = 0; r < world; r++) {
      slabs[(size_t)r].plan = plans[(size_t)r];
      slabs[(size_t)r].ctx = context_for(name, r, devices[r]);
    }
    for_each_slab(name, slabs, [&](FilterSlab &s) {
      drop_pending_stage_events(s.ctx);
      s.clock.begin(s.ctx->stream);
      filter_slab(s, f, nx, ny, nz, src_host, mask_host, nullptr, 0);
    });
    // every slab has read its planes: delivering cannot overwrite a plane that a slab has still to read
    for_each_slab(name, slabs, [&](FilterSlab &s) {
      deliver_slab(s, nx, ny, dst_host);
      s.out.free();
      s.clock.end(s.ctx->stream);
      // a slab's blocks are volume-sized and a later call's slabs may not fit them: cached, they would keep that
      // memory from every other context on the device
      release_cache(s.ctx);
    });

    if (A_out) *A_out = slabs[0].A;   // the peak heights depend on the taps alone
    if (B_out) *B_out = slabs[0].B;
    if (device_ms)
      for (int r = 0; r < ndev; r++) device_ms[r] = r < world ? slabs[(size_t)r].clock.ms : 0.0;
    return 0;
  } catch (const std::exception &ex) {
    set_last_error(ex.what());
    return 1;
  }
}

int filter_stream(const char *name, visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, const float *src_host,
                  const float *mask_host, const visfd_filter_params *p, int64_t device_bytes, float *dst_host,
                  float *A_out, float *B_out, int64_t *n_slabs_out) {
  try {
    const std::string who(name);
    check_filter_args(who, nx, ny, nz, src_host, mask_host, dst_host);
    const Filter f = filter_args(who, p);
    VREQUIRE(device_bytes >= 0, who + ": negative device_bytes");
    VREQUIRE(ctx != nullptr, who + ": context is NULL");
    const int64_t budget = stream_budget(ctx, device_bytes);
    const int zhw = f.z_halfwidth();
    size_t need = 0;
    const int n = fewest_slabs(nz, zhw, 0, 0, budget, [&](const SlabPlan &pl) {
      return filter_slab_bytes(pl, nx, ny, mask_host != nullptr, f);
    }, &need);
    if (n == 0) throw too_small(who, "the filter", need, budget);
    const std::vector<SlabPlan> plans = make_plans(nz, n, zhw, 0, 0);
    const size_t plane = (size_t)nx * (size_t)ny;
    // dst_host == src_host: the raw planes [carry0, own0 of the next slab) that a later slab still reads.  Slab
    // starts never decrease, so the planes below the next slab's start are dropped: at most halo + 7 planes.
    const bool aliased = dst_host == src_host;
    std::vector<float> carry;
    int64_t carry0 = 0;
    float A = 0.0f, B = 0.0f;
    for (int r = 0; r < n; r++) {
      FilterSlab s;
      s.ctx = ctx;
      s.plan = plans[(size_t)r];
      try {
        filter_slab(s, f, nx, ny, nz, src_host, mask_host, aliased ? carry.data() : nullptr, carry0);
        if (aliased && r + 1 < n) {
          const int64_t keep0 = plans[(size_t)r + 1].slab0, mid = std::max(keep0, s.plan.own0);
          std::vector<float> next((size_t)(s.plan.own1 - keep0) * plane);
          if (keep0 < s.plan.own0)
            std::copy(carry.begin() + (keep0 - carry0) * plane, carry.begin() + (s.plan.own0 - carry0) * plane,
                      next.begin());
          std::copy(src_host + (size_t)mid * plane, src_host + (size_t)s.plan.own1 * plane,
                    next.begin() + (mid - keep0) * plane);
          carry.swap(next);
          carry0 = keep0;
        }
        deliver_slab(s, nx, ny, dst_host);
      } catch (const std::exception &ex) {
        throw Error(who + ", slab " + std::to_string(r) + " of " + std::to_string(n) + ": " + ex.what());
      }
      if (r == 0) {   // the peak heights depend on the taps alone
        A = s.A;
        B = s.B;
      }
      s.out.free();
      release_cache(ctx);
    }
    if (A_out) *A_out = A;
    if (B_out) *B_out = B;
    if (n_slabs_out) *n_slabs_out = n;
    return 0;
  } catch (const std::exception &ex) {
    set_last_error(ex.what());
    reset_after_failure(ctx);
    return 1;
  }
}

}  // namespace

extern "C" int visfd_cuda_filter_multi(int ndev, const int *devices, int64_t nx, int64_t ny, int64_t nz,
                                       const float *src_host, const float *mask_host, const visfd_filter_params *p,
                                       float *dst_host, float *A_out, float *B_out, double *device_ms) {
  return filter_multi("visfd_cuda_filter_multi", ndev, devices, nx, ny, nz, src_host, mask_host, p, dst_host, A_out,
                      B_out, device_ms);
}

extern "C" int visfd_cuda_filter_stream(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, const float *src_host,
                                        const float *mask_host, const visfd_filter_params *p, int64_t device_bytes,
                                        float *dst_host, float *A_out, float *B_out, int64_t *n_slabs_out) {
  return filter_stream("visfd_cuda_filter_stream", ctx, nx, ny, nz, src_host, mask_host, p, device_bytes, dst_host,
                       A_out, B_out, n_slabs_out);
}

extern "C" int visfd_cuda_membrane_multi(int ndev, const int *devices, int64_t nx, int64_t ny, int64_t nz,
                                         const float *src_host, const float *mask_host,
                                         const visfd_membrane_params *p, float *out_host, float *threshold_out,
                                         double *device_ms /* ndev values or NULL */) {
  return membrane_multi("visfd_cuda_membrane_multi", ndev, devices, nx, ny, nz, src_host, mask_host, p, 0.0f, 1,
                        out_host, threshold_out, device_ms);
}

extern "C" int visfd_cuda_membrane_multi_background(int ndev, const int *devices, int64_t nx, int64_t ny, int64_t nz,
                                                    const float *src_host, const float *mask_host,
                                                    const visfd_membrane_params *p, float background_sigma,
                                                    int normalize_near_boundaries, float *out_host,
                                                    float *threshold_out, double *device_ms) {
  return membrane_multi("visfd_cuda_membrane_multi_background", ndev, devices, nx, ny, nz, src_host, mask_host, p,
                        background_sigma, normalize_near_boundaries, out_host, threshold_out, device_ms);
}

extern "C" int visfd_cuda_membrane_stream(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, const float *src_host,
                                          const float *mask_host, const visfd_membrane_params *p,
                                          int64_t device_bytes, float *out_host, float *threshold_out,
                                          int64_t *n_slabs_out) {
  return membrane_stream("visfd_cuda_membrane_stream", ctx, nx, ny, nz, src_host, mask_host, p, 0.0f, 1,
                         device_bytes, out_host, threshold_out, n_slabs_out);
}

extern "C" int visfd_cuda_membrane_stream_background(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz,
                                                     const float *src_host, const float *mask_host,
                                                     const visfd_membrane_params *p, float background_sigma,
                                                     int normalize_near_boundaries, int64_t device_bytes,
                                                     float *out_host, float *threshold_out, int64_t *n_slabs_out) {
  return membrane_stream("visfd_cuda_membrane_stream_background", ctx, nx, ny, nz, src_host, mask_host, p,
                         background_sigma, normalize_near_boundaries, device_bytes, out_host, threshold_out,
                         n_slabs_out);
}

extern "C" int visfd_cuda_membrane_connect_multi(int ndev, const int *devices, int64_t nx, int64_t ny, int64_t nz,
                                                 const float *src_host, const float *mask_host,
                                                 const visfd_membrane_params *p, float background_sigma,
                                                 int normalize_near_boundaries, const visfd_connect_params *c,
                                                 float *out_host, float *threshold_out, int64_t *labels_host,
                                                 float *direction_host, int64_t *n_clusters, float *cluster_maxima,
                                                 int64_t maxima_capacity, int64_t *n_maxima, double *device_ms) {
  const char *name = "visfd_cuda_membrane_connect_multi";
  try {
    VREQUIRE(ndev >= 1 && devices, std::string(name) + ": need at least one device");
    Connect cn = connect_args(name, nx, ny, nz, src_host, p, background_sigma, c, out_host, labels_host,
                              direction_host, maxima_capacity);
    cn.n_clusters = n_clusters;
    cn.n_maxima = n_maxima;
    cn.maxima = cluster_maxima;
    return membrane_multi(name, ndev, devices, nx, ny, nz, src_host, mask_host, p, background_sigma,
                          normalize_near_boundaries, out_host, threshold_out, device_ms, &cn);
  } catch (const std::exception &ex) {
    set_last_error(ex.what());
    return 1;
  }
}

extern "C" int visfd_cuda_membrane_connect_stream(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz,
                                                  const float *src_host, const float *mask_host,
                                                  const visfd_membrane_params *p, float background_sigma,
                                                  int normalize_near_boundaries, const visfd_connect_params *c,
                                                  int64_t device_bytes, float *out_host, float *threshold_out,
                                                  int64_t *labels_host, float *direction_host, int64_t *n_clusters,
                                                  float *cluster_maxima, int64_t maxima_capacity, int64_t *n_maxima,
                                                  int64_t *n_slabs_out) {
  const char *name = "visfd_cuda_membrane_connect_stream";
  try {
    // the arguments are checked before the context is used
    Connect cn = connect_args(name, nx, ny, nz, src_host, p, background_sigma, c, out_host, labels_host,
                              direction_host, maxima_capacity);
    VREQUIRE(device_bytes >= 0, std::string(name) + ": negative device_bytes");
    cn.n_clusters = n_clusters;
    cn.n_maxima = n_maxima;
    cn.maxima = cluster_maxima;
    return membrane_stream(name, ctx, nx, ny, nz, src_host, mask_host, p, background_sigma, normalize_near_boundaries,
                           device_bytes, out_host, threshold_out, n_slabs_out, &cn);
  } catch (const std::exception &ex) {
    set_last_error(ex.what());
    return 1;
  }
}

extern "C" int visfd_cuda_blob_dog_multi(int ndev, const int *devices, int64_t nx, int64_t ny, int64_t nz,
                                         const float *src_host, const float *mask_host, const float *sigmas,
                                         int n_sigmas, float delta, float truncate_ratio, float minima_threshold,
                                         float maxima_threshold, int use_threshold_ratios, int64_t capacity,
                                         float *min_crds, float *min_sigma, float *min_score, int64_t *n_minima,
                                         float *max_crds, float *max_sigma, float *max_score, int64_t *n_maxima,
                                         double *device_ms) {
  const BlobArgs a{sigmas, n_sigmas, delta, truncate_ratio, minima_threshold, maxima_threshold, use_threshold_ratios};
  return blob_multi("visfd_cuda_blob_dog_multi", ndev, devices, nx, ny, nz, src_host, mask_host, a, capacity,
                    min_crds, min_sigma, min_score, n_minima, max_crds, max_sigma, max_score, n_maxima, device_ms);
}

extern "C" int visfd_cuda_blob_dog_stream(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, const float *src_host,
                                          const float *mask_host, const float *sigmas, int n_sigmas, float delta,
                                          float truncate_ratio, float minima_threshold, float maxima_threshold,
                                          int use_threshold_ratios, int64_t device_bytes, int64_t capacity,
                                          float *min_crds, float *min_sigma, float *min_score, int64_t *n_minima,
                                          float *max_crds, float *max_sigma, float *max_score, int64_t *n_maxima,
                                          int64_t *n_slabs_out) {
  const BlobArgs a{sigmas, n_sigmas, delta, truncate_ratio, minima_threshold, maxima_threshold, use_threshold_ratios};
  return blob_stream("visfd_cuda_blob_dog_stream", ctx, nx, ny, nz, src_host, mask_host, a, device_bytes, capacity,
                     min_crds, min_sigma, min_score, n_minima, max_crds, max_sigma, max_score, n_maxima, n_slabs_out);
}
