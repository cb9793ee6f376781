// multi.cu -- the membrane pipeline over Z-slabs behind ONE C call, for host arrays (SURVEY 8b/8e): a C++ host such
// as filter_mrc hands over its host arrays and gets the result back, with no MPI, no Python and no process per GPU.
//
//   visfd_cuda_membrane_multi(ndev, devices, nx, ny, nz, src_host, mask_host, params, out_host, &threshold)
//     one slab per device, all slabs at once: every GPU of the node on one volume;
//   visfd_cuda_membrane_stream(ctx, nx, ny, nz, src_host, mask_host, params, device_bytes, out_host, &threshold)
//     one device, the slabs one after another within a device-memory budget: volumes whose working set does not fit.
// Their _background forms add `-membrane-background`: both scores multiplied by the peak height
// source - Gauss(source, background_sigma), as visfd_cuda_membrane_background does on one GPU.
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

visfd_ctx *context_for(int slot, int device) {
  if ((int)g_ctx.size() <= slot) g_ctx.resize((size_t)slot + 1, {-1, nullptr});
  auto &e = g_ctx[(size_t)slot];
  if (e.second && e.first != device) {
    visfd_cuda_destroy(e.second);
    e.second = nullptr;
  }
  if (!e.second) {
    visfd_ctx *c = nullptr;
    if (visfd_cuda_init(device, &c) != 0) throw Error(std::string("visfd_cuda_membrane_multi: ") + visfd_cuda_last_error());
    e = {device, c};
  }
  return e.second;
}

// What a slab keeps on its device from one step to the next.
struct Slab {
  visfd_ctx *ctx = nullptr;
  SlabPlan plan;
  Scratch<float> mask, smoothed, saliency;
  Scratch<float> peak;   // with the background: the peak height of every plane of the slab, until the vote ends
  cudaEvent_t start = nullptr, stop = nullptr;   // device time: first upload to last download
  double ms = 0.0;
  uint64_t hist[HIST_BINS];
  ~Slab() {
    if (start) cudaEventDestroy(start);
    if (stop) cudaEventDestroy(stop);
  }
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
template <typename Fn>
void for_each_slab(const char *name, std::vector<Slab> &slabs, const Fn &fn) {
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
size_t slab_bytes(const SlabPlan &pl, int64_t nx, int64_t ny, bool masked, const visfd_membrane_params *p,
                  int gauss_hw, const Background &bg, bool vote, uint64_t voters) {
  const size_t plane = (size_t)nx * (size_t)ny;
  const int64_t slab = pl.slab1 - pl.slab0;
  const size_t vol = visfd_ctx::block_bytes((size_t)slab * plane * sizeof(float));
  const int hw[3] = {gauss_hw, gauss_hw, gauss_hw}, hw_bg[3] = {bg.hw, bg.hw, bg.hw};
  const size_t peak = bg.on() ? vol : 0;
  const size_t bg_taps = bg.on() ? separable_workspace_bytes(nx, ny, slab, hw_bg, false, false) - vol : 0;
  const size_t ridge = (masked ? 4 : 3) * vol + peak + separable_workspace_bytes(nx, ny, slab, hw, masked, true) + bg_taps;
  if (!vote) return ridge + visfd_ctx::block_bytes(HIST_BINS * sizeof(uint64_t));
  size_t voting = (masked ? 3 : 2) * vol + peak +
                  visfd_ctx::block_bytes((size_t)(pl.own1 - pl.own0) * plane * sizeof(float));
  if (p->tv_sigma > 0.0f) {
    // visfd_cuda_vote_slab_host widens the voter planes down to a global multiple of 8: up to 7 more planes, whose
    // saliency may be incomplete, so they may add up to 7 planes of voters to the count of the whole volume
    const int64_t vplanes = std::min(pl.vote1 - pl.vote0 + 7, slab);
    const uint64_t vox = (uint64_t)vplanes * plane;
    const uint64_t n = voters < vox ? std::min(vox, voters + 7 * (uint64_t)plane) : vox;
    voting += tv_workspace_bytes(nx, ny, vplanes, pl.own1 - pl.own0, n);
  }
  return std::max(ridge, voting);
}

// The ridge step's scratch and every block a finished slab leaves behind go back to the device, so that the next
// step or slab allocates afresh rather than next to cached blocks it cannot reuse.
void release_cache(visfd_ctx *ctx) {
  VCK(cudaStreamSynchronize(ctx->stream));
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

int membrane_multi(const char *name, int ndev, const int *devices, int64_t nx, int64_t ny, int64_t nz,
                   const float *src_host, const float *mask_host, const visfd_membrane_params *p,
                   float background_sigma, int normalize, float *out_host, float *threshold_out,
                   double *device_ms) {
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
    for (int r = 0; r < world; r++) slabs[(size_t)r].ctx = context_for(r, devices[r]);
    auto concurrently = [&](const auto &step) { for_each_slab(name, slabs, step); };

    for_each_slab(name, slabs, [&](Slab &s) {
      VCK(cudaEventCreate(&s.start));
      VCK(cudaEventCreate(&s.stop));
      VCK(cudaEventRecord(s.start, s.ctx->stream));
      upload_and_ridge(s, nx, ny, nz, src_host, mask_host, p, bg);
    });

    float threshold = p->cut;
    if (p->cut_is_fraction)
      threshold = select_threshold(p->cut, [&](uint32_t prefix, int prefix_bits, uint64_t *hist) {
        summed_own_hist(slabs, concurrently, plane, mask_host != nullptr, prefix, prefix_bits, hist);
      });

    for_each_slab(name, slabs, [&](Slab &s) {
      vote_to_host(s, nx, ny, nz, threshold, p, out_host);
      VCK(cudaEventRecord(s.stop, s.ctx->stream));
      VCK(cudaEventSynchronize(s.stop));
      float t = 0;
      VCK(cudaEventElapsedTime(&t, s.start, s.stop));
      s.ms = t;
    });

    if (threshold_out) *threshold_out = threshold;
    if (device_ms)
      for (int r = 0; r < ndev; r++) device_ms[r] = r < world ? slabs[(size_t)r].ms : 0.0;
    return 0;
  } catch (const std::exception &ex) {
    set_last_error(ex.what());
    return 1;
  }
}

int membrane_stream(const char *name, visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, const float *src_host,
                    const float *mask_host, const visfd_membrane_params *p, float background_sigma, int normalize,
                    int64_t device_bytes, float *out_host, float *threshold_out, int64_t *n_slabs_out) {
  try {
    const std::string who(name);
    VREQUIRE(ctx != nullptr, who + ": context is NULL");
    VREQUIRE(nx > 0 && ny > 0 && nz > 0 && src_host && p && out_host && device_bytes >= 0, who + ": bad arguments");
    VREQUIRE(!is_device_pointer(src_host) && !is_device_pointer(out_host) && !is_device_pointer(mask_host),
             who + " takes HOST arrays (use visfd_cuda_membrane for device-resident data)");
    const Background bg = background(who, p, background_sigma, normalize);
    VCK(cudaSetDevice(ctx->device));
    drop_pending_stage_events(ctx);
    release_cache(ctx);   // blocks cached by earlier calls count against the budget
    int64_t budget = device_bytes;
    if (budget == 0) {
      // the margin covers what the call needs outside the pool: the allocation granularity of cudaMalloc, code
      // of kernels loaded on first use, local memory
      size_t free_b = 0, total_b = 0;
      VCK(cudaMemGetInfo(&free_b, &total_b));
      budget = (int64_t)free_b - (int64_t)(1u << 30);
    }
    const int gauss_hw = (int)floor(p->sigma * p->truncate_ratio);
    const int tv_hw = p->tv_sigma > 0.0f ? tv_halfwidth(p->tv_sigma, p->tv_cutoff_ratio) : 0;
    const size_t plane = (size_t)nx * (size_t)ny;
    const bool masked = mask_host != nullptr, vote = p->tv_sigma > 0.0f;

    // The fewest slabs whose every slab fits the budget, 0 if none does; *need: the bytes of the largest slab of
    // the last plan tried.
    auto fewest_slabs = [&](bool vote_pass, uint64_t voters, size_t *need) {
      for (int world = 1; world <= max_slabs(nz); world++) {
        *need = 0;
        for (const SlabPlan &pl : make_plans(nz, world, gauss_hw, tv_hw, bg.hw))
          *need = std::max(*need, slab_bytes(pl, nx, ny, masked, p, gauss_hw, bg, vote_pass, voters));
        if (*need <= (size_t)std::max<int64_t>(budget, 0)) return world;
      }
      return 0;
    };
    auto too_small = [&](const char *pass, size_t need) {
      return Error(who + ": " + std::string(pass) + " needs " + std::to_string(need) +
                   " bytes of device memory in slabs of 8 planes; the budget is " + std::to_string(budget) +
                   " bytes");
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
    const int n_cut = fewest_slabs(false, 0, &need);
    if (n_cut == 0) throw too_small("the upload and ridge step", need);
    float threshold = p->cut;
    uint64_t voters = UINT64_MAX;   // unknown: every voxel of a slab's voter planes may vote
    if (p->cut_is_fraction || (vote && fewest_slabs(true, voters, &need) != n_cut)) {
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

    const int n_vote = fewest_slabs(true, voters, &need);
    if (n_vote == 0) throw too_small("the vote pass", need);
    std::vector<Slab> slabs((size_t)n_vote);
    make_slabs(slabs, make_plans(nz, n_vote, gauss_hw, tv_hw, bg.hw), ctx);
    one_by_one(slabs, [&](Slab &s) {
      release_cache(ctx);   // the ridge step's scratch
      vote_to_host(s, nx, ny, nz, threshold, p, out_host);
    });

    if (threshold_out) *threshold_out = threshold;
    if (n_slabs_out) *n_slabs_out = n_vote;
    return 0;
  } catch (const std::exception &ex) {
    set_last_error(ex.what());
    if (ctx) {
      cudaStreamSynchronize(ctx->stream);
      cudaGetLastError();
      ctx->trim();
    }
    return 1;
  }
}

}  // namespace

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
