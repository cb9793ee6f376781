// multi.cu -- the membrane pipeline on several GPUs of one node behind ONE C call (SURVEY 8b/8e): a C++ host such
// as filter_mrc hands over its host arrays and gets the result back, with no MPI, no Python and no process per GPU.
//
//   visfd_cuda_membrane_multi(ndev, devices, nx, ny, nz, src_host, mask_host, params, out_host, &threshold)
//
// One slab per device.  The volume is cut into Z-slabs exactly as visfd_b200/slab.py does for the
// process-per-GPU driver (rank boundaries on multiples of 8 planes, slabs widened by a halo of RAW SOURCE planes,
// halo = tv_halfwidth + 1 + gauss_halfwidth, slab start rounded down to a multiple of 8), so every stage is
// slab-local and the result is bit-identical to the one-GPU result.  Because the source lives in host memory, each
// device uploads its slab -- halo included -- straight from the caller's array over its own PCIe link: there is no
// device-to-device halo traffic at all.
//
// The call runs in phases.  A phase runs every slab at once (slab 0 on the calling thread, the others on threads of
// their own) and is joined on the host before the next one starts, so a slab that fails cannot leave the others
// waiting for it: (1) upload + ridge saliency; (2) for the `-tv-best` cut, one phase per round of the radix select
// (select_threshold), in which every slab histograms its own planes into 2048 bins and the calling thread sums them
// (the cut must be a GLOBAL order statistic, bin/filter_mrc/handlers.cpp:1766-1782); (3) voting, each device
// delivering its planes of the result into the caller's array chunk by chunk behind its voting kernels
// (visfd_cuda_vote_slab_host).
//
// The same device may be listed several times (two slabs on one GPU): that is how the one-GPU test box exercises
// the slab logic.
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

// visfd_b200/slab.py: partition() + make_plan()
std::vector<SlabPlan> make_plans(int64_t nz, int world, int gauss_hw, int tv_hw) {
  const int64_t unit = (nz / 8 >= world) ? 8 : 1;
  const int64_t base = (nz / unit) / world, rem = (nz / unit) % world;
  const int64_t halo = tv_hw > 0 ? tv_hw + 1 + gauss_hw : 1 + gauss_hw;
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

// What a slab keeps on its device from one phase to the next.
struct Slab {
  visfd_ctx *ctx = nullptr;
  SlabPlan plan;
  Scratch<float> mask, smoothed, saliency;
  cudaEvent_t start = nullptr, stop = nullptr;   // device time: first upload to last download
  double ms = 0.0;
  uint64_t hist[HIST_BINS];
  ~Slab() {
    if (start) cudaEventDestroy(start);
    if (stop) cudaEventDestroy(stop);
  }
};

// Runs fn(slab) for every slab at once, slab 0 on the calling thread and the others on threads of their own, each
// on its slab's device.  Returns when all of them have finished, and then throws the error of the first slab that
// failed.
template <typename Fn>
void for_each_slab(std::vector<Slab> &slabs, const Fn &fn) {
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
      throw Error("visfd_cuda_membrane_multi, slab " + std::to_string(r) + " on device " +
                  std::to_string(slabs[r].ctx->device) + ": " + errors[r]);
}

}  // namespace

extern "C" int visfd_cuda_membrane_multi(int ndev, const int *devices, int64_t nx, int64_t ny, int64_t nz,
                                         const float *src_host, const float *mask_host,
                                         const visfd_membrane_params *p, float *out_host, float *threshold_out,
                                         double *device_ms /* ndev values or NULL */) {
  try {
    VREQUIRE(ndev >= 1 && devices, "visfd_cuda_membrane_multi: need at least one device");
    VREQUIRE(nx > 0 && ny > 0 && nz > 0 && src_host && p && out_host, "visfd_cuda_membrane_multi: bad arguments");
    VREQUIRE(!is_device_pointer(src_host) && !is_device_pointer(out_host) && !is_device_pointer(mask_host),
             "visfd_cuda_membrane_multi takes HOST arrays (use the slab entry points for device-resident data)");
    const int gauss_hw = (int)floor(p->sigma * p->truncate_ratio);
    const int tv_hw = p->tv_sigma > 0.0f ? tv_halfwidth(p->tv_sigma, p->tv_cutoff_ratio) : 0;
    const int world = (int)std::min<int64_t>(ndev, std::max<int64_t>(1, nz / 8));   // at least 8 planes per worker
    const std::vector<SlabPlan> plans = make_plans(nz, world, gauss_hw, tv_hw);
    const size_t plane = (size_t)nx * (size_t)ny;

    std::lock_guard<std::mutex> lock(g_call_mutex);
    std::vector<Slab> slabs((size_t)world);
    for (int r = 0; r < world; r++) {
      slabs[(size_t)r].ctx = context_for(r, devices[r]);
      slabs[(size_t)r].plan = plans[(size_t)r];
    }

    // ---- upload the slab, halo included, and compute its ridge saliency ----
    for_each_slab(slabs, [&](Slab &s) {
      const SlabPlan &pl = s.plan;
      const size_t n = (size_t)(pl.slab1 - pl.slab0) * plane;
      VCK(cudaEventCreate(&s.start));
      VCK(cudaEventCreate(&s.stop));
      VCK(cudaEventRecord(s.start, s.ctx->stream));
      Scratch<float> src(s.ctx, n);   // the raw slab is not needed after this phase
      s.smoothed.reset(s.ctx, n);
      s.saliency.reset(s.ctx, n);
      VCK(cudaMemcpyAsync(src.get(), src_host + (size_t)pl.slab0 * plane, n * sizeof(float), cudaMemcpyHostToDevice,
                          s.ctx->stream));
      if (mask_host) {
        s.mask.reset(s.ctx, n);
        VCK(cudaMemcpyAsync(s.mask.get(), mask_host + (size_t)pl.slab0 * plane, n * sizeof(float),
                            cudaMemcpyHostToDevice, s.ctx->stream));
      }
      if (visfd_cuda_ridge_saliency_slab(s.ctx, nx, ny, pl.slab1 - pl.slab0, pl.slab0, nz, src.get(), s.mask.get(),
                                         p->sigma, p->truncate_ratio, p->eival_order, VISFD_SCORE_PLANAR,
                                         s.smoothed.get(), s.saliency.get()) != 0)
        throw Error(visfd_cuda_last_error());
    });

    // ---- global cut: radix select over the slabs' own planes ----
    float threshold = p->cut;
    if (p->cut_is_fraction)
      threshold = select_threshold(p->cut, [&](uint32_t prefix, int prefix_bits, uint64_t *hist) {
        for_each_slab(slabs, [&](Slab &s) {
          const size_t own = (size_t)(s.plan.own0 - s.plan.slab0) * plane;
          select_hist_device(s.ctx, (i64)((s.plan.own1 - s.plan.own0) * (int64_t)plane), s.saliency.get() + own,
                             mask_host ? s.mask.get() + own : nullptr, prefix, prefix_bits, s.hist);
        });
        std::fill(hist, hist + HIST_BINS, 0);
        for (const Slab &s : slabs)
          for (int b = 0; b < HIST_BINS; b++) hist[b] += s.hist[b];
      });

    // ---- voting on the own planes, delivered into the caller's array ----
    for_each_slab(slabs, [&](Slab &s) {
      const SlabPlan &pl = s.plan;
      Scratch<float> out(s.ctx, (size_t)(pl.own1 - pl.own0) * plane);
      if (visfd_cuda_vote_slab_host(s.ctx, nx, ny, pl.slab1 - pl.slab0, pl.slab0, nz, pl.own0 - pl.slab0,
                                    pl.own1 - pl.slab0, pl.vote0 - pl.slab0, pl.vote1 - pl.slab0, s.saliency.get(),
                                    s.smoothed.get(), s.mask.get(), threshold, p, out.get(), nullptr,
                                    out_host + (size_t)pl.own0 * plane) != 0)
        throw Error(visfd_cuda_last_error());
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
