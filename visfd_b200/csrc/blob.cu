// blob.cu -- scale-space blob detection, BlobDog (lib/visfd/feature.hpp:56-427):
// a ring of three LoG-filtered volumes (ApplyLog per scale, gauss.cu) and, for every
// interior scale, a strict 80-neighbour extremum test in (x,y,z,scale) that appends
// candidates (x,y,z,score) to a device list through a warp-aggregated atomic cursor.
// Scan traffic: the three volumes are read once from HBM (12 B/voxel); the voxel's own scale
// is held as separable row minima / maxima in registers, the two adjacent scales are only
// touched around the extrema of the own scale.
//
// The reference's running score filter (:267-303) depends on OpenMP thread order; only
// its deterministic consequences are kept: in absolute mode a candidate must beat the
// threshold strictly, in ratio mode candidates are pre-filtered on the device against
// the best score of the PREVIOUS scales (never stricter than the final filter, :362-417)
// and the final filter runs on the host once the global best scores are known.
#include "common.cuh"
#include "kernels.cuh"
#include <algorithm>
#include <cmath>
#include <limits>
#include <numeric>

namespace visfd_cuda {

struct BlobCand {
  float x, y, z, score;
};

struct BlobScanArgs {
  const float *prev, *cur, *next, *mask;
  int nx, ny, nz;             // nz: planes of the slab
  int z_offset, nz_global;    // the slab's first plane in the image, the image's planes
  int own_z0;                 // first receiver plane (slab-local); the grid spans the receiver planes
  float min_thr, max_thr;     // device pre-filter: minima need score < min_thr, maxima > max_thr
  BlobCand *mins, *maxs;
  unsigned long long *counters;  // [0] minima, [1] maxima
  unsigned long long capacity;
};

__device__ __forceinline__ void append(BlobCand *list, unsigned long long *counter,
                                       unsigned long long capacity, bool pred, const BlobCand &c) {
  unsigned m = __ballot_sync(0xffffffffu, pred);
  if (!m) return;
  const int lane = threadIdx.x & 31;
  unsigned long long base = 0;
  const int leader = __ffs(m) - 1;
  if (lane == leader) base = atomicAdd(counter, (unsigned long long)__popc(m));
  base = __shfl_sync(0xffffffffu, base, leader);
  if (pred) {
    unsigned long long slot = base + __popc(m & ((1u << lane) - 1u));
    if (slot < capacity) list[slot] = c;
  }
}

// A warp owns 32 consecutive x of one y and marches through BLOB_ZC planes.
// Phase A -- the 26 neighbours of the voxel's own scale.  The warp keeps the rows y-1, y, y+1 of the planes
// z-1, z, z+1 in registers (own column per lane; the x-1 / x+1 columns come from the neighbouring lanes by
// shuffle, lanes 0 and 31 load theirs); stepping to the next plane loads three rows, and they are
// requested one plane ahead, so the latency of the kernel's only compulsory traffic (4 B/voxel) is hidden
// behind the comparisons of the plane before.  A strict extremum of its own scale survives.
// Phase B -- survivors are queued in shared memory and, 32 at a time, tested against their 27 + 27
// neighbours in the scales below and above by the WHOLE warp (lane = neighbour, four survivors in
// flight), instead of every voxel's lane walking 54 dependent loads while its 31 neighbours wait.
constexpr int BLOB_ZC = 16;

struct BlobPending {
  unsigned long long at;   // linear index of the voxel in the slab
  float e;
  int x, gz;
  int flags;               // 1 minimum candidate, 2 maximum candidate
};

__device__ __forceinline__ void blob_flush(const BlobScanArgs &a, BlobPending *q, int n, int iy) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const size_t sy = a.nx, sz = (size_t)a.nx * a.ny;
  const ptrdiff_t off = (lane < 27) ? (lane / 9 - 1) * (ptrdiff_t)sz + ((lane / 3) % 3 - 1) * (ptrdiff_t)sy + (lane % 3 - 1) : 0;
  bool my_min = false, my_max = false;
  for (int j0 = 0; j0 < n; j0 += 4) {
    float p[4], nx_[4], es[4];
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const int j = min(j0 + u, n - 1);
      es[u] = q[j].e;
      const size_t at = (size_t)q[j].at + off;
      p[u] = (lane < 27) ? __ldg(a.prev + at) : 0.0f;
      nx_[u] = (lane < 27) ? __ldg(a.next + at) : 0.0f;
    }
#pragma unroll
    for (int u = 0; u < 4; u++) {
      // the reference's tests (feature.hpp:245-258): nb <= e spoils a minimum, nb >= e a maximum
      const bool ok_min = __all_sync(full, lane >= 27 || (!(p[u] <= es[u]) && !(nx_[u] <= es[u])));
      const bool ok_max = __all_sync(full, lane >= 27 || (!(p[u] >= es[u]) && !(nx_[u] >= es[u])));
      if (lane == j0 + u) { my_min = ok_min; my_max = ok_max; }
    }
  }
  const bool mine = lane < n;
  BlobCand cand{0.f, 0.f, 0.f, 0.f};
  int flags = 0;
  if (mine) {
    cand = BlobCand{(float)q[lane].x, (float)iy, (float)q[lane].gz, q[lane].e};
    flags = q[lane].flags;
  }
  __syncwarp();
  append(a.mins, a.counters + 0, a.capacity, mine && (flags & 1) && my_min && cand.score < a.min_thr, cand);
  append(a.maxs, a.counters + 1, a.capacity, mine && (flags & 2) && my_max && cand.score > a.max_thr, cand);
}

// What a warp keeps of one plane of the voxel's own scale (rows y-1, y, y+1 of its 32 columns): the
// minimum and maximum over x-1, x, x+1 of every row -- the separable part of the 3x3x3 test -- plus, for
// the voxel's own row, the value itself and the minimum / maximum of its two x neighbours.
struct BlobPlane {
  float rmin[3], rmax[3];   // per row, over x-1..x+1
  float pmin, pmax;         // over the three rows (the plane as the voxel's z-1 or z+1 neighbour)
  float e, smin, smax;      // own row: centre value, min / max of the x-1 and x+1 values
};

__global__ void __launch_bounds__(256) blob_scan_kernel(BlobScanArgs a, int own_z1) {
  __shared__ BlobPending pending[8][32];
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  BlobPending *q = pending[warp];
  const int ix = blockIdx.x * 64 + (threadIdx.x & 63);
  const int iy = blockIdx.y * 4 + (threadIdx.x >> 6);
  // every neighbour must be inside the image (feature.hpp:245-258); the slab's halo guarantees that a
  // neighbour inside the image is inside the slab.  Row conditions are uniform over the warp.
  if (iy < 1 || iy >= a.ny - 1) return;
  const int z_begin = a.own_z0 + blockIdx.z * BLOB_ZC, z_end = min(z_begin + BLOB_ZC, own_z1);
  const size_t sy = a.nx, sz = (size_t)a.nx * a.ny;
  const bool in_x = ix < a.nx, interior = ix >= 1 && ix < a.nx - 1;
  const bool left = lane == 0 && interior, right = lane == 31 && interior;
  const size_t col = (size_t)iy * sy + ix;

  // raw rows y-1, y, y+1 of plane z (own column, and the outer columns on lanes 0 / 31); planes outside
  // the slab are never needed by a valid voxel
  auto load_plane = [&](int z, float v[3], float l[3], float r[3]) {
    const bool ok = z >= 0 && z < a.nz;
#pragma unroll
    for (int k = 0; k < 3; k++) {
      const size_t row = (size_t)max(z, 0) * sz + col + (k - 1) * (ptrdiff_t)sy;
      v[k] = (ok && in_x) ? __ldg(a.cur + row) : 0.0f;
      l[k] = (ok && left) ? __ldg(a.cur + row - 1) : 0.0f;
      r[k] = (ok && right) ? __ldg(a.cur + row + 1) : 0.0f;
    }
  };
  auto reduce_plane = [&](const float v[3], const float l[3], const float r[3], BlobPlane &p) {
#pragma unroll
    for (int k = 0; k < 3; k++) {
      const float sl = __shfl_up_sync(full, v[k], 1), sr = __shfl_down_sync(full, v[k], 1);
      const float xl = (lane == 0) ? l[k] : sl, xr = (lane == 31) ? r[k] : sr;
      const float mn = fminf(xl, xr), mx = fmaxf(xl, xr);
      p.rmin[k] = fminf(mn, v[k]);
      p.rmax[k] = fmaxf(mx, v[k]);
      if (k == 1) { p.e = v[k]; p.smin = mn; p.smax = mx; }
    }
    p.pmin = fminf(fminf(p.rmin[0], p.rmin[1]), p.rmin[2]);
    p.pmax = fmaxf(fmaxf(p.rmax[0], p.rmax[1]), p.rmax[2]);
  };

  int n_pending = 0;
  // the voxel of plane iz with the planes below (A), its own (B) and above (C)
  auto test_plane = [&](int iz, const BlobPlane &A, const BlobPlane &B, const BlobPlane &C) {
    const int gz = a.z_offset + iz;
    const bool plane_ok = gz >= 1 && gz < a.nz_global - 1 && iz >= 1 && iz < a.nz - 1;   // uniform
    const float e = B.e;
    const float nmin = fminf(fminf(A.pmin, C.pmin), fminf(fminf(B.rmin[0], B.rmin[2]), B.smin));
    const float nmax = fmaxf(fmaxf(A.pmax, C.pmax), fmaxf(fmaxf(B.rmax[0], B.rmax[2]), B.smax));
    const size_t c = (size_t)iz * sz + col;
    bool unmasked = true;
    if (a.mask && plane_ok) {   // the voxel and its 26 neighbours must all be un-masked (feature.hpp:245-258)
#pragma unroll
      for (int rr = 0; rr < 9; rr++) {
        const size_t row = c + (rr / 3 - 1) * (ptrdiff_t)sz + (rr % 3 - 1) * (ptrdiff_t)sy;
        const bool m = in_x && __ldg(a.mask + row) != 0.0f;
        bool ml = __shfl_up_sync(full, m, 1), mr = __shfl_down_sync(full, m, 1);
        if (left) ml = __ldg(a.mask + row - 1) != 0.0f;
        if (right) mr = __ldg(a.mask + row + 1) != 0.0f;
        unmasked = unmasked && m && ml && mr;
      }
    }
    // minima need score < 0, maxima score > 0 (:270-271, :289-290); strict against every neighbour
    const bool is_min = plane_ok && interior && unmasked && e < 0.0f && e < nmin;
    const bool is_max = plane_ok && interior && unmasked && e > 0.0f && e > nmax;
    const unsigned alive = __ballot_sync(full, is_min || is_max);
    if (!alive) return;
    const int n_new = __popc(alive);
    if (n_pending + n_new > 32) {
      __syncwarp();
      blob_flush(a, q, n_pending, iy);
      n_pending = 0;
      __syncwarp();
    }
    if (is_min || is_max) {
      BlobPending &slot = q[n_pending + __popc(alive & ((1u << lane) - 1u))];
      slot.at = (unsigned long long)c;
      slot.e = e;
      slot.x = ix;
      slot.gz = gz;
      slot.flags = (is_min ? 1 : 0) | (is_max ? 2 : 0);
    }
    n_pending += n_new;
  };

  // three plane slots used in rotation (the loop is unrolled by three so that the roles are compile-time);
  // the raw rows of the plane after next are in flight while a plane is tested
  BlobPlane P0, P1, P2;
  float v[3], l[3], r[3];
  load_plane(z_begin - 1, v, l, r);
  reduce_plane(v, l, r, P0);
  load_plane(z_begin, v, l, r);
  reduce_plane(v, l, r, P1);
  load_plane(z_begin + 1, v, l, r);
  for (int iz = z_begin; iz < z_end; iz += 3) {
    reduce_plane(v, l, r, P2);          // plane iz + 1
    load_plane(iz + 2, v, l, r);
    test_plane(iz, P0, P1, P2);
    if (iz + 1 >= z_end) break;
    reduce_plane(v, l, r, P0);          // plane iz + 2
    load_plane(iz + 3, v, l, r);
    test_plane(iz + 1, P1, P2, P0);
    if (iz + 2 >= z_end) break;
    reduce_plane(v, l, r, P1);          // plane iz + 3
    load_plane(iz + 4, v, l, r);
    test_plane(iz + 2, P2, P0, P1);
  }
  __syncwarp();
  if (n_pending) blob_flush(a, q, n_pending, iy);
}

static void sort_raster(std::vector<BlobCand> &v) {
  std::sort(v.begin(), v.end(), [](const BlobCand &p, const BlobCand &q) {
    if (p.z != q.z) return p.z < q.z;
    if (p.y != q.y) return p.y < q.y;
    return p.x < q.x;
  });
}

// feature.hpp:362-417: the final score filter, once the best scores of the WHOLE image are known
void blob_final_filter(BlobList &minima, BlobList &maxima, float minima_threshold, float maxima_threshold,
                       int use_threshold_ratios, float gmin, float gmax) {
  const float INF = std::numeric_limits<float>::infinity();
  bool filt = (minima_threshold != INF) || (maxima_threshold != -INF);
  bool drop_min = false, drop_max = false;
  if (use_threshold_ratios) {
    // An infinite RATIO admits (almost) nothing in the reference's running filter
    // (+-inf times the running best score); the deterministic reading is an empty list.
    if (maxima_threshold == -INF) drop_max = true;
    if (minima_threshold == INF) drop_min = true;
    if (filt) {
      minima_threshold *= gmin;
      maxima_threshold *= gmax;
    }
  }
  auto keep = [&](BlobList &l, bool drop, bool is_min) {
    BlobList out;
    if (!drop)
      for (size_t i = 0; i < l.score.size(); i++)
        if (!filt || (is_min ? l.score[i] <= minima_threshold : l.score[i] >= maxima_threshold)) {
          out.crds.insert(out.crds.end(), {l.crds[3 * i], l.crds[3 * i + 1], l.crds[3 * i + 2]});
          out.sigma.push_back(l.sigma[i]);
          out.score.push_back(l.score[i]);
        }
    l = std::move(out);
  };
  keep(minima, drop_min, true);
  keep(maxima, drop_max, false);
}

// Slab form: the slab holds image planes [z_offset, z_offset + nz); candidates are produced for the
// slab-local planes [own_z0, own_z1) with z reported as the IMAGE plane.  best[0] / best[1] receive the
// best minimum / maximum score found (1 / -1 if none, feature.hpp:122-123).  finalize = false leaves out
// the final filter, which needs the best scores of the whole image (blob_final_filter).  capacity: rows of each
// device candidate list (0: N / 32, at least 65536); a scale that overflows them is scanned again into larger lists.
void blob_dog_device(visfd_ctx *ctx, i64 nx, i64 ny, i64 nz, i64 z_offset, i64 nz_global, i64 own_z0, i64 own_z1,
                     const float *src, const float *mask,
                     const float *sigmas, int n_sigmas, float delta, float truncate_ratio,
                     float minima_threshold, float maxima_threshold, int use_threshold_ratios,
                     BlobList &minima, BlobList &maxima, bool finalize, float best[2], i64 capacity_rows) {
  VREQUIRE(nx > 0 && ny > 0 && nz > 0, "empty volume");
  VREQUIRE(z_offset >= 0 && z_offset + nz <= nz_global && 0 <= own_z0 && own_z0 <= own_z1 && own_z1 <= nz,
           "slab / receiver planes outside the image");
  VREQUIRE(nx < 2147483647LL / 2 && ny <= 4 * 65535LL && nz <= 65535 && nz_global < 2147483647LL,
           "volume too large for the blob scan launch");
  const i64 N = nx * ny * nz;
  const float INF = std::numeric_limits<float>::infinity();
  Scratch<float> ring[3];
  for (int k = 0; k < 3; k++) ring[k].reset(ctx, N);
  unsigned long long capacity =
      (unsigned long long)(capacity_rows > 0 ? capacity_rows : std::max<i64>(1 << 16, N / 32));
  Scratch<BlobCand> dmins(ctx, capacity), dmaxs(ctx, capacity);
  Scratch<unsigned long long> counters(ctx, 2);

  std::vector<BlobCand> mins, maxs;
  std::vector<float> min_sig, max_sig;
  std::vector<i64> min_rows(n_sigmas, 0), max_rows(n_sigmas, 0);
  float gmin = 1.0f, gmax = -1.0f;  // feature.hpp:122-123 ("impossible" initial values)

  for (int ir = 0; ir < n_sigmas; ir++) {
    float s3[3] = {sigmas[ir], sigmas[ir], sigmas[ir]};
    float sa[3], sb[3], scale;
    int hw[3];
    log_params(s3, delta, truncate_ratio, sa, sb, hw, &scale);
    // an interior slab end needs hw planes for the LoG of the receiver planes' neighbours, + 1 for those
    VREQUIRE((z_offset == 0 || own_z0 >= hw[2] + 1) && (z_offset + nz == nz_global || nz - own_z1 >= hw[2] + 1),
             "slab lacks the halo (LoG half-width + 1 planes) around the receiver planes");
    dog_device(ctx, nx, ny, nz, z_offset, nz_global, src, ring[ir % 3].get(), mask, sa, sb, hw, scale, nullptr, nullptr);
    if (ir < 2 || own_z1 == own_z0) continue;
    // device pre-filter thresholds for this scale
    float min_thr = minima_threshold, max_thr = maxima_threshold;
    if (use_threshold_ratios) {
      // final cut will be ratio * (global best); the best of the previous scales gives a
      // bound that can only be looser (for ratios >= 0)
      min_thr = (gmin < 0.0f && minima_threshold >= 0.0f && minima_threshold != INF) ? minima_threshold * gmin : INF;
      max_thr = (gmax > 0.0f && maxima_threshold >= 0.0f && maxima_threshold != -INF) ? maxima_threshold * gmax : -INF;
      // (<= becomes < on the device: widen by one ulp so that equality survives to the host filter)
      if (min_thr != INF) min_thr = std::nextafter(min_thr, INF);
      if (max_thr != -INF) max_thr = std::nextafter(max_thr, -INF);
    }
    for (int attempt = 0; attempt < 2; attempt++) {
      BlobScanArgs a;
      a.prev = ring[(ir - 2) % 3].get();
      a.cur = ring[(ir - 1) % 3].get();
      a.next = ring[ir % 3].get();
      a.mask = mask;
      a.nx = (int)nx; a.ny = (int)ny; a.nz = (int)nz;
      a.z_offset = (int)z_offset; a.nz_global = (int)nz_global; a.own_z0 = (int)own_z0;
      a.min_thr = min_thr; a.max_thr = max_thr;
      a.mins = dmins.get(); a.maxs = dmaxs.get();
      a.counters = counters.get();
      a.capacity = capacity;
      unsigned long long h[2];
      {
        StageTimer t(ctx, "blob_scan");
        VCK(cudaMemsetAsync(counters.get(), 0, 2 * sizeof(unsigned long long), ctx->stream));
        dim3 grid(div_up(nx, 64), div_up(ny, 4), div_up(own_z1 - own_z0, BLOB_ZC));
        blob_scan_kernel<<<grid, 256, 0, ctx->stream>>>(a, (int)own_z1);
        VCK(cudaGetLastError());
        ctx->count_launch();
      }
      VCK(cudaMemcpyAsync(h, counters.get(), sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
      VCK(cudaStreamSynchronize(ctx->stream));
      if (h[0] > capacity || h[1] > capacity) {
        VREQUIRE(attempt == 0, "blob candidate list overflow");
        capacity = std::max(h[0], h[1]);
        dmins.reset(ctx, capacity);
        dmaxs.reset(ctx, capacity);
        continue;
      }
      std::vector<BlobCand> lm(h[0]), lx(h[1]);
      if (h[0]) VCK(cudaMemcpyAsync(lm.data(), dmins.get(), h[0] * sizeof(BlobCand), cudaMemcpyDeviceToHost, ctx->stream));
      if (h[1]) VCK(cudaMemcpyAsync(lx.data(), dmaxs.get(), h[1] * sizeof(BlobCand), cudaMemcpyDeviceToHost, ctx->stream));
      VCK(cudaStreamSynchronize(ctx->stream));
      sort_raster(lm);
      sort_raster(lx);
      for (auto &c : lm) { mins.push_back(c); min_sig.push_back(sigmas[ir - 1]); gmin = std::min(gmin, c.score); }
      for (auto &c : lx) { maxs.push_back(c); max_sig.push_back(sigmas[ir - 1]); gmax = std::max(gmax, c.score); }
      min_rows[ir - 1] = (i64)lm.size();
      max_rows[ir - 1] = (i64)lx.size();
      break;
    }
  }

  minima = BlobList();
  maxima = BlobList();
  for (size_t i = 0; i < mins.size(); i++) {
    minima.crds.insert(minima.crds.end(), {mins[i].x, mins[i].y, mins[i].z});
    minima.sigma.push_back(min_sig[i]);
    minima.score.push_back(mins[i].score);
  }
  for (size_t i = 0; i < maxs.size(); i++) {
    maxima.crds.insert(maxima.crds.end(), {maxs[i].x, maxs[i].y, maxs[i].z});
    maxima.sigma.push_back(max_sig[i]);
    maxima.score.push_back(maxs[i].score);
  }
  minima.scale_rows = std::move(min_rows);
  maxima.scale_rows = std::move(max_rows);
  if (best) { best[0] = gmin; best[1] = gmax; }
  if (finalize) blob_final_filter(minima, maxima, minima_threshold, maxima_threshold, use_threshold_ratios, gmin, gmax);
}

}  // namespace visfd_cuda
