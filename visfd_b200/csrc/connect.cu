// connect.cu -- LabelConnected (lib/visfd/connect.hpp:171-1432) as HandleTV calls it
// (bin/filter_mrc/handlers.cpp:1927-2034): clustering of the voxels above a saliency threshold
// into surfaces, refusing voxels and voxel pairs whose vote tensors / directions disagree.
//
// The reference is one serial loop: a priority-queue flood from the saliency maxima that, for
// every voxel it pops, computes a finite-difference Hessian of the saliency, diagonalises it,
// compares it with the voxel's vote tensor and direction, and then tests each of the six
// neighbours' tensors and directions against the voxel's own.  All of that arithmetic depends
// only on the voxel and its neighbours, not on the flood.  So:
//
//   device (connect_predicates_kernel, one thread per voxel, everything in one pass)
//     * the voxel's admissibility (saliency >= threshold, mask) and, for admissible voxels, the
//       two "saliency vs tensor / vector" tests of connect.hpp:462-578 -- 19-point Hessian of the
//       saliency, its principal eigenvector (double closed form, eigen3.cuh), trace products;
//     * the six DIRECTED neighbour tests of connect.hpp:609-676 (bounds, mask, tensor, vector);
//     * the local-extremum flags _FindExtrema needs (morphology_implementation.hpp:57-515):
//       "no neighbour is greater", "some neighbour is equal" (plateaus);
//     packed into 16 bits per voxel.
//   host (flood_host)
//     * seeds from the flags (plateaus resolved by a breadth-first search over equal voxels),
//       sorted as the reference sorts its maxima;
//     * the flood itself, in the reference's pop order, reading only the 16-bit flags: the basin
//       a voxel lands in, the polarity (sign) bookkeeping of the standardised directions and the
//       order of the cluster merges depend on that order, so it is kept; what is left of it is
//       integer work on the admissible voxels;
//     * cluster renumbering by size, direction standardisation (connect.hpp:1060-1300).
//
// Reference quirks reproduced on purpose: TraceProductSym3 / FrobeniusNormSym3 index the wrong
// lookup table (lin3_utils.hpp:516-528 uses MapIndices_linear_to_3x3 where MapIndices_3x3_to_linear
// is meant) and so only combine DIAGONAL entries, in a particular order with repeats -- the
// compiled reference computes a0b0+a0b1+a1b2+a1b0+a1b1+a2b2+a2b1+a2b2+a0b0, checked against
// the reference build; the neighbour vector test sits inside `if (aaaafSymmetricTensor)`
// (connect.hpp:648); the basin number travels through a float (connect.hpp:438); voxels outside the
// mask keep the internal marker n_maxima + 1 (connect.hpp:1398-1401 skips them).
// Not offered: must-link constraints (connect.hpp:830-1040), sorting by value, voxel weights.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <queue>

#include "common.cuh"
#include "kernels.cuh"
#include "eigen3.cuh"
#include "stencil.cuh"

namespace visfd_cuda {

enum : uint16_t {
  CS_CAND = 1,        // inside the mask and not below the saliency threshold
  CS_PASS = 2,        // survives the saliency-vs-tensor and saliency-vs-vector tests
  CS_EDGE0 = 4,       // bits 2..7: neighbour k is inside the image and the mask and compatible (directed test)
  CS_GE = 1 << 8,     // no neighbour (inside image and mask) has a greater saliency
  CS_EQ = 1 << 9,     // some neighbour has an equal saliency (plateau)
  CS_MASK = 1 << 10,  // inside the mask
};

// connect.hpp:212-240 with connectivity 1: jz, jy, jx loops
__constant__ int c_nbr[6][3] = {{0, 0, -1}, {0, -1, 0}, {-1, 0, 0}, {1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
static const int h_nbr[6][3] = {{0, 0, -1}, {0, -1, 0}, {-1, 0, 0}, {1, 0, 0}, {0, 1, 0}, {0, 0, 1}};

// The arrays hold nz planes starting at global plane z_offset of a volume of nz_global planes: the stencil clamp and
// the neighbour bounds are those of the whole volume, so a slab computes the flags of the undivided image.
struct ConnArgs {
  const float *sal, *mask, *tensor, *dir;
  int nx, ny, nz, z_offset, nz_global;
  float thr_sal, thr_vs, thr_vn, thr_ts, thr_tn;
  int order, signed_dot;
  uint16_t *state;
};

// TraceProductSym3 as the reference build evaluates it (see the header): diagonal entries only.
__device__ __forceinline__ float trace_product_ref(const float a[3], const float b[3]) {
  float s = __fmul_rn(a[0], b[0]);
  s = __fadd_rn(s, __fmul_rn(a[0], b[1]));
  s = __fadd_rn(s, __fmul_rn(a[1], b[2]));
  s = __fadd_rn(s, __fmul_rn(a[1], b[0]));
  s = __fadd_rn(s, __fmul_rn(a[1], b[1]));
  s = __fadd_rn(s, __fmul_rn(a[2], b[2]));
  s = __fadd_rn(s, __fmul_rn(a[2], b[1]));
  s = __fadd_rn(s, __fmul_rn(a[2], b[2]));
  s = __fadd_rn(s, __fmul_rn(a[0], b[0]));
  return s;
}
__device__ __forceinline__ float dot3_ref(const float a[3], const float b[3]) {  // lin3_utils.hpp:60-62
  return __fadd_rn(__fadd_rn(__fmul_rn(a[0], b[0]), __fmul_rn(a[1], b[1])), __fmul_rn(a[2], b[2]));
}

// a is compatible with b?  (connect.hpp:648-676; `ta`, `tb`: diagonal tensor entries or NULL)
__device__ __forceinline__ bool pair_ok(const ConnArgs &g, const float *ta, const float *tb, const float va[3],
                                        const float vb[3]) {
  if (!ta) return true;
  {
    const float tp = trace_product_ref(ta, tb);
    const float fa = sqrtf(trace_product_ref(ta, ta)), fb = sqrtf(trace_product_ref(tb, tb));
    if (tp < __fmul_rn(__fmul_rn(g.thr_tn, fa), fb)) return false;
  }
  const float d = dot3_ref(va, vb);
  if (g.signed_dot) {
    // (sic) the signed branch compares with the TENSOR threshold, connect.hpp:654
    const float la = sqrtf(dot3_ref(va, va)), lb = sqrtf(dot3_ref(vb, vb));
    if (d < __fmul_rn(__fmul_rn(g.thr_tn, la), lb)) return false;
  } else {
    const float lhs = __fmul_rn(d, d);
    const float rhs = __fmul_rn(__fmul_rn(__fmul_rn(g.thr_vn, g.thr_vn), dot3_ref(va, va)), dot3_ref(vb, vb));
    if (lhs < rhs) return false;
  }
  return true;
}

__global__ void __launch_bounds__(256) connect_predicates_kernel(ConnArgs g, int z0) {
  const int ix = blockIdx.x * blockDim.x + threadIdx.x;
  const int iy = blockIdx.y * blockDim.y + threadIdx.y;
  const int iz = z0 + blockIdx.z;
  if (ix >= g.nx || iy >= g.ny) return;
  const i64 sy = g.nx, sz = (i64)g.nx * g.ny;
  const i64 i = iz * sz + iy * sy + ix;
  uint16_t st = 0;
  if (g.mask && __ldg(g.mask + i) == 0.0f) {
    g.state[i] = 0;
    return;
  }
  st |= CS_MASK;
  const float s = __ldg(g.sal + i);
  const bool cand = !(s < g.thr_sal);   // connect.hpp:445-449 (a NaN is not rejected there either)
  float t_own[3] = {0.f, 0.f, 0.f}, v_own[3] = {0.f, 0.f, 0.f};
  if (cand) {
    st |= CS_CAND;
    if (g.tensor) {
      t_own[0] = __ldg(g.tensor + 6 * i); t_own[1] = __ldg(g.tensor + 6 * i + 1); t_own[2] = __ldg(g.tensor + 6 * i + 2);
    }
    if (g.dir) {
      v_own[0] = __ldg(g.dir + 3 * i); v_own[1] = __ldg(g.dir + 3 * i + 1); v_own[2] = __ldg(g.dir + 3 * i + 2);
    }
    // ---- saliency vs tensor / vector at this voxel (connect.hpp:462-578) ----
    bool discard = false;
    if (g.tensor || g.dir) {
      Stencil sten = make_stencil(g.sal, g.nx, g.ny, g.z_offset, g.nz_global, ix, iy, iz);
      float h[6];
      fd_hessian(sten, 1.0f, h);
      // tensor positive definite near the target and clusters start at maxima: the Hessian changes sign (:487-492)
#pragma unroll
      for (int k = 0; k < 6; k++) h[k] = -h[k];
      if (g.tensor) {
        const float tp = trace_product_ref(h, t_own);
        const float fs = sqrtf(trace_product_ref(h, h)), ft = sqrtf(trace_product_ref(t_own, t_own));
        if (tp < __fmul_rn(__fmul_rn(g.thr_ts, fs), ft)) discard = true;
      }
      if (g.dir) {
        Sym3d m = {h[0], h[1], h[2], h[3], h[4], h[5]};
        double ev[3], e0d[3];
        sym3_eigen_first(m, g.order, ev, e0d);
        const float e0[3] = {(float)e0d[0], (float)e0d[1], (float)e0d[2]};
        const float d = dot3_ref(e0, v_own);
        if (g.signed_dot) {
          if (d < __fmul_rn(__fmul_rn(g.thr_vs, sqrtf(dot3_ref(e0, e0))), sqrtf(dot3_ref(v_own, v_own)))) discard = true;
        } else {
          const float rhs = __fmul_rn(__fmul_rn(__fmul_rn(g.thr_vs, g.thr_vs), dot3_ref(e0, e0)), dot3_ref(v_own, v_own));
          if (__fmul_rn(d, d) < rhs) discard = true;
        }
      }
    }
    if (!discard) st |= CS_PASS;
  }
  // ---- neighbours: extremum flags for every voxel, directed compatibility for admissible ones ----
  bool ge = true, eq = false;
#pragma unroll
  for (int k = 0; k < 6; k++) {
    const int jx = ix + c_nbr[k][0], jy = iy + c_nbr[k][1], jz = iz + c_nbr[k][2];
    if (jx < 0 || jx >= g.nx || jy < 0 || jy >= g.ny || jz + g.z_offset < 0 || jz + g.z_offset >= g.nz_global) continue;
    const i64 j = jz * sz + jy * sy + jx;
    if (g.mask && __ldg(g.mask + j) == 0.0f) continue;
    const float sj = __ldg(g.sal + j);
    if (sj > s) ge = false;
    else if (sj == s) eq = true;
    if (st & CS_PASS) {
      bool ok = true;
      if (g.tensor) {
        const float tj[3] = {__ldg(g.tensor + 6 * j), __ldg(g.tensor + 6 * j + 1), __ldg(g.tensor + 6 * j + 2)};
        const float vj[3] = {__ldg(g.dir + 3 * j), __ldg(g.dir + 3 * j + 1), __ldg(g.dir + 3 * j + 2)};
        ok = pair_ok(g, t_own, tj, v_own, vj);
      }
      if (ok) st |= (uint16_t)(CS_EDGE0 << k);
    }
  }
  if (ge) st |= CS_GE;
  if (eq) st |= CS_EQ;
  g.state[i] = st;
}

void connect_predicates_device(visfd_ctx *ctx, i64 nx, i64 ny, i64 nz_local, i64 z_offset, i64 nz_global, i64 z0,
                               i64 z1, const float *sal, const float *mask, const float *tensor, const float *dir,
                               int eival_order, int signed_dot, float thr_sal, float thr_vs, float thr_vn, float thr_ts,
                               float thr_tn, uint16_t *state) {
  VREQUIRE(nx >= 3 && ny >= 3 && nz_global >= 3, "LabelConnected needs an image at least 3 voxels wide (finite-difference Hessian)");
  VREQUIRE(!tensor || dir, "tensors without directions");
  // the clamped stencil and the neighbours of planes [z0, z1) must lie in the slab
  const i64 lo = std::max<i64>(0, std::min(z_offset + z0 - 1, nz_global - 3));
  const i64 hi = std::min(nz_global, std::max<i64>(z_offset + z1 + 1, 3));
  VREQUIRE(0 <= z0 && z0 <= z1 && z1 <= nz_local && z_offset >= 0 && z_offset + nz_local <= nz_global &&
               (z1 == z0 || (lo >= z_offset && hi <= z_offset + nz_local)),
           "connect: the slab lacks the planes next to the planes it computes");
  ConnArgs g{sal, mask, tensor, dir, (int)nx, (int)ny, (int)nz_local, (int)z_offset, (int)nz_global, thr_sal, thr_vs,
             thr_vn, thr_ts, thr_tn, eival_order, signed_dot, state};
  StageTimer t(ctx, "connect_predicates");
  dim3 block(64, 4, 1);
  for (i64 zc = z0; zc < z1; zc += 65535) {
    dim3 grid(div_up(nx, 64), div_up(ny, 4), (unsigned)std::min<i64>(65535, z1 - zc));
    connect_predicates_kernel<<<grid, block, 0, ctx->stream>>>(g, (int)zc);
    VCK(cudaGetLastError());
    ctx->count_launch();
  }
}

void first_eigenvectors_device(visfd_ctx *ctx, i64 n, const float *tensor, const float *mask, int eival_order,
                               float *dir) {
  // handlers.cpp:1933-1950: the first eigenvector of every vote tensor (masked voxels: left as they are -> zero here)
  VCK(cudaMemsetAsync(dir, 0, 3 * (size_t)n * sizeof(float), ctx->stream));
  tensor_score_device(ctx, n, tensor, mask, eival_order, 0, 1, nullptr, nullptr, dir);
}

// ---------------------------------------------------------------------------------------------------
// host: seeds + ordered flood over the 16-bit flags
// ---------------------------------------------------------------------------------------------------
namespace {

struct QEntry {
  float sal;
  i64 basin;
  int x, y, z;
};
// std::less on tuple<Scalar, ptrdiff_t, array<Coordinate,3>> (connect.hpp:307-315): a max-heap
struct QLess {
  bool operator()(const QEntry &a, const QEntry &b) const {
    if (a.sal < b.sal) return true;
    if (b.sal < a.sal) return false;
    if (a.basin != b.basin) return a.basin < b.basin;
    if (a.x != b.x) return a.x < b.x;
    if (a.y != b.y) return a.y < b.y;
    return a.z < b.z;
  }
};

struct Seed {
  float score;
  i64 voxel;   // raster index of the plateau's first voxel
};

}  // namespace

// Returns the number of clusters.  labels: N int64 (host).  dir: N*3 floats (host) or NULL; sign-standardised in place
// when unsigned_dot (aaaafVectorStandardized aliases aaaafVector in HandleTV, handlers.cpp:1985).
i64 connect_flood_host(i64 nx, i64 ny, i64 nz, const float *sal, const uint16_t *state, float *dir, bool unsigned_dot,
                       float thr_sal, i64 *labels, std::vector<float> *cluster_maxima, i64 *n_maxima_out) {
  const i64 sy = nx, sz = nx * ny, N = nx * ny * nz;
  // ---- _FindExtrema: maxima (plateaus allowed, borders allowed), morphology_implementation.hpp:57-515 ----
  // maxima_threshold = threshold (or -inf when the caller passed +inf, :549-550)
  const float max_thr = (thr_sal == INFINITY) ? -INFINITY : thr_sal;
  std::vector<Seed> seeds;
  {
    std::vector<bool> seen;   // plateau members already visited (allocated on first need)
    std::vector<i64> q;
    for (i64 i = 0; i < N; i++) {
      const uint16_t st = state[i];
      if (!(st & CS_MASK)) continue;
      if (!(st & CS_EQ)) {
        if ((st & CS_GE) && sal[i] >= max_thr) seeds.push_back({sal[i], i});
        continue;
      }
      if (!(sal[i] >= max_thr)) continue;   // a plateau below the threshold cannot be recorded
      if (seen.empty()) seen.assign((size_t)N, false);
      if (seen[(size_t)i]) continue;
      // breadth-first search over the equal-valued neighbours: a maximum iff every member has CS_GE
      bool is_max = true;
      q.clear();
      q.push_back(i);
      seen[(size_t)i] = true;
      for (size_t h = 0; h < q.size(); h++) {
        const i64 v = q[h];
        if (!(state[v] & CS_GE)) is_max = false;
        const int x = (int)(v % nx), y = (int)((v / nx) % ny), z = (int)(v / sz);
        for (int k = 0; k < 6; k++) {
          const int jx = x + h_nbr[k][0], jy = y + h_nbr[k][1], jz = z + h_nbr[k][2];
          if (jx < 0 || jx >= nx || jy < 0 || jy >= ny || jz < 0 || jz >= nz) continue;
          const i64 j = jz * sz + jy * sy + jx;
          if (!(state[j] & CS_MASK) || seen[(size_t)j] || !(sal[j] == sal[v])) continue;
          seen[(size_t)j] = true;
          q.push_back(j);
        }
      }
      if (is_max) seeds.push_back({sal[i], i});
    }
  }
  // sort(rbegin, rend) on (score, position in the list): decreasing score, ties by decreasing position (:449-470)
  {
    std::vector<std::pair<float, i64> > key(seeds.size());
    for (size_t k = 0; k < seeds.size(); k++) key[k] = {seeds[k].score, (i64)k};
    std::sort(key.rbegin(), key.rend());
    std::vector<Seed> sorted(seeds.size());
    for (size_t k = 0; k < seeds.size(); k++) sorted[k] = seeds[(size_t)key[k].second];
    seeds.swap(sorted);
  }
  const i64 n_basins = (i64)seeds.size();
  if (n_maxima_out) *n_maxima_out = n_basins;
  const i64 UNDEFINED = n_basins + 1, QUEUED = n_basins + 2;   // connect.hpp:288-289
  std::fill(labels, labels + N, UNDEFINED);

  std::priority_queue<QEntry, std::vector<QEntry>, QLess> pq;
  for (i64 b = 0; b < n_basins; b++) {
    const i64 v = seeds[(size_t)b].voxel;
    pq.push({seeds[(size_t)b].score, b, (int)(v % nx), (int)((v / nx) % ny), (int)(v / sz)});
    labels[v] = QUEUED;
  }
  std::vector<i64> basin2cluster((size_t)n_basins);
  std::vector<std::vector<i64> > cluster2basins((size_t)n_basins);
  for (i64 b = 0; b < n_basins; b++) {
    basin2cluster[(size_t)b] = b;
    cluster2basins[(size_t)b].push_back(b);
  }
  std::vector<signed char> polarity((size_t)n_basins, 1);
  const bool standardise = dir != nullptr && unsigned_dot;
  std::vector<i64> accepted;   // voxels that joined a basin, in pop order

  while (!pq.empty()) {
    const QEntry e = pq.top();
    pq.pop();
    const i64 basin = (i64)(float)e.basin;   // (sic) the basin number passes through a Scalar, connect.hpp:438
    const i64 i = e.z * sz + e.y * sy + e.x;
    const uint16_t st = state[i];
    if (!(st & CS_CAND)) {   // below the threshold or outside the mask, :445-456
      labels[i] = UNDEFINED;
      continue;
    }
    if (!(st & CS_PASS)) {   // :580-591
      labels[i] = UNDEFINED;
      if (basin >= 0 && basin < n_basins && seeds[(size_t)basin].voxel == i) basin2cluster[(size_t)basin] = -1;
      continue;
    }
    labels[i] = basin;
    accepted.push_back(i);
    for (int k = 0; k < 6; k++) {
      if (!(st & (CS_EDGE0 << k))) continue;
      const int jx = e.x + h_nbr[k][0], jy = e.y + h_nbr[k][1], jz = e.z + h_nbr[k][2];
      const i64 j = jz * sz + jy * sy + jx;
      const i64 lj = labels[j];
      if (lj == QUEUED) continue;
      if (lj == UNDEFINED) {
        labels[j] = QUEUED;
        pq.push({sal[j], basin, jx, jy, jz});
        if (standardise) {   // :698-722
          float *a = dir + 3 * i, *b = dir + 3 * j;
          if (a[0] * b[0] + a[1] * b[1] + a[2] * b[2] < 0.0f) { b[0] *= -1.0f; b[1] *= -1.0f; b[2] *= -1.0f; }
        }
        continue;
      }
      // the neighbour already belongs to a basin: merge the two clusters (:727-803)
      const i64 bi = basin, bj = lj;
      const i64 ci = basin2cluster[(size_t)bi], cj = basin2cluster[(size_t)bj];
      bool polarity_match = true;
      if (standardise) {
        const float *a = dir + 3 * i, *b = dir + 3 * j;
        if ((a[0] * b[0] + a[1] * b[1] + a[2] * b[2]) * polarity[(size_t)bi] * polarity[(size_t)bj] < 0.0f)
          polarity_match = false;
      }
      if (ci == cj) continue;
      const i64 keep = std::min(ci, cj), gone = std::max(ci, cj);
      for (i64 b : cluster2basins[(size_t)gone]) {
        cluster2basins[(size_t)keep].push_back(b);
        basin2cluster[(size_t)b] = keep;
        if (standardise && !polarity_match) polarity[(size_t)b] = (signed char)-polarity[(size_t)b];
      }
      cluster2basins[(size_t)gone].clear();
      cluster2basins[(size_t)gone].shrink_to_fit();
    }
  }
  cluster2basins.clear();

  // ---- clusters: count, renumber (:1045-1068) ----
  i64 n_clusters = 0;
  std::vector<i64> old2new((size_t)n_basins), deepest;
  for (i64 b = 0; b < n_basins; b++) {
    old2new[(size_t)b] = n_clusters;
    if (basin2cluster[(size_t)b] == b) {
      deepest.push_back(b);
      n_clusters++;
    }
  }
  for (i64 b = 0; b < n_basins; b++)
    if (basin2cluster[(size_t)b] >= 0) basin2cluster[(size_t)b] = old2new[(size_t)basin2cluster[(size_t)b]];

  std::sort(accepted.begin(), accepted.end());   // raster order, as the reference's image loops
  if (standardise)
    for (i64 v : accepted) {   // :1080-1105
      const float p = (float)polarity[(size_t)labels[v]];
      dir[3 * v] *= p; dir[3 * v + 1] *= p; dir[3 * v + 2] *= p;
    }
  std::vector<long double> size((size_t)n_clusters, 0.0L);
  for (i64 v : accepted) {
    labels[v] = basin2cluster[(size_t)labels[v]];
    size[(size_t)labels[v]] += 1.0L;
  }
  if (standardise && n_clusters > 0) {   // outward normals: centre of mass test, :1183-1284
    std::vector<long double> com((size_t)n_clusters * 3, 0.0L), sum((size_t)n_clusters, 0.0L);
    for (i64 v : accepted) {
      const size_t c = (size_t)labels[v];
      com[3 * c] += (long double)(v % nx);
      com[3 * c + 1] += (long double)((v / nx) % ny);
      com[3 * c + 2] += (long double)(v / sz);
    }
    for (size_t c = 0; c < (size_t)n_clusters; c++)
      for (int d = 0; d < 3; d++) com[3 * c + d] /= size[c];
    for (i64 v : accepted) {
      const size_t c = (size_t)labels[v];
      const float r[3] = {(float)((long double)(v % nx) - com[3 * c]), (float)((long double)((v / nx) % ny) - com[3 * c + 1]),
                          (float)((long double)(v / sz) - com[3 * c + 2])};
      const float *n = dir + 3 * v;
      sum[c] += (long double)(r[0] * n[0] + r[1] * n[1] + r[2] * n[2]);
    }
    for (i64 v : accepted)
      if (sum[(size_t)labels[v]] < 0.0L) { dir[3 * v] *= -1.0f; dir[3 * v + 1] *= -1.0f; dir[3 * v + 2] *= -1.0f; }
  }
  // ---- order by size: sort(rbegin, rend) on (float size, cluster) (:1310-1355) ----
  std::vector<i64> rank_of((size_t)n_clusters);
  {
    std::vector<std::pair<float, i64> > key((size_t)n_clusters);
    for (i64 c = 0; c < n_clusters; c++) key[(size_t)c] = {(float)size[(size_t)c], c};
    std::sort(key.rbegin(), key.rend());
    for (i64 r = 0; r < n_clusters; r++) rank_of[(size_t)key[(size_t)r].second] = r;
    if (cluster_maxima) {
      cluster_maxima->resize((size_t)n_clusters * 3);
      for (i64 r = 0; r < n_clusters; r++) {
        const i64 v = seeds[(size_t)deepest[(size_t)key[(size_t)r].second]].voxel;
        (*cluster_maxima)[3 * r] = (float)(v % nx);
        (*cluster_maxima)[3 * r + 1] = (float)((v / nx) % ny);
        (*cluster_maxima)[3 * r + 2] = (float)(v / sz);
      }
    }
  }
  for (i64 v : accepted) labels[v] = rank_of[(size_t)labels[v]] + 1;   // cluster numbers start at 1 (:1418)
  // everything else inside the mask that is still UNDEFINED (or was queued and thrown out) becomes -1 (:1403-1406)
  for (i64 i = 0; i < N; i++)
    if ((state[i] & CS_MASK) && labels[i] == UNDEFINED) labels[i] = -1;
  return n_clusters;
}

}  // namespace visfd_cuda

using namespace visfd_cuda;

extern "C" int visfd_cuda_label_connected(visfd_ctx *ctx, int64_t nx, int64_t ny, int64_t nz, const float *saliency,
                                          const float *mask, const float *tensor, float *direction,
                                          int direction_from_tensor, int eival_order, int consider_dot_product_sign,
                                          float threshold_saliency, float threshold_vector_saliency,
                                          float threshold_vector_neighbor, float threshold_tensor_saliency,
                                          float threshold_tensor_neighbor, int64_t *labels, int64_t *n_clusters,
                                          float *cluster_maxima, int64_t maxima_capacity, int64_t *n_maxima) {
  try {
    VREQUIRE(ctx != nullptr, "context is NULL");
    VCK(cudaSetDevice(ctx->device));
    drop_pending_stage_events(ctx);
    VREQUIRE(nx > 0 && ny > 0 && nz > 0 && nx < (1LL << 31) && ny < (1LL << 31) && nz < (1LL << 31), "bad image dimensions");
    VREQUIRE(saliency && labels, "NULL argument");
    VREQUIRE(!(direction_from_tensor && !tensor), "direction_from_tensor without a tensor");
    const size_t N = (size_t)nx * ny * nz;
    const bool host = !is_device_pointer(saliency);
    const bool have_dir = direction != nullptr || tensor != nullptr;
    // connect.hpp:190-205: with unsigned dot products a negative vector threshold means "do not test"
    if (!consider_dot_product_sign) {
      if (threshold_vector_saliency < 0) threshold_vector_saliency = 0.0f;
      if (threshold_vector_neighbor < 0) threshold_vector_neighbor = 0.0f;
    }
    Staged<float> s(ctx, saliency, N, Dir::In, host), m(ctx, mask, N, Dir::In, host), t(ctx, tensor, 6 * N, Dir::In, host);
    const bool compute_dir = tensor && (direction_from_tensor || !direction);
    Scratch<float> dir_tmp;
    Staged<float> d;
    float *dir_dev = nullptr;
    if (direction) {
      d.init(ctx, direction, 3 * N, compute_dir ? Dir::Out : Dir::In, host);
      dir_dev = d.get();
    } else if (have_dir) {
      dir_tmp.reset(ctx, 3 * N);
      dir_dev = dir_tmp.get();
    }
    if (compute_dir) first_eigenvectors_device(ctx, (i64)N, t.get(), m.get(), eival_order, dir_dev);
    Scratch<uint16_t> state(ctx, N);
    // the Hessian of the saliency is diagonalised with DECREASING eigenvalues (clusters start at maxima, connect.hpp:173-177)
    connect_predicates_device(ctx, nx, ny, nz, 0, nz, 0, nz, s.get(), m.get(), t.get(), dir_dev, 1, consider_dot_product_sign != 0,
                              threshold_saliency, threshold_vector_saliency, threshold_vector_neighbor,
                              threshold_tensor_saliency, threshold_tensor_neighbor, state.get());
    // ---- to the host: flags, saliency (if it was on the device), directions (if they are wanted back) ----
    std::vector<uint16_t> h_state(N);
    VCK(cudaMemcpyAsync(h_state.data(), state.get(), N * sizeof(uint16_t), cudaMemcpyDeviceToHost, ctx->stream));
    std::vector<float> h_sal_buf, h_dir_buf;
    const float *h_sal = saliency;
    if (!host) {
      h_sal_buf.resize(N);
      VCK(cudaMemcpyAsync(h_sal_buf.data(), saliency, N * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
      h_sal = h_sal_buf.data();
    }
    float *h_dir = nullptr;
    if (direction) {
      if (host) {
        if (compute_dir) VCK(cudaMemcpyAsync(direction, dir_dev, 3 * N * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
        h_dir = direction;
      } else {
        h_dir_buf.resize(3 * N);
        VCK(cudaMemcpyAsync(h_dir_buf.data(), dir_dev, 3 * N * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
        h_dir = h_dir_buf.data();
      }
      d.delivered = true;
    }
    VCK(cudaStreamSynchronize(ctx->stream));
    std::vector<int64_t> h_lab_buf;
    int64_t *h_lab = labels;
    if (is_device_pointer(labels)) {
      h_lab_buf.resize(N);
      h_lab = h_lab_buf.data();
    }
    std::vector<float> maxima;
    i64 n_max = 0;
    const auto t0 = std::chrono::steady_clock::now();
    const i64 nc = connect_flood_host(nx, ny, nz, h_sal, h_state.data(), h_dir, consider_dot_product_sign == 0,
                                      threshold_saliency, h_lab, &maxima, &n_max);
    const double flood_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (h_lab != labels) VCK(cudaMemcpyAsync(labels, h_lab, N * sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream));
    if (direction && !host)
      VCK(cudaMemcpyAsync(direction, h_dir, 3 * N * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    if (n_clusters) *n_clusters = nc;
    if (n_maxima) *n_maxima = n_max;
    if (cluster_maxima && maxima_capacity > 0)
      memcpy(cluster_maxima, maxima.data(), sizeof(float) * 3 * (size_t)std::min<i64>(nc, maxima_capacity));
    VCK(cudaStreamSynchronize(ctx->stream));
    resolve_stage_times(ctx);
    ctx->stage_ms["flood"] += flood_ms;   // host time of the ordered flood
    return 0;
  } catch (const std::exception &ex) {
    set_last_error(ex.what());
    if (ctx) { cudaStreamSynchronize(ctx->stream); cudaGetLastError(); }
    return 1;
  }
}
