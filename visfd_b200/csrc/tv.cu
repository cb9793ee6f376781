// tv.cu -- TV3D dense stick voting (lib/visfd/feature.hpp:1712-2037, receiver loop
// TVReceiveStickVotes :2218-2384) as a sparse-voter / dense-receiver gather.
//
// The reference visits all (2hw+1)^3 offsets of every receiver and skips the ~95 % of
// them whose voter has zero saliency.  Here the voters (saliency != 0 after the cut,
// mask != 0) are first compacted into a list ordered by 4x4x4 BRICK (count -> exclusive
// scan -> fill -> direction: two row-streaming passes over the saliency volume, a warp per
// run of 8 bricks, and one thread per voter for its normal), 48 B per voter, laid out as the
// voting kernels consume them (struct VoterRec).  The gather runs one WARP per 4x4x4 receiver patch (lane = (x, y, half);
// four z-receivers per lane; the two half-warps take different voters): it builds the table of
// brick rows that can reach the patch, streams their voters through an exact voter-to-patch
// distance test into a warp-private cp.async ring in shared memory, and drains the ring 32
// voters at a time.  Two kernels share that code:
//   * tv_gather_kernel     -- 4 warps per CTA (one 8x8x4 tile), radial decay by MUFU.EX2 / MUFU.RCP;
//                             every exponent, curves, non-positive weights, mixed support shells.
//   * tv_gather_lut_kernel -- persistent, one 16-warp CTA per SM; exp(-r^2/2 sigma^2) (zero outside
//                             the support) and -1/r^2 come from a shared-memory table indexed by
//                             the INTEGER r^2 (positions are lattice points), 16 replicas so that
//                             the lanes of a half-warp never share a bank.  Exponent 4, positive
//                             weights, vote radius <= 24: the filter_mrc default and BASELINE's
//                             configurations.  No MUFU, no support mask, no address arithmetic in
//                             the loop: the r^2 accumulator is a DENORMAL float whose bit pattern is
//                             the shared-memory address of the table row (see LUT_* below).
// The reference's decay TABLE (lib/visfd/filter3d.hpp:546-601) is only needed for two things,
// both computed on the host with the reference's own float expressions: the normalisation
// constant (sum over the cube) and which lattice points on the shell r^2 == hw^2 survive the
// truncation threshold.
//
// Epilogue (fused, accumulators still in registers): optional store of the 6-component
// tensor (-save-progress) and DiagonalizeFlatSym3 + ScoreTensorPlanar/Linear
// (bin/filter_mrc/handlers.cpp:1870-1892), eigenvalues in double (eigen3.cuh: sym3_eigenvalues_newton).
#include <cstdlib>

#include "common.cuh"
#include "kernels.cuh"
#include "eigen3.cuh"
#include <cmath>
#include <algorithm>

namespace visfd_cuda {

constexpr int BR = 8;            // edge of a receiver tile and of the regions the list kernels work on
constexpr int VSH = 2;           // voters are ordered by bricks of edge 1 << VSH = 4: a receiver patch tests
constexpr int VBR = 1 << VSH;    // the voters of the bricks that touch its reach, and 4^3 bricks hug a
                                 // radius-20 sphere better than 8^3 ones (72 % instead of 53 % accepted)
// Warps never synchronise with each other; four per CTA cover one 8x8x4 receiver tile and share its
// candidates in L1.  Measured on the 256^3 run: 1 warp per CTA 32.0 ms, 2: 29.6, 4: 29.5, 8: 30.6
// (fewer: less sharing; more: registers and shared memory wait for the slowest of eight patches).
constexpr int TV_WARPS = 4;
constexpr int TV_THREADS = 32 * TV_WARPS;
constexpr int TV_MIN_CTAS = 16 / TV_WARPS;
constexpr int TV_TILE_Z = 4;      // receiver planes per CTA
constexpr int TV_MAX_REACH = 7;  // bricks; hw <= 56
constexpr int TV_MAX_SHELL = 512;

int tv_halfwidth(float sigma, float cutoff_ratio) {
  return (int)floor(sigma * cutoff_ratio);  // feature.hpp:1669-1675
}

// ---------------------------------------------------------------------------------
// host: what we need from the reference's decay table
// ---------------------------------------------------------------------------------
struct DecayInfo {
  float total;                      // sum of the un-normalised table (float, raster order)
  int shell_total = 0, shell_kept = 0;  // lattice points with r^2 == hw^2: all / surviving the truncation
  std::vector<uint32_t> shell_keep; // packed |dx| | |dy|<<8 | |dz|<<16 of surviving shell points
};

// GenFilterGenGauss3D(sigma, m=2, hw): lib/visfd/filter3d.hpp:546-601
static DecayInfo decay_info(float sigma, int hw) {
  DecayInfo info;
  float thr = 1.0f;
  {
    float h = (sigma > 0) ? expf(-powf(hw / sigma, 2.0f)) : 1.0f;
    if (h < thr) thr = h;
  }
  float total = 0;
  const int hw2 = hw * hw;
  for (int iz = -hw; iz <= hw; iz++)
    for (int iy = -hw; iy <= hw; iy++)
      for (int ix = -hw; ix <= hw; ix++) {
        float x = (!((sigma == 0.0f) && (ix == 0))) ? ix / sigma : 0.0f;
        float y = (!((sigma == 0.0f) && (iy == 0))) ? iy / sigma : 0.0f;
        float z = (!((sigma == 0.0f) && (iz == 0))) ? iz / sigma : 0.0f;
        float r = sqrtf(x * x + y * y + z * z);
        float h = (r > 0) ? expf(-powf(r, 2.0f)) : 1.0f;
        if (fabsf(h) < thr) h = 0.0f;
        total += h;
        int r2 = ix * ix + iy * iy + iz * iz;
        if (r2 == hw2) {
          info.shell_total++;
          if (h != 0.0f) info.shell_kept++;
        }
        if (r2 == hw2 && h != 0.0f && ix >= 0 && iy >= 0 && iz >= 0)
          info.shell_keep.push_back((uint32_t)ix | ((uint32_t)iy << 8) | ((uint32_t)iz << 16));
        // Lattice points strictly inside (outside) the shell are kept (dropped) by a
        // margin of exp(1/sigma^2) - 1 >> float epsilon, so r^2 < hw^2 decides them.
      }
  info.total = total;
  return info;
}

// ---------------------------------------------------------------------------------
// voter list construction
// ---------------------------------------------------------------------------------
struct VoterSrc {
  const float *sal;
  const float *mask_src;
  float thr;
  int nx, ny;
  i64 nz;  // slab planes
  int vbx, vby, vbz;     // 4^3 voter bricks: the order of the list, the index of counts[] / off[]
};

// The list kernels stream the saliency (and mask) volume by ROWS: a warp owns 8 consecutive bricks of one brick
// row -- 32 columns x 4 rows x 4 planes -- and issues its sixteen 128-byte row loads back to back before it
// looks at any of them (16 independent, fully coalesced loads per lane in flight; the round-1 kernels walked
// 8^3 regions with 32-byte row pieces and reached 1.2 TB/s).  Lane = x column; the nibble of a ballot that
// belongs to a brick gives its voters of that row, so counts and ranks in (z, y, x) order are popcounts.
constexpr int VL_WARPS = 8;                 // warps per CTA, side by side along x: 1 KB of every row
constexpr int VL_ROWS = VBR * VBR;          // 16 rows (y, z) per brick row

struct VoterRows {
  float s[VL_ROWS];       // saliency * mask weight, or 0 where the voxel is no voter
  __device__ __forceinline__ void load(const VoterSrc &v, int x, int by, int bz) {
    float m[VL_ROWS];
    // one base index and two strides instead of sixteen 64-bit index computations
    const int ylim = v.ny - by * VBR;                 // rows (r & 3) < ylim exist
    const i64 zlim = v.nz - (i64)bz * VBR;            // planes (r >> 2) < zlim exist
    const i64 sy = v.nx, sz = (i64)v.nx * v.ny;
    const i64 i0 = ((i64)bz * VBR * v.ny + (i64)by * VBR) * v.nx + x;
    const bool xin = x < v.nx;
#pragma unroll
    for (int r = 0; r < VL_ROWS; r++) {
      const bool in = xin && (r & 3) < ylim && (r >> 2) < zlim;
      const i64 i = i0 + (r & 3) * sy + (r >> 2) * sz;
      s[r] = in ? __ldg(v.sal + i) : 0.0f;
      m[r] = (in && v.mask_src) ? __ldg(v.mask_src + i) : 1.0f;
    }
#pragma unroll
    for (int r = 0; r < VL_ROWS; r++) {
      // cut: handlers.cpp:1792; zero saliency never votes: feature.hpp:2268; masked voxels: :2259-2260;
      // a mask weight multiplies the decay, :2261-2265
      const bool voter = (s[r] >= v.thr) && s[r] != 0.0f && m[r] != 0.0f;
      s[r] = voter ? (v.mask_src ? s[r] * m[r] : s[r]) : 0.0f;
    }
  }
  // (a voter whose weighted saliency is exactly 0 cannot occur: both factors are non-zero floats, and a
  // product that underflows to 0 would vote with weight 0 anyway)
};

__global__ void __launch_bounds__(32 * VL_WARPS) voter_count_kernel(VoterSrc v, uint32_t *__restrict__ counts) {
  const int lane = threadIdx.x & 31;
  const int bx0 = (blockIdx.x * VL_WARPS + (threadIdx.x >> 5)) * 8;
  if (bx0 >= v.vbx) return;
  const int by = blockIdx.y, bz = blockIdx.z;
  VoterRows rows;
  rows.load(v, bx0 * VBR + lane, by, bz);
  uint32_t cnt = 0;
#pragma unroll
  for (int r = 0; r < VL_ROWS; r++) {
    const unsigned bal = __ballot_sync(0xffffffffu, rows.s[r] != 0.0f);
    cnt += __popc((bal >> (lane & 28)) & 15u);
  }
  if ((lane & 3) == 0 && bx0 + (lane >> 2) < v.vbx) counts[((i64)bz * v.vby + by) * v.vbx + bx0 + (lane >> 2)] = cnt;
}

// Exclusive scan of n uint32 counters into off[0..n] (off[n] = total): per-block scan,
// scan of the block sums by one CTA, then offset add.
constexpr int SCAN_T = 1024, SCAN_I = 4, SCAN_B = SCAN_T * SCAN_I;

__device__ __forceinline__ uint32_t block_excl_scan(uint32_t v, uint32_t *sh, uint32_t &total) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  uint32_t x = v;
  for (int o = 1; o < 32; o <<= 1) {
    uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) sh[w] = x;
  __syncthreads();
  if (w == 0) {
    uint32_t s = sh[lane];
    for (int o = 1; o < 32; o <<= 1) {
      uint32_t y = __shfl_up_sync(0xffffffffu, s, o);
      if (lane >= o) s += y;
    }
    sh[lane] = s;
  }
  __syncthreads();
  uint32_t base = w ? sh[w - 1] : 0;
  total = sh[31];
  __syncthreads();
  return base + x - v;
}

__global__ void __launch_bounds__(SCAN_T)
scan_local_kernel(const uint32_t *__restrict__ in, uint32_t *__restrict__ out, uint32_t *__restrict__ sums, i64 n) {
  __shared__ uint32_t sh[32];
  i64 base = (i64)blockIdx.x * SCAN_B + (i64)threadIdx.x * SCAN_I;
  uint32_t v[SCAN_I], s = 0;
#pragma unroll
  for (int k = 0; k < SCAN_I; k++) {
    v[k] = (base + k < n) ? in[base + k] : 0u;
    s += v[k];
  }
  uint32_t tot;
  uint32_t ex = block_excl_scan(s, sh, tot);
#pragma unroll
  for (int k = 0; k < SCAN_I; k++) {
    if (base + k < n) out[base + k] = ex;
    ex += v[k];
  }
  if (threadIdx.x == 0) sums[blockIdx.x] = tot;
}

__global__ void __launch_bounds__(SCAN_T) scan_sums_kernel(uint32_t *__restrict__ sums, i64 m, uint32_t *__restrict__ total_out) {
  __shared__ uint32_t sh[32];
  uint32_t carry = 0;
  for (i64 base = 0; base < m; base += SCAN_T) {
    i64 i = base + threadIdx.x;
    uint32_t v = (i < m) ? sums[i] : 0u;
    uint32_t tot;
    uint32_t ex = block_excl_scan(v, sh, tot);
    if (i < m) sums[i] = carry + ex;
    carry += tot;
  }
  if (threadIdx.x == 0) *total_out = carry;
}

__global__ void __launch_bounds__(SCAN_T)
scan_add_kernel(uint32_t *__restrict__ out, const uint32_t *__restrict__ sums, i64 n, const uint32_t *__restrict__ total) {
  i64 base = (i64)blockIdx.x * SCAN_B + (i64)threadIdx.x * SCAN_I;
  uint32_t add = sums[blockIdx.x];
#pragma unroll
  for (int k = 0; k < SCAN_I; k++)
    if (base + k < n) out[base + k] += add;
  if (blockIdx.x == 0 && threadIdx.x == 0) out[n] = *total;
}

// One voter as the gather kernel consumes it (48 B; copied verbatim into shared memory).
struct __align__(16) VoterRec {
  float4 a;  // {-x, -y, -z, log2(4w)/2}
  float4 b;  // {nx, ny, nz, log2(4w)}
  float4 c;  // {nx/2, ny/2, nz/2, 4w}       w = saliency * mask weight / table total
  // table kernel (lut), L = (4w)^(1/6): the vote u = sqrt(4w decay) cos^2 (n/2 - q r) picks up L from the dot
  // product, L^2 from cos^2 and L from n/2, so the weight costs no instruction in the loop.  The fields carry
  // power-of-two scales (exact; see LUT_* below) chosen so that the r^2 accumulator of the loop is a DENORMAL
  // float whose bit pattern is the shared-memory address of the table row:
  //   a = {-x rho, -y rho, -z rho, L^2 K}, b = {L n beta, L}, c = {L n beta2, 0}
};
// rho^2 = 2^-142 = LUT_ROW ulps of the denormal range: (rho r)^2 accumulates to bits = base + 128 r^2.
// With ninv' = -tau / r^2 from the table: d' = (rho r).(beta L n) = rho beta L d, qn' = d' ninv' = -(rho beta tau) L q,
// ang' = qn' d' + K L^2 = K L^2 cos^2 (K = rho^2 beta^2 tau), h' = qn' (rho r) + beta2 L n = 2 beta2 L (n/2 - q r)
// (beta2 = rho^2 beta tau / 2), and the table's E' = E / (2 beta2 K) restores the scale.  Every intermediate is a
// normal float of moderate exponent; all scalings are powers of two, so the results are those of the unscaled form.
constexpr int LUT_RHO_LOG2 = -71, LUT_BETA_LOG2 = 40, LUT_TAU_LOG2 = 100;
constexpr int LUT_K_LOG2 = 2 * LUT_RHO_LOG2 + 2 * LUT_BETA_LOG2 + LUT_TAU_LOG2;        // 38
constexpr int LUT_BETA2_LOG2 = 2 * LUT_RHO_LOG2 + LUT_BETA_LOG2 + LUT_TAU_LOG2 - 1;    // -3
constexpr int LUT_E_LOG2 = -(1 + LUT_BETA2_LOG2 + LUT_K_LOG2);                         // -36
__host__ __device__ __forceinline__ float pow2f(int e) {   // 2^e, -126 <= e <= 127
  union { unsigned u; float f; } v; v.u = (unsigned)(e + 127) << 23; return v.f;
}

struct DirSrc {
  const float *direction;  // N*3, or NULL
  const float *smoothed;   // used when direction == NULL
  float ridge_sigma;
  int order;
  i64 z_offset, nz_global;
};

// Declared in ridge.cu's translation unit as static device code; restated here because
// the fill kernel needs the same stencil (kept tiny on purpose).
__device__ __forceinline__ void voter_direction(const DirSrc &d, int nx, int ny, int x, int y, i64 z, float n[3]) {
  i64 i = (z * ny + y) * (i64)nx + x;
  if (d.direction) {
    n[0] = __ldg(d.direction + 3 * i + 0);
    n[1] = __ldg(d.direction + 3 * i + 1);
    n[2] = __ldg(d.direction + 3 * i + 2);
    return;
  }
  // finite-difference Hessian of the smoothed image with the centre clamped at the
  // GLOBAL border (visfd_utils.hpp:530-616), times sigma^2 (feature.hpp:1331-1333)
  int cx = x, cy = y;
  i64 zg = d.z_offset + z;
  if (cx == 0) cx++; else if (cx == nx - 1) cx--;
  if (cy == 0) cy++; else if (cy == ny - 1) cy--;
  if (zg == 0) zg++; else if (zg == d.nz_global - 1) zg--;
  const i64 sy = nx, sz = (i64)nx * ny;
  const float *p = d.smoothed + ((zg - d.z_offset) * ny + cy) * (i64)nx + cx;
#define F(a, b, c) __ldg(p + (a) + (b) * sy + (c) * sz)
  float s2 = __fmul_rn(d.ridge_sigma, d.ridge_sigma);
  float c = F(0, 0, 0), c2 = __fmul_rn(2.0f, c);
  float hxx = __fmul_rn(__fsub_rn(__fadd_rn(F(1, 0, 0), F(-1, 0, 0)), c2), s2);
  float hyy = __fmul_rn(__fsub_rn(__fadd_rn(F(0, 1, 0), F(0, -1, 0)), c2), s2);
  float hzz = __fmul_rn(__fsub_rn(__fadd_rn(F(0, 0, 1), F(0, 0, -1)), c2), s2);
  float xy = __fsub_rn(__fsub_rn(__fadd_rn(F(1, 1, 0), F(-1, -1, 0)), F(1, -1, 0)), F(-1, 1, 0));
  float yz = __fsub_rn(__fsub_rn(__fadd_rn(F(0, 1, 1), F(0, -1, -1)), F(0, 1, -1)), F(0, -1, 1));
  float xz = __fsub_rn(__fsub_rn(__fadd_rn(F(1, 0, 1), F(-1, 0, -1)), F(-1, 0, 1)), F(1, 0, -1));
#undef F
  Sym3d m = {hxx, hyy, hzz, __fmul_rn(__fmul_rn(0.25f, xy), s2), __fmul_rn(__fmul_rn(0.25f, yz), s2),
             __fmul_rn(__fmul_rn(0.25f, xz), s2)};
  double e0[3];
  sym3_first_eigenvector_newton(m, d.order, e0);
  n[0] = (float)e0[0];
  n[1] = (float)e0[1];
  n[2] = (float)e0[2];
}

// Pass 1 of the fill: positions and weights in brick order, voxels of a brick in (z, y, x) order.  The records it
// writes are the same for both gather kernels; voter_direction_kernel puts them in the chosen kernel's form.
__global__ void __launch_bounds__(32 * VL_WARPS)
voter_fill_kernel(VoterSrc v, const uint32_t *__restrict__ off, float inv_total,
                  VoterRec *__restrict__ rec, uint32_t *__restrict__ nonpos_flag) {
  const int lane = threadIdx.x & 31;
  const int bx0 = (blockIdx.x * VL_WARPS + (threadIdx.x >> 5)) * 8;
  if (bx0 >= v.vbx) return;
  const int by = blockIdx.y, bz = blockIdx.z;
  const int x = bx0 * VBR + lane;
  VoterRows rows;
  rows.load(v, x, by, bz);
  const int bx = bx0 + (lane >> 2);
  const uint32_t base = (bx < v.vbx) ? __ldg(off + ((i64)bz * v.vby + by) * v.vbx + bx) : 0u;
  const unsigned below = (1u << (lane & 3)) - 1u;   // lanes of my nibble that come before me
  uint32_t rank = 0;                                 // voters of my brick in the rows done so far
#pragma unroll
  for (int r = 0; r < VL_ROWS; r++) {
    const unsigned nib = (__ballot_sync(0xffffffffu, rows.s[r] != 0.0f) >> (lane & 28)) & 15u;
    if (rows.s[r] != 0.0f) {
      const float wgt = rows.s[r] * inv_total;
      if (!(wgt > 0.0f)) *nonpos_flag = 1u;  // benign race: every writer stores the same value
      // position and raw weight only: the forms of the weight that the gather kernels fold into their arithmetic
      // (a logarithm, a sixth root) are computed by voter_direction_kernel, where every lane has a voter -- here
      // ~5 % of the lanes do, and a warp would run the libm sequence for them at that lane efficiency
      VoterRec *q = rec + base + rank + __popc(nib & below);
      q->a = make_float4(-(float)x, -(float)(by * VBR + (r & 3)), -(float)(bz * VBR + (r >> 2)), 0.0f);
      q->c.w = 4.0f * wgt;
    }
    rank += __popc(nib);
  }
}

// Pass 2: one THREAD per voter (dense lanes -- in the brick pass only ~5 % of the lanes are
// voters and the double-precision eigenvector would run at that lane efficiency).  Finishes each
// record for the gather kernel the host chose: lut = the table kernel.
__global__ void __launch_bounds__(256)
voter_direction_kernel(DirSrc d, int nx, int ny, uint32_t n_voters, bool lut, VoterRec *__restrict__ rec) {
  const uint32_t i = blockIdx.x * 256u + threadIdx.x;
  if (i >= n_voters) return;
  VoterRec *r = rec + i;
  const float4 a = r->a;
  float n[3];
  voter_direction(d, nx, ny, (int)(-a.x), (int)(-a.y), (i64)(-a.z), n);
  // the weight w4 = 4 * saliency * mask weight / table total in the three forms vote() / vote_lut() use
  const float w4 = r->c.w;
  float sb = 1.0f, sc = 0.5f;
  if (lut) {   // only used when every weight is positive (checked by the host before the launch)
    const float lam = (float)pow((double)fmaxf(w4, 0.0f), 1.0 / 6.0);
    sb = lam * pow2f(LUT_BETA_LOG2); sc = lam * pow2f(LUT_BETA2_LOG2);
    const float rho = pow2f(LUT_RHO_LOG2);   // the table kernel's position scale (exact: a power of two)
    r->a = make_float4(a.x * rho, a.y * rho, a.z * rho, lam * lam * pow2f(LUT_K_LOG2));
    r->b.w = lam;
    r->c.w = 0.0f;
  } else {
    const float l4 = log2f(w4);
    r->a.w = 0.5f * l4;
    r->b.w = l4;
  }
  r->b.x = sb * n[0]; r->b.y = sb * n[1]; r->b.z = sb * n[2];
  r->c.x = sc * n[0]; r->c.y = sc * n[1]; r->c.z = sc * n[2];
}

// ---------------------------------------------------------------------------------
// gather
// ---------------------------------------------------------------------------------
struct GatherArgs {
  const VoterRec *rec;
  const uint32_t *off;
  const uint32_t *shell;  // device copy of DecayInfo::shell_keep
  int n_shell;
  int nx, ny;
  i64 nz;                 // slab planes (voter bricks cover [0,nz))
  int nbx, nby, nbz;
  i64 own_z0, own_z1;     // receiver planes (slab-local)
  int ntx, nty;           // receiver tiles in x,y
  int hw;
  int row_cap;            // per-warp capacity of the row table
  float hw2;              // (float) hw*hw
  float lim_in;           // pairs with r2 < lim_in get the full weight ...
  float lim_pass;         // ... pairs with r2 in [lim_in, lim_pass) sit on the shell (SHELL kernels only)
  float neg_c;            // -log2(e)/sigma^2 (half of it for the SQRTW kernels)
  float half_exp;         // exponent/2, generic path
  const float *mask_dst;  // slab-indexed, or NULL
  float *tensor;          // own-planes-indexed * 6, or NULL
  float *score;           // own-planes-indexed, or NULL
  int order, score_kind;
  // table kernel only
  const float2 *lut;      // n_lut entries {sqrt(decay(r2)) or 0 outside the support, -1/r2 (0 at r2 = 0)}
  int n_lut;              // the last entry is {0, 0}: r2 is clamped to it when the table is shorter than the reach
  unsigned n_tiles;       // 8x8x4 receiver tiles of this launch
  unsigned *ticket;       // device counter handing out tiles, zeroed before the launch
};

__device__ __forceinline__ void cp_async16(void *smem, const void *gmem) {
  unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sa), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

__device__ __forceinline__ float fast_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float fast_rcp(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float fast_lg2(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __noinline__ float shell_weight(const uint32_t *shell, int n, float dx, float dy, float dz) {
  uint32_t key = (uint32_t)fabsf(dx) | ((uint32_t)fabsf(dy) << 8) | ((uint32_t)fabsf(dz) << 16);
  for (int k = 0; k < n; k++)
    if (__ldg(shell + k) == key) return 1.0f;
  return 0.0f;
}

__device__ __forceinline__ int axis_gap(int lo_a, int hi_a, int lo_b, int hi_b) {
  // distance between integer intervals [lo_a,hi_a] and [lo_b,hi_b]
  return max(0, max(lo_b - hi_a, lo_a - hi_b));
}

constexpr int TV_DRAIN = 32;             // voters evaluated per drain
constexpr int TV_GROUP = 8;              // voters per unrolled iteration of a drain (4 per half-warp) ...
#ifndef TV_GROUP_LUT_N
#define TV_GROUP_LUT_N 16
#endif
constexpr int TV_GROUP_LUT = TV_GROUP_LUT_N;   // ... and in the table kernel (8 per half-warp: -2.7 % in isolation)
// ring capacity: at most TV_DRAIN - 1 + 64 voters are queued when a streaming iteration (64 candidates,
// two per lane; three per lane measured no faster) starts, and it adds up to 64 more before the whole
// batches among the former are drained
constexpr int TV_QCAP = 5 * TV_DRAIN;
constexpr float TV_R2_EPS = 1e-30f;      // keeps 1/r^2 finite for the self vote (r = 0, d.n = 0)

__device__ __forceinline__ float2 bc(float x) { return make_float2(x, x); }  // FFMA2 takes scalar (.F32) operands

// The vote of one voter on the two receivers (x, y, z) and (x, y, z+1) of a lane.
// With r = receiver - voter, r2 = |r|^2, d = r.n, q = d/r2:  sin^2 = q*d (cos^2 = 1 - q*d),
// rotated normal v = n - 2 q r (feature.hpp:2341-2351; its sign does not matter for
// v v^T, so surfaces and curves share it).  We accumulate with h = v/2 = n/2 - q r and
// fold the factor 4 into the weight.  The two receivers share x and y, so the x/y terms
// of r2 and d are scalar; everything else is packed FP32 (FFMA2/FMUL2, whose scalar
// operand form reads a shared value without a register pair).
//   SQRTW (exponent 4, all weights > 0): weight*decay*ang^2*4 = (sE*ang)^2 with
//     sE = exp2(r2*neg_c/2 + log2(4w)/2);  T += (sE*ang*h)(sE*ang*h)^T
//   otherwise: w = decay*ang^(e/2)*weight*4,  T += (w h) h^T
// Pairs outside the support get weight 0.  Lattice points exactly on the shell
// r2 == hw^2 are kept or dropped by float rounding in the reference's table
// (filter3d.hpp:546-601); the host evaluates that table: all kept (every parameter set we
// have seen) or all dropped is folded into lim_in = hw^2 +- 0.5; a mixed shell runs the
// SHELL kernels, which look each on-shell pair up in the list of kept points.
template <int EXPO, bool CURVES, bool POSW, bool SHELL>
__device__ __forceinline__ void vote_pair(float rx, float ry, float rxy2, float dxy, float2 fz, const float4 &ea,
                                          const float4 &eb, const float4 &ec, const GatherArgs &g, float negc,
                                          float lim_in, float2 T[6]) {
  constexpr bool SQRTW = (EXPO == 4) && POSW;
  const float2 rz = __fadd2_rn(fz, bc(ea.z));
  const float2 r2 = __ffma2_rn(rz, rz, bc(rxy2));
  const float2 d = __ffma2_rn(rz, bc(eb.z), bc(dxy));
  float2 ee;
  if (POSW) {
    const float2 arg = __ffma2_rn(r2, bc(negc), bc(SQRTW ? ea.w : eb.w));
    ee = make_float2(fast_ex2(arg.x), fast_ex2(arg.y));
  } else {
    const float2 arg = __fmul2_rn(r2, bc(negc));
    ee = __fmul2_rn(make_float2(fast_ex2(arg.x), fast_ex2(arg.y)), bc(ec.w));
  }
  const float2 ninv = make_float2(fast_rcp(-r2.x), fast_rcp(-r2.y));
  const float2 qn = __fmul2_rn(d, ninv);  // -q
  float2 ang2;                             // cos^2 (surfaces) / -sin^2 (curves)
  if (CURVES) ang2 = __fmul2_rn(qn, d);
  else ang2 = __ffma2_rn(qn, d, make_float2(1.0f, 1.0f));
  float2 w;
  if (SQRTW) {
    w = __fmul2_rn(ee, ang2);              // sign irrelevant: it is squared below
  } else {
    if (CURVES) ang2 = make_float2(-ang2.x, -ang2.y);
    float2 ang;
    if (EXPO == 2) ang = ang2;
    else if (EXPO == 4) ang = __fmul2_rn(ang2, ang2);
    else ang = make_float2(fast_ex2(g.half_exp * fast_lg2(fmaxf(ang2.x, 0.0f))),
                           fast_ex2(g.half_exp * fast_lg2(fmaxf(ang2.y, 0.0f))));
    w = __fmul2_rn(ee, ang);
  }
  {
    const float2 wfull = w;
    w.x = (r2.x < lim_in) ? w.x : 0.0f;
    w.y = (r2.y < lim_in) ? w.y : 0.0f;
    if (SHELL) {
      const bool sx = r2.x >= lim_in && r2.x < g.lim_pass, sy = r2.y >= lim_in && r2.y < g.lim_pass;
      if (__any_sync(0xffffffffu, sx || sy)) {
        if (sx) w.x = wfull.x * shell_weight(g.shell, g.n_shell, rx, ry, rz.x);
        if (sy) w.y = wfull.y * shell_weight(g.shell, g.n_shell, rx, ry, rz.y);
      }
    }
  }
  const float2 hx = __ffma2_rn(qn, bc(rx), bc(ec.x));
  const float2 hy = __ffma2_rn(qn, bc(ry), bc(ec.y));
  const float2 hz = __ffma2_rn(qn, rz, bc(ec.z));
  const float2 wx = __fmul2_rn(w, hx), wy = __fmul2_rn(w, hy), wz = __fmul2_rn(w, hz);
  if (SQRTW) {
    T[0] = __ffma2_rn(wx, wx, T[0]);
    T[3] = __ffma2_rn(wx, wy, T[3]);
    T[5] = __ffma2_rn(wx, wz, T[5]);
    T[1] = __ffma2_rn(wy, wy, T[1]);
    T[4] = __ffma2_rn(wy, wz, T[4]);
    T[2] = __ffma2_rn(wz, wz, T[2]);
  } else {
    T[0] = __ffma2_rn(wx, hx, T[0]);
    T[3] = __ffma2_rn(wx, hy, T[3]);
    T[5] = __ffma2_rn(wx, hz, T[5]);
    T[1] = __ffma2_rn(wy, hy, T[1]);
    T[4] = __ffma2_rn(wy, hz, T[4]);
    T[2] = __ffma2_rn(wz, hz, T[2]);
  }
}

// One voter on the FOUR receivers (x, y, z..z+3) of a lane: the x/y terms once, then the two
// z pairs.  T[0..5]: receivers z, z+1; T[6..11]: z+2, z+3.
template <int EXPO, bool CURVES, bool POSW, bool SHELL>
__device__ __forceinline__ void vote(const VoterRec *q, float fx, float fy, float2 fz01, float2 fz23,
                                     const GatherArgs &g, float negc, float lim_in, float2 T[12]) {
  const float4 ea = q->a, eb = q->b, ec = q->c;
  const float rx = fx + ea.x, ry = fy + ea.y;
  const float rxy2 = fmaf(ry, ry, fmaf(rx, rx, TV_R2_EPS));
  const float dxy = fmaf(ry, eb.y, rx * eb.x);
  vote_pair<EXPO, CURVES, POSW, SHELL>(rx, ry, rxy2, dxy, fz01, ea, eb, ec, g, negc, lim_in, T);
  vote_pair<EXPO, CURVES, POSW, SHELL>(rx, ry, rxy2, dxy, fz23, ea, eb, ec, g, negc, lim_in, T + 6);
}


// ---- table variant (exponent 4, weights > 0) ---------------------------------------------------
// The table holds 128-byte rows, one per integer r^2: 16 replicas of {E', -tau/r^2}; a lane reads replica
// lane & 15, so the 16 lanes of a half-warp -- which share the voter -- cover all 32 banks exactly once.
// The r^2 accumulator starts at the bit pattern of the lane's replica address (a denormal float, the shared
// window is < 2^23 bytes) and every (rho r)^2 term adds 128 ulps per unit of r^2 exactly (denormal arithmetic is
// fixed point), so its bits ARE the address of the row: no conversion, no add.  (Round 1 of this kernel used
// MAGIC = 65536 + r^2 and an IADD3 per lookup; together with the MOVs that re-paired the two lookups for a
// packed multiply that was 10 of ~106 issue slots per voter and lane.)
constexpr int LUT_ROW = 128;            // bytes per r2
constexpr int LUT_MAX_HW = 24;
struct LutState {
  float base;        // bit pattern = shared-window address of the lane's replica of row 0
  float r2m_max;     // bit pattern = address of the lane's replica of the last row (CLAMP)
};
__device__ __forceinline__ float2 lut_fetch(float r2m) {
  float2 t;
  asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(t.x), "=f"(t.y) : "r"(__float_as_uint(r2m)));
  return t;
}
__device__ __forceinline__ float fmul_s(float a, float b) {   // a scalar multiply ptxas may not re-pair
  float d;
  asm("mul.rn.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b));
  return d;
}
template <bool CURVES, bool CLAMP>
__device__ __forceinline__ void vote_pair_lut(float rx, float ry, float rxy2m, float dxy, float2 fz, const float4 &ea,
                                              const float4 &eb, const float4 &ec, const LutState &L, float2 T[6]) {
  const float2 rz = __fadd2_rn(fz, bc(ea.z));
  float2 r2m = __ffma2_rn(rz, rz, bc(rxy2m));
  if (CLAMP) { r2m.x = fminf(r2m.x, L.r2m_max); r2m.y = fminf(r2m.y, L.r2m_max); }
  const float2 d = __ffma2_rn(rz, bc(eb.z), bc(dxy));        // d'
  const float2 t0 = lut_fetch(r2m.x), t1 = lut_fetch(r2m.y);
  // {E', ninv'} of the two receivers arrive as two register pairs; multiplying them in scalar form costs the
  // same two FMA-pipe cycles as one packed multiply and saves the two MOVs that would re-pair them
  float2 qn, w;
  qn.x = fmul_s(d.x, t0.y); qn.y = fmul_s(d.y, t1.y);        // qn'
  float2 ang2;                                               // K L^2 cos^2 (surfaces) / -K L^2 sin^2 (curves)
  if (CURVES) ang2 = __fmul2_rn(qn, d);
  else ang2 = __ffma2_rn(qn, d, bc(ea.w));
  w.x = fmul_s(t0.x, ang2.x); w.y = fmul_s(t1.x, ang2.y);    // sign irrelevant: squared below
  const float2 hx = __ffma2_rn(qn, bc(rx), bc(ec.x));        // h'
  const float2 hy = __ffma2_rn(qn, bc(ry), bc(ec.y));
  const float2 hz = __ffma2_rn(qn, rz, bc(ec.z));
  const float2 wx = __fmul2_rn(w, hx), wy = __fmul2_rn(w, hy), wz = __fmul2_rn(w, hz);
  T[0] = __ffma2_rn(wx, wx, T[0]);
  T[3] = __ffma2_rn(wx, wy, T[3]);
  T[5] = __ffma2_rn(wx, wz, T[5]);
  T[1] = __ffma2_rn(wy, wy, T[1]);
  T[4] = __ffma2_rn(wy, wz, T[4]);
  T[2] = __ffma2_rn(wz, wz, T[2]);
}
template <bool CURVES, bool CLAMP>
__device__ __forceinline__ void vote_lut(const VoterRec *q, float fx, float fy, float2 fz01, float2 fz23, const LutState &L,
                                         float2 T[12]) {
  const float4 ea = q->a, eb = q->b, ec = q->c;
  const float rx = fx + ea.x, ry = fy + ea.y;                // rho r
  const float rxy2m = fmaf(ry, ry, fmaf(rx, rx, L.base));
  const float dxy = fmaf(ry, eb.y, rx * eb.x);
  vote_pair_lut<CURVES, CLAMP>(rx, ry, rxy2m, dxy, fz01, ea, eb, ec, L, T);
  vote_pair_lut<CURVES, CLAMP>(rx, ry, rxy2m, dxy, fz23, ea, eb, ec, L, T + 6);
}

// n consecutive ring entries (n a multiple of 4; a drain never wraps, see the kernel): the
// lanes of half-warp h take entries h, h+2, h+4, ... -- two voters per warp iteration.
// LUT: 0 = decay by MUFU (vote), 1 = table covering the whole reach, 2 = table with clamped index
template <int EXPO, bool CURVES, bool POSW, bool SHELL, int LUT>
__device__ __forceinline__ void drain(const VoterRec *q, int n, float fx, float fy, float2 fz01, float2 fz23,
                                      const GatherArgs &g, float negc, float lim_in, const LutState &L, float2 T[12]) {
  const VoterRec *end = q + n;
  constexpr int G = LUT ? TV_GROUP_LUT : TV_GROUP;
#pragma unroll 1
  for (; q < end; q += G) {
#pragma unroll
    for (int u = 0; u < G; u += 2) {
      if (LUT) vote_lut<CURVES, LUT == 2>(q + u, fx, fy, fz01, fz23, L, T);
      else vote<EXPO, CURVES, POSW, SHELL>(q + u, fx, fy, fz01, fz23, g, negc, lim_in, T);
    }
  }
}
// The two halves' tensors are added (half 0 finishes receivers z, z+1, half 1 z+2, z+3), then the optional
// 6-component store and the post-vote score, accumulators still in registers.
__device__ __forceinline__ void patch_epilogue(const GatherArgs &g, const float2 T[12], int half, int ix, int iy, int pz) {
  float2 Tm[6];
#pragma unroll
  for (int k = 0; k < 6; k++) {
    const float2 give = half ? T[k] : T[k + 6];      // what the partner lane finishes
    const float2 keep = half ? T[k + 6] : T[k];
    Tm[k].x = keep.x + __shfl_xor_sync(0xffffffffu, give.x, 16);
    Tm[k].y = keep.y + __shfl_xor_sync(0xffffffffu, give.y, 16);
  }
  const int iz = pz + 2 * half;
  if (ix < g.nx && iy < g.ny) {
#pragma unroll
    for (int r = 0; r < 2; r++) {
      const i64 z = iz + r;
      if (z >= g.own_z1) break;
      float Tr[6];
#pragma unroll
      for (int k = 0; k < 6; k++) Tr[k] = r ? Tm[k].y : Tm[k].x;
      const i64 slab_i = (z * g.ny + iy) * (i64)g.nx + ix;
      const i64 out_i = ((z - g.own_z0) * g.ny + iy) * (i64)g.nx + ix;
      const bool masked = g.mask_dst && __ldg(g.mask_dst + slab_i) == 0.0f;  // feature.hpp:2002-2003
      if (g.tensor) {
        float *o = g.tensor + 6 * out_i;
#pragma unroll
        for (int k = 0; k < 6; k++) o[k] = masked ? 0.0f : Tr[k];
      }
      if (g.score) {
        float sc = 0.0f;
        if (!masked) {
          Sym3d mm = {Tr[0], Tr[1], Tr[2], Tr[3], Tr[4], Tr[5]};
          double ev[3];
          sym3_eigenvalues(mm, g.order, ev);
          sc = score_from_eivals(ev, g.score_kind, 1);
        }
        g.score[out_i] = sc;
      }
    }
  }
}

// One WARP per 4x4x4 receiver patch.  Lane = (x, y, h): the lanes of half-warp h hold all four
// z-receivers of their (x, y) column (24 accumulators as twelve packed pairs), and the two
// half-warps evaluate DIFFERENT voters in the same iteration -- h takes every second ring entry
// -- and add their tensors at the end.  A lane thus amortises the x/y terms and the three
// LDS.128 of a voter over four receivers instead of two (-9 % per evaluation in isolation),
// while the patch a voter is culled against stays the 4x4x4 cube.  The 4 warps of a CTA cover
// an 8x8x4 tile and never synchronise with each other.  A warp
//   1. builds the table of brick rows (contiguous ranges of the brick-ordered voter
//      list) whose bricks can reach its patch,
//   2. streams them 64 candidates at a time: each lane loads the positions of two
//      candidates (one iteration ahead, straight from L1/L2), tests the exact distance between
//      the voter and the patch box against the support radius, and -- if the voter can
//      reach the patch -- copies its 48-byte record with cp.async into the next free slot
//      of a warp-private shared-memory ring (slot = ballot rank),
//   3. whenever the ring held >= 32 voters BEFORE the current iteration appended to it, waits
//      for all but the newest cp.async group and drains them 32 at a time: 16 iterations of
//      two voters (the three LDS.128 carry one address per half-warp).
// Ring invariant: capacity 160, head a multiple of 32; an iteration tests 64 candidates.
// Before it the ring holds <= 95 voters, it adds <= 64 (159 < 160 live), and it drains the
// whole groups of 32 among the voters queued before it -- all of which belong to cp.async
// groups older than the newest one -- leaving <= 31 + 64.
template <int EXPO, bool CURVES, bool POSW, bool SHELL, int LUT>
__device__ __forceinline__ void gather_patch(const GatherArgs &g, const unsigned slot, unsigned char *mine, const LutState &L) {
  const int lane = threadIdx.x & 31;
  const int warp = slot & 3;
  VoterRec *ring = reinterpret_cast<VoterRec *>(mine);
  uint32_t *row_start = reinterpret_cast<uint32_t *>(ring + TV_QCAP);
  uint32_t *row_pref = row_start + g.row_cap;  // [row_cap + 1]

  // CTA tile: 8 x 8 x 4 receivers (ntx x nty x layers of 4 planes)
  const int tile = slot >> 2;
  const int tx = tile % g.ntx, ty = (tile / g.ntx) % g.nty, tz = tile / (g.ntx * g.nty);
  const int px = tx * BR + (warp & 1) * 4, py = ty * BR + (warp >> 1) * 4;
  const int pz = (int)g.own_z0 + tz * TV_TILE_Z;
  if (px >= g.nx || py >= g.ny || pz >= g.own_z1) return;  // whole warp: no receivers
  const int pz_hi = (int)min((i64)pz + 3, g.own_z1 - 1), py_hi = min(py + 3, g.ny - 1), px_hi = min(px + 3, g.nx - 1);

  // ---- 1. brick rows that can reach the patch ----------------------------------------
  const int bz_lo = max(0, (pz - g.hw) >> VSH), bz_hi = min(g.nbz - 1, (pz_hi + g.hw) >> VSH);
  const int by_lo = max(0, (py - g.hw) >> VSH), by_hi = min(g.nby - 1, (py_hi + g.hw) >> VSH);
  const int nry = by_hi - by_lo + 1;
  const int nrows = (bz_hi - bz_lo + 1) * nry;  // <= row_cap by construction
  uint32_t carry = 0;
  for (int r0 = 0; r0 < nrows; r0 += 32) {
    const int r = r0 + lane;
    uint32_t start = 0, len = 0;
    if (r < nrows) {
      const int bz = bz_lo + r / nry, by = by_lo + r % nry;
      const int dz = axis_gap(pz, pz_hi, bz * VBR, bz * VBR + VBR - 1);
      const int dy = axis_gap(py, py_hi, by * VBR, by * VBR + VBR - 1);
      const int rem = g.hw * g.hw - dz * dz - dy * dy;
      if (rem >= 0) {
        int d = (int)floorf(sqrtf((float)rem));
        while ((d + 1) * (d + 1) <= rem) d++;
        while (d * d > rem) d--;
        const int bx_lo = max(0, (px - d) >> VSH), bx_hi = min(g.nbx - 1, (px_hi + d) >> VSH);
        const i64 rb = ((i64)bz * g.nby + by) * g.nbx;
        start = __ldg(g.off + rb + bx_lo);
        len = __ldg(g.off + rb + bx_hi + 1) - start;
      }
    }
    uint32_t incl = len;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      uint32_t y = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += y;
    }
    if (r < nrows) {
      row_start[r] = start;
      row_pref[r] = carry + incl - len;
    }
    carry += __shfl_sync(0xffffffffu, incl, 31);
  }
  if (lane == 0) row_pref[nrows] = carry;
  __syncwarp();
  const uint32_t total = carry;

  // ---- receivers of this lane: (ix, iy, pz .. pz+3); its voters: every second ring entry ----
  const int ix = px + (lane & 3), iy = py + ((lane >> 2) & 3), half = lane >> 4;
  // (the table kernel works in coordinates scaled by rho = 2^-71, see LUT_*: every comparison below is exact in
  // either scale, the squared distances of the scaled form being fixed-point denormals)
  const float cs = LUT ? pow2f(LUT_RHO_LOG2) : 1.0f;
  const float fx = (float)ix * cs, fy = (float)iy * cs;
  const float2 fz01 = make_float2((float)pz * cs, (float)(pz + 1) * cs), fz23 = make_float2((float)(pz + 2) * cs, (float)(pz + 3) * cs);
  const float pcx = (px + 1.5f) * cs, pcy = (py + 1.5f) * cs, pcz = (pz + 1.5f) * cs, box = 1.5f * cs;
  const float negc = g.neg_c;  // already halved on the host for the SQRTW kernels
  const float lim_in = g.lim_in, lim_pass = (g.lim_pass * cs) * cs;
  float2 T[12];
#pragma unroll
  for (int k = 0; k < 12; k++) T[k] = make_float2(0.0f, 0.0f);

  // ---- 2./3. stream, cull, vote ---------------------------------------------------------
  int cur_row = 0;  // per-lane cursor into the row table (flat indices only grow)
  auto locate = [&](uint32_t e) -> uint32_t {
    while (e >= row_pref[cur_row + 1]) cur_row++;
    return row_start[cur_row] + (e - row_pref[cur_row]);
  };
  auto reach = [&](const float4 &a) -> bool {
    // exact distance from the voter (a holds the NEGATED position) to the patch box
    const float gx = fmaxf(fabsf(a.x + pcx) - box, 0.0f);
    const float gy = fmaxf(fabsf(a.y + pcy) - box, 0.0f);
    const float gz = fmaxf(fabsf(a.z + pcz) - box, 0.0f);
    return fmaf(gx, gx, fmaf(gy, gy, gz * gz)) < lim_pass;
  };
  auto enqueue = [&](int slot, uint32_t gi) {
    if (slot >= TV_QCAP) slot -= TV_QCAP;
    VoterRec *dst = ring + slot;
    const VoterRec *src = g.rec + gi;
    cp_async16(&dst->a, &src->a);
    cp_async16(&dst->b, &src->b);
    cp_async16(&dst->c, &src->c);
  };
  int head = 0, cnt = 0;
  // candidate e of the stream, clamped to the last one so that every lane always loads (an
  // unconditional load keeps the prefetch out of the way of the registers in use; lanes past
  // the end are masked when their candidate is tested)
  auto fetch = [&](uint32_t e, uint32_t &gi, float4 &a) {
    gi = locate(min(e, total - 1));
    a = __ldg(&g.rec[gi].a);
  };
  uint32_t ng0 = 0, ng1 = 0;
  float4 na0 = make_float4(0.f, 0.f, 0.f, 0.f), na1 = na0;
  if (total > 0) {
    fetch(lane, ng0, na0);
    fetch(32 + lane, ng1, na1);
  }
  for (uint32_t base = 0; base < total; base += 64) {
    const float4 a0 = na0, a1 = na1;
    const uint32_t g0 = ng0, g1 = ng1;
    fetch(base + 64 + lane, ng0, na0);
    fetch(base + 96 + lane, ng1, na1);
    const bool p0 = base + lane < total && reach(a0), p1 = base + 32 + lane < total && reach(a1);
    const unsigned m0 = __ballot_sync(0xffffffffu, p0), m1 = __ballot_sync(0xffffffffu, p1);
    const unsigned below = (1u << lane) - 1u;
    const int n0 = __popc(m0);
    if (p0) enqueue(head + cnt + __popc(m0 & below), g0);
    if (p1) enqueue(head + cnt + n0 + __popc(m1 & below), g1);
    cp_async_commit();
    const int ndrain = cnt & ~(TV_DRAIN - 1);   // whole drains among the voters queued BEFORE this iteration
    cnt += n0 + __popc(m1);
    if (ndrain) {
      cp_async_wait<1>();
      __syncwarp();
      for (int d = 0; d < ndrain; d += TV_DRAIN) {
        drain<EXPO, CURVES, POSW, SHELL, LUT>(ring + head + half, TV_DRAIN, fx, fy, fz01, fz23, g, negc, lim_in, L, T);
        head = (head + TV_DRAIN == TV_QCAP) ? 0 : head + TV_DRAIN;
      }
      cnt -= ndrain;
      __syncwarp();
    }
  }
  // leftovers (< 160), padded to a multiple of 4 with zero-weight voters
  cp_async_wait<0>();
  constexpr int G = LUT ? TV_GROUP_LUT : TV_GROUP;   // voters per unrolled drain iteration
  if (lane < ((G - (cnt & (G - 1))) & (G - 1))) {
    int slot = head + cnt + lane;
    if (slot >= TV_QCAP) slot -= TV_QCAP;
    if (LUT) {
      // a zero vote: the lane's own position (r = 0, so the index stays inside the table) and L = 0
      ring[slot].a = make_float4(-(float)px * cs, -(float)py * cs, -(float)pz * cs, 0.0f);
      ring[slot].b = make_float4(0.f, 0.f, 0.f, 0.f);
    } else {
      const float ninf = __int_as_float(0xff800000u);  // ex2(-inf) = 0
      ring[slot].a = make_float4(1.0e4f, 1.0e4f, 1.0e4f, ninf);
      ring[slot].b = make_float4(0.f, 0.f, 0.f, ninf);
    }
    ring[slot].c = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  __syncwarp();
  cnt = (cnt + G - 1) & ~(G - 1);
  while (cnt > 0) {
    const int n = min(cnt, min(TV_DRAIN, TV_QCAP - head));
    drain<EXPO, CURVES, POSW, SHELL, LUT>(ring + head + half, n, fx, fy, fz01, fz23, g, negc, lim_in, L, T);
    head = (head + n == TV_QCAP) ? 0 : head + n;
    cnt -= n;
  }

  patch_epilogue(g, T, half, ix, iy, pz);
}


// 4 warps per CTA = one 8x8x4 receiver tile; decay by MUFU.
template <int EXPO, bool CURVES, bool POSW, bool SHELL>
__global__ void __launch_bounds__(TV_THREADS, TV_MIN_CTAS) tv_gather_kernel(GatherArgs g) {
  extern __shared__ __align__(16) unsigned char tv_smem[];
  const unsigned slot = blockIdx.x * TV_WARPS + (threadIdx.x >> 5);   // warp slot: 4 per tile
  const size_t per_warp = TV_QCAP * sizeof(VoterRec) + (2 * (size_t)g.row_cap + 4) * sizeof(uint32_t);
  unsigned char *mine = tv_smem + (threadIdx.x >> 5) * ((per_warp + 15) & ~(size_t)15);
  LutState L{0.0f, 0.0f};
  gather_patch<EXPO, CURVES, POSW, SHELL, 0>(g, slot, mine, L);
}

// Persistent table kernel: one CTA of 16 warps per SM, the table once per CTA.  The warps never wait for
// each other after the table is in place.  Work is handed out per QUAD of warps (4 quads per CTA): the four
// patches of an 8x8x4 tile go to the four next tickets of one quad, so that they run on the same SM at about the
// same time and find each other's candidates in L1, and a warp that finishes early takes the first patch of the
// quad's next tile instead of idling.  The warp that draws a tile's first ticket fetches the tile number from the
// device-wide counter and publishes it in shared memory; the other three pick it up there.
#ifndef LUT_WARPS_N
#define LUT_WARPS_N 16
#endif
constexpr int LUT_WARPS = LUT_WARPS_N, LUT_QUADS = LUT_WARPS / 4, LUT_SEQ = 8;   // a slot is reused 32 tickets later
template <bool CURVES, bool CLAMP>
__global__ void __launch_bounds__(32 * LUT_WARPS, 1) tv_gather_lut_kernel(GatherArgs g) {
  extern __shared__ __align__(16) unsigned char tv_smem[];
  __shared__ unsigned quad_ticket[LUT_QUADS];
  __shared__ volatile unsigned quad_tile[LUT_QUADS][LUT_SEQ], quad_seq[LUT_QUADS][LUT_SEQ];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, quad = w >> 2;
  const size_t tab_bytes = (size_t)g.n_lut * LUT_ROW;
  {
    float2 *tab = reinterpret_cast<float2 *>(tv_smem);
    for (int i = threadIdx.x; i < g.n_lut * (LUT_ROW / 8); i += 32 * LUT_WARPS) tab[i] = __ldg(g.lut + i / (LUT_ROW / 8));
    if (threadIdx.x < LUT_QUADS) quad_ticket[threadIdx.x] = 0u;
    if (threadIdx.x < LUT_QUADS * LUT_SEQ) quad_seq[threadIdx.x / LUT_SEQ][threadIdx.x % LUT_SEQ] = 0u;
  }
  __syncthreads();
  const size_t per_warp = (TV_QCAP * sizeof(VoterRec) + (2 * (size_t)g.row_cap + 4) * sizeof(uint32_t) + 15) & ~(size_t)15;
  unsigned char *mine = tv_smem + tab_bytes + w * per_warp;
  LutState L;
  const unsigned replica = (unsigned)__cvta_generic_to_shared(tv_smem) + 8u * (lane & 15);
  L.base = __uint_as_float(replica);
  L.r2m_max = __uint_as_float(replica + (unsigned)LUT_ROW * (unsigned)(g.n_lut - 1));
  for (;;) {
    unsigned t = 0, tile = 0;
    if (lane == 0) {
      t = atomicAdd(&quad_ticket[quad], 1u);
      const unsigned k = t >> 2, s = k % LUT_SEQ;
      if ((t & 3u) == 0u) {
        tile = atomicAdd(g.ticket, 1u);
        quad_tile[quad][s] = tile;
        __threadfence_block();
        quad_seq[quad][s] = k + 1u;
      } else {
        while (quad_seq[quad][s] != k + 1u) {}
        __threadfence_block();
        tile = quad_tile[quad][s];
      }
    }
    t = __shfl_sync(0xffffffffu, t, 0);
    tile = __shfl_sync(0xffffffffu, tile, 0);
    if (tile >= g.n_tiles) break;   // the counter only grows: every later ticket of this quad ends here too
    gather_patch<4, CURVES, true, false, CLAMP ? 2 : 1>(g, tile * 4u + (t & 3u), mine, L);
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------------
// host driver
// ---------------------------------------------------------------------------------
// Count, scan, fill: the voter list in brick order (off = the list's offset of every brick), its records in the
// form voter_fill_kernel leaves them.  Returns the number of voters; nonpos: some voter's weight is <= 0.
static uint32_t build_voter_list(visfd_ctx *ctx, const VoterSrc &vs, float inv_total, Scratch<uint32_t> &off,
                                 Scratch<VoterRec> &rec, bool &nonpos) {
  const i64 n_bricks = (i64)vs.vbx * vs.vby * vs.vbz;
  const dim3 grid((unsigned)div_up(vs.vbx, 8 * VL_WARPS), (unsigned)vs.vby, (unsigned)vs.vbz);
  Scratch<uint32_t> counts(ctx, n_bricks);
  off.reset(ctx, n_bricks + 1);
  const i64 n_scan_blocks = (n_bricks + SCAN_B - 1) / SCAN_B;
  Scratch<uint32_t> sums(ctx, n_scan_blocks + 2);   // block sums, [n] = total, [n+1] = non-positive-weight flag
  uint32_t *total = sums.get() + n_scan_blocks, *flag = total + 1;
  voter_count_kernel<<<grid, 32 * VL_WARPS, 0, ctx->stream>>>(vs, counts.get());
  VCK(cudaGetLastError());
  scan_local_kernel<<<(unsigned)n_scan_blocks, SCAN_T, 0, ctx->stream>>>(counts.get(), off.get(), sums.get(), n_bricks);
  VCK(cudaGetLastError());
  scan_sums_kernel<<<1, SCAN_T, 0, ctx->stream>>>(sums.get(), n_scan_blocks, total);
  VCK(cudaGetLastError());
  scan_add_kernel<<<(unsigned)n_scan_blocks, SCAN_T, 0, ctx->stream>>>(off.get(), sums.get(), n_bricks, total);
  VCK(cudaGetLastError());
  ctx->count_launch(4);
  uint32_t n_voters = 0, nonpos_flag = 0;
  VCK(cudaMemcpyAsync(&n_voters, total, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  VCK(cudaStreamSynchronize(ctx->stream));
  // (a 32-bit voter count: 4.29e9 voters would need 137 GB of voter records anyway)
  rec.reset(ctx, std::max<size_t>(n_voters, 1));
  if (n_voters > 0) {
    VCK(cudaMemsetAsync(flag, 0, sizeof(uint32_t), ctx->stream));
    voter_fill_kernel<<<grid, 32 * VL_WARPS, 0, ctx->stream>>>(vs, off.get(), inv_total, rec.get(), flag);
    VCK(cudaGetLastError());
    ctx->count_launch();
    VCK(cudaMemcpyAsync(&nonpos_flag, flag, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    VCK(cudaStreamSynchronize(ctx->stream));
  }
  nonpos = nonpos_flag != 0;
  return n_voters;
}

// Which gather kernel runs, and with what arguments.
struct GatherPlan {
  int kernel = 0;           // 0: tv_gather_kernel, 1: tv_gather_lut_kernel, 2: the same with a clamped table index
  int expo;                 // tv_gather_kernel<EXPO, CURVES, POSW, SHELL>: EXPO 2 or 4, 0 for any other exponent
  bool curves, posw, shell;
  float lim_in, lim_pass;   // GatherArgs::lim_in / lim_pass
  int row_cap;              // GatherArgs::row_cap
  int n_lut = 0;            // table rows (kernels 1 and 2)
  size_t smem;              // dynamic shared memory per CTA
  float neg_c;              // GatherArgs::neg_c
};

// The table kernel wants exponent 4, positive weights, a support whose shell is all kept or all dropped, and a
// radius whose table fits beside its 16 voter rings in smem_optin bytes of shared memory.  No voters: kernel 0.
static GatherPlan plan_gather(const TVParams &p, int hw, const DecayInfo &info, uint32_t n_voters, bool nonpos,
                              int smem_optin) {
  GatherPlan pl;
  // lattice points on the shell r2 == hw^2: all kept / all dropped / mixed (see vote())
  const bool mixed_shell = info.shell_total != 0 && info.shell_kept != 0 && info.shell_kept != info.shell_total;
  const bool shell_in = info.shell_total != 0 && info.shell_kept == info.shell_total;
  const float hw2 = (float)(hw * hw);
  pl.lim_in = hw2 + ((shell_in && !mixed_shell) ? 0.5f : -0.5f);
  pl.lim_pass = hw2 + ((shell_in || mixed_shell) ? 0.5f : -0.5f);
  const int per_axis = ((2 * hw + 3) >> VSH) + 2;
  pl.row_cap = per_axis * per_axis;
  const size_t per_warp = (TV_QCAP * sizeof(VoterRec) + (2 * (size_t)pl.row_cap + 4) * sizeof(uint32_t) + 15) & ~(size_t)15;
  pl.expo = (p.exponent == 2 || p.exponent == 4) ? p.exponent : 0;
  pl.curves = p.curves != 0;
  pl.shell = mixed_shell;
  // POSW: all voter weights > 0 (always true for the planar ridge score), so log2(weight) rides in the decay exponent
  pl.posw = !mixed_shell && !nonpos;
  pl.neg_c = (float)(-1.4426950408889634 / ((double)p.sigma * (double)p.sigma));
  pl.smem = TV_WARPS * per_warp;
  if (p.exponent == 4 && pl.posw && hw <= LUT_MAX_HW && n_voters > 0) {
    const size_t budget = (size_t)smem_optin - 1024;   // the kernel's static shared memory (work tickets)
    // largest r2 between a receiver of a 4x4x4 patch and a voter the cull lets through (gap vector g, |g|^2 < lim_pass)
    int r2_reach = 27;
    for (int gz = 0; gz <= hw; gz++)
      for (int gy = 0; gy <= hw; gy++)
        for (int gx = 0; gx <= hw; gx++)
          if ((float)(gx * gx + gy * gy + gz * gz) < pl.lim_pass)
            r2_reach = std::max(r2_reach, (gx + 3) * (gx + 3) + (gy + 3) * (gy + 3) + (gz + 3) * (gz + 3));
    const int r2_in = (int)floorf(pl.lim_in);          // largest r2 with a non-zero weight (lim_in = hw^2 +- 0.5)
    const int n_full = r2_reach + 1, n_clamped = r2_in + 2;
    if ((size_t)n_full * LUT_ROW + LUT_WARPS * per_warp <= budget) { pl.kernel = 1; pl.n_lut = n_full; }
    else if ((size_t)n_clamped * LUT_ROW + LUT_WARPS * per_warp <= budget) { pl.kernel = 2; pl.n_lut = n_clamped; }
    if (pl.kernel) pl.smem = (size_t)pl.n_lut * LUT_ROW + LUT_WARPS * per_warp;
  }
  if (!pl.kernel && pl.expo == 4 && pl.posw) pl.neg_c *= 0.5f;   // SQRTW: the decay of sqrt(weight)
  return pl;
}

// The table kernel's rows r2 = 0 .. n_lut - 1: {E', ninv'} in the scales of its records (LUT_*).
static void upload_table(visfd_ctx *ctx, const GatherPlan &pl, float sigma, Scratch<float2> &lut) {
  std::vector<float2> h(pl.n_lut);
  for (int r2 = 0; r2 < pl.n_lut; r2++) {
    const float e = ((float)r2 < pl.lim_in) ? (float)exp(-0.5 * (double)r2 / ((double)sigma * (double)sigma)) : 0.0f;
    // powers of two: exact
    h[r2] = make_float2(ldexpf(e, LUT_E_LOG2), r2 ? ldexpf((float)(-1.0 / (double)r2), LUT_TAU_LOG2) : 0.0f);
  }
  if (pl.kernel == 2) h[pl.n_lut - 1] = make_float2(0.0f, 0.0f);
  lut.reset(ctx, h.size());
  VCK(cudaMemcpyAsync(lut.get(), h.data(), h.size() * sizeof(float2), cudaMemcpyHostToDevice, ctx->stream));
  VCK(cudaStreamSynchronize(ctx->stream));   // h goes out of scope
}

typedef void (*GatherKernel)(GatherArgs);
template <int E, bool C>
static GatherKernel mufu_kernel(const GatherPlan &pl) {
  if (pl.shell) return tv_gather_kernel<E, C, false, true>;
  return pl.posw ? tv_gather_kernel<E, C, true, false> : tv_gather_kernel<E, C, false, false>;
}
template <bool C>
static GatherKernel gather_kernel(const GatherPlan &pl) {
  if (pl.kernel) return pl.kernel == 2 ? tv_gather_lut_kernel<C, true> : tv_gather_lut_kernel<C, false>;
  return pl.expo == 2 ? mufu_kernel<2, C>(pl) : pl.expo == 4 ? mufu_kernel<4, C>(pl) : mufu_kernel<0, C>(pl);
}

// One launch over the 8x8x4 receiver tiles of g: one 4-warp CTA per tile in tv_gather_kernel; the persistent table
// kernel takes them from g.ticket.
static void launch_gather(visfd_ctx *ctx, const GatherPlan &pl, const GatherArgs &g, unsigned tiles) {
  const GatherKernel k = pl.curves ? gather_kernel<true>(pl) : gather_kernel<false>(pl);
  const unsigned ctas = pl.kernel ? (unsigned)std::min<i64>(ctx->sm_count, ((i64)tiles + LUT_QUADS - 1) / LUT_QUADS) : tiles;
  VCK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
  k<<<ctas, pl.kernel ? 32 * LUT_WARPS : TV_THREADS, pl.smem, ctx->stream>>>(g);
  VCK(cudaGetLastError());
  ctx->count_launch();
}

// The pool blocks of tv_device below, each at its largest.
size_t tv_workspace_bytes(i64 nx, i64 ny, i64 nz_local, i64 own_planes, uint64_t n_voters) {
  static_assert(sizeof(VoterRec) == 48, "voter record size");
  const size_t n_bricks = (size_t)div_up(nx, VBR) * (size_t)div_up(ny, VBR) * (size_t)div_up(nz_local, VBR);
  const size_t n_scan_blocks = (n_bricks + SCAN_B - 1) / SCAN_B;
  const size_t max_lut = 3 * (LUT_MAX_HW + 3) * (LUT_MAX_HW + 3) + 1;   // plan_gather's r2_reach + 1 at most
  auto b = visfd_ctx::block_bytes;
  return b(n_bricks * 4) + b((n_bricks + 1) * 4) + b((n_scan_blocks + 2) * 4) +   // counts, off, sums
         b(std::max<uint64_t>(n_voters, 1) * sizeof(VoterRec)) + b(TV_MAX_SHELL * 4) +   // rec, shell
         b(max_lut * sizeof(float2)) + b(std::max<size_t>(div_up(own_planes, BR), 1) * 4);   // lut, tickets
}

bool tv_device(visfd_ctx *ctx, i64 nx, i64 ny, i64 nz_local, i64 z_offset, i64 nz_global,
               i64 own_z0, i64 own_z1, const float *saliency, float thr, const float *direction,
               const float *smoothed, float ridge_sigma, int eival_order, int score_kind,
               const float *mask_src, const float *mask_dst, const TVParams &p, float *tensor,
               float *score, float *score_host, const float *peak) {
  VREQUIRE(nx > 0 && ny > 0 && nz_local > 0, "empty volume");
  VREQUIRE(!peak || score, "the peak height scales the score: score must be given");
  VREQUIRE(own_z0 >= 0 && own_z1 <= nz_local && own_z0 <= own_z1, "receiver planes outside the slab");
  VREQUIRE(p.sigma > 0.0f, "tensor-voting sigma must be positive");
  VREQUIRE(p.exponent >= 1, "tensor-voting angle exponent must be >= 1");
  VREQUIRE(direction || smoothed, "tensor voting needs voter directions");
  const int hw = tv_halfwidth(p.sigma, p.cutoff_ratio);
  VREQUIRE(hw >= 0 && hw <= TV_MAX_REACH * BR, "tensor-voting radius too large (max 56 voxels)");
  VREQUIRE(nx <= (1 << 23) && ny <= (1 << 23) && nz_local <= (1 << 23), "slab too large");
  if (own_z1 == own_z0) return false;
  DecayInfo info = decay_info(p.sigma, hw);
  VREQUIRE((int)info.shell_keep.size() <= TV_MAX_SHELL, "too many lattice points on the support shell");

  const int nbx = (int)div_up(nx, BR), nby = (int)div_up(ny, BR);   // 8x8 receiver tiles per layer
  const int vbx = (int)div_up(nx, VBR), vby = (int)div_up(ny, VBR), vbz = (int)div_up(nz_local, VBR);
  VREQUIRE((i64)vbx * vby * vbz < 2147483647LL, "too many bricks for one launch");
  VREQUIRE(vby <= 65535 && vbz <= 65535, "slab too large for the voter list kernels");
  int smem_optin = 0;
  VCK(cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, ctx->device));
  Scratch<uint32_t> off;
  Scratch<VoterRec> rec;
  uint32_t n_voters = 0;
  GatherPlan pl;
  {
    StageTimer t(ctx, "compact");
    bool nonpos = false;
    n_voters = build_voter_list(ctx, VoterSrc{saliency, mask_src, thr, (int)nx, (int)ny, nz_local, vbx, vby, vbz},
                                1.0f / info.total, off, rec, nonpos);
    pl = plan_gather(p, hw, info, n_voters, nonpos, smem_optin);
    if (n_voters > 0) {   // the direction pass
      DirSrc ds{direction, smoothed, ridge_sigma, eival_order, z_offset, nz_global};
      voter_direction_kernel<<<div_up(n_voters, 256), 256, 0, ctx->stream>>>(ds, (int)nx, (int)ny, n_voters,
                                                                            pl.kernel != 0, rec.get());
      VCK(cudaGetLastError());
      ctx->count_launch();
    }
  }
  ctx->last_voters = n_voters;
  ctx->last_tv_kernel = pl.kernel;

  Scratch<uint32_t> shell(ctx, std::max<size_t>(info.shell_keep.size(), 1));
  if (!info.shell_keep.empty())
    VCK(cudaMemcpyAsync(shell.get(), info.shell_keep.data(), info.shell_keep.size() * sizeof(uint32_t),
                        cudaMemcpyHostToDevice, ctx->stream));

  GatherArgs g;
  g.rec = rec.get(); g.off = off.get();
  g.shell = shell.get(); g.n_shell = (int)info.shell_keep.size();
  g.nx = (int)nx; g.ny = (int)ny; g.nz = nz_local;
  g.nbx = vbx; g.nby = vby; g.nbz = vbz;   // the voter bricks
  g.own_z0 = own_z0; g.own_z1 = own_z1;
  g.ntx = nbx; g.nty = nby;
  g.hw = hw; g.hw2 = (float)(hw * hw);
  g.row_cap = pl.row_cap;
  g.lim_in = pl.lim_in; g.lim_pass = pl.lim_pass;
  g.neg_c = pl.neg_c;
  g.half_exp = 0.5f * (float)p.exponent;
  g.mask_dst = mask_dst; g.tensor = tensor; g.score = score;
  g.order = eival_order; g.score_kind = score_kind;
  g.lut = nullptr; g.n_lut = pl.n_lut; g.n_tiles = 0; g.ticket = nullptr;
  // receiver planes in chunks (multiples of the 8-plane tile): one launch each, so that a
  // finished chunk of the result can travel to the host while the next one is computed
  const i64 planes = own_z1 - own_z0;
  const bool overlap_d2h = score_host && score && planes >= 8 * BR;
  // up to 16 chunks: only the last one's copy (1/16 of the result) is not hidden behind a kernel;
  // but every chunk keeps >= 64 waves of CTAs, or the tails of the launches cost more than the copy
  // (VISFD_CUDA_CHUNK_WAVES overrides the 64, for tests that want many small chunks)
  const char *waves_env = getenv("VISFD_CUDA_CHUNK_WAVES");
  const i64 waves = waves_env ? std::max(0, atoi(waves_env)) : 64;
  const i64 tiles_per_layer = (i64)div_up(nx, BR) * div_up(ny, BR);
  const i64 min_chunk = (TV_TILE_Z * ((waves * 4 * (i64)ctx->sm_count + tiles_per_layer - 1) / tiles_per_layer) + BR - 1) / BR * BR;
  const i64 chunk_planes = overlap_d2h ? std::max(((planes + 15) / 16 + BR - 1) / BR * BR, min_chunk) : planes;
  const int n_chunks = (int)((planes + chunk_planes - 1) / chunk_planes);
  VREQUIRE((i64)g.ntx * g.nty * div_up(chunk_planes, TV_TILE_Z) * 4 / TV_WARPS < 2147483647LL,
           "too many receiver tiles for one launch");
  // score planes [z0, z1) of the slab *= their peak height, where mask_dst != 0
  auto scale_own_planes = [&](i64 z0, i64 z1, float *s) {
    const size_t o = (size_t)z0 * (size_t)nx * (size_t)ny;
    scale_by_peak_device(ctx, (i64)((size_t)(z1 - z0) * (size_t)nx * (size_t)ny), s, peak + o, nullptr,
                         mask_dst ? mask_dst + o : nullptr);
  };
  EventList chunk_events(ctx);
  std::vector<cudaEvent_t> &chunk_done = chunk_events.ev;
  Scratch<float2> lut;
  Scratch<unsigned> tickets;
  if (pl.kernel) {
    upload_table(ctx, pl, p.sigma, lut);
    g.lut = lut.get();
    tickets.reset(ctx, (size_t)n_chunks);
    VCK(cudaMemsetAsync(tickets.get(), 0, (size_t)n_chunks * sizeof(unsigned), ctx->stream));
  }
  {
    StageTimer t(ctx, "tv");
    for (int c = 0; c < n_chunks; c++) {
      GatherArgs gc = g;
      gc.own_z0 = g.own_z0 + c * chunk_planes;
      gc.own_z1 = std::min(g.own_z1, gc.own_z0 + chunk_planes);
      const size_t chunk_off = (size_t)(gc.own_z0 - g.own_z0) * (size_t)nx * (size_t)ny;
      if (g.score) gc.score = g.score + chunk_off;
      if (g.tensor) gc.tensor = g.tensor + 6 * chunk_off;
      const unsigned grid = (unsigned)((i64)gc.ntx * gc.nty * div_up(gc.own_z1 - gc.own_z0, TV_TILE_Z) * 4 / TV_WARPS);
      if (pl.kernel) {
        gc.n_tiles = grid;   // one 4-warp tile per CTA of the MUFU kernel
        gc.ticket = tickets.get() + c;
      }
      launch_gather(ctx, pl, gc, grid);
      if (overlap_d2h) {
        if (peak) scale_own_planes(gc.own_z0, gc.own_z1, gc.score);   // before the chunk's copy is queued
        VCK(cudaEventRecord(chunk_events.add(), ctx->stream));
      }
    }
  }
  if (peak && !overlap_d2h) scale_own_planes(own_z0, own_z1, score);
  if (overlap_d2h) {
    // all launches are queued; now the copies, each behind its chunk (with pageable host memory
    // cudaMemcpyAsync blocks the host, which no longer delays any launch)
    if (!ctx->copy_stream) VCK(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    const size_t plane = (size_t)nx * (size_t)ny;
    for (int c = 0; c < n_chunks; c++) {
      const size_t off = (size_t)c * (size_t)chunk_planes * plane;
      const size_t cnt = (size_t)std::min(chunk_planes, planes - c * chunk_planes) * plane;
      VCK(cudaStreamWaitEvent(ctx->copy_stream, chunk_done[c], 0));
      VCK(cudaMemcpyAsync(score_host + off, g.score + off, cnt * sizeof(float), cudaMemcpyDeviceToHost,
                          ctx->copy_stream));
    }
    VCK(cudaStreamSynchronize(ctx->copy_stream));
  }
  // the Scratch buffers are returned to the pool on scope exit; the pool is
  // stream-ordered, so the kernels above keep exclusive use until they finish.
  VCK(cudaStreamSynchronize(ctx->stream));
  return overlap_d2h;
}

}  // namespace visfd_cuda
