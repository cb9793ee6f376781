// gauss.cu -- separable 3-D filtering (ApplySeparable / ApplyGauss / ApplyDog / ApplyLog)
// as three streaming sweeps Z -> Y -> X, the order of lib/visfd/filter3d.hpp:741-981.
//
// Data layout: dense float32 [nz][ny][nx], x fastest.  Every sweep reads 4 B and
// writes 4 B per voxel (24 B/voxel per Gaussian); the un-masked normalisation
// (filter3d.hpp:1004-1022) and the DoG / LoG combine (filter3d.hpp:1387-1390,
// :1493-1498) are fused into the X sweep's epilogue, so they cost no extra pass.
//
// Kernels
//  sweep_axis3_kernel : Y or Z sweep, the default.  A CTA owns 128 columns x 96 outputs along the axis in 3 chunks;
//      the whole tile is requested up front by TMA (cp.async.bulk.tensor boxes of 8 rows, zero-filled outside the
//      volume, one mbarrier per chunk); tap-stationary compute: a thread keeps a window of 8 input rows in registers
//      and produces 4 outputs x float4 with every tap useful.
//  sweep_x2_kernel    : X sweep, the default.  64 rows x (128 + 2 hw) columns by TMA in two chunks; first / last tap
//      steps specialised on hw mod 4; normalisation and DoG / LoG combine in the epilogue.
//  sweep_axis2_kernel / sweep_axis_kernel / sweep_x_kernel : fall-backs for ragged nx (no float4 / TMA alignment),
//      very wide filters, and masks (sweep_axis_kernel<EXACT_MASKED>: (h*m)*f per tap from two shared-memory tiles).
// Out-of-volume taps are zero (the reference skips them, filter1d.hpp:98-99); the
// renormalisation divides by the product of the three 1-D edge profiles.
//
// Arithmetic modes (template parameter MODE of both kernels):
//  EXACT (default)  every tap is a separate IEEE multiply and add, accumulated in the
//      reference's order (filter index j ascending = input index descending,
//      filter1d.hpp:96-101), so the output is BIT-IDENTICAL to the reference's
//      x86-64 (non-FMA) build.  Zero-padded taps / rows add +-0 and change nothing.
//      This is what makes DoG/LoG (a 2500x amplified difference of two Gaussians), the
//      blob extremum tests and the ridge saliency (4th power of second differences)
//      reproducible rather than "close".
//  EXACT_MASKED  Z sweep with a mask: (h*m)*f per tap as in filter1d.hpp:273-286, from
//      two shared-memory tiles.
//  FAST  one FFMA per tap (and mask pre-multiplied while staging): half the FP32
//      instructions, ~1e-7 absolute / 1e-5 relative differences from the reference.
//      Selected per context (visfd_cuda_set_fast_gauss / VISFD_CUDA_FAST_GAUSS=1).
#include "common.cuh"
#include "kernels.cuh"
#include <cuda.h>
#include <cudaTypedefs.h>
#include <cmath>
#include <algorithm>

namespace visfd_cuda {

// ---------------------------------------------------------------------------------
// TMA (cp.async.bulk.tensor): the sweeps' shared-memory tiles are boxes of a 2-D / 3-D
// tensor map over the volume; one thread issues the copies, the hardware zero-fills
// everything outside the volume, and an mbarrier per chunk tells the CTA when it landed.
// ---------------------------------------------------------------------------------
static PFN_cuTensorMapEncodeTiled tensor_map_encoder() {
  // resolved once; the initialisation of a function-local static is thread-safe (several host threads filter at once)
  static const PFN_cuTensorMapEncodeTiled fn = [] {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      return reinterpret_cast<PFN_cuTensorMapEncodeTiled>(p);
    cudaGetLastError();
    return PFN_cuTensorMapEncodeTiled(nullptr);
  }();
  return fn;
}

// float32 tensor of `rank` dims (x fastest), dense; box = tile extents.  false if TMA
// cannot describe it (alignment, size) -- the caller falls back to cp.async staging.
static bool make_tensor_map(CUtensorMap *map, const float *ptr, int rank, const i64 *dims, const int *box) {
  PFN_cuTensorMapEncodeTiled enc = tensor_map_encoder();
  if (!enc || ((uintptr_t)ptr & 15) != 0) return false;
  cuuint64_t gdim[3], gstride[2];
  cuuint32_t bdim[3], estr[3] = {1, 1, 1};
  i64 stride = sizeof(float);
  for (int d = 0; d < rank; d++) {
    if (dims[d] <= 0 || dims[d] > 0xffffffffLL || box[d] <= 0 || box[d] > 256) return false;
    gdim[d] = (cuuint64_t)dims[d];
    bdim[d] = (cuuint32_t)box[d];
    stride *= dims[d];
    if (d + 1 < rank) {
      if (stride % 16 != 0 || stride >= (1LL << 40)) return false;
      gstride[d] = (cuuint64_t)stride;
    }
  }
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, (cuuint32_t)rank, const_cast<float *>(ptr), gdim, gstride,
                   bdim, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned parity) {
  unsigned done;
  do {
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                 : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  } while (!done);
}
__device__ __forceinline__ void tma_load_3d(void *dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
               ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
               ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}

// ---------------------------------------------------------------------------------
// host: taps
// ---------------------------------------------------------------------------------
// GenFilterGauss1D<float>: lib/visfd/filter1d.hpp:411-460.  Discrete Gaussian kernel
// exp(-s^2) I_|i|(s^2) for s<=10 and |i|<=20, sampled continuous Gaussian otherwise,
// in long double; stored as float; normalised by the long double sum of the floats.
void gen_gauss1d(float sigma, int hw, float *taps) {
  long double sum = 0.0L;
  for (int i = -hw; i <= hw; i++) {
    float v;
    if (sigma == 0.0f) {
      v = (i == 0) ? 1.0f : 0.0f;
    } else {
      long double S = sigma, I = i;
      if ((S <= 10.0) && (fabsl(I) <= 20.0))
        v = (float)(expl(-S * S) * std::cyl_bessel_i(fabsl(I), S * S));
      else
        v = (float)(expl(-(I * I) / (2.0 * S * S)) / sqrtl(2 * S * S * M_PI));
    }
    taps[i + hw] = v;
    sum += v;
  }
  for (int i = 0; i < 2 * hw + 1; i++) taps[i] = (float)(taps[i] / sum);
}

// Response of the filter to an all-ones line of length n, float, j ascending
// (lib/visfd/filter3d.hpp:1005-1011 via filter1d.hpp:96-101): the edge profile the
// un-masked normalisation divides by.
static void edge_profile(const float *taps, int hw, i64 n, i64 first, i64 count,
                         float *d) {
  for (i64 t = 0; t < count; t++) {
    i64 i = first + t;
    float acc = 0.0f;
    for (int j = -hw; j <= hw; j++) {
      i64 k = i - j;
      if (k < 0 || k >= n) continue;
      acc += taps[j + hw] * 1.0f;
    }
    d[t] = acc;
  }
}

// ---------------------------------------------------------------------------------
// device kernels
// ---------------------------------------------------------------------------------
constexpr int AX_R = 8;        // outputs per thread along the sweep axis
constexpr int AX_WARPS = 8;    // warps per CTA
constexpr int AX_TA = AX_R * AX_WARPS;  // 64 outputs along the axis per CTA
constexpr int AX_TX = 128;     // columns per CTA (32 lanes x float4)
constexpr int TAP_PAD_LO = 16; // zero padding below/above the taps in shared memory
constexpr int TAP_PAD_HI = 8;

__device__ __forceinline__ float4 ld4(const float *p) {
  return __ldg(reinterpret_cast<const float4 *>(p));
}

enum { MODE_FAST = 0, MODE_EXACT = 1, MODE_EXACT_MASKED = 2 };

template <int MODE>
__device__ __forceinline__ float tap_acc(float acc, float h, float v) {
  if (MODE == MODE_FAST) return fmaf(h, v, acc);
  return __fadd_rn(acc, __fmul_rn(h, v));
}

// Packed FP32 (FMUL2 / FADD2 / FFMA2, each lane-wise IEEE round-to-nearest like the scalar
// forms, so EXACT stays bit-exact): half the issue slots for the same arithmetic.
// (ptxas 12.9 contracts mul.rn.f32x2 + add.rn.f32x2 into one FFMA2 -- unlike the scalar .rn
// forms, and whatever -fmad says -- so EXACT cannot write the sum as a packed add; see
// mul_then_add2 for the form it uses: two instructions per two taps instead of four.)
__device__ __forceinline__ unsigned long long f2_bits(float2 v) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(v.x), "f"(v.y));
  return r;
}
__device__ __forceinline__ float2 bits_f2(unsigned long long b) {
  float2 v;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(v.x), "=f"(v.y) : "l"(b));
  return v;
}
// The sum: a packed FMA of the ROUNDED product with a multiplier of one -- fma(p, 1, acc) rounds p + acc once,
// which is the rounded addition.  The one comes from constant memory, so ptxas can neither fold it away nor
// contract anything: two issue slots per pair of taps (FMUL2 + FFMA2) instead of three (FMUL2 + 2 FADD).
__constant__ float c_one = 1.0f;
__device__ __forceinline__ float2 mul_then_add2(float2 acc, float2 a, float2 b) {
  unsigned long long p, r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(p) : "l"(f2_bits(a)), "l"(f2_bits(b)));
  const float one = c_one;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(p), "l"(f2_bits(make_float2(one, one))), "l"(f2_bits(acc)));
  return bits_f2(r);
}
template <int MODE>
__device__ __forceinline__ float2 tap_acc2(float2 acc, float h, float2 v) {
  if (MODE == MODE_FAST) return __ffma2_rn(v, make_float2(h, h), acc);
  return mul_then_add2(acc, make_float2(h, h), v);
}
template <int MODE>
__device__ __forceinline__ float2 tap_acc2(float2 acc, float2 h, float v) {
  if (MODE == MODE_FAST) return __ffma2_rn(h, make_float2(v, v), acc);
  return mul_then_add2(acc, h, make_float2(v, v));
}

// in/out: volumes; the sweep axis has n_axis entries with stride s_axis (floats);
// the third ("other") dimension has stride s_other and is indexed by blockIdx.z.
// mask (optional): FAST: multiplied into the input while staging; EXACT_MASKED: staged
// in a second tile and multiplied into the TAP first, as the reference does.
template <int MODE>
__global__ void __launch_bounds__(32 * AX_WARPS)
sweep_axis_kernel(const float *__restrict__ in, float *__restrict__ out,
                  const float *__restrict__ mask, const float *__restrict__ taps,
                  int hw, int nx, i64 n_axis, i64 s_axis, i64 s_other, int vec_ok) {
  extern __shared__ __align__(128) float smem[];
  const int rows = AX_TA + 2 * hw + 8;          // staged rows (+8 zero rows for the unrolled tail)
  float *tile = smem;                           // [rows][AX_TX]
  float *mtile = smem + (size_t)rows * AX_TX;   // [rows][AX_TX], EXACT_MASKED only
  float *tp = smem + (size_t)rows * AX_TX * (MODE == MODE_EXACT_MASKED ? 2 : 1);  // padded taps
  const int lane = threadIdx.x, wy = threadIdx.y;
  const int tid = wy * 32 + lane;
  const int x0 = blockIdx.x * AX_TX;
  const i64 a0 = (i64)blockIdx.y * AX_TA;
  const i64 base = (i64)blockIdx.z * s_other;

  const int ntap = 2 * hw + 1;
  for (int k = tid; k < ntap + TAP_PAD_LO + TAP_PAD_HI; k += 32 * AX_WARPS) {
    int t = k - TAP_PAD_LO;
    tp[k] = (t >= 0 && t < ntap) ? taps[t] : 0.0f;
  }
  // stage rows a0-hw .. a0-hw+rows-1 (zero outside the volume / beyond 2hw+TA)
  const int xl = x0 + 4 * lane;
  for (int r = wy; r < rows; r += AX_WARPS) {
    i64 a = a0 - hw + r;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f), m = make_float4(0.f, 0.f, 0.f, 0.f);
    if (a >= 0 && a < n_axis && r < AX_TA + 2 * hw) {
      const float *p = in + base + a * s_axis + xl;
      const float *pm = mask ? mask + base + a * s_axis + xl : nullptr;
      if (vec_ok && xl + 3 < nx) {
        v = ld4(p);
        if (pm) m = ld4(pm);
      } else {
        if (xl + 0 < nx) { v.x = __ldg(p + 0); if (pm) m.x = __ldg(pm + 0); }
        if (xl + 1 < nx) { v.y = __ldg(p + 1); if (pm) m.y = __ldg(pm + 1); }
        if (xl + 2 < nx) { v.z = __ldg(p + 2); if (pm) m.z = __ldg(pm + 2); }
        if (xl + 3 < nx) { v.w = __ldg(p + 3); if (pm) m.w = __ldg(pm + 3); }
      }
      if (MODE == MODE_FAST && pm) { v.x *= m.x; v.y *= m.y; v.z *= m.z; v.w *= m.w; }
    }
    *reinterpret_cast<float4 *>(tile + (size_t)r * AX_TX + 4 * lane) = v;
    if (MODE == MODE_EXACT_MASKED) *reinterpret_cast<float4 *>(mtile + (size_t)r * AX_TX + 4 * lane) = m;
  }
  __syncthreads();

  float4 acc[AX_R];
#pragma unroll
  for (int r = 0; r < AX_R; r++) acc[r] = make_float4(0.f, 0.f, 0.f, 0.f);
  const int ob = AX_R * wy;
  const float *trow = tile + (size_t)ob * AX_TX + 4 * lane;
  const float *mrow = mtile + (size_t)ob * AX_TX + 4 * lane;
  // output o=ob+r (axis position a0+o) takes input row p=ob+q with tap index
  // 2hw + r - q;  q runs over [0, 2hw+7] in blocks of 8, from the HIGHEST input index
  // down: that is the reference's accumulation order (tap index ascending).
  const int nblk = (2 * hw + AX_R + 7) / 8;
  for (int q0 = 8 * (nblk - 1); q0 >= 0; q0 -= 8) {
    float t[15];
    const float *tb = tp + TAP_PAD_LO + (2 * hw - q0) - 7;
#pragma unroll
    for (int d = 0; d < 15; d++) t[d] = tb[d];
#pragma unroll
    for (int u = 7; u >= 0; u--) {
      float4 v = *reinterpret_cast<const float4 *>(trow + (size_t)(q0 + u) * AX_TX);
      float4 m = make_float4(1.f, 1.f, 1.f, 1.f);
      if (MODE == MODE_EXACT_MASKED) m = *reinterpret_cast<const float4 *>(mrow + (size_t)(q0 + u) * AX_TX);
#pragma unroll
      for (int r = 0; r < AX_R; r++) {
        float h = t[r - u + 7];
        if (MODE == MODE_EXACT_MASKED) {
          // filter1d.hpp:273-286: filter_val = h*mask; delta = filter_val*f; g += delta
          acc[r].x = __fadd_rn(acc[r].x, __fmul_rn(__fmul_rn(h, m.x), v.x));
          acc[r].y = __fadd_rn(acc[r].y, __fmul_rn(__fmul_rn(h, m.y), v.y));
          acc[r].z = __fadd_rn(acc[r].z, __fmul_rn(__fmul_rn(h, m.z), v.z));
          acc[r].w = __fadd_rn(acc[r].w, __fmul_rn(__fmul_rn(h, m.w), v.w));
        } else {
          acc[r].x = tap_acc<MODE>(acc[r].x, h, v.x);
          acc[r].y = tap_acc<MODE>(acc[r].y, h, v.y);
          acc[r].z = tap_acc<MODE>(acc[r].z, h, v.z);
          acc[r].w = tap_acc<MODE>(acc[r].w, h, v.w);
        }
      }
    }
  }
#pragma unroll
  for (int r = 0; r < AX_R; r++) {
    i64 a = a0 + ob + r;
    if (a >= n_axis) break;
    float *p = out + base + a * s_axis + xl;
    if (vec_ok && xl + 3 < nx) {
      *reinterpret_cast<float4 *>(p) = acc[r];
    } else {
      if (xl + 0 < nx) p[0] = acc[r].x;
      if (xl + 1 < nx) p[1] = acc[r].y;
      if (xl + 2 < nx) p[2] = acc[r].z;
      if (xl + 3 < nx) p[3] = acc[r].w;
    }
  }
}

// ---- un-masked Y / Z sweep, tap-stationary --------------------------------------------
// CTA = 8 warps x 32 lanes: 128 columns (float4 per lane) x 32 outputs along the axis,
// warp w owns outputs 4w..4w+3.  The CTA stages the ntap8 + 31 input rows it needs once
// (ntap8 = taps rounded up to a multiple of 8, zero taps at the end).  A thread keeps a
// window of 8 input rows in registers, indexed by k mod 8 where row k is input position
// a0 + hw - k: output r takes tap t from row k = t - r, so one group of 4 taps needs
// rows 4g-3 .. 4g+3 -- 4 new rows per group, 16 useful mul+add per float4 column, and all
// register indices static after unrolling two groups.  Taps are visited in ascending order
// for every output: the reference's accumulation order (filter1d.hpp:96-101).
constexpr int A2_S = 32;   // outputs along the axis per CTA
constexpr int A2_R = 4;    // outputs per thread

template <int MODE>
__global__ void __launch_bounds__(256, 4)
sweep_axis2_kernel(const float *__restrict__ in, float *__restrict__ out,
                   const float *__restrict__ taps, int hw, int ntap8, int nx, i64 n_axis,
                   i64 s_axis, i64 s_other, int vec_ok) {
  extern __shared__ __align__(128) float smem[];
  const int rows = ntap8 + A2_S - 1;
  float *tile = smem;                          // [rows][AX_TX]
  float *tp = smem + (size_t)rows * AX_TX;     // [ntap8]
  const int lane = threadIdx.x, wy = threadIdx.y;
  const int tid = wy * 32 + lane;
  const int x0 = blockIdx.x * AX_TX;
  const i64 A0 = (i64)blockIdx.y * A2_S;
  const i64 base = (i64)blockIdx.z * s_other;
  const int ntap = 2 * hw + 1;
  for (int k = tid; k < ntap8; k += 256) tp[k] = (k < ntap) ? taps[k] : 0.0f;
  // tile row rho holds input position lo + rho
  const i64 lo = A0 + hw - ntap8 + 1;
  const int xl = x0 + 4 * lane;
  for (int r = wy; r < rows; r += 8) {
    const i64 a = lo + r;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (a >= 0 && a < n_axis) {
      const float *p = in + base + a * s_axis + xl;
      if (vec_ok && xl + 3 < nx) {
        v = ld4(p);
      } else {
        if (xl + 0 < nx) v.x = __ldg(p + 0);
        if (xl + 1 < nx) v.y = __ldg(p + 1);
        if (xl + 2 < nx) v.z = __ldg(p + 2);
        if (xl + 3 < nx) v.w = __ldg(p + 3);
      }
    }
    *reinterpret_cast<float4 *>(tile + (size_t)r * AX_TX + 4 * lane) = v;
  }
  __syncthreads();

  float4 acc[A2_R];
#pragma unroll
  for (int r = 0; r < A2_R; r++) acc[r] = make_float4(0.f, 0.f, 0.f, 0.f);
  // row k of this warp = tile row A2_R*wy + ntap8 - 1 - k
  const float *row0 = tile + (size_t)(A2_R * wy + ntap8 - 1) * AX_TX + 4 * lane;
#define ROW(k) (*reinterpret_cast<const float4 *>(row0 - (ptrdiff_t)(k) * AX_TX))
  float4 win[8];
  win[5] = ROW(-3);
  win[6] = ROW(-2);
  win[7] = ROW(-1);
#define TAP4(h, tt, base_idx)                                                     \
  _Pragma("unroll") for (int r = 0; r < A2_R; r++) {                              \
    const float4 v = win[((base_idx) + (tt) - r) & 7];                            \
    acc[r].x = tap_acc<MODE>(acc[r].x, h, v.x);                                   \
    acc[r].y = tap_acc<MODE>(acc[r].y, h, v.y);                                   \
    acc[r].z = tap_acc<MODE>(acc[r].z, h, v.z);                                   \
    acc[r].w = tap_acc<MODE>(acc[r].w, h, v.w);                                   \
  }
  for (int k0 = 0; k0 < ntap8; k0 += 8) {
    const float4 ha = *reinterpret_cast<const float4 *>(tp + k0);
    const float4 hb = *reinterpret_cast<const float4 *>(tp + k0 + 4);
    win[0] = ROW(k0 + 0);
    win[1] = ROW(k0 + 1);
    win[2] = ROW(k0 + 2);
    win[3] = ROW(k0 + 3);
    TAP4(ha.x, 0, 0) TAP4(ha.y, 1, 0) TAP4(ha.z, 2, 0) TAP4(ha.w, 3, 0)
    win[4] = ROW(k0 + 4);
    win[5] = ROW(k0 + 5);
    win[6] = ROW(k0 + 6);
    win[7] = ROW(k0 + 7);
    TAP4(hb.x, 0, 4) TAP4(hb.y, 1, 4) TAP4(hb.z, 2, 4) TAP4(hb.w, 3, 4)
  }
#undef TAP4
#undef ROW
#pragma unroll
  for (int r = 0; r < A2_R; r++) {
    const i64 a = A0 + A2_R * wy + r;
    if (a >= n_axis) break;
    float *p = out + base + a * s_axis + xl;
    if (vec_ok && xl + 3 < nx) {
      *reinterpret_cast<float4 *>(p) = acc[r];
    } else {
      if (xl + 0 < nx) p[0] = acc[r].x;
      if (xl + 1 < nx) p[1] = acc[r].y;
      if (xl + 2 < nx) p[2] = acc[r].z;
      if (xl + 3 < nx) p[3] = acc[r].w;
    }
  }
}

// ---- the same with the loads pipelined (cp.async) ------------------------------------------
// One CTA covers A3_NCH chunks of 32 outputs along the axis.  All rows of the tile are
// requested up front with cp.async (LDGSTS, zero-fill outside the volume), one commit
// group per chunk, so a CTA has its whole tile (tens of KB) in flight while it computes
// the chunks that have already landed; with 3 CTAs per SM that is > 100 KB of loads in
// flight per SM, enough to cover the DRAM latency at full bandwidth.  Needs float4-aligned
// rows (nx % 4 == 0); sweep_axis2_kernel handles the ragged case.
constexpr int A3_NCH = 3;

__device__ __forceinline__ void cp_async16_zfill(void *smem, const void *gmem, bool valid) {
  unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
  int sz = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(sa), "l"(gmem), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_commit_group() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

// TMA = true: the tile is fetched by cp.async.bulk.tensor boxes of 8 rows x 128 columns of
// the 3-D tensor map `tmap` (axis_dim = 1: Y sweep, 2: Z sweep), issued by one thread and
// tracked by one mbarrier per chunk; TMA = false: per-thread cp.async as described above.
// DUAL = true: two filters of the same (zero-padded) length over ONE staged tile -- the pair of Gaussians of a
// DoG / LoG reads the source once: taps_b -> out_b next to taps -> out.
template <int MODE, bool TMA, bool DUAL>
__global__ void __launch_bounds__(256, 3)
sweep_axis3_kernel(const __grid_constant__ CUtensorMap tmap, int axis_dim,
                   const float *__restrict__ in, float *__restrict__ out, float *__restrict__ out_b,
                   const float *__restrict__ taps, const float *__restrict__ taps_b, int hw, int ntap8, int nx,
                   i64 n_axis, i64 s_axis, i64 s_other) {
  extern __shared__ __align__(128) float smem[];
  const int rows = ntap8 + A3_NCH * A2_S;      // multiple of 8
  float *tile = smem;                          // [rows][AX_TX]
  float *tp = smem + (size_t)rows * AX_TX;     // [ntap8] (x 2 if DUAL)
  uint64_t *bars = reinterpret_cast<uint64_t *>(tp + (DUAL ? 2 : 1) * ntap8);   // [A3_NCH], TMA only
  const int lane = threadIdx.x, wy = threadIdx.y;
  const int tid = wy * 32 + lane;
  const int xl = blockIdx.x * AX_TX + 4 * lane;
  const i64 A0 = (i64)blockIdx.y * (A3_NCH * A2_S);
  const i64 base = (i64)blockIdx.z * s_other;
  const i64 lo = A0 + hw - ntap8;              // tile row rho holds input position lo + rho
  const bool xin = xl < nx;
  if (TMA) {
    if (tid == 0) {
#pragma unroll
      for (int c = 0; c < A3_NCH; c++) mbar_init(bars + c, 1);
      mbar_init_fence();
#pragma unroll
      for (int c = 0; c < A3_NCH; c++) {
        if (A0 + A2_S * c >= n_axis) break;
        const int r_begin = c == 0 ? 0 : ntap8 + A2_S * c, r_end = ntap8 + A2_S * (c + 1);
        mbar_expect_tx(bars + c, (unsigned)(r_end - r_begin) * AX_TX * sizeof(float));
        for (int r = r_begin; r < r_end; r += 8) {
          const int a = (int)(lo + r), o = (int)blockIdx.z;
          tma_load_3d(tile + (size_t)r * AX_TX, &tmap, bars + c, blockIdx.x * AX_TX, axis_dim == 1 ? a : o,
                      axis_dim == 1 ? o : a);
        }
      }
    }
  }
  // every thread copies its 16-byte column of rows wy, wy+8, ...: one pointer increment per copy
  const float *colbase = in + base + xl;
#pragma unroll
  for (int c = 0; c < A3_NCH; c++) {
    if (TMA) break;
    const int r_begin = c == 0 ? 0 : ntap8 + A2_S * c, r_end = ntap8 + A2_S * (c + 1);
    if (A0 + A2_S * c < n_axis) {
      i64 a = lo + r_begin + wy;
      const float *src = colbase + a * s_axis;
      float *dst = tile + (size_t)(r_begin + wy) * AX_TX + 4 * lane;
      for (int r = r_begin + wy; r < r_end; r += 8) {
        const bool ok = xin && a >= 0 && a < n_axis;
        cp_async16_zfill(dst, ok ? src : in, ok);
        a += 8;
        src += 8 * s_axis;
        dst += 8 * AX_TX;
      }
    }
    cp_async_commit_group();
  }
  if (tid < ntap8) {   // ntap8 <= 256 (checked by the host)
    tp[tid] = (tid < 2 * hw + 1) ? taps[tid] : 0.0f;
    if (DUAL) tp[ntap8 + tid] = (tid < 2 * hw + 1) ? taps_b[tid] : 0.0f;
  }
  if (TMA) __syncthreads();   // barriers initialised, taps staged

#pragma unroll 1
  for (int c = 0; c < A3_NCH; c++) {
    if (A0 + A2_S * c >= n_axis) break;   // uniform
    if (TMA) {
      mbar_wait(bars + c, 0);
    } else {
      if (c == 0) cp_async_wait_group<A3_NCH - 1>();
      else if (c == 1) cp_async_wait_group<A3_NCH - 2>();
      else cp_async_wait_group<0>();
      __syncthreads();
    }
#pragma unroll 1
    for (int f = 0; f < (DUAL ? 2 : 1); f++) {
    const float *tpf = tp + f * ntap8;
    float *outf = f ? out_b : out;
    float2 acc[A2_R][2];
#pragma unroll
    for (int r = 0; r < A2_R; r++) acc[r][0] = acc[r][1] = make_float2(0.f, 0.f);
    const float *row0 = tile + (size_t)(A2_S * c + A2_R * wy + ntap8) * AX_TX + 4 * lane;
#define ROW(k) (*reinterpret_cast<const float4 *>(row0 - (ptrdiff_t)(k) * AX_TX))
    float4 win[8];
    win[5] = ROW(-3);
    win[6] = ROW(-2);
    win[7] = ROW(-1);
#define TAP4(h, tt, base_idx)                                                     \
  _Pragma("unroll") for (int r = 0; r < A2_R; r++) {                              \
    const float4 v = win[((base_idx) + (tt) - r) & 7];                            \
    acc[r][0] = tap_acc2<MODE>(acc[r][0], h, make_float2(v.x, v.y));              \
    acc[r][1] = tap_acc2<MODE>(acc[r][1], h, make_float2(v.z, v.w));              \
  }
    const int ntap = 2 * hw + 1;
    int k0 = 0;
    for (; k0 + 8 <= ntap; k0 += 8) {
      const float4 ha = *reinterpret_cast<const float4 *>(tpf + k0);
      const float4 hb = *reinterpret_cast<const float4 *>(tpf + k0 + 4);
      win[0] = ROW(k0 + 0);
      win[1] = ROW(k0 + 1);
      win[2] = ROW(k0 + 2);
      win[3] = ROW(k0 + 3);
      TAP4(ha.x, 0, 0) TAP4(ha.y, 1, 0) TAP4(ha.z, 2, 0) TAP4(ha.w, 3, 0)
      win[4] = ROW(k0 + 4);
      win[5] = ROW(k0 + 5);
      win[6] = ROW(k0 + 6);
      win[7] = ROW(k0 + 7);
      TAP4(hb.x, 0, 4) TAP4(hb.y, 1, 4) TAP4(hb.z, 2, 4) TAP4(hb.w, 3, 4)
    }
    {
      // the last 1, 3, 5 or 7 taps (the count is odd): the taps that pad the group to 8 are zeros and add
      // nothing, so they are not evaluated (FP32-pipe time at sigma >= 4)
      const int rem = ntap - k0;
      const float4 ha = *reinterpret_cast<const float4 *>(tpf + k0);
      const float4 hb = *reinterpret_cast<const float4 *>(tpf + k0 + 4);
      win[0] = ROW(k0 + 0);
      TAP4(ha.x, 0, 0)
      if (rem >= 3) {
        win[1] = ROW(k0 + 1);
        win[2] = ROW(k0 + 2);
        TAP4(ha.y, 1, 0) TAP4(ha.z, 2, 0)
      }
      if (rem >= 5) {
        win[3] = ROW(k0 + 3);
        win[4] = ROW(k0 + 4);
        TAP4(ha.w, 3, 0) TAP4(hb.x, 0, 4)
      }
      if (rem >= 7) {
        win[5] = ROW(k0 + 5);
        win[6] = ROW(k0 + 6);
        TAP4(hb.y, 1, 4) TAP4(hb.z, 2, 4)
      }
    }
#undef TAP4
#undef ROW
    if (xin) {
#pragma unroll
      for (int r = 0; r < A2_R; r++) {
        const i64 a = A0 + A2_S * c + A2_R * wy + r;
        if (a < n_axis)
          *reinterpret_cast<float4 *>(outf + base + a * s_axis + xl) =
              make_float4(acc[r][0].x, acc[r][0].y, acc[r][1].x, acc[r][1].y);
      }
    }
    }
  }
}

constexpr int XS_ROWS = 32;  // rows per CTA (8 warps x 4 rows per thread)
constexpr int XS_TX = 128;   // outputs along x per CTA
constexpr int XS_RR = 4;     // rows per thread

struct XEpilogue {
  // normalisation: out = v / (dx[x]*dy[y]*dz[z]) (un-masked) or v / den3[i] where >0
  const float *dx, *dy, *dz;   // un-masked edge profiles (NULL = no normalisation)
  const float *den3;           // masked: 3-D denominator after its own X sweep
  // combine: out = (minuend[i] - v) * scale when minuend != NULL (DoG / LoG)
  const float *minuend;
  float scale;
  // dual X sweep (DoG / LoG): the edge profiles of the second Gaussian; out = (a / den_a - b / den_b) * scale
  const float *dx_b, *dy_b, *dz_b;
};

template <int MODE>
__global__ void __launch_bounds__(256)
sweep_x_kernel(const float *__restrict__ in, float *__restrict__ out,
               const float *__restrict__ taps, int hw, int nx, i64 nrows, int ny,
               XEpilogue ep, int vec_ok) {
  extern __shared__ __align__(128) float smem[];
  const int hwpad = (hw + 3) & ~3;
  const int pitch = XS_TX + 2 * hwpad + 4;   // +4: keeps rows 16 B aligned, staggers banks
  float *tile = smem;                        // [XS_ROWS][pitch]
  float *tp = smem + (size_t)XS_ROWS * pitch;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int tid = threadIdx.x;
  const int x0 = blockIdx.y * XS_TX;
  const i64 row0 = (i64)blockIdx.x * XS_ROWS;
  const int ntap = 2 * hw + 1;
  for (int k = tid; k < ntap + TAP_PAD_LO + TAP_PAD_HI; k += 256) {
    int t = k - TAP_PAD_LO;
    tp[k] = (t >= 0 && t < ntap) ? taps[t] : 0.0f;
  }
  // stage: each row segment covers x in [x0-hwpad, x0+XS_TX+hwpad)
  const int segw = XS_TX + 2 * hwpad;         // multiple of 4
  const int nvec = segw >> 2;
  for (int r = w; r < XS_ROWS; r += 8) {
    i64 row = row0 + r;
    const float *prow = in + row * (i64)nx;
    for (int c = lane; c < nvec; c += 32) {
      int x = x0 - hwpad + 4 * c;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (row < nrows) {
        if (vec_ok && x >= 0 && x + 3 < nx) {
          v = ld4(prow + x);
        } else {
          if (x + 0 >= 0 && x + 0 < nx) v.x = __ldg(prow + x + 0);
          if (x + 1 >= 0 && x + 1 < nx) v.y = __ldg(prow + x + 1);
          if (x + 2 >= 0 && x + 2 < nx) v.z = __ldg(prow + x + 2);
          if (x + 3 >= 0 && x + 3 < nx) v.w = __ldg(prow + x + 3);
        }
      }
      *reinterpret_cast<float4 *>(tile + (size_t)r * pitch + 4 * c) = v;
    }
  }
  __syncthreads();

  float acc[XS_RR][4];
#pragma unroll
  for (int i = 0; i < XS_RR; i++)
#pragma unroll
    for (int e = 0; e < 4; e++) acc[i][e] = 0.f;
  // thread: outputs x0+4*lane+e (e=0..3) of rows w*4+i.  Input float4 step m holds
  // tile columns 4*lane+4m+c; output e sits at column 4*lane+hwpad+e; tap index
  // = hw + hwpad + e - c - 4m.
  const int nsteps = (2 * hwpad + 4) >> 2;
  const float *tb0 = tp + TAP_PAD_LO + hw + hwpad - 3;
  const float *trow = tile + (size_t)(w * XS_RR) * pitch + 4 * lane;
  // highest input column first = the reference's accumulation order (tap index ascending)
  for (int m = nsteps - 1; m >= 0; m--) {
    float t[7];
    const float *tb = tb0 - 4 * m;
#pragma unroll
    for (int d = 0; d < 7; d++) t[d] = tb[d];
#pragma unroll
    for (int i = 0; i < XS_RR; i++) {
      float4 v = *reinterpret_cast<const float4 *>(trow + (size_t)i * pitch + 4 * m);
      float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int e = 0; e < 4; e++)
#pragma unroll
        for (int c = 3; c >= 0; c--) acc[i][e] = tap_acc<MODE>(acc[i][e], t[e - c + 3], vv[c]);
    }
  }
  const int xo = x0 + 4 * lane;
#pragma unroll
  for (int i = 0; i < XS_RR; i++) {
    i64 row = row0 + w * XS_RR + i;
    if (row >= nrows) break;
    float r4[4] = {acc[i][0], acc[i][1], acc[i][2], acc[i][3]};
    const i64 o = row * (i64)nx + xo;
    if (ep.dx) {
      const int iy = (int)(row % ny);
      const i64 iz = row / ny;
      const float dyz_y = __ldg(ep.dy + iy), dz = __ldg(ep.dz + iz);
#pragma unroll
      for (int e = 0; e < 4; e++)
        if (xo + e < nx) {
          // filter3d.hpp:1016-1019: den = (dx*dy)*dz, IEEE division
          float den = __fmul_rn(__fmul_rn(__ldg(ep.dx + xo + e), dyz_y), dz);
          r4[e] = __fdiv_rn(r4[e], den);
        }
    } else if (ep.den3) {
#pragma unroll
      for (int e = 0; e < 4; e++)
        if (xo + e < nx) {
          float den = __ldg(ep.den3 + o + e);
          if (den > 0.0f) r4[e] = __fdiv_rn(r4[e], den);  // filter3d.hpp:991-992
        }
    }
    if (ep.minuend) {
#pragma unroll
      for (int e = 0; e < 4; e++)
        if (xo + e < nx) r4[e] = __fmul_rn(__fsub_rn(__ldg(ep.minuend + o + e), r4[e]), ep.scale);
    }
    if (vec_ok && xo + 3 < nx) {
      *reinterpret_cast<float4 *>(out + o) = make_float4(r4[0], r4[1], r4[2], r4[3]);
    } else {
#pragma unroll
      for (int e = 0; e < 4; e++)
        if (xo + e < nx) out[o + e] = r4[e];
    }
  }
}

// ---- X sweep with pipelined loads ---------------------------------------------------------
// Same arithmetic as sweep_x_kernel; differences: the tile (64 rows in two chunks of 32)
// is requested up front with cp.async and computed chunk by chunk; x tiles are the FASTEST
// grid index, so the two CTAs that share a halo run back to back and the second finds it
// in L2; the 7 taps of a step come from two aligned LDS.128; the epilogue does one
// integer division per thread instead of two 64-bit ones per row.
constexpr int X2_ROWS = 64;

// One step of the X sweep: the aligned input float4 at column offset 4m feeds the four
// outputs of the thread through taps t[e - c + 3].  POS 1 / 2 = the highest / lowest step,
// where the taps outside [0, 2hw] are known at compile time from DELTA = hwpad - hw and the
// packed operations that would only multiply zero taps are dropped.
template <int MODE, int DELTA, int POS>
__device__ __forceinline__ void x2_step(float2 (&acc)[XS_RR][2], const float *tb0, const float *tb1,
                                        const float *trow, int pitch, int m) {
  // tap pairs (t[j], t[j+1]): even j from tp, odd j from the shifted copy
  const float4 e0 = *reinterpret_cast<const float4 *>(tb0 - 4 * m);      // t0 t1 t2 t3
  const float4 e1 = *reinterpret_cast<const float4 *>(tb0 - 4 * m + 4);  // t4 t5 t6 .
  const float4 o0 = *reinterpret_cast<const float4 *>(tb1 - 4 * m);      // t1 t2 t3 t4
  const float4 o1 = *reinterpret_cast<const float4 *>(tb1 - 4 * m + 4);  // t5 t6 . .
  const float2 t01 = make_float2(e0.x, e0.y), t23 = make_float2(e0.z, e0.w), t45 = make_float2(e1.x, e1.y);
  const float2 t12 = make_float2(o0.x, o0.y), t34 = make_float2(o0.z, o0.w), t56 = make_float2(o1.x, o1.y);
  // pair p (outputs 2p, 2p+1) and input column c are live unless both taps are out of range
#define X2_LIVE(p, c) (POS == 0 || (POS == 1 ? (2 * (p) + 1 - (c) >= DELTA) : (2 * (p) - (c) <= -DELTA)))
#pragma unroll
  for (int i = 0; i < XS_RR; i++) {
    const float4 v = *reinterpret_cast<const float4 *>(trow + (size_t)i * pitch + 4 * m);
    // output e takes tap t[e - c + 3] from input column c; c descending = taps ascending
    if (X2_LIVE(0, 3)) acc[i][0] = tap_acc2<MODE>(acc[i][0], t01, v.w);
    if (X2_LIVE(1, 3)) acc[i][1] = tap_acc2<MODE>(acc[i][1], t23, v.w);
    if (X2_LIVE(0, 2)) acc[i][0] = tap_acc2<MODE>(acc[i][0], t12, v.z);
    if (X2_LIVE(1, 2)) acc[i][1] = tap_acc2<MODE>(acc[i][1], t34, v.z);
    if (X2_LIVE(0, 1)) acc[i][0] = tap_acc2<MODE>(acc[i][0], t23, v.y);
    if (X2_LIVE(1, 1)) acc[i][1] = tap_acc2<MODE>(acc[i][1], t45, v.y);
    if (X2_LIVE(0, 0)) acc[i][0] = tap_acc2<MODE>(acc[i][0], t34, v.x);
    if (X2_LIVE(1, 0)) acc[i][1] = tap_acc2<MODE>(acc[i][1], t56, v.x);
  }
#undef X2_LIVE
}

// EPI: 0 = no normalisation, 1 = divide by the product of the edge profiles, 2 = divide by den3
// TMA: the two 32-row chunks are boxes (128 + 2 hwpad) x 32 of the 2-D tensor map (x, row).
// DUAL (EPI 1 only): the two chunks are the SAME 32 rows of two inputs (in / tmap with taps, in_b / tmap_b with
// taps_b, equal half-widths): the last sweep of both Gaussians of a DoG / LoG in one pass.  The first result waits
// in registers, the second is subtracted from it: neither the first Gaussian nor the "minuend" read of the
// separate passes ever touches HBM.
template <int MODE, int DELTA, int EPI, bool TMA, bool DUAL>
__global__ void __launch_bounds__(256, (DUAL && !TMA) ? 2 : 3)   // (the cp.async fall-back of the dual form needs 4 more registers)
sweep_x2_kernel(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ CUtensorMap tmap_b,
                const float *__restrict__ in, const float *__restrict__ in_b, float *__restrict__ out,
                const float *__restrict__ taps, const float *__restrict__ taps_b, int hw, int nx, i64 nrows, int ny,
                int nxt, XEpilogue ep) {
  static_assert(!DUAL || EPI == 1, "the dual sweep is the normalised, un-masked DoG");
  extern __shared__ __align__(128) float smem[];
  const int hwpad = (hw + 3) & ~3;
  const int pitch = XS_TX + 2 * hwpad + (TMA ? 0 : 4);
  float *tile = smem;                        // [X2_ROWS][pitch]
  uint64_t *bars = reinterpret_cast<uint64_t *>(smem + (size_t)X2_ROWS * pitch);   // [2] (+2 pad), TMA only
  float *tp = smem + (size_t)X2_ROWS * pitch + 8;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int tid = threadIdx.x;
  const int xt = blockIdx.x % nxt;
  const i64 row0 = (i64)(blockIdx.x / nxt) * (DUAL ? 32 : X2_ROWS);
  const int chunk_rows = DUAL ? 0 : 32;      // first row of chunk c = row0 + chunk_rows * c
  const int x0 = xt * XS_TX;
  const int nvec = (XS_TX + 2 * hwpad) >> 2;
  if (TMA && tid == 0) {
    mbar_init(bars + 0, 1);
    mbar_init(bars + 1, 1);
    mbar_init_fence();
#pragma unroll
    for (int c = 0; c < 2; c++) {
      if (row0 + chunk_rows * c >= nrows) break;
      mbar_expect_tx(bars + c, 32u * (unsigned)pitch * sizeof(float));
      tma_load_2d(tile + (size_t)32 * c * pitch, (DUAL && c) ? &tmap_b : &tmap, bars + c, x0 - hwpad,
                  (int)(row0 + chunk_rows * c));
    }
  }
  // (cp.async) every thread copies a fixed 16-byte column of the tile (two of them for the
  // few that cover the halo) in rows w, w+8, ...: one pointer increment per copy
#pragma unroll
  for (int c = 0; c < 2; c++) {
    if (TMA) break;
    const float *inc = (DUAL && c) ? in_b : in;
    if (row0 + chunk_rows * c < nrows) {
      for (int cc = lane; cc < nvec; cc += 32) {
        const int x = x0 - hwpad + 4 * cc;
        const bool okx = x >= 0 && x < nx;
        i64 row = row0 + chunk_rows * c + w;
        const float *src = okx ? inc + row * (i64)nx + x : inc;
        float *dst = tile + (size_t)(32 * c + w) * pitch + 4 * cc;
#pragma unroll
        for (int k = 0; k < 4; k++) {
          const bool ok = okx && row < nrows;
          cp_async16_zfill(dst, ok ? src : inc, ok);
          row += 8;
          src += 8 * (i64)nx;
          dst += 8 * pitch;
        }
      }
    }
    cp_async_commit_group();
  }
  // taps, placed so that the 8-float window of every step is 16-byte aligned, plus a copy
  // shifted by one float (tp1[k] = tp[k+1]) so that odd tap pairs are aligned pairs too
  // (DUAL: the same pair of arrays for taps_b behind them)
  const int ntap = 2 * hw + 1;
  const int P = 16 + ((3 - hw - hwpad) & 3);
  const int tplen = (P + ntap + 16 + 3) & ~3;
  for (int k = tid; k < tplen; k += 256) {
    const int t = k - P;
    tp[k] = (t >= 0 && t < ntap) ? taps[t] : 0.0f;
    tp[tplen + k] = (t + 1 >= 0 && t + 1 < ntap) ? taps[t + 1] : 0.0f;
    if (DUAL) {
      tp[2 * tplen + k] = (t >= 0 && t < ntap) ? taps_b[t] : 0.0f;
      tp[3 * tplen + k] = (t + 1 >= 0 && t + 1 < ntap) ? taps_b[t + 1] : 0.0f;
    }
  }
  const int nsteps = (2 * hwpad + 4) >> 2;
  const int xo = x0 + 4 * lane;
  float dxv[4] = {1.f, 1.f, 1.f, 1.f};
  if (EPI == 1 && !DUAL && xo < nx) {
#pragma unroll
    for (int e = 0; e < 4; e++) dxv[e] = __ldg(ep.dx + xo + e);
  }
  float keep[XS_RR][4];   // DUAL: the first Gaussian's rows

#pragma unroll 1
  for (int c = 0; c < 2; c++) {
    if (row0 + chunk_rows * c >= nrows) break;  // uniform
    if (TMA) {
      if (c == 0) __syncthreads();   // barriers initialised, taps staged
      mbar_wait(bars + c, 0);
    } else {
      if (c == 0) cp_async_wait_group<1>(); else cp_async_wait_group<0>();
      __syncthreads();
    }
    const bool second = DUAL && c == 1;
    const float *tb0 = tp + (second ? 2 * tplen : 0) + P + hw + hwpad - 3;
    const float *tb1 = tb0 + tplen;
    float2 acc[XS_RR][2];   // outputs (0,1) and (2,3) of each row
#pragma unroll
    for (int i = 0; i < XS_RR; i++) acc[i][0] = acc[i][1] = make_float2(0.f, 0.f);
    const float *trow = tile + (size_t)(32 * c + w * XS_RR) * pitch + 4 * lane;
    // highest input column first = the reference's accumulation order (tap index ascending)
    if (nsteps >= 2) {
      x2_step<MODE, DELTA, 1>(acc, tb0, tb1, trow, pitch, nsteps - 1);
      for (int m = nsteps - 2; m >= 1; m--) x2_step<MODE, DELTA, 0>(acc, tb0, tb1, trow, pitch, m);
      x2_step<MODE, DELTA, 2>(acc, tb0, tb1, trow, pitch, 0);
    } else {
      x2_step<MODE, DELTA, 0>(acc, tb0, tb1, trow, pitch, 0);
    }
    if (xo >= nx) continue;
    const i64 rb = row0 + chunk_rows * c + w * XS_RR;
    unsigned iz = 0, iy = 0;
    if (EPI == 1) {   // rows < 2^32 (checked by the host)
      iz = (unsigned)rb / (unsigned)ny;
      iy = (unsigned)rb - iz * (unsigned)ny;
    }
    const i64 o0 = rb * (i64)nx + xo;
    float *op = out + o0;
    const float *mp = ep.minuend ? ep.minuend + o0 : nullptr;
    const float *dp = EPI == 2 ? ep.den3 + o0 : nullptr;
    const float *pdy = second ? ep.dy_b : ep.dy, *pdz = second ? ep.dz_b : ep.dz;
    const int nrow_here = (int)min((i64)XS_RR, nrows - rb);
    if (DUAL) {   // each Gaussian has its own profile
#pragma unroll
      for (int e = 0; e < 4; e++) dxv[e] = __ldg((second ? ep.dx_b : ep.dx) + xo + e);
    }
#pragma unroll
    for (int i = 0; i < XS_RR; i++) {
      if (i >= nrow_here) break;
      float r4[4] = {acc[i][0].x, acc[i][0].y, acc[i][1].x, acc[i][1].y};
      if (EPI == 1) {
        while (iy >= (unsigned)ny) { iy -= ny; iz++; }
        const float dy = __ldg(pdy + iy), dz = __ldg(pdz + iz);
        iy++;
        // filter3d.hpp:1016-1019: den = (dx*dy)*dz, IEEE division.  x / 1 == x, so the
        // interior is skipped whenever the taps sum to exactly 1 (one test per row).
        float den[4];
#pragma unroll
        for (int e = 0; e < 4; e++) den[e] = __fmul_rn(__fmul_rn(dxv[e], dy), dz);
        if (!(den[0] == 1.0f && den[1] == 1.0f && den[2] == 1.0f && den[3] == 1.0f)) {
#pragma unroll
          for (int e = 0; e < 4; e++) r4[e] = __fdiv_rn(r4[e], den[e]);
        }
      } else if (EPI == 2) {
        const float4 den = ld4(dp + (size_t)i * nx);
        if (den.x > 0.0f) r4[0] = __fdiv_rn(r4[0], den.x);  // filter3d.hpp:991-992
        if (den.y > 0.0f) r4[1] = __fdiv_rn(r4[1], den.y);
        if (den.z > 0.0f) r4[2] = __fdiv_rn(r4[2], den.z);
        if (den.w > 0.0f) r4[3] = __fdiv_rn(r4[3], den.w);
      }
      if (DUAL) {
        if (c == 0) {
#pragma unroll
          for (int e = 0; e < 4; e++) keep[i][e] = r4[e];
          continue;
        }
#pragma unroll
        for (int e = 0; e < 4; e++) r4[e] = __fmul_rn(__fsub_rn(keep[i][e], r4[e]), ep.scale);
      } else if (mp) {
        const float4 mn = ld4(mp + (size_t)i * nx);
        r4[0] = __fmul_rn(__fsub_rn(mn.x, r4[0]), ep.scale);
        r4[1] = __fmul_rn(__fsub_rn(mn.y, r4[1]), ep.scale);
        r4[2] = __fmul_rn(__fsub_rn(mn.z, r4[2]), ep.scale);
        r4[3] = __fmul_rn(__fsub_rn(mn.w, r4[3]), ep.scale);
      }
      *reinterpret_cast<float4 *>(op + (size_t)i * nx) = make_float4(r4[0], r4[1], r4[2], r4[3]);
    }
  }
}

__global__ void fill_kernel(float *p, float v, i64 n) {
  i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
  i64 stride = (i64)gridDim.x * blockDim.x;
  for (; i < n; i += stride) p[i] = v;
}

// ---------------------------------------------------------------------------------
// host drivers (device pointers)
// ---------------------------------------------------------------------------------
template <int MODE>
static void launch_axis_mode(visfd_ctx *ctx, const float *in, float *out, const float *mask,
                             const float *d_taps, int hw, i64 nx, i64 n_axis, i64 s_axis,
                             i64 n_other, i64 s_other) {
  const int rows = AX_TA + 2 * hw + 8;
  size_t smem = ((size_t)rows * AX_TX * (MODE == MODE_EXACT_MASKED ? 2 : 1) +
                 (2 * hw + 1 + TAP_PAD_LO + TAP_PAD_HI)) * sizeof(float);
  VREQUIRE(smem <= 220 * 1024, "filter half-width too large for the sweep kernel");
  VREQUIRE(n_other <= 65535 && div_up(n_axis, AX_TA) <= 65535, "volume too large in y/z for one launch");
  // per launch: the attribute is per DEVICE and a process may hold contexts on several GPUs
  VCK(cudaFuncSetAttribute(sweep_axis_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
  int vec_ok = (nx % 4 == 0) && (((uintptr_t)in & 15) == 0) && (((uintptr_t)out & 15) == 0) &&
               (!mask || ((uintptr_t)mask & 15) == 0);
  dim3 grid(div_up(nx, AX_TX), div_up(n_axis, AX_TA), (unsigned)n_other);
  dim3 block(32, AX_WARPS);
  sweep_axis_kernel<MODE><<<grid, block, smem, ctx->stream>>>(in, out, mask, d_taps, hw, (int)nx, n_axis,
                                                              s_axis, s_other, vec_ok);
  VCK(cudaGetLastError());
  ctx->count_launch();
}

template <int MODE>
static void launch_axis2_mode(visfd_ctx *ctx, const float *in, float *out, const float *d_taps, int hw,
                              i64 nx, i64 n_axis, i64 s_axis, i64 n_other, i64 s_other) {
  const int ntap8 = (2 * hw + 1 + 7) & ~7;
  const size_t smem = ((size_t)(ntap8 + A2_S - 1) * AX_TX + ntap8) * sizeof(float);
  VREQUIRE(smem <= 220 * 1024, "filter half-width too large for the sweep kernel");
  VREQUIRE(n_other <= 65535 && div_up(n_axis, A2_S) <= 65535, "volume too large in y/z for one launch");
  // per launch: the attribute is per DEVICE and a process may hold contexts on several GPUs
  VCK(cudaFuncSetAttribute(sweep_axis2_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
  int vec_ok = (nx % 4 == 0) && (((uintptr_t)in & 15) == 0) && (((uintptr_t)out & 15) == 0);
  dim3 grid(div_up(nx, AX_TX), div_up(n_axis, A2_S), (unsigned)n_other);
  dim3 block(32, 8);
  sweep_axis2_kernel<MODE><<<grid, block, smem, ctx->stream>>>(in, out, d_taps, hw, ntap8, (int)nx, n_axis,
                                                               s_axis, s_other, vec_ok);
  VCK(cudaGetLastError());
  ctx->count_launch();
}

// out_b / d_taps_b != NULL: the dual form (both tap arrays hold 2 hw + 1 entries)
template <int MODE, bool DUAL>
static bool launch_axis3_impl(visfd_ctx *ctx, const float *in, float *out, float *out_b, const float *d_taps,
                              const float *d_taps_b, int hw, i64 nx, i64 n_axis, i64 s_axis, i64 n_other,
                              i64 s_other) {
  const int ntap8 = (2 * hw + 1 + 7) & ~7;
  const size_t smem = ((size_t)(ntap8 + A3_NCH * A2_S) * AX_TX + (DUAL ? 2 : 1) * ntap8) * sizeof(float) +
                      A3_NCH * sizeof(uint64_t);
  const bool vec_ok = (nx % 4 == 0) && (((uintptr_t)in & 15) == 0) && (((uintptr_t)out & 15) == 0) &&
                      (((uintptr_t)out_b & 15) == 0);
  if (!vec_ok || smem > 100 * 1024 || ntap8 > 256 || n_other > 65535 || div_up(n_axis, A3_NCH * A2_S) > 65535) return false;
  // per launch: the attribute is per DEVICE and a process may hold contexts on several GPUs
  VCK(cudaFuncSetAttribute(sweep_axis3_kernel<MODE, true, DUAL>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
  VCK(cudaFuncSetAttribute(sweep_axis3_kernel<MODE, false, DUAL>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
  dim3 grid(div_up(nx, AX_TX), div_up(n_axis, A3_NCH * A2_S), (unsigned)n_other);
  dim3 block(32, 8);
  // the volume as a 3-D tensor (x, y, z): Y sweep: s_axis == nx; Z sweep: s_other == nx
  const int axis_dim = (s_axis == nx) ? 1 : 2;
  const i64 dims[3] = {nx, axis_dim == 1 ? n_axis : n_other, axis_dim == 1 ? n_other : n_axis};
  const int box[3] = {AX_TX, axis_dim == 1 ? 8 : 1, axis_dim == 1 ? 1 : 8};
  CUtensorMap tmap;
  memset(&tmap, 0, sizeof(tmap));
  const bool consistent = axis_dim == 1 ? (s_other == nx * n_axis) : (s_axis == nx * n_other);
  if (ctx->use_tma && consistent && make_tensor_map(&tmap, in, 3, dims, box))
    sweep_axis3_kernel<MODE, true, DUAL><<<grid, block, smem, ctx->stream>>>(
        tmap, axis_dim, in, out, out_b, d_taps, d_taps_b, hw, ntap8, (int)nx, n_axis, s_axis, s_other);
  else
    sweep_axis3_kernel<MODE, false, DUAL><<<grid, block, smem, ctx->stream>>>(
        tmap, axis_dim, in, out, out_b, d_taps, d_taps_b, hw, ntap8, (int)nx, n_axis, s_axis, s_other);
  VCK(cudaGetLastError());
  ctx->count_launch();
  return true;
}

template <int MODE>
static bool launch_axis3_mode(visfd_ctx *ctx, const float *in, float *out, const float *d_taps, int hw,
                              i64 nx, i64 n_axis, i64 s_axis, i64 n_other, i64 s_other) {
  return launch_axis3_impl<MODE, false>(ctx, in, out, nullptr, d_taps, nullptr, hw, nx, n_axis, s_axis, n_other,
                                        s_other);
}

static void launch_axis(visfd_ctx *ctx, const float *in, float *out, const float *mask,
                        const float *d_taps, int hw, i64 nx, i64 n_axis, i64 s_axis,
                        i64 n_other, i64 s_other) {
  if (!mask) {
    if (ctx->fast_gauss ? launch_axis3_mode<MODE_FAST>(ctx, in, out, d_taps, hw, nx, n_axis, s_axis, n_other, s_other)
                        : launch_axis3_mode<MODE_EXACT>(ctx, in, out, d_taps, hw, nx, n_axis, s_axis, n_other, s_other))
      return;
    if (ctx->fast_gauss) launch_axis2_mode<MODE_FAST>(ctx, in, out, d_taps, hw, nx, n_axis, s_axis, n_other, s_other);
    else launch_axis2_mode<MODE_EXACT>(ctx, in, out, d_taps, hw, nx, n_axis, s_axis, n_other, s_other);
    return;
  }
  if (ctx->fast_gauss)
    launch_axis_mode<MODE_FAST>(ctx, in, out, mask, d_taps, hw, nx, n_axis, s_axis, n_other, s_other);
  else if (mask)
    launch_axis_mode<MODE_EXACT_MASKED>(ctx, in, out, mask, d_taps, hw, nx, n_axis, s_axis, n_other, s_other);
  else
    launch_axis_mode<MODE_EXACT>(ctx, in, out, mask, d_taps, hw, nx, n_axis, s_axis, n_other, s_other);
}

static size_t x2_smem_bytes(bool dual, int hw) {
  const int hwpad = (hw + 3) & ~3;
  const int pitch = XS_TX + 2 * hwpad + 4;
  return ((size_t)X2_ROWS * pitch + 8 + (dual ? 4 : 2) * (2 * hw + 1 + 40)) * sizeof(float);
}
static bool x2_qualifies(bool dual, i64 nx, i64 nrows, int hw) {
  const i64 nxt = div_up(nx, XS_TX), nrt = div_up(nrows, (i64)(dual ? 32 : X2_ROWS));
  return nx % 4 == 0 && x2_smem_bytes(dual, hw) <= 100 * 1024 && nxt * nrt <= 2147483647LL && nrows < 4294967296LL;
}

// The pipelined X sweep; in_b / d_taps_b != NULL: its dual form (DoG / LoG, see the kernel).  Returns false when the
// volume does not qualify (nothing launched).
static bool launch_x2(visfd_ctx *ctx, const float *in, const float *in_b, float *out, const float *d_taps,
                      const float *d_taps_b, int hw, i64 nx, i64 ny, i64 nrows, const XEpilogue &ep) {
  const bool dual = in_b != nullptr;
  const int hwpad = (hw + 3) & ~3;
  const bool vec_ok = (((uintptr_t)in & 15) == 0) && (((uintptr_t)in_b & 15) == 0) &&
                      (((uintptr_t)out & 15) == 0) && (!ep.den3 || ((uintptr_t)ep.den3 & 15) == 0) &&
                      (!ep.minuend || ((uintptr_t)ep.minuend & 15) == 0);
  if (!vec_ok || !x2_qualifies(dual, nx, nrows, hw)) return false;
  const size_t smem2 = x2_smem_bytes(dual, hw);
  const i64 nxt = div_up(nx, XS_TX), nrt = div_up(nrows, (i64)(dual ? 32 : X2_ROWS));
  if (dual && !(ep.dx && ep.dx_b && !ep.den3 && !ep.minuend)) return false;
  CUtensorMap tmap, tmap_b;
  memset(&tmap, 0, sizeof(tmap));
  memset(&tmap_b, 0, sizeof(tmap_b));
  const i64 dims2[2] = {nx, nrows};
  const int box2[2] = {XS_TX + 2 * hwpad, 32};
  const bool tma = ctx->use_tma && make_tensor_map(&tmap, in, 2, dims2, box2) &&
                   (!dual || make_tensor_map(&tmap_b, in_b, 2, dims2, box2));
  const unsigned grid = (unsigned)(nxt * nrt);   // 1-D grid, x tiles fastest
  // (the attribute is set per launch: it is per DEVICE and a process may hold contexts on several GPUs)
#define X2_LAUNCH_T(M, D, E, T, U)                                                                                \
  do {                                                                                                            \
    VCK(cudaFuncSetAttribute(sweep_x2_kernel<M, D, E, T, U>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024)); \
    sweep_x2_kernel<M, D, E, T, U><<<grid, 256, smem2, ctx->stream>>>(tmap, tmap_b, in, in_b, out, d_taps, d_taps_b, hw, \
                                                                      (int)nx, nrows, (int)ny, (int)nxt, ep);     \
  } while (0)
#define X2_LAUNCH_E(M, D, E, U)                          \
  do {                                                   \
    if (tma) X2_LAUNCH_T(M, D, E, true, U);              \
    else X2_LAUNCH_T(M, D, E, false, U);                 \
  } while (0)
#define X2_LAUNCH(M, D)                                  \
  do {                                                   \
    if (dual) X2_LAUNCH_E(M, D, 1, true);                \
    else if (ep.dx) X2_LAUNCH_E(M, D, 1, false);         \
    else if (ep.den3) X2_LAUNCH_E(M, D, 2, false);       \
    else X2_LAUNCH_E(M, D, 0, false);                    \
  } while (0)
#define X2_LAUNCH_D(M)                                   \
  switch (hwpad - hw) {                                  \
    case 0: X2_LAUNCH(M, 0); break;                      \
    case 1: X2_LAUNCH(M, 1); break;                      \
    case 2: X2_LAUNCH(M, 2); break;                      \
    default: X2_LAUNCH(M, 3); break;                     \
  }
  if (ctx->fast_gauss) { X2_LAUNCH_D(MODE_FAST) } else { X2_LAUNCH_D(MODE_EXACT) }
#undef X2_LAUNCH_D
#undef X2_LAUNCH
#undef X2_LAUNCH_E
#undef X2_LAUNCH_T
  VCK(cudaGetLastError());
  ctx->count_launch();
  return true;
}

static void launch_x(visfd_ctx *ctx, const float *in, float *out, const float *d_taps, int hw,
                     i64 nx, i64 ny, i64 nrows, const XEpilogue &ep) {
  if (launch_x2(ctx, in, nullptr, out, d_taps, nullptr, hw, nx, ny, nrows, ep)) return;
  const int hwpad = (hw + 3) & ~3;
  const int pitch = XS_TX + 2 * hwpad + 4;
  size_t smem = ((size_t)XS_ROWS * pitch + (2 * hw + 1 + TAP_PAD_LO + TAP_PAD_HI)) * sizeof(float);
  VREQUIRE(smem <= 220 * 1024, "filter half-width too large for the x sweep kernel");
  // per launch: the attribute is per DEVICE and a process may hold contexts on several GPUs
  VCK(cudaFuncSetAttribute(sweep_x_kernel<MODE_FAST>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
  VCK(cudaFuncSetAttribute(sweep_x_kernel<MODE_EXACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
  int vec_ok = (nx % 4 == 0) && (((uintptr_t)in & 15) == 0) && (((uintptr_t)out & 15) == 0) &&
               (!ep.den3 || ((uintptr_t)ep.den3 & 15) == 0) && (!ep.minuend || ((uintptr_t)ep.minuend & 15) == 0);
  // rows go on grid.x (2^31-1 blocks), x tiles on grid.y
  i64 gx = (nrows + XS_ROWS - 1) / XS_ROWS;
  VREQUIRE(gx <= 2147483647LL && div_up(nx, XS_TX) <= 65535, "volume too large for one launch");
  dim3 grid((unsigned)gx, div_up(nx, XS_TX), 1);
  if (ctx->fast_gauss)
    sweep_x_kernel<MODE_FAST><<<grid, 256, smem, ctx->stream>>>(in, out, d_taps, hw, (int)nx, nrows, (int)ny, ep, vec_ok);
  else
    sweep_x_kernel<MODE_EXACT><<<grid, 256, smem, ctx->stream>>>(in, out, d_taps, hw, (int)nx, nrows, (int)ny, ep, vec_ok);
  VCK(cudaGetLastError());
  ctx->count_launch();
}

void fill_device(visfd_ctx *ctx, float *p, float v, i64 n) {
  fill_kernel<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(p, v, n);
  VCK(cudaGetLastError());
  ctx->count_launch();
}

// ApplySeparable on device memory.  src/dst/mask: device pointers to the slab
// (nz_local planes = global planes [z_offset, z_offset+nz_local) of nz_global).
// tmp: device scratch of N floats (dst may not alias src).  If combine_minuend is
// given the result written to dst is (combine_minuend - filtered) * combine_scale.
float separable_device(visfd_ctx *ctx, i64 nx, i64 ny, i64 nz_local, i64 z_offset, i64 nz_global,
                       const float *src, float *dst, const float *mask, const float *const taps[3],
                       const int hw[3], bool normalize, const float *combine_minuend,
                       float combine_scale, bool z_swept) {
  StageTimer timer(ctx, "gauss");
  const i64 N = nx * ny * nz_local;
  VREQUIRE(nx > 0 && ny > 0 && nz_local > 0, "empty volume");
  VREQUIRE(hw[0] >= 0 && hw[1] >= 0 && hw[2] >= 0, "negative filter half-width");
  VREQUIRE(z_offset >= 0 && z_offset + nz_local <= nz_global, "slab outside the volume");
  // The Z sweep reads src while other CTAs already write dst: unlike the reference (one temporary per line,
  // filter3d.hpp:710-713 copies first) the device path cannot filter in place
  // (z_swept: dst already holds the Z sweep of the source -- dog_device's shared sweep -- and src is not read)
  VREQUIRE((z_swept || src != dst) && (!mask || mask != dst) && (!combine_minuend || combine_minuend != dst),
           "separable filter: dst must not alias src, mask or the minuend (device pointers)");
  VREQUIRE(!z_swept || !mask, "separable filter: the shared Z sweep has no masked form");
  // upload taps (+ edge profiles) in one host buffer
  const int nt[3] = {2 * hw[0] + 1, 2 * hw[1] + 1, 2 * hw[2] + 1};
  const i64 n_dim[3] = {nx, ny, nz_local};
  size_t total = nt[0] + nt[1] + nt[2] + nx + ny + nz_local;
  std::vector<float> h(total);
  size_t off_t[3], off_d[3], o = 0;
  for (int d = 0; d < 3; d++) { off_t[d] = o; memcpy(&h[o], taps[d], nt[d] * sizeof(float)); o += nt[d]; }
  for (int d = 0; d < 3; d++) { off_d[d] = o; o += n_dim[d]; }
  bool plain_norm = normalize && !mask;
  if (plain_norm) {
    edge_profile(taps[0], hw[0], nx, 0, nx, &h[off_d[0]]);
    edge_profile(taps[1], hw[1], ny, 0, ny, &h[off_d[1]]);
    edge_profile(taps[2], hw[2], nz_global, z_offset, nz_local, &h[off_d[2]]);
  }
  Scratch<float> dconst(ctx, total);
  VCK(cudaMemcpyAsync(dconst.get(), h.data(), total * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  // The host vector must outlive the async copy from pageable memory: cudaMemcpyAsync
  // from pageable memory returns after staging, so this is safe.
  const float *tx = dconst.get() + off_t[0], *ty = dconst.get() + off_t[1], *tz = dconst.get() + off_t[2];

  Scratch<float> tmp(ctx, N);
  XEpilogue ep{};
  ep.minuend = combine_minuend;
  ep.scale = combine_scale;
  if (!mask) {
    // Z: src -> dst ; Y: dst -> tmp ; X: tmp -> dst
    if (!z_swept) launch_axis(ctx, src, dst, nullptr, tz, hw[2], nx, nz_local, nx * ny, ny, nx);
    launch_axis(ctx, dst, tmp.get(), nullptr, ty, hw[1], nx, ny, nx, nz_local, nx * ny);
    if (plain_norm) {
      ep.dx = dconst.get() + off_d[0];
      ep.dy = dconst.get() + off_d[1];
      ep.dz = dconst.get() + off_d[2];
    }
    launch_x(ctx, tmp.get(), dst, tx, hw[0], nx, ny, ny * nz_local, ep);
  } else {
    // masked: filter mask*src and (if normalising) the mask itself
    // (filter3d.hpp:799-803, 868-879, 948-959, 986-992)
    Scratch<float> den, den2;
    launch_axis(ctx, src, dst, mask, tz, hw[2], nx, nz_local, nx * ny, ny, nx);
    launch_axis(ctx, dst, tmp.get(), nullptr, ty, hw[1], nx, ny, nx, nz_local, nx * ny);
    if (normalize) {
      den.reset(ctx, N);
      den2.reset(ctx, N);
      XEpilogue none{};
      launch_axis(ctx, mask, den.get(), nullptr, tz, hw[2], nx, nz_local, nx * ny, ny, nx);
      launch_axis(ctx, den.get(), den2.get(), nullptr, ty, hw[1], nx, ny, nx, nz_local, nx * ny);
      launch_x(ctx, den2.get(), den.get(), tx, hw[0], nx, ny, ny * nz_local, none);
      ep.den3 = den.get();
    }
    launch_x(ctx, tmp.get(), dst, tx, hw[0], nx, ny, ny * nz_local, ep);
  }
  return taps[0][hw[0]] * taps[1][hw[1]] * taps[2][hw[2]];  // filter3d.hpp:1044-1046
}

float gauss_device(visfd_ctx *ctx, i64 nx, i64 ny, i64 nz_local, i64 z_offset, i64 nz_global,
                   const float *src, float *dst, const float *mask, const float sigma[3],
                   const int hw[3], bool normalize, const float *combine_minuend, float combine_scale,
                   bool z_swept) {
  std::vector<float> t[3];
  const float *tp[3];
  for (int d = 0; d < 3; d++) {
    VREQUIRE(hw[d] >= 0 && sigma[d] >= 0.0f, "negative sigma or half-width");
    t[d].resize(2 * hw[d] + 1);
    gen_gauss1d(sigma[d], hw[d], t[d].data());
    tp[d] = t[d].data();
  }
  return separable_device(ctx, nx, ny, nz_local, z_offset, nz_global, src, dst, mask, tp, hw,
                          normalize, combine_minuend, combine_scale, z_swept);
}

// The Z sweeps of two Gaussians over one read of the source: src -> (dst_a, dst_b).  Both tap arrays are centred in
// 2 hw + 1 entries, hw = the larger half-width; the padding taps are zeros, which add +-0 to the running sums in
// the same order as before and so leave every finite result bit for bit what the separate sweeps give.
// Returns false (nothing launched) when the pair does not qualify.
static bool dual_z_sweep(visfd_ctx *ctx, i64 nx, i64 ny, i64 nz_local, const float *src, float *dst_a, float *dst_b,
                         float sigma_a, int hw_a, float sigma_b, int hw_b) {
  const int hw = std::max(hw_a, hw_b);
  // padding the shorter filter costs arithmetic: measured on B200, one extra group of 8 taps still pays with FMA
  // accumulation (DoG sigma 2 / 3.2: 1.34 -> 1.29 ms at 512^3) and does not in the bit-exact mode (1.63 -> 1.67)
  const int extra = ((2 * hw + 8) & ~7) - ((2 * std::min(hw_a, hw_b) + 8) & ~7);
  if (extra > (ctx->fast_gauss ? 8 : 0)) return false;
  if (src == dst_a || src == dst_b || dst_a == dst_b) return false;
  const int nt = 2 * hw + 1;
  std::vector<float> h(2 * (size_t)nt, 0.0f);
  gen_gauss1d(sigma_a, hw_a, h.data() + (hw - hw_a));
  gen_gauss1d(sigma_b, hw_b, h.data() + nt + (hw - hw_b));
  Scratch<float> d(ctx, 2 * (size_t)nt);
  VCK(cudaMemcpyAsync(d.get(), h.data(), h.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  StageTimer timer(ctx, "gauss");
  return ctx->fast_gauss
             ? launch_axis3_impl<MODE_FAST, true>(ctx, src, dst_a, dst_b, d.get(), d.get() + nt, hw, nx, nz_local,
                                                  nx * ny, ny, nx)
             : launch_axis3_impl<MODE_EXACT, true>(ctx, src, dst_a, dst_b, d.get(), d.get() + nt, hw, nx, nz_local,
                                                   nx * ny, ny, nx);
}

// ApplyDog (filter3d.hpp:1340-1402): dst = G_a(src) - G_b(src), optionally * scale (ApplyLog).
void dog_device(visfd_ctx *ctx, i64 nx, i64 ny, i64 nz_local, i64 z_offset, i64 nz_global,
                const float *src, float *dst, const float *mask, const float sigma_a[3],
                const float sigma_b[3], const int hw[3], float scale, float *A, float *B, const int *hw_b) {
  const i64 N = nx * ny * nz_local;
  Scratch<float> ga(ctx, N);
  const int *hb = hw_b ? hw_b : hw;
  for (int d = 0; d < 3; d++)
    VREQUIRE(hw[d] >= 0 && hb[d] >= 0 && sigma_a[d] >= 0.0f && sigma_b[d] >= 0.0f, "negative sigma or half-width");
  if (!mask && hw[0] == hb[0] && hw[1] == hb[1] && hw[2] == hb[2] && ((uintptr_t)dst & 15) == 0 && src != dst &&
      x2_qualifies(true, nx, ny * nz_local, hw[0])) {
    // Both Gaussians in four launches and 40 B / voxel instead of six and 52 (ApplyLog's pair always has equal
    // half-widths, filter3d.hpp:1460-1464): one Z sweep of the source for both, a Y sweep each, one X sweep that
    // normalises both, subtracts and scales.  Same operations on the same values in the same order as the two
    // separate filters: bit-identical to them.
    StageTimer timer(ctx, "gauss");
    VREQUIRE(nx > 0 && ny > 0 && nz_local > 0, "empty volume");
    VREQUIRE(z_offset >= 0 && z_offset + nz_local <= nz_global, "slab outside the volume");
    const int nt[3] = {2 * hw[0] + 1, 2 * hw[1] + 1, 2 * hw[2] + 1};
    const i64 n_dim[3] = {nx, ny, nz_local};
    const size_t per = (size_t)nt[0] + nt[1] + nt[2] + nx + ny + nz_local;
    std::vector<float> h(2 * per);
    size_t off_t[3], off_d[3], o = 0;
    for (int d = 0; d < 3; d++) { off_t[d] = o; o += nt[d]; }
    for (int d = 0; d < 3; d++) { off_d[d] = o; o += n_dim[d]; }
    float centre[2] = {1.0f, 1.0f};
    for (int f = 0; f < 2; f++) {
      float *hf = h.data() + f * per;
      const float *sg = f ? sigma_b : sigma_a;
      for (int d = 0; d < 3; d++) {
        gen_gauss1d(sg[d], hw[d], hf + off_t[d]);
        centre[f] *= hf[off_t[d] + hw[d]];   // filter3d.hpp:1044-1046
      }
      edge_profile(hf + off_t[0], hw[0], nx, 0, nx, hf + off_d[0]);
      edge_profile(hf + off_t[1], hw[1], ny, 0, ny, hf + off_d[1]);
      edge_profile(hf + off_t[2], hw[2], nz_global, z_offset, nz_local, hf + off_d[2]);
    }
    Scratch<float> dconst(ctx, 2 * per), tmp(ctx, N);
    VCK(cudaMemcpyAsync(dconst.get(), h.data(), h.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    const float *ca = dconst.get(), *cb = dconst.get() + per;
    // Z: src -> (ga, dst)
    const bool z_dual =
        ctx->fast_gauss ? launch_axis3_impl<MODE_FAST, true>(ctx, src, ga.get(), dst, ca + off_t[2], cb + off_t[2], hw[2],
                                                             nx, nz_local, nx * ny, ny, nx)
                        : launch_axis3_impl<MODE_EXACT, true>(ctx, src, ga.get(), dst, ca + off_t[2], cb + off_t[2], hw[2],
                                                              nx, nz_local, nx * ny, ny, nx);
    if (!z_dual) {
      launch_axis(ctx, src, ga.get(), nullptr, ca + off_t[2], hw[2], nx, nz_local, nx * ny, ny, nx);
      launch_axis(ctx, src, dst, nullptr, cb + off_t[2], hw[2], nx, nz_local, nx * ny, ny, nx);
    }
    // Y: ga -> tmp, dst -> ga
    launch_axis(ctx, ga.get(), tmp.get(), nullptr, ca + off_t[1], hw[1], nx, ny, nx, nz_local, nx * ny);
    launch_axis(ctx, dst, ga.get(), nullptr, cb + off_t[1], hw[1], nx, ny, nx, nz_local, nx * ny);
    // X: (tmp, ga) -> dst
    XEpilogue ep{};
    ep.scale = scale;
    ep.dx = ca + off_d[0]; ep.dy = ca + off_d[1]; ep.dz = ca + off_d[2];
    ep.dx_b = cb + off_d[0]; ep.dy_b = cb + off_d[1]; ep.dz_b = cb + off_d[2];
    const bool x_dual = launch_x2(ctx, tmp.get(), ga.get(), dst, ca + off_t[0], cb + off_t[0], hw[0], nx, ny,
                                  ny * nz_local, ep);
    VREQUIRE(x_dual, "dog: the shared X sweep did not launch");   // x2_qualifies() said it would
    if (A) *A = centre[0];
    if (B) *B = centre[1];
    return;
  }
  const bool z_swept = !mask && dual_z_sweep(ctx, nx, ny, nz_local, src, ga.get(), dst, sigma_a[2], hw[2],
                                             sigma_b[2], hb[2]);
  float a = gauss_device(ctx, nx, ny, nz_local, z_offset, nz_global, src, ga.get(), mask, sigma_a, hw,
                         true, nullptr, 1.0f, z_swept);
  float b = gauss_device(ctx, nx, ny, nz_local, z_offset, nz_global, src, dst, mask, sigma_b, hb, true,
                         ga.get(), scale, z_swept);
  if (A) *A = a;
  if (B) *B = b;
}

// ApplyLog parameter derivation: filter3d.hpp:1451-1464, :1493
void log_params(const float sigma[3], float delta, float truncate_ratio, float sigma_a[3],
                float sigma_b[3], int hw[3], float *scale) {
  for (int d = 0; d < 3; d++) {
    sigma_a[d] = (float)(sigma[d] * (1.0 - 0.5 * delta));
    sigma_b[d] = (float)(sigma[d] * (1.0 + 0.5 * delta));
    hw[d] = (int)floor(truncate_ratio * std::max(sigma_a[d], sigma_b[d]));
  }
  *scale = (float)(1.0 / (delta * delta));
}

}  // namespace visfd_cuda
