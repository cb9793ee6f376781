// select.cu -- the saliency cut of HandleTV (bin/filter_mrc/handlers.cpp:1751-1797)
// without a sort: the threshold is the element of rank k = floor(n*f) in DECREASING
// order, found by a 3-pass (11+11+10 bit) radix select over order-preserving 32-bit
// keys.  Each pass is one streaming read of the saliency volume (4 B/voxel) into a
// 2048-bin histogram; between passes only the 2048 counters visit the host, which is
// also where a multi-GPU driver all-reduces them (the cut is a global order statistic).
#include "common.cuh"
#include "kernels.cuh"
#include <cmath>

namespace visfd_cuda {

__host__ __device__ __forceinline__ uint32_t key_of_bits(uint32_t u) {
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
uint32_t float_to_key(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  return key_of_bits(u);
}
float key_to_float(uint32_t k) {
  uint32_t u = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
  float f;
  memcpy(&f, &u, 4);
  return f;
}

__device__ __forceinline__ void hist_add(unsigned int *sh, bool valid, uint32_t bin) {
  // warp-uniform bins (long runs of equal saliency, e.g. zeros) cost one atomic
  const unsigned full = 0xffffffffu;
  uint32_t b0 = __shfl_sync(full, bin, 0);
  bool same = __all_sync(full, valid && bin == b0);
  if (same) {
    if ((threadIdx.x & 31) == 0) atomicAdd(&sh[b0], 32u);
  } else if (valid) {
    atomicAdd(&sh[bin], 1u);
  }
}

// One key into the CTA's histogram.  Saliencies cluster in a few bins of the first pass, so lanes of
// a warp that hold the same bin as lane 0 are counted with one atomic (the common long runs: zeros,
// one exponent), the others individually.
__device__ __forceinline__ void hist_add4(unsigned int *sh, const bool valid[4], const uint32_t bin[4]) {
  const unsigned full = 0xffffffffu;
#pragma unroll
  for (int e = 0; e < 4; e++) {
    const uint32_t b0 = __shfl_sync(full, bin[e], 0);
    const unsigned same = __ballot_sync(full, valid[e] && bin[e] == b0);
    if ((threadIdx.x & 31) == 0 && same) atomicAdd(&sh[b0], (unsigned)__popc(same));
    if (valid[e] && bin[e] != b0) atomicAdd(&sh[bin[e]], 1u);
  }
}

// Four consecutive voxels per thread and iteration (one 16-byte load; the ragged tail and unaligned
// volumes go through the scalar path of the last iterations).
__global__ void __launch_bounds__(512)
select_hist_kernel(const float *__restrict__ sal, const float *__restrict__ mask, i64 n,
                   uint32_t prefix, int prefix_bits, int bin_bits,
                   unsigned long long *__restrict__ hist) {
  __shared__ unsigned int sh[HIST_BINS];
  for (int k = threadIdx.x; k < HIST_BINS; k += blockDim.x) sh[k] = 0;
  __syncthreads();
  const int shift = 32 - prefix_bits - bin_bits;
  const uint32_t bin_mask = (1u << bin_bits) - 1u;
  const int pshift = 32 - prefix_bits;            // 32 when there is no prefix yet (never shifted by)
  const bool vec = ((reinterpret_cast<uintptr_t>(sal) | (mask ? reinterpret_cast<uintptr_t>(mask) : 0)) & 15) == 0;
  const i64 n4 = vec ? n / 4 : 0;                 // float4 groups
  const i64 stride = (i64)gridDim.x * blockDim.x;
  // loop bounds are warp-uniform so that the warp collectives are safe
  const i64 n4_round = (n4 + 31) & ~(i64)31;
  for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n4_round; i += stride) {
    bool valid[4] = {false, false, false, false};
    uint32_t bin[4] = {0, 0, 0, 0};
    if (i < n4) {
      const float4 v = __ldg(reinterpret_cast<const float4 *>(sal) + i);
      const uint32_t key[4] = {key_of_bits(__float_as_uint(v.x)), key_of_bits(__float_as_uint(v.y)),
                               key_of_bits(__float_as_uint(v.z)), key_of_bits(__float_as_uint(v.w))};
      float4 m = make_float4(1.f, 1.f, 1.f, 1.f);
      if (mask) m = __ldg(reinterpret_cast<const float4 *>(mask) + i);
      const float mm[4] = {m.x, m.y, m.z, m.w};
#pragma unroll
      for (int e = 0; e < 4; e++) {
        valid[e] = mm[e] != 0.0f && (prefix_bits == 0 || (key[e] >> pshift) == prefix);
        bin[e] = (key[e] >> shift) & bin_mask;
      }
    }
    // later passes: almost nothing matches the prefix any more
    if (!__any_sync(0xffffffffu, valid[0] || valid[1] || valid[2] || valid[3])) continue;
    hist_add4(sh, valid, bin);
  }
  const i64 tail0 = n4 * 4, n_tail = n - tail0;
  const i64 tail_round = (n_tail + 31) & ~(i64)31;
  for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < tail_round; i += stride) {
    bool valid = i < n_tail;
    uint32_t key = 0;
    if (valid) {
      key = key_of_bits(__float_as_uint(__ldg(sal + tail0 + i)));
      if (mask && __ldg(mask + tail0 + i) == 0.0f) valid = false;
      if (prefix_bits > 0 && (key >> pshift) != prefix) valid = false;
    }
    hist_add(sh, valid, (key >> shift) & bin_mask);
  }
  __syncthreads();
  for (int k = threadIdx.x; k < HIST_BINS; k += blockDim.x)
    if (sh[k]) atomicAdd(&hist[k], (unsigned long long)sh[k]);
}

static int bits_for_pass(int prefix_bits) { return (32 - prefix_bits) >= 11 ? 11 : (32 - prefix_bits); }

void select_hist_device(visfd_ctx *ctx, i64 n, const float *sal, const float *mask,
                        uint32_t prefix, int prefix_bits, uint64_t *hist_host) {
  VREQUIRE(prefix_bits >= 0 && prefix_bits < 32, "select: bad prefix length");
  int bin_bits = bits_for_pass(prefix_bits);
  Scratch<unsigned long long> d(ctx, HIST_BINS);
  {
    StageTimer t(ctx, "select");
    VCK(cudaMemsetAsync(d.get(), 0, HIST_BINS * sizeof(unsigned long long), ctx->stream));
    if (n > 0) {
      int grid = (int)std::min<i64>((n + 511) / 512, (i64)ctx->sm_count * 8);
      select_hist_kernel<<<grid, 512, 0, ctx->stream>>>(sal, mask, n, prefix, prefix_bits, bin_bits, d.get());
      VCK(cudaGetLastError());
      ctx->count_launch();
    }
  }
  VCK(cudaMemcpyAsync(hist_host, d.get(), HIST_BINS * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
  VCK(cudaStreamSynchronize(ctx->stream));
}

// One narrowing step on the host.  `rank` = how many keys, among those matching the
// current prefix, are strictly greater than the wanted one (0-based rank in decreasing
// order).  Bins are scanned from the top.
int select_step_host(const uint64_t *hist, uint32_t *prefix, int *prefix_bits, uint64_t *rank) {
  int bin_bits = bits_for_pass(*prefix_bits);
  int nb = 1 << bin_bits;
  uint64_t cum = 0;
  for (int b = nb - 1; b >= 0; b--) {
    if (*rank < cum + hist[b]) {
      *rank -= cum;
      *prefix = (*prefix_bits == 0) ? (uint32_t)b : ((*prefix << bin_bits) | (uint32_t)b);
      *prefix_bits += bin_bits;
      return 0;
    }
    cum += hist[b];
  }
  return 1;  // rank beyond the population
}

float select_threshold(float fraction,
                       const std::function<void(uint32_t prefix, int prefix_bits, uint64_t *hist)> &summed_hist,
                       uint64_t *n_at_or_above) {
  uint64_t hist[HIST_BINS];
  uint32_t prefix = 0;
  int prefix_bits = 0;
  uint64_t rank = 0;
  uint64_t above = 0, equal = 0;   // keys above the threshold's / equal to it
  bool first = true;
  while (prefix_bits < 32) {
    const int bin_bits = bits_for_pass(prefix_bits);
    summed_hist(prefix, prefix_bits, hist);
    if (first) {
      uint64_t total = 0;
      for (int b = 0; b < HIST_BINS; b++) total += hist[b];
      VREQUIRE(total > 0, "saliency cut: no un-masked voxels");
      // handlers.cpp:1779-1782: i = floor(n_voxels * fraction) with a float product.
      // (fraction >= 1 indexes past the end in the reference; clamp to the last element.)
      float prod = (float)total * fraction;
      double fl = std::floor((double)prod);
      if (fl < 0) fl = 0;
      rank = (fl >= (double)total) ? total - 1 : (uint64_t)fl;
      first = false;
    }
    const uint64_t skip = rank;
    int rc = select_step_host(hist, &prefix, &prefix_bits, &rank);
    VREQUIRE(rc == 0, "saliency cut: rank outside the population");
    above += skip - rank;   // the keys of the bins above the chosen one
    equal = hist[prefix & ((1u << bin_bits) - 1u)];
  }
  if (n_at_or_above) *n_at_or_above = above + equal;
  return key_to_float(prefix);
}

float select_threshold_device(visfd_ctx *ctx, i64 n, const float *sal, const float *mask,
                              float fraction) {
  return select_threshold(fraction, [&](uint32_t prefix, int prefix_bits, uint64_t *hist) {
    select_hist_device(ctx, n, sal, mask, prefix, prefix_bits, hist);
  });
}

__global__ void cut_kernel(float *__restrict__ sal, float thr, i64 n) {
  i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
  i64 stride = (i64)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    float v = sal[i];
    if (v < thr) sal[i] = 0.0f;  // handlers.cpp:1792 (ties survive)
  }
}

void apply_cut_device(visfd_ctx *ctx, i64 n, float *sal, float thr) {
  if (n == 0) return;
  StageTimer t(ctx, "select");
  int grid = (int)std::min<i64>((n + 255) / 256, (i64)ctx->sm_count * 16);
  cut_kernel<<<grid, 256, 0, ctx->stream>>>(sal, thr, n);
  VCK(cudaGetLastError());
  ctx->count_launch();
}

// peak_height of `-membrane-background` (handlers.cpp:1698-1702, :1883-1887): score *= source - background, for the
// voxels the reference visits (mask != 0).  bg == NULL: src already holds the peak height.
__global__ void scale_by_peak_kernel(float *__restrict__ score, const float *__restrict__ src, const float *__restrict__ bg,
                                     const float *__restrict__ mask, i64 n) {
  i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
  i64 stride = (i64)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    if (mask && __ldg(mask + i) == 0.0f) continue;
    const float peak = bg ? __fsub_rn(__ldg(src + i), __ldg(bg + i)) : __ldg(src + i);
    score[i] = __fmul_rn(score[i], peak);
  }
}

void scale_by_peak_device(visfd_ctx *ctx, i64 n, float *score, const float *src, const float *background, const float *mask) {
  if (n == 0) return;
  StageTimer t(ctx, "ridge");
  int grid = (int)std::min<i64>((n + 255) / 256, (i64)ctx->sm_count * 16);
  scale_by_peak_kernel<<<grid, 256, 0, ctx->stream>>>(score, src, background, mask, n);
  VCK(cudaGetLastError());
  ctx->count_launch();
}

__global__ void count_unmasked_kernel(const float *__restrict__ mask, i64 n, unsigned long long *out) {
  i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
  i64 stride = (i64)gridDim.x * blockDim.x;
  unsigned long long c = 0;
  for (; i < n; i += stride) c += (__ldg(mask + i) != 0.0f);
  for (int o = 16; o; o >>= 1) c += __shfl_down_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, c);
}

i64 count_unmasked_device(visfd_ctx *ctx, i64 n, const float *mask) {
  if (!mask) return n;
  Scratch<unsigned long long> d(ctx, 1);
  VCK(cudaMemsetAsync(d.get(), 0, sizeof(unsigned long long), ctx->stream));
  int grid = (int)std::min<i64>((n + 255) / 256, (i64)ctx->sm_count * 16);
  if (n > 0) {
    count_unmasked_kernel<<<grid, 256, 0, ctx->stream>>>(mask, n, d.get());
    VCK(cudaGetLastError());
    ctx->count_launch();
  }
  unsigned long long h = 0;
  VCK(cudaMemcpyAsync(&h, d.get(), sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
  VCK(cudaStreamSynchronize(ctx->stream));
  return (i64)h;
}

}  // namespace visfd_cuda
