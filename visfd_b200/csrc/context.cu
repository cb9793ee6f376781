// context.cu -- context lifetime, device workspace pool, stage timing, error state.
#include "common.cuh"
#include <algorithm>
#include <mutex>
#include <stdlib.h>

namespace visfd_cuda {

static thread_local std::string g_last_error;
void set_last_error(const std::string &m) { g_last_error = m; }   // g_last_error is thread_local
const char *get_last_error() { return g_last_error.c_str(); }

bool is_device_pointer(const void *p) {
  if (!p) return false;
  cudaPointerAttributes a;
  cudaError_t e = cudaPointerGetAttributes(&a, p);
  if (e != cudaSuccess) {
    cudaGetLastError();  // clear
    return false;
  }
  return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

StageTimer::StageTimer(visfd_ctx *c, const char *n) : ctx(c), name(n) {
  if (!ctx->timing) return;
  VCK(cudaEventCreate(&a));
  VCK(cudaEventCreate(&b));
  VCK(cudaEventRecord(a, ctx->stream));
}
StageTimer::~StageTimer() {
  if (!a) return;
  cudaEventRecord(b, ctx->stream);
  ctx->pending_events.push_back({name, a, b});
}

void drop_pending_stage_events(visfd_ctx *ctx) {
  for (auto &pe : ctx->pending_events) {
    cudaEventDestroy(pe.a);
    cudaEventDestroy(pe.b);
  }
  ctx->pending_events.clear();
}

void reset_stage_times(visfd_ctx *ctx) {
  drop_pending_stage_events(ctx);
  ctx->stage_ms.clear();
}

void resolve_stage_times(visfd_ctx *ctx) {
  for (auto &pe : ctx->pending_events) {
    float ms = 0.0f;
    if (cudaEventElapsedTime(&ms, pe.a, pe.b) == cudaSuccess) ctx->stage_ms[pe.name] += ms;
    cudaEventDestroy(pe.a);
    cudaEventDestroy(pe.b);
  }
  cudaGetLastError();
  ctx->pending_events.clear();
}

}  // namespace visfd_cuda

using namespace visfd_cuda;

void *visfd_ctx::alloc(size_t bytes) {
  bytes = block_bytes(bytes);
  // best fit among cached blocks that are not wastefully large
  int best = -1;
  for (int i = 0; i < (int)free_blocks.size(); i++) {
    size_t b = free_blocks[i].bytes;
    if (b >= bytes && b <= bytes + bytes / 4 + (1 << 20)) {
      if (best < 0 || b < free_blocks[best].bytes) best = i;
    }
  }
  if (best >= 0) {
    Block blk = free_blocks[best];
    free_blocks.erase(free_blocks.begin() + best);
    live_blocks[blk.p] = blk.bytes;
    return blk.p;
  }
  void *p = nullptr;
  cudaError_t e = cudaMalloc(&p, bytes);
  if (e != cudaSuccess) {
    cudaGetLastError();
    // release the cache (after the stream drained: cached blocks may still be in use
    // by enqueued kernels) and retry once
    cudaStreamSynchronize(stream);
    trim();
    e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) {
      cudaGetLastError();
      throw Error("visfd_cuda: out of device memory allocating " + std::to_string(bytes >> 20) +
                  " MiB (" + cudaGetErrorString(e) + ")");
    }
  }
  live_blocks[p] = bytes;
  reserved_bytes += (int64_t)bytes;
  peak_reserved_bytes = std::max(peak_reserved_bytes, reserved_bytes);
  return p;
}

void visfd_ctx::release(void *p) {
  if (!p) return;
  auto it = live_blocks.find(p);
  if (it == live_blocks.end()) return;
  // Stream-ordered reuse: all work is enqueued on ctx->stream, so a later kernel that
  // receives this block runs after every earlier kernel that used it.
  free_blocks.push_back({p, it->second});
  live_blocks.erase(it);
}

void visfd_ctx::trim() {
  for (auto &b : free_blocks) {
    cudaFree(b.p);
    reserved_bytes -= (int64_t)b.bytes;
  }
  free_blocks.clear();
}

extern "C" {

int visfd_cuda_version(void) { return 1; }

const char *visfd_cuda_last_error(void) { return visfd_cuda::get_last_error(); }

int visfd_cuda_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

int visfd_cuda_init(int device, visfd_ctx **out) {
  try {
    VREQUIRE(out != nullptr, "visfd_cuda_init: ctx pointer is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
      cudaGetLastError();
      throw Error(std::string("visfd_cuda: no usable CUDA device (") +
                  (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") +
                  "); there is no CPU fallback");
    }
    if (device < 0) VCK(cudaGetDevice(&device));
    VREQUIRE(device < count, "visfd_cuda_init: device index out of range");
    VCK(cudaSetDevice(device));
    cudaDeviceProp prop;
    VCK(cudaGetDeviceProperties(&prop, device));
    VREQUIRE(prop.major >= 10,
             "visfd_cuda: this library is built for sm_100a (B200) only; device is sm_" +
                 std::to_string(prop.major) + std::to_string(prop.minor));
    visfd_ctx *c = new visfd_ctx();
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    VCK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    c->own_stream = true;
    const char *fg = getenv("VISFD_CUDA_FAST_GAUSS");
    c->fast_gauss = fg && fg[0] == '1';
    const char *nt = getenv("VISFD_CUDA_NO_TMA");
    c->use_tma = !(nt && nt[0] == '1');
    *out = c;
    return 0;
  } catch (const std::exception &ex) {
    set_last_error(ex.what());
    return 1;
  }
}

void visfd_cuda_destroy(visfd_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  reset_stage_times(ctx);
  ctx->trim();
  for (auto &kv : ctx->live_blocks) cudaFree(kv.first);
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  delete ctx;
}

int visfd_cuda_set_stream(visfd_ctx *ctx, void *cuda_stream) {
  if (!ctx) return 1;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  ctx->stream = (cudaStream_t)cuda_stream;
  ctx->own_stream = false;
  return 0;
}

int visfd_cuda_trim(visfd_ctx *ctx) {
  if (!ctx) return 1;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  ctx->trim();
  return 0;
}

int64_t visfd_cuda_launch_count(visfd_ctx *ctx) { return ctx ? ctx->launches : -1; }

int64_t visfd_cuda_peak_reserved_bytes(visfd_ctx *ctx) { return ctx ? ctx->peak_reserved_bytes : -1; }

void visfd_cuda_reset_peak_reserved_bytes(visfd_ctx *ctx) {
  if (ctx) ctx->peak_reserved_bytes = ctx->reserved_bytes;
}

void visfd_cuda_set_fast_gauss(visfd_ctx *ctx, int enabled) {
  if (ctx) ctx->fast_gauss = enabled != 0;
}

void visfd_cuda_reset_stage_ms(visfd_ctx *ctx) {
  if (ctx) reset_stage_times(ctx);
}

void visfd_cuda_set_timing(visfd_ctx *ctx, int enabled) {
  if (ctx) ctx->timing = enabled != 0;
}

double visfd_cuda_stage_ms(visfd_ctx *ctx, const char *stage) {
  if (!ctx || !stage) return -1.0;
  auto it = ctx->stage_ms.find(stage);
  if (it == ctx->stage_ms.end()) return -1.0;
  return it->second;
}

}  // extern "C"
