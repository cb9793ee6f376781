// common.cuh -- context, error handling, device workspace pool, host<->device staging.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <map>
#include <string>
#include <vector>
#include <stdexcept>

#include "../../include/visfd_cuda.h"

namespace visfd_cuda {

typedef int64_t i64;

struct Error : std::runtime_error {
  explicit Error(const std::string &m) : std::runtime_error(m) {}
};

void set_last_error(const std::string &m);
const char *get_last_error();

#define VCK(call)                                                              \
  do {                                                                         \
    cudaError_t e__ = (call);                                                  \
    if (e__ != cudaSuccess)                                                    \
      throw ::visfd_cuda::Error(std::string(#call) + " failed: " +             \
                                cudaGetErrorString(e__) + " (" __FILE__ ":" +  \
                                std::to_string(__LINE__) + ")");               \
  } while (0)

#define VREQUIRE(cond, msg)                                                    \
  do {                                                                         \
    if (!(cond)) throw ::visfd_cuda::Error(std::string("visfd_cuda: ") + (msg)); \
  } while (0)

}  // namespace visfd_cuda

// Opaque handle of the C ABI.
struct visfd_ctx {
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  cudaStream_t copy_stream = nullptr;       // lazily created: D2H of finished result chunks behind the kernels
  int64_t launches = 0;
  int64_t last_voters = 0;
  int last_tv_kernel = 0;                   // voting kernel of the last call: 0 MUFU, 1 table, 2 table with clamped index
  bool fast_gauss = false;                  // FFMA sweeps instead of the bit-exact mul+add
  bool use_tma = true;                      // stage the sweeps' tiles with TMA (VISFD_CUDA_NO_TMA=1: cp.async)
  bool timing = true;                       // record per-stage CUDA events
  std::map<std::string, double> stage_ms;   // resolved at the end of each API call
  struct PendingEvent { const char *name; cudaEvent_t a, b; };
  std::vector<PendingEvent> pending_events;

  struct Block { void *p; size_t bytes; };
  std::vector<Block> free_blocks;           // cached, not in use
  std::map<void *, size_t> live_blocks;     // handed out
  int64_t reserved_bytes = 0;               // held from cudaMalloc: live + cached
  int64_t peak_reserved_bytes = 0;          // highest reserved_bytes since creation or the last reset

  // What alloc(bytes) takes from the device: requests are rounded up to whole 512-byte units.
  static size_t block_bytes(size_t bytes) { return ((bytes ? bytes : 16) + 511) & ~size_t(511); }
  // Whether alloc serves a request of `bytes` (block_bytes) from a cached block of `cached` bytes.
  static bool reuses(size_t cached, size_t bytes) { return cached >= bytes && cached <= bytes + bytes / 4 + (1 << 20); }
  void *alloc(size_t bytes);
  void release(void *p);
  void trim();
  void count_launch(int n = 1) { launches += n; }
};

namespace visfd_cuda {

// RAII device scratch buffer from the context pool.
template <typename T>
struct Scratch {
  visfd_ctx *ctx = nullptr;
  T *p = nullptr;
  size_t n = 0;
  Scratch() {}
  Scratch(visfd_ctx *c, size_t count) { reset(c, count); }
  void reset(visfd_ctx *c, size_t count) {
    free();
    ctx = c;
    n = count;
    p = count ? static_cast<T *>(c->alloc(count * sizeof(T))) : nullptr;
  }
  void free() {
    if (p && ctx) ctx->release(p);
    p = nullptr;
  }
  ~Scratch() { free(); }
  Scratch(const Scratch &) = delete;
  Scratch &operator=(const Scratch &) = delete;
  T *get() const { return p; }
};

bool is_device_pointer(const void *p);

// Stage timing helper: records CUDA events on the context stream around a scope.
struct StageTimer {
  visfd_ctx *ctx;
  const char *name;
  cudaEvent_t a = nullptr, b = nullptr;
  StageTimer(visfd_ctx *c, const char *n);
  ~StageTimer();
};
void reset_stage_times(visfd_ctx *ctx);
void drop_pending_stage_events(visfd_ctx *ctx);
void resolve_stage_times(visfd_ctx *ctx);  // call after stream sync

// CUDA events with a guaranteed end of life: on scope exit (normal or by exception) both streams of the
// context are drained first, so that copies still in flight on copy_stream cannot write into staging blocks
// the pool has already handed to someone else, and then the events are destroyed.
struct EventList {
  visfd_ctx *ctx;
  std::vector<cudaEvent_t> ev;
  explicit EventList(visfd_ctx *c) : ctx(c) {}
  cudaEvent_t add() {
    cudaEvent_t e;
    VCK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    ev.push_back(e);
    return e;
  }
  ~EventList() {
    if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
    cudaStreamSynchronize(ctx->stream);
    for (cudaEvent_t e : ev) cudaEventDestroy(e);
  }
  EventList(const EventList &) = delete;
  EventList &operator=(const EventList &) = delete;
};

// A user array that may live on the host or on the device.
enum class Dir { In, Out, InOut };
template <typename T>
struct Staged {
  visfd_ctx *ctx = nullptr;
  T *user = nullptr;
  T *dev = nullptr;
  size_t n = 0;
  bool host = false;
  Dir dir = Dir::In;
  Staged() {}
  Staged(visfd_ctx *c, const T *ptr, size_t count, Dir d, bool is_host) {
    init(c, const_cast<T *>(ptr), count, d, is_host);
  }
  void init(visfd_ctx *c, T *ptr, size_t count, Dir d, bool is_host) {
    ctx = c; user = ptr; n = count; dir = d; host = is_host && ptr != nullptr;
    if (!ptr) { dev = nullptr; return; }
    if (!host) { dev = ptr; return; }
    dev = static_cast<T *>(c->alloc(count * sizeof(T)));
    if (d != Dir::Out) {
      StageTimer t(c, "h2d");
      VCK(cudaMemcpyAsync(dev, user, count * sizeof(T), cudaMemcpyHostToDevice, c->stream));
    }
  }
  bool delivered = false;  // the producer already copied the result to the user's array
  void finish() {  // copy results back (outputs only)
    if (host && dev && dir != Dir::In && !delivered) {
      StageTimer t(ctx, "d2h");
      VCK(cudaMemcpyAsync(user, dev, n * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
    }
  }
  ~Staged() {
    if (host && dev) ctx->release(dev);
  }
  Staged(const Staged &) = delete;
  Staged &operator=(const Staged &) = delete;
  T *get() const { return dev; }
};

static inline unsigned div_up(i64 a, i64 b) { return (unsigned)((a + b - 1) / b); }

}  // namespace visfd_cuda
