// common.cuh -- shared host/device helpers of librlvi_b200 (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/rlvi_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "librlvi_b200 is written for sm_100a (B200); compile with -gencode arch=compute_100a,code=sm_100a"
#endif

// ---------------------------------------------------------------------------------------------
// context + error plumbing (host)
// ---------------------------------------------------------------------------------------------
struct rlvi_ctx {
  int device;
  int sm_count;
  int64_t launches;
  void* scratch;         // device scratch for reduction partials, barriers, small results
  size_t scratch_bytes;
  void* big;             // device-resident copy of host inputs (rlvi_em_step_logistic_host)
  size_t big_bytes;
  void* pinned;          // small pinned staging buffer
  size_t pinned_bytes;
  cudaStream_t copy_stream;
  cudaEvent_t ev[4];
};

void rlvi_set_error(const char* fmt, ...);
int rlvi_scratch(rlvi_ctx* ctx, size_t bytes, void** out);   // grows ctx->scratch if needed

// Scratch header: the first kScratchHeaderBytes of ctx->scratch, zero when allocated.  Byte offsets:
//   [0, 64)       control words.  The fixed point uses [1] as its failure flag; stats_allreduce (dist.cu) uses [0] as
//                 its ticket and [1] as its failure flag.  Each launcher clears them before its launch.
//   [128, 132)    the ticket of grid_total.  Left at zero by every kernel that takes it (the last block resets it).
//   [256, 448)    the fixed point's local LL window when world == 1 (4 slots x 6 LL words), cleared by its launcher.
//   [2048, 2064)  the TF32 Gram's error flag (u32) and, at 2056, the weight maximum (u64), cleared by its launcher.
//   [4096, ...)   per-launch partials.
constexpr size_t kScratchControlBytes = 64;
constexpr size_t kScratchTicket = 128;
constexpr size_t kScratchFpWindow = 256;
constexpr size_t kScratchTf32Err = 2048;
constexpr size_t kScratchTf32Wmax = 2056;
constexpr size_t kScratchHeaderBytes = 4096;

struct RlviScratch {
  unsigned int* control;
  unsigned int* ticket;
  double* fp_window;
  unsigned int* tf32_err;
  unsigned long long* tf32_wmax;
  double* partials;
};

// Scratch for the header plus `partial_bytes` of partials, as typed pointers (valid until the next rlvi_scratch call).
static inline int rlvi_scratch_header(rlvi_ctx* ctx, size_t partial_bytes, RlviScratch* out) {
  void* scratch = nullptr;
  const int rc = rlvi_scratch(ctx, kScratchHeaderBytes + partial_bytes, &scratch);
  if (rc != RLVI_OK) return rc;
  char* base = static_cast<char*>(scratch);
  out->control = reinterpret_cast<unsigned int*>(base);
  out->ticket = reinterpret_cast<unsigned int*>(base + kScratchTicket);
  out->fp_window = reinterpret_cast<double*>(base + kScratchFpWindow);
  out->tf32_err = reinterpret_cast<unsigned int*>(base + kScratchTf32Err);
  out->tf32_wmax = reinterpret_cast<unsigned long long*>(base + kScratchTf32Wmax);
  out->partials = reinterpret_cast<double*>(base + kScratchHeaderBytes);
  return RLVI_OK;
}

// Grid for a 256-thread grid-stride pass of about `per_thread` elements per thread, capped at 8 CTAs per SM.
static inline int grid_for(const rlvi_ctx* ctx, int64_t n, int per_thread) {
  int64_t want = (n + 256 * per_thread - 1) / (256 * per_thread);
  const int64_t cap = int64_t(ctx->sm_count) * 8;
  return int(want < 1 ? 1 : (want > cap ? cap : want));
}

// gram_tma.cu: general-d Gram on the FP64 tensor pipe; RLVI_ERR_UNSUPPORTED = shape not covered (fall back)
int rlvi_gram_tma_f64(rlvi_ctx* ctx, const double* X, const double* y, const double* weights, const double* center,
                      int64_t n, int d, int power, int want_gram, double* out, cudaStream_t st);

#define RLVI_CUDA(expr)                                                                   \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess) {                                                              \
      rlvi_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return RLVI_ERR_CUDA;                                                               \
    }                                                                                     \
  } while (0)

#define RLVI_REQUIRE(cond, msg)                                      \
  do {                                                               \
    if (!(cond)) {                                                   \
      rlvi_set_error("%s: %s (%s)", __func__, msg, #cond);           \
      return RLVI_ERR_INVALID;                                       \
    }                                                                \
  } while (0)

#define RLVI_LAUNCH_CHECK(ctx)                                                      \
  do {                                                                              \
    cudaError_t _e = cudaGetLastError();                                            \
    if (_e != cudaSuccess) {                                                        \
      rlvi_set_error("%s:%d: kernel launch -> %s", __FILE__, __LINE__, cudaGetErrorString(_e)); \
      return RLVI_ERR_CUDA;                                                         \
    }                                                                               \
    (ctx)->launches++;                                                              \
  } while (0)

static inline bool rlvi_aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// RAII device guard so the library never changes the caller's current device.
struct RlviDeviceGuard {
  int prev;
  bool changed;
  explicit RlviDeviceGuard(int dev) : prev(-1), changed(false) {
    if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) {
      cudaSetDevice(dev);
      changed = true;
    }
  }
  ~RlviDeviceGuard() {
    if (changed) cudaSetDevice(prev);
  }
};

// ---------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------
#ifdef __CUDACC__

constexpr int kWarp = 32;

// Streaming 128-bit loads: read-only path, do not allocate in L1 (every byte is used once).
__device__ __forceinline__ double2 ld_stream_d2(const double* p) {
  double2 r;
  asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0, %1}, [%2];" : "=d"(r.x), "=d"(r.y) : "l"(p));
  return r;
}
__device__ __forceinline__ double ld_stream_d1(const double* p) {
  double r;
  asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(r) : "l"(p));
  return r;
}
__device__ __forceinline__ float4 ld_stream_f4(const float* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Block-wide sum of NV values per thread.  Fixed order: xor-shuffle tree inside each warp, then
// warp 0 adds the per-warp partials in warp order.  Result valid in thread 0.
// `smem` must hold NV * (blockDim.x / 32) doubles.  Contains two __syncthreads().
template <int NV>
__device__ __forceinline__ void block_sum(double (&v)[NV], double* smem) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = warp_sum(v[i]);
  __syncthreads();   // protect smem reuse across consecutive calls
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < NV; ++i) smem[i * nwarp + warp] = v[i];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      double s = 0.0;
      for (int w = 0; w < nwarp; ++w) s += smem[i * nwarp + w];
      v[i] = s;
    }
  }
}

// "Last block finishes" ticket: returns true in ALL threads of the block that arrives last.
// `counter` must be zero before the launch and is reset to zero by the last block, so the same
// counter can be reused by the next launch on the stream.
__device__ __forceinline__ bool last_block_ticket(unsigned int* counter, unsigned int nblocks) {
  __shared__ unsigned int s_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned int t = atomicAdd(counter, 1u);
    s_last = (t == nblocks - 1) ? 1u : 0u;
    if (s_last) *counter = 0u;
  }
  __syncthreads();
  if (s_last) __threadfence();
  return s_last != 0u;
}

// Deterministic cross-block sum of NV values, called by every thread of the grid.  Thread 0 holds the block's totals
// in `v`; they are stored as partials[block][NV].  Returns true in lane 0 of warp 0 of the block that arrives last,
// with `v` holding the grid totals.  Fixed order: lane j adds partials j, j + 32, ... in increasing order, then the
// warp_sum xor tree.  `ticket` is the scratch header's ticket.
template <int NV>
__device__ __forceinline__ bool grid_total(double (&v)[NV], double* partials, unsigned int* ticket) {
  if (threadIdx.x == 0) {
#pragma unroll
    for (int i = 0; i < NV; ++i) partials[NV * blockIdx.x + i] = v[i];
  }
  if (!last_block_ticket(ticket, gridDim.x) || threadIdx.x >= 32) return false;
  double a[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) a[i] = 0.0;
  for (unsigned int j = threadIdx.x; j < gridDim.x; j += 32) {
#pragma unroll
    for (int i = 0; i < NV; ++i) a[i] += partials[NV * j + i];
  }
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = warp_sum(a[i]);
  return threadIdx.x == 0;
}

#endif  // __CUDACC__
