// fixed_point.cu -- the epsilon fixed point of the E-step as ONE persistent cooperative kernel.
//
// Replaces the Python loops of
//   standard-learning/rlvi.py:8-20        (update_weights,          RLVI_FP_STANDARD, FP64)
//   online-learning/main.py:45-58         (update_weights_rlvi,     RLVI_FP_ONLINE,   FP64)
//   deep-learning/methods/train_rlvi.py:14-38 (update_sample_weights, RLVI_FP_DEEP,   FP32)
// which launch ~10 array operations (and, on the GPU path, one host sync) per pass.
//
// Design (SURVEY.md H2): the posterior of pass k is a function of (e_i, rho_k) only, so no pi array
// is kept between passes.  Pass 1 reads the losses, writes e_i = exp(-s*l_i) once, and every later
// pass streams ONLY e (8 B/sample FP64) while accumulating  S = sum pi'  and  E = sum (pi' - pi)^2
// with pi recomputed from the previous rho.  The scalar recurrence (eps, rho, stop test) is evaluated
// redundantly by every block from the same bits, in the reference's FP64 operation order, so the
// loop exits on the device without a host round trip.  A final pass writes pi.
//
// Cross-block reduction is deterministic, two hops, no atomics: block partials as self-validating "LL" words ->
// block 0 sums them in a fixed order and publishes the rank's totals as LL words (to a local window, or with
// `dist` set to every peer's inbox over NVLink) -> all blocks poll their own window (which is the grid barrier)
// and add the `world` slots in rank order, so every block of every rank sees identical totals and takes the
// same stop decision.
//
// How the later passes get e[] (fp_cache_slots): up to 2^22 samples per GPU the head of the vector stays in shared
// memory and the rest comes from L2 with per-thread loads; above that every warp streams its own contiguous segment
// through a private ring of bulk copies (the TMA engine runs ahead of the arithmetic; each pass arms the next pass's
// first copies before the grid reduction; the head of an HBM-sized vector is kept in L2 by cache hints).
// Series passes (STANDARD): once rho dominates max e, a pass takes its two sums from power sums of e built once per call
// (series_sums) and reads no e at all; only the passes before that switch, and the final pass, stream the vector.
// RLVI_FP_TRACE=1 prints the per-round timeline of a call (profiles/r02_fixed_point_trace.txt).
#include <math.h>
#include <stdlib.h>

#include "tma.cuh"

namespace {

constexpr int kFpThreads = 256;
constexpr int kFpUnroll = 8;            // independent 128-bit loads in flight per thread
constexpr int kFpCacheSlots = 24;       // whole trips: 24 x 256 x 16 B = 96 KiB of e[] per CTA stay in shared memory (2 CTAs/SM)
constexpr unsigned long long kSpinTimeoutNs = 20ull * 1000ull * 1000ull * 1000ull;
// Series passes (STANDARD, VEC): power sums P_j = sum z^j, z = e / 2^E, j = 1..kFpSeriesJ, built once per call.  They
// travel through the grid reduction as (kFpSeriesJ + 1) / 3 rounds of three values: the power sums and, last, min z.
constexpr int kFpSeriesJ = 17;
static_assert(kFpSeriesJ % 3 == 2, "the power sums and min z fill whole reduction rounds");

enum ReduceOp { OP_SUM = 0, OP_MIN = 1, OP_MAX = 2 };

template <typename T>
struct FpParams {
  const T* losses;        // STANDARD/ONLINE: losses or NULL; DEEP: unused (residuals is in/out)
  const double* scale;    // device scalar or NULL
  T* e;                   // scratch e_i
  T* pi_out;              // STANDARD/ONLINE output; DEEP: weights (in/out)
  T* residuals;           // DEEP only (in/out)
  int64_t n;
  int64_t n_global;
  double tol;
  int maxiter;
  double* partials;       // [2][grid][6] LL words (two per double)
  unsigned int* control;  // [1] failure flag
  rlvi_fp_result* result;
  int rank, world;
  double* inbox;
  double* const* peer_inbox;
  unsigned long long call_index;
  int cache_slots;        // FP64 VEC kernels: chunks per thread kept in shared memory
  int l2_head;            // ring mode: keep the head of the vector L2-resident across passes (cache-hinted bulk copies)
  double pi0;             // initial posterior; 0 = the variant's constant (0.95 / 0.5)
  int series;             // STANDARD, VEC: allow series passes (RLVI_FP_SERIES=0 forces streaming)
  unsigned long long* trace;   // bring-up only (RLVI_FP_TRACE=1): [round][grid][4] globaltimer stamps, else NULL
};
constexpr int kFpTraceRounds = 64;

__device__ __forceinline__ unsigned long long gtime_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ unsigned int ld_acquire_u32(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_gpu_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ double ld_volatile_f64(const double* p) {
  double v;
  asm volatile("ld.volatile.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
  return v;
}

struct FpShared {
  double warp_part[3 * (kFpThreads / 32)];
  double total[3];
  int failed;
};

// ---- "LL" words (the idea of NCCL's low-latency protocol): 8 bytes = 32 bits of payload + a 32-bit sequence tag,
// written with ONE store and read with ONE load, so a word is either old or complete and needs no fence, flag or
// atomic around it.  A double travels as two words (low half, high half); a reader spins until both carry the tag.
__device__ __forceinline__ void st_ll(unsigned long long* p, double v, unsigned int tag, bool sys) {
  const unsigned long long b = (unsigned long long)__double_as_longlong(v);
  const unsigned long long w0 = (b & 0xffffffffull) | ((unsigned long long)tag << 32);
  const unsigned long long w1 = (b >> 32) | ((unsigned long long)tag << 32);
  if (sys) asm volatile("st.relaxed.sys.global.v2.u64 [%0], {%1, %2};" ::"l"(p), "l"(w0), "l"(w1) : "memory");
  else asm volatile("st.relaxed.gpu.global.v2.u64 [%0], {%1, %2};" ::"l"(p), "l"(w0), "l"(w1) : "memory");
}
// true when both words of the double at p carry `tag`
__device__ __forceinline__ bool ld_ll(const unsigned long long* p, unsigned int tag, bool sys, double& v) {
  unsigned long long w0, w1;
  if (sys) asm volatile("ld.relaxed.sys.global.v2.u64 {%0, %1}, [%2];" : "=l"(w0), "=l"(w1) : "l"(p) : "memory");
  else asm volatile("ld.relaxed.gpu.global.v2.u64 {%0, %1}, [%2];" : "=l"(w0), "=l"(w1) : "l"(p) : "memory");
  v = __longlong_as_double((long long)((w0 & 0xffffffffull) | (w1 << 32)));
  return (unsigned int)(w0 >> 32) == tag && (unsigned int)(w1 >> 32) == tag;
}

// Grid-wide (and, with dist, cross-GPU) reduction of three values; v2 uses OP2.  On return all threads
// of all blocks (of all ranks) hold the same totals.  `round` counts reduction rounds and is advanced here.
// Returns false if a wait timed out (a peer died / launch was not co-resident).
//
// Two hops, no atomics, no fences on the critical path: every block stores its partial as LL words; BLOCK 0 of the rank
// gathers them (all its threads poll, block j by thread j mod 256; fixed summation order) and stores the rank's totals
// as LL words into slot `rank` of every rank's window (over NVLink for the peers; world == 1 uses a local window in
// the context scratch); every block then polls its own window for the `world` totals -- which is also the grid
// barrier -- and adds them in rank order, so all blocks of all ranks hold the same bits.  (Round 1 of the build passed
// through the last-arriving block with a ticket atomic, __threadfence and a release/acquire flag.)
// PUBLISH: the reduction must also make the blocks' earlier global writes visible to each other (pass 1 of the
// fixed point writes e[], which the bulk-copy ring of other warps reads later): one fence on each side.
template <typename T, int OP2, bool PUBLISH>
__device__ bool grid_allreduce3(const FpParams<T>& p, FpShared& sh, double& v0, double& v1, double& v2,
                                unsigned int& round) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int NW = kFpThreads / 32;
  const bool sys = p.world > 1;
  if (p.trace && round < kFpTraceRounds && threadIdx.x == 0)
    p.trace[(size_t(round) * gridDim.x + blockIdx.x) * 4 + 0] = gtime_ns();
  const unsigned int buf = round & 1u;
  const unsigned int tag = (unsigned int)((p.call_index << 12) + round + 1ull);     // never 0: round + 1 in [1, 4096)
  unsigned long long* part = reinterpret_cast<unsigned long long*>(p.partials) + size_t(buf) * gridDim.x * 6;
  // window slot: two per call parity and two per round parity, so a fast rank that already started the NEXT round / call
  // can never overwrite a slot a slow rank has not read yet (a rank is at most one published round ahead of any peer)
  const size_t slot = (size_t(((p.call_index & 1ull) << 1) | buf) * p.world) * 6;
  // ---- block stage: fixed xor tree per warp, then warp partials in warp order
  v0 = warp_sum(v0);
  v1 = warp_sum(v1);
  v2 = (OP2 == OP_SUM) ? warp_sum(v2) : (OP2 == OP_MIN ? warp_min(v2) : warp_max(v2));
  __syncthreads();
  if (lane == 0) {
    sh.warp_part[warp] = v0;
    sh.warp_part[NW + warp] = v1;
    sh.warp_part[2 * NW + warp] = v2;
  }
  if (threadIdx.x == 0) sh.failed = 0;
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0.0, b = 0.0, c = sh.warp_part[2 * NW];
    for (int w = 0; w < NW; ++w) {
      a += sh.warp_part[w];
      b += sh.warp_part[NW + w];
      const double t = sh.warp_part[2 * NW + w];
      c = (OP2 == OP_SUM) ? (w == 0 ? t : c + t) : (OP2 == OP_MIN ? fmin(c, t) : fmax(c, t));
    }
    if (PUBLISH) __threadfence();        // this block's global writes (ordered before by the barrier) first
    unsigned long long* mine = part + size_t(blockIdx.x) * 6;
    st_ll(mine + 0, a, tag, false);
    st_ll(mine + 2, b, tag, false);
    st_ll(mine + 4, c, tag, false);
    if (p.trace && round < kFpTraceRounds) p.trace[(size_t(round) * gridDim.x + blockIdx.x) * 4 + 1] = gtime_ns();
  }
  if (blockIdx.x == 0) {
    // ---- block 0 gathers the block partials (thread t: blocks t, t + 256, ...) and sums them in a fixed order; the
    // timeout clock is read on the slow path only (a %globaltimer read per partial sat on every pass's critical path)
    double a = 0.0, b = 0.0;
    double c = (OP2 == OP_SUM) ? 0.0 : (OP2 == OP_MIN ? INFINITY : -INFINITY);
    int failed = 0;
    for (unsigned int j = threadIdx.x; j < gridDim.x && !failed; j += 2 * kFpThreads) {
      // two partials per thread and sweep (blocks j and j + 256), polled TOGETHER: the blocks beyond the first 256 tend
      // to arrive last, and polling them only after the thread's first partial put a second L2 round trip on the path
      const bool two = j + kFpThreads < gridDim.x;
      const unsigned long long* src = part + size_t(j) * 6;
      const unsigned long long* src2 = two ? part + size_t(j + kFpThreads) * 6 : src;
      double x0, x1, x2, y0, y1, y2;
      unsigned long long t0 = 0ull;
      unsigned int spins = 0;
      for (;;) {
        const bool k0 = ld_ll(src + 0, tag, false, x0), k1 = ld_ll(src + 2, tag, false, x1), k2 = ld_ll(src + 4, tag, false, x2);
        const bool m0 = ld_ll(src2 + 0, tag, false, y0), m1 = ld_ll(src2 + 2, tag, false, y1), m2 = ld_ll(src2 + 4, tag, false, y2);
        if (k0 && k1 && k2 && m0 && m1 && m2) break;
        if ((++spins & 63u) == 0u) {
          if (ld_acquire_u32(p.control + 1) != 0u) { failed = 1; break; }
          const unsigned long long now = gtime_ns();
          if (t0 == 0ull) t0 = now;
          if (now - t0 > kSpinTimeoutNs) { atomicExch(p.control + 1, 1u); failed = 1; break; }
        }
      }
      if (!failed) {
        a += x0;
        b += x1;
        c = (OP2 == OP_SUM) ? c + x2 : (OP2 == OP_MIN ? fmin(c, x2) : fmax(c, x2));
        if (two) {
          a += y0;
          b += y1;
          c = (OP2 == OP_SUM) ? c + y2 : (OP2 == OP_MIN ? fmin(c, y2) : fmax(c, y2));
        }
      }
    }
    a = warp_sum(a);
    b = warp_sum(b);
    c = (OP2 == OP_SUM) ? warp_sum(c) : (OP2 == OP_MIN ? warp_min(c) : warp_max(c));
    if (failed) sh.failed = 1;
    __syncthreads();                     // warp_part was consumed by thread 0 above
    if (lane == 0) {
      sh.warp_part[warp] = a;
      sh.warp_part[NW + warp] = b;
      sh.warp_part[2 * NW + warp] = c;
    }
    __syncthreads();
    if (warp == 0 && !sh.failed) {
      double ta = 0.0, tb = 0.0, tc = sh.warp_part[2 * NW];
      for (int w = 0; w < NW; ++w) {
        ta += sh.warp_part[w];
        tb += sh.warp_part[NW + w];
        const double t = sh.warp_part[2 * NW + w];
        tc = (OP2 == OP_SUM) ? (w == 0 ? t : tc + t) : (OP2 == OP_MIN ? fmin(tc, t) : fmax(tc, t));
      }
      // ---- ... and publishes the rank's totals to every rank's window (lane r -> rank r)
      if (PUBLISH) __threadfence();
      for (int r = lane; r < p.world; r += 32) {
        unsigned long long* dst =
            reinterpret_cast<unsigned long long*>(p.world > 1 ? p.peer_inbox[r] : p.inbox) + slot + size_t(p.rank) * 6;
        st_ll(dst + 0, ta, tag, sys);
        st_ll(dst + 2, tb, tag, sys);
        st_ll(dst + 4, tc, tag, sys);
      }
      if (p.trace && round < kFpTraceRounds && lane == 0) p.trace[(size_t(round) * gridDim.x) * 4 + 2] = gtime_ns();
    }
  }
  if (warp == 0) {
    // ---- every block: wait for the `world` totals in its own window, add them in rank order
    double ra = 0.0, rb = 0.0, rc = 0.0;
    int failed = 0;
    if (lane < p.world) {
      const unsigned long long* src = reinterpret_cast<const unsigned long long*>(p.inbox) + slot + size_t(lane) * 6;
      unsigned long long t0 = 0ull;        // the timeout clock is read on the slow path only
      unsigned int spins = 0;
      for (;;) {
        const bool k0 = ld_ll(src + 0, tag, sys, ra), k1 = ld_ll(src + 2, tag, sys, rb), k2 = ld_ll(src + 4, tag, sys, rc);
        if (k0 && k1 && k2) break;
        if ((++spins & 63u) == 0u) {
          if (ld_acquire_u32(p.control + 1) != 0u) { failed = 1; break; }
          const unsigned long long now = gtime_ns();
          if (t0 == 0ull) t0 = now;
          if (now - t0 > kSpinTimeoutNs) { atomicExch(p.control + 1, 1u); failed = 1; break; }
        }
      }
    }
    failed = __any_sync(0xffffffffu, failed);
    if (PUBLISH) __threadfence();        // acquire side: the other blocks' writes are visible to this block from here on
    double a = 0.0, b = 0.0;
    double c = (OP2 == OP_SUM) ? 0.0 : (OP2 == OP_MIN ? INFINITY : -INFINITY);
    for (int r = 0; r < p.world; ++r) {      // rank-ordered sequential sum (world <= 32), same bits everywhere
      a += __shfl_sync(0xffffffffu, ra, r);
      b += __shfl_sync(0xffffffffu, rb, r);
      const double t = __shfl_sync(0xffffffffu, rc, r);
      c = (OP2 == OP_SUM) ? c + t : (OP2 == OP_MIN ? fmin(c, t) : fmax(c, t));
    }
    if (lane == 0) {
      sh.total[0] = a;
      sh.total[1] = b;
      sh.total[2] = c;
      if (failed) sh.failed = 1;
    }
  }
  __syncthreads();
  if (p.trace && round < kFpTraceRounds && threadIdx.x == 0)
    p.trace[(size_t(round) * gridDim.x + blockIdx.x) * 4 + 3] = gtime_ns();
  v0 = sh.total[0];
  v1 = sh.total[1];
  v2 = sh.total[2];
  round += 1u;
  return sh.failed == 0;
}

// ---- vector access helpers ---------------------------------------------------------------------
template <typename T> struct Vec;
template <> struct Vec<double> {
  static constexpr int W = 2;
  typedef double2 type;
  __device__ static void load(const double* p, double (&o)[2]) { double2 v = *reinterpret_cast<const double2*>(p); o[0] = v.x; o[1] = v.y; }
  __device__ static void store(double* p, const double (&o)[2]) { *reinterpret_cast<double2*>(p) = make_double2(o[0], o[1]); }
};
template <> struct Vec<float> {
  static constexpr int W = 4;
  typedef float4 type;
  __device__ static void load(const float* p, float (&o)[4]) { float4 v = *reinterpret_cast<const float4*>(p); o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w; }
  __device__ static void store(float* p, const float (&o)[4]) { *reinterpret_cast<float4*>(p) = make_float4(o[0], o[1], o[2], o[3]); }
};

// Load / store one chunk of W = (VEC ? Vec<T>::W : 1) consecutive elements starting at i; elements
// at or past n read as `fill` and are not written.
template <typename T, bool VEC, int W>
__device__ __forceinline__ void load_chunk(const T* p, int64_t i, int64_t n, T (&o)[W], T fill) {
  if constexpr (VEC) {
    if (i + W <= n) {
      Vec<T>::load(p + i, o);
      return;
    }
  }
#pragma unroll
  for (int j = 0; j < W; ++j) o[j] = (i + j < n) ? p[i + j] : fill;
}
template <typename T, bool VEC, int W>
__device__ __forceinline__ void store_chunk(T* p, int64_t i, int64_t n, const T (&o)[W]) {
  if constexpr (VEC) {
    if (i + W <= n) {
      Vec<T>::store(p + i, o);
      return;
    }
  }
#pragma unroll
  for (int j = 0; j < W; ++j)
    if (i + j < n) p[i + j] = o[j];
}

// Apply F(index, nvalid, ptr-relative lambda) over [0, n) with a grid-stride loop of vector chunks.
// VEC: all arrays are 16-byte aligned -> 128-bit accesses, kFpUnroll chunks per thread per trip.
template <typename T, bool VEC, typename F>
__device__ __forceinline__ void for_each_chunk(int64_t n, F&& f) {
  constexpr int W = VEC ? Vec<T>::W : 1;
  const int64_t nchunks = (n + W - 1) / W;
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  int64_t c = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  // unrolled main part: kFpUnroll independent chunks per trip
  for (; c + (kFpUnroll - 1) * stride < nchunks; c += kFpUnroll * stride) {
#pragma unroll
    for (int u = 0; u < kFpUnroll; ++u) f(c + u * stride, u);
  }
  for (; c < nchunks; c += stride) f(c, 0);
}

// posterior formulas ------------------------------------------------------------------------------
// STANDARD: pi = e / (rho + e)            (rlvi.py:15)
// ONLINE/DEEP: pi = rho e / (1 + rho e)   (online main.py:52, train_rlvi.py:31)
template <int VARIANT>
__device__ __forceinline__ double post_f64(double e, double rho) {
  if (VARIANT == RLVI_FP_STANDARD) return e / (rho + e);
  const double a = rho * e;
  return a / (1.0 + a);
}

// 1/x for x in the normal range to <= 1 ulp: MUFU.RCP64H seed r0 (relative error d ~ 2^-20), then ONE
// second-order correction  r = r0 (1 + d + d^2)  -- 3 dependent DFMA, residual d^3 ~ 2^-60 -- instead of two
// Newton steps (4 DFMA).  The IEEE division the compiler emits for `e / prod` is ~25 instructions with a slow
// path; the hot pass is bound by FP64 issue (tools/ubench_fp.cu: realistic DFMA/DADD/DMUL mixes run at about half
// the DFMA peak because of operand bandwidth), so every FP64 instruction per sample counts.
__device__ __forceinline__ double rcp_fast(double x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  const double d = fma(-x, r, 1.0);
  const double s = fma(d, d, d);
  return fma(r, s, r);
}

// pi' and (pi' - pi) with the reference's own two IEEE divisions (scalar / unaligned path, loop tails and
// the out-of-range fallback of the fast path below).
template <int VARIANT>
__device__ __forceinline__ void post_pair_f64(double e, double rho_new, double rho_old, double& pnew, double& diff) {
  pnew = post_f64<VARIANT>(e, rho_new);
  diff = pnew - post_f64<VARIANT>(e, rho_old);
}

// The hot pass (k >= 2) over a 16-byte aligned e[]: kFpUnroll independent 128-bit loads are issued
// before any arithmetic so that ~128 B per thread are in flight; two accumulator pairs halve the DADD/DFMA
// dependency chains.  Loads bypass L1 (every byte is used once per pass; at <= 64 MiB per GPU the vector
// stays L2 resident between passes).  Each thread re-reads exactly the chunks it wrote in pass 1.
__device__ __forceinline__ double2 ld_e2(const double2* p) {
  double2 r;
  asm volatile("ld.global.L1::no_allocate.v2.f64 {%0, %1}, [%2];" : "=d"(r.x), "=d"(r.y) : "l"(p) : "memory");
  return r;
}
// On-chip residency of e[] between passes: the first `slots` chunks of every thread (chunk ordinal =
// 8 trip + u) are kept in shared memory (filled during pass 1), the rest is re-read from L2 / HBM.  At 8 GPUs a
// shard is 64 MiB and ~40 % of it fits the 148 x ~216 KB of shared memory, which cuts the L2 traffic of the
// L2-bound passes by that much; the values are identical to the global ones, so results do not change.
struct ECache {
  double2* buf;    // cache: [slots][blockDim.x]; ring: [kFpRingDepth][kFpUnroll][blockDim.x]
  int slots;       // > 0: the first `slots` chunks of every thread are resident (small shards)
  int ring;        // != 0: the buffer is a per-WARP TMA prefetch ring instead (HBM-sized vectors)
  uint64_t* bars;  // ring mode: [warps][kFpRingDepth] mbarriers (kernel lifetime; phases persist across passes)
  uint32_t phase;  // ring mode: bit s = parity to wait for on this warp's slot s
  int armed;       // ring mode: slots 0 .. armed - 1 already hold (or are receiving) the NEXT pass's first trips: e[] does not
                   // change after pass 1, so a pass ends by issuing the next pass's first copies and their latency runs
                   // under the grid reduction instead of in front of the first trip
  // ring mode, L2 residency: the vector (512 MiB at the headline shape) is streamed once per pass and plain LRU keeps
  // none of it in the 126 MB L2.  The first `head_trips` trips of every warp's segment (~75 MiB in all) are loaded under
  // an L2 evict_last policy, the rest under evict_first, so that head is served from L2 in every pass after the first
  // (measured in isolation, tools/ubench_l2hint.cu: 80.7 -> 72.9 us per pass)
  int head_trips;
  uint64_t pol_last, pol_first;
};
constexpr int64_t kFpL2HeadBytes = int64_t(76) << 20;

__device__ __forceinline__ void bulk_g2s_hint(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar, uint64_t pol) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
          smem_u32(dst_smem)),
      "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)), "l"(pol)
      : "memory");
}
constexpr int kFpRingDepth = 3;   // 4 KiB slots per warp (8 warps x 3 x 4 KiB = 96 KiB per CTA)

__device__ __forceinline__ double2 ld_e2c(const ECache& ec, int slot, const double2* gptr) {
  return (slot < ec.slots) ? ec.buf[slot * kFpThreads + threadIdx.x] : ld_e2(gptr);
}

// Branch-free fast evaluation of one trip (kFpUnroll chunks of two samples).  The issue slots are what bounds
// the hot pass (ncu: 27 warp-instructions per sample and pass, 11 of them FP64 at half issue rate), so:
//   * no per-sample range test -- an operand at the low end of rcp_fast's domain (0, a denormal product) or an
//     infinite one (rho = inf, an overflowed product) surfaces as a NaN / inf in the trip's sums, which the caller
//     tests ONCE per trip and then redoes the trip with the IEEE divisions.  The high end does not: .ftz flushes
//     1/x to a finite 0 for x in [2^1022, 2^1024), so fp_kernel_f64 tests the largest argument of a pass once
//     (rcp_fast_in_range) and takes the IEEE path for the whole pass when it is that large;
//   * STANDARD accumulates sum t^2 and the caller multiplies by (rho_old - rho_new)^2 once per pass
//     (pi' - pi = t (rho_old - rho_new)): one DMUL per sample less.
// q2 = sum t^2 (STANDARD) or sum (pi' - pi)^2 (ONLINE).
template <int VARIANT>
__device__ __forceinline__ void trip_fast(const double2 (&v)[kFpUnroll], double rho_new, double rho_old, double& t1a,
                                          double& t1b, double& q2a, double& q2b) {
  auto one = [&](double e, double& t1, double& q2) {
    if (VARIANT == RLVI_FP_STANDARD) {
      const double b = rho_old + e;
      const double t = e * rcp_fast((rho_new + e) * b);
      t1 = fma(t, b, t1);                  // pi' = t (rho_old + e)
      q2 = fma(t, t, q2);
    } else {
      const double a = rho_new * e, b = rho_old * e;
      const double b1 = 1.0 + b;
      const double t = rcp_fast((1.0 + a) * b1);
      const double d = (a - b) * t;
      t1 = fma(a * b1, t, t1);
      q2 = fma(d, d, q2);
    }
  };
#pragma unroll
  for (int u = 0; u < kFpUnroll; ++u) {
    one(v[u].x, t1a, q2a);
    one(v[u].y, t1b, q2b);
  }
}
// STANDARD only: the trip WITHOUT the stop-test sum -- sum pi' alone, pi' = e / (rho' + e): 5 FP64 instructions per
// sample instead of 10.  Used for the passes whose stop test is decided by the bound of fp_kernel_f64 (see there).
__device__ __forceinline__ void trip_sum_only(const double2 (&v)[kFpUnroll], double rho_new, double& t1a, double& t1b) {
#pragma unroll
  for (int u = 0; u < kFpUnroll; ++u) {
    t1a = fma(v[u].x, rcp_fast(rho_new + v[u].x), t1a);
    t1b = fma(v[u].y, rcp_fast(rho_new + v[u].y), t1b);
  }
}
__device__ __forceinline__ bool finite_f64(double x) {
  return (((unsigned int)__double2hiint(x) >> 20) & 0x7ffu) != 0x7ffu;
}

// false when some sample of a pass would hand rcp_fast an argument at or above 2^1022, where rcp.approx.ftz.f64 returns 0 (1/x
// is subnormal and flushed) and the sample would drop out of the sums without a trace.  trip_fast's argument grows with e
// (rho, rho' >= 0; rounding is monotone), so the largest of a pass is the one at max e; inf and NaN count as out of range.
// It also bounds trip_sum_only's rho' + e: rho' + e > (rho' + e)(rho + e) needs rho + e < 1, and then rho' + e >= 2^1022
// needs rho' = inf (rho' = eps / (1 - eps) or avg / (1 - avg) is below 2^54 when finite), which makes the product inf too.
// emax and rho are the grid's (and the ranks') reduced values, so every block takes the same branch.
template <int VARIANT>
__device__ __forceinline__ bool rcp_fast_in_range(double emax, double rho_new, double rho_old) {
  const double x = (VARIANT == RLVI_FP_STANDARD) ? (rho_new + emax) * (rho_old + emax)
                                                 : (1.0 + rho_new * emax) * (1.0 + rho_old * emax);
  return x < 0x1p1022;
}

// ---- series passes (STANDARD; DESIGN.md section 4, "Series passes") ------------------------------------------------
// Once rho dominates max e, both sums of a pass follow from the power sums P_j = sum z^j of z = e / 2^E (2^E = the
// smallest power of two >= max e, so z is in [0, 1] and the scaling is exact).  With a = 2^E / rho', b = 2^E / rho:
//   sum pi'   = sum_{k >= 1} (-1)^(k-1) a^k P_k
//   sum t^2   = (a b / 2^E)^2 sum_{m >= 0} (-1)^m c_m P_{m+2},   c_m = sum_{i=0..m} (i+1)(m-i+1) a^i b^(m-i)
//             ((-1)^m c_m: the coefficients of 1 / ((1 + a x)^2 (1 + b x)^2))
// (t = (pi' - pi) / (rho - rho'), as in trip_fast).  The build pass accumulates them next to its ordinary sums.
__device__ __forceinline__ void trip_powers(const double2 (&v)[kFpUnroll], double zs, double (&P)[kFpSeriesJ], double& zmin) {
#pragma unroll
  for (int u = 0; u < kFpUnroll; ++u) {
    const double za = v[u].x * zs, zb = v[u].y * zs;
    zmin = fmin(zmin, fmin(za, zb));
    double pa = za, pb = zb;
#pragma unroll
    for (int j = 0; j < kFpSeriesJ; ++j) {
      P[j] += pa + pb;
      if (j + 1 < kFpSeriesJ) {
        pa *= za;
        pb *= zb;
      }
    }
  }
}

// The a-priori truncation bounds of both series after kFpSeriesJ power sums, relative to the sums themselves, at
// q = 2^E / min(rho', rho) >= a, b (derivation: DESIGN.md section 4).  A pass is evaluated from the series only when
// both are <= 2^-60, i.e. well below the rounding of the direct sums.
__device__ __forceinline__ bool series_admits(double q) {
  constexpr int J = kFpSeriesJ;
  const double r = q * double(J + 3) / double(J);
  if (!(q > 0.0 && r < 1.0)) return false;           // also rejects NaN
  double qm = 1.0;                                    // q^(J-1)
  for (int j = 0; j < J - 1; ++j) qm *= q;
  const double b1 = qm * q * (1.0 + q) / (1.0 - q);  // sum pi':  q^J (1 + q) / (1 - q)
  const double q1 = (1.0 + q) * (1.0 + q);
  const double b2 = q1 * q1 * (double(J + 2) * double(J + 1) * double(J) / 6.0) * qm / (1.0 - r);   // sum t^2
  constexpr double kTol = 8.673617379884035e-19;     // 2^-60
  return b1 <= kTol && b2 <= kTol;
}

// Evaluates both series from the published power sums P (shared memory, P[j] = P_{j+1}) in a fixed order: every
// thread of every block (of every rank) computes the same bits.  s2 = sum (pi' - pi)^2 as the streamed pass forms it.
__device__ __forceinline__ void series_sums(const double* P, double two_e, double zs, double rho_new, double rho_old,
                                            double& s1, double& s2) {
  constexpr int J = kFpSeriesJ;
  const double a = two_e / rho_new, b = two_e / rho_old;
  double h = P[J - 1];
#pragma unroll
  for (int j = J - 2; j >= 0; --j) h = fma(-a, h, P[j]);
  s1 = a * h;
  // sum_{m=0..J-2} g_m P_{m+2} with g_m = (-1)^m c_m, the coefficients of 1 / D(x), D(x) = (1 + a x)^2 (1 + b x)^2 =
  // 1 + d1 x + d2 x^2 + d3 x^3 + d4 x^4: g_0 = 1, g_m = -(d1 g_{m-1} + d2 g_{m-2} + d3 g_{m-3} + d4 g_{m-4}).  O(J) and a
  // short dependency chain, instead of the O(J^2) double sum (a series pass is on the critical path of every block).
  const double ab = a * b;
  const double d1 = 2.0 * (a + b), d2 = fma(a, a, fma(b, b, 4.0 * ab)), d3 = 2.0 * ab * (a + b), d4 = ab * ab;
  double g0 = 1.0, g1 = 0.0, g2 = 0.0, g3 = 0.0, acc = P[1];
#pragma unroll
  for (int m = 1; m <= J - 2; ++m) {
    const double g = -fma(d1, g0, fma(d2, g1, fma(d3, g2, d4 * g3)));
    g3 = g2;
    g2 = g1;
    g1 = g0;
    g0 = g;
    acc = fma(g, P[m + 1], acc);
  }
  const double w = a * b * zs, drho = rho_old - rho_new;
  s2 = (drho * drho) * ((w * w) * acc);
}

// SUM_ONLY (STANDARD): accumulate sum pi' only (s2 comes back 0); the IEEE / remainder paths still form (pi' - pi)^2 but
// their sum is discarded.  POW (STANDARD): the build pass of the series -- also accumulate this thread's power sums P and
// min z of z = e zs (trip_powers; zero-filled lanes add nothing).
template <int VARIANT, bool SUM_ONLY, bool POW = false>
__device__ __forceinline__ void stream_pass_vec(const double* e, ECache& ec, int64_t n, double rho_new,
                                                double rho_old, double& s1, double& s2, double zs = 0.0,
                                                double* P = nullptr, double* zmin = nullptr) {
  static_assert(!SUM_ONLY || VARIANT == RLVI_FP_STANDARD, "the sum-only pass exists for the STANDARD variant");
  static_assert(!POW || VARIANT == RLVI_FP_STANDARD, "the series exists for the STANDARD variant");
  double pw[kFpSeriesJ], zm = 0.0;
  if (POW) {
#pragma unroll
    for (int j = 0; j < kFpSeriesJ; ++j) pw[j] = 0.0;
    zm = INFINITY;
  }
  const double2* ev = reinterpret_cast<const double2*>(e);
  const int64_t nvec = n >> 1;
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  const double drho = rho_old - rho_new;
  int64_t c = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  double s1a = 0.0, s1b = 0.0, s2a = 0.0, s2b = 0.0;   // s2*: exact (pi' - pi)^2 sums of the IEEE-path samples
  double q2sa = 0.0, q2sb = 0.0;                        // fast trips: sum t^2 (STANDARD) / sum d^2 (ONLINE)
  int slot0 = 0;
  if (ec.ring) {
    // HBM-sized vector: every WARP streams its own contiguous segment through a private ring of
    // kFpRingDepth x 4 KiB slots filled by the TMA engine (one cp.async.bulk per 256-chunk trip, issued by
    // lane 0, completing on the slot's mbarrier): 8-12 KiB per warp in flight without holding registers, and
    // bulk requests reach ~6.6 TB/s where per-thread 16-byte loads (LDG or LDGSTS) level off at ~5.7 TB/s.
    // e[] reached L2 before the previous grid barrier; the bulk copies read L2.
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int kWarpTrip = kFpUnroll * 32;                     // chunks per warp trip (4 KiB)
    const int64_t nwarps = int64_t(gridDim.x) * (kFpThreads / 32);
    const int64_t wg = int64_t(blockIdx.x) * (kFpThreads / 32) + warp;
    const int64_t seg = (nvec + nwarps - 1) / nwarps;
    const int64_t lo = wg * seg < nvec ? wg * seg : nvec;
    const int64_t hi = (lo + seg < nvec) ? lo + seg : nvec;
    const int64_t ntrips = (hi - lo) / kWarpTrip;
    // the segment's partial last trip goes through the ring too (a shorter copy; lanes beyond it read zeros: e = 0 adds nothing
    // to either sum) instead of a batch of direct loads whose L2 latency stood at the end of every pass
    const int rem = int((hi - lo) - ntrips * kWarpTrip);
    const int64_t nt = ntrips + (rem > 0 ? 1 : 0);
    double2* ringw = ec.buf + size_t(warp) * kFpRingDepth * kWarpTrip;
    uint64_t* bar = ec.bars + warp * kFpRingDepth;
    uint32_t phase = ec.phase;
    // The trips are bound by issue slots (~200 SASS instructions per 16-sample trip and warp, profiles/r02_fixed_point_trace.txt),
    // so the loop works on 32-bit shared-memory addresses formed ONCE per pass (the generic-pointer helpers re-derive the
    // shared window on every call) and tests the sums for non-finite values once per PASS and lane instead of per trip.
    const uint32_t ring_s = smem_u32(ringw), bar_s = smem_u32(bar);
    const uint32_t lane_s = ring_s + uint32_t(lane) * 16u;
    const double2* gsrc = ev + lo;
    auto issue = [&](int64_t j, int slot) {
      if (lane == 0) {
        const uint32_t bytes = (j < ntrips) ? uint32_t(kWarpTrip * 16) : uint32_t(rem) * 16u;
        const uint32_t b32 = bar_s + uint32_t(slot) * 8u, dst = ring_s + uint32_t(slot) * uint32_t(kWarpTrip * 16);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(b32), "r"(bytes) : "memory");
        if (ec.head_trips > 0)
          asm volatile(
              "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(dst),
              "l"(gsrc + j * kWarpTrip), "r"(bytes), "r"(b32), "l"(j < ec.head_trips ? ec.pol_last : ec.pol_first)
              : "memory");
        else
          asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                       "l"(gsrc + j * kWarpTrip), "r"(bytes), "r"(b32)
                       : "memory");
      }
    };
    auto wait_slot = [&](int slot) {
      const uint32_t b32 = bar_s + uint32_t(slot) * 8u, parity = (phase >> slot) & 1u;
      uint32_t ok;
      do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(b32), "r"(parity)
            : "memory");
      } while (!ok);
      phase ^= 1u << slot;
    };
    auto lds2 = [](uint32_t addr) {
      double2 r;
      asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(r.x), "=d"(r.y) : "r"(addr) : "memory");
      return r;
    };
    if (ec.armed == 0) {          // the first ring pass; later passes were armed by their predecessor
#pragma unroll
      for (int j = 0; j < kFpRingDepth - 1; ++j)
        if (j < nt) issue(j, j);
    }
    int rd = 0, wr = kFpRingDepth - 1;
    for (int64_t j = 0; j < nt; ++j) {
      if (j + kFpRingDepth - 1 < nt) issue(j + kFpRingDepth - 1, wr);   // slot wr was read in iteration j - 1
      wait_slot(rd);
      const uint32_t src = lane_s + uint32_t(rd) * uint32_t(kWarpTrip * 16);
      double2 v[kFpUnroll];
      if (j < ntrips) {
#pragma unroll
        for (int u = 0; u < kFpUnroll; ++u) v[u] = lds2(src + uint32_t(u) * 512u);
      } else {
#pragma unroll
        for (int u = 0; u < kFpUnroll; ++u) v[u] = (u * 32 + lane < rem) ? lds2(src + uint32_t(u) * 512u) : make_double2(0.0, 0.0);
      }
      __syncwarp();                              // every lane has its data: the slot may be re-armed next trip
      if (POW) trip_powers(v, zs, pw, zm);
      if (SUM_ONLY) trip_sum_only(v, rho_new, s1a, s1b);
      else trip_fast<VARIANT>(v, rho_new, rho_old, s1a, s1b, q2sa, q2sb);
      rd = (rd + 1 == kFpRingDepth) ? 0 : rd + 1;
      wr = (wr + 1 == kFpRingDepth) ? 0 : wr + 1;
    }
    if (!(finite_f64(s1a + s1b) && finite_f64(q2sa + q2sb))) {
      // rare: rho = inf / 0 or an e at the edge of the exponent range made the fast reciprocal produce inf / NaN somewhere in
      // this lane's share of the segment -> that share again with the IEEE divisions (exact (pi' - pi)^2 sums)
      s1a = s1b = q2sa = q2sb = 0.0;
#pragma unroll 1
      for (int64_t i = lo + lane; i < hi; i += 32) {
        const double2 w = ld_e2(ev + i);
        double pn, d;
        post_pair_f64<VARIANT>(w.x, rho_new, rho_old, pn, d);
        s1a += pn;
        s2a = fma(d, d, s2a);
        post_pair_f64<VARIANT>(w.y, rho_new, rho_old, pn, d);
        s1b += pn;
        s2b = fma(d, d, s2b);
      }
    }
    // every slot has been read (the __syncwarp of the last trip): arm the next pass's first trips now
    ec.armed = 0;
#pragma unroll
    for (int j = 0; j < kFpRingDepth - 1; ++j)
      if (j < nt) {
        issue(j, j);
        ec.armed = j + 1;
      }
    ec.phase = phase;
    c = nvec;                                    // the grid-stride loops below have nothing left to do
  }
  for (; c + (kFpUnroll - 1) * stride < nvec; c += kFpUnroll * stride, slot0 += kFpUnroll) {
    double2 v[kFpUnroll];
    if (slot0 + kFpUnroll <= ec.slots) {   // whole trip on chip (uniform branch; keeps the 8 loads back to back)
#pragma unroll
      for (int u = 0; u < kFpUnroll; ++u) v[u] = ec.buf[(slot0 + u) * kFpThreads + threadIdx.x];
    } else {
#pragma unroll
      for (int u = 0; u < kFpUnroll; ++u) v[u] = ld_e2(ev + c + u * stride);
    }
    if (POW) trip_powers(v, zs, pw, zm);
    double t1a = 0.0, t1b = 0.0, q2a = 0.0, q2b = 0.0;
    if (SUM_ONLY) trip_sum_only(v, rho_new, t1a, t1b);
    else trip_fast<VARIANT>(v, rho_new, rho_old, t1a, t1b, q2a, q2b);
    if (finite_f64(t1a + t1b) && finite_f64(q2a + q2b)) {
      s1a += t1a;
      s1b += t1b;
      q2sa += q2a;
      q2sb += q2b;
    } else {   // rare: rho = inf / 0 or e at the edge of the exponent range -> IEEE path for this trip
#pragma unroll 1
      for (int u = 0; u < kFpUnroll; ++u) {
        const double2 w = ld_e2c(ec, slot0 + u, ev + c + u * stride);   // re-load: keeps v[] in registers
        double pn, d;
        post_pair_f64<VARIANT>(w.x, rho_new, rho_old, pn, d);
        s1a += pn;
        s2a = fma(d, d, s2a);
        post_pair_f64<VARIANT>(w.y, rho_new, rho_old, pn, d);
        s1b += pn;
        s2b = fma(d, d, s2b);
      }
    }
  }
  if (c < nvec) {
    // remainder: ONE predicated trip with all loads in flight together (a chunk-at-a-time tail loop costs a
    // full memory latency per chunk, which dominated the pass once a shard is L2 resident), zero-filled and pushed
    // through the same fast trip as the full ones (e = 0 adds nothing to either sum; at 2^23 samples per GPU the
    // remainder is 1 of 7 trips, and with the IEEE divisions it cost more than the other six together)
    double2 v[kFpUnroll];
#pragma unroll
    for (int u = 0; u < kFpUnroll; ++u) {
      const int64_t i = c + u * stride;
      v[u] = (i < nvec) ? ld_e2c(ec, slot0 + u, ev + i) : make_double2(0.0, 0.0);
    }
    if (POW) trip_powers(v, zs, pw, zm);
    double t1a = 0.0, t1b = 0.0, q2a = 0.0, q2b = 0.0;
    if (SUM_ONLY) trip_sum_only(v, rho_new, t1a, t1b);
    else trip_fast<VARIANT>(v, rho_new, rho_old, t1a, t1b, q2a, q2b);
    if (finite_f64(t1a + t1b) && finite_f64(q2a + q2b)) {
      s1a += t1a;
      s1b += t1b;
      q2sa += q2a;
      q2sb += q2b;
    } else {
#pragma unroll 1
      for (int u = 0; u < kFpUnroll; ++u) {
        if (c + u * stride < nvec) {
          const double2 w = ld_e2c(ec, slot0 + u, ev + c + u * stride);
          double pn, d;
          post_pair_f64<VARIANT>(w.x, rho_new, rho_old, pn, d);
          s1a += pn;
          s2a = fma(d, d, s2a);
          post_pair_f64<VARIANT>(w.y, rho_new, rho_old, pn, d);
          s1b += pn;
          s2b = fma(d, d, s2b);
        }
      }
    }
  }
  if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0) {
    double pn, d;
    post_pair_f64<VARIANT>(e[n - 1], rho_new, rho_old, pn, d);
    s1a += pn;
    s2a = fma(d, d, s2a);
    if (POW) {
      const double z = e[n - 1] * zs;
      double pz = z;
      zm = fmin(zm, z);
#pragma unroll
      for (int j = 0; j < kFpSeriesJ; ++j) {
        pw[j] += pz;
        pz *= z;
      }
    }
  }
  if (POW) {
#pragma unroll
    for (int j = 0; j < kFpSeriesJ; ++j) P[j] = pw[j];
    *zmin = zm;
  }
  s1 = s1a + s1b;
  s2 = SUM_ONLY ? 0.0 : (s2a + s2b) + ((VARIANT == RLVI_FP_STANDARD) ? (drho * drho) * (q2sa + q2sb) : (q2sa + q2sb));
}

// Pass 1 over a precomputed, 16-byte aligned e[] (the loss kernel wrote it): pi' against the constant
// initial posterior, plus max e (ONLINE's normalisation).  Same load batching as stream_pass_vec.
template <int VARIANT>
__device__ __forceinline__ void first_pass_vec(const double* e, const ECache& ec, int64_t n, double rho, double pi0,
                                               double& s1, double& s2, double& mx) {
  const double2* ev = reinterpret_cast<const double2*>(e);
  const int64_t nvec = n >> 1;
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  int64_t c = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  double s1a = 0.0, s1b = 0.0, s2a = 0.0, s2b = 0.0, m = 0.0;
  auto one = [&](double x, double& sa, double& sb) {
    const double pn = post_f64<VARIANT>(x, rho);
    const double d = pn - pi0;
    sa += pn;
    sb = fma(d, d, sb);
    m = fmax(m, x);
  };
  int slot0 = 0;
  for (; c + (kFpUnroll - 1) * stride < nvec; c += kFpUnroll * stride, slot0 += kFpUnroll) {
    double2 v[kFpUnroll];
#pragma unroll
    for (int u = 0; u < kFpUnroll; ++u) v[u] = ld_e2(ev + c + u * stride);
#pragma unroll
    for (int u = 0; u < kFpUnroll; ++u)
      if (slot0 + u < ec.slots) ec.buf[(slot0 + u) * kFpThreads + threadIdx.x] = v[u];
#pragma unroll
    for (int u = 0; u < kFpUnroll; ++u) {
      one(v[u].x, s1a, s2a);
      one(v[u].y, s1b, s2b);
    }
  }
  if (c < nvec) {
    double2 v[kFpUnroll];
#pragma unroll
    for (int u = 0; u < kFpUnroll; ++u) {
      const int64_t i = c + u * stride;
      v[u] = (i < nvec) ? ld_e2(ev + i) : make_double2(0.0, 0.0);
      if (i < nvec && slot0 + u < ec.slots) ec.buf[(slot0 + u) * kFpThreads + threadIdx.x] = v[u];
    }
#pragma unroll
    for (int u = 0; u < kFpUnroll; ++u) {
      if (c + u * stride < nvec) {
        one(v[u].x, s1a, s2a);
        one(v[u].y, s1b, s2b);
      }
    }
  }
  if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0) one(e[n - 1], s1a, s2a);
  s1 = s1a + s1b;
  s2 = s2a + s2b;
  mx = m;
}

// Final pass: pi = the reference's own expression (IEEE division), optionally divided by `norm` (ONLINE).
template <int VARIANT>
__device__ __forceinline__ void final_pass_vec(const double* e, const ECache& ec, double* out, int64_t n, double rho,
                                               double norm) {
  const double2* ev = reinterpret_cast<const double2*>(e);
  double2* ov = reinterpret_cast<double2*>(out);
  const int64_t nvec = n >> 1;
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  int64_t c = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  auto one = [&](double x) {
    double pv = post_f64<VARIANT>(x, rho);
    if (VARIANT == RLVI_FP_ONLINE) pv = pv / norm;
    return pv;
  };
  int slot0 = 0;
  for (; c + (kFpUnroll - 1) * stride < nvec; c += kFpUnroll * stride, slot0 += kFpUnroll) {
    double2 v[kFpUnroll];
    if (slot0 + kFpUnroll <= ec.slots) {   // whole trip on chip (uniform branch; keeps the 8 loads back to back)
#pragma unroll
      for (int u = 0; u < kFpUnroll; ++u) v[u] = ec.buf[(slot0 + u) * kFpThreads + threadIdx.x];
    } else {
#pragma unroll
      for (int u = 0; u < kFpUnroll; ++u) v[u] = ld_e2(ev + c + u * stride);
    }
#pragma unroll
    for (int u = 0; u < kFpUnroll; ++u) ov[c + u * stride] = make_double2(one(v[u].x), one(v[u].y));
  }
  if (c < nvec) {
    double2 v[kFpUnroll];
#pragma unroll
    for (int u = 0; u < kFpUnroll; ++u) {
      const int64_t i = c + u * stride;
      v[u] = (i < nvec) ? ld_e2c(ec, slot0 + u, ev + i) : make_double2(0.0, 0.0);
    }
#pragma unroll
    for (int u = 0; u < kFpUnroll; ++u) {
      const int64_t i = c + u * stride;
      if (i < nvec) ov[i] = make_double2(one(v[u].x), one(v[u].y));
    }
  }
  if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0) out[n - 1] = one(e[n - 1]);
}

// The build pass of the series (STANDARD, VEC): a sum-only streamed pass that also accumulates the
// power sums, then the pass's own sums reduced as usual, then the power sums and min z in (kFpSeriesJ + 1) / 3 further
// rounds of the same fixed-order reduction, so every block of every rank holds the same P_j.  They are kept in
// shared memory (`pw`, block-wide) rather than in registers across the later passes.
template <int VARIANT>
__device__ __forceinline__ void build_power_sums(const FpParams<double>& p, FpShared& sh, ECache& ec, const double* e,
                                              double rho_new, double rho_old, double zs, double* pw,
                                              double& s1, double& s2, int& pw_state, bool& ok, unsigned int& round) {
  double P[kFpSeriesJ], zmin = 0.0;
  stream_pass_vec<VARIANT, true, true>(e, ec, p.n, rho_new, rho_old, s1, s2, zs, P, &zmin);
  double z = 0.0;
  ok = grid_allreduce3<double, OP_SUM, false>(p, sh, s1, s2, z, round);
  bool fin = true;
#pragma unroll
  for (int j = 0; j + 2 < kFpSeriesJ; j += 3) {
    ok = ok && grid_allreduce3<double, OP_SUM, false>(p, sh, P[j], P[j + 1], P[j + 2], round);
    fin = fin && finite_f64(P[j]) && finite_f64(P[j + 1]) && finite_f64(P[j + 2]);
  }
  ok = ok && grid_allreduce3<double, OP_MIN, false>(p, sh, P[kFpSeriesJ - 2], P[kFpSeriesJ - 1], zmin, round);
  fin = fin && finite_f64(P[kFpSeriesJ - 2]) && finite_f64(P[kFpSeriesJ - 1]);
  if (threadIdx.x == 0) {
#pragma unroll
    for (int j = 0; j < kFpSeriesJ; ++j) pw[j] = P[j];
  }
  __syncthreads();
  pw_state = (fin && zmin >= 0.0) ? 1 : -1;
}

// =================================================================================================
// FP64 kernel: STANDARD and ONLINE
// =================================================================================================
// VEC: two CTAs per SM, which the shared-memory budget (kFpCacheSlots, the ring) is sized for.  Left to itself ptxas gave
// the STANDARD instantiation 174 registers (one CTA per SM, hence another grid and summation order) once the per-pass range
// test was added; at 128 it spills what it spilled before.
template <int VARIANT, bool VEC>
__global__ void __launch_bounds__(kFpThreads, VEC ? 2 : 0) fp_kernel_f64(const FpParams<double> p) {
  __shared__ FpShared sh;
  unsigned int round = 0;
  const double n_glob = double(p.n_global);
  const double pi0 = (p.pi0 > 0.0) ? p.pi0 : ((VARIANT == RLVI_FP_STANDARD) ? 0.95 : 0.5);
  const double s = p.scale ? *p.scale : 1.0;
  const bool have_losses = p.losses != nullptr;
  const double* losses = p.losses;
  double* e = p.e;
  constexpr int W = VEC ? 2 : 1;
  extern __shared__ __align__(16) unsigned char fp_dyn_smem[];
  ECache ec;
  ec.buf = reinterpret_cast<double2*>(fp_dyn_smem);
  ec.slots = (VEC && p.cache_slots > 0) ? p.cache_slots : 0;
  ec.ring = (VEC && p.cache_slots < 0) ? 1 : 0;      // cache_slots < 0 selects the prefetch ring
  __shared__ uint64_t fp_ring_bars[(kFpThreads / 32) * kFpRingDepth];
  ec.bars = fp_ring_bars;
  ec.phase = 0u;
  ec.armed = 0;
  ec.head_trips = 0;
  ec.pol_last = ec.pol_first = 0ull;
  if (ec.ring && p.l2_head) {
    const int64_t nwarps = int64_t(gridDim.x) * (kFpThreads / 32);
    ec.head_trips = int(kFpL2HeadBytes / (nwarps * int64_t(kFpUnroll * 32 * 16)));
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(ec.pol_last));
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(ec.pol_first));
  }
  if (ec.ring) {
    if (threadIdx.x == 0) {
      for (int i = 0; i < (kFpThreads / 32) * kFpRingDepth; ++i) mbar_init(&fp_ring_bars[i], 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
  }
  const int64_t chunk0 = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t cstride = int64_t(gridDim.x) * blockDim.x;
  // rho for pass 1 from the constant initial posterior, in the reference's operation order
  double rho_new, rho_old = 0.0, eps;
  if (VARIANT == RLVI_FP_STANDARD) {
    eps = 1.0 - pi0;
    rho_new = eps / (1.0 - eps);
  } else {
    eps = 1.0 - pi0;
    rho_new = pi0 / (1.0 - pi0);
  }

  double S = n_glob * pi0, E = 0.0, emax = 0.0, err = 0.0;
  const double sqrt_n = sqrt(n_glob);
  double bound_prev = 0.0, bound_prev2 = 0.0;
  int k = 1, converged = 0;
  bool ok = true;
  // series passes: the power sums (block-wide copy), 2^E and 2^-E; pw_state 0 = not built, 1 = usable, -1 = built, unusable
  constexpr bool kSeries = VEC && VARIANT == RLVI_FP_STANDARD;
  __shared__ double fp_pw[kFpSeriesJ];
  double two_e = 0.0, zs = 0.0;
  int pw_state = 0;
  for (;; ++k) {
    double s1 = 0.0, s2 = 0.0, mx = 0.0;
    bool sum_only = false, series = false, build = false;
    if (kSeries && k >= 2 && pw_state == 1 && series_admits(two_e / fmin(rho_new, rho_old))) {
      // a series pass: no stream, no grid barrier.  An err within 2^-40 tol of tol is re-taken from the streamed sums,
      // so a stop decision never rests on the series' rounding.
      series_sums(fp_pw, two_e, zs, rho_new, rho_old, s1, s2);
      series = !(fabs(sqrt(s2) - p.tol) <= 0x1p-40 * fabs(p.tol));
    }
    if (series) {
      // s1, s2 came from the series
    } else if (k == 1 && VEC && !have_losses) {
      first_pass_vec<VARIANT>(e, ec, p.n, rho_new, pi0, s1, s2, mx);
    } else if (k == 1) {
      for_each_chunk<double, VEC>(p.n, [&](int64_t c, int) {
        const int64_t i = c * W;
        double ev[W];
        if (have_losses) {
          double lv[W];
          load_chunk<double, VEC, W>(losses, i, p.n, lv, 0.0);
#pragma unroll
          for (int j = 0; j < W; ++j) ev[j] = exp(-(s * lv[j]));
          store_chunk<double, VEC, W>(e, i, p.n, ev);
        } else {
          load_chunk<double, VEC, W>(e, i, p.n, ev, 0.0);
        }
        if (VEC) {   // keep the chunk on chip for the later passes (chunk ordinal of this thread = slot)
          const int64_t slot = (c - chunk0) / cstride;
          if (slot < ec.slots && i + W <= p.n) ec.buf[slot * kFpThreads + threadIdx.x] = make_double2(ev[0], ev[W - 1]);
        }
#pragma unroll
        for (int j = 0; j < W; ++j) {
          if (i + j < p.n) {
            const double pn = post_f64<VARIANT>(ev[j], rho_new);
            const double d = pn - pi0;
            s1 += pn;
            s2 = fma(d, d, s2);
            mx = fmax(mx, ev[j]);
          }
        }
      });
    } else if (VEC && rcp_fast_in_range<VARIANT>(emax, rho_new, rho_old)) {
      // Which trip?  By Cauchy-Schwarz  ||pi' - pi||_2 >= |sum pi' - sum pi| / sqrt(N): when that lower bound is above tol
      // the stop test `err < tol` (rlvi.py:18) is decided WITHOUT the sum of squared differences, and the pass needs
      // half the FP64 instructions.  The bound is predicted from the last two (it decays geometrically: in the
      // collapse regime it is within 10 % of err itself, so all passes but the last qualify); a pass that was run
      // sum-only and whose bound then fails to prove anything is repeated in full, so every decision is the exact one.
      sum_only = (VARIANT == RLVI_FP_STANDARD) && k < p.maxiter && bound_prev2 > 0.0 &&
                 bound_prev * fmin(1.0, bound_prev / bound_prev2) > 2.0 * p.tol;
      // Build the power sums (once per call) in a sum-only pass whose last two ratios predict that the series will be
      // admitted two passes on: rho grows by r = rho' / rho per pass, so q falls to q / r^2.  Data that never nears
      // the switch (r ~ 1, q >= 1) never builds them.  Only the sum-only trip has the registers to spare for them.
      if (kSeries && p.series && sum_only && pw_state == 0 && rho_old > 0.0) {
        const double r = rho_new / rho_old;
        build = series_admits(two_e / fmin(rho_new, rho_old) / (r * r));
      }
      if constexpr (kSeries) {
        if (build) build_power_sums<VARIANT>(p, sh, ec, e, rho_new, rho_old, zs, fp_pw, s1, s2, pw_state, ok, round);
      }
      if (!build) {
        if (sum_only) stream_pass_vec<VARIANT, VARIANT == RLVI_FP_STANDARD>(e, ec, p.n, rho_new, rho_old, s1, s2);
        else stream_pass_vec<VARIANT, false>(e, ec, p.n, rho_new, rho_old, s1, s2);
      }
    } else {
      // the scalar path, and a pass of the aligned one that is out of rcp_fast's range (leaves the ring's armed copies alone)
      for_each_chunk<double, VEC>(p.n, [&](int64_t c, int) {
        const int64_t i = c * W;
        double ev[W];
        load_chunk<double, VEC, W>(e, i, p.n, ev, 0.0);
#pragma unroll
        for (int j = 0; j < W; ++j) {
          if (i + j < p.n) {
            double pn, d;
            post_pair_f64<VARIANT>(ev[j], rho_new, rho_old, pn, d);
            s1 += pn;
            s2 = fma(d, d, s2);
          }
        }
      });
    }
    if (k == 1) {
      // ring mode reads e[] with the TMA engine (async proxy) in the later passes: order this thread's generic
      // stores of e before them (the grid barrier below then publishes them to the other CTAs)
      if (ec.ring && have_losses) asm volatile("fence.proxy.async;" ::: "memory");
      ok = grid_allreduce3<double, OP_MAX, true>(p, sh, s1, s2, mx, round);
      emax = mx;
      if (kSeries && emax > 0x1p-1000 && emax < 0x1p1000) {     // normal and finite: 2^E and 2^-E are exact
        int ex;
        const double m = frexp(emax, &ex);                     // emax = m 2^ex, m in [0.5, 1)
        two_e = (m == 0.5) ? emax : ldexp(1.0, ex);
        zs = 1.0 / two_e;
      } else {
        pw_state = -1;
      }
    } else if (series || build) {
      // the sums are complete (series) or were reduced with the power sums
    } else {
      double z = 0.0;
      ok = grid_allreduce3<double, OP_SUM, false>(p, sh, s1, s2, z, round);
    }
    if (!ok) break;
    const double bound = fabs(s1 - S) / sqrt_n;          // S still holds the previous pass's sum (N pi0 before pass 1)
    if (sum_only && !(bound > p.tol * (1.0 + 1e-6))) {
      // the bound proves nothing this time: repeat the pass with the full trip (all blocks of all ranks hold the
      // same `bound` bits and come here together)
      sum_only = false;
      s1 = 0.0;
      s2 = 0.0;
      double z = 0.0;
      stream_pass_vec<VARIANT, false>(e, ec, p.n, rho_new, rho_old, s1, s2);
      ok = grid_allreduce3<double, OP_SUM, false>(p, sh, s1, s2, z, round);
      if (!ok) break;
    }
    bound_prev2 = bound_prev;
    bound_prev = bound;
    S = s1;
    if (sum_only) {
      err = bound;                                       // a lower bound of the true error, already above tol
    } else {
      E = s2;
      err = sqrt(E);
      if (err < p.tol) { converged = 1; break; }   // rlvi.py:18 / online main.py:54
    }
    if (k >= p.maxiter) break;
    // next pass's ratio from the mean of the posteriors just computed
    rho_old = rho_new;
    const double avg = S / n_glob;
    if (VARIANT == RLVI_FP_STANDARD) {
      eps = 1.0 - avg;                 // rlvi.py:13
      rho_new = eps / (1.0 - eps);     // rlvi.py:14
    } else {
      eps = 1.0 - avg;
      rho_new = avg / (1.0 - avg);     // online main.py:51
    }
  }

  // ring mode: the last stream pass armed copies for a pass that will not run -- let them land before the CTA can exit
  if (ec.ring) {
    uint64_t* bar = ec.bars + (threadIdx.x >> 5) * kFpRingDepth;
    for (int sl = 0; sl < ec.armed; ++sl) mbar_wait(&bar[sl], (ec.phase >> sl) & 1u);
    ec.armed = 0;
  }
  // final pass: write the last pi' with the reference's own expression (single correctly rounded
  // division), then the variant's normalisation
  double norm = 1.0;
  if (VARIANT == RLVI_FP_ONLINE) norm = post_f64<VARIANT>(emax, rho_new) * n_glob;   // max(pi') * n
  if (ok && VEC) {
    final_pass_vec<VARIANT>(e, ec, p.pi_out, p.n, rho_new, norm);
  } else if (ok) {
    double* out = p.pi_out;
    for_each_chunk<double, VEC>(p.n, [&](int64_t c, int) {
      const int64_t i = c * W;
      double ev[W], pv[W];
      load_chunk<double, VEC, W>(e, i, p.n, ev, 0.0);
#pragma unroll
      for (int j = 0; j < W; ++j) {
        pv[j] = post_f64<VARIANT>(ev[j], rho_new);
        if (VARIANT == RLVI_FP_ONLINE) pv[j] = pv[j] / norm;
      }
      store_chunk<double, VEC, W>(out, i, p.n, pv);
    });
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    rlvi_fp_result r;
    r.eps = eps;
    r.rho = rho_new;
    r.sum_pi = S;
    r.err = err;
    r.iters = ok ? k : -1;
    r.converged = ok ? converged : -1;
    *p.result = r;
  }
}

// =================================================================================================
// FP32 kernel: DEEP (train_rlvi.py:14-38).  Elementwise arithmetic in FP32 exactly as torch does it;
// the two sums are accumulated in FP64 and rounded to FP32 where torch holds an FP32 scalar.
// =================================================================================================
__device__ __forceinline__ float post_f32(float e, float rho) {
  const float a = rho * e;
  return __fdiv_rn(a, 1.0f + a);
}

template <bool VEC>
__global__ void __launch_bounds__(kFpThreads) fp_kernel_deep_f32(const FpParams<float> p) {
  __shared__ FpShared sh;
  unsigned int round = 0;
  const double n_glob = double(p.n_global);
  constexpr int W = VEC ? 4 : 1;
  float* res = p.residuals;
  float* wts = p.pi_out;
  float* e = p.e;
  bool ok = true;

  // residuals.min()  (train_rlvi.py:26)
  double mn = INFINITY, z0 = 0.0, z1 = 0.0;
  for_each_chunk<float, VEC>(p.n, [&](int64_t c, int) {
    const int64_t i = c * W;
    float rv[W];
    load_chunk<float, VEC, W>(res, i, p.n, rv, INFINITY);
#pragma unroll
    for (int j = 0; j < W; ++j) mn = fmin(mn, double(rv[j]));
  });
  ok = grid_allreduce3<float, OP_MIN, true>(p, sh, z0, z1, mn, round);
  const float rmin = float(mn);

  float rho_new = float(0.95 / (1.0 - 0.95));   // Python-float ratio, cast when it meets the FP32 tensor
  float rho_old = 0.0f;
  float avg = 0.95f;
  double S = 0.0, err = 0.0, emax = 0.0;
  int k = 1, converged = 0;
  if (ok) {
    for (;; ++k) {
      double s1 = 0.0, s2 = 0.0, mx = 0.0;
      if (k == 1) {
        for_each_chunk<float, VEC>(p.n, [&](int64_t c, int) {
          const int64_t i = c * W;
          float rv[W], wv[W], ev[W];
          load_chunk<float, VEC, W>(res, i, p.n, rv, 0.f);
          load_chunk<float, VEC, W>(wts, i, p.n, wv, 0.f);
#pragma unroll
          for (int j = 0; j < W; ++j) {
            rv[j] = rv[j] - rmin;          // residuals.sub_(min)
            ev[j] = expf(-rv[j]);          // torch.exp(-residuals)
          }
          store_chunk<float, VEC, W>(res, i, p.n, rv);
          store_chunk<float, VEC, W>(e, i, p.n, ev);
#pragma unroll
          for (int j = 0; j < W; ++j) {
            if (i + j < p.n) {
              const float pn = post_f32(ev[j], rho_new);
              const float d = pn - wv[j];    // first pass: against the INCOMING weights (line 32)
              s1 += double(pn);
              s2 = fma(double(d), double(d), s2);
              mx = fmax(mx, double(ev[j]));
            }
          }
        });
      } else {
        for_each_chunk<float, VEC>(p.n, [&](int64_t c, int) {
          const int64_t i = c * W;
          float ev[W];
          load_chunk<float, VEC, W>(e, i, p.n, ev, 0.f);
#pragma unroll
          for (int j = 0; j < W; ++j) {
            if (i + j < p.n) {
              const float pn = post_f32(ev[j], rho_new);
              const float po = post_f32(ev[j], rho_old);   // == what `weights` held after the last pass
              const float d = pn - po;
              s1 += double(pn);
              s2 = fma(double(d), double(d), s2);
            }
          }
        });
      }
      if (k == 1) {
        ok = grid_allreduce3<float, OP_MAX, true>(p, sh, s1, s2, mx, round);
        emax = mx;
      } else {
        double z = 0.0;
        ok = grid_allreduce3<float, OP_SUM, true>(p, sh, s1, s2, z, round);
      }
      if (!ok) break;
      S = s1;
      err = double(float(sqrt(s2)));          // torch.norm returns an FP32 scalar
      avg = float(S / n_glob);                // weights.mean() (line 34) -- computed BEFORE the test
      rho_old = rho_new;
      const float rho_next = __fdiv_rn(avg, 1.0f - avg);
      if (float(err) < float(p.tol)) { converged = 1; break; }
      if (k >= p.maxiter) break;
      rho_new = rho_next;
    }
  }
  // weights[:] = pi'; weights /= weights.max()   (lines 33, 37)
  const float rho_fin = rho_old;   // the ratio the last executed pass used
  if (ok) {
    const float wmax = post_f32(float(emax), rho_fin);
    for_each_chunk<float, VEC>(p.n, [&](int64_t c, int) {
      const int64_t i = c * W;
      float ev[W], pv[W];
      load_chunk<float, VEC, W>(e, i, p.n, ev, 0.f);
#pragma unroll
      for (int j = 0; j < W; ++j) pv[j] = __fdiv_rn(post_f32(ev[j], rho_fin), wmax);
      store_chunk<float, VEC, W>(wts, i, p.n, pv);
    });
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    rlvi_fp_result r;
    r.eps = 1.0 - double(avg);
    r.rho = double(rho_fin);
    r.sum_pi = S;
    r.err = err;
    r.iters = ok ? k : -1;
    r.converged = ok ? converged : -1;
    *p.result = r;
  }
}

// =================================================================================================
// Small-n path: the WHOLE loop in one CTA, e[] resident in shared memory (n <= 28 K doubles / 56 K floats:
// the online batches of 100 and the deep path's N_train = 45 000).  No grid barrier, no global traffic
// between passes: a pass is n/1024 shared-memory reads per thread plus one block reduction (~1-2 us).
// =================================================================================================
constexpr int kSmallThreads = 1024;
constexpr size_t kSmallSmemBytes = size_t(224) * 1024;

struct SmallRed {
  double part[2][3][kSmallThreads / 32];
};

// Block-wide reduction of three values (v2 with OP2); every thread returns the totals.  Fixed order: xor tree
// per warp, then every warp adds the 32 warp partials in the same lane-strided order.  One __syncthreads per
// call (the partial buffers alternate by `round` parity).
template <int OP2>
__device__ __forceinline__ void block_allreduce3(SmallRed& red, double& v0, double& v1, double& v2, unsigned int& round) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned int b = round & 1u;
  v0 = warp_sum(v0);
  v1 = warp_sum(v1);
  v2 = (OP2 == OP_SUM) ? warp_sum(v2) : (OP2 == OP_MIN ? warp_min(v2) : warp_max(v2));
  if (lane == 0) {
    red.part[b][0][warp] = v0;
    red.part[b][1][warp] = v1;
    red.part[b][2][warp] = v2;
  }
  __syncthreads();
  v0 = warp_sum(red.part[b][0][lane]);
  v1 = warp_sum(red.part[b][1][lane]);
  const double t = red.part[b][2][lane];
  v2 = (OP2 == OP_SUM) ? warp_sum(t) : (OP2 == OP_MIN ? warp_min(t) : warp_max(t));
  round += 1u;
}

template <int VARIANT>
__global__ void __launch_bounds__(kSmallThreads, 1) fp_small_kernel_f64(const FpParams<double> p) {
  extern __shared__ __align__(16) unsigned char small_smem[];
  double* se = reinterpret_cast<double*>(small_smem);
  __shared__ SmallRed red;
  unsigned int round = 0;
  const int n = int(p.n);
  const double n_glob = double(p.n_global);
  const double pi0 = (p.pi0 > 0.0) ? p.pi0 : ((VARIANT == RLVI_FP_STANDARD) ? 0.95 : 0.5);
  const double s = p.scale ? *p.scale : 1.0;
  double eps = 1.0 - pi0;
  double rho_new = (VARIANT == RLVI_FP_STANDARD) ? eps / (1.0 - eps) : pi0 / (1.0 - pi0);
  double rho_old = 0.0;
  // pass 1: e -> shared memory (+ global e_work, part of the contract), sums against the constant pi0
  double s1 = 0.0, s2 = 0.0, mx = 0.0;
  for (int i = threadIdx.x; i < n; i += kSmallThreads) {
    const double ev = p.losses ? exp(-(s * p.losses[i])) : p.e[i];
    se[i] = ev;
    if (p.losses) p.e[i] = ev;
    const double pn = post_f64<VARIANT>(ev, rho_new);
    const double d = pn - pi0;
    s1 += pn;
    s2 = fma(d, d, s2);
    mx = fmax(mx, ev);
  }
  block_allreduce3<OP_MAX>(red, s1, s2, mx, round);
  const double emax = mx;
  double S = s1, err = sqrt(s2);
  int k = 1, converged = 0;
  while (true) {
    if (err < p.tol) { converged = 1; break; }
    if (k >= p.maxiter) break;
    rho_old = rho_new;
    const double avg = S / n_glob;
    eps = 1.0 - avg;
    rho_new = (VARIANT == RLVI_FP_STANDARD) ? eps / (1.0 - eps) : avg / (1.0 - avg);
    ++k;
    double a1 = 0.0, a2 = 0.0, z = 0.0;
    for (int i = threadIdx.x; i < n; i += kSmallThreads) {
      double pn, d;
      post_pair_f64<VARIANT>(se[i], rho_new, rho_old, pn, d);
      a1 += pn;
      a2 = fma(d, d, a2);
    }
    block_allreduce3<OP_SUM>(red, a1, a2, z, round);
    S = a1;
    err = sqrt(a2);
  }
  double norm = 1.0;
  if (VARIANT == RLVI_FP_ONLINE) norm = post_f64<VARIANT>(emax, rho_new) * n_glob;
  for (int i = threadIdx.x; i < n; i += kSmallThreads) {
    double pv = post_f64<VARIANT>(se[i], rho_new);
    if (VARIANT == RLVI_FP_ONLINE) pv = pv / norm;
    p.pi_out[i] = pv;
  }
  if (threadIdx.x == 0) {
    rlvi_fp_result r;
    r.eps = eps;
    r.rho = rho_new;
    r.sum_pi = S;
    r.err = err;
    r.iters = k;
    r.converged = converged;
    *p.result = r;
  }
}

__global__ void __launch_bounds__(kSmallThreads, 1) fp_small_kernel_deep_f32(const FpParams<float> p) {
  extern __shared__ __align__(16) unsigned char small_smem[];
  float* se = reinterpret_cast<float*>(small_smem);
  __shared__ SmallRed red;
  unsigned int round = 0;
  const int n = int(p.n);
  const double n_glob = double(p.n_global);
  float* res = p.residuals;
  float* wts = p.pi_out;
  double mn = INFINITY, z0 = 0.0, z1 = 0.0;
  for (int i = threadIdx.x; i < n; i += kSmallThreads) mn = fmin(mn, double(res[i]));
  block_allreduce3<OP_MIN>(red, z0, z1, mn, round);
  const float rmin = float(mn);
  float rho_new = float(0.95 / (1.0 - 0.95)), rho_old = 0.0f, avg = 0.95f;
  double s1 = 0.0, s2 = 0.0, mx = 0.0;
  for (int i = threadIdx.x; i < n; i += kSmallThreads) {
    const float r = res[i] - rmin;           // residuals.sub_(min)
    const float ev = expf(-r);               // torch.exp(-residuals)
    res[i] = r;
    se[i] = ev;
    p.e[i] = ev;
    const float pn = post_f32(ev, rho_new);
    const float d = pn - wts[i];             // first pass: against the INCOMING weights
    s1 += double(pn);
    s2 = fma(double(d), double(d), s2);
    mx = fmax(mx, double(ev));
  }
  block_allreduce3<OP_MAX>(red, s1, s2, mx, round);
  const double emax = mx;
  double S = s1, err = double(float(sqrt(s2)));
  int k = 1, converged = 0;
  while (true) {
    avg = float(S / n_glob);                 // weights.mean(), computed BEFORE the test (train_rlvi.py:34-35)
    rho_old = rho_new;
    const float rho_next = __fdiv_rn(avg, 1.0f - avg);
    if (float(err) < float(p.tol)) { converged = 1; break; }
    if (k >= p.maxiter) break;
    rho_new = rho_next;
    ++k;
    double a1 = 0.0, a2 = 0.0, z = 0.0;
    for (int i = threadIdx.x; i < n; i += kSmallThreads) {
      const float ev = se[i];
      const float pn = post_f32(ev, rho_new);
      const float d = pn - post_f32(ev, rho_old);
      a1 += double(pn);
      a2 = fma(double(d), double(d), a2);
    }
    block_allreduce3<OP_SUM>(red, a1, a2, z, round);
    S = a1;
    err = double(float(sqrt(a2)));
  }
  const float rho_fin = rho_old;
  const float wmax = post_f32(float(emax), rho_fin);
  for (int i = threadIdx.x; i < n; i += kSmallThreads) wts[i] = __fdiv_rn(post_f32(se[i], rho_fin), wmax);
  if (threadIdx.x == 0) {
    rlvi_fp_result r;
    r.eps = 1.0 - double(avg);
    r.rho = double(rho_fin);
    r.sum_pi = S;
    r.err = err;
    r.iters = k;
    r.converged = converged;
    *p.result = r;
  }
}

template <typename T, typename K>
int launch_fp_small(rlvi_ctx* ctx, K kernel, const FpParams<T>& p, cudaStream_t stream) {
  const size_t smem = (size_t(p.n) * sizeof(T) + 15) & ~size_t(15);
  RLVI_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kSmallSmemBytes)));
  kernel<<<1, kSmallThreads, smem, stream>>>(p);
  RLVI_LAUNCH_CHECK(ctx);
  return RLVI_OK;
}

// ---- host launch -----------------------------------------------------------------------------
template <typename T, typename K>
int launch_fp(rlvi_ctx* ctx, K kernel, FpParams<T>& p, int64_t n_chunks, cudaStream_t stream, int cache_slots = 0) {
  int per_sm = 0;
  const size_t dyn_smem = size_t(cache_slots < 0 ? kFpRingDepth * kFpUnroll : cache_slots) * kFpThreads * sizeof(double2);
  p.cache_slots = cache_slots;
  {
    static const char* env = getenv("RLVI_FP_L2HEAD");      // =0 switches the L2-residency hints off (experiments)
    p.l2_head = (cache_slots < 0 && !(env && atoi(env) == 0)) ? 1 : 0;
  }
  if (dyn_smem > 0)
    RLVI_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(dyn_smem)));
  RLVI_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kFpThreads, dyn_smem));
  if (per_sm < 1) {
    rlvi_set_error("fixed-point kernel does not fit on an SM");
    return RLVI_ERR_CUDA;
  }
  if (per_sm > 4) per_sm = 4;
  int64_t max_grid = int64_t(ctx->sm_count) * per_sm;
  int64_t want = (n_chunks + int64_t(kFpThreads) * kFpUnroll - 1) / (int64_t(kFpThreads) * kFpUnroll);
  int grid = int(want < 1 ? 1 : (want > max_grid ? max_grid : want));
  RlviScratch s;
  const size_t part_bytes = size_t(2) * grid * 6 * sizeof(unsigned long long);   // [2 round parities][grid][3 doubles as LL words]
  int rc = rlvi_scratch_header(ctx, part_bytes, &s);
  if (rc != RLVI_OK) return rc;
  p.control = s.control;
  p.partials = s.partials;
  // The whole header (failure flag, local LL window) and the block partials are zeroed: LL tags start at 1, so a zeroed
  // (or any earlier call's) word never matches.
  RLVI_CUDA(cudaMemsetAsync(p.control, 0, kScratchHeaderBytes + part_bytes, stream));
  if (p.world == 1) p.inbox = s.fp_window;
  p.trace = nullptr;
  static const char* trace_env = getenv("RLVI_FP_TRACE");
  const size_t trace_bytes = size_t(kFpTraceRounds) * grid * 4 * sizeof(unsigned long long);
  if (trace_env && atoi(trace_env) != 0) {
    RLVI_CUDA(cudaMalloc(&p.trace, trace_bytes));
    RLVI_CUDA(cudaMemsetAsync(p.trace, 0, trace_bytes, stream));
  }
  void* args[] = {&p};
  RLVI_CUDA(cudaLaunchCooperativeKernel(reinterpret_cast<const void*>(kernel), dim3(grid), dim3(kFpThreads), args,
                                        dyn_smem, stream));
  RLVI_LAUNCH_CHECK(ctx);
  if (p.trace) {   // bring-up only: per round, when the blocks finished their trips / stored partials / saw the totals
    RLVI_CUDA(cudaStreamSynchronize(stream));
    unsigned long long* h = static_cast<unsigned long long*>(malloc(trace_bytes));
    cudaMemcpy(h, p.trace, trace_bytes, cudaMemcpyDeviceToHost);
    unsigned long long prev_done = 0ull;
    for (int r = 0; r < kFpTraceRounds; ++r) {
      const unsigned long long* t = h + size_t(r) * grid * 4;
      if (t[0] == 0ull) break;
      unsigned long long base = t[0];
      for (int b = 0; b < grid; ++b) if (t[b * 4] < base) base = t[b * 4];
      double a_min = 1e30, a_max = 0, a_mean = 0, st_max = 0, done_min = 1e30, done_max = 0, done_mean = 0;
      int argmax = 0;
      for (int b = 0; b < grid; ++b) {
        const double a = double(t[b * 4 + 0] - base), s1 = double(t[b * 4 + 1] - base), dn = double(t[b * 4 + 3] - base);
        if (a > a_max) { a_max = a; argmax = b; }
        a_min = a < a_min ? a : a_min;
        a_mean += a / grid;
        st_max = s1 > st_max ? s1 : st_max;
        done_min = dn < done_min ? dn : done_min;
        done_max = dn > done_max ? dn : done_max;
        done_mean += dn / grid;
      }
      fprintf(stderr, "[fp trace] round %2d: since prev done %7.0f ns | arrive min 0 mean %5.0f max %5.0f (block %d) | partials "
              "stored by %5.0f | block 0 arrived %5.0f published %5.0f | totals seen min %5.0f mean %5.0f max %5.0f\n", r,
              prev_done > 0ull ? double((long long)(base - prev_done)) : 0.0, a_mean, a_max, argmax, st_max, double(t[0] - base),
              double(t[2] - base), done_min, done_mean, done_max);
      if (grid >= 8) {      // arrival by eighths of the grid (which blocks are late?)
        fprintf(stderr, "           mean arrival by eighth of the grid:");
        for (int q = 0; q < 8; ++q) {
          double m = 0;
          const int lo = grid * q / 8, hi = grid * (q + 1) / 8;
          for (int b = lo; b < hi; ++b) m += double(t[b * 4 + 0] - base) / (hi - lo);
          fprintf(stderr, " %5.0f", m);
        }
        fprintf(stderr, "\n");
      }
      prev_done = base + (unsigned long long)done_mean;
    }
    free(h);
    cudaFree(p.trace);
  }
  return RLVI_OK;
}

template <typename T>
int fill_dist(FpParams<T>& p, const rlvi_fp_dist* dist, int64_t n) {
  p.rank = 0;
  p.world = 1;
  p.n_global = n;
  p.inbox = nullptr;
  p.peer_inbox = nullptr;
  p.call_index = 0;
  if (dist && dist->world > 1) {
    RLVI_REQUIRE(dist->world <= 32 && dist->rank >= 0 && dist->rank < dist->world, "bad rank/world");
    RLVI_REQUIRE(dist->inbox && dist->peer_inbox && dist->n_global >= n, "incomplete rlvi_fp_dist");
    RLVI_REQUIRE(p.maxiter < 4000, "sharded fixed point: maxiter must be below 4000 (sequence tags of the peer windows)");
    p.rank = dist->rank;
    p.world = dist->world;
    p.n_global = dist->n_global;
    p.inbox = dist->inbox;
    p.peer_inbox = dist->peer_inbox;
    p.call_index = dist->call_index;
  } else if (dist) {
    p.n_global = dist->n_global > 0 ? dist->n_global : n;
  }
  return RLVI_OK;
}

}  // namespace

// window layout (doubles): [0, 24 world) fixed-point slots (4 x world x 6 LL words) | [24 world, 26 world) statistics tags
// (2 parities) | then 2 parities x world x RLVI_DIST_STATS_CAPACITY statistics slots (dist.cu)
extern "C" int rlvi_fp_dist_inbox_doubles(int world) {
  return 24 * world + 2 * world + 2 * world * RLVI_DIST_STATS_CAPACITY;
}

static int fixed_point_f64_impl(rlvi_ctx* ctx, int variant, const double* losses, const double* scale,
                                double* e_work, int64_t n, double tol, int maxiter, double pi0, double* pi_out,
                                rlvi_fp_result* result, const rlvi_fp_dist* dist, void* stream);

// How the later passes get e[]: resident head in shared memory (small shards) or the bulk-copy ring.
// RLVI_FP_CACHE_SLOTS overrides (experiments, tests).
static int fp_cache_slots(int64_t n) {
  const char* env = getenv("RLVI_FP_CACHE_SLOTS");       // read per call: tests switch it
  if (env && *env) {
    const int v = atoi(env);
    return v < 0 ? -1 : (v > kFpCacheSlots ? kFpCacheSlots : v);
  }
  // <= 2^22 samples: keep the head of the vector resident in shared memory; larger: the buffer becomes a bulk-copy prefetch
  // ring (-1) -- from 2^23 samples on the ring wins even while the vector is L2 resident (12.9 vs 14.4 us per pass at 2^23,
  // 24.1 vs 27.9 at 2^24, 9.0 vs 8.1 at 2^22: tools/fp_pass_time.py), because its copies run ahead of the arithmetic
  return n <= (int64_t(1) << 22) ? kFpCacheSlots : -1;
}

// Series passes of the STANDARD kernel (on by default; the kernel switches from the data).  RLVI_FP_SERIES=0 streams
// every pass (A/B comparisons, tests); read per call.
static int fp_series_enabled() {
  const char* env = getenv("RLVI_FP_SERIES");
  return (env && *env && atoi(env) == 0) ? 0 : 1;
}

extern "C" int rlvi_fixed_point_f64(rlvi_ctx* ctx, int variant, const double* losses, const double* scale,
                                    double* e_work, int64_t n, double tol, int maxiter, double* pi_out,
                                    rlvi_fp_result* result, const rlvi_fp_dist* dist, void* stream) {
  return fixed_point_f64_impl(ctx, variant, losses, scale, e_work, n, tol, maxiter, 0.0, pi_out, result, dist, stream);
}

extern "C" int rlvi_fixed_point_init_f64(rlvi_ctx* ctx, int variant, const double* losses, const double* scale,
                                         double* e_work, int64_t n, double tol, int maxiter, double pi0,
                                         double* pi_out, rlvi_fp_result* result, const rlvi_fp_dist* dist,
                                         void* stream) {
  RLVI_REQUIRE(pi0 > 0.0 && pi0 < 1.0, "pi0 must be in (0, 1)");
  return fixed_point_f64_impl(ctx, variant, losses, scale, e_work, n, tol, maxiter, pi0, pi_out, result, dist, stream);
}

static int fixed_point_f64_impl(rlvi_ctx* ctx, int variant, const double* losses, const double* scale,
                                double* e_work, int64_t n, double tol, int maxiter, double pi0, double* pi_out,
                                rlvi_fp_result* result, const rlvi_fp_dist* dist, void* stream) {
  RLVI_REQUIRE(ctx && e_work && pi_out && result, "null pointer");
  RLVI_REQUIRE(n > 0, "n must be positive");
  RLVI_REQUIRE(maxiter >= 1, "maxiter must be >= 1");
  RLVI_REQUIRE(variant == RLVI_FP_STANDARD || variant == RLVI_FP_ONLINE, "FP64 variants: STANDARD, ONLINE");
  RLVI_REQUIRE(pi_out != e_work, "pi_out may not alias e_work");
  RlviDeviceGuard guard(ctx->device);
  FpParams<double> p;
  memset(&p, 0, sizeof(p));
  p.losses = losses;
  p.scale = scale;
  p.e = e_work;
  p.pi_out = pi_out;
  p.n = n;
  p.tol = tol;
  p.maxiter = maxiter;
  p.result = result;
  int rc = fill_dist(p, dist, n);
  if (rc != RLVI_OK) return rc;
  p.pi0 = pi0;
  p.series = fp_series_enabled();
  const bool vec = rlvi_aligned16(e_work) && rlvi_aligned16(pi_out) && (!losses || rlvi_aligned16(losses));
  const int64_t chunks = vec ? (n + 1) / 2 : n;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (p.world == 1 && size_t(n) * sizeof(double) <= kSmallSmemBytes && losses != pi_out)
    return variant == RLVI_FP_STANDARD ? launch_fp_small(ctx, fp_small_kernel_f64<RLVI_FP_STANDARD>, p, st)
                                       : launch_fp_small(ctx, fp_small_kernel_f64<RLVI_FP_ONLINE>, p, st);
  if (variant == RLVI_FP_STANDARD)
    return vec ? launch_fp(ctx, fp_kernel_f64<RLVI_FP_STANDARD, true>, p, chunks, st, fp_cache_slots(n))
               : launch_fp(ctx, fp_kernel_f64<RLVI_FP_STANDARD, false>, p, chunks, st);
  return vec ? launch_fp(ctx, fp_kernel_f64<RLVI_FP_ONLINE, true>, p, chunks, st, fp_cache_slots(n))
             : launch_fp(ctx, fp_kernel_f64<RLVI_FP_ONLINE, false>, p, chunks, st);
}

extern "C" int rlvi_fixed_point_deep_f32(rlvi_ctx* ctx, float* residuals, float* weights, float* e_work,
                                         int64_t n, float tol, int maxiter, rlvi_fp_result* result,
                                         const rlvi_fp_dist* dist, void* stream) {
  RLVI_REQUIRE(ctx && residuals && weights && e_work && result, "null pointer");
  RLVI_REQUIRE(n > 0, "n must be positive");
  RLVI_REQUIRE(maxiter >= 1, "maxiter must be >= 1");
  RlviDeviceGuard guard(ctx->device);
  FpParams<float> p;
  memset(&p, 0, sizeof(p));
  p.residuals = residuals;
  p.pi_out = weights;
  p.e = e_work;
  p.n = n;
  p.tol = double(tol);
  p.maxiter = maxiter;
  p.result = result;
  int rc = fill_dist(p, dist, n);
  if (rc != RLVI_OK) return rc;
  const bool vec = rlvi_aligned16(residuals) && rlvi_aligned16(weights) && rlvi_aligned16(e_work);
  const int64_t chunks = vec ? (n + 3) / 4 : n;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (p.world == 1 && size_t(n) * sizeof(float) <= kSmallSmemBytes)
    return launch_fp_small(ctx, fp_small_kernel_deep_f32, p, st);
  return vec ? launch_fp(ctx, fp_kernel_deep_f32<true>, p, chunks, st)
             : launch_fp(ctx, fp_kernel_deep_f32<false>, p, chunks, st);
}
