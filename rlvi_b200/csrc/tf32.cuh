// tf32.cuh -- shared by the TF32 weighted-Gram kernels (gram_tf32.cu: one CTA per SM, d <= 128; gram_tf32_pair.cu: CTA
// pairs, cta_group::2, d = 129..512): tensor-map encode entry point, tile constants, launch parameters, the cross-file
// host entry points, tcgen05 / TMA PTX wrappers.
#pragma once

#include <cuda.h>
#include <math.h>
#include <stdlib.h>

#include "tma.cuh"

namespace tf32 {


typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn encode_tiled_fn32() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

constexpr int kMB = 128;                     // feature block edge = UMMA M
constexpr int kR = 16;                       // rows per tile (two K = 8 steps)
constexpr int kChunkBytes = kR * 128;        // 32 floats x 16 rows
constexpr int kBlkBytes = 4 * kChunkBytes;   // one 128-feature block of one tile: 8 KiB
constexpr int kThreads = 512;
constexpr int kTpc = 8;                      // tiles per TMEM accumulation (128 rows)
constexpr int kSmemBudget = 200 * 1024;      // stages
constexpr int kTailBytes = 16 * 1024;        // barriers, TMEM slot, per-team reduction scratch
constexpr int kSmemTotal = kSmemBudget + kTailBytes + 1024;   // + alignment slack
constexpr int kFlushTiles = 16;              // column sums: FP32 per thread for 16 of the team's tiles, then FP64
constexpr int kPairTypes = 3;                // CTA-pair types (0,0), (0,1), (1,1) over 256-feature blocks

// What both routes read.  rlvi_weighted_moments_f32 fills the inputs and the scratch header (err, wmax); each route lays
// out its own G / column-sum partials behind the header (their shapes are in CtaParams / PairParams).
struct Tf32Params {
  const double* w;        // pi [n]
  const double* y;        // [n] or null
  int64_t n;
  int d;
  int power;
  int chunks_per_flush;   // register (level 2) accumulation length, in chunks
  int box3d;              // 1: one 3-D TMA box per feature block (d % 32 == 0); 0: four 2-D boxes
  double* gpart64;        // per-CTA FP64 partials of G
  double* spart;          // per-CTA FP64 partials of S1, Sy
  unsigned int* err;      // device flag: a bounded wait expired
  const unsigned long long* wmax;   // bits of max_i pi_i (device): the weights are normalised by a power of two
};

// The CTA-pair route of one call (gram_tf32_pair.cu), fixed before anything is queued.
struct PairPlan {
  int nsplit;                  // 1: TF32X1; 2: TF32X3 with BF16 corrections; 3: TF32X3 in TF32 (RLVI_TF32_PURE3=1)
  int ntypes;                  // 1 (d <= 256) or 3
  int first[kPairTypes + 1];   // first pair of each type; first[ntypes] = pairs, 0 when the device cannot hold ntypes
  int coef_blocks;             // blocks of the row-coefficient kernel
  size_t part_bytes;           // partials and row coefficients, behind the scratch header
};

// The even exponent e with max pi <= 2^e (0 when max pi is 0 or not finite): rows are scaled by pi 2^-e so that
// the FP32 products pi^2 x^2 of the collapse regime (SURVEY.md H1: pi ~ 1e-7 .. 1e-20) stay in FP32 range; the
// statistics are scaled back by exact powers of two in the finalize kernel.
__device__ __forceinline__ int weight_exponent(const unsigned long long* wmax) {
  const unsigned long long b = *wmax;
  const int ex = int((b >> 52) & 0x7FFull);
  if (ex == 0 || ex == 0x7FF) return 0;
  int e = ex - 1022;              // max pi = m 2^e, m in [0.5, 1)
  e += (e & 1);
  return e;
}

// ---- PTX wrappers ------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_2d_f32(uint32_t dst_smem, const CUtensorMap* tmap, int x, int y, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
          dst_smem),
      "l"(tmap), "r"(x), "r"(y), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_f32(uint32_t dst_smem, const CUtensorMap* tmap, int x, int y, int z, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
          dst_smem),
      "l"(tmap), "r"(x), "r"(y), "r"(z), "r"(smem_u32(bar))
      : "memory");
}
// round-to-nearest (ties away from zero in magnitude) onto the TF32 grid, on the bit pattern: what cvt.rna.tf32.f32
// computes, without its NaN/Inf special-casing (Inf stays Inf, NaN stays NaN under the mask)
__device__ __forceinline__ uint32_t to_tf32(float v) { return (__float_as_uint(v) + 0x1000u) & 0xFFFFE000u; }
// Packed FP32 pairs (SASS FMUL2 / FFMA2: two FP32 lanes per issue slot)
__device__ __forceinline__ float2 f2mul(float2 a, float2 b) {
  float2 r;
  asm("{.reg .b64 ra, rb, rc; mov.b64 ra, {%2,%3}; mov.b64 rb, {%4,%5}; mul.f32x2 rc, ra, rb; mov.b64 {%0,%1}, rc;}"
      : "=f"(r.x), "=f"(r.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
  return r;
}
__device__ __forceinline__ float2 f2fma(float2 a, float2 b, float2 c) {
  float2 r;
  asm("{.reg .b64 ra, rb, rc, rd; mov.b64 ra, {%2,%3}; mov.b64 rb, {%4,%5}; mov.b64 rc, {%6,%7}; fma.rn.f32x2 rd, ra, rb, rc; "
      "mov.b64 {%0,%1}, rd;}"
      : "=f"(r.x), "=f"(r.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
  return r;
}
// Dekker / Veltkamp split of FP32 onto the TF32 grid with FP32 arithmetic only: hi = the 11 significant bits of z rounded
// to nearest (C = 2^13 + 1: t = C z, hi = t - (t - z)), lo = z - hi exactly (|lo| <= 2^-11 |z|; the tensor core reads the
// upper 11 of its <= 13 significant bits).  Three / four packed instructions per TWO elements instead of two / four
// integer ones per element.
__device__ __forceinline__ float2 tf32_hi2(float2 z) {
  const float2 c = make_float2(8193.f, 8193.f), m1 = make_float2(-1.f, -1.f);
  const float2 t = f2mul(z, c);
  const float2 u = f2fma(z, m1, t);
  return f2fma(u, m1, t);
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tc_mma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// 32 lanes x 16 consecutive 32-bit columns -> 16 registers per thread (thread l = TMEM lane base + l)
__device__ __forceinline__ void tc_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// UMMA shared-memory descriptor, MN-major, SWIZZLE_128B_BASE32B: start >> 4 | LBO >> 4 << 16 | SBO >> 4 << 32 |
// version 1 << 46 | layout type 1 << 61.  LBO = byte stride between 32-feature column groups, SBO = between 4-row atoms.
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr) {
  return uint64_t((smem_addr & 0x3FFFFu) >> 4) | (uint64_t(kChunkBytes >> 4) << 16) | (uint64_t(512 >> 4) << 32) |
         (uint64_t(1) << 46) | (uint64_t(1) << 61);
}
// instruction descriptor: D = F32 (1 << 4), A = B = TF32 (2 << 7, 2 << 10), A and B MN-major (bits 15, 16),
// N >> 3 at bit 17, M >> 4 at bit 24
__device__ __forceinline__ uint32_t umma_idesc(int n_cols) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) | (uint32_t(n_cols >> 3) << 17) |
         (uint32_t(kMB >> 4) << 24);
}

// Bounded mbarrier wait: a protocol error must end in an error flag, never in a hung GPU.
__device__ __forceinline__ bool wait_or_abort(uint64_t* bar, uint32_t parity, unsigned int* err) {
  if (mbar_try_wait(bar, parity)) return true;
  const long long t0 = clock64();
  unsigned int spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 255u) == 0u) {
      if (clock64() - t0 > 6000000000LL) {
        atomicExch(err, 1u);
        return false;
      }
      if (*reinterpret_cast<volatile unsigned int*>(err) != 0u) return false;
    }
  }
  return true;
}

}  // namespace tf32

// gram_tf32_pair.cu.  rlvi_tf32_pair_plan: host-side queries only (d = 129..512).  rlvi_tf32_pair_moments: queues the
// route; `p` has the inputs and the scratch header filled in and the weight-maximum kernel queued, `part` is plan.part_bytes
// of scratch behind the header.
int rlvi_tf32_pair_plan(rlvi_ctx* ctx, int64_t n, int d, int power, bool has_y, int precision, tf32::PairPlan* plan);
int rlvi_tf32_pair_moments(rlvi_ctx* ctx, const CUtensorMap& tmap, const CUtensorMap& tmap3, const tf32::Tf32Params& p,
                           const tf32::PairPlan& plan, char* part, int want_gram, double* out, cudaStream_t st);
