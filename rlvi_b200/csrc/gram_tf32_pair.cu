// gram_tf32_pair.cu -- the TF32 weighted Gram of FP32-stored samples on CTA PAIRS (tcgen05.mma.cta_group::2, M = 256):
// the d = 129..512 shapes of rlvi_weighted_moments_f32 (config C3: N = 2^24, d = 512; d = 257..384 runs as 512 with the
// fourth 128-feature block zero-filled by the TMA).  Same
// statistics, same three-level accumulation and the same operand layout as gram_tf32.cu (read its header first);
// what changes is who computes what:
//
//   standard-learning/utils.py:82-84   PCA of the rows pi_i x_i      (power = 2:  G = sum pi_i^2 x_i x_i^T)
//   standard-learning/rlvi.py:70-71    sqrt(pi)-scaled least squares (power = 1:  G = sum pi_i x_i x_i^T)
//
// Why pairs.  The single-CTA kernel is bound by shared-memory bandwidth and by the tile loads, not by the tensor pipe
// (profiles/r02_tf32_stats.txt): a kind::tf32 instruction covers only K = 8 rows, so M128 x N256 reads 12 KiB of
// operands per 128 clk (96 of the SM's 128 B/clk) before the TMA fill and the in-place transform get any, and every
// CTA loads three 128-feature blocks per tile.  With cta_group::2 the two SMs of a TPC run ONE M = 256, N = 256
// instruction: each CTA supplies its 128 rows of A and only HALF of B (128 columns) from its own shared memory, the
// hardware shares the halves.  Per CTA and K step that is 8 KiB instead of 12, and a CTA loads / transforms one block
// per tile (diagonal pair: A half = B half) or two (off-diagonal) instead of three.
//
// Decomposition.  The features are cut into 256-wide pair blocks P (1 or 2 of them).  A pair of TYPE (P, Q), P <= Q,
// accumulates the 256 x 256 block G[P, Q]: CTA r holds rows 256 P + 128 r .. + 127 (TMEM lanes) x 256 columns.  Types:
// (0,0) for d <= 256; (0,0), (0,1), (1,1) for d <= 512.  Every type sweeps ALL row tiles, split over its own pairs
// (tile t of slot s: s, s + nslots, ...); the off-diagonal type has twice the load / transform work per tile and gets
// proportionally more pairs.  CTA r of a diagonal pair also owns the column sums of feature block 2 P + r.
//
// Per CTA, warp-specialised (16 warps; setmaxnreg 96 for warpgroups 0-1, 160 for warpgroups 2-3):
//   warp 0      TMA producer: per tile ONE 3-D tensor-map box per loaded feature block (32 floats x 16 rows x 4 column
//               groups) + bulk copies of the tile's FP32 row coefficients (written once per call by pair_coef_kernel: no
//               FP64 instruction runs in this kernel's inner loops -- FP64 issued while the tensor pipe is busy waits for it);
//   warp 1      MMA issuer, in the LEADER CTA (cluster rank 0) only: tcgen05.mma.cta_group::2.kind::tf32, then
//               tcgen05.commit ... multicast::cluster releases the stage (`empty`) and publishes the chunk (`tfull`) in
//               both CTAs;
//   warps 2-7   six single-warp TRANSFORM workers, tile t -> worker t mod 6, in place on the landed tile (z = s x split into
//               TF32 hi + exact remainder lo with packed FP32 arithmetic); a finished tile is announced by one elected
//               lane per CTA on the LEADER's `ready` barrier (remote mbarrier arrive, default scope);
//   warps 8-15  ACCUMULATOR warps: TMEM -> registers (tcgen05.ld) every 128 rows, FP64 partials every 32 Ki rows; they arrive
//               on the leader's `tempty`;
//   cluster barriers after set-up and before TMEM is freed, and each producer drains its `empty` barriers before
//   leaving, so no multicast arrive can land in a CTA that has exited.
// Measured history and what bounded each version: profiles/r02_tf32_pair_stats.txt.
#include "tf32.cuh"

namespace {

using namespace tf32;

constexpr int kPairStages = 12;             // upper bound; the ring uses min(kPairStages, budget / stage bytes)
constexpr int kWorkers = 6;                 // transform warps per CTA (warps 2-7), one whole 16-row tile each
constexpr int kCoefBytes = 256;             // per stage: s, c1, cy of the tile's 16 rows (64 B each)
constexpr int kCoefThreads = 256;

struct PairParams {
  Tf32Params b;                 // gpart64: [grid][2][128][128]; spart: [grid][kWorkers][2][128] (diagonal pairs)
  int nbp;                      // 256-feature pair blocks: 1 or 2
  int ntypes;                   // 1 or 3
  int first[kPairTypes + 1];    // first pair of each type; first[ntypes] = number of pairs (grid = 2 x that)
  // per-row FP32 coefficients written by pair_coef_kernel (padded with zeros to a multiple of kR rows):
  const float* coef_sc;         // s_i: z_i = s_i x_i
  const float* coef_c1;         // the X^T pi coefficient; == coef_sc for power 2
  const float* coef_cy;         // the X^T (w y) coefficient, or null
  double* s0blocks;             // [coef_blocks][2] partial S0 / Swy of the coefficient kernel
  int coef_blocks;
  long long* stats;             // optional [grid][8] per-role cycle counters (RLVI_TF32_STATS=1)
};

__host__ __device__ __forceinline__ void pair_type(int t, int nbp, int& pa, int& pb) {
  if (nbp == 1 || t == 0) {
    pa = 0;
    pb = 0;
  } else if (t == 1) {
    pa = 0;
    pb = 1;
  } else {
    pa = 1;
    pb = 1;
  }
}

// ---- cluster-scope PTX ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `local` (a shared::cta address of THIS CTA) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t map_to_cta(uint32_t local, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  // default semantics (release at CTA scope), as CUTLASS's ClusterBarrier::arrive(cta_id): the data the waiter needs are
  // this CTA's shared-memory writes, published to the tensor core by fence.proxy.async; a release.cluster arrive costs
  // ~1100 clk per call (measured, profiles/r02_tf32_pair_ablation.txt)
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ bool wait_or_abort_cluster(uint64_t* bar, uint32_t parity, unsigned int* err) {
  if (mbar_try_wait_cluster(bar, parity)) return true;
  const long long t0 = clock64();
  unsigned int spins = 0;
  while (!mbar_try_wait_cluster(bar, parity)) {
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
__device__ __forceinline__ void tc2_commit_both(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"((unsigned short)3)
      : "memory");
}
__device__ __forceinline__ void tc2_mma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// BF16 correction products of the mixed mode (NSPLIT == 2): kind::f16, K = 16 per instruction
__device__ __forceinline__ void tc2_mma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D = F32, A = B = BF16 (format 1 at bits 7 and 10), both MN-major, N >> 3 at bit 17, M = 256
__device__ __forceinline__ uint32_t umma_idesc_pair_bf16(int n_cols) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | (uint32_t(n_cols >> 3) << 17) |
         (uint32_t(256 >> 4) << 24);
}
// 16-bit MN-major operand block (128 features x 16 rows = 4 KiB), SWIZZLE_128B: atom = 64 features (128 B) x 8 rows,
// LBO = 2048 B between the two feature atoms, SBO = 1024 B between the two 8-row groups (tools/bf16_debug.cu,
// profiles/r02_bf16_descriptor_probe.txt)
constexpr int kBlk16Bytes = 4096;
__device__ __forceinline__ uint64_t umma_desc_bf16(uint32_t smem_addr) {
  return uint64_t((smem_addr & 0x3FFFFu) >> 4) | (uint64_t(2048 >> 4) << 16) | (uint64_t(1024 >> 4) << 32) |
         (uint64_t(1) << 46) | (uint64_t(2) << 61);
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {      // lo -> bits 0..15
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
// instruction descriptor of the pair instruction: as umma_idesc, M = 256
__device__ __forceinline__ uint32_t umma_idesc_pair(int n_cols) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) | (uint32_t(n_cols >> 3) << 17) |
         (uint32_t(256 >> 4) << 24);
}

struct PairCtx {
  unsigned char* smem;
  uint64_t *full_bar, *empty_bar, *tfull_bar;
  uint32_t ready_remote, tempty_remote;    // the LEADER's `ready[0]` / `tempty[0]` as shared::cluster addresses
  float* red_all;            // [kWorkers][2][128] column-sum exchange, private to each transform warp
  uint32_t tmem_base;
  int stage_bytes, nst, nfb, slot, nslots;
  int my_tiles, my_chunks;
  bool c1_is_sc;             // power 2: the column-sum coefficient is the row scale itself
  uint32_t coef_off;         // byte offset of the coefficient slots (kCoefBytes per stage) behind the stages
};

// One TRANSFORM warp (worker w of kWorkers): tiles w, w + kWorkers, ... of the CTA, in place on the landed tile:
// z = s_i x rounded to TF32 (Z_hi) and, for 3xTF32, the remainder Z_lo into the second buffer; with HAS_SUMS (diagonal
// pairs) the column sums of the CTA's feature block ride along.  Single warps (not four-warp teams): a tile's transform
// is a chain of dependent shared-memory round trips whose latency triples under load, so what counts is how many
// tiles are in flight, and a warp needs no barrier but __syncwarp.
template <int NSPLIT, bool HAS_Y, bool HAS_SUMS>
__device__ __forceinline__ void pair_transform_warp(const PairParams& pp, const PairCtx& cx, const int worker) {
  const Tf32Params& p = pp.b;
  unsigned char* smem = cx.smem;
  uint64_t *full_bar = cx.full_bar, *empty_bar = cx.empty_bar;
  const int stage_bytes = cx.stage_bytes, nst = cx.nst, nfb = cx.nfb, slot = cx.slot;
  const int my_tiles = cx.my_tiles;
  const int lane = threadIdx.x & 31;
  const int q = lane & 7, r4 = lane >> 3;                // logical 16-byte unit, row within a pass of 4 rows
  // SWIZZLE_128B_ATOM_32B: the 32-byte unit q >> 1 of row rr sits at unit (q >> 1) ^ (rr & 3); rr & 3 = r4 in every pass
  const uint32_t off0 = uint32_t(r4 * 128 + (((((q >> 1) ^ r4) << 1) | (q & 1)) << 4));
  const uint32_t lo_off = uint32_t(nfb * kBlkBytes);
  float* red = cx.red_all + worker * 256;
  float2 s1acc[HAS_SUMS ? 4 : 1][2], syacc[(HAS_SUMS && HAS_Y) ? 4 : 1][2];       // [chunk][float pair of the 16-byte unit]
#pragma unroll
  for (int c = 0; c < (HAS_SUMS ? 4 : 1); ++c) s1acc[c][0] = s1acc[c][1] = make_float2(0.f, 0.f);
#pragma unroll
  for (int c = 0; c < ((HAS_SUMS && HAS_Y) ? 4 : 1); ++c) syacc[c][0] = syacc[c][1] = make_float2(0.f, 0.f);
  double s1d[4] = {0.0, 0.0, 0.0, 0.0}, syd[4] = {0.0, 0.0, 0.0, 0.0};
  bool ok = true;

  // FP32 column sums of the last kFlushTiles tiles -> FP64 (lane l keeps columns l, l + 32, l + 64, l + 96)
  auto flush_sums = [&]() {
    if (HAS_SUMS) {
      if (NSPLIT == 2 && (r4 & 1)) {      // odd rows accumulated chunk c ^ 1 in slot c (see the chunk order below)
#pragma unroll
        for (int c = 0; c < (HAS_SUMS ? 4 : 1); c += 2)
#pragma unroll
          for (int k = 0; k < 2; ++k) {
            const float2 t1 = s1acc[c][k];
            s1acc[c][k] = s1acc[HAS_SUMS ? c + 1 : 0][k];
            s1acc[HAS_SUMS ? c + 1 : 0][k] = t1;
            if (HAS_Y) {
              const float2 t2 = syacc[(HAS_SUMS && HAS_Y) ? c : 0][k];
              syacc[(HAS_SUMS && HAS_Y) ? c : 0][k] = syacc[(HAS_SUMS && HAS_Y) ? c + 1 : 0][k];
              syacc[(HAS_SUMS && HAS_Y) ? c + 1 : 0][k] = t2;
            }
          }
      }
#pragma unroll
      for (int c = 0; c < (HAS_SUMS ? 4 : 1); ++c)
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          float v = (k & 1) ? s1acc[c][k >> 1].y : s1acc[c][k >> 1].x;
          v += __shfl_xor_sync(0xffffffffu, v, 8);
          v += __shfl_xor_sync(0xffffffffu, v, 16);
          if (lane < 8) red[c * 32 + lane * 4 + k] = v;
          if (HAS_Y) {
            float u = (k & 1) ? syacc[(HAS_SUMS && HAS_Y) ? c : 0][k >> 1].y : syacc[(HAS_SUMS && HAS_Y) ? c : 0][k >> 1].x;
            u += __shfl_xor_sync(0xffffffffu, u, 8);
            u += __shfl_xor_sync(0xffffffffu, u, 16);
            if (lane < 8) red[128 + c * 32 + lane * 4 + k] = u;
          }
        }
#pragma unroll
      for (int c = 0; c < (HAS_SUMS ? 4 : 1); ++c) s1acc[c][0] = s1acc[c][1] = make_float2(0.f, 0.f);
#pragma unroll
      for (int c = 0; c < ((HAS_SUMS && HAS_Y) ? 4 : 1); ++c) syacc[c][0] = syacc[c][1] = make_float2(0.f, 0.f);
      __syncwarp();
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        s1d[j] += double(red[j * 32 + lane]);
        if (HAS_Y) syd[j] += double(red[128 + j * 32 + lane]);
      }
      __syncwarp();
    }
  };

  int done = 0;
  long long t_full = 0, t_busy = 0;
  int s = worker % nst;
  uint32_t ph = uint32_t(worker / nst) & 1u;
  for (int it = worker; it < my_tiles; it += kWorkers) {
    const long long k1 = pp.stats ? clock64() : 0;
    // see gram_tf32.cu: `empty` one phase back first, so that `full` cannot be mistaken for the previous phase
    ok = wait_or_abort(&empty_bar[s], ph ^ 1u, p.err) && wait_or_abort(&full_bar[s], ph, p.err);
    if (!ok) break;
    const long long k2 = pp.stats ? clock64() : 0;
    t_full += k2 - k1;
    unsigned char* sb = smem + size_t(s) * stage_bytes;
    // the tile's row coefficients arrived with it (FP32, from pair_coef_kernel): no FP64 and no global load in this loop --
    // FP64 instructions issued while the tensor pipe is busy wait for it (stall_math was 47 % of these warps' time)
    const float* cf = reinterpret_cast<const float*>(smem + cx.coef_off + uint32_t(s) * kCoefBytes);
#pragma unroll
    for (int pass = 0; pass < kR / 4; ++pass) {
      const int rr = pass * 4 + r4;
      const float sc = cf[rr];
      const float c1 = cx.c1_is_sc ? sc : cf[kR + rr];
      const float cy = HAS_Y ? cf[2 * kR + rr] : 0.f;
      const float2 scv = make_float2(sc, sc), c1v = make_float2(c1, c1), cyv = make_float2(cy, cy), m1v = make_float2(-1.f, -1.f);
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        if (i < nfb) {
          const bool sums = HAS_SUMS && (i == 0);
#pragma unroll
          for (int c0 = 0; c0 < 4; ++c0) {
            // mixed mode: odd rows of a pass take the chunks in the order 1, 0, 3, 2, so that the 8-byte BF16 stores of the
            // four rows spread over both halves of the 128-byte lines (2 wavefronts per store instead of 4)
            const int c = (NSPLIT == 2) ? (c0 ^ (r4 & 1)) : c0;
            float4* ptr = reinterpret_cast<float4*>(sb + i * kBlkBytes + c * kChunkBytes + pass * 512 + off0);
            const float4 x = *ptr;
            const float2 xa = make_float2(x.x, x.y), xb = make_float2(x.z, x.w);
            if (sums) {
              s1acc[HAS_SUMS ? c0 : 0][0] = f2fma(xa, c1v, s1acc[HAS_SUMS ? c0 : 0][0]);
              s1acc[HAS_SUMS ? c0 : 0][1] = f2fma(xb, c1v, s1acc[HAS_SUMS ? c0 : 0][1]);
              if (HAS_Y) {
                syacc[(HAS_SUMS && HAS_Y) ? c0 : 0][0] = f2fma(xa, cyv, syacc[(HAS_SUMS && HAS_Y) ? c0 : 0][0]);
                syacc[(HAS_SUMS && HAS_Y) ? c0 : 0][1] = f2fma(xb, cyv, syacc[(HAS_SUMS && HAS_Y) ? c0 : 0][1]);
              }
            }
            const float2 za = f2mul(xa, scv), zb = f2mul(xb, scv);
            const float2 ha = tf32_hi2(za), hb = tf32_hi2(zb);
            *ptr = make_float4(ha.x, ha.y, hb.x, hb.y);
            if (NSPLIT == 3) {
              const float2 la = f2fma(ha, m1v, za), lb = f2fma(hb, m1v, zb);       // exact remainders
              *reinterpret_cast<float4*>(reinterpret_cast<unsigned char*>(ptr) + lo_off) = make_float4(la.x, la.y, lb.x, lb.y);
            }
            if (NSPLIT == 2) {
              // mixed mode: the two correction products run as BF16 (K = 16 per instruction, half the tensor time and half
              // the operand bytes of a TF32 pass): z to 8 bits and the exact remainder to 8 bits, in the 16-bit operands'
              // own MN-major layout.  Features 32 c + 4 q .. + 3 of row rr: 8 bytes in 16-byte unit 4 (c & 1) + (q >> 1)
              // (XOR rr & 7) of the row's 128-byte line, feature atom c >> 1, row group rr >> 3.
              const float2 la = f2fma(ha, m1v, za), lb = f2fma(hb, m1v, zb);
              const uint32_t o16 = uint32_t((c >> 1) * 2048 + (rr >> 3) * 1024 + (rr & 7) * 128 +
                                            (((4 * (c & 1) + (q >> 1)) ^ (rr & 7)) << 4) + (q & 1) * 8);
              unsigned char* h16 = sb + nfb * kBlkBytes + i * kBlk16Bytes + o16;
              *reinterpret_cast<uint2*>(h16) = make_uint2(pack_bf16x2(za.x, za.y), pack_bf16x2(zb.x, zb.y));
              *reinterpret_cast<uint2*>(h16 + nfb * kBlk16Bytes) = make_uint2(pack_bf16x2(la.x, la.y), pack_bf16x2(lb.x, lb.y));
            }
          }
        }
      }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic writes -> visible to the tensor core
    __syncwarp();
    if (lane == 0) mbar_arrive_cluster(cx.ready_remote + uint32_t(s) * 8u);   // the leader's barrier: 1 + 1 warps per tile
    if ((++done % kFlushTiles) == 0) flush_sums();
    s += kWorkers;
    while (s >= nst) {
      s -= nst;
      ph ^= 1u;
    }
    if (pp.stats) t_busy += clock64() - k2;
  }
  if (pp.stats && lane == 0 && worker == 0) {
    pp.stats[size_t(blockIdx.x) * 8 + 1] = t_full * kWorkers;   // scaled to "per tile of the CTA" like the other roles
    pp.stats[size_t(blockIdx.x) * 8 + 2] = t_busy * kWorkers;
  }
  if (ok) {
    flush_sums();
    if (HAS_SUMS) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        p.spart[((size_t(blockIdx.x) * kWorkers + worker) * 2 + 0) * 128 + j * 32 + lane] = s1d[j];
        p.spart[((size_t(blockIdx.x) * kWorkers + worker) * 2 + 1) * 128 + j * 32 + lane] = syd[j];
      }
    }
  }
}

// One ACCUMULATOR warp (warps 8-15): TMEM lanes 32 (warp % 4) .. + 31 of column half h = (warp - 8) / 4.  The tensor core
// adds in FP32 with truncation, so a TMEM accumulator only lives for kTpc tiles; it is read back (tcgen05.ld) and
// added, round-to-nearest, into 128 FP32 registers, themselves flushed into the CTA's FP64 partial every
// `chunks_per_flush` chunks.  Two TMEM buffers alternate, so chunk c is drained while chunk c + 1 accumulates.
__device__ __forceinline__ void pair_acc_warp(const PairParams& pp, const PairCtx& cx) {
  const Tf32Params& p = pp.b;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int h = (warp - 8) >> 2, quarter = warp & 3;
  float acc[128];
#pragma unroll
  for (int i = 0; i < 128; ++i) acc[i] = 0.f;
  double* gp = p.gpart64 + ((size_t(blockIdx.x) * 2 + h) * 128 + size_t(quarter * 32 + lane)) * 128;
  bool flushed = false;
  bool ok = true;
  long long t_drain = 0;
  auto flush_acc = [&]() {
#pragma unroll
    for (int i = 0; i < 128; i += 2) {
      double2 v = make_double2(double(acc[i]), double(acc[i + 1]));
      if (flushed) {
        const double2 o = *reinterpret_cast<const double2*>(gp + i);
        v.x += o.x;
        v.y += o.y;
      }
      *reinterpret_cast<double2*>(gp + i) = v;
      acc[i] = 0.f;
      acc[i + 1] = 0.f;
    }
    flushed = true;
  };
  for (int ch = 0; ch < cx.my_chunks; ++ch) {
    const int buf = ch & 1;
    if (!wait_or_abort(&cx.tfull_bar[buf], uint32_t(ch >> 1) & 1u, p.err)) {
      ok = false;
      break;
    }
    const long long k0 = pp.stats ? clock64() : 0;
    tc_fence_after();
    {
      const uint32_t taddr = cx.tmem_base + (uint32_t(quarter * 32) << 16) + uint32_t(buf * 256 + h * 128);
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        float v[16];
        tc_ld16(taddr + uint32_t(c * 16), v);
#pragma unroll
        for (int j = 0; j < 16; ++j) acc[c * 16 + j] += v[j];
      }
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive_cluster(cx.tempty_remote + uint32_t(buf) * 8u);
    if (((ch + 1) % p.chunks_per_flush) == 0) flush_acc();
    if (pp.stats) t_drain += clock64() - k0;
  }
  if (pp.stats && lane == 0 && warp == 8) pp.stats[size_t(blockIdx.x) * 8 + 6] = t_drain * kTpc;   // per chunk -> per 8 tiles
  if (ok) flush_acc();
}

template <int NSPLIT, bool HAS_Y>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
    gram_tf32_pair_kernel(const __grid_constant__ CUtensorMap tmap2, const __grid_constant__ CUtensorMap tmap3,
                          const PairParams pp) {
  const Tf32Params& p = pp.b;
  extern __shared__ unsigned char smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  unsigned char* smem = smem_raw + ((1024u - (raw & 1023u)) & 1023u);   // same offset in both CTAs of the pair
  const uint32_t smem_base = smem_u32(smem);
  unsigned char* tail = smem + kSmemBudget;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(tail);          // [kPairStages] TMA -> transform (own CTA)
  uint64_t* ready_bar = full_bar + kPairStages;                     // [kPairStages] transform (both CTAs) -> MMA (leader)
  uint64_t* empty_bar = ready_bar + kPairStages;                    // [kPairStages] MMA -> TMA (multicast to both)
  uint64_t* tfull_bar = empty_bar + kPairStages;                    // [2] MMA -> accumulator warps (multicast)
  uint64_t* tempty_bar = tfull_bar + 2;                             // [2] accumulator warps (both CTAs) -> MMA (leader)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
  float* red_all = reinterpret_cast<float*>(tail + 512);            // [kWorkers][2][128] column-sum exchange (per warp)

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1;
  int type = 0;
  while (type + 1 < pp.ntypes && pair >= pp.first[type + 1]) ++type;
  const int slot = pair - pp.first[type];
  const int nslots = pp.first[type + 1] - pp.first[type];
  int pa, pb;
  pair_type(type, pp.nbp, pa, pb);
  const bool diag = (pa == pb);
  const int fb_a = 2 * pa + int(rank), fb_b = 2 * pb + int(rank);
  const int nfb = diag ? 1 : 2;
  const uint32_t a_off = 0u, b_off = diag ? 0u : uint32_t(kBlkBytes);
  const int stage_bytes = nfb * kBlkBytes * (NSPLIT == 1 ? 1 : 2);      // mixed mode: 8 KiB TF32 hi + 2 x 4 KiB BF16 per block
  int nst = (kSmemBudget - kPairStages * kCoefBytes) / stage_bytes;
  if (nst > kPairStages) nst = kPairStages;
  const uint32_t coef_off = uint32_t(nst) * uint32_t(stage_bytes);      // coefficient slots behind the stages
  const int ntiles = int((p.n + kR - 1) / kR);
  const int my_tiles = (ntiles > slot) ? (ntiles - slot + nslots - 1) / nslots : 0;
  const int my_chunks = (my_tiles + kTpc - 1) / kTpc;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kPairStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&ready_bar[s], 2);      // the tile's transform warp of each CTA
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tfull_bar[b], 1);
      mbar_init(&tempty_bar[b], 16);    // 8 accumulator warps of each CTA
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {   // TMEM of both SMs: all 512 columns (two 256-column accumulator buffers)
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();              // the peer's barriers are initialised before anything arrives on them
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);

  PairCtx cx;
  cx.smem = smem;
  cx.full_bar = full_bar;
  cx.empty_bar = empty_bar;
  cx.tfull_bar = tfull_bar;
  cx.ready_remote = map_to_cta(smem_u32(ready_bar), 0u);
  cx.tempty_remote = map_to_cta(smem_u32(tempty_bar), 0u);
  cx.red_all = red_all;
  cx.tmem_base = tmem_base;
  cx.stage_bytes = stage_bytes;
  cx.nst = nst;
  cx.nfb = nfb;
  cx.slot = slot;
  cx.nslots = nslots;
  cx.my_tiles = my_tiles;
  cx.my_chunks = my_chunks;
  cx.c1_is_sc = (pp.coef_c1 == pp.coef_sc);
  cx.coef_off = coef_off;

  if (warp < 8) {
    // ===== warpgroups 0, 1: TMA producer (warp 0, both CTAs), MMA issuer (warp 1 of the leader), six transform warps ======
    asm volatile("setmaxnreg.dec.sync.aligned.u32 96;");
    if (warp == 0 && lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      long long t_wait = 0;
      const long long t_begin = clock64();
      bool ok = true;
      for (int it = 0; it < my_tiles; ++it) {
        const long long c0 = pp.stats ? clock64() : 0;
        if (!wait_or_abort(&empty_bar[s], ph ^ 1u, p.err)) {
          ok = false;
          break;
        }
        if (pp.stats) t_wait += clock64() - c0;
        const int row0 = (slot + it * nslots) * kR;
        const uint32_t sb = smem_base + uint32_t(s) * uint32_t(stage_bytes);
        const bool c1_sep = (pp.coef_c1 != pp.coef_sc);
        const uint32_t coef_tx = uint32_t(kR * 4) * (1u + (c1_sep ? 1u : 0u) + (HAS_Y ? 1u : 0u));
        mbar_arrive_expect_tx(&full_bar[s], uint32_t(nfb * kBlkBytes) + coef_tx);
        {
          unsigned char* cdst = smem + coef_off + uint32_t(s) * kCoefBytes;
          bulk_g2s(cdst, pp.coef_sc + row0, kR * 4, &full_bar[s]);
          if (c1_sep) bulk_g2s(cdst + kR * 4, pp.coef_c1 + row0, kR * 4, &full_bar[s]);
          if (HAS_Y) bulk_g2s(cdst + 2 * kR * 4, pp.coef_cy + row0, kR * 4, &full_bar[s]);
        }
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          if (i < nfb) {
            const int fbi = (i == 0) ? fb_a : fb_b;
            if (p.box3d) {       // one box: 32 floats x 16 rows x 4 column groups
              tma_load_3d_f32(sb + uint32_t(i * kBlkBytes), &tmap3, 0, row0, fbi * 4, &full_bar[s]);
            } else {
#pragma unroll
              for (int c = 0; c < 4; ++c)
                tma_load_2d_f32(sb + uint32_t(i * kBlkBytes + c * kChunkBytes), &tmap2, fbi * kMB + c * 32, row0,
                                &full_bar[s]);
            }
          }
        }
        if (++s == nst) {
          s = 0;
          ph ^= 1u;
        }
      }
      // tail: every release of a stage this CTA filled must have landed before the CTA may exit (multicast arrives
      // from the leader's tcgen05.commit target this CTA's shared memory)
      for (int k = 0; ok && k < nst && k < my_tiles; ++k) {
        if (!wait_or_abort(&empty_bar[s], ph ^ 1u, p.err)) break;
        if (++s == nst) {
          s = 0;
          ph ^= 1u;
        }
      }
      if (pp.stats) {
        pp.stats[size_t(blockIdx.x) * 8 + 0] = t_wait;
        pp.stats[size_t(blockIdx.x) * 8 + 7] = clock64() - t_begin;
      }
    } else if (warp == 1 && lane == 0 && rank == 0) {
      const uint32_t idesc = umma_idesc_pair(256);
      const uint32_t idesc16 = umma_idesc_pair_bf16(256);
      const uint32_t lo_off = uint32_t(nfb * kBlkBytes);   // Z_lo blocks follow the Z_hi blocks of a stage
      const uint64_t dconst = umma_desc(0);
      auto desc = [&](uint32_t addr) { return dconst | uint64_t((addr & 0x3FFFFu) >> 4); };
      int s = 0;
      uint32_t ph = 0;
      bool ok = true;
      long long t_ready = 0, t_tempty = 0, t_issue = 0;
      for (int it = 0; it < my_tiles && ok; ++it) {
        const int ch = it / kTpc;
        const int tin = it - ch * kTpc;
        const int buf = ch & 1;
        const long long c0 = pp.stats ? clock64() : 0;     // (the issuer's loop is on the critical path: no clock reads unless asked)
        if (tin == 0) {
          ok = wait_or_abort_cluster(&tempty_bar[buf], (uint32_t(ch >> 1) & 1u) ^ 1u, p.err);
          if (!ok) break;
          tc_fence_after();
        }
        const long long c1 = pp.stats ? clock64() : 0;
        ok = wait_or_abort_cluster(&ready_bar[s], ph, p.err);
        if (!ok) break;
        tc_fence_after();
        const long long c2 = pp.stats ? clock64() : 0;
        t_tempty += c1 - c0;
        t_ready += c2 - c1;
        const uint32_t sb = smem_base + uint32_t(s) * uint32_t(stage_bytes);
        const uint32_t dcol = tmem_base + uint32_t(buf * 256);
#pragma unroll
        for (int ks = 0; ks < kR / 8; ++ks) {
          const uint32_t first = (tin == 0 && ks == 0) ? 0u : 1u;
          const uint32_t kb = sb + uint32_t(ks * 1024);
          const uint64_t a_hi = desc(kb + a_off), b_hi = desc(kb + b_off);
          tc2_mma_tf32(dcol, a_hi, b_hi, idesc, first);
          if (NSPLIT == 3) {
            tc2_mma_tf32(dcol, desc(kb + lo_off + a_off), b_hi, idesc, 1u);
            tc2_mma_tf32(dcol, a_hi, desc(kb + lo_off + b_off), idesc, 1u);
          }
        }
        if (NSPLIT == 2) {      // lo . hi + hi . lo in BF16: one K = 16 instruction each for the whole tile
          const uint32_t h16 = sb + uint32_t(nfb * kBlkBytes), l16 = h16 + uint32_t(nfb * kBlk16Bytes);
          const uint32_t a16 = a_off / 2u, b16 = b_off / 2u;     // block index x 4 KiB
          tc2_mma_bf16(dcol, umma_desc_bf16(l16 + a16), umma_desc_bf16(h16 + b16), idesc16, 1u);
          tc2_mma_bf16(dcol, umma_desc_bf16(h16 + a16), umma_desc_bf16(l16 + b16), idesc16, 1u);
        }
        tc2_commit_both(&empty_bar[s]);                                        // stage free in both CTAs
        if (tin == kTpc - 1 || it == my_tiles - 1) tc2_commit_both(&tfull_bar[buf]);   // chunk complete in both TMEMs
        if (pp.stats) t_issue += clock64() - c2;
        if (++s == nst) {
          s = 0;
          ph ^= 1u;
        }
      }
      if (pp.stats) {
        pp.stats[size_t(blockIdx.x) * 8 + 3] = t_ready;
        pp.stats[size_t(blockIdx.x) * 8 + 4] = t_tempty;
        pp.stats[size_t(blockIdx.x) * 8 + 5] = t_issue;
      }
    } else if (warp >= 2) {
      if (diag) pair_transform_warp<NSPLIT, HAS_Y, true>(pp, cx, warp - 2);
      else pair_transform_warp<NSPLIT, HAS_Y, false>(pp, cx, warp - 2);
    }
  } else {
    // ===== warpgroups 2, 3: the accumulator warps (TMEM -> FP32 registers -> FP64 partials) ===========================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 160;");
    pair_acc_warp(pp, cx);
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();              // both CTAs are done with each other's shared memory, barriers and TMEM
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// Row coefficients in FP32, once per call (HBM-bound, ~20 B per row): s_i = pi_i 2^-e (power 2) or sqrt(pi_i 2^-e)
// (power 1) -- the factor of z_i = s_i x_i --, c1_i = pi_i 2^-e for X^T pi, cy_i = w_i y_i (normalised) for X^T (w y);
// rows n .. npad - 1 are zero.  Also S0 = sum w_i and Swy = sum w_i y_i in FP64 (w = pi^2 or pi), as per-block partials.
__global__ void __launch_bounds__(kCoefThreads) pair_coef_kernel(const double* __restrict__ w, const double* __restrict__ y,
                                                                 int64_t n, int64_t npad, int power,
                                                                 const unsigned long long* wmax, float* __restrict__ sc,
                                                                 float* __restrict__ c1, float* __restrict__ cy,
                                                                 double* __restrict__ s0blocks) {
  const double wscale = ldexp(1.0, -weight_exponent(wmax));      // exact power of two
  double s0 = 0.0, swy = 0.0;
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < npad; i += int64_t(gridDim.x) * blockDim.x) {
    const double pid = (i < n) ? w[i] : 0.0;
    const double yd = (y && i < n) ? y[i] : 0.0;
    const double wd = (power == 2) ? pid * pid : pid;
    const double pis = pid * wscale;                               // normalised weight, <= 1
    sc[i] = (power == 2) ? float(pis) : float(sqrt(pis));
    if (c1 != sc) c1[i] = float(pis);
    if (cy) cy[i] = float(((power == 2) ? pis * pis : pis) * yd);
    s0 += wd;
    swy = fma(wd, yd, swy);
  }
  __shared__ double red[2][kCoefThreads / 32];
  s0 = warp_sum(s0);
  swy = warp_sum(swy);
  if ((threadIdx.x & 31) == 0) {
    red[0][threadIdx.x >> 5] = s0;
    red[1][threadIdx.x >> 5] = swy;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0.0, b = 0.0;
    for (int k = 0; k < kCoefThreads / 32; ++k) {
      a += red[0][k];
      b += red[1][k];
    }
    s0blocks[size_t(blockIdx.x) * 2 + 0] = a;
    s0blocks[size_t(blockIdx.x) * 2 + 1] = b;
  }
}

// Sum the per-CTA partials in slot order, mirror the upper triangle, write [S0, Swy, S1, Sy, G] (FP64).
__global__ void __launch_bounds__(256) gram_tf32_pair_finalize_kernel(const PairParams pp, int has_y, int want_gram,
                                                                      double* out) {
  const Tf32Params& p = pp.b;
  const int d = p.d, nb = 2 * pp.nbp;
  const int npairs_blk = nb * (nb + 1) / 2;
  const int64_t gtotal = int64_t(npairs_blk) * kMB * kMB;
  const int64_t idx = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const bool bad = *p.err != 0u;
  const int wexp = weight_exponent(p.wmax);
  const double up1 = ldexp(1.0, wexp), upw = ldexp(1.0, wexp * p.power);   // undo the weight normalisation
  if (idx < gtotal) {
    if (!want_gram) return;
    int pidx = int(idx / (kMB * kMB));
    const int i = int((idx / kMB) % kMB), j = int(idx % kMB);     // G block (a, b), a <= b, element (i, j)
    int a = 0;
    while (pidx >= nb - a) {
      pidx -= nb - a;
      ++a;
    }
    const int b = a + pidx;
    const int fi = a * kMB + i, fj = b * kMB + j;
    if (fi >= d || fj >= d) return;
    if (a == b && i > j) return;
    const int pa = a >> 1, r = a & 1, pb = b >> 1, h = b & 1;
    const int type = (pp.nbp == 1) ? 0 : (pa == 0 ? pb : 2);
    double s = 0.0;
    for (int sl = pp.first[type]; sl < pp.first[type + 1]; ++sl)
      s += p.gpart64[((size_t(sl) * 2 + r) * 2 + h) * (kMB * kMB) + size_t(i) * kMB + j];
    s *= upw;
    if (bad) s = nan("");
    double* G = out + 2 + 2 * d;
    G[size_t(fi) * d + fj] = s;
    G[size_t(fj) * d + fi] = s;
    return;
  }
  const int64_t k = idx - gtotal;
  if (k < 2) {          // S0, Swy: block partials of the coefficient kernel, in block order
    double s = 0.0;
    for (int b = 0; b < pp.coef_blocks; ++b) s += pp.s0blocks[size_t(b) * 2 + k];
    out[k] = bad ? nan("") : ((k == 1 && !has_y) ? 0.0 : s);
    return;
  }
  const int64_t f2 = k - 2;
  if (f2 < 2 * int64_t(d)) {
    const int which = int(f2 / d), f = int(f2 % d);
    const int blk = f / kMB, fin = f % kMB;
    const int type = (pp.nbp == 1) ? 0 : ((blk >> 1) == 0 ? 0 : 2);     // the diagonal pair of the block
    const int r = blk & 1;
    double s = 0.0;
    if (which == 0 || has_y)
      for (int sl = pp.first[type]; sl < pp.first[type + 1]; ++sl)
        for (int t = 0; t < kWorkers; ++t) s += p.spart[(((size_t(sl) * 2 + r) * kWorkers + t) * 2 + which) * 128 + fin];
    out[2 + which * d + f] = bad ? nan("") : s * (which == 0 ? up1 : upw);
  }
}

// The partials and row coefficients of a pair grid, in scratch order behind the header.
struct PairLayout {
  size_t gbytes, sbytes, s0bytes, cbytes;
  int ncoef;
  size_t total() const { return gbytes + sbytes + s0bytes + cbytes * size_t(ncoef); }
};
PairLayout pair_layout(int grid, int64_t npad, int coef_blocks, int power, bool has_y) {
  PairLayout l;
  l.gbytes = size_t(grid) * 2 * kMB * kMB * sizeof(double);
  l.sbytes = size_t(grid) * kWorkers * 2 * 128 * sizeof(double);
  l.s0bytes = (size_t(coef_blocks) * 2 * sizeof(double) + 255) / 256 * 256;
  l.cbytes = (size_t(npad) * 4 + 255) / 256 * 256;
  l.ncoef = 1 + (power == 1 ? 1 : 0) + (has_y ? 1 : 0);
  return l;
}

}  // namespace

// Host-side queries only: which kernel, how many pairs of each type, how much scratch.  The caller guarantees
// d = 129..512.  first[ntypes] == 0 when the device cannot co-schedule one pair per type.
int rlvi_tf32_pair_plan(rlvi_ctx* ctx, int64_t n, int d, int power, bool has_y, int precision, PairPlan* plan) {
  memset(plan, 0, sizeof(*plan));
  const int nb = (d + kMB - 1) / kMB;
  const int nbp = (nb + 1) / 2;                         // d = 257..384: the fourth block is zero-filled by the TMA
  plan->ntypes = (nbp == 1) ? 1 : 3;

  // RLVI_TF32X3 = the ~1e-6 mode: TF32 hi.hi + the two correction products.  By default the corrections run as BF16
  // (NSPLIT = 2: a third less tensor time); RLVI_TF32_PURE3=1 keeps all three passes in TF32 (NSPLIT = 3).
  const char* pure_env = getenv("RLVI_TF32_PURE3");      // read per call: tests switch it
  plan->nsplit = (precision == RLVI_TF32X1) ? 1 : ((pure_env && atoi(pure_env) != 0) ? 3 : 2);
  const int variant = (plan->nsplit == 1 ? 0 : (plan->nsplit == 3 ? 2 : 4)) + (has_y ? 1 : 0);
  const void* fns[6] = {(const void*)gram_tf32_pair_kernel<1, false>, (const void*)gram_tf32_pair_kernel<1, true>,
                        (const void*)gram_tf32_pair_kernel<3, false>, (const void*)gram_tf32_pair_kernel<3, true>,
                        (const void*)gram_tf32_pair_kernel<2, false>, (const void*)gram_tf32_pair_kernel<2, true>};
  const void* fn = fns[variant];
  // once per (device, kernel): the shared-memory opt-in and how many pairs can be resident at once (one CTA per SM,
  // the two SMs of a TPC per pair) -- both are host-side driver calls of ~1 ms
  static int cached_pairs[64][6];
  const int dev_slot = (ctx->device >= 0 && ctx->device < 64) ? ctx->device : 0;
  int max_pairs = cached_pairs[dev_slot][variant];
  if (max_pairs == 0) {
    RLVI_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemTotal));
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(unsigned(ctx->sm_count / 2 * 2), 1, 1);
    cfg.blockDim = dim3(kThreads, 1, 1);
    cfg.dynamicSmemBytes = kSmemTotal;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = 2;
    attr.val.clusterDim.y = 1;
    attr.val.clusterDim.z = 1;
    cfg.attrs = &attr;
    cfg.numAttrs = 1;
    // pairs are independent of each other: a wrong answer here costs speed (a second wave), never correctness
    if (cudaOccupancyMaxActiveClusters(&max_pairs, fn, &cfg) != cudaSuccess || max_pairs < 1) {
      cudaGetLastError();
      max_pairs = ctx->sm_count / 2;
    }
    cached_pairs[dev_slot][variant] = max_pairs;
  }
  if (max_pairs > ctx->sm_count / 2) max_pairs = ctx->sm_count / 2;
  if (getenv("RLVI_TF32_STATS")) fprintf(stderr, "[tf32 pair] resident pairs: %d\n", max_pairs);
  if (max_pairs < plan->ntypes) return RLVI_OK;
  const int64_t ntiles = (n + kR - 1) / kR;

  // pairs per type: in proportion to the per-tile cost (off-diagonal pairs load and transform two blocks per tile)
  int count[kPairTypes] = {0, 0, 0};
  if (plan->ntypes == 1) {
    count[0] = int(ntiles < max_pairs ? ntiles : max_pairs);
  } else {
    // measured per-tile cost (profiles/r02_tf32_pair_stats.txt): the tensor pipe bounds both kinds of pair alike
    // ... except in the mixed mode, where the stages of an off-diagonal pair are twice as large and half as many, and the
    // pair is bound by the round trip of a stage instead (986 vs 738 clk per tile): 28.2 -> 26.9 ms at config 3 with 1.25
    const double wdiag = 1.0, woff = (plan->nsplit == 2) ? 1.25 : 1.0;
    int total = max_pairs;
    if (ntiles * 3 < total) total = int(ntiles) * 3;
    int off = int(double(total) * woff / (2.0 * wdiag + woff) + 0.5);
    if (off < 1) off = 1;
    int dg = (total - off) / 2;
    if (dg < 1) dg = 1;
    off = total - 2 * dg;                               // >= 1: total >= 3
    count[0] = dg;
    count[1] = off;
    count[2] = dg;
  }
  for (int t = 0; t < plan->ntypes; ++t) plan->first[t + 1] = plan->first[t] + count[t];
  for (int t = plan->ntypes; t < kPairTypes; ++t) plan->first[t + 1] = plan->first[plan->ntypes];
  const int64_t npad = ntiles * kR;
  plan->coef_blocks = int((npad + kCoefThreads * 4 - 1) / (kCoefThreads * 4));
  if (plan->coef_blocks > ctx->sm_count * 8) plan->coef_blocks = ctx->sm_count * 8;
  plan->part_bytes = pair_layout(2 * plan->first[plan->ntypes], npad, plan->coef_blocks, power, has_y).total();
  return RLVI_OK;
}

int rlvi_tf32_pair_moments(rlvi_ctx* ctx, const CUtensorMap& tmap, const CUtensorMap& tmap3, const Tf32Params& p,
                           const PairPlan& plan, char* part, int want_gram, double* out, cudaStream_t st) {
  PairParams pp;
  memset(&pp, 0, sizeof(pp));
  pp.b = p;
  pp.nbp = (plan.ntypes == 1) ? 1 : 2;
  pp.ntypes = plan.ntypes;
  for (int t = 0; t <= kPairTypes; ++t) pp.first[t] = plan.first[t];
  const int grid = 2 * plan.first[plan.ntypes];
  const int64_t ntiles = (p.n + kR - 1) / kR;
  const int64_t npad = ntiles * kR;
  const PairLayout l = pair_layout(grid, npad, plan.coef_blocks, p.power, p.y != nullptr);
  pp.b.gpart64 = reinterpret_cast<double*>(part);
  pp.b.spart = reinterpret_cast<double*>(part + l.gbytes);
  pp.s0blocks = reinterpret_cast<double*>(part + l.gbytes + l.sbytes);
  pp.coef_blocks = plan.coef_blocks;
  {
    float* c0 = reinterpret_cast<float*>(part + l.gbytes + l.sbytes + l.s0bytes);
    float* c1 = (p.power == 1) ? reinterpret_cast<float*>(reinterpret_cast<char*>(c0) + l.cbytes) : c0;
    float* c2 = p.y ? reinterpret_cast<float*>(reinterpret_cast<char*>(c0) + l.cbytes * size_t(l.ncoef - 1)) : nullptr;
    pp.coef_sc = c0;
    pp.coef_c1 = c1;
    pp.coef_cy = c2;
    pair_coef_kernel<<<plan.coef_blocks, kCoefThreads, 0, st>>>(p.w, p.y, p.n, npad, p.power, p.wmax, c0, c1, c2, pp.s0blocks);
    RLVI_LAUNCH_CHECK(ctx);
  }
  const size_t stats_bytes = size_t(grid) * 8 * sizeof(long long);
  if (getenv("RLVI_TF32_STATS")) {
    RLVI_CUDA(cudaMalloc(&pp.stats, stats_bytes));
    RLVI_CUDA(cudaMemset(pp.stats, 0, stats_bytes));
  }

  switch ((plan.nsplit == 1 ? 0 : (plan.nsplit == 3 ? 2 : 4)) + (p.y ? 1 : 0)) {
    case 0: gram_tf32_pair_kernel<1, false><<<grid, kThreads, kSmemTotal, st>>>(tmap, tmap3, pp); break;
    case 1: gram_tf32_pair_kernel<1, true><<<grid, kThreads, kSmemTotal, st>>>(tmap, tmap3, pp); break;
    case 2: gram_tf32_pair_kernel<3, false><<<grid, kThreads, kSmemTotal, st>>>(tmap, tmap3, pp); break;
    case 3: gram_tf32_pair_kernel<3, true><<<grid, kThreads, kSmemTotal, st>>>(tmap, tmap3, pp); break;
    case 4: gram_tf32_pair_kernel<2, false><<<grid, kThreads, kSmemTotal, st>>>(tmap, tmap3, pp); break;
    default: gram_tf32_pair_kernel<2, true><<<grid, kThreads, kSmemTotal, st>>>(tmap, tmap3, pp); break;
  }
  RLVI_LAUNCH_CHECK(ctx);
  if (pp.stats) {    // bring-up only: synchronise and print the per-role cycle counters (mean over the CTAs of a type)
    RLVI_CUDA(cudaStreamSynchronize(st));
    long long* hst = static_cast<long long*>(malloc(stats_bytes));
    cudaMemcpy(hst, pp.stats, stats_bytes, cudaMemcpyDeviceToHost);
    const char* names[8] = {"producer wait empty", "worker0 wait full (x6)", "worker0 busy (x6)", "mma wait ready", "mma wait tempty",
                            "mma issue", "acc warp drain (x8)", "producer total"};
    for (int t = 0; t < pp.ntypes; ++t) {
      const int cnt = pp.first[t + 1] - pp.first[t];
      const double tiles = double(ntiles) / cnt;
      for (int r = 0; r < 2; ++r) {
        double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        for (int sl = pp.first[t]; sl < pp.first[t + 1]; ++sl)
          for (int k = 0; k < 8; ++k) acc[k] += double(hst[(size_t(sl) * 2 + r) * 8 + k]) / cnt;
        fprintf(stderr, "[tf32 pair stats] type %d cta %d (%d pairs, %.0f tiles/CTA), cycles per tile:", t, r, cnt, tiles);
        for (int k = 0; k < 8; ++k) fprintf(stderr, " %s=%.0f", names[k], acc[k] / tiles);
        fprintf(stderr, "\n");
      }
    }
    free(hst);
    cudaFree(pp.stats);
    pp.stats = nullptr;
  }
  const int nb = 2 * pp.nbp;
  const int64_t total = int64_t(nb) * (nb + 1) / 2 * kMB * kMB + 2 + 2 * int64_t(p.d);
  gram_tf32_pair_finalize_kernel<<<int((total + 255) / 256), 256, 0, st>>>(pp, p.y ? 1 : 0, want_gram, out);
  RLVI_LAUNCH_CHECK(ctx);
  return RLVI_OK;
}
