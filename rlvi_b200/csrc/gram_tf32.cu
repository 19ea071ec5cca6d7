// gram_tf32.cu -- pi-weighted M-step statistics of FP32-STORED samples on the 5th-generation tensor cores
// (tcgen05.mma kind::tf32, accumulators in TMEM): the FP32 mode of SURVEY.md section 8(d), config C3
// (robust PCA, N = 2^24, d = 512).  Replaces, for float32 X, the contractions of
//   standard-learning/utils.py:82-84   PCA of the rows pi_i x_i      (power = 2:  G = sum pi_i^2 x_i x_i^T)
//   standard-learning/rlvi.py:70-71    sqrt(pi)-scaled least squares (power = 1:  G = sum pi_i x_i x_i^T)
//   standard-learning/utils.py:36-38,103-105                         (power = 1)
//
// Routes.  rlvi_weighted_moments_f32 (at the end of this file) picks exactly one per call, before anything is queued:
//   d > 512, d % 4 != 0, unaligned X, n >= 2^31 - 16, no tensor-map entry point: X is converted to FP64 chunk by chunk
//               and handed to rlvi_weighted_moments_f64;
//   d = 129..512  CTA pairs, cta_group::2 (gram_tf32_pair.cu);
//   d <= 128      the single-CTA kernel below.
//
// Formulation.  With s_i = pi_i (power 2) or sqrt(pi_i) (power 1) and z_i = s_i x_i -- the very rows the reference
// forms -- G = Z^T Z.  For d <= 128 the features are ONE 128-feature block (zero-filled past d by the TMA), so G is one
// M = 128, N = 128 product whose A and B are the same shared-memory block.  CTA c (persistent, one per SM) takes the
// row tiles c, c + nslots, c + 2 nslots, ... (16 rows each).
//
// Per CTA, warp-specialised (16 warps = 4 warpgroups with their own register budgets, setmaxnreg 40/88/192/88):
//   warp 0      TMA producer: per tile ONE cp.async.bulk.tensor.3d box (32 floats x 16 rows x 4 column groups; four 2-D
//               boxes when d % 32 != 0), CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B -> exactly the one canonical MN-major
//               layout tcgen05 accepts for 32-bit operands, SWIZZLE_128B_BASE32B (Swizzle<2,5,2>: atoms of 128 B x 4
//               rows, the 32-byte unit index XORed with row mod 4), LBO = 2048 B (next 32 features), SBO = 512 B (next
//               4 rows).  The plain SWIZZLE_128B / no-swizzle MN-major layouts silently give zeros for kind::tf32
//               (tools/tf32_debug.cu, profiles/r02_tf32_descriptor_probe.txt);
//   warps 4-15  three transform TEAMS of four warps; team t takes the CTA's tiles t, t + 3, ... (CUDA cores, in
//               place on the landed tile): z = s_i x rounded to TF32 (round-to-nearest on the bit pattern) = Z_hi,
//               and for the 3xTF32 mode the remainder Z_lo = tf32(z - Z_hi) into a second buffer; the column
//               sums S1 = X^T pi, Sy = X^T (w y), S0, sum w y ride along; fence.proxy.async, mbarrier arrive;
//   warp 1      MMA issuer (one thread): D += Z_hi^T Z_hi (+ Z_lo^T Z_hi + Z_hi^T Z_lo), K = 8 per instruction, both
//               operands MN-major straight from shared memory; tcgen05.commit frees the stage / publishes the chunk;
//   warps 8-11  (team 1) are also the accumulator: the tensor core adds in FP32 (round-toward-zero inside the
//               datapath), so a TMEM accumulator only lives for 8 tiles (128 rows); it is then read back (tcgen05.ld
//               32x32b) and added, round-to-nearest, into 128 FP32 registers per thread, which are themselves flushed
//               into this CTA's FP64 partial in global memory every `chunks_per_flush` chunks.  Two TMEM buffers
//               (2 x 128 columns) alternate so the read-back overlaps the next chunk's MMAs; team 1 drains chunk c - 2
//               just before it transforms its first tile of chunk c (complete by then).
// A finalize kernel adds the per-CTA partials in slot order (deterministic) and mirrors the upper triangle.
// The weights are normalised by a power of two (max pi <= 2^e) so that the collapse regime (pi ~ 1e-7 .. 1e-20,
// SURVEY.md H1) stays inside the FP32 range; the statistics are scaled back exactly.
//
// Accuracy: 3xTF32 keeps ~2^-21 per product, the three-level accumulation keeps the sums at FP32 level over
// any N -> entry by entry, |G - G_ref| <= 1e-5 B with B = |X|^T diag(w) |X| against FP64 on the same float32 samples
// (measured <= 7e-7 B here, <= 2.8e-6 B on the CTA pairs, on inputs whose TF32 remainders all have one sign; B200,
// 1000 W), for scaled samples 2^-60 <= |z| < 2^56 (or 0): below, the products leave the FP32 normal range and lose their
// corrections first; from 2^56 on, a 32 Ki-row register sum of z^2 can overflow.  tests/test_gpu_fp32_mode.py checks
// both ends.  Single-pass TF32 (precision = RLVI_TF32X1) rounds operands to 11 bits: ~1e-3/sqrt(rows) on zero-mean
// remainders, up to ~5e-4 B when they share a sign.
#include "tf32.cuh"

namespace {

using namespace tf32;

constexpr int kTeams = 3;
constexpr int kStages = 8;                   // 8 KiB (TF32X1) or 16 KiB (3xTF32: Z_hi + Z_lo) each
static_assert(kStages * 2 * kBlkBytes <= kSmemBudget, "stages exceed the shared-memory budget");

struct CtaParams {
  Tf32Params b;           // gpart64: [grid][128][128]; spart: [grid][kTeams][2][128] (S1, Sy)
  int nslots;             // = grid
  double* s0part;         // [grid][kTeams][2]   S0, Swy
};

// One transform team (four warps): tiles team, team + 3, ... of the CTA.  The IS_ACC team (1) also owns the level-2
// accumulator.  A separate instantiation per register budget (setmaxnreg 88 / 192).
struct TeamCtx {
  unsigned char* smem;
  uint64_t *full_bar, *ready_bar, *empty_bar, *tfull_bar, *tempty_bar;
  float* red_all;
  double* dred_all;
  uint32_t tmem_base;
  int slot, team;
  int my_tiles, my_chunks;
};

template <int NSPLIT, bool HAS_Y, bool IS_ACC>
__device__ __forceinline__ void team_body(const CtaParams& cp, const TeamCtx& cx) {
  const Tf32Params& p = cp.b;
  constexpr int kStageBytes = kBlkBytes * (NSPLIT == 3 ? 2 : 1);
  unsigned char* smem = cx.smem;
  uint64_t *full_bar = cx.full_bar, *ready_bar = cx.ready_bar, *tfull_bar = cx.tfull_bar, *tempty_bar = cx.tempty_bar;
  uint64_t* empty_bar = cx.empty_bar;
  const uint32_t tmem_base = cx.tmem_base;
  const int slot = cx.slot, team = cx.team;
  const int my_tiles = cx.my_tiles, my_chunks = cx.my_chunks;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tt = threadIdx.x & 127;                      // thread of the team
  const int q = tt & 7, rr = tt >> 3;                    // logical 16-byte unit, row of the tile
  // SWIZZLE_128B_ATOM_32B: the 32-byte unit q >> 1 of row rr sits at unit (q >> 1) ^ (rr & 3)
  const uint32_t off = uint32_t(rr * 128 + (((((q >> 1) ^ (rr & 3)) << 1) | (q & 1)) << 4));
  const bool own_s0 = (q == 0);
  float* red = cx.red_all + team * 1024;
  double* dred = cx.dred_all + team * 32;
  const int bar_id = 1 + team;
  float s1acc[4][4], syacc[4][4];
#pragma unroll
  for (int c = 0; c < 4; ++c)
#pragma unroll
    for (int k = 0; k < 4; ++k) s1acc[c][k] = syacc[c][k] = 0.f;
  double s1d = 0.0, syd = 0.0, s0 = 0.0, swy = 0.0;
  const double wscale = ldexp(1.0, -weight_exponent(p.wmax));      // exact power of two

  // ---- accumulator state (team 1 only; thread = TMEM lane quarter * 32 + lane) ----
  const int quarter = warp & 3;                          // hardware: a warp reaches TMEM lanes 32 (warp id % 4) ..
  float acc[128];
#pragma unroll
  for (int i = 0; i < 128; ++i) acc[i] = 0.f;
  double* gp = p.gpart64 + (size_t(blockIdx.x) * 128 + size_t(quarter * 32 + lane)) * 128;
  bool flushed = false;
  int next_drain = 0;
  bool ok = true;

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
  auto drain = [&](int ch) -> bool {
    const int buf = ch & 1;
    if (!wait_or_abort(&tfull_bar[buf], uint32_t(ch >> 1) & 1u, p.err)) return false;
    tc_fence_after();
    const uint32_t taddr = tmem_base + (uint32_t(quarter * 32) << 16) + uint32_t(buf * kMB);
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      float v[16];
      tc_ld16(taddr + uint32_t(c * 16), v);
#pragma unroll
      for (int j = 0; j < 16; ++j) acc[c * 16 + j] += v[j];
    }
    tc_fence_before();
    mbar_arrive(&tempty_bar[buf]);
    if (((ch + 1) % p.chunks_per_flush) == 0) flush_acc();
    return true;
  };

  auto flush_sums = [&]() {
    const int wq = tt >> 5;
#pragma unroll
    for (int c = 0; c < 4; ++c)
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        float v = s1acc[c][k];
        v += __shfl_xor_sync(0xffffffffu, v, 8);
        v += __shfl_xor_sync(0xffffffffu, v, 16);
        if (lane < 8) red[(wq * 2 + 0) * 128 + c * 32 + lane * 4 + k] = v;
        s1acc[c][k] = 0.f;
        if (HAS_Y) {
          float u = syacc[c][k];
          u += __shfl_xor_sync(0xffffffffu, u, 8);
          u += __shfl_xor_sync(0xffffffffu, u, 16);
          if (lane < 8) red[(wq * 2 + 1) * 128 + c * 32 + lane * 4 + k] = u;
          syacc[c][k] = 0.f;
        }
      }
    asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
    s1d += double((red[0 * 128 + tt] + red[2 * 128 + tt]) + (red[4 * 128 + tt] + red[6 * 128 + tt]));
    if (HAS_Y) syd += double((red[1 * 128 + tt] + red[3 * 128 + tt]) + (red[5 * 128 + tt] + red[7 * 128 + tt]));
    asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
  };

  auto load_row = [&](int it, double& pid, double& yd) {
    const int64_t row = (int64_t(slot) + int64_t(it) * cp.nslots) * kR + rr;
    pid = (it < my_tiles && row < p.n) ? p.w[row] : 0.0;
    yd = (HAS_Y && it < my_tiles && row < p.n) ? p.y[row] : 0.0;
  };

  double pid, yd;
  load_row(team, pid, yd);
  int done = 0;
  int s = team;                                          // team < kStages
  uint32_t ph = 0;
  for (int it = team; it < my_tiles; it += kTeams) {
    double pid_n, yd_n;
    load_row(it + kTeams, pid_n, yd_n);                  // prefetch the row coefficients of the team's next tile
    if constexpr (IS_ACC) {                              // chunk c - 2 is complete by now: drain it before chunk c
      const int ch = it / kTpc;
      while (ok && next_drain + 2 <= ch) ok = drain(next_drain++);
      if (!ok) break;
    }
    const double wd = (p.power == 2) ? pid * pid : pid;
    const double pis = pid * wscale;                       // normalised weight, <= 1
    const float sc = (p.power == 2) ? float(pis) : float(sqrt(pis));
    const float c1 = float(pis);
    const float cy = HAS_Y ? float(((p.power == 2) ? pis * pis : pis) * yd) : 0.f;
    if (own_s0) {
      s0 += wd;
      if (HAS_Y) swy = fma(wd, yd, swy);
    }
    // Tiles land out of order and the stage's previous tile belonged to another team: `full` could still be one
    // phase behind, which try_wait.parity cannot tell from "complete".  The MMA's release of the previous use
    // (`empty`, one phase back) implies that phase of `full` is over, so wait for that first.
    ok = wait_or_abort(&empty_bar[s], ph ^ 1u, p.err) && wait_or_abort(&full_bar[s], ph, p.err);
    if (!ok) break;
    unsigned char* sb = smem + size_t(s) * kStageBytes;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      float4* ptr = reinterpret_cast<float4*>(sb + c * kChunkBytes + off);
      const float4 x = *ptr;
      s1acc[c][0] = fmaf(c1, x.x, s1acc[c][0]);
      s1acc[c][1] = fmaf(c1, x.y, s1acc[c][1]);
      s1acc[c][2] = fmaf(c1, x.z, s1acc[c][2]);
      s1acc[c][3] = fmaf(c1, x.w, s1acc[c][3]);
      if (HAS_Y) {
        syacc[c][0] = fmaf(cy, x.x, syacc[c][0]);
        syacc[c][1] = fmaf(cy, x.y, syacc[c][1]);
        syacc[c][2] = fmaf(cy, x.z, syacc[c][2]);
        syacc[c][3] = fmaf(cy, x.w, syacc[c][3]);
      }
      const float z0 = sc * x.x, z1 = sc * x.y, z2 = sc * x.z, z3 = sc * x.w;
      const uint32_t h0 = to_tf32(z0), h1 = to_tf32(z1), h2 = to_tf32(z2), h3 = to_tf32(z3);
      *reinterpret_cast<uint4*>(ptr) = make_uint4(h0, h1, h2, h3);
      if (NSPLIT == 3) {                                   // Z_lo: the block behind Z_hi in the stage
        const uint32_t l0 = to_tf32(z0 - __uint_as_float(h0)), l1 = to_tf32(z1 - __uint_as_float(h1)),
                       l2 = to_tf32(z2 - __uint_as_float(h2)), l3 = to_tf32(z3 - __uint_as_float(h3));
        *reinterpret_cast<uint4*>(reinterpret_cast<unsigned char*>(ptr) + kBlkBytes) = make_uint4(l0, l1, l2, l3);
      }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic writes -> visible to the tensor core
    mbar_arrive(&ready_bar[s]);
    if ((++done % kFlushTiles) == 0) flush_sums();
    pid = pid_n;
    yd = yd_n;
    s += kTeams;                                           // kStages > kTeams: at most one wrap
    if (s >= kStages) {
      s -= kStages;
      ph ^= 1u;
    }
  }
  if (ok) {
    flush_sums();
    p.spart[((size_t(blockIdx.x) * kTeams + team) * 2 + 0) * 128 + tt] = s1d;
    p.spart[((size_t(blockIdx.x) * kTeams + team) * 2 + 1) * 128 + tt] = syd;
    if (q == 0) {
      dred[rr * 2 + 0] = s0;
      dred[rr * 2 + 1] = swy;
    }
    asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
    if (tt == 0) {
      double a = 0.0, b = 0.0;
      for (int r = 0; r < kR; ++r) {
        a += dred[r * 2 + 0];
        b += dred[r * 2 + 1];
      }
      cp.s0part[(size_t(blockIdx.x) * kTeams + team) * 2 + 0] = a;
      cp.s0part[(size_t(blockIdx.x) * kTeams + team) * 2 + 1] = b;
    }
    if constexpr (IS_ACC) {
      while (ok && next_drain < my_chunks) ok = drain(next_drain++);
      if (ok) flush_acc();
    }
  }
}

template <int NSPLIT, bool HAS_Y>
__global__ void __launch_bounds__(kThreads, 1)
    gram_tf32_kernel(const __grid_constant__ CUtensorMap tmap2, const __grid_constant__ CUtensorMap tmap3, const CtaParams cp) {
  const Tf32Params& p = cp.b;
  constexpr int kStageBytes = kBlkBytes * (NSPLIT == 3 ? 2 : 1);
  extern __shared__ unsigned char smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  unsigned char* smem = smem_raw + ((1024u - (raw & 1023u)) & 1023u);
  const uint32_t smem_base = smem_u32(smem);
  unsigned char* tail = smem + kSmemBudget;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(tail);          // [kStages] TMA -> transform
  uint64_t* ready_bar = full_bar + kStages;                         // [kStages] transform -> MMA
  uint64_t* empty_bar = ready_bar + kStages;                        // [kStages] MMA -> TMA
  uint64_t* tfull_bar = empty_bar + kStages;                        // [2] MMA -> accumulator team
  uint64_t* tempty_bar = tfull_bar + 2;                             // [2] accumulator team -> MMA
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
  float* red_all = reinterpret_cast<float*>(tail + 512);            // [kTeams][4 warps][2][128] column-sum exchange
  double* dred_all = reinterpret_cast<double*>(tail + 512 + kTeams * 4096);   // [kTeams][16][2] S0 / Swy exchange

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int slot = blockIdx.x;
  const int ntiles = int((p.n + kR - 1) / kR);
  const int my_tiles = (ntiles > slot) ? (ntiles - slot + cp.nslots - 1) / cp.nslots : 0;
  const int my_chunks = (my_tiles + kTpc - 1) / kTpc;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&ready_bar[s], 128);
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tfull_bar[b], 1);
      mbar_init(&tempty_bar[b], 128);   // team 1
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {   // TMEM: two 128-column accumulator buffers
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(2 * kMB)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);

  if (warp < 4) {
    // ===== warpgroup 0: TMA producer (warp 0) and MMA issuer (warp 1) ==========================================
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    if (warp == 0 && lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int it = 0; it < my_tiles; ++it) {
        if (!wait_or_abort(&empty_bar[s], ph ^ 1u, p.err)) break;
        const int row0 = (slot + it * cp.nslots) * kR;
        const uint32_t sb = smem_base + uint32_t(s) * uint32_t(kStageBytes);
        mbar_arrive_expect_tx(&full_bar[s], uint32_t(kBlkBytes));
        if (p.box3d) {       // one box: 32 floats x 16 rows x 4 column groups
          tma_load_3d_f32(sb, &tmap3, 0, row0, 0, &full_bar[s]);
        } else {
#pragma unroll
          for (int c = 0; c < 4; ++c) tma_load_2d_f32(sb + uint32_t(c * kChunkBytes), &tmap2, c * 32, row0, &full_bar[s]);
        }
        if (++s == kStages) {
          s = 0;
          ph ^= 1u;
        }
      }
    } else if (warp == 1 && lane == 0) {
      const uint32_t idesc = umma_idesc(kMB);
      // descriptor = constant | (address >> 4): only the low 14 bits change
      const uint64_t dconst = umma_desc(0);
      auto desc = [&](uint32_t addr) { return dconst | uint64_t((addr & 0x3FFFFu) >> 4); };
      int s = 0;
      uint32_t ph = 0;
      bool ok = true;
      for (int it = 0; it < my_tiles && ok; ++it) {
        const int ch = it / kTpc;
        const int tin = it - ch * kTpc;
        const int buf = ch & 1;
        if (tin == 0) {
          ok = wait_or_abort(&tempty_bar[buf], (uint32_t(ch >> 1) & 1u) ^ 1u, p.err);
          if (!ok) break;
          tc_fence_after();
        }
        ok = wait_or_abort(&ready_bar[s], ph, p.err);
        if (!ok) break;
        tc_fence_after();
        const uint32_t sb = smem_base + uint32_t(s) * uint32_t(kStageBytes);
        const uint32_t dcol = tmem_base + uint32_t(buf * kMB);
#pragma unroll
        for (int ks = 0; ks < kR / 8; ++ks) {
          const uint32_t first = (tin == 0 && ks == 0) ? 0u : 1u;
          const uint32_t kb = sb + uint32_t(ks * 1024);
          const uint64_t hi = desc(kb);
          tc_mma_tf32(dcol, hi, hi, idesc, first);
          if (NSPLIT == 3) {
            const uint64_t lo = desc(kb + kBlkBytes);
            tc_mma_tf32(dcol, lo, hi, idesc, 1u);
            tc_mma_tf32(dcol, hi, lo, idesc, 1u);
          }
        }
        tc_commit(&empty_bar[s]);                                        // stage free once these MMAs have read it
        if (tin == kTpc - 1 || it == my_tiles - 1) tc_commit(&tfull_bar[buf]);   // chunk complete in TMEM
        if (++s == kStages) {
          s = 0;
          ph ^= 1u;
        }
      }
    }
  } else {
    // ===== warpgroups 1-3: the transform teams; team 1 also holds the level-2 accumulator =========================
    TeamCtx cx;
    cx.smem = smem;
    cx.full_bar = full_bar;
    cx.ready_bar = ready_bar;
    cx.empty_bar = empty_bar;
    cx.tfull_bar = tfull_bar;
    cx.tempty_bar = tempty_bar;
    cx.red_all = red_all;
    cx.dred_all = dred_all;
    cx.tmem_base = tmem_base;
    cx.slot = slot;
    cx.team = (warp >> 2) - 1;
    cx.my_tiles = my_tiles;
    cx.my_chunks = my_chunks;
    if (cx.team == 1) {
      asm volatile("setmaxnreg.inc.sync.aligned.u32 192;");
      team_body<NSPLIT, HAS_Y, true>(cp, cx);
    } else {
      asm volatile("setmaxnreg.dec.sync.aligned.u32 88;");
      team_body<NSPLIT, HAS_Y, false>(cp, cx);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(2 * kMB) : "memory");
  }
}

// Sum the per-CTA partials in slot order, mirror the upper triangle, write [S0, Swy, S1, Sy, G] (FP64).
__global__ void __launch_bounds__(256) gram_tf32_finalize_kernel(const CtaParams cp, int has_y, int want_gram, double* out) {
  const Tf32Params& p = cp.b;
  const int d = p.d;
  const int64_t gtotal = int64_t(kMB) * kMB;
  const int64_t idx = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const bool bad = *p.err != 0u;
  const int wexp = weight_exponent(p.wmax);
  const double up1 = ldexp(1.0, wexp), upw = ldexp(1.0, wexp * p.power);   // undo the weight normalisation
  if (idx < gtotal) {
    if (!want_gram) return;
    const int i = int(idx / kMB), j = int(idx % kMB);
    if (j >= d || i > j) return;                                   // upper triangle, i <= j < d
    double s = 0.0;
    for (int sl = 0; sl < cp.nslots; ++sl) s += p.gpart64[size_t(sl) * (kMB * kMB) + size_t(i) * kMB + j];
    s *= upw;
    if (bad) s = nan("");
    double* G = out + 2 + 2 * d;
    G[size_t(i) * d + j] = s;
    G[size_t(j) * d + i] = s;
    return;
  }
  const int64_t k = idx - gtotal;
  if (k < 2) {          // S0, Swy
    double s = 0.0;
    for (int sl = 0; sl < cp.nslots; ++sl)
      for (int t = 0; t < kTeams; ++t) s += cp.s0part[(size_t(sl) * kTeams + t) * 2 + k];
    out[k] = bad ? nan("") : ((k == 1 && !has_y) ? 0.0 : s);
    return;
  }
  const int64_t f2 = k - 2;
  if (f2 < 2 * int64_t(d)) {
    const int which = int(f2 / d), f = int(f2 % d);
    double s = 0.0;
    if (which == 0 || has_y)
      for (int sl = 0; sl < cp.nslots; ++sl)
        for (int t = 0; t < kTeams; ++t) s += p.spart[((size_t(sl) * kTeams + t) * 2 + which) * 128 + f];
    out[2 + which * d + f] = bad ? nan("") : s * (which == 0 ? up1 : upw);
  }
}

__global__ void __launch_bounds__(256) wmax_kernel(const double* __restrict__ w, int64_t n, unsigned long long* out) {
  double m = 0.0;
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x)
    m = fmax(m, w[i]);                   // weights are >= 0; fmax drops NaN
  m = warp_max(m);
  if ((threadIdx.x & 31) == 0 && m > 0.0) atomicMax(out, (unsigned long long)__double_as_longlong(m));
}

__global__ void __launch_bounds__(256) f32_to_f64_kernel(const float* __restrict__ src, double* __restrict__ dst, int64_t count) {
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < count; i += int64_t(gridDim.x) * blockDim.x)
    dst[i] = double(src[i]);
}
__global__ void __launch_bounds__(256) add_f64_kernel(double* __restrict__ dst, const double* __restrict__ src, int count, int first) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) dst[i] = first ? src[i] : dst[i] + src[i];
}

}  // namespace

// Shapes the tensor path does not cover: convert row chunks to FP64 and reuse the FP64 statistics kernels.
static int moments_f32_via_f64(rlvi_ctx* ctx, const float* X, const double* y, const double* weights, int64_t n, int d,
                               int power, int want_gram, double* out, cudaStream_t st) {
  const int nm = rlvi_moments_out_doubles(d);
  const int nsum = want_gram ? nm : 2 + 2 * d;             // want_gram == 0 leaves G in `out` untouched

  int64_t chunk = (int64_t(64) << 20) / (int64_t(d) * 8);   // 64 MiB of converted rows at a time
  if (chunk < 64) chunk = 64;
  if (chunk > n) chunk = n;
  const size_t need = size_t(chunk) * d * 8 + size_t(nm) * 8 + 256;
  if (need > ctx->big_bytes) {
    RLVI_CUDA(cudaDeviceSynchronize());
    if (ctx->big) cudaFree(ctx->big);
    ctx->big = nullptr;
    ctx->big_bytes = 0;
    if (cudaMalloc(&ctx->big, need) != cudaSuccess) {
      rlvi_set_error("cudaMalloc of %zu bytes for the FP32 -> FP64 staging buffer failed", need);
      return RLVI_ERR_NOMEM;
    }
    ctx->big_bytes = need;
  }
  double* xd = static_cast<double*>(ctx->big);
  double* tmp = xd + size_t(chunk) * d;
  bool first = true;
  for (int64_t r0 = 0; r0 < n; r0 += chunk) {
    const int64_t rows = (n - r0 < chunk) ? (n - r0) : chunk;
    f32_to_f64_kernel<<<ctx->sm_count * 4, 256, 0, st>>>(X + r0 * d, xd, rows * d);
    RLVI_LAUNCH_CHECK(ctx);
    RLVI_CUDA(cudaMemsetAsync(tmp, 0, size_t(nsum) * 8, st));
    const int rc = rlvi_weighted_moments_f64(ctx, xd, y ? y + r0 : nullptr, weights + r0, rows, d, power, want_gram, tmp, st);
    if (rc != RLVI_OK) return rc;
    add_f64_kernel<<<(nsum + 255) / 256, 256, 0, st>>>(out, tmp, nsum, first ? 1 : 0);
    RLVI_LAUNCH_CHECK(ctx);
    first = false;
  }
  return RLVI_OK;
}

extern "C" int rlvi_weighted_moments_f32(rlvi_ctx* ctx, const float* X, const double* y, const double* weights, int64_t n,
                                         int d, int power, int want_gram, int precision, double* out, void* stream) {
  RLVI_REQUIRE(ctx && X && weights && out, "null pointer");
  RLVI_REQUIRE(n > 0 && d > 0, "n and d must be positive");
  RLVI_REQUIRE(power == 1 || power == 2, "power must be 1 or 2");
  RLVI_REQUIRE(precision == RLVI_TF32X3 || precision == RLVI_TF32X1, "precision must be RLVI_TF32X3 or RLVI_TF32X1");
  if (d > 1024) {
    rlvi_set_error("rlvi_weighted_moments_f32: d = %d > 1024 is not supported", d);
    return RLVI_ERR_UNSUPPORTED;
  }
  RlviDeviceGuard guard(ctx->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  EncodeTiledFn encode = encode_tiled_fn32();
  if (!encode || d > 4 * kMB || d % 4 != 0 || n >= (int64_t(1) << 31) - kR || !rlvi_aligned16(X))
    return moments_f32_via_f64(ctx, X, y, weights, n, d, power, want_gram, out, st);

  // The route and its partials (behind the 4 KiB scratch header), decided before anything is queued.  d = 129..512 runs
  // on CTA pairs when the device can co-schedule one pair per pair type, and otherwise takes the FP64 route; a B200
  // always can (148 SMs hold up to 74 pairs, at most 3 are needed).
  const bool pairs = d > kMB;
  PairPlan plan;
  CtaParams cp;
  memset(&cp, 0, sizeof(cp));
  size_t part_bytes = 0;
  if (pairs) {
    const int rc = rlvi_tf32_pair_plan(ctx, n, d, power, y != nullptr, precision, &plan);
    if (rc != RLVI_OK) return rc;
    if (plan.first[plan.ntypes] == 0) return moments_f32_via_f64(ctx, X, y, weights, n, d, power, want_gram, out, st);
    part_bytes = plan.part_bytes;
  } else {
    const int64_t ntiles = (n + kR - 1) / kR;
    cp.nslots = int(ntiles < ctx->sm_count ? ntiles : ctx->sm_count);
    part_bytes = size_t(cp.nslots) * (size_t(kMB) * kMB + kTeams * 2 * 128 + kTeams * 2) * sizeof(double);
  }

  CUtensorMap tmap, tmap3;
  const cuuint64_t gdim[2] = {cuuint64_t(d), cuuint64_t(n)};
  const cuuint64_t gstride[1] = {cuuint64_t(d) * 4};
  const cuuint32_t box[2] = {32, cuuint32_t(kR)};
  const cuuint32_t estr[3] = {1, 1, 1};
  CUresult cr = encode(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(X), gdim, gstride, box, estr,
                       CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                       CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (cr != CUDA_SUCCESS) {
    rlvi_set_error("cuTensorMapEncodeTiled (FP32) failed (%d)", int(cr));
    return RLVI_ERR_CUDA;
  }
  Tf32Params& p = cp.b;
  // d % 32 == 0: view X as [d/32 column groups][n rows][32 floats] so ONE box (32 x 16 x 4) fetches a whole
  // 128-feature block of a tile (TMA instructions issue at ~60 clk each); column groups past d/32 are zero-filled
  tmap3 = tmap;
  if (d % 32 == 0) {
    const cuuint64_t gdim3[3] = {32, cuuint64_t(n), cuuint64_t(d / 32)};
    const cuuint64_t gstride3[2] = {cuuint64_t(d) * 4, 128};
    const cuuint32_t box3[3] = {32, cuuint32_t(kR), 4};
    cr = encode(&tmap3, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(X), gdim3, gstride3, box3, estr,
                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    p.box3d = (cr == CUDA_SUCCESS) ? 1 : 0;
    if (!p.box3d) tmap3 = tmap;
  }
  p.w = weights;
  p.y = y;
  p.n = n;
  p.d = d;
  p.power = power;
  p.chunks_per_flush = 256;     // 32 Ki rows per register accumulation

  RlviScratch s;
  const int rc = rlvi_scratch_header(ctx, part_bytes, &s);
  if (rc != RLVI_OK) return rc;
  p.err = s.tf32_err;
  p.wmax = s.tf32_wmax;
  RLVI_CUDA(cudaMemsetAsync(p.err, 0, 16, st));          // error flag + the weight maximum
  wmax_kernel<<<grid_for(ctx, n, 8), 256, 0, st>>>(weights, n, s.tf32_wmax);
  RLVI_LAUNCH_CHECK(ctx);
  if (pairs)
    return rlvi_tf32_pair_moments(ctx, tmap, tmap3, p, plan, reinterpret_cast<char*>(s.partials), want_gram, out, st);

  const int grid = cp.nslots;
  p.gpart64 = s.partials;
  p.spart = p.gpart64 + size_t(grid) * kMB * kMB;
  cp.s0part = p.spart + size_t(grid) * kTeams * 2 * 128;
#define RLVI_TF32_LAUNCH(NS, HY)                                                                                   \
  {                                                                                                                \
    RLVI_CUDA(cudaFuncSetAttribute(gram_tf32_kernel<NS, HY>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemTotal)); \
    gram_tf32_kernel<NS, HY><<<grid, kThreads, kSmemTotal, st>>>(tmap, tmap3, cp);                                        \
  }
  if (precision == RLVI_TF32X1) {
    if (y) RLVI_TF32_LAUNCH(1, true) else RLVI_TF32_LAUNCH(1, false)
  } else {
    if (y) RLVI_TF32_LAUNCH(3, true) else RLVI_TF32_LAUNCH(3, false)
  }
#undef RLVI_TF32_LAUNCH
  RLVI_LAUNCH_CHECK(ctx);
  const int64_t total = int64_t(kMB) * kMB + 2 + 2 * int64_t(d);
  gram_tf32_finalize_kernel<<<int((total + 255) / 256), 256, 0, st>>>(cp, y ? 1 : 0, want_gram, out);
  RLVI_LAUNCH_CHECK(ctx);
  return RLVI_OK;
}
