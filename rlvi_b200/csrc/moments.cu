// moments.cu -- pi-weighted sufficient statistics of the M-step: ONE pass over X.
//
//   S0 = sum w,  Swy = sum w y,  S1 = X^T w,  Sy = X^T (w y),  G = X^T diag(w) X
//
// replaces the NumPy/BLAS contractions at standard-learning/rlvi.py:48,56 (mean), :70-71,79-80 (the
// normal equations of the sqrt(pi)-scaled lstsq), utils.py:36-38 (MM majoriser), :82-84 (Gram of the
// pi-scaled rows handed to PCA; power = 2) and :103-105 (covariance), none of which can run past
// N ~ 3e4 in the reference because of its N x N np.diag (SURVEY.md quirk Q5).
//
// d == 64 fast path (the headline shape, N = 2^26):
//   * persistent kernel, one CTA per SM, 8 consumer warps + 1 producer warp;
//   * the producer streams 64-row tiles (32 KiB of X + the rows' w and y) into a 6-stage shared-memory
//     ring with cp.async.bulk (the TMA engine; SASS UBLKCP) completing on mbarriers -- four 8 KiB copies
//     per tile, skewed by 16 bytes each so that the fragment reads are bank-conflict free;
//   * each consumer warp takes 4-sample k-groups and issues mma.sync.m8n8k4.f64 (SASS DMMA.8x8x4, the
//     only FP64 tensor shape sm_100a has; tcgen05 has no f64 kind) for the 36 upper-triangular 8x8
//     tiles of G, A = w * x (row scaling done in registers), B = x; all 72 accumulators of a lane stay
//     in registers for the whole kernel.  S1/Sy ride along as 16 DFMA per k-group;
//   * feature permutation: lane (g,t) of a warp reads, for J = 0..3, the 16 bytes holding features
//     16J + 2c(g) + {0,1}, c(g) = (g>>1)|((g&1)<<2); the two halves are MMA blocks 2J and 2J+1.  A
//     permutation of features is only a relabelling of G's rows/columns and is undone in the finalize
//     kernel.
//   * FP64-pipe bound: 36 DMMA x 512 flop per 4 rows = 4608 flop per 512-byte row (SURVEY.md H3).
//   * deterministic: per-CTA partials, then a fixed-order sum over CTAs in moments_finalize_kernel.
// Any other d (or unaligned pointers): generic register-tiled fallback (correct for all d, not tuned).
#include <math.h>

#include "rowmap.cuh"
#include "tma_ring.cuh"

namespace {

// ---------------------------------------------------------------------------------------------
// d = 64 fast path
// ---------------------------------------------------------------------------------------------
constexpr int kD = 64;
constexpr int kTileRows = 64;
constexpr int kGroupRows = 16;                        // rows per TMA copy; a tile = 4 groups
constexpr int kGroupPitch = kGroupRows * 512 + 16;    // groups land 16 B further round the banks (see consumer)
constexpr int kStages = 6;
constexpr int kConsumers = 8;                         // consumer warps
constexpr int kGramThreads = 384;                    // 2 consumer warpgroups + 1 producer warpgroup (1 active warp)
constexpr int kXBytes = 4 * kGroupPitch;              // 32832
constexpr int kStageBytes = ((kXBytes + 2 * kTileRows * 8) + 127) / 128 * 128;   // X tile + w + y
constexpr int kTiles36 = 36;
constexpr int kCompact = kTiles36 * 64;               // 2304 doubles: 36 tiles of 8x8
constexpr int kPartialStride = 2 + 2 * kD + kCompact; // S0, Swy, S1, Sy, G(compact)
constexpr int kGramSmem = kStages * kStageBytes + 2 * kStages * 8 + 64;

__host__ __device__ __forceinline__ int feat_of(int block, int r) {
  // MMA block `block` (0..7), fragment row/col r (0..7) -> feature index (see header comment)
  const int c = (r >> 1) | ((r & 1) << 2);
  return 16 * (block >> 1) + 2 * c + (block & 1);
}

struct GramParams {
  const double* X;
  const double* y;
  const double* w;
  const double* center;   // CENTERED: x_i is replaced by x_i - center
  int64_t n;
  int power;
  double* partials;   // [grid][kPartialStride]
};

template <bool HAS_Y, bool CENTERED>
__global__ void __launch_bounds__(kGramThreads, 1) gram64_kernel(const GramParams p) {
  extern __shared__ __align__(128) unsigned char smem[];
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kStages * kStageBytes);
  uint64_t* empty_bar = full_bar + kStages;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t ntiles = (p.n + kTileRows - 1) / kTileRows;
  double* smG = reinterpret_cast<double*>(smem);                 // epilogue view: [8][2304]
  double* smV = smG + kConsumers * kCompact;                      // [8][64] S1, [8][64] Sy, [8][2]

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], kConsumers);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  if (warp >= kConsumers) {
    // ===== producer warpgroup: hand its registers to the consumers (16 K regs per SM sub-partition:
    // 3 warps there would cap every warp at 168; the consumers need ~224) ========================
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    if (warp == kConsumers) {
      int stage = 0;
      uint32_t phase = 0;
      for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        mbar_wait(&empty_bar[stage], phase ^ 1u);
        unsigned char* sX = smem + stage * kStageBytes;
        double* sW = reinterpret_cast<double*>(sX + kXBytes);
        double* sY = sW + kTileRows;
        const int64_t row0 = tile * kTileRows;
        if (row0 + kTileRows <= p.n) {
          // FOUR 8 KiB copies per tile, one per 16-row group, each landing 16 bytes further round the banks.
          // (Per-row 512-byte copies into a padded pitch made the fragment reads conflict free but the
          // serialised UBLKCP issue, ~60 clk per row, left the tensor pipe 40 % idle.)  The four k-slots of
          // one DMMA take one row from EACH group, so the 16-byte skew between groups is what separates the
          // banks of the four rows a quarter-warp reads together.
          if (lane == 0) {
            mbar_arrive_expect_tx(&full_bar[stage], kTileRows * 512 + 512 + (HAS_Y ? 512 : 0));
#pragma unroll
            for (int q = 0; q < 4; ++q)
              bulk_g2s(sX + q * kGroupPitch, p.X + (row0 + q * kGroupRows) * kD, kGroupRows * 512, &full_bar[stage]);
            bulk_g2s(sW, p.w + row0, 512, &full_bar[stage]);
            if (HAS_Y) bulk_g2s(sY, p.y + row0, 512, &full_bar[stage]);
          }
        } else {
          // ragged last tile: plain loads, zero fill (w = 0 and x = 0 => no contribution)
          for (int idx = lane; idx < kTileRows * kD; idx += 32) {
            const int r = idx >> 6, c = idx & 63;
            double* dst = reinterpret_cast<double*>(sX + (r / kGroupRows) * kGroupPitch + (r % kGroupRows) * 512);
            dst[c] = (row0 + r < p.n) ? p.X[(row0 + r) * kD + c] : 0.0;
          }
          for (int r = lane; r < kTileRows; r += 32) {
            sW[r] = (row0 + r < p.n) ? p.w[row0 + r] : 0.0;
            sY[r] = (HAS_Y && row0 + r < p.n) ? p.y[row0 + r] : 0.0;
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&full_bar[stage]);
        }
        if (++stage == kStages) {
          stage = 0;
          phase ^= 1u;
        }
      }
    }
  } else {
    // ===== consumer warps ====================================================================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 232;");
    double acc[2 * kTiles36];
    double s1[8], sy[8];
    double s0 = 0.0, swy = 0.0;
#pragma unroll
    for (int i = 0; i < 2 * kTiles36; ++i) acc[i] = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      s1[i] = 0.0;
      sy[i] = 0.0;
    }
    const int g = lane >> 2, t = lane & 3;
    const int cidx = (g >> 1) | ((g & 1) << 2);
    double cb[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) cb[j] = CENTERED ? p.center[feat_of(j, g)] : 0.0;
    int stage = 0;
    uint32_t phase = 0;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      mbar_wait(&full_bar[stage], phase);
      const unsigned char* sX = smem + stage * kStageBytes;
      const double* sW = reinterpret_cast<const double*>(sX + kXBytes);
      const double* sY = sW + kTileRows;
#pragma unroll
      for (int kk = 0; kk < kTileRows / (4 * kConsumers); ++kk) {
        // k-group kg = warp + 8 kk: its four samples are row kg of each 16-row group (k-slot t <-> group t)
        const int kg = warp + kConsumers * kk;
        const int r = t * kGroupRows + kg;
        const unsigned char* xr = sX + t * kGroupPitch + kg * 512 + cidx * 16;
        const double2 x0 = *reinterpret_cast<const double2*>(xr);
        const double2 x1 = *reinterpret_cast<const double2*>(xr + 128);
        const double2 x2 = *reinterpret_cast<const double2*>(xr + 256);
        const double2 x3 = *reinterpret_cast<const double2*>(xr + 384);
        double b[8] = {x0.x, x0.y, x1.x, x1.y, x2.x, x2.y, x3.x, x3.y};
        if (CENTERED) {
#pragma unroll
          for (int j = 0; j < 8; ++j) b[j] -= cb[j];
        }
        const double w1 = sW[r];
        const double we = (p.power == 2) ? w1 * w1 : w1;
        double wy = 0.0;
        if (HAS_Y) wy = we * sY[r];
        if (g == 0) {
          s0 += we;
          swy += wy;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          s1[j] = fma(w1, b[j], s1[j]);
          if (HAS_Y) sy[j] = fma(wy, b[j], sy[j]);
        }
        // all eight scaled A fragments first (one register each): with a single temporary the DMUL ->
        // DMMA -> DMUL chain serialised the tensor pipe (ncu: 60 % DMMA utilisation, stall_math on DMUL)
        double a[8];
#pragma unroll
        for (int I = 0; I < 8; ++I) a[I] = we * b[I];
        // ptxas sinks each DMUL to just before its first DMMA (one shared temporary); a never-taken store that reads all
        // eight products pins them here (same-box A/B at N = 2^26: 9.620 -> 9.598 ms -- the scheduler's other warp
        // already covered most of that latency)
        if (p.n < 0) {
#pragma unroll
          for (int I = 0; I < 8; ++I) reinterpret_cast<volatile double*>(smem)[lane + 32 * I] = a[I];
        }
        int idx = 0;
#pragma unroll
        for (int I = 0; I < 8; ++I) {
#pragma unroll
          for (int J = I; J < 8; ++J) {
            dmma884(acc[2 * idx], acc[2 * idx + 1], a[I], b[J]);
            ++idx;
          }
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty_bar[stage]);
      if (++stage == kStages) {
        stage = 0;
        phase ^= 1u;
      }
    }
    // all consumers are done reading the ring (and every issued copy has been consumed): reuse it
    asm volatile("bar.sync 1, %0;" ::"n"(kConsumers * 32) : "memory");
#pragma unroll
    for (int idx = 0; idx < kTiles36; ++idx) {
      *reinterpret_cast<double2*>(smG + (warp * kTiles36 + idx) * 64 + g * 8 + 2 * t) =
          make_double2(acc[2 * idx], acc[2 * idx + 1]);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      double v = s1[j];
      v += __shfl_xor_sync(0xffffffffu, v, 1);
      v += __shfl_xor_sync(0xffffffffu, v, 2);
      double u = sy[j];
      u += __shfl_xor_sync(0xffffffffu, u, 1);
      u += __shfl_xor_sync(0xffffffffu, u, 2);
      if (t == 0) {
        smV[warp * 64 + feat_of(j, g)] = v;
        smV[kConsumers * 64 + warp * 64 + feat_of(j, g)] = u;
      }
    }
    const double t0 = warp_sum(s0), t1 = warp_sum(swy);
    if (lane == 0) {
      smV[2 * kConsumers * 64 + 2 * warp] = t0;
      smV[2 * kConsumers * 64 + 2 * warp + 1] = t1;
    }
  }

  // ===== cross-warp sum in shared memory, fixed warp order =======================================
  __syncthreads();
  double* out = p.partials + size_t(blockIdx.x) * kPartialStride;
  for (int e = threadIdx.x; e < kCompact; e += blockDim.x) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < kConsumers; ++w) s += smG[w * kCompact + e];
    out[2 + 2 * kD + e] = s;
  }
  if (threadIdx.x < 2 * kD) {
    const int which = threadIdx.x >> 6, f = threadIdx.x & 63;
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < kConsumers; ++w) s += smV[which * kConsumers * 64 + w * 64 + f];
    out[2 + which * kD + f] = s;
  } else if (threadIdx.x < 2 * kD + 2) {
    const int which = threadIdx.x - 2 * kD;
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < kConsumers; ++w) s += smV[2 * kConsumers * 64 + 2 * w + which];
    out[which] = s;
  }
}

// Sum the per-CTA partials in CTA order and scatter to the public layout.
__global__ void gram64_finalize_kernel(const double* __restrict__ partials, int nparts, int want_gram,
                                       double* __restrict__ out) {
  // four lanes per output element: lane q adds the CTA partials c = q, q + 4, ... in order, then a fixed
  // two-level shuffle tree (148 dependent loads per thread made this 15 us; it matters once a GPU's shard of
  // the statistics pass takes ~1 ms)
  const int gid = blockIdx.x * blockDim.x + threadIdx.x;
  const int e = gid >> 2, q = gid & 3;
  double s = 0.0;
  if (e < kPartialStride && (want_gram || e < 2 + 2 * kD)) {
    for (int c = q; c < nparts; c += 4) s += partials[size_t(c) * kPartialStride + e];
  }
  s += __shfl_xor_sync(0xffffffffu, s, 1);
  s += __shfl_xor_sync(0xffffffffu, s, 2);
  if (q != 0 || e >= kPartialStride) return;
  if (!want_gram && e >= 2 + 2 * kD) return;
  if (e < 2 + 2 * kD) {
    out[e] = s;
    return;
  }
  const int ce = e - (2 + 2 * kD);
  const int tile = ce >> 6, r = (ce >> 3) & 7, c = ce & 7;
  int I = 0, rem = tile;
  while (rem >= 8 - I) {
    rem -= 8 - I;
    ++I;
  }
  const int J = I + rem;
  const int fi = feat_of(I, r), fj = feat_of(J, c);
  double* G = out + 2 + 2 * kD;
  if (I < J) {
    G[fi * kD + fj] = s;
    G[fj * kD + fi] = s;
  } else if (fi <= fj) {   // diagonal tile: keep one triangle so G is exactly symmetric
    G[fi * kD + fj] = s;
    G[fj * kD + fi] = s;
  }
}

// ---------------------------------------------------------------------------------------------
// generic fallback, any d: (a) column sums, (b) register-tiled Gram, (c) finalize
// ---------------------------------------------------------------------------------------------
constexpr int kColThreads = 256;

struct ColParams {
  const double* X;
  const double* y;
  const double* w;
  const double* params;   // logistic gradient: [b, theta(d)]
  const double* center;   // MODE 0, optional: x_i - center
  int64_t n;
  int d;
  int power;
  int L;
  double* partials;       // [grid][2 + 2*d]
};

// MODE 0: moments  c1 = w (first power), c2 = we*y, S0 = sum we, Swy = sum we*y
// MODE 1: logistic gradient  c1 = w (sigmoid(b + x.theta) - y); out[0] = sum c1, out[2..2+d) = X^T c1
template <int MODE, int FPL, bool VEC>
__global__ void __launch_bounds__(kColThreads) colsum_kernel(const ColParams p) {
  extern __shared__ double smc[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  const int L = p.L, q = lane & (L - 1), sub = lane / L, R = 32 / L;
  double th[FPL];
  double b0 = 0.0;
  if (MODE == 1) {
    for (int i = threadIdx.x; i < p.d + 1; i += blockDim.x) smc[i] = p.params[i];
    __syncthreads();
    b0 = smc[0];
    RowMap<FPL, VEC>::load_vec(smc + 1, p.d, q, L, th);
    __syncthreads();
  }
  double a1[FPL], a2[FPL], cen[FPL];
#pragma unroll
  for (int k = 0; k < FPL; ++k) {
    a1[k] = 0.0;
    a2[k] = 0.0;
    const int f = RowMap<FPL, VEC>::feature(k, q, L);
    cen[k] = (MODE == 0 && p.center && f < p.d) ? p.center[f] : 0.0;
  }
  double s0 = 0.0, swy = 0.0;
  const int64_t warps_total = int64_t(gridDim.x) * nwarp;
  const int64_t warp_id = int64_t(blockIdx.x) * nwarp + warp;
  for (int64_t row0 = warp_id * R; row0 < p.n; row0 += warps_total * R) {
    const int64_t row = row0 + sub;
    const bool valid = row < p.n;
    double x[FPL];
    RowMap<FPL, VEC>::load_row(p.X, row, p.d, q, L, valid, x);
    if (MODE == 0) {
#pragma unroll
      for (int k = 0; k < FPL; ++k) x[k] -= cen[k];   // rows past n carry w = 0
    }
    const double w1 = valid ? p.w[row] : 0.0;
    const double yi = (valid && p.y) ? p.y[row] : 0.0;
    double c1, c2 = 0.0;
    if (MODE == 0) {
      const double we = (p.power == 2) ? w1 * w1 : w1;
      c1 = w1;
      c2 = we * yi;
      if (q == 0) {
        s0 += we;
        swy += c2;
      }
    } else {
      double a = 0.0;
#pragma unroll
      for (int k = 0; k < FPL; ++k) a = fma(x[k], th[k], a);
      a = group_sum(a, L);
      const double phi = b0 + a;
      // utils.py:7-16 sigmoid, overflow-free form
      const double z = exp(-fabs(phi));
      const double sg = (phi >= 0.0 ? 1.0 : z) / (1.0 + z);
      c1 = w1 * (sg - yi);
      if (q == 0) s0 += c1;
    }
#pragma unroll
    for (int k = 0; k < FPL; ++k) {
      a1[k] = fma(c1, x[k], a1[k]);
      if (MODE == 0) a2[k] = fma(c2, x[k], a2[k]);
    }
  }
  // lanes with the same q hold partial sums of the same features: fold the row groups of the warp
#pragma unroll
  for (int k = 0; k < FPL; ++k) {
    for (int o = L; o < 32; o <<= 1) {
      a1[k] += __shfl_xor_sync(0xffffffffu, a1[k], o);
      if (MODE == 0) a2[k] += __shfl_xor_sync(0xffffffffu, a2[k], o);
    }
  }
  s0 = warp_sum(s0);
  swy = warp_sum(swy);
  // per-warp vectors to shared memory, then a fixed-order sum over warps
  const int stride = 2 + 2 * p.d;
  double* mine = smc + size_t(warp) * stride;
  __syncthreads();
  if (sub == 0) {
#pragma unroll
    for (int k = 0; k < FPL; ++k) {
      const int f = RowMap<FPL, VEC>::feature(k, q, L);
      if (f < p.d) {
        mine[2 + f] = a1[k];
        mine[2 + p.d + f] = a2[k];
      }
    }
  }
  if (lane == 0) {
    mine[0] = s0;
    mine[1] = swy;
  }
  __syncthreads();
  double* out = p.partials + size_t(blockIdx.x) * stride;
  for (int e = threadIdx.x; e < stride; e += blockDim.x) {
    double s = 0.0;
    for (int w = 0; w < nwarp; ++w) s += smc[size_t(w) * stride + e];
    out[e] = s;
  }
}

// out[e] = sum over parts of element src(e), e < count (fixed order).  skip1: the gradient layout
// drops slot 1 (Swy) of the partial vector: src(0) = 0, src(e) = e + 1.
__global__ void sum_parts_kernel(const double* __restrict__ partials, int nparts, int stride, int count,
                                 int skip1, double* __restrict__ out) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= count) return;
  const int src = (skip1 && e > 0) ? e + 1 : e;
  double s = 0.0;
  for (int c = 0; c < nparts; ++c) s += partials[size_t(c) * stride + src];
  out[e] = s;
}

// Register-tiled Gram for arbitrary d: CTA (bx <= by pair, row chunk) computes a 64x64 block of
// X^T diag(we) X over its rows; 16x16 threads, 4x4 outputs each.
constexpr int kGT = 64;   // block edge
constexpr int kGR = 16;   // rows per shared-memory step

struct GenGramParams {
  const double* X;
  const double* w;
  const double* center;
  int64_t n;
  int d;
  int power;
  int nb;            // ceil(d/64)
  int nchunks;
  int64_t rows_per_chunk;
  double* partials;  // [nchunks][npairs][64*64]
};

__global__ void __launch_bounds__(256) gen_gram_kernel(const GenGramParams p) {
  __shared__ double As[kGR][kGT + 4];
  __shared__ double Bs[kGR][kGT + 4];
  // pair index -> (bi, bj), bi <= bj
  int bi = 0, rem = blockIdx.x;
  while (rem >= p.nb - bi) {
    rem -= p.nb - bi;
    ++bi;
  }
  const int bj = bi + rem;
  const int chunk = blockIdx.y;
  const int64_t r_begin = int64_t(chunk) * p.rows_per_chunk;
  const int64_t r_end = (r_begin + p.rows_per_chunk < p.n) ? r_begin + p.rows_per_chunk : p.n;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  double acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0;
  for (int64_t r0 = r_begin; r0 < r_end; r0 += kGR) {
    for (int idx = threadIdx.x; idx < kGR * kGT; idx += blockDim.x) {
      const int r = idx >> 6, c = idx & 63;
      const int64_t row = r0 + r;
      double wa = 0.0, xa = 0.0, xb = 0.0;
      if (row < r_end) {
        const double w1 = p.w[row];
        wa = (p.power == 2) ? w1 * w1 : w1;
        const int fa = bi * kGT + c, fb = bj * kGT + c;
        if (fa < p.d) xa = p.X[row * int64_t(p.d) + fa] - (p.center ? p.center[fa] : 0.0);
        if (fb < p.d) xb = p.X[row * int64_t(p.d) + fb] - (p.center ? p.center[fb] : 0.0);
      }
      As[r][c] = wa * xa;
      Bs[r][c] = xb;
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < kGR; ++r) {
      double a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        a[i] = As[r][ty * 4 + i];
        b[i] = Bs[r][tx * 4 + i];
      }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fma(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
  const int npairs = p.nb * (p.nb + 1) / 2;
  double* out = p.partials + (size_t(chunk) * npairs + blockIdx.x) * (kGT * kGT);
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) out[(ty * 4 + i) * kGT + tx * 4 + j] = acc[i][j];
}

__global__ void gen_gram_finalize_kernel(const double* __restrict__ partials, int nchunks, int nb, int d,
                                         double* __restrict__ G) {
  const int npairs = nb * (nb + 1) / 2;
  const int64_t e = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (e >= int64_t(npairs) * kGT * kGT) return;
  const int pair = int(e / (kGT * kGT)), within = int(e % (kGT * kGT));
  int bi = 0, rem = pair;
  while (rem >= nb - bi) {
    rem -= nb - bi;
    ++bi;
  }
  const int bj = bi + rem;
  const int fi = bi * kGT + within / kGT, fj = bj * kGT + within % kGT;
  if (fi >= d || fj >= d) return;
  if (bi == bj && fi > fj) return;   // one triangle of diagonal blocks, mirrored below
  double s = 0.0;
  for (int c = 0; c < nchunks; ++c) s += partials[(size_t(c) * npairs + pair) * (kGT * kGT) + within];
  G[size_t(fi) * d + fj] = s;
  G[size_t(fj) * d + fi] = s;
}

template <int MODE>
int launch_colsum(rlvi_ctx* ctx, const RowMapCfg& cfg, ColParams& p, int grid, size_t smem, cudaStream_t st) {
#define RLVI_COL_CASE(F, V)                                                                                   \
  if (cfg.fpl == F && cfg.vec == V) {                                                                         \
    if (smem > 48 * 1024)                                                                                     \
      RLVI_CUDA(cudaFuncSetAttribute(colsum_kernel<MODE, F, V>, cudaFuncAttributeMaxDynamicSharedMemorySize,  \
                                     int(smem)));                                                             \
    colsum_kernel<MODE, F, V><<<grid, kColThreads, smem, st>>>(p);                                            \
    RLVI_LAUNCH_CHECK(ctx);                                                                                   \
    return RLVI_OK;                                                                                           \
  }
  RLVI_COL_CASE(4, true)
  RLVI_COL_CASE(4, false)
  RLVI_COL_CASE(16, true)
  RLVI_COL_CASE(16, false)
  RLVI_COL_CASE(32, true)
  RLVI_COL_CASE(32, false)
#undef RLVI_COL_CASE
  rlvi_set_error("no colsum kernel for fpl=%d", cfg.fpl);
  return RLVI_ERR_UNSUPPORTED;
}

// ---------------------------------------------------------------------------------------------
// TMA-fed column sums (d % 16 == 0, d <= 256, 16-byte aligned pointers): the producer / private-ring skeleton
// of tma_ring.cuh (shared with loss_tma_kernel) feeding a two-phase consumer.
//   phase 1 (MODE 1 only): lane = row, rotated conflict-free walk, phi = b + x.theta,
//                          c1 = w (sigmoid(phi) - y)                       utils.py:40-41
//           (MODE 0)      : c1 = w, c2 = we * y                           rlvi.py:48,56,71,80
//   phase 2: lane = feature pair(s): acc[f] += c_r * x[r][f] over the 32 rows of the tile, c_r broadcast from
//            shared memory; every 128-bit read of x is one conflict-free wavefront per 8 lanes.
// Per-warp d-vectors are summed in warp order, per-CTA partials in CTA order (sum_parts_kernel).
// ---------------------------------------------------------------------------------------------
struct ColTmaParams {
  const double* X;
  const double* y;
  const double* w;
  const double* params;
  const double* center;   // MODE 0, optional
  int64_t n;
  int d;
  int power;
  RingGeom geom;
  double* partials;  // [grid][2 + 2 d]
};

static inline size_t colsum_tma_tail(int d) {
  return size_t(d + 2) * 8 + kRingBarrierBytes + size_t(kRingConsumers) * 64 * 8 + size_t(kRingConsumers) * (2 + 2 * d) * 8 + 128;
}

template <int MODE>
__global__ void __launch_bounds__(kRingThreads, 1) colsum_tma_kernel(const ColTmaParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int C = p.geom.ncons;
  Ring ring;
  ring.base = smem_raw;
  ring.g = p.geom;
  ring.d = p.d;
  double* sTheta = reinterpret_cast<double*>(smem_raw + ring_bytes(p.geom));              // d (+ 2)
  ring.full_bar = reinterpret_cast<uint64_t*>(sTheta + p.d + 2);
  ring.empty_bar = ring.full_bar + kRingMaxStages;
  double* sC = reinterpret_cast<double*>(ring.empty_bar + kRingMaxStages);                 // [C][2][32] row coefficients
  double* sOut = sC + kRingConsumers * 64;                                                  // [C][2 + 2 d]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int d = p.d, npair = d >> 1;
  const int stride = 2 + 2 * d;
  if (MODE == 1)
    for (int i = threadIdx.x; i < d; i += blockDim.x) sTheta[i] = p.params[1 + i];
  ring_init(ring);
  const double b0 = (MODE == 1) ? p.params[0] : 0.0;
  const int64_t my_tiles = ring_my_tiles(p.n);
  const bool has_y = p.y != nullptr;

  if (warp == kRingConsumers) {
    // rows past n of the ragged tile enter the sums with weight 0: clear them (a stale NaN x 0 would poison)
    ring_produce(ring, p.X, p.y, p.w, p.n, my_tiles, true);
  } else if (warp < C) {
    const double2* th2 = reinterpret_cast<const double2*>(sTheta);
    double* myC = sC + warp * 64;
    constexpr int kMaxUnitsPerLane = 4;          // d <= 256 -> <= 128 units of 16 bytes per row
    double a1[2 * kMaxUnitsPerLane], a2[2 * kMaxUnitsPerLane];
#pragma unroll
    for (int i = 0; i < 2 * kMaxUnitsPerLane; ++i) {
      a1[i] = 0.0;
      a2[i] = 0.0;
    }
    double cen[2 * kMaxUnitsPerLane];
#pragma unroll
    for (int v = 0; v < kMaxUnitsPerLane; ++v) {
      const int unit = lane + 32 * v;
      const bool on = (MODE == 0) && p.center && unit < npair;
      cen[2 * v] = on ? p.center[2 * unit] : 0.0;
      cen[2 * v + 1] = on ? p.center[2 * unit + 1] : 0.0;
    }
    double s0 = 0.0, swy = 0.0;
    for (int64_t t = warp; t < my_tiles; t += C) {
      const RingStage st = ring_acquire(ring, warp, t);
      const double2* xt = reinterpret_cast<const double2*>(st.x);
      // ---- phase 1: one row per lane -> its coefficients
      const double w1 = st.w[lane];
      const double yi = has_y ? st.y[lane] : 0.0;
      double c1, c2 = 0.0;
      if (MODE == 0) {
        const double we = (p.power == 2) ? w1 * w1 : w1;
        c1 = w1;
        c2 = we * yi;
        s0 += we;
        swy += c2;
      } else {
        const double2* xr = xt + size_t(lane) * npair;
        double q0 = 0.0, q1 = 0.0, q2 = 0.0, q3 = 0.0;
        int u = lane % npair;
#pragma unroll 4
        for (int j = 0; j < npair; j += 2) {
          int u1 = u + 1;
          if (u1 == npair) u1 = 0;
          const double2 x0 = xr[u], x1 = xr[u1];
          const double2 t0 = th2[u], t1 = th2[u1];
          u = u1 + 1;
          if (u == npair) u = 0;
          q0 = fma(x0.x, t0.x, q0);
          q1 = fma(x0.y, t0.y, q1);
          q2 = fma(x1.x, t1.x, q2);
          q3 = fma(x1.y, t1.y, q3);
        }
        const double phi = b0 + ((q0 + q1) + (q2 + q3));
        const double z = exp(-fabs(phi));                       // utils.py:7-16 sigmoid, overflow-free form
        const double sg = (phi >= 0.0 ? 1.0 : z) / (1.0 + z);
        c1 = w1 * (sg - yi);
        s0 += c1;
      }
      myC[lane] = c1;
      if (MODE == 0) myC[32 + lane] = c2;
      __syncwarp();
      // ---- phase 2: lane = feature pair(s); acc += c_r * x[r][.] over the tile's rows
#pragma unroll 4
      for (int rr = 0; rr < kRingRows; ++rr) {
        const double k1 = myC[rr];
        const double k2 = (MODE == 0) ? myC[32 + rr] : 0.0;
        const double2* xrow = xt + size_t(rr) * npair;
#pragma unroll
        for (int v = 0; v < kMaxUnitsPerLane; ++v) {
          const int unit = lane + 32 * v;
          if (unit < npair) {
            double2 x = xrow[unit];
            if (MODE == 0) {
              x.x -= cen[2 * v];
              x.y -= cen[2 * v + 1];
            }
            a1[2 * v] = fma(k1, x.x, a1[2 * v]);
            a1[2 * v + 1] = fma(k1, x.y, a1[2 * v + 1]);
            if (MODE == 0) {
              a2[2 * v] = fma(k2, x.x, a2[2 * v]);
              a2[2 * v + 1] = fma(k2, x.y, a2[2 * v + 1]);
            }
          }
        }
      }
      ring_release(ring, st);
    }
    // per-warp vector to shared memory
    double* mine = sOut + size_t(warp) * stride;
    s0 = warp_sum(s0);
    swy = warp_sum(swy);
    if (lane == 0) {
      mine[0] = s0;
      mine[1] = swy;
    }
#pragma unroll
    for (int v = 0; v < kMaxUnitsPerLane; ++v) {
      const int unit = lane + 32 * v;
      if (unit < npair) {
        mine[2 + 2 * unit] = a1[2 * v];
        mine[2 + 2 * unit + 1] = a1[2 * v + 1];
        mine[2 + d + 2 * unit] = a2[2 * v];
        mine[2 + d + 2 * unit + 1] = a2[2 * v + 1];
      }
    }
  }
  __syncthreads();
  double* out = p.partials + size_t(blockIdx.x) * stride;
  for (int e = threadIdx.x; e < stride; e += blockDim.x) {
    double s = 0.0;
    for (int w = 0; w < C; ++w) s += sOut[size_t(w) * stride + e];
    out[e] = s;
  }
}

// shared host driver for the two colsum modes; result lands in out[0 .. 2+2d)
template <int MODE>
int run_colsum(rlvi_ctx* ctx, const double* X, const double* y, const double* w, const double* params,
               const double* center, int64_t n, int d, int power, double* out, int count, cudaStream_t st) {
  // ---- TMA-fed path -------------------------------------------------------------------------------
  if (d % 16 == 0 && d <= 256 && n >= kRingRows && rlvi_aligned16(X) && rlvi_aligned16(w) && (!y || rlvi_aligned16(y))) {
    ColTmaParams q;
    q.X = X;
    q.y = y;
    q.w = w;
    q.params = params;
    q.center = center;
    q.n = n;
    q.d = d;
    q.power = power;
    const int stride = 2 + 2 * d;
    const size_t tail = colsum_tma_tail(d);
    if (ring_geometry(d, tail, &q.geom)) {
      const int grid = ring_grid(q.geom, n, ctx->sm_count);
      RlviScratch s;
      const int rc = rlvi_scratch_header(ctx, size_t(grid) * stride * sizeof(double), &s);
      if (rc != RLVI_OK) return rc;
      q.partials = s.partials;
      const size_t smem = ring_bytes(q.geom) + tail;
      RLVI_CUDA(cudaFuncSetAttribute(colsum_tma_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
      colsum_tma_kernel<MODE><<<grid, kRingThreads, smem, st>>>(q);
      RLVI_LAUNCH_CHECK(ctx);
      sum_parts_kernel<<<(count + 255) / 256, 256, 0, st>>>(q.partials, grid, stride, count, MODE == 1 ? 1 : 0, out);
      RLVI_LAUNCH_CHECK(ctx);
      return RLVI_OK;
    }
  }

  RowMapCfg cfg;
  if (!rowmap_pick(d, rlvi_aligned16(X), &cfg)) {
    rlvi_set_error("column-sum kernels support 1 <= d <= 1024 (got %d)", d);
    return RLVI_ERR_UNSUPPORTED;
  }
  const int nwarp = kColThreads / 32;
  const int R = 32 / cfg.L;
  const int64_t steps = (n + R - 1) / R;
  int64_t want = (steps + nwarp - 1) / nwarp;
  // fewer, fatter CTAs: every CTA ends with a (2+2d)-vector reduction
  const int64_t cap = int64_t(ctx->sm_count) * 2;
  const int grid = int(want < 1 ? 1 : (want > cap ? cap : want));
  const int stride = 2 + 2 * d;
  RlviScratch s;
  int rc = rlvi_scratch_header(ctx, size_t(grid) * stride * sizeof(double), &s);
  if (rc != RLVI_OK) return rc;
  ColParams p;
  p.X = X;
  p.y = y;
  p.w = w;
  p.params = params;
  p.center = center;
  p.n = n;
  p.d = d;
  p.power = power;
  p.L = cfg.L;
  p.partials = s.partials;
  size_t smem = size_t(nwarp) * stride * sizeof(double);
  if (smem < size_t(d + 1) * sizeof(double)) smem = size_t(d + 1) * sizeof(double);
  rc = launch_colsum<MODE>(ctx, cfg, p, grid, smem, st);
  if (rc != RLVI_OK) return rc;
  sum_parts_kernel<<<(count + 255) / 256, 256, 0, st>>>(p.partials, grid, stride, count, MODE == 1 ? 1 : 0, out);
  RLVI_LAUNCH_CHECK(ctx);
  return RLVI_OK;
}

}  // namespace

extern "C" int rlvi_moments_out_doubles(int d) { return 2 + 2 * d + d * d; }

static int weighted_moments_impl(rlvi_ctx* ctx, const double* X, const double* y, const double* weights,
                                 const double* center, int64_t n, int d, int power, int want_gram, double* out,
                                 void* stream);

extern "C" int rlvi_weighted_moments_f64(rlvi_ctx* ctx, const double* X, const double* y, const double* weights,
                                         int64_t n, int d, int power, int want_gram, double* out, void* stream) {
  return weighted_moments_impl(ctx, X, y, weights, nullptr, n, d, power, want_gram, out, stream);
}

extern "C" int rlvi_weighted_moments_centered_f64(rlvi_ctx* ctx, const double* X, const double* y,
                                                  const double* weights, const double* center, int64_t n, int d,
                                                  int power, int want_gram, double* out, void* stream) {
  RLVI_REQUIRE(center != nullptr, "null centre");
  return weighted_moments_impl(ctx, X, y, weights, center, n, d, power, want_gram, out, stream);
}

static int weighted_moments_impl(rlvi_ctx* ctx, const double* X, const double* y, const double* weights,
                                 const double* center, int64_t n, int d, int power, int want_gram, double* out,
                                 void* stream) {
  RLVI_REQUIRE(ctx && X && weights && out, "null pointer");
  RLVI_REQUIRE(n > 0 && d > 0, "n and d must be positive");
  RLVI_REQUIRE(power == 1 || power == 2, "power must be 1 or 2");
  RlviDeviceGuard guard(ctx->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);

  const bool fast = (d == kD) && rlvi_aligned16(X) && rlvi_aligned16(weights) && (!y || rlvi_aligned16(y)) &&
                    want_gram;
  if (fast) {
    const int64_t ntiles = (n + kTileRows - 1) / kTileRows;
    const int grid = int(ntiles < ctx->sm_count ? ntiles : ctx->sm_count);
    RlviScratch s;
    const int rc = rlvi_scratch_header(ctx, size_t(grid) * kPartialStride * sizeof(double), &s);
    if (rc != RLVI_OK) return rc;
    GramParams p;
    p.X = X;
    p.y = y;
    p.w = weights;
    p.n = n;
    p.power = power;
    p.partials = s.partials;
    p.center = center;
#define RLVI_GRAM64_LAUNCH(HY, CE)                                                                              \
  {                                                                                                             \
    RLVI_CUDA(cudaFuncSetAttribute(gram64_kernel<HY, CE>, cudaFuncAttributeMaxDynamicSharedMemorySize, kGramSmem)); \
    gram64_kernel<HY, CE><<<grid, kGramThreads, kGramSmem, st>>>(p);                                            \
  }
    if (y && center) RLVI_GRAM64_LAUNCH(true, true)
    else if (y) RLVI_GRAM64_LAUNCH(true, false)
    else if (center) RLVI_GRAM64_LAUNCH(false, true)
    else RLVI_GRAM64_LAUNCH(false, false)
#undef RLVI_GRAM64_LAUNCH
    RLVI_LAUNCH_CHECK(ctx);
    gram64_finalize_kernel<<<(4 * kPartialStride + 255) / 256, 256, 0, st>>>(p.partials, grid, want_gram, out);
    RLVI_LAUNCH_CHECK(ctx);
    return RLVI_OK;
  }

  // ---- general d on the FP64 tensor pipe, TMA tensor-map fed (gram_tma.cu) --------------------------
  if (want_gram) {
    const int trc = rlvi_gram_tma_f64(ctx, X, y, weights, center, n, d, power, want_gram, out, st);
    if (trc != RLVI_ERR_UNSUPPORTED) return trc;
  }

  // ---- fallback (odd d, unaligned pointers, tiny n): vectors first, then a register-tiled Gram ------
  int rc = run_colsum<0>(ctx, X, y, weights, nullptr, center, n, d, power, out, 2 + 2 * d, st);
  if (rc != RLVI_OK) return rc;
  if (!want_gram) return RLVI_OK;
  if (d > 4096) {
    rlvi_set_error("generic Gram supports d <= 4096 (got %d)", d);
    return RLVI_ERR_UNSUPPORTED;
  }
  GenGramParams g;
  g.X = X;
  g.w = weights;
  g.center = center;
  g.n = n;
  g.d = d;
  g.power = power;
  g.nb = (d + kGT - 1) / kGT;
  const int npairs = g.nb * (g.nb + 1) / 2;
  int64_t nchunks = (int64_t(ctx->sm_count) * 4 + npairs - 1) / npairs;
  const int64_t max_chunks = (n + kGR - 1) / kGR;
  if (nchunks > max_chunks) nchunks = max_chunks;
  if (nchunks < 1) nchunks = 1;
  if (nchunks > 65535) nchunks = 65535;
  g.rows_per_chunk = ((n + nchunks - 1) / nchunks + kGR - 1) / kGR * kGR;
  nchunks = (n + g.rows_per_chunk - 1) / g.rows_per_chunk;
  g.nchunks = int(nchunks);
  RlviScratch s;
  rc = rlvi_scratch_header(ctx, size_t(nchunks) * npairs * kGT * kGT * sizeof(double), &s);
  if (rc != RLVI_OK) return rc;
  g.partials = s.partials;
  gen_gram_kernel<<<dim3(npairs, g.nchunks), 256, 0, st>>>(g);
  RLVI_LAUNCH_CHECK(ctx);
  const int64_t total = int64_t(npairs) * kGT * kGT;
  gen_gram_finalize_kernel<<<int((total + 255) / 256), 256, 0, st>>>(g.partials, g.nchunks, g.nb, d,
                                                                     out + 2 + 2 * d);
  RLVI_LAUNCH_CHECK(ctx);
  return RLVI_OK;
}

extern "C" int rlvi_logistic_grad_f64(rlvi_ctx* ctx, const double* X, const double* y, const double* weights,
                                      int64_t n, int d, const double* params, double* out, void* stream) {
  RLVI_REQUIRE(ctx && X && y && weights && params && out, "null pointer");
  RLVI_REQUIRE(n > 0 && d > 0, "n and d must be positive");
  RlviDeviceGuard guard(ctx->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // colsum MODE 1 leaves [sum c, -, X^T c (d), -] per CTA; the final sum gathers [sum c, X^T c]
  return run_colsum<1>(ctx, X, y, weights, params, nullptr, n, d, 1, out, 1 + d, st);
}
