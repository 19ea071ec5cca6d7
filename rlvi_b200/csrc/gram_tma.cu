// gram_tma.cu -- pi-weighted Gram X^T diag(w) X for GENERAL d on the FP64 tensor pipe (the d = 64 headline
// shape has its own kernel in moments.cu).
//
//   * the d features are cut into nb = ceil(d/64) blocks; a work unit is (row chunk, block pair bi <= bj): one
//     CTA computes the 64 x 64 block G[bi][bj] over its rows -- the 36 upper-triangular 8x8 tiles when
//     bi == bj, all 64 tiles otherwise -- with mma.sync.m8n8k4.f64 (SASS DMMA.8x8x4);
//   * units are ordered pair-minor, so the CTAs resident at the same time work on the same rows and X comes
//     from HBM once and from L2 for the other pairs;
//   * X tiles (64 rows x 64 features of block bi, and of bj) are fetched by the TMA engine through a 2-D
//     TENSOR MAP (cp.async.bulk.tensor.2d, SASS UTMALDG): box = 16 features (128 B) x 64 rows,
//     CU_TENSOR_MAP_SWIZZLE_128B, four boxes per 64-feature tile.  The hardware swizzle (16-byte unit index
//     XOR row mod 8) makes the consumers' fragment reads bank-conflict free at the dense pitch, rows past n
//     and features past d arrive as zeros, and one instruction moves 8 KiB (per-row bulk copies are
//     issue-bound, see moments.cu);
//   * warp roles as in gram64_kernel: 1 producer warp + 8 consumer warps (setmaxnreg 40 / 232), 3-stage ring;
//   * S0, sum w y, X^T w, X^T (w y) ride along in the diagonal units;
//   * deterministic: per-unit partials, fixed-order sum over the row chunks in the finalize kernel.
// FP64-pipe bound: (nb(nb-1)/2 * 64 + nb * 36) DMMA per 4 rows; d = 512: 2080 DMMA -> 7.5 ms per 2^20 rows.
#include <cuda.h>
#include <math.h>

#include "tma.cuh"

namespace {

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled_fn() {
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

constexpr int kB = 64;                    // feature block edge
constexpr int kRows = 64;                 // rows per tile
constexpr int kBoxBytes = kRows * 128;    // one TMA box: 64 rows x 16 doubles
constexpr int kTileBytes = 4 * kBoxBytes; // 64 rows x 64 features
constexpr int kGStages = 3;
constexpr int kGConsumers = 8;
constexpr int kGThreads = 384;
constexpr int kGStageBytes = 2 * kTileBytes + 2 * kRows * 8;           // tile(bi), tile(bj), w, y = 66560 = 65 KiB
constexpr int kGSmem = kGStages * kGStageBytes + 2 * kGStages * 8 + 64 + 1024;   // + alignment slack
constexpr int kUnitStride = 2 + 2 * kB + kB * kB;                      // S0, Swy, S1, Sy, 64 tiles x 64

__host__ __device__ __forceinline__ int feat_of64(int block, int r) {
  const int c = (r >> 1) | ((r & 1) << 2);
  return 16 * (block >> 1) + 2 * c + (block & 1);
}

__device__ __forceinline__ void tma_load_2d(void* dst_smem, const CUtensorMap* tmap, int x, int y, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
          smem_u32(dst_smem)),
      "l"(tmap), "r"(x), "r"(y), "r"(smem_u32(bar))
      : "memory");
}

struct GramTmaParams {
  const double* y;
  const double* w;
  const double* center;   // optional: x_i - center
  int64_t n;
  int d;
  int power;
  int nb;
  int npairs;
  int64_t rows_per_chunk;   // multiple of kRows
  double* partials;         // [units][kUnitStride]
};

// Fragment of one 64-feature tile for lane (g, t) and row r: the 16-byte units c(g) + 8 J, J = 0..3.
__device__ __forceinline__ void load_frag(const unsigned char* tile, int r, int cidx, double (&x)[8]) {
  const unsigned char* base = tile + r * 128 + ((cidx ^ (r & 7)) << 4);
#pragma unroll
  for (int J = 0; J < 4; ++J) {
    const double2 v = *reinterpret_cast<const double2*>(base + J * kBoxBytes);
    x[2 * J] = v.x;
    x[2 * J + 1] = v.y;
  }
}

// ---- diagonal unit (bi == bj): 36 upper-triangular tiles per warp, every warp takes 2 of the 16 k-groups of
// a tile; S0, Swy, S1, Sy ride along -----------------------------------------------------------------
template <bool HAS_Y, bool CENTERED>
__device__ __forceinline__ void consume_diag(const GramTmaParams& p, unsigned char* ring, uint64_t* full_bar,
                                             uint64_t* empty_bar, int64_t ntiles, double* smG, double* out, int bi) {
  constexpr int NT = 36;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int cidx = (g >> 1) | ((g & 1) << 2);
  double acc[2 * NT];
  double s1[8], sy[8];
  double s0 = 0.0, swy = 0.0;
  double ca[8];
#pragma unroll
  for (int i = 0; i < 2 * NT; ++i) acc[i] = 0.0;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    s1[i] = 0.0;
    sy[i] = 0.0;
    const int f = bi * kB + feat_of64(i, g);
    ca[i] = (CENTERED && f < p.d) ? p.center[f] : 0.0;
  }
  int stage = 0;
  uint32_t phase = 0;
  for (int64_t tile = 0; tile < ntiles; ++tile) {
    mbar_wait(&full_bar[stage], phase);
    const unsigned char* sA = ring + size_t(stage) * kGStageBytes;
    const double* sW = reinterpret_cast<const double*>(sA + 2 * kTileBytes);
    const double* sY = sW + kRows;
#pragma unroll
    for (int kk = 0; kk < kRows / (4 * kGConsumers); ++kk) {
      const int r = (warp + kGConsumers * kk) * 4 + t;
      double xa[8];
      load_frag(sA, r, cidx, xa);
      if (CENTERED) {
#pragma unroll
        for (int j = 0; j < 8; ++j) xa[j] -= ca[j];
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
        s1[j] = fma(w1, xa[j], s1[j]);
        if (HAS_Y) sy[j] = fma(wy, xa[j], sy[j]);
      }
      double a[8];
#pragma unroll
      for (int I = 0; I < 8; ++I) a[I] = we * xa[I];
      int idx = 0;
#pragma unroll
      for (int I = 0; I < 8; ++I) {
#pragma unroll
        for (int J = I; J < 8; ++J) {
          dmma884(acc[2 * idx], acc[2 * idx + 1], a[I], xa[J]);
          ++idx;
        }
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty_bar[stage]);
    if (++stage == kGStages) {
      stage = 0;
      phase ^= 1u;
    }
  }
  // ---- cross-warp sum through shared memory (8 warps x 36 tiles x 512 B = 144 KiB), fixed warp order ----
  asm volatile("bar.sync 1, %0;" ::"n"(kGConsumers * 32) : "memory");   // the ring is free now
#pragma unroll
  for (int idx = 0; idx < NT; ++idx)
    *reinterpret_cast<double2*>(smG + (warp * NT + idx) * 64 + g * 8 + 2 * t) = make_double2(acc[2 * idx], acc[2 * idx + 1]);
  double* smV = smG + kGConsumers * NT * 64;   // [8][64] S1, [8][64] Sy, [8][2]
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    double v = s1[j];
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    double u = sy[j];
    u += __shfl_xor_sync(0xffffffffu, u, 1);
    u += __shfl_xor_sync(0xffffffffu, u, 2);
    if (t == 0) {
      smV[warp * 64 + feat_of64(j, g)] = v;
      smV[kGConsumers * 64 + warp * 64 + feat_of64(j, g)] = u;
    }
  }
  const double t0 = warp_sum(s0), t1 = warp_sum(swy);
  if (lane == 0) {
    smV[2 * kGConsumers * 64 + 2 * warp] = t0;
    smV[2 * kGConsumers * 64 + 2 * warp + 1] = t1;
  }
  asm volatile("bar.sync 1, %0;" ::"n"(kGConsumers * 32) : "memory");
  for (int e = threadIdx.x; e < NT * 64; e += kGConsumers * 32) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < kGConsumers; ++w) s += smG[w * NT * 64 + e];
    out[2 + 2 * kB + e] = s;
  }
  if (threadIdx.x < 2 * kB) {
    const int which = threadIdx.x >> 6, f = threadIdx.x & 63;
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < kGConsumers; ++w) s += smV[which * kGConsumers * 64 + w * 64 + f];
    out[2 + which * kB + f] = s;
  } else if (threadIdx.x < 2 * kB + 2) {
    const int which = threadIdx.x - 2 * kB;
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < kGConsumers; ++w) s += smV[2 * kGConsumers * 64 + 2 * w + which];
    out[which] = s;
  }
}

// ---- off-diagonal unit (bi < bj): all 64 tiles.  Warps 0-3 own the tile rows I = 0..3, warps 4-7 the rows
// I = 4..7 (32 tiles = 64 accumulator registers per lane); each warp takes 4 of the 16 k-groups of a tile. ----
template <bool CENTERED>
__device__ __forceinline__ void consume_offdiag(const GramTmaParams& p, unsigned char* ring, uint64_t* full_bar,
                                                uint64_t* empty_bar, int64_t ntiles, double* smG, double* out, int bi,
                                                int bj) {
  constexpr int NT = 32;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int cidx = (g >> 1) | ((g & 1) << 2);
  const int ih = warp >> 2, wq = warp & 3;
  double acc[2 * NT];
#pragma unroll
  for (int i = 0; i < 2 * NT; ++i) acc[i] = 0.0;
  double cbv[8], cav[4];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int f = bj * kB + feat_of64(j, g);
    cbv[j] = (CENTERED && f < p.d) ? p.center[f] : 0.0;
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int f = bi * kB + feat_of64(4 * ih + i, g);
    cav[i] = (CENTERED && f < p.d) ? p.center[f] : 0.0;
  }
  int stage = 0;
  uint32_t phase = 0;
  for (int64_t tile = 0; tile < ntiles; ++tile) {
    mbar_wait(&full_bar[stage], phase);
    const unsigned char* sA = ring + size_t(stage) * kGStageBytes;
    const unsigned char* sB = sA + kTileBytes;
    const double* sW = reinterpret_cast<const double*>(sA + 2 * kTileBytes);
#pragma unroll 2
    for (int kk = 0; kk < 4; ++kk) {
      const int r = (wq + 4 * kk) * 4 + t;
      double xb[8];
      load_frag(sB, r, cidx, xb);
      // A side: only the blocks I = 4 ih .. 4 ih + 3, i.e. the 16-byte units c(g) + 8 J for J = 2 ih, 2 ih + 1
      const unsigned char* abase = sA + r * 128 + ((cidx ^ (r & 7)) << 4) + (2 * ih) * kBoxBytes;
      const double2 v0 = *reinterpret_cast<const double2*>(abase);
      const double2 v1 = *reinterpret_cast<const double2*>(abase + kBoxBytes);
      const double w1 = sW[r];
      const double we = (p.power == 2) ? w1 * w1 : w1;
      if (CENTERED) {
#pragma unroll
        for (int j = 0; j < 8; ++j) xb[j] -= cbv[j];
      }
      const double a[4] = {we * (v0.x - cav[0]), we * (v0.y - cav[1]), we * (v1.x - cav[2]), we * (v1.y - cav[3])};
#pragma unroll
      for (int I = 0; I < 4; ++I) {
#pragma unroll
        for (int J = 0; J < 8; ++J) dmma884(acc[2 * (I * 8 + J)], acc[2 * (I * 8 + J) + 1], a[I], xb[J]);
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty_bar[stage]);
    if (++stage == kGStages) {
      stage = 0;
      phase ^= 1u;
    }
  }
  asm volatile("bar.sync 1, %0;" ::"n"(kGConsumers * 32) : "memory");   // the ring is free now
#pragma unroll
  for (int idx = 0; idx < NT; ++idx)
    *reinterpret_cast<double2*>(smG + (warp * NT + idx) * 64 + g * 8 + 2 * t) = make_double2(acc[2 * idx], acc[2 * idx + 1]);
  asm volatile("bar.sync 1, %0;" ::"n"(kGConsumers * 32) : "memory");
  // output tile index = 32 ih + local; sum over the four warps of that half in warp order
  for (int e = threadIdx.x; e < 64 * 64; e += kGConsumers * 32) {
    const int half = e / (NT * 64), local = e - half * (NT * 64);
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < 4; ++w) s += smG[((half * 4 + w) * NT) * 64 + local];
    out[2 + 2 * kB + e] = s;
  }
}

template <bool HAS_Y, bool CENTERED>
__global__ void __launch_bounds__(kGThreads, 1) gram_tma_kernel(const __grid_constant__ CUtensorMap tmap,
                                                                const GramTmaParams p) {
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* ring = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(ring + kGStages * kGStageBytes);
  uint64_t* empty_bar = full_bar + kGStages;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // unit -> (chunk, pair) -> (bi, bj)
  const int unit = blockIdx.x;
  const int chunk = unit / p.npairs;
  int rem = unit - chunk * p.npairs, bi = 0;
  while (rem >= p.nb - bi) {
    rem -= p.nb - bi;
    ++bi;
  }
  const int bj = bi + rem;
  const int64_t r_begin = int64_t(chunk) * p.rows_per_chunk;
  const int64_t r_end = (r_begin + p.rows_per_chunk < p.n) ? r_begin + p.rows_per_chunk : p.n;
  const int64_t ntiles = (r_end - r_begin + kRows - 1) / kRows;
  const bool diag = (bi == bj);

  if (threadIdx.x == 0) {
    for (int s = 0; s < kGStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], kGConsumers);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap) : "memory");
  }
  __syncthreads();

  if (warp >= kGConsumers) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    if (warp == kGConsumers) {
      int stage = 0;
      uint32_t phase = 0;
      for (int64_t tile = 0; tile < ntiles; ++tile) {
        mbar_wait(&empty_bar[stage], phase ^ 1u);
        unsigned char* sA = ring + size_t(stage) * kGStageBytes;
        unsigned char* sB = sA + kTileBytes;
        double* sW = reinterpret_cast<double*>(sA + 2 * kTileBytes);
        double* sY = sW + kRows;
        const int64_t row0 = r_begin + tile * kRows;
        const bool full_rows = (row0 + kRows <= p.n);
        if (!full_rows) {   // ragged tail: w / y by plain loads with zero fill (X rows past n arrive as zeros)
          for (int r = lane; r < kRows; r += 32) {
            sW[r] = (row0 + r < p.n) ? p.w[row0 + r] : 0.0;
            sY[r] = (HAS_Y && diag && row0 + r < p.n) ? p.y[row0 + r] : 0.0;
          }
          __syncwarp();
        }
        if (lane == 0) {
          uint32_t bytes = uint32_t(kTileBytes) * (diag ? 1u : 2u);
          if (full_rows) bytes += 512u + ((HAS_Y && diag) ? 512u : 0u);
          mbar_arrive_expect_tx(&full_bar[stage], bytes);
#pragma unroll
          for (int q = 0; q < 4; ++q) tma_load_2d(sA + q * kBoxBytes, &tmap, bi * kB + 16 * q, int(row0), &full_bar[stage]);
          if (!diag) {
#pragma unroll
            for (int q = 0; q < 4; ++q)
              tma_load_2d(sB + q * kBoxBytes, &tmap, bj * kB + 16 * q, int(row0), &full_bar[stage]);
          }
          if (full_rows) {
            bulk_g2s(sW, p.w + row0, 512, &full_bar[stage]);
            if (HAS_Y && diag) bulk_g2s(sY, p.y + row0, 512, &full_bar[stage]);
          }
        }
        if (++stage == kGStages) {
          stage = 0;
          phase ^= 1u;
        }
      }
    }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 232;");
    double* out = p.partials + size_t(unit) * kUnitStride;
    double* smG = reinterpret_cast<double*>(ring);
    if (diag)
      consume_diag<HAS_Y, CENTERED>(p, ring, full_bar, empty_bar, ntiles, smG, out, bi);
    else
      consume_offdiag<CENTERED>(p, ring, full_bar, empty_bar, ntiles, smG, out, bi, bj);
  }
}

// Sum the per-unit partials over the row chunks (chunk order) and scatter to the public layout.
__global__ void gram_tma_finalize_kernel(const double* __restrict__ partials, int nchunks, int nb, int npairs, int d,
                                         int want_gram, double* __restrict__ out) {
  const int64_t e = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t per_pair = kUnitStride;
  if (e >= int64_t(npairs) * per_pair) return;
  const int pair = int(e / per_pair), within = int(e % per_pair);
  int bi = 0, rem = pair;
  while (rem >= nb - bi) {
    rem -= nb - bi;
    ++bi;
  }
  const int bj = bi + rem;
  const bool diag = (bi == bj);
  if (within < 2 + 2 * kB && !diag) return;
  if (within >= 2 + 2 * kB && !want_gram) return;
  double s = 0.0;
  for (int c = 0; c < nchunks; ++c) s += partials[(size_t(c) * npairs + pair) * kUnitStride + within];
  if (within < 2) {
    if (bi == 0) out[within] = s;       // S0 / Swy: identical in every diagonal unit set, take block 0's
    return;
  }
  if (within < 2 + 2 * kB) {
    const int which = (within - 2) / kB, f = bi * kB + (within - 2) % kB;
    if (f < d) out[2 + which * d + f] = s;
    return;
  }
  const int ce = within - (2 + 2 * kB);
  const int tile = ce >> 6, r = (ce >> 3) & 7, c = ce & 7;
  int I, J;
  if (diag) {
    if (tile >= 36) return;
    I = 0;
    int tr = tile;
    while (tr >= 8 - I) {
      tr -= 8 - I;
      ++I;
    }
    J = I + tr;
  } else {
    I = tile >> 3;
    J = tile & 7;
  }
  const int fi = bi * kB + feat_of64(I, r), fj = bj * kB + feat_of64(J, c);
  if (fi >= d || fj >= d) return;
  if (diag && I == J && fi > fj) return;   // one triangle of the diagonal tiles, mirrored below
  double* G = out + 2 + 2 * d;
  G[size_t(fi) * d + fj] = s;
  G[size_t(fj) * d + fi] = s;
}

}  // namespace

// Returns RLVI_OK, or RLVI_ERR_UNSUPPORTED when this path does not apply (caller falls back).
int rlvi_gram_tma_f64(rlvi_ctx* ctx, const double* X, const double* y, const double* weights, const double* center,
                      int64_t n, int d, int power, int want_gram, double* out, cudaStream_t st) {
  EncodeTiledFn encode = encode_tiled_fn();
  if (!encode || d % 2 != 0 || d < 16 || d > 2048 || n < kRows || n >= (int64_t(1) << 31) || !rlvi_aligned16(X) ||
      !rlvi_aligned16(weights) || (y && !rlvi_aligned16(y)))
    return RLVI_ERR_UNSUPPORTED;
  CUtensorMap tmap;
  const cuuint64_t gdim[2] = {cuuint64_t(d), cuuint64_t(n)};
  const cuuint64_t gstride[1] = {cuuint64_t(d) * 8};
  const cuuint32_t box[2] = {16, cuuint32_t(kRows)};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult cr = encode(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double*>(X), gdim, gstride, box, estr,
                             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (cr != CUDA_SUCCESS) {
    rlvi_set_error("cuTensorMapEncodeTiled failed (%d)", int(cr));
    return RLVI_ERR_UNSUPPORTED;
  }
  GramTmaParams p;
  p.y = y;
  p.w = weights;
  p.center = center;
  p.n = n;
  p.d = d;
  p.power = power;
  p.nb = (d + kB - 1) / kB;
  p.npairs = p.nb * (p.nb + 1) / 2;
  int64_t nchunks = (int64_t(ctx->sm_count) * 4 + p.npairs - 1) / p.npairs;
  const int64_t max_chunks = (n + kRows - 1) / kRows;
  if (nchunks > max_chunks) nchunks = max_chunks;
  if (nchunks < 1) nchunks = 1;
  p.rows_per_chunk = ((n + nchunks - 1) / nchunks + kRows - 1) / kRows * kRows;
  nchunks = (n + p.rows_per_chunk - 1) / p.rows_per_chunk;
  const int64_t units = nchunks * p.npairs;
  RlviScratch s;
  const int rc = rlvi_scratch_header(ctx, size_t(units) * kUnitStride * sizeof(double), &s);
  if (rc != RLVI_OK) return rc;
  p.partials = s.partials;
#define RLVI_GRAM_TMA_LAUNCH(HY, CE)                                                                          \
  {                                                                                                           \
    RLVI_CUDA(cudaFuncSetAttribute(gram_tma_kernel<HY, CE>, cudaFuncAttributeMaxDynamicSharedMemorySize, kGSmem)); \
    gram_tma_kernel<HY, CE><<<int(units), kGThreads, kGSmem, st>>>(tmap, p);                                  \
  }
  if (y && center) RLVI_GRAM_TMA_LAUNCH(true, true)
  else if (y) RLVI_GRAM_TMA_LAUNCH(true, false)
  else if (center) RLVI_GRAM_TMA_LAUNCH(false, true)
  else RLVI_GRAM_TMA_LAUNCH(false, false)
#undef RLVI_GRAM_TMA_LAUNCH
  RLVI_LAUNCH_CHECK(ctx);
  const int64_t total = int64_t(p.npairs) * kUnitStride;
  gram_tma_finalize_kernel<<<int((total + 255) / 256), 256, 0, st>>>(p.partials, int(nchunks), p.nb, p.npairs, d,
                                                                     want_gram, out);
  RLVI_LAUNCH_CHECK(ctx);
  return RLVI_OK;
}
