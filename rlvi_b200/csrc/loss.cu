// loss.cu -- per-sample negative log-likelihoods: ONE streaming pass over X (HBM-bound).
//
// Replaces the NumPy expressions of
//   standard-learning/utils.py:19-21   cross_entropy            (RLVI_LOSS_LOGISTIC_CE)
//   standard-learning/utils.py:62-64   sklearn_log_reg's loss   (RLVI_LOSS_SOFTPLUS)
//   standard-learning/rlvi.py:72,81    (y - X theta)^2          (RLVI_LOSS_SQRES)
//   standard-learning/rlvi.py:49,57    ||theta - x||^2          (RLVI_LOSS_SQDIST)
//   standard-learning/utils.py:77-79   PCA reconstruction       (RLVI_LOSS_PCA)
//   standard-learning/utils.py:93-101  Gaussian NLL             (RLVI_LOSS_GAUSSIAN, DMMA kernel below)
// and fuses e_i = exp(-l_i) (the fixed point's input) and the pi-weighted loss sum
// (sigma2 = pi.r2 / sum pi, rlvi.py:50,58,73,82) into the same pass.
//
// Algorithmic bytes per sample: d*8 (X) + 8 (y) + 8 (pi, optional) + 8 (l) + 8 (e).
#include <math.h>

#include "rowmap.cuh"
#include "tma_ring.cuh"

namespace {

constexpr int kLossThreads = 256;

// What every loss kernel writes: l, exp(-l), and with weights the grid totals (sum w l, sum w) into wsum_out.
struct LossOut {
  const double* w;
  double* losses;
  double* e_out;
  double* wsum_out;
  double* partials;       // [grid][2]
  unsigned int* ticket;
};

// One row's outputs; wi is only read when o.w is set.
__device__ __forceinline__ void loss_row(const LossOut& o, int64_t row, double loss, double wi, double& s_wl,
                                         double& s_w) {
  if (o.losses) o.losses[row] = loss;
  if (o.e_out) o.e_out[row] = exp(-loss);
  if (o.w) {
    s_wl = fma(wi, loss, s_wl);
    s_w += wi;
  }
}

// End of a loss kernel: block then grid totals of (sum w l, sum w).  `red` holds 2 * nwarps doubles.
__device__ __forceinline__ void loss_sums(const LossOut& o, double s_wl, double s_w, double* red) {
  if (!o.w) return;   // uniform across the grid
  double v[2] = {s_wl, s_w};
  block_sum<2>(v, red);
  if (grid_total<2>(v, o.partials, o.ticket)) {
    o.wsum_out[0] = v[0];
    o.wsum_out[1] = v[1];
  }
}

struct LossParams {
  const double* X;
  const double* y;
  const double* params;
  LossOut o;
  int64_t n;
  int d;
  int kind;
  int intercept;
  int L;
};

// a = x.theta (or ||theta - x||^2 for SQDIST), b = x.x (PCA only), b0 = intercept, yi = label / target.
__device__ __forceinline__ double finish_loss(int kind, double a, double b, double b0, double yi) {
  switch (kind) {
    case RLVI_LOSS_LOGISTIC_CE: {
      const double phi = b0 + a;
      return (-yi * phi + phi) + log1p(exp(-phi));          // utils.py:21, same operation order
    }
    case RLVI_LOSS_SOFTPLUS: {
      const double phi = b0 + a;
      return fmax(phi, 0.0) + log1p(exp(-fabs(phi)));        // logaddexp(0, phi)
    }
    case RLVI_LOSS_SQRES: {
      const double r = yi - (b0 + a);
      return r * r;
    }
    case RLVI_LOSS_SQDIST: {
      const double r = sqrt(a);                              // np.linalg.norm(...)**2
      return r * r;
    }
    default:                                                 // RLVI_LOSS_PCA
      return b - a * a;
  }
}

// DOTK 0: a = x.theta          (LOGISTIC_CE, SOFTPLUS, SQRES)
// DOTK 1: a = x.theta, b = x.x (PCA)
// DOTK 2: a = ||theta - x||^2  (SQDIST)
template <int DOTK, int FPL, bool VEC>
__global__ void __launch_bounds__(kLossThreads) loss_kernel(const LossParams p) {
  extern __shared__ double sm[];
  double* sm_params = sm;                    // d + 1
  double* sm_red = sm + (p.d + 2);           // 2 * nwarps
  const int np = p.d + (p.intercept ? 1 : 0);
  for (int i = threadIdx.x; i < np; i += blockDim.x) sm_params[i] = p.params[i];
  __syncthreads();

  const int lane = threadIdx.x & 31;
  const int L = p.L;
  const int q = lane & (L - 1);
  const int sub = lane / L;
  const int R = 32 / L;
  const double b0 = p.intercept ? sm_params[0] : 0.0;
  double th[FPL];
  RowMap<FPL, VEC>::load_vec(sm_params + (p.intercept ? 1 : 0), p.d, q, L, th);

  const int64_t warps_total = int64_t(gridDim.x) * (blockDim.x >> 5);
  const int64_t warp_id = int64_t(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  double s_wl = 0.0, s_w = 0.0;

  for (int64_t row0 = warp_id * R; row0 < p.n; row0 += warps_total * R) {
    const int64_t row = row0 + sub;
    const bool valid = row < p.n;
    double x[FPL];
    RowMap<FPL, VEC>::load_row(p.X, row, p.d, q, L, valid, x);
    double a = 0.0, b = 0.0;
#pragma unroll
    for (int k = 0; k < FPL; ++k) {
      if (DOTK == 2) {
        const double t = th[k] - x[k];
        a = fma(t, t, a);
      } else {
        a = fma(x[k], th[k], a);
        if (DOTK == 1) b = fma(x[k], x[k], b);
      }
    }
    a = group_sum(a, L);
    if (DOTK == 1) b = group_sum(b, L);
    if (q == 0 && valid) {
      const double loss = finish_loss(p.kind, a, b, b0, (p.kind == RLVI_LOSS_LOGISTIC_CE || p.kind == RLVI_LOSS_SQRES) ? p.y[row] : 0.0);
      loss_row(p.o, row, loss, p.o.w ? p.o.w[row] : 0.0, s_wl, s_w);
    }
  }
  loss_sums(p.o, s_wl, s_w, sm_red);
}

// ---------------------------------------------------------------------------------------------
// TMA-fed streaming kernel (d % 16 == 0, d <= 256, 16-byte aligned pointers): the headline path.
// Producer / private-ring skeleton: tma_ring.cuh.  Consumer: lane l owns row l of its warp's 32-row tile and
// does the whole d-long dot product itself.  Rows sit at their natural d*8-byte pitch (a multiple of 128
// bytes), so lane l walks its row ROTATED by l 16-byte units -- unit (j + l) mod (d/2) at step j -- which
// makes every 128-bit shared-memory read of x and of theta bank-conflict free; the exp / log1p tail then runs
// with ALL 32 lanes busy (the register-tiled kernel above leaves 3/4 of the lanes idle there and exposes the
// global-load latency once per row group); outputs are one coalesced 256-byte store per warp and array.
// Algorithmic bytes per sample: d*8 (X) + 8 (y) [+ 8 (pi)] in, 8 (l) and/or 8 (e) out.
// ---------------------------------------------------------------------------------------------
struct LossTmaParams {
  const double* X;
  const double* y;
  const double* params;
  LossOut o;
  int64_t n;
  int d;
  int kind;
  int intercept;
  RingGeom geom;
};

// shared-memory tail after the ring: theta (d doubles, padded), the barriers, the block-reduction scratch
static inline size_t loss_tma_tail(int d) {
  return size_t(((d + 1) & ~1) + 2) * 8 + kRingBarrierBytes + 2 * (kRingConsumers + 1) * 8 + 128;
}

template <int DOTK>
__global__ void __launch_bounds__(kRingThreads, 1) loss_tma_kernel(const LossTmaParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int d = p.d;
  Ring ring;
  ring.base = smem_raw;
  ring.g = p.geom;
  ring.d = d;
  double* sTheta = reinterpret_cast<double*>(smem_raw + ring_bytes(p.geom));         // d (+ pad to even)
  ring.full_bar = reinterpret_cast<uint64_t*>(sTheta + ((d + 1) & ~1) + 2);
  ring.empty_bar = ring.full_bar + kRingMaxStages;
  double* sRed = reinterpret_cast<double*>(ring.empty_bar + kRingMaxStages);          // 2 * 17 doubles
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < d; i += blockDim.x) sTheta[i] = p.params[i + (p.intercept ? 1 : 0)];
  ring_init(ring);
  const double b0 = p.intercept ? p.params[0] : 0.0;
  const int64_t my_tiles = ring_my_tiles(p.n);
  const bool need_y = (p.kind == RLVI_LOSS_LOGISTIC_CE || p.kind == RLVI_LOSS_SQRES);
  double s_wl = 0.0, s_w = 0.0;

  if (warp == kRingConsumers) {
    ring_produce(ring, p.X, need_y ? p.y : nullptr, p.o.w, p.n, my_tiles, false);
  } else if (warp < p.geom.ncons) {
    const double2* th2 = reinterpret_cast<const double2*>(sTheta);
    const int npair = d >> 1;                      // 16-byte units per row, a multiple of 8
    for (int64_t t = warp; t < my_tiles; t += p.geom.ncons) {
      const RingStage st = ring_acquire(ring, warp, t);
      const double2* xr = reinterpret_cast<const double2*>(st.x) + size_t(lane) * npair;
      double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0, q0 = 0.0, q1 = 0.0;
      int u = lane % npair;                         // rotated walk: conflict-free at the natural pitch
#pragma unroll 4
      for (int j = 0; j < npair; j += 2) {
        int u1 = u + 1;
        if (u1 == npair) u1 = 0;
        const double2 x0 = xr[u], x1 = xr[u1];
        const double2 t0 = th2[u], t1 = th2[u1];
        u = u1 + 1;
        if (u == npair) u = 0;
        if (DOTK == 2) {
          const double v0 = t0.x - x0.x, v1 = t0.y - x0.y, v2 = t1.x - x1.x, v3 = t1.y - x1.y;
          a0 = fma(v0, v0, a0);
          a1 = fma(v1, v1, a1);
          a2 = fma(v2, v2, a2);
          a3 = fma(v3, v3, a3);
        } else {
          a0 = fma(x0.x, t0.x, a0);
          a1 = fma(x0.y, t0.y, a1);
          a2 = fma(x1.x, t1.x, a2);
          a3 = fma(x1.y, t1.y, a3);
          if (DOTK == 1) {
            q0 = fma(x0.x, x0.x, q0);
            q1 = fma(x0.y, x0.y, q1);
            q0 = fma(x1.x, x1.x, q0);
            q1 = fma(x1.y, x1.y, q1);
          }
        }
      }
      const double a = (a0 + a1) + (a2 + a3);
      const double b = q0 + q1;
      const double yi = st.y[lane];
      const double wi = st.w[lane];
      ring_release(ring, st);                        // the stage can be refilled while we do the tail
      const int64_t row = ring_row0(t) + lane;
      if (row < p.n) loss_row(p.o, row, finish_loss(p.kind, a, b, b0, need_y ? yi : 0.0), wi, s_wl, s_w);
    }
  }
  loss_sums(p.o, s_wl, s_w, sRed);
}

// ---------------------------------------------------------------------------------------------
// Gaussian NLL through the FP64 tensor pipe.
//   l_i = 0.5 (||U (x_i - mu)||^2 + c),  U upper triangular with U^T U = cov^-1.
// A warp takes 8 rows per step.  Z = C U^T is accumulated with mma.sync.m8n8k4.f64 (SASS DMMA.8x8x4):
// A fragment = centred samples (row g, feature pair of lane t), B fragment = U rows from shared memory
// (pitch d+8 doubles: conflict-free 128-bit reads), only the block-upper-triangular part is visited:
// nb(nb+1) DMMAs per 8 rows, nb = ceil(d/8).  The k-slots of one DMMA pair are the two halves of one
// 128-bit load, i.e. features (8kk+2t, 8kk+2t+1); the same permutation is applied to U's columns, so
// the contraction is unchanged.
// ---------------------------------------------------------------------------------------------
struct GaussParams {
  const double* X;
  const double* params;   // [c, mu(d), U(d*d) row-major upper triangular]
  LossOut o;
  int64_t n;
  int d;
};

template <int NB_MAX, bool VEC>
__global__ void __launch_bounds__(kLossThreads) gaussian_loss_kernel(const GaussParams p) {
  extern __shared__ __align__(16) double smg[];
  const int d = p.d;
  const int nb = (d + 7) >> 3;
  const int dp = nb * 8;
  const int pitch = dp + 8;
  double* sU = smg;                       // dp * pitch
  double* sMu = sU + size_t(dp) * pitch;  // dp
  double* sRed = sMu + dp;                // 2 * nwarps
  for (int i = threadIdx.x; i < dp * pitch; i += blockDim.x) {
    const int r = i / pitch, c = i - r * pitch;
    sU[i] = (r < d && c < d && c >= r) ? p.params[1 + d + size_t(r) * d + c] : 0.0;
  }
  for (int i = threadIdx.x; i < dp; i += blockDim.x) sMu[i] = (i < d) ? p.params[1 + i] : 0.0;
  __syncthreads();
  const double cst = p.params[0];

  const int lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int64_t warps_total = int64_t(gridDim.x) * (blockDim.x >> 5);
  const int64_t warp_id = int64_t(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  double s_wl = 0.0, s_w = 0.0;

  for (int64_t row0 = warp_id * 8; row0 < p.n; row0 += warps_total * 8) {
    const int64_t row = row0 + g;
    const bool valid = row < p.n;
    double2 c[NB_MAX];
#pragma unroll
    for (int kk = 0; kk < NB_MAX; ++kk) {
      const int f = 8 * kk + 2 * t;
      double2 v = make_double2(0.0, 0.0);
      if (kk < nb && valid) {
        const double* src = p.X + row * int64_t(d) + f;
        if (VEC) {
          if (f < d) v = ld_stream_d2(src);
        } else {
          if (f < d) v.x = ld_stream_d1(src);
          if (f + 1 < d) v.y = ld_stream_d1(src + 1);
        }
        const double2 m = *reinterpret_cast<const double2*>(sMu + f);
        v.x -= m.x;
        v.y -= m.y;
        if (f >= d) v.x = 0.0;
        if (f + 1 >= d) v.y = 0.0;
      }
      c[kk] = v;
    }
    double quad = 0.0;
#pragma unroll
    for (int nbk = 0; nbk < NB_MAX; ++nbk) {
      if (nbk < nb) {
        double z0 = 0.0, z1 = 0.0;
        const double* urow = sU + size_t(8 * nbk + g) * pitch + 2 * t;
#pragma unroll
        for (int kk = nbk; kk < NB_MAX; ++kk) {
          if (kk < nb) {
            const double2 u = *reinterpret_cast<const double2*>(urow + 8 * kk);
            dmma884(z0, z1, c[kk].x, u.x);
            dmma884(z0, z1, c[kk].y, u.y);
          }
        }
        quad = fma(z0, z0, quad);
        quad = fma(z1, z1, quad);
      }
    }
    quad += __shfl_xor_sync(0xffffffffu, quad, 1);
    quad += __shfl_xor_sync(0xffffffffu, quad, 2);
    if (t == 0 && valid) {
      const double loss = 0.5 * (quad + cst);                    // utils.py:101
      loss_row(p.o, row, loss, p.o.w ? p.o.w[row] : 0.0, s_wl, s_w);
    }
  }
  loss_sums(p.o, s_wl, s_w, sRed);
}

// ---------------------------------------------------------------------------------------------
// TMA-fed Gaussian NLL (d % 16 == 0, d <= 64, aligned): same producer / private-ring skeleton as
// loss_tma_kernel; a consumer warp walks its 32-row tile as four 8-row DMMA groups, gathers the four groups'
// quadratic forms so that lane l ends with row l (one shuffle per group), and then runs the exp tail and the
// 256-byte stores with all 32 lanes.  (gaussian_loss_kernel above fetches its fragments straight from global
// memory: latency-bound at 47 % of the DMMA peak.)
// ---------------------------------------------------------------------------------------------
struct GaussTmaParams {
  const double* X;
  const double* params;   // [c, mu(d), U(d*d) row-major upper triangular]
  LossOut o;
  int64_t n;
  int d;
  RingGeom geom;
};

static inline size_t gauss_tma_tail(int d) {
  return (size_t(d) * (d + 8) + d) * 8 + kRingBarrierBytes + 2 * (kRingConsumers + 1) * 8 + 128;
}

template <int NB>   // NB = d / 8 MMA blocks (exact)
__global__ void __launch_bounds__(kRingThreads, 1) gaussian_tma_kernel(const GaussTmaParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr int D = NB * 8;
  constexpr int kPitchU = D + 8;                 // doubles: conflict-free 128-bit reads of U rows
  Ring ring;
  ring.base = smem_raw;
  ring.g = p.geom;
  ring.d = D;
  double* sU = reinterpret_cast<double*>(smem_raw + ring_bytes(p.geom));       // D * kPitchU
  double* sMu = sU + D * kPitchU;                                               // D
  ring.full_bar = reinterpret_cast<uint64_t*>(sMu + D);
  ring.empty_bar = ring.full_bar + kRingMaxStages;
  double* sRed = reinterpret_cast<double*>(ring.empty_bar + kRingMaxStages);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < D * kPitchU; i += blockDim.x) {
    const int r = i / kPitchU, c = i - r * kPitchU;
    sU[i] = (c < D && c >= r) ? p.params[1 + D + size_t(r) * D + c] : 0.0;
  }
  for (int i = threadIdx.x; i < D; i += blockDim.x) sMu[i] = p.params[1 + i];
  ring_init(ring);
  const double cst = p.params[0];
  const int64_t my_tiles = ring_my_tiles(p.n);
  double s_wl = 0.0, s_w = 0.0;

  if (warp == kRingConsumers) {
    ring_produce(ring, p.X, nullptr, p.o.w, p.n, my_tiles, false);
  } else if (warp < p.geom.ncons) {
    const int g = lane >> 2, t = lane & 3;
    for (int64_t tl = warp; tl < my_tiles; tl += p.geom.ncons) {
      const RingStage st = ring_acquire(ring, warp, tl);
      double myquad = 0.0;
#pragma unroll 1
      for (int grp = 0; grp < 4; ++grp) {
        // centred fragment of row 8 grp + g: features (8 kk + 2 t, + 1)
        const double2* xrow = reinterpret_cast<const double2*>(st.x + size_t(8 * grp + g) * D * 8);
        double2 c[NB];
#pragma unroll
        for (int kk = 0; kk < NB; ++kk) {
          double2 v = xrow[4 * kk + t];
          const double2 m = *reinterpret_cast<const double2*>(sMu + 8 * kk + 2 * t);
          v.x -= m.x;
          v.y -= m.y;
          c[kk] = v;
        }
        double quad = 0.0;
#pragma unroll
        for (int nbk = 0; nbk < NB; ++nbk) {
          double z0 = 0.0, z1 = 0.0;
          const double* urow = sU + size_t(8 * nbk + g) * kPitchU + 2 * t;
#pragma unroll
          for (int kk = nbk; kk < NB; ++kk) {
            const double2 u = *reinterpret_cast<const double2*>(urow + 8 * kk);
            dmma884(z0, z1, c[kk].x, u.x);
            dmma884(z0, z1, c[kk].y, u.y);
          }
          quad = fma(z0, z0, quad);
          quad = fma(z1, z1, quad);
        }
        quad += __shfl_xor_sync(0xffffffffu, quad, 1);
        quad += __shfl_xor_sync(0xffffffffu, quad, 2);
        // row 8 grp + g's form sits in lanes 4 g .. 4 g + 3; lane l wants row l
        const double got = __shfl_sync(0xffffffffu, quad, 4 * (lane & 7));
        if ((lane >> 3) == grp) myquad = got;
      }
      const double wi = st.w[lane];
      ring_release(ring, st);
      const int64_t row = ring_row0(tl) + lane;
      if (row < p.n) loss_row(p.o, row, 0.5 * (myquad + cst), wi, s_wl, s_w);   // utils.py:101
    }
  }
  loss_sums(p.o, s_wl, s_w, sRed);
}

template <int DOTK>
int launch_loss(rlvi_ctx* ctx, const RowMapCfg& cfg, LossParams& p, int grid, size_t smem, cudaStream_t st) {
#define RLVI_LOSS_CASE(F, V)                                                            \
  if (cfg.fpl == F && cfg.vec == V) {                                                   \
    loss_kernel<DOTK, F, V><<<grid, kLossThreads, smem, st>>>(p);                       \
    RLVI_LAUNCH_CHECK(ctx);                                                             \
    return RLVI_OK;                                                                     \
  }
  RLVI_LOSS_CASE(4, true)
  RLVI_LOSS_CASE(4, false)
  RLVI_LOSS_CASE(16, true)
  RLVI_LOSS_CASE(16, false)
  RLVI_LOSS_CASE(32, true)
  RLVI_LOSS_CASE(32, false)
#undef RLVI_LOSS_CASE
  rlvi_set_error("no loss kernel for fpl=%d", cfg.fpl);
  return RLVI_ERR_UNSUPPORTED;
}

// The grid's (sum w l, sum w) partials and the ticket, from the scratch header.
int loss_scratch(rlvi_ctx* ctx, int grid, LossOut& o) {
  RlviScratch s;
  const int rc = rlvi_scratch_header(ctx, size_t(grid) * 2 * sizeof(double), &s);
  o.partials = s.partials;
  o.ticket = s.ticket;
  return rc;
}


// ---------------------------------------------------------------------------------------------
// FP32-STORED X (the FP32 mode of SURVEY.md section 8d, config C3): the same losses from float32 samples.
// The per-sample vectors stay FP64 (l, e, pi, y); products and sums are formed in FP64 from the converted
// samples, so the only difference to the FP64 path is the storage rounding of X itself.  One warp per row:
// lane l takes the 16-byte units l, l + 32, ... (coalesced 512-byte requests), theta sits in shared memory.
// HBM-bound: d*4 (X) + 8 (y) [+ 8 (pi)] in, 8 (l) and/or 8 (e) out per sample.
// ---------------------------------------------------------------------------------------------
struct LossF32Params {
  const float* X;
  const double* y;
  const double* params;
  LossOut o;
  int64_t n;
  int d;
  int kind;
  int intercept;
  int vec;                // X 16-byte aligned and d % 4 == 0
};

// float -> double on the integer pipe: F2F.F64.F32 issues at ~4 lanes / clk / SM on B200 (measured: the conversion, not
// HBM, bounded the first version of this kernel at 3.9 TB/s), a shift / add / select sequence at 64.  Exact for normal
// numbers and zero; denormals (|x| < 2^-126) flush to zero; Inf / NaN take the slow path.
__device__ __forceinline__ double f32_to_f64(float f) {
  const uint32_t u = __float_as_uint(f);
  const uint32_t a = u & 0x7FFFFFFFu;
  if (a >= 0x7F800000u) return double(f);
  const uint32_t hi = (a < 0x00800000u) ? 0u : ((a >> 3) + 0x38000000u);   // exponent bias 127 -> 1023
  const uint32_t lo = (a < 0x00800000u) ? 0u : (u << 29);
  return __hiloint2double(int(hi | (u & 0x80000000u)), int(lo));
}

// theta in shared memory for the vector path: lane l of a warp multiplies the four samples 4l .. 4l+3 of every
// 128-feature group, i.e. 32 bytes of theta per lane -- at that stride two 16-byte reads per lane collide four ways
// (ncu: 55 % of the shared-memory wavefronts were conflicts and the kernel sat at 3.9 TB/s).  Stored as two planes
// per group, {theta[4l], theta[4l+1]} for all lanes then {theta[4l+2], theta[4l+3]}, each read is one conflict-free
// 16-byte access per lane.
__device__ __forceinline__ int theta_slot(int e) {
  const int g = e >> 7, r = e & 127, l = r >> 2, k = r & 3;
  return (g << 7) + ((k >> 1) << 6) + (l << 1) + (k & 1);
}

template <int DOTK>
__global__ void __launch_bounds__(kLossThreads) loss_f32_kernel(const LossF32Params p) {
  extern __shared__ double sm[];
  const int dpad = (p.d + 127) & ~127;
  double* th = sm;                                  // theta, dpad doubles (permuted when p.vec), 16-byte aligned
  double* sm_red = sm + dpad + 2;                   // 2 * nwarps
  for (int i = threadIdx.x; i < dpad; i += blockDim.x) th[i] = 0.0;
  __syncthreads();
  for (int i = threadIdx.x; i < p.d; i += blockDim.x) th[p.vec ? theta_slot(i) : i] = p.params[i + (p.intercept ? 1 : 0)];
  __syncthreads();
  const double b0 = p.intercept ? p.params[0] : 0.0;
  const int lane = threadIdx.x & 31;
  const int64_t warps_total = int64_t(gridDim.x) * (blockDim.x >> 5);
  const int64_t warp_id = int64_t(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  double s_wl = 0.0, s_w = 0.0;

  for (int64_t row = warp_id; row < p.n; row += warps_total) {
    const float* xr = p.X + row * p.d;
    double a = 0.0, b = 0.0;
    if (p.vec) {
      for (int j0 = 0; j0 < p.d; j0 += 512) {       // up to 4 independent 16-byte loads in flight per lane
        float4 x[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int j = j0 + u * 128 + lane * 4;
          x[u] = (j < p.d) ? ld_stream_f4(xr + j) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int j = j0 + u * 128 + lane * 4;
          if (j < p.d) {
            const double xv[4] = {f32_to_f64(x[u].x), f32_to_f64(x[u].y), f32_to_f64(x[u].z), f32_to_f64(x[u].w)};
            const double2 t01 = *reinterpret_cast<const double2*>(th + (j0 + u * 128) + lane * 2);
            const double2 t23 = *reinterpret_cast<const double2*>(th + (j0 + u * 128) + 64 + lane * 2);
            const double tv[4] = {t01.x, t01.y, t23.x, t23.y};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              if (DOTK == 2) {
                const double t = tv[k] - xv[k];
                a = fma(t, t, a);
              } else {
                a = fma(xv[k], tv[k], a);
                if (DOTK == 1) b = fma(xv[k], xv[k], b);
              }
            }
          }
        }
      }
    } else {
      for (int j = lane; j < p.d; j += 32) {
        const double xv = double(xr[j]);
        if (DOTK == 2) {
          const double t = th[j] - xv;
          a = fma(t, t, a);
        } else {
          a = fma(xv, th[j], a);
          if (DOTK == 1) b = fma(xv, xv, b);
        }
      }
    }
    a = warp_sum(a);
    if (DOTK == 1) b = warp_sum(b);
    if (lane == 0) {
      const double loss = finish_loss(p.kind, a, b, b0, (p.kind == RLVI_LOSS_LOGISTIC_CE || p.kind == RLVI_LOSS_SQRES) ? p.y[row] : 0.0);
      loss_row(p.o, row, loss, p.o.w ? p.o.w[row] : 0.0, s_wl, s_w);
    }
  }
  loss_sums(p.o, s_wl, s_w, sm_red);
}

}  // namespace

extern "C" int rlvi_loss_f64(rlvi_ctx* ctx, int kind, int intercept, const double* X, const double* y, int64_t n,
                             int d, const double* params, const double* weights, double* losses_out,
                             double* e_out, double* wsum_out, void* stream) {
  RLVI_REQUIRE(ctx && X && params, "null pointer");
  RLVI_REQUIRE(n > 0 && d > 0, "n and d must be positive");
  RLVI_REQUIRE(kind >= RLVI_LOSS_LOGISTIC_CE && kind <= RLVI_LOSS_GAUSSIAN, "unknown loss kind");
  RLVI_REQUIRE(losses_out || e_out || weights, "nothing to compute");
  RLVI_REQUIRE(!weights || wsum_out, "weights given but wsum_out is null");
  if (kind == RLVI_LOSS_LOGISTIC_CE || kind == RLVI_LOSS_SQRES) RLVI_REQUIRE(y != nullptr, "this loss needs y");
  RlviDeviceGuard guard(ctx->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int warps_per_block = kLossThreads / 32;
  const LossOut o = {weights, losses_out, e_out, wsum_out, nullptr, nullptr};

  if (kind == RLVI_LOSS_GAUSSIAN) {
    if (d > 128) {
      rlvi_set_error("RLVI_LOSS_GAUSSIAN supports d <= 128 (got %d)", d);
      return RLVI_ERR_UNSUPPORTED;
    }
    // ---- TMA-fed path: d in {16, 32, 48, 64}, aligned, at least one full tile ------------------------
    if (d % 16 == 0 && d <= 64 && n >= kRingRows && rlvi_aligned16(X) && (!weights || rlvi_aligned16(weights))) {
      GaussTmaParams q;
      q.X = X;
      q.params = params;
      q.o = o;
      q.n = n;
      q.d = d;
      const size_t tail = gauss_tma_tail(d);
      if (!ring_geometry(d, tail, &q.geom)) return RLVI_ERR_UNSUPPORTED;
      const int grid = ring_grid(q.geom, n, ctx->sm_count);
      const int rc = loss_scratch(ctx, grid, q.o);
      if (rc != RLVI_OK) return rc;
      const size_t smem = ring_bytes(q.geom) + tail;
#define RLVI_GTMA_CASE(NB)                                                                                    \
  if (d == 8 * NB) {                                                                                          \
    RLVI_CUDA(cudaFuncSetAttribute(gaussian_tma_kernel<NB>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem))); \
    gaussian_tma_kernel<NB><<<grid, kRingThreads, smem, st>>>(q);                                              \
    RLVI_LAUNCH_CHECK(ctx);                                                                                   \
    return RLVI_OK;                                                                                           \
  }
      RLVI_GTMA_CASE(2)
      RLVI_GTMA_CASE(4)
      RLVI_GTMA_CASE(6)
      RLVI_GTMA_CASE(8)
#undef RLVI_GTMA_CASE
    }
    const int nb = (d + 7) / 8, dp = nb * 8;
    const size_t smem = (size_t(dp) * (dp + 8) + dp + 2 * warps_per_block) * sizeof(double);
    const bool vec = rlvi_aligned16(X) && (d % 2 == 0);
    int64_t steps = (n + 7) / 8;
    int64_t want = (steps + warps_per_block - 1) / warps_per_block;
    int grid = int(want < 1 ? 1 : (want > int64_t(ctx->sm_count) * 2 ? int64_t(ctx->sm_count) * 2 : want));
    GaussParams p;
    p.X = X;
    p.params = params;
    p.o = o;
    p.n = n;
    p.d = d;
    const int rc = loss_scratch(ctx, grid, p.o);
    if (rc != RLVI_OK) return rc;
#define RLVI_GAUSS_CASE(NB, V)                                                                             \
  if (nb <= NB && vec == V) {                                                                              \
    RLVI_CUDA(cudaFuncSetAttribute(gaussian_loss_kernel<NB, V>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                   int(smem)));                                                            \
    gaussian_loss_kernel<NB, V><<<grid, kLossThreads, smem, st>>>(p);                                      \
    RLVI_LAUNCH_CHECK(ctx);                                                                                \
    return RLVI_OK;                                                                                        \
  }
    RLVI_GAUSS_CASE(8, true)
    RLVI_GAUSS_CASE(8, false)
    RLVI_GAUSS_CASE(16, true)
    RLVI_GAUSS_CASE(16, false)
#undef RLVI_GAUSS_CASE
    return RLVI_ERR_UNSUPPORTED;
  }

  // ---- TMA-fed path: d % 16 == 0, <= 256, all streamed arrays 16-byte aligned, at least one full tile ----
  if (d % 16 == 0 && d <= 256 && n >= kRingRows && rlvi_aligned16(X) && (!y || rlvi_aligned16(y)) &&
      (!weights || rlvi_aligned16(weights))) {
    LossTmaParams q;
    q.X = X;
    q.y = y;
    q.params = params;
    q.o = o;
    q.n = n;
    q.d = d;
    q.kind = kind;
    q.intercept = intercept ? 1 : 0;
    const size_t tail = loss_tma_tail(d);
    if (ring_geometry(d, tail, &q.geom)) {
      const int grid = ring_grid(q.geom, n, ctx->sm_count);
      const int rc = loss_scratch(ctx, grid, q.o);
      if (rc != RLVI_OK) return rc;
      const size_t smem = ring_bytes(q.geom) + tail;
#define RLVI_TMA_CASE(K)                                                                                   \
  {                                                                                                        \
    RLVI_CUDA(cudaFuncSetAttribute(loss_tma_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem))); \
    loss_tma_kernel<K><<<grid, kRingThreads, smem, st>>>(q);                                                \
    RLVI_LAUNCH_CHECK(ctx);                                                                                \
    return RLVI_OK;                                                                                        \
  }
      if (kind == RLVI_LOSS_PCA) RLVI_TMA_CASE(1)
      if (kind == RLVI_LOSS_SQDIST) RLVI_TMA_CASE(2)
      RLVI_TMA_CASE(0)
#undef RLVI_TMA_CASE
    }
  }

  RowMapCfg cfg;
  if (!rowmap_pick(d, rlvi_aligned16(X), &cfg)) {
    rlvi_set_error("loss kernels support 1 <= d <= 1024 (got %d)", d);
    return RLVI_ERR_UNSUPPORTED;
  }
  const int R = 32 / cfg.L;
  int64_t steps = (n + R - 1) / R;
  int64_t want = (steps + warps_per_block - 1) / warps_per_block;
  int64_t cap = int64_t(ctx->sm_count) * 8;    // 8 resident 256-thread CTAs per SM at <= 32 registers/thread... grid-stride covers the rest
  int grid = int(want < 1 ? 1 : (want > cap ? cap : want));
  LossParams p;
  p.X = X;
  p.y = y;
  p.params = params;
  p.o = o;
  p.n = n;
  p.d = d;
  p.kind = kind;
  p.intercept = intercept ? 1 : 0;
  p.L = cfg.L;
  const int rc = loss_scratch(ctx, grid, p.o);
  if (rc != RLVI_OK) return rc;
  const size_t smem = (size_t(d) + 2 + 2 * warps_per_block) * sizeof(double);
  if (kind == RLVI_LOSS_PCA) return launch_loss<1>(ctx, cfg, p, grid, smem, st);
  if (kind == RLVI_LOSS_SQDIST) return launch_loss<2>(ctx, cfg, p, grid, smem, st);
  return launch_loss<0>(ctx, cfg, p, grid, smem, st);
}

extern "C" int rlvi_loss_f32(rlvi_ctx* ctx, int kind, int intercept, const float* X, const double* y, int64_t n, int d,
                             const double* params, const double* weights, double* losses_out, double* e_out,
                             double* wsum_out, void* stream) {
  RLVI_REQUIRE(ctx && X && params, "null pointer");
  RLVI_REQUIRE(n > 0 && d > 0, "n and d must be positive");
  RLVI_REQUIRE(kind >= RLVI_LOSS_LOGISTIC_CE && kind <= RLVI_LOSS_PCA, "loss kind not available for FP32 samples");
  RLVI_REQUIRE(losses_out || e_out || weights, "nothing to compute");
  RLVI_REQUIRE(!weights || wsum_out, "weights given but wsum_out is null");
  if (kind == RLVI_LOSS_LOGISTIC_CE || kind == RLVI_LOSS_SQRES) RLVI_REQUIRE(y != nullptr, "this loss needs y");
  if (d > 4096) {
    rlvi_set_error("rlvi_loss_f32 supports d <= 4096 (got %d)", d);
    return RLVI_ERR_UNSUPPORTED;
  }
  RlviDeviceGuard guard(ctx->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int warps_per_block = kLossThreads / 32;
  int64_t want = (n + warps_per_block - 1) / warps_per_block;
  const int64_t cap = int64_t(ctx->sm_count) * 8;
  const int grid = int(want < 1 ? 1 : (want > cap ? cap : want));
  LossF32Params p;
  p.X = X;
  p.y = y;
  p.params = params;
  p.o = {weights, losses_out, e_out, wsum_out, nullptr, nullptr};
  p.n = n;
  p.d = d;
  p.kind = kind;
  p.intercept = intercept ? 1 : 0;
  p.vec = (rlvi_aligned16(X) && d % 4 == 0) ? 1 : 0;
  const int rc = loss_scratch(ctx, grid, p.o);
  if (rc != RLVI_OK) return rc;
  const size_t smem = (size_t((d + 127) & ~127) + 2 + 2 * warps_per_block) * sizeof(double);
  if (kind == RLVI_LOSS_PCA) loss_f32_kernel<1><<<grid, kLossThreads, smem, st>>>(p);
  else if (kind == RLVI_LOSS_SQDIST) loss_f32_kernel<2><<<grid, kLossThreads, smem, st>>>(p);
  else loss_f32_kernel<0><<<grid, kLossThreads, smem, st>>>(p);
  RLVI_LAUNCH_CHECK(ctx);
  return RLVI_OK;
}
