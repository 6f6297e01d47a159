// gpb_kern.cu -- fused covariance construction and its gradient reductions.
//
// Forward (gpb_kern_fwd) replaces Kernel.K (gptorch/kernels.py:189-222, 258-262) together with
// Stationary.squared_dist/dist (:149-172), util.squared_distance (gptorch/util.py:73-88) and the noise
// diagonal of GPR._compute_kyy (gptorch/models/gpr.py:69-86): one pass, one N^2 write, no temporaries.
// The X.X'^T term of the reference's expansion |a|^2 + |b|^2 - 2 a.b runs on FP64 DMMA; the clamp, sqrt,
// kernel non-linearity, variance and noise are applied in the accumulator epilogue.
//
// Backward (gpb_kern_bwd / gpb_gpr_grad) replaces torch autograd through those composite ops: it reduces an
// upstream gradient against dK/d(length scales, variance, X2) in one pass over G, recomputing K on the fly.
// For the GPR loss the upstream gradient W = 1/2 (dy Kinv - a a^T) is itself formed on the fly from the
// blocked inverse left by gpb_potri_lower, so neither W nor K is ever materialised.
#include "gpb_kernfn.cuh"
#include "gpb_kernbwd.cuh"
#include <algorithm>
#include <cstdlib>

namespace gpb {

// ================================================================================================
// forward
// ================================================================================================
constexpr int KF_TM = 64;     // tile rows  (2 warps x 32)
constexpr int KF_TN = 128;    // tile cols  (4 warps x 32)
constexpr int KF_MI = 4, KF_NI = 4;   // 8x8 DMMA fragments per warp tile (32 x 32): 32 accumulators per thread
constexpr int KF_DC = 16;    // feature chunk staged per pass
constexpr int KF_LD = 20;    // padded row stride (doubles): 20 mod 16 == 4 -> conflict-free DMMA fragment loads
constexpr int KF_THREADS = 256;
constexpr long KF_SQUARE_MIN_TILES = 4096;   // ~9 waves of 148 x 3 CTAs

struct KfwdParams {
  int kind;
  const double* X; int n1; long ldx;
  const double* X2; int n2; long ldx2;
  int D;
  const double* ell; int ell_len;
  const double* sigma2;
  const double* noise;
  int symmetric;   // X2 == NULL
  int lower;       // only tiles with tn <= tm
  double* K; long ldk;
  int tiles_n;
};

// 64 x 128 tile per CTA, 8 warps (2 x 4) of 32 x 32: 32 fp64 accumulators per thread keeps the kernel at two CTAs
// (16 warps) per SM, which is what hides the latency of the exp() chains in the epilogue.
// KIND is a compile-time constant: the family switch inside kern_base() folds away, and the polynomial constants of
// the one exp() that remains are shared by the 32 unrolled elements instead of being re-materialised per branch.
template <int KIND>
__global__ void __launch_bounds__(KF_THREADS, 2) kern_fwd_kernel(const KfwdParams p) {
  __shared__ double As[KF_TM * KF_LD];
  __shared__ double Bs[KF_TN * KF_LD];
  __shared__ double na[KF_TM], nbv[KF_TN];
  __shared__ double scale[KF_DC];

  int tm, tn;
  {
    const int t = blockIdx.x;
    if (p.lower) {
      // lower triangle in units of 128-column blocks: tile row tm (64 rows) needs column tiles 0 .. tm/2
      // enumerate pairs of tile rows: rows (2q, 2q+1) each have q+1 column tiles
      int q = static_cast<int>((sqrt(4.0 * t + 1.0) - 1.0) * 0.5);
      while ((q + 1) * (q + 2) <= t) ++q;
      while (q * (q + 1) > t) --q;
      const int rem = t - q * (q + 1);      // 0 .. 2(q+1)-1
      tm = 2 * q + rem / (q + 1);
      tn = rem % (q + 1);
    } else {
      tm = t / p.tiles_n;
      tn = t - tm * p.tiles_n;
    }
  }
  const int m0 = tm * KF_TM, n0 = tn * KF_TN;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int wm = warp & 1, wn = warp >> 1;
  const int r = lane >> 2, kk = lane & 3;
  constexpr bool linear = KIND == KERN_LINEAR;

  double acc[KF_MI][KF_NI][2];
#pragma unroll
  for (int i = 0; i < KF_MI; ++i)
#pragma unroll
    for (int j = 0; j < KF_NI; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
  double my_n = 0.0;  // thread t < 64: squared norm of A row t; 64 <= t < 192: of B row t - 64

  for (int d0 = 0; d0 < p.D; d0 += KF_DC) {
    __syncthreads();
    if (tid < KF_DC) {
      // per-dimension factor: the variance v_d for Linear, 1 / ell_d otherwise -- ONE division per dimension and CTA; the
      // staging loop below multiplies (a division per staged element was a quarter of this kernel's instructions)
      const int d = d0 + tid;
      double s = 1.0;
      if (d < p.D) s = p.ell[p.ell_len == 1 ? 0 : d];
      scale[tid] = linear ? s : 1.0 / s;
    }
    __syncthreads();
    for (int idx = tid; idx < (KF_TM + KF_TN) * KF_DC; idx += KF_THREADS) {
      const int row = idx >> 4, k = idx & 15;
      const int d = d0 + k;
      double v = 0.0;
      if (row < KF_TM) {
        if (d < p.D && m0 + row < p.n1) {
          const double x = p.X[static_cast<long>(m0 + row) * p.ldx + d];
          v = x * scale[k];
        }
        As[row * KF_LD + k] = v;
      } else {
        const int rb = row - KF_TM;
        if (d < p.D && n0 + rb < p.n2) {
          const double x = p.X2[static_cast<long>(n0 + rb) * p.ldx2 + d];
          v = linear ? x : x * scale[k];
        }
        Bs[rb * KF_LD + k] = v;
      }
    }
    __syncthreads();
    if (tid < KF_TM + KF_TN) {
      const double* src = tid < KF_TM ? &As[tid * KF_LD] : &Bs[(tid - KF_TM) * KF_LD];
#pragma unroll
      for (int k = 0; k < KF_DC; ++k) my_n += src[k] * src[k];
    }
    const int ksteps = min(KF_DC, p.D - d0 + 3) / 4;   // skip k4-steps that are all padding
    for (int ks = 0; ks < ksteps; ++ks) {
      double a[KF_MI], b[KF_NI];
#pragma unroll
      for (int i = 0; i < KF_MI; ++i) a[i] = As[(wm * 32 + 8 * i + r) * KF_LD + ks * 4 + kk];
#pragma unroll
      for (int j = 0; j < KF_NI; ++j) b[j] = Bs[(wn * 32 + 8 * j + r) * KF_LD + ks * 4 + kk];
#pragma unroll
      for (int i = 0; i < KF_MI; ++i)
#pragma unroll
        for (int j = 0; j < KF_NI; ++j) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
    }
  }
  if (tid < KF_TM) na[tid] = my_n;
  else if (tid < KF_TM + KF_TN) nbv[tid - KF_TM] = my_n;
  __syncthreads();

  const double sig2 = linear ? 1.0 : *p.sigma2;
  const double noise = (p.symmetric && p.noise) ? *p.noise : 0.0;
  // Two fragment rows (16 elements) per basic block: the fp64 chains (distance, exp polynomial) of different elements are
  // independent, and only when they sit in the same branch-free block does the scheduler interleave them.  The row bound
  // is applied at the stores, not as a branch around the arithmetic.
#pragma unroll
  for (int ip = 0; ip < KF_MI; ip += 2) {
    double v[2][KF_NI][2];
#pragma unroll
    for (int ii = 0; ii < 2; ++ii) {
      const int i = ip + ii;
      const int lr = wm * 32 + 8 * i + r;
      const int row = m0 + lr;
      const double nrow = na[lr];
#pragma unroll
      for (int j = 0; j < KF_NI; ++j) {
        const int lc = wn * 32 + 8 * j + 2 * kk;
        const int col = n0 + lc;
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const double dot = acc[i][j][e];
          const bool diag = p.symmetric && row == col + e;
          double val;
          if (linear) {
            val = dot;
          } else {
            double r2 = (nrow + nbv[lc + e]) - 2.0 * dot;  // gptorch/util.py:84
            r2 = fmax(r2, 0.0);                             // value of r2 - clamp(r2, max=0) (gptorch/util.py:88)
            // K(X) diagonal: the reference's expansion leaves O(1e-16) round-off here, which sqrt() turns into
            // O(1e-8) noise for Exp/Matern; the distance of a point to itself is exactly 0.
            r2 = diag ? 0.0 : r2;
            val = sig2 * kern_base(KIND, r2);
          }
          v[ii][j][e] = diag ? val + noise : val;
        }
      }
    }
#pragma unroll
    for (int ii = 0; ii < 2; ++ii) {
      const int row = m0 + wm * 32 + 8 * (ip + ii) + r;
      if (row >= p.n1) continue;
      double* krow = p.K + static_cast<long>(row) * p.ldk;
#pragma unroll
      for (int j = 0; j < KF_NI; ++j) {
        const int col = n0 + wn * 32 + 8 * j + 2 * kk;
        if (col + 1 < p.n2 && ((p.ldk & 1) == 0)) {
          __stcs(reinterpret_cast<double2*>(krow + col), make_double2(v[ii][j][0], v[ii][j][1]));
        } else {
          if (col < p.n2) krow[col] = v[ii][j][0];
          if (col + 1 < p.n2) krow[col + 1] = v[ii][j][1];
        }
      }
    }
  }
}

// D <= 16: the whole feature range is ONE staging chunk, so the distance tile can be produced in passes of 16 fragment
// rows -- 16 instead of 32 live accumulators per thread, which brings the kernel under 85 registers and THREE CTAs (24
// warps) per SM.  Round-2 ncu (profiles/r02_ncu_covariance_kernels_n32768.txt): 47 % of the stall samples of the first
// version sat in the staging prologue (a load -> scale -> store loop of 12 dependent global-memory round trips per CTA,
// plus spills in the epilogue), not in the exp chains; the one-thread-per-row staging below exposes ONE round trip, and
// four-element batches (kern_base_vec) keep the epilogue free of spills: 1.80 -> 1.34 ms at N = 32768, D = 8 (RBF).
template <int KIND, int HALVES>
__global__ void __launch_bounds__(KF_THREADS, 3) kern_fwd_d16_kernel(const KfwdParams p) {
  constexpr int RP = 2;                // fragment rows per pass
  constexpr int TM = KF_TM * HALVES;   // HALVES = 2: two 64-row halves share one staged X2 block (128 x 128 tile)
  __shared__ __align__(16) double As[TM * KF_LD];
  __shared__ __align__(16) double Bs[KF_TN * KF_LD];
  __shared__ double na[TM], nbv[KF_TN];
  __shared__ double scale[KF_DC];
  int tm, tn;
  {
    const int t = blockIdx.x;
    if (p.lower && HALVES == 2) {
      // square tiles: plain triangular enumeration, tile row tm holds column tiles 0 .. tm
      int q = static_cast<int>((sqrtf(8.0f * static_cast<float>(t) + 1.0f) - 1.0f) * 0.5f);   // estimate, corrected below
      while ((q + 1) * (q + 2) / 2 <= t) ++q;
      while (q * (q + 1) / 2 > t) --q;
      tm = q;
      tn = t - q * (q + 1) / 2;
    } else if (p.lower) {
      int q = static_cast<int>((sqrtf(4.0f * static_cast<float>(t) + 1.0f) - 1.0f) * 0.5f);   // estimate, corrected below
      while ((q + 1) * (q + 2) <= t) ++q;
      while (q * (q + 1) > t) --q;
      const int rem = t - q * (q + 1);
      tm = 2 * q + rem / (q + 1);
      tn = rem % (q + 1);
    } else {
      tm = t / p.tiles_n;
      tn = t - tm * p.tiles_n;
    }
  }
  const int m0 = tm * TM, n0 = tn * KF_TN;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int wm = warp & 1, wn = warp >> 1;
  const int r = lane >> 2, kk = lane & 3;
  constexpr bool linear = KIND == KERN_LINEAR;

  // Staging: one thread per row (64 rows of X, 128 of X2).  The row's loads are independent instructions issued BEFORE
  // the barrier that publishes the reciprocal length scales, so a CTA exposes one global-memory latency, not one per
  // staging iteration; scaling, the padded shared-memory row and the row's squared norm then come out of registers in
  // the same thread (the norm is the k-ordered sum of the staged values, as before).
  const bool is_a = tid < TM;
  const int srow = is_a ? tid : tid - TM;
  const double sig2 = linear ? 1.0 : __ldg(p.sigma2);   // issued with the row loads, ahead of the barriers
  const double noise = (p.symmetric && p.noise) ? __ldg(p.noise) : 0.0;
  double xr[KF_DC];
  if (tid < TM + KF_TN) {
    const bool in = is_a ? (m0 + srow < p.n1) : (n0 + srow < p.n2);
    const double* src = is_a ? p.X + static_cast<long>(m0 + srow) * p.ldx : p.X2 + static_cast<long>(n0 + srow) * p.ldx2;
    const bool vec = (((p.ldx | p.ldx2 | static_cast<long>(p.D)) & 1) == 0) &&
                     (((reinterpret_cast<uintptr_t>(p.X) | reinterpret_cast<uintptr_t>(p.X2)) & 15) == 0);
    if (vec) {
#pragma unroll
      for (int k = 0; k < KF_DC; k += 2) {
        double2 v = make_double2(0.0, 0.0);
        if (in && k < p.D) v = __ldg(reinterpret_cast<const double2*>(src + k));
        xr[k] = v.x;
        xr[k + 1] = v.y;
      }
    } else {
#pragma unroll
      for (int k = 0; k < KF_DC; ++k) xr[k] = (in && k < p.D) ? __ldg(src + k) : 0.0;
    }
  }
  if (tid >= KF_THREADS - KF_DC) {
    const int k = tid - (KF_THREADS - KF_DC);
    double s = 1.0;
    if (k < p.D) s = p.ell[p.ell_len == 1 ? 0 : k];
    scale[k] = linear ? s : 1.0 / s;
  }
  __syncthreads();
  if (tid < TM + KF_TN) {
    double* dst = is_a ? &As[srow * KF_LD] : &Bs[srow * KF_LD];
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < KF_DC; k += 2) {
      double2 v;
      v.x = (linear && !is_a) ? xr[k] : xr[k] * scale[k];
      v.y = (linear && !is_a) ? xr[k + 1] : xr[k + 1] * scale[k + 1];
      *reinterpret_cast<double2*>(dst + k) = v;
      s += v.x * v.x;
      s += v.y * v.y;
    }
    if (is_a) na[srow] = s;
    else nbv[srow] = s;
  }
  __syncthreads();

  const int ksteps = min(KF_DC, p.D + 3) / 4;
#pragma unroll 1
  for (int ihh = 0; ihh < HALVES * 4 / RP; ++ihh) {
    const int ih = ihh % (4 / RP), h0 = (ihh / (4 / RP)) * KF_TM;
    double acc[RP][KF_NI][2];
#pragma unroll
    for (int i = 0; i < RP; ++i)
#pragma unroll
      for (int j = 0; j < KF_NI; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
    for (int ks = 0; ks < ksteps; ++ks) {
      double a[RP], b[KF_NI];
#pragma unroll
      for (int i = 0; i < RP; ++i) a[i] = As[(h0 + wm * 32 + 8 * (RP * ih + i) + r) * KF_LD + ks * 4 + kk];
#pragma unroll
      for (int j = 0; j < KF_NI; ++j) b[j] = Bs[(wn * 32 + 8 * j + r) * KF_LD + ks * 4 + kk];
#pragma unroll
      for (int i = 0; i < RP; ++i)
#pragma unroll
        for (int j = 0; j < KF_NI; ++j) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
    }
#pragma unroll
    for (int i = 0; i < RP; ++i) {
      const int lr = h0 + wm * 32 + 8 * (RP * ih + i) + r;
      const int row = m0 + lr;
      const double nrow = na[lr];
      double* krow = p.K + static_cast<long>(row) * p.ldk;
      // four elements (two column pairs) per batch: their exp chains are issued interleaved (kern_base_vec)
#pragma unroll
      for (int jp = 0; jp < KF_NI; jp += 2) {
        double v[4];
        bool diag[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int j = jp + (q >> 1), e = q & 1;
          const int lc = wn * 32 + 8 * j + 2 * kk;
          const double dot = acc[i][j][e];
          diag[q] = p.symmetric && row == n0 + lc + e;
          if (linear) {
            v[q] = dot;
          } else {
            double r2 = (nrow + nbv[lc + e]) - 2.0 * dot;  // gptorch/util.py:84
            r2 = fmax(r2, 0.0);                             // gptorch/util.py:88
            v[q] = diag[q] ? 0.0 : r2;                      // exact zero self-distance (see kern_fwd_kernel)
          }
        }
        if constexpr (KIND == KERN_RBF || KIND == KERN_EXP || KIND == KERN_MATERN32 || KIND == KERN_MATERN52) {
          kern_base_vec<KIND, 4>(v);
        } else if (!linear) {
#pragma unroll
          for (int q = 0; q < 4; ++q) v[q] = kern_base(KIND, v[q]);
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          if (!linear) v[q] = sig2 * v[q];
          v[q] = diag[q] ? v[q] + noise : v[q];
        }
        if (row < p.n1) {
#pragma unroll
          for (int jj = 0; jj < 2; ++jj) {
            const int col = n0 + wn * 32 + 8 * (jp + jj) + 2 * kk;
            if (col + 1 < p.n2 && ((p.ldk & 1) == 0)) {
              __stcs(reinterpret_cast<double2*>(krow + col), make_double2(v[2 * jj], v[2 * jj + 1]));
            } else {
              if (col < p.n2) krow[col] = v[2 * jj];
              if (col + 1 < p.n2) krow[col + 1] = v[2 * jj + 1];
            }
          }
        }
      }
    }
  }
}

int kern_fwd(int kind, const double* X, int n1, long ldx, const double* X2, int n2, long ldx2, int D,
             const double* ell, int ell_len, const double* sigma2, const double* noise, int fill, double* K,
             long ldk, cudaStream_t stream) {
  if (kind < 0 || kind > KERN_PERIODIC) return GPB_ERR_BADARG;
  if (!X || !K || !ell || D <= 0 || (ell_len != 1 && ell_len != D)) return GPB_ERR_BADARG;
  if (kind != KERN_LINEAR && !sigma2) return GPB_ERR_BADARG;
  if (kind == KERN_LINEAR && ell_len != D) return GPB_ERR_BADARG;
  KfwdParams p;
  p.kind = kind;
  p.X = X; p.n1 = n1; p.ldx = ldx;
  p.symmetric = (X2 == nullptr);
  if (p.symmetric) { p.X2 = X; p.n2 = n1; p.ldx2 = ldx; }
  else { p.X2 = X2; p.n2 = n2; p.ldx2 = ldx2; }
  if (n1 <= 0 || p.n2 <= 0) return GPB_OK;
  if (ldx < D || p.ldx2 < D || ldk < p.n2) return GPB_ERR_BADARG;
  if (reinterpret_cast<uintptr_t>(K) & 15) return GPB_ERR_ALIGN;
  p.D = D; p.ell = ell; p.ell_len = ell_len; p.sigma2 = sigma2; p.noise = noise;
  p.lower = (fill == 1);
  if (p.lower && !p.symmetric) return GPB_ERR_BADARG;
  p.K = K; p.ldk = ldk;
  // D <= 16 kernel: 128 x 128 tiles (two row halves per staged X2 block) once the 64-row tiling has CTAs to spare
  static const int force_square = [] { const char* e = getenv("GPB_KFWD_SQUARE"); return e ? atoi(e) : -1; }();
  const long tiles64 = static_cast<long>((n1 + KF_TM - 1) / KF_TM) * ((p.n2 + KF_TN - 1) / KF_TN) / (p.lower ? 2 : 1);
  const bool square = D <= KF_DC && (force_square >= 0 ? force_square != 0 : tiles64 >= KF_SQUARE_MIN_TILES);
  const int tile_rows = square ? 2 * KF_TM : KF_TM;
  const int tiles_m = (n1 + tile_rows - 1) / tile_rows;
  p.tiles_n = (p.n2 + KF_TN - 1) / KF_TN;
  // lower fill: tile row tm (64 rows) covers column tiles 0 .. tm/2 (128 columns each)
  int ntiles = tiles_m * p.tiles_n;
  if (p.lower && square) {
    ntiles = tiles_m * (tiles_m + 1) / 2;
  } else if (p.lower) {
    const int q = tiles_m / 2;               // complete pairs of tile rows
    ntiles = q * (q + 1) + ((tiles_m & 1) ? (q + 1) : 0);
  }
  if (D <= KF_DC) {
#define GPB_KF16(KIND)                                                                                   \
  do {                                                                                                   \
    if (square) kern_fwd_d16_kernel<KIND, 2><<<ntiles, KF_THREADS, 0, stream>>>(p);                      \
    else kern_fwd_d16_kernel<KIND, 1><<<ntiles, KF_THREADS, 0, stream>>>(p);                             \
  } while (0)
    switch (kind) {
      case KERN_RBF: GPB_KF16(KERN_RBF); break;
      case KERN_EXP: GPB_KF16(KERN_EXP); break;
      case KERN_MATERN32: GPB_KF16(KERN_MATERN32); break;
      case KERN_MATERN52: GPB_KF16(KERN_MATERN52); break;
      case KERN_LINEAR: GPB_KF16(KERN_LINEAR); break;
      default: GPB_KF16(KERN_PERIODIC); break;
    }
#undef GPB_KF16
    count_launch();
    GPB_CUDA_CHECK(cudaGetLastError());
    return GPB_OK;
  }
  switch (kind) {
    case KERN_RBF: kern_fwd_kernel<KERN_RBF><<<ntiles, KF_THREADS, 0, stream>>>(p); break;
    case KERN_EXP: kern_fwd_kernel<KERN_EXP><<<ntiles, KF_THREADS, 0, stream>>>(p); break;
    case KERN_MATERN32: kern_fwd_kernel<KERN_MATERN32><<<ntiles, KF_THREADS, 0, stream>>>(p); break;
    case KERN_MATERN52: kern_fwd_kernel<KERN_MATERN52><<<ntiles, KF_THREADS, 0, stream>>>(p); break;
    case KERN_LINEAR: kern_fwd_kernel<KERN_LINEAR><<<ntiles, KF_THREADS, 0, stream>>>(p); break;
    default: kern_fwd_kernel<KERN_PERIODIC><<<ntiles, KF_THREADS, 0, stream>>>(p); break;
  }
  count_launch();
  GPB_CUDA_CHECK(cudaGetLastError());
  return GPB_OK;
}

// ================================================================================================
// Linear.Kdiag
// ================================================================================================
__global__ void linear_kdiag_kernel(const double* __restrict__ X, int n, long ldx, int D, const double* __restrict__ v,
                                    double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double s = 0.0;
  for (int d = 0; d < D; ++d) {
    const double x = X[static_cast<long>(i) * ldx + d];
    s += x * x * v[d];  // gptorch/kernels.py:265
  }
  out[i] = s;
}

int linear_kdiag(const double* X, int n, long ldx, int D, const double* v, double* out, cudaStream_t stream) {
  if (n <= 0) return GPB_OK;
  if (!X || !v || !out || D <= 0) return GPB_ERR_BADARG;
  linear_kdiag_kernel<<<(n + 255) / 256, 256, 0, stream>>>(X, n, ldx, D, v, out);
  count_launch();
  GPB_CUDA_CHECK(cudaGetLastError());
  return GPB_OK;
}

// ================================================================================================
// backward reductions
// ================================================================================================
constexpr int KB_COLS = 128;     // columns (second argument) per CTA, one per thread pair
constexpr int KB_RT = 8;         // rows per thread per chunk
constexpr int KB_ROWS = 2 * KB_RT;  // rows per chunk (two thread halves)
constexpr int KB_THREADS = 256;
// accumulator chunk of feature dimensions (template parameter KB_DC): 8 when D <= 8, else 16
constexpr int KB_DMAX = 160;     // shared-memory staging limit on D
constexpr int KB_DY = 8;         // a-vector chunk


// G2: also accumulate the per-column sums needed for dLoss/dX2 (and for the Linear kernel's variance gradient).
// KIND >= 0: the covariance family as a compile-time constant (stationary families); KIND < 0: read p.kind at run time
// (Linear, Constant, White -- no transcendental in their derivative).
template <bool GPR, int KB_DC, bool G2, int KIND>
__global__ void __launch_bounds__(KB_THREADS, 2) kern_bwd_kernel(const KbwdParams p) {
  const int kind = KIND >= 0 ? KIND : p.kind;
  extern __shared__ double kb_smem[];
  const int D = p.D;
  double* X2s = kb_smem;                       // [D][128]
  double* X1s = X2s + static_cast<size_t>(D) * KB_COLS;    // [KB_ROWS][D]
  double* ellv = X1s + static_cast<size_t>(KB_ROWS) * D;   // [D]
  double* acol = ellv + D;                     // [KB_DY][128]
  double* arow = acol + KB_COLS * KB_DY;       // [KB_ROWS][KB_DY]
  double* red = arow + KB_ROWS * KB_DY;        // [32] + [2][128] combine scratch
  double* comb = red + 32;

  const int t = threadIdx.x, c = t & 127, half = t >> 7;
  const int cb = blockIdx.x, strip = blockIdx.y;
  const int c0 = cb * KB_COLS;
  const int j = c0 + c;
  const bool jvalid = j < p.n2;
  const bool linear = kind == KERN_LINEAR;
  const int cta = blockIdx.y * gridDim.x + blockIdx.x;

  for (int d = t; d < D; d += KB_THREADS) ellv[d] = p.ell[p.ell_len == 1 ? 0 : d];
  __syncthreads();
  for (int idx = t; idx < KB_COLS * D; idx += KB_THREADS) {
    const int cc = idx / D, d = idx - cc * D;
    double v = 0.0;
    if (c0 + cc < p.n2) {
      v = p.X2[static_cast<long>(c0 + cc) * p.ldx2 + d];
      if (!linear) v /= ellv[d];
    }
    X2s[d * KB_COLS + cc] = v;
  }
  const double sig2 = linear ? 1.0 : *p.sigma2;
  // GPR: rows start at the column block's own 128-block (lower triangle only)
  const int rc_start = GPR ? (c0 / KB_ROWS) : 0;

  double sK = 0.0, gn = 0.0;
  const int ndc = (D + KB_DC - 1) / KB_DC;
  for (int dc = 0; dc < ndc; ++dc) {
    double S[KB_DC], g2[KB_DC];
#pragma unroll
    for (int dd = 0; dd < KB_DC; ++dd) S[dd] = g2[dd] = 0.0;

    for (int rc = rc_start + strip; rc < p.nrc; rc += p.strips) {
      const int i0 = rc * KB_ROWS;
      __syncthreads();
      for (int idx = t; idx < KB_ROWS * D; idx += KB_THREADS) {
        const int rr = idx / D, d = idx - rr * D;
        double v = 0.0;
        if (i0 + rr < p.n1) {
          v = p.X1[static_cast<long>(i0 + rr) * p.ldx1 + d];
          if (!linear) v /= ellv[d];
        }
        X1s[rr * D + d] = v;
      }
      double hreg[KB_RT];
      if (GPR) {
        // aa[rr] = sum_o a[i][o] a[j][o], staged in chunks of KB_DY outputs
#pragma unroll
        for (int rr = 0; rr < KB_RT; ++rr) hreg[rr] = 0.0;
        for (int o0 = 0; o0 < p.dy; o0 += KB_DY) {
          __syncthreads();
          for (int idx = t; idx < KB_COLS * KB_DY; idx += KB_THREADS) {
            const int cc = idx / KB_DY, o = idx - cc * KB_DY;
            acol[o * KB_COLS + cc] = (c0 + cc < p.n2 && o0 + o < p.dy) ? p.a[static_cast<long>(c0 + cc) * p.lda + o0 + o] : 0.0;
          }
          for (int idx = t; idx < KB_ROWS * KB_DY; idx += KB_THREADS) {
            const int rr = idx / KB_DY, o = idx - rr * KB_DY;
            arow[idx] = (i0 + rr < p.n1 && o0 + o < p.dy) ? p.a[static_cast<long>(i0 + rr) * p.lda + o0 + o] : 0.0;
          }
          __syncthreads();
#pragma unroll
          for (int o = 0; o < KB_DY; ++o) {
            const double aj = acol[o * KB_COLS + c];
#pragma unroll
            for (int rr = 0; rr < KB_RT; ++rr) hreg[rr] += arow[(half * KB_RT + rr) * KB_DY + o] * aj;
          }
        }
      }
      __syncthreads();

      // ---- phase A: scaled squared distances of this thread's KB_RT rows against its column ----
      double r2[KB_RT];
#pragma unroll
      for (int rr = 0; rr < KB_RT; ++rr) r2[rr] = 0.0;
      if (!linear) {
        for (int d = 0; d < D; ++d) {
          const double x2d = X2s[d * KB_COLS + c];
#pragma unroll
          for (int rr = 0; rr < KB_RT; ++rr) {
            const double diff = X1s[(half * KB_RT + rr) * D + d] - x2d;
            r2[rr] += diff * diff;
          }
        }
      }
#pragma unroll
      for (int rr = 0; rr < KB_RT; ++rr) {
        const int i = i0 + half * KB_RT + rr;
        bool valid = jvalid && i < p.n1;
        double g = 0.0;
        if (GPR) {
          valid = valid && i >= j;
          if (valid) {
            const bool same_blk = (i / NB) == (j / NB);
            const double kinv = same_blk ? p.kd[static_cast<long>(i) * NB + (j - (j / NB) * NB)]
                                         : __ldcs(&p.Kinv[static_cast<long>(i) * p.ldk + j]);
            const double w = 0.5 * (static_cast<double>(p.dy) * kinv - hreg[rr]);
            if (i == j) {
              if (dc == 0) gn += w;
              g = w;
            } else {
              g = 2.0 * w;
            }
          }
        } else if (valid) {
          g = p.g_trans ? p.G[static_cast<long>(j) * p.ldg + i] : __ldcs(&p.G[static_cast<long>(i) * p.ldg + j]);
          if (p.Mul) g *= p.g_trans ? p.Mul[static_cast<long>(j) * p.ldm + i] : __ldcs(&p.Mul[static_cast<long>(i) * p.ldm + j]);
        }
        double h = 0.0;
        if (valid) {
          if (linear) {
            h = g;
          } else if (kind >= KERN_CONSTANT) {
            // Constant: K = sigma2; White: K = sigma2 [i == j] for K(X), 0 for K(X, X2) (gptorch/kernels.py:83-101)
            if (dc == 0 && (kind == KERN_CONSTANT || (p.symmetric && i == j))) sK += g;
          } else {
            double kbase, fac1;
            kern_base_fac(kind, r2[rr], kbase, fac1);
            if (dc == 0) sK += g * kbase;
            h = g * fac1 * sig2;
          }
        }
        hreg[rr] = h;
      }

      // ---- phase B: accumulate this chunk of feature dimensions -------------------------------------
#pragma unroll
      for (int dd = 0; dd < KB_DC; ++dd) {
        const int d = dc * KB_DC + dd;
        if (d < D) {
          const double x2d = X2s[d * KB_COLS + c];
#pragma unroll
          for (int rr = 0; rr < KB_RT; ++rr) {
            const double x1d = X1s[(half * KB_RT + rr) * D + d];
            if (linear) {
              if (G2) g2[dd] += hreg[rr] * x1d;
            } else {
              const double diff = x1d - x2d;
              const double u = hreg[rr] * diff;
              if (G2) g2[dd] += u;
              S[dd] += u * diff;
            }
          }
        }
      }
    }  // row chunks

    // ---- flush this feature chunk: S -> per-CTA partial, g2 -> per-strip partial ---------------------
#pragma unroll
    for (int dd = 0; dd < KB_DC; ++dd) {
      const int d = dc * KB_DC + dd;
      if (d >= D) break;  // uniform across the block
      double s = linear ? g2[dd] * X2s[d * KB_COLS + c] : S[dd];
      s = block_sum(s, red);
      if (t == 0) p.part_h[static_cast<long>(cta) * (D + 2) + d] = s;
      if (G2 && p.part_g2) {
        __syncthreads();
        comb[half * KB_COLS + c] = g2[dd];
        __syncthreads();
        if (half == 0 && jvalid)
          p.part_g2[(static_cast<long>(strip) * p.n2 + j) * D + d] = comb[c] + comb[KB_COLS + c];
      }
    }
  }
  sK = block_sum(sK, red);
  if (t == 0) p.part_h[static_cast<long>(cta) * (D + 2) + D] = sK;
  gn = block_sum(gn, red);
  if (t == 0) p.part_h[static_cast<long>(cta) * (D + 2) + D + 1] = gn;
}

// Final deterministic reduction of the per-CTA partials and scaling to gradients w.r.t. the kernel's own
// (transformed) hyper-parameters ell, sigma2 (the exp-transform chain rule is left to torch autograd,
// gptorch/param.py:35).
__global__ void kbwd_finalize_kernel(int kind, int D, int ell_len, const double* __restrict__ ell, int ncta,
                                     const double* __restrict__ part_h, int strips, int n2,
                                     const double* __restrict__ part_g2, double* __restrict__ g_ell,
                                     double* __restrict__ g_sigma2, double* __restrict__ g_noise,
                                     double* __restrict__ gX2) {
  const long gid = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const bool linear = kind == KERN_LINEAR;
  if (gid < D + 2) {
    double s = 0.0;
    for (int cta = 0; cta < ncta; ++cta) s += part_h[static_cast<long>(cta) * (D + 2) + gid];
    if (gid < D) {
      if (linear) {
        g_ell[gid] = s;
      } else if (ell_len == D) {
        g_ell[gid] = s / ell[gid];
      } else {
        // isotropic: handled below by thread D-th? -> accumulate serially here for determinism
      }
    } else if (gid == D) {
      if (g_sigma2) g_sigma2[0] = s;
    } else {
      if (g_noise) g_noise[0] = s;
    }
  }
  if (gid == 0 && !linear && ell_len == 1) {
    double tot = 0.0;
    for (int d = 0; d < D; ++d) {
      double s = 0.0;
      for (int cta = 0; cta < ncta; ++cta) s += part_h[static_cast<long>(cta) * (D + 2) + d];
      tot += s;
    }
    g_ell[0] = tot / ell[0];
  }
  if (gX2 != nullptr && part_g2 != nullptr) {
    const long total = static_cast<long>(n2) * D;
    for (long idx = gid; idx < total; idx += static_cast<long>(gridDim.x) * blockDim.x) {
      const int d = static_cast<int>(idx % D);
      double s = 0.0;
      for (int st = 0; st < strips; ++st) s += part_g2[static_cast<long>(st) * total + idx];
      const double e = ell[ell_len == 1 ? 0 : d];
      gX2[idx] = linear ? s * e : s / e;
    }
  }
}

static inline size_t kbwd_smem_bytes(int D) {
  return (static_cast<size_t>(D) * KB_COLS + static_cast<size_t>(KB_ROWS) * D + D + KB_COLS * KB_DY + KB_ROWS * KB_DY +
          32 + 2 * KB_COLS) * sizeof(double);
}

static inline void kbwd_grid(int nrows, int ncols, bool lower, int& ncb, int& nrc, int& strips) {
  ncb = (ncols + KB_COLS - 1) / KB_COLS;
  nrc = (nrows + KB_ROWS - 1) / KB_ROWS;
  const int target = 4 * 148;
  strips = std::max(1, std::min(nrc, (target + ncb - 1) / ncb));
  (void)lower;
}

size_t kern_bwd_workspace_bytes(int n1, int n2, int D) {
  int ncb, nrc, strips;
  kbwd_grid(n1, n2, false, ncb, nrc, strips);
  const size_t ncta = static_cast<size_t>(ncb) * strips;
  return (ncta * (D + 2) + static_cast<size_t>(strips) * n2 * D) * sizeof(double) + 256;
}

template <bool GPR, int DC, bool G2, int KIND>
static int kbwd_launch_kind(const KbwdParams& p, int ncb, size_t smem, cudaStream_t stream) {
  static std::atomic<int> smem_state[GPB_MAX_DEVICES];
  if (int rc = ensure_dynamic_smem(kern_bwd_kernel<GPR, DC, G2, KIND>, static_cast<int>(smem), smem_state)) return rc;
  dim3 grid(ncb, p.strips);
  kern_bwd_kernel<GPR, DC, G2, KIND><<<grid, KB_THREADS, smem, stream>>>(p);
  count_launch();
  GPB_CUDA_CHECK(cudaGetLastError());
  return GPB_OK;
}

template <bool GPR, int DC, bool G2>
static int kbwd_launch_cfg(const KbwdParams& p, int ncb, size_t smem, cudaStream_t stream) {
  switch (p.kind) {
    case KERN_RBF: return kbwd_launch_kind<GPR, DC, G2, KERN_RBF>(p, ncb, smem, stream);
    case KERN_EXP: return kbwd_launch_kind<GPR, DC, G2, KERN_EXP>(p, ncb, smem, stream);
    case KERN_MATERN32: return kbwd_launch_kind<GPR, DC, G2, KERN_MATERN32>(p, ncb, smem, stream);
    case KERN_MATERN52: return kbwd_launch_kind<GPR, DC, G2, KERN_MATERN52>(p, ncb, smem, stream);
    case KERN_PERIODIC: return kbwd_launch_kind<GPR, DC, G2, KERN_PERIODIC>(p, ncb, smem, stream);
    default: return kbwd_launch_kind<GPR, DC, G2, -1>(p, ncb, smem, stream);
  }
}

// ---- DMMA path (gpb_kern_mma.cuh, one translation unit per covariance family) -------------------------------------------
int kbwd_mma_launch_rbf(const KbwdParams& p, int ncb, bool gpr, bool g2, cudaStream_t stream);
int kbwd_mma_launch_exp(const KbwdParams& p, int ncb, bool gpr, bool g2, cudaStream_t stream);
int kbwd_mma_launch_matern32(const KbwdParams& p, int ncb, bool gpr, bool g2, cudaStream_t stream);
int kbwd_mma_launch_matern52(const KbwdParams& p, int ncb, bool gpr, bool g2, cudaStream_t stream);

static int kbwd_mma_launch(const KbwdParams& p, int ncb, bool gpr, bool g2, cudaStream_t stream) {
  switch (p.kind) {
    case KERN_RBF: return kbwd_mma_launch_rbf(p, ncb, gpr, g2, stream);
    case KERN_EXP: return kbwd_mma_launch_exp(p, ncb, gpr, g2, stream);
    case KERN_MATERN32: return kbwd_mma_launch_matern32(p, ncb, gpr, g2, stream);
    default: return kbwd_mma_launch_matern52(p, ncb, gpr, g2, stream);
  }
}

static inline bool kbwd_use_mma(const KbwdParams& p, bool gpr) {
  const bool family = p.kind == KERN_RBF || p.kind == KERN_EXP || p.kind == KERN_MATERN32 || p.kind == KERN_MATERN52;
  return family && p.D <= 32 && p.Mul == nullptr && !p.g_trans && (!gpr || p.dy <= BM_DY);
}

template <bool GPR>
static int kbwd_launch(KbwdParams& p, int ncb, double* g_ell, double* g_sigma2, double* g_noise, double* gX2,
                       cudaStream_t stream) {
  if (kbwd_use_mma(p, GPR)) {
    // 64-row tiles; the strips never exceed the scalar kernel's (its row chunks are shorter), so the caller's workspace
    // -- sized by kern_bwd_workspace_bytes / gpr_grad_workspace_bytes -- covers the per-CTA partials of this path too
    const int ntr = (p.n1 + BM_TM - 1) / BM_TM;
    p.strips = std::max(1, std::min(p.strips, ntr));
    if (gX2) p.part_g2 = p.part_h + static_cast<size_t>(ncb) * p.strips * (p.D + 2);
    // K(X) evaluated as K(X, X): the distance of a point to itself is exactly 0, as in the forward kernel
    if (p.X1 == p.X2 && p.ldx1 == p.ldx2 && p.n1 == p.n2) p.symmetric = 1;
    const int rc = kbwd_mma_launch(p, ncb, GPR, !GPR && gX2 != nullptr, stream);
    if (rc) return rc;
    const int ncta = ncb * p.strips;
    const long work = std::max<long>(p.D + 2, gX2 ? static_cast<long>(p.n2) * p.D : 0);
    const int blocks = static_cast<int>(std::min<long>((work + 255) / 256, 1024));
    kbwd_finalize_kernel<<<blocks, 256, 0, stream>>>(p.kind, p.D, p.ell_len, p.ell, ncta, p.part_h, p.strips, p.n2,
                                                     gX2 ? p.part_g2 : nullptr, g_ell, g_sigma2, g_noise, gX2);
    count_launch();
    GPB_CUDA_CHECK(cudaGetLastError());
    return GPB_OK;
  }
  const size_t smem = kbwd_smem_bytes(p.D);
  const bool g2 = (gX2 != nullptr) || p.kind == KERN_LINEAR;
  int rc;
  if (p.D <= 8) rc = g2 ? kbwd_launch_cfg<GPR, 8, true>(p, ncb, smem, stream) : kbwd_launch_cfg<GPR, 8, false>(p, ncb, smem, stream);
  else rc = g2 ? kbwd_launch_cfg<GPR, 16, true>(p, ncb, smem, stream) : kbwd_launch_cfg<GPR, 16, false>(p, ncb, smem, stream);
  if (rc) return rc;
  const int ncta = ncb * p.strips;
  const long work = std::max<long>(p.D + 2, gX2 ? static_cast<long>(p.n2) * p.D : 0);
  const int blocks = static_cast<int>(std::min<long>((work + 255) / 256, 1024));
  kbwd_finalize_kernel<<<blocks, 256, 0, stream>>>(p.kind, p.D, p.ell_len, p.ell, ncta, p.part_h, p.strips, p.n2,
                                                   gX2 ? p.part_g2 : nullptr, g_ell, g_sigma2, g_noise, gX2);
  count_launch();
  GPB_CUDA_CHECK(cudaGetLastError());
  return GPB_OK;
}

int kern_bwd_mul(int kind, const double* X, int n1, long ldx, const double* X2, int n2, long ldx2, int D,
                 const double* ell, int ell_len, const double* sigma2, const double* G, long ldg, int g_transposed,
                 const double* Mul, long ldm, int symmetric, double* g_ell, double* g_sigma2, double* gX2,
                 void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  if (kind < 0 || kind > KERN_WHITE) return GPB_ERR_BADARG;
  if (!X || !G || !ell || !g_ell || D <= 0 || (ell_len != 1 && ell_len != D)) return GPB_ERR_BADARG;
  if (kind != KERN_LINEAR && !sigma2) return GPB_ERR_BADARG;
  if (kind == KERN_LINEAR && ell_len != D) return GPB_ERR_BADARG;
  if (D > KB_DMAX) return GPB_ERR_UNSUPPORTED;
  KbwdParams p{};
  p.kind = kind;
  p.X1 = X; p.n1 = n1; p.ldx1 = ldx;
  if (X2) { p.X2 = X2; p.n2 = n2; p.ldx2 = ldx2; }
  else { p.X2 = X; p.n2 = n1; p.ldx2 = ldx; }
  if (n1 <= 0 || p.n2 <= 0) return GPB_ERR_BADARG;
  p.D = D; p.ell = ell; p.ell_len = ell_len; p.sigma2 = sigma2;
  p.G = G; p.ldg = ldg; p.g_trans = g_transposed;
  p.Mul = Mul; p.ldm = ldm; p.symmetric = (symmetric || !X2) ? 1 : 0;
  int ncb;
  kbwd_grid(n1, p.n2, false, ncb, p.nrc, p.strips);
  if (!workspace || workspace_bytes < kern_bwd_workspace_bytes(n1, p.n2, D)) return GPB_ERR_BADARG;
  p.part_h = static_cast<double*>(workspace);
  p.part_g2 = gX2 ? p.part_h + static_cast<size_t>(ncb) * p.strips * (D + 2) : nullptr;
  return kbwd_launch<false>(p, ncb, g_ell, g_sigma2, nullptr, gX2, stream);
}

int kern_bwd(int kind, const double* X, int n1, long ldx, const double* X2, int n2, long ldx2, int D,
             const double* ell, int ell_len, const double* sigma2, const double* G, long ldg, int g_transposed,
             double* g_ell, double* g_sigma2, double* gX2, void* workspace, size_t workspace_bytes,
             cudaStream_t stream) {
  if (kind > KERN_PERIODIC) return GPB_ERR_BADARG;
  return kern_bwd_mul(kind, X, n1, ldx, X2, n2, ldx2, D, ell, ell_len, sigma2, G, ldg, g_transposed, nullptr, 0, 0,
                      g_ell, g_sigma2, gX2, workspace, workspace_bytes, stream);
}

size_t gpr_grad_workspace_bytes(int n, int D) {
  int ncb, nrc, strips;
  kbwd_grid(n, n, true, ncb, nrc, strips);
  return static_cast<size_t>(ncb) * strips * (D + 2) * sizeof(double) + 256;
}

// ================================================================================================
// input gradient of the fused GPR loss
// ================================================================================================
// gX_t = sum_s 2 W_ts dK_ts/dx_t with W = 1/2 (dy Kinv - a a^T) formed on the fly from the blocked lower Kinv
// (W_ts = W_st: the pair is read from row max(t, s), column min(t, s)).  One CTA owns 128 target rows (one per thread
// pair, the two halves take alternate source rows) and one chunk of KB_DC feature dimensions (blockIdx.y), and sweeps
// EVERY source row: each pair of the lower triangle is visited twice, once per end, so each target's sum is complete
// inside its CTA and is combined in a fixed order -- no per-CTA partials, no workspace, deterministic.
//   stationary: dK_ts/dx_td = -sigma2 fac1(r2) (x~_td - x~_sd) / ell_d   (the g_ell reduction's fac1; zero below the
//               r2 clamp, gptorch/kernels.py:171-172, so coincident points contribute nothing)
//   Linear:     dK_ts/dx_td = v_d x_sd  (the diagonal pair included: dK_tt/dx_t = 2 v x_t)
template <int KB_DC, int KIND>
__global__ void __launch_bounds__(KB_THREADS, 2) gpr_gx_kernel(const KbwdParams p, double* __restrict__ gX, long ldgx) {
  const int kind = KIND >= 0 ? KIND : p.kind;
  extern __shared__ double kb_smem[];
  const int D = p.D;
  double* Xts = kb_smem;                                   // [D][128] target coordinates (scaled)
  double* Xss = Xts + static_cast<size_t>(D) * KB_COLS;    // [KB_ROWS][D] source coordinates (scaled)
  double* ellv = Xss + static_cast<size_t>(KB_ROWS) * D;   // [D]
  double* at = ellv + D;                                   // [KB_DY][128]
  double* as = at + KB_COLS * KB_DY;                       // [KB_ROWS][KB_DY]
  double* comb = as + KB_ROWS * KB_DY + 32;                // [2][128]

  const int t = threadIdx.x, c = t & 127, half = t >> 7;
  const int c0 = blockIdx.x * KB_COLS;
  const int j = c0 + c;                                    // target row
  const bool jvalid = j < p.n1;
  const int d0 = blockIdx.y * KB_DC;
  const bool linear = kind == KERN_LINEAR;

  for (int d = t; d < D; d += KB_THREADS) ellv[d] = p.ell[p.ell_len == 1 ? 0 : d];
  __syncthreads();
  for (int idx = t; idx < KB_COLS * D; idx += KB_THREADS) {
    const int cc = idx / D, d = idx - cc * D;
    double v = 0.0;
    if (c0 + cc < p.n1) {
      v = p.X1[static_cast<long>(c0 + cc) * p.ldx1 + d];
      if (!linear) v /= ellv[d];
    }
    Xts[d * KB_COLS + cc] = v;
  }
  const double sig2 = linear ? 1.0 : *p.sigma2;

  double acc[KB_DC];
#pragma unroll
  for (int dd = 0; dd < KB_DC; ++dd) acc[dd] = 0.0;

  for (int rc = 0; rc < p.nrc; ++rc) {
    const int i0 = rc * KB_ROWS;
    __syncthreads();
    for (int idx = t; idx < KB_ROWS * D; idx += KB_THREADS) {
      const int rr = idx / D, d = idx - rr * D;
      double v = 0.0;
      if (i0 + rr < p.n1) {
        v = p.X1[static_cast<long>(i0 + rr) * p.ldx1 + d];
        if (!linear) v /= ellv[d];
      }
      Xss[rr * D + d] = v;
    }
    // aa[rr] = sum_o a[s][o] a[t][o], staged in chunks of KB_DY outputs
    double hreg[KB_RT];
#pragma unroll
    for (int rr = 0; rr < KB_RT; ++rr) hreg[rr] = 0.0;
    for (int o0 = 0; o0 < p.dy; o0 += KB_DY) {
      __syncthreads();
      for (int idx = t; idx < KB_COLS * KB_DY; idx += KB_THREADS) {
        const int cc = idx / KB_DY, o = idx - cc * KB_DY;
        at[o * KB_COLS + cc] = (c0 + cc < p.n1 && o0 + o < p.dy) ? p.a[static_cast<long>(c0 + cc) * p.lda + o0 + o] : 0.0;
      }
      for (int idx = t; idx < KB_ROWS * KB_DY; idx += KB_THREADS) {
        const int rr = idx / KB_DY, o = idx - rr * KB_DY;
        as[idx] = (i0 + rr < p.n1 && o0 + o < p.dy) ? p.a[static_cast<long>(i0 + rr) * p.lda + o0 + o] : 0.0;
      }
      __syncthreads();
#pragma unroll
      for (int o = 0; o < KB_DY; ++o) {
        const double aj = at[o * KB_COLS + c];
#pragma unroll
        for (int rr = 0; rr < KB_RT; ++rr) hreg[rr] += as[(half * KB_RT + rr) * KB_DY + o] * aj;
      }
    }
    __syncthreads();

    double r2[KB_RT];
#pragma unroll
    for (int rr = 0; rr < KB_RT; ++rr) r2[rr] = 0.0;
    if (!linear) {
      for (int d = 0; d < D; ++d) {
        const double xt = Xts[d * KB_COLS + c];
#pragma unroll
        for (int rr = 0; rr < KB_RT; ++rr) {
          const double diff = Xss[(half * KB_RT + rr) * D + d] - xt;
          r2[rr] += diff * diff;
        }
      }
    }
#pragma unroll
    for (int rr = 0; rr < KB_RT; ++rr) {
      const int i = i0 + half * KB_RT + rr;
      double h = 0.0;
      if (jvalid && i < p.n1) {
        const int hi = i > j ? i : j, lo = i > j ? j : i;
        const bool same_blk = (hi / NB) == (lo / NB);
        const double kinv = same_blk ? p.kd[static_cast<long>(hi) * NB + (lo - (lo / NB) * NB)]
                                     : p.Kinv[static_cast<long>(hi) * p.ldk + lo];
        const double g = 2.0 * (0.5 * (static_cast<double>(p.dy) * kinv - hreg[rr]));
        if (linear) {
          h = g;
        } else {
          double kbase, fac1;
          kern_base_fac(kind, r2[rr], kbase, fac1);
          h = g * fac1 * sig2;
        }
      }
      hreg[rr] = h;
    }
#pragma unroll
    for (int dd = 0; dd < KB_DC; ++dd) {
      const int d = d0 + dd;
      if (d < D) {
        const double xt = Xts[d * KB_COLS + c];
#pragma unroll
        for (int rr = 0; rr < KB_RT; ++rr) {
          const double xs = Xss[(half * KB_RT + rr) * D + d];
          acc[dd] += linear ? hreg[rr] * xs : hreg[rr] * (xs - xt);
        }
      }
    }
  }

  // the two halves' sums of each target, in a fixed order; then the 1/ell (stationary) or v (Linear) factor
#pragma unroll
  for (int dd = 0; dd < KB_DC; ++dd) {
    const int d = d0 + dd;
    if (d >= D) break;  // uniform across the block
    __syncthreads();
    comb[half * KB_COLS + c] = acc[dd];
    __syncthreads();
    if (half == 0 && jvalid) {
      const double s = comb[c] + comb[KB_COLS + c];
      gX[static_cast<long>(j) * ldgx + d] = linear ? s * ellv[d] : s / ellv[d];
    }
  }
}

template <int DC, int KIND>
static int gpr_gx_launch_kind(const KbwdParams& p, dim3 grid, size_t smem, double* gX, long ldgx, cudaStream_t stream) {
  static std::atomic<int> smem_state[GPB_MAX_DEVICES];
  if (int rc = ensure_dynamic_smem(gpr_gx_kernel<DC, KIND>, static_cast<int>(smem), smem_state)) return rc;
  gpr_gx_kernel<DC, KIND><<<grid, KB_THREADS, smem, stream>>>(p, gX, ldgx);
  count_launch();
  GPB_CUDA_CHECK(cudaGetLastError());
  return GPB_OK;
}

template <int DC>
static int gpr_gx_launch_cfg(const KbwdParams& p, double* gX, long ldgx, cudaStream_t stream) {
  const dim3 grid((p.n1 + KB_COLS - 1) / KB_COLS, (p.D + DC - 1) / DC);
  const size_t smem = kbwd_smem_bytes(p.D);
  switch (p.kind) {
    case KERN_RBF: return gpr_gx_launch_kind<DC, KERN_RBF>(p, grid, smem, gX, ldgx, stream);
    case KERN_EXP: return gpr_gx_launch_kind<DC, KERN_EXP>(p, grid, smem, gX, ldgx, stream);
    case KERN_MATERN32: return gpr_gx_launch_kind<DC, KERN_MATERN32>(p, grid, smem, gX, ldgx, stream);
    case KERN_MATERN52: return gpr_gx_launch_kind<DC, KERN_MATERN52>(p, grid, smem, gX, ldgx, stream);
    case KERN_PERIODIC: return gpr_gx_launch_kind<DC, KERN_PERIODIC>(p, grid, smem, gX, ldgx, stream);
    default: return gpr_gx_launch_kind<DC, -1>(p, grid, smem, gX, ldgx, stream);
  }
}

int gpr_grad(int kind, const double* X, int n, long ldx, int D, const double* ell, int ell_len,
             const double* sigma2, const double* Kinv, long ldk, const double* kdiag_blocks, const double* a,
             int dy, long lda_a, double* g_ell, double* g_sigma2, double* g_noise, void* workspace,
             size_t workspace_bytes, double* gX, long ldgx, cudaStream_t stream) {
  if (kind < 0 || kind > KERN_PERIODIC) return GPB_ERR_BADARG;
  if (!X || !Kinv || !kdiag_blocks || !a || !ell || !g_ell || D <= 0 || n <= 0 || dy <= 0) return GPB_ERR_BADARG;
  if (ell_len != 1 && ell_len != D) return GPB_ERR_BADARG;
  if (kind != KERN_LINEAR && !sigma2) return GPB_ERR_BADARG;
  if (gX && ldgx < D) return GPB_ERR_BADARG;
  if (D > KB_DMAX) return GPB_ERR_UNSUPPORTED;
  KbwdParams p{};
  p.kind = kind;
  p.X1 = X; p.n1 = n; p.ldx1 = ldx;
  p.X2 = X; p.n2 = n; p.ldx2 = ldx;
  p.D = D; p.ell = ell; p.ell_len = ell_len; p.sigma2 = sigma2;
  p.Kinv = Kinv; p.ldk = ldk; p.kd = kdiag_blocks; p.a = a; p.dy = dy; p.lda = lda_a;
  int ncb;
  kbwd_grid(n, n, true, ncb, p.nrc, p.strips);
  if (!workspace || workspace_bytes < gpr_grad_workspace_bytes(n, D)) return GPB_ERR_BADARG;
  p.part_h = static_cast<double*>(workspace);
  p.part_g2 = nullptr;
  const KbwdParams px = p;     // kbwd_launch adapts the strips to its path; the input gradient sweeps whole columns
  if (int rc = kbwd_launch<true>(p, ncb, g_ell, g_sigma2, g_noise, nullptr, stream)) return rc;
  if (!gX) return GPB_OK;
  return D <= 8 ? gpr_gx_launch_cfg<8>(px, gX, ldgx, stream) : gpr_gx_launch_cfg<16>(px, gX, ldgx, stream);
}

}  // namespace gpb
