// gpb_chol.cu -- blocked FP64 Cholesky, triangular inverse and (L L^T)^-1 on the DMMA GEMM engine.
//
// Replaces torch.cholesky / torch.cholesky_inverse behind gptorch/functions.py:46-54 and the O(N^3) part of
// autograd's CholeskyBackward0 in the GPR loss gradient (SURVEY 8a rows F2, F5, M2).
//
// All matrices are row-major, LOWER storage.  Everything O(n^3) is expressed as NT / TN GEMMs on 128-aligned
// sub-blocks addressed through ONE whole-buffer TMA tensor map, so a recursion step is just new coordinates:
//
//   potrf(A):   A11 = L11 L11^T (recurse) ; A21 <- A21 L11^-T (right TRSM, recursive, base case = NT GEMM with
//               the explicit inverse of a 128x128 diagonal block) ; A22 -= A21 A21^T (SYRK, lower tiles) ;
//               recurse on A22.  The 128x128 diagonal blocks are factored AND inverted in shared memory by
//               one CTA (diag_block_kernel); the inverses are kept in `dinv` for every later solve.
//   potri(L):   T = L^-T is built in the UPPER triangle of the same buffer, level by level (all sub-problems
//               of one size are batched in one launch):  P^T = T22^T L21 (TN, triangular k-range),
//               T12 = -T11 P  (NT, triangular k-range).  Then Kinv = T T^T (NT, k >= row-tile) is written
//               to the strictly-lower blocks; diagonal blocks go to a side buffer because the diagonal
//               blocks of T are still being read by other CTAs.
#include "gpb_gemm.cuh"
#include "gpb_ozaki.cuh"
#include <vector>
#include <map>
#include <mutex>
#include <utility>
#include <cstdlib>
#include <algorithm>
#include <algorithm>

namespace gpb {

void set_last_error_msg(const char* msg);

// ================================================================================================
// 128 x 128 diagonal block: Cholesky + inverse in shared memory (one CTA, on the critical path)
// ================================================================================================
// Blocked on 16 x 16 sub-blocks.  Per sub-block: warp 0 factors it and inverts it in REGISTERS (lane i owns
// row i; pivots and columns travel by shuffles; rsqrt() replaces sqrt + divide and doubles as 1/L_kk for the
// inverse), then all 16 warps apply the panel solve and the rank-16 trailing update with DMMA on fragments
// read straight from shared memory (row stride 132 doubles: conflict free).  The inverse of the whole block
// follows from the 16 x 16 inverses by block forward substitution, again on DMMA:  M_ik = I_ii L_ik, then
// X_ij = -sum_{k=j}^{i-1} M_ik X_kj level by level (i - j = 1..7).
constexpr int DG_THREADS = 512;
constexpr int DG_LD = 132;   // 132 mod 16 == 4
constexpr int DG_SB = 16;    // sub-block
constexpr int DG_NSB = NB / DG_SB;
constexpr int DG_ILD = 20;   // row stride of the 16 x 16 inverse blocks (20 mod 16 == 4)
constexpr int DG_SMEM_BYTES = (NB * DG_LD + DG_NSB * DG_SB * DG_ILD) * 8 + 16;

// Warp-level Cholesky of a 16x16 block held one row per lane (lanes >= 16 carry zeros), in place; rs[k] =
// 1/L_kk.  `bad` returns the first column (0-based) with a non-positive / NaN pivot, or -1.
__device__ __forceinline__ void warp_potrf16(double (&a)[DG_SB], double (&rs)[DG_SB], int lane, int& bad) {
  bad = -1;
#pragma unroll
  for (int k = 0; k < DG_SB; ++k) {
    const double dk = __shfl_sync(0xffffffffu, a[k], k);
    if (!(dk > 0.0) && bad < 0) bad = k;
    const double r = rsqrt(dk);
    rs[k] = r;
    if (lane == k) a[k] = dk * r;
    else if (lane > k) a[k] *= r;
    const double lk = a[k];
#pragma unroll
    for (int j = 0; j < DG_SB; ++j) {
      if (j > k) {
        const double ljk = __shfl_sync(0xffffffffu, lk, j);
        if (lane >= j) a[j] -= lk * ljk;
      }
    }
  }
}

// Inverse of the lower-triangular 16x16 block held one row per lane: lane c ends with column c in x[].
__device__ __forceinline__ void warp_trtri16(const double (&a)[DG_SB], const double (&rs)[DG_SB], double (&x)[DG_SB],
                                             int lane) {
#pragma unroll
  for (int i = 0; i < DG_SB; ++i) x[i] = (i == lane) ? rs[i] : 0.0;
#pragma unroll
  for (int i = 1; i < DG_SB; ++i) {
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < DG_SB; ++k) {
      if (k < i) {
        const double lik = __shfl_sync(0xffffffffu, a[k], i);   // L[i][k]
        s += lik * x[k];
      }
    }
    if (i > lane) x[i] = -rs[i] * s;
  }
}

// blockIdx.x selects the diagonal block; A0 points at element (0,0) of the matrix; j_first is the index of
// the first diagonal block handled by this launch.
__global__ void __launch_bounds__(DG_THREADS, 1)
diag_block_kernel(double* __restrict__ A0, long lda, int n, double* __restrict__ dinv, int* info, int j_first,
                  int do_factor) {
  extern __shared__ double dg_smem[];
  double* S = dg_smem;                     // [128][132]
  double* Ib = S + NB * DG_LD;             // [8][16][20]: inverses of the diagonal 16x16 sub-blocks
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int r8 = lane >> 2, kk = lane & 3;
  const int j0 = (j_first + blockIdx.x) * NB;
  const int nb = min(NB, n - j0);
  double* A = A0 + static_cast<long>(j0) * lda + j0;
  double* dinv_blk = dinv + static_cast<long>(j0) * NB;

  for (int idx = t; idx < NB * NB; idx += DG_THREADS) {
    const int r = idx >> 7, c = idx & 127;
    double v = 0.0;
    if (c <= r) {
      if (r < nb) v = A[static_cast<long>(r) * lda + c];
      else v = (r == c) ? 1.0 : 0.0;
    }
    S[r * DG_LD + c] = v;
  }
  __syncthreads();

  for (int b = 0; b < DG_NSB; ++b) {
    const int o = b * DG_SB;
    // ---- (a) one warp: factor + invert the 16x16 diagonal sub-block in registers --------------------
    if (warp == 0) {
      double a[DG_SB], rs[DG_SB], x[DG_SB];
#pragma unroll
      for (int j = 0; j < DG_SB; ++j) a[j] = (lane < DG_SB && j <= lane) ? S[(o + lane) * DG_LD + o + j] : 0.0;
      if (do_factor) {
        int bad;
        warp_potrf16(a, rs, lane, bad);
        if (bad >= 0 && lane == 0 && o + bad < nb) atomicCAS(info, 0, j0 + o + bad + 1);
        if (lane < DG_SB) {
#pragma unroll
          for (int j = 0; j < DG_SB; ++j)
            if (j <= lane) S[(o + lane) * DG_LD + o + j] = a[j];
        }
      } else {
#pragma unroll
        for (int k = 0; k < DG_SB; ++k) rs[k] = 1.0 / __shfl_sync(0xffffffffu, a[k], k);
      }
      warp_trtri16(a, rs, x, lane);
      if (lane < DG_SB) {
#pragma unroll
        for (int i = 0; i < DG_SB; ++i) Ib[(b * DG_SB + i) * DG_ILD + lane] = x[i];
      }
    }
    if (!do_factor) continue;   // inverse-only: the sub-block inverses are all that phase 1 provides
    __syncthreads();
    const int R0 = o + DG_SB;
    // ---- (b) panel: rows below the sub-block  <-  rows * I_bb^T  (strips of 8 rows, one per warp) ------
    for (int strip = warp; strip < (NB - R0) / 8; strip += DG_THREADS / 32) {
      const int row = R0 + 8 * strip + r8;
      double af[4], acc[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) af[ks] = S[row * DG_LD + o + 4 * ks + kk];
#pragma unroll
      for (int jn = 0; jn < 2; ++jn)
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
          const double bf = Ib[(b * DG_SB + 8 * jn + r8) * DG_ILD + 4 * ks + kk];
          dmma884(acc[jn][0], acc[jn][1], af[ks], bf);
        }
      // the strip is rewritten in place by the lanes of this warp: every lane's operand loads precede the warp-collective
      // DMMA, the barrier makes that ordering explicit (compute-sanitizer racecheck: WAR between lanes otherwise)
      __syncwarp();
#pragma unroll
      for (int jn = 0; jn < 2; ++jn) {
        S[row * DG_LD + o + 8 * jn + 2 * kk] = acc[jn][0];
        S[row * DG_LD + o + 8 * jn + 2 * kk + 1] = acc[jn][1];
      }
    }
    __syncthreads();
    // ---- (c) trailing update: lower 8x8 tiles of S[R0:, R0:] -= P P^T, K = 16 -------------------------
    {
      const int T = (NB - R0) / 8;
      const int ntile = T * (T + 1) / 2;
      for (int tile = warp; tile < ntile; tile += DG_THREADS / 32) {
        int ti = static_cast<int>((sqrtf(8.0f * tile + 1.0f) - 1.0f) * 0.5f);
        while ((ti + 1) * (ti + 2) / 2 <= tile) ++ti;
        while (ti * (ti + 1) / 2 > tile) --ti;
        const int tj = tile - ti * (ti + 1) / 2;
        double acc0 = 0.0, acc1 = 0.0;
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
          const double af = S[(R0 + 8 * ti + r8) * DG_LD + o + 4 * ks + kk];
          const double bf = S[(R0 + 8 * tj + r8) * DG_LD + o + 4 * ks + kk];
          dmma884(acc0, acc1, af, bf);
        }
        double* c = &S[(R0 + 8 * ti + r8) * DG_LD + R0 + 8 * tj + 2 * kk];
        c[0] -= acc0;
        c[1] -= acc1;
      }
    }
    __syncthreads();
  }
  __syncthreads();

  if (do_factor) {
    for (int idx = t; idx < NB * NB; idx += DG_THREADS) {
      const int r = idx >> 7, c = idx & 127;
      if (r < nb && c <= r) A[static_cast<long>(r) * lda + c] = S[r * DG_LD + c];
    }
  }

  // ---- phase 2: X = L^-1 from the sub-block inverses ----------------------------------------------------
  // step A: M_ik = I_ii L_ik for every strictly-lower 16x16 block (28 blocks x 4 tiles of 8x8), in place.
  {
    constexpr int NTILE = (DG_NSB * (DG_NSB - 1) / 2) * 4;   // 112
    double m0[NTILE / 16], m1[NTILE / 16];
#pragma unroll
    for (int q = 0; q < NTILE / 16; ++q) {
      const int tile = warp + 16 * q;
      const int blk = tile >> 2, tm = (tile >> 1) & 1, tn = tile & 1;
      int bi = static_cast<int>((sqrtf(8.0f * blk + 1.0f) - 1.0f) * 0.5f);
      while ((bi + 1) * (bi + 2) / 2 <= blk) ++bi;
      while (bi * (bi + 1) / 2 > blk) --bi;
      const int bk = blk - bi * (bi + 1) / 2;
      const int i = bi + 1;   // block row 1..7, block col bk 0..i-1
      double acc0 = 0.0, acc1 = 0.0;
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        const double af = Ib[(i * DG_SB + 8 * tm + r8) * DG_ILD + 4 * ks + kk];
        const double bf = S[(i * DG_SB + 4 * ks + kk) * DG_LD + bk * DG_SB + 8 * tn + r8];
        dmma884(acc0, acc1, af, bf);
      }
      m0[q] = acc0;
      m1[q] = acc1;
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < NTILE / 16; ++q) {
      const int tile = warp + 16 * q;
      const int blk = tile >> 2, tm = (tile >> 1) & 1, tn = tile & 1;
      int bi = static_cast<int>((sqrtf(8.0f * blk + 1.0f) - 1.0f) * 0.5f);
      while ((bi + 1) * (bi + 2) / 2 <= blk) ++bi;
      while (bi * (bi + 1) / 2 > blk) --bi;
      const int bk = blk - bi * (bi + 1) / 2;
      const int i = bi + 1;
      double* c = &S[(i * DG_SB + 8 * tm + r8) * DG_LD + bk * DG_SB + 8 * tn + 2 * kk];
      c[0] = m0[q];
      c[1] = m1[q];
    }
    __syncthreads();
  }
  // levels d = i - j: X_ij = -sum_{k=j}^{i-1} M_ik X_kj, with X_jj = I_jj and X_kj (k > j) kept at the mirrored
  // (upper) block position S[16 j + . ][16 k + . ].
  for (int d = 1; d < DG_NSB; ++d) {
    const int ntile = (DG_NSB - d) * 4;
    for (int tile = warp; tile < ntile; tile += DG_THREADS / 32) {
      const int j = tile >> 2, tm = (tile >> 1) & 1, tn = tile & 1;
      const int i = j + d;
      double acc0 = 0.0, acc1 = 0.0;
      for (int k = j; k < i; ++k) {
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
          const double af = S[(i * DG_SB + 8 * tm + r8) * DG_LD + k * DG_SB + 4 * ks + kk];   // M_ik
          const double bf = (k == j) ? Ib[(j * DG_SB + 4 * ks + kk) * DG_ILD + 8 * tn + r8]
                                     : S[(j * DG_SB + 4 * ks + kk) * DG_LD + k * DG_SB + 8 * tn + r8];  // X_kj
          dmma884(acc0, acc1, af, bf);
        }
      }
      double* c = &S[(j * DG_SB + 8 * tm + r8) * DG_LD + i * DG_SB + 8 * tn + 2 * kk];
      c[0] = -acc0;
      c[1] = -acc1;
    }
    __syncthreads();
  }

  for (int idx = t; idx < NB * NB; idx += DG_THREADS) {
    const int r = idx >> 7, c = idx & 127;
    const int bi = r >> 4, bj = c >> 4;
    double v = 0.0;
    if (bi == bj) v = Ib[(bi * DG_SB + (r & 15)) * DG_ILD + (c & 15)];
    else if (bi > bj) v = S[(bj * DG_SB + (r & 15)) * DG_LD + bi * DG_SB + (c & 15)];
    dinv_blk[r * NB + c] = v;
  }
}

static int launch_diag_blocks(double* A0, long lda, int n, double* dinv, int* info, int j_first, int nblocks,
                              int do_factor, cudaStream_t stream) {
  static std::atomic<int> smem_state[GPB_MAX_DEVICES];
  if (int rc = ensure_dynamic_smem(diag_block_kernel, DG_SMEM_BYTES, smem_state)) return rc;
  diag_block_kernel<<<nblocks, DG_THREADS, DG_SMEM_BYTES, stream>>>(A0, lda, n, dinv, info, j_first, do_factor);
  count_launch();
  GPB_CUDA_CHECK(cudaGetLastError());
  return GPB_OK;
}

// ================================================================================================
// potrf driver
// ================================================================================================
struct CholCtx {
  double* A;
  long lda;
  int n;
  double* dinv;
  int* info;
  CUtensorMap mapA128;   // whole buffer, box rows 128
  CUtensorMap mapD128;   // dinv [npad x 128], box rows 128
  cudaStream_t stream;
};

static inline int split_point(int n) {
  // first part: floor(half of the 128-blocks) * 128  (>= 128 because n > 128)
  const int nblk = (n + NB - 1) / NB;
  return (nblk / 2) * NB;
}

// X[r0:r0+m, c0:c0+n] <- X * L[c0:c0+n, c0:c0+n]^-T
static int trsm_right_rec(CholCtx& c, int r0, int m, int c0, int n) {
  if (m <= 0 || n <= 0) return GPB_OK;
  if (n <= NB) {
    GemmArgs g;
    g.M = m; g.N = n; g.K = NB;
    g.alpha = 1.0; g.beta = 0.0;
    g.C = c.A + static_cast<long>(r0) * c.lda + c0;
    g.ldc = c.lda;
    g.ax = c0; g.ay = r0;
    g.bx = 0; g.by = c0;
    g.flags = GF_ROWS_INPLACE;
    return gemm_launch(GEMM_NT, c.mapA128, c.mapD128, g, c.stream);
  }
  const int n1 = split_point(n), n2 = n - n1;
  int rc = trsm_right_rec(c, r0, m, c0, n1);
  if (rc) return rc;
  GemmArgs g;
  g.M = m; g.N = n2; g.K = n1;
  g.alpha = -1.0; g.beta = 1.0;
  g.C = c.A + static_cast<long>(r0) * c.lda + c0 + n1;
  g.ldc = c.lda;
  g.ax = c0; g.ay = r0;
  g.bx = c0; g.by = c0 + n1;
  rc = gemm_launch(GEMM_NT, c.mapA128, c.mapA128, g, c.stream);
  if (rc) return rc;
  return trsm_right_rec(c, r0, m, c0 + n1, n2);
}

static int potrf_rec(CholCtx& c, int j0, int n) {
  if (n <= 0) return GPB_OK;
  if (n <= NB) return launch_diag_blocks(c.A, c.lda, c.n, c.dinv, c.info, j0 / NB, 1, 1, c.stream);
  const int n1 = split_point(n), n2 = n - n1;
  int rc = potrf_rec(c, j0, n1);
  if (rc) return rc;
  rc = trsm_right_rec(c, j0 + n1, n2, j0, n1);
  if (rc) return rc;
  GemmArgs g;
  g.M = n2; g.N = n2; g.K = n1;
  g.alpha = -1.0; g.beta = 1.0;
  g.C = c.A + static_cast<long>(j0 + n1) * c.lda + (j0 + n1);
  g.ldc = c.lda;
  g.ax = j0; g.ay = j0 + n1;
  g.bx = j0; g.by = j0 + n1;
  g.flags = GF_LOWER_TILES;
  rc = gemm_launch(GEMM_NT, c.mapA128, c.mapA128, g, c.stream);
  if (rc) return rc;
  return potrf_rec(c, j0 + n1, n2);
}

static inline long npad128(long n) { return (n + NB - 1) / NB * NB; }

// ---- look-ahead driver ---------------------------------------------------------------------------------
// For large n the factorisation is organised in column panels of LA_PANEL columns.  The latency-bound work
// (recursive factorisation of the panel's diagonal block, its TRSM) runs on a high-priority side stream
// while the bulk trailing update of the PREVIOUS panel still occupies the chip on the caller's stream:
//
//   S0 (caller)  : ... 3a(p): update cols of panel p+1 | 3b(p): update everything right of panel p+1 | 3a(p+1) ...
//   S1 (priority):                                     | potrf(diag p+1), trsm(panel p+1)            |
//
// 3b(p) only reads panel p and writes columns right of panel p+1, S1 only touches the columns of panel p+1.
constexpr int LA_PANEL = 2048;
constexpr int LA_MIN_N = 3072;

struct AuxStream {
  cudaStream_t stream = nullptr;
  cudaEvent_t ev_panel = nullptr, ev_update = nullptr, ev_fork = nullptr;
  int device = -1;
};

// One side stream + event set per (device, caller stream): two factorisations issued on different caller streams of the
// same device never share events, and the table itself is guarded (the library may be called from several host threads).
static int get_aux(cudaStream_t caller, AuxStream** out) {
  static std::mutex mu;
  static std::map<std::pair<int, cudaStream_t>, AuxStream> table;
  int dev = 0;
  GPB_CUDA_CHECK(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(mu);
  AuxStream& a = table[std::make_pair(dev, caller)];
  if (a.stream == nullptr) {
    int lo = 0, hi = 0;
    GPB_CUDA_CHECK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    GPB_CUDA_CHECK(cudaStreamCreateWithPriority(&a.stream, cudaStreamNonBlocking, hi));
    GPB_CUDA_CHECK(cudaEventCreateWithFlags(&a.ev_panel, cudaEventDisableTiming));
    GPB_CUDA_CHECK(cudaEventCreateWithFlags(&a.ev_update, cudaEventDisableTiming));
    GPB_CUDA_CHECK(cudaEventCreateWithFlags(&a.ev_fork, cudaEventDisableTiming));
    a.device = dev;
  }
  *out = &a;
  return GPB_OK;
}

// Large trailing updates on the INT8 tensor path (gpb_ozaki.cu: the fused tcgen05 kernel by default, GPB_I8MMA=0 turns it
// off).  Shapes that path does not take fall through to the DMMA engine.
static int syrk_update(CholCtx& c, int r0, int m, int k0, int k) {
  // A[r0:r0+m, r0:r0+m] (lower tiles) -= P P^T with P = A[r0:r0+m, k0:k0+k]
  if (const int oz = sliced_slices(); oz > 0 && m >= OZ_MIN_ROWS && k >= OZ_MIN_K) {
    const double* P = c.A + static_cast<long>(r0) * c.lda + k0;
    const int rc = gemm_ozaki_nt(m, m, k, -1.0, P, c.lda, P, c.lda, 1.0, c.A + static_cast<long>(r0) * c.lda + r0, c.lda, 1,
                                 oz, c.stream);
    if (rc != GPB_ERR_UNSUPPORTED) return rc;
  }
  GemmArgs g;
  g.M = m; g.N = m; g.K = k;
  g.alpha = -1.0; g.beta = 1.0;
  g.C = c.A + static_cast<long>(r0) * c.lda + r0;
  g.ldc = c.lda;
  g.ax = k0; g.ay = r0;
  g.bx = k0; g.by = r0;
  g.flags = GF_LOWER_TILES;
  return gemm_launch(GEMM_NT, c.mapA128, c.mapA128, g, c.stream);
}

// Panel schedule: widths (multiples of the 128 block) of the look-ahead panels; the last entry is the tail, which is
// factored by the plain recursion once the trailing matrix is too small for a bulk update to hide the panel chain.
// GPB_LA_PANEL / GPB_LA_FIRST / GPB_LA_TAIL override the defaults (tuning aid; read once).
static int env_int(const char* name, int fallback) {
  const char* v = getenv(name);
  if (!v || !*v) return fallback;
  const int x = atoi(v);
  return x > 0 ? (x + NB - 1) / NB * NB : fallback;
}

static void panel_schedule(int n, std::vector<int>& starts) {
  // measured on B200 (tools/bench_potrf.py sweeps, profiles/r02_potrf_panel_sweep.txt): narrow panels win while the
  // trailing updates are short (n = 8192: 512 columns 10.7 ms vs 2048 columns 12.7 ms vs plain recursion 13.4 ms), wide
  // panels once the k-length of the trailing GEMMs dominates (n = 32768: 2048 columns 354 ms, 1024 columns 357 ms)
  int def = n <= 16384 ? 512 : (n <= 24576 ? 1024 : LA_PANEL);
  // int8-sliced products: they run the bulk updates so much faster than the panel chain that wide panels pay earlier
  // (library engine, n = 16384, 8 slices: 512 columns 49.6 ms, 1024 columns 43.9 ms, 2048 columns 39.5 ms; n = 32768 flat)
  if (sliced_slices() > 0 && n >= 12288) def = LA_PANEL;
  static const int w_env = env_int("GPB_LA_PANEL", 0), first_env = env_int("GPB_LA_FIRST", 0),
                   tail_env = env_int("GPB_LA_TAIL", 0);
  const int w = w_env ? w_env : def, first = first_env ? first_env : w, tail = tail_env ? tail_env : w;
  starts.clear();
  int c = 0;
  starts.push_back(0);
  c = std::min(first, n);
  while (n - c > tail) {
    starts.push_back(c);
    c += w;
  }
  if (c < n) starts.push_back(c);
  starts.push_back(n);
}

static int potrf_lookahead(CholCtx& c) {
  AuxStream* aux = nullptr;
  int rc = get_aux(c.stream, &aux);
  if (rc) return rc;
  const cudaStream_t s0 = c.stream, s1 = aux->stream;
  const int n = c.n;
  std::vector<int> st;
  panel_schedule(n, st);
  const int np = static_cast<int>(st.size()) - 1;     // panels [st[p], st[p+1])
  GPB_CUDA_CHECK(cudaEventRecord(aux->ev_fork, s0));
  GPB_CUDA_CHECK(cudaStreamWaitEvent(s1, aux->ev_fork, 0));
  // panel 0
  c.stream = s1;
  rc = potrf_rec(c, 0, st[1]);
  if (rc) return rc;
  if (st[1] < n) {
    rc = trsm_right_rec(c, st[1], n - st[1], 0, st[1]);
    if (rc) return rc;
  }
  GPB_CUDA_CHECK(cudaEventRecord(aux->ev_panel, s1));
  for (int p = 0; p + 1 < np; ++p) {
    const int c0 = st[p], w = st[p + 1] - st[p];
    const int c1 = st[p + 1];
    const int w1 = st[p + 2] - c1;
    const int c2 = c1 + w1;
    GPB_CUDA_CHECK(cudaStreamWaitEvent(s0, aux->ev_panel, 0));
    // 3a: bring the columns of the next panel up to date
    c.stream = s0;
    rc = syrk_update(c, c1, w1, c0, w);
    if (rc) return rc;
    if (c2 < n) {
      GemmArgs g;
      g.M = n - c2; g.N = w1; g.K = w;
      g.alpha = -1.0; g.beta = 1.0;
      g.C = c.A + static_cast<long>(c2) * c.lda + c1;
      g.ldc = c.lda;
      g.ax = c0; g.ay = c2;
      g.bx = c0; g.by = c1;
      rc = GPB_ERR_UNSUPPORTED;
      if (const int oz = sliced_slices(); oz > 0 && g.M >= OZ_MIN_ROWS && g.N >= OZ_MIN_COLS && g.K >= OZ_MIN_K)
        rc = gemm_ozaki_nt(g.M, g.N, g.K, -1.0, c.A + static_cast<long>(c2) * c.lda + c0, c.lda,
                           c.A + static_cast<long>(c1) * c.lda + c0, c.lda, 1.0, g.C, c.lda, 0, oz, s0);
      if (rc == GPB_ERR_UNSUPPORTED) rc = gemm_launch(GEMM_NT, c.mapA128, c.mapA128, g, s0);
      if (rc) return rc;
    }
    GPB_CUDA_CHECK(cudaEventRecord(aux->ev_update, s0));
    // side stream: factor the next panel while 3b runs
    GPB_CUDA_CHECK(cudaStreamWaitEvent(s1, aux->ev_update, 0));
    c.stream = s1;
    rc = potrf_rec(c, c1, w1);
    if (rc) return rc;
    if (c2 < n) {
      rc = trsm_right_rec(c, c2, n - c2, c1, w1);
      if (rc) return rc;
    }
    GPB_CUDA_CHECK(cudaEventRecord(aux->ev_panel, s1));
    // 3b: the rest of the trailing matrix
    c.stream = s0;
    if (c2 < n) {
      rc = syrk_update(c, c2, n - c2, c0, w);
      if (rc) return rc;
    }
  }
  GPB_CUDA_CHECK(cudaStreamWaitEvent(s0, aux->ev_panel, 0));
  c.stream = s0;
  return GPB_OK;
}

int potrf_lower(double* A, int n, long lda, double* dinv, int* info, cudaStream_t stream) {
  if (n <= 0) return GPB_OK;
  if (!A || !dinv || !info || lda < n) return GPB_ERR_BADARG;
  CholCtx c;
  c.A = A; c.lda = lda; c.n = n; c.dinv = dinv; c.info = info; c.stream = stream;
  int rc = make_tmap_f64(&c.mapA128, A, n, n, lda, 32);
  if (rc) return rc;
  rc = make_tmap_f64(&c.mapD128, dinv, npad128(n), NB, NB, 32);
  if (rc) return rc;
  static const int la_min = env_int("GPB_LA_MIN_N", LA_MIN_N);
  if (n >= la_min) return potrf_lookahead(c);
  return potrf_rec(c, 0, n);
}

int trsm_right_lt(const double* L, int n, long ldl, const double* dinv, double* X, int m, long ldx,
                  cudaStream_t stream);

// ================================================================================================
// right-side solve on a separate panel X (m x n):  X <- X L^-T
// ================================================================================================
struct TrsmCtx {
  double* X; long ldx; int m;
  CUtensorMap mapX128, mapL128, mapD128;
  cudaStream_t stream;
};

static int trsm_panel_rec(TrsmCtx& c, int c0, int n) {
  if (n <= 0) return GPB_OK;
  if (n <= NB) {
    GemmArgs g;
    g.M = c.m; g.N = n; g.K = NB;
    g.alpha = 1.0; g.beta = 0.0;
    g.C = c.X + c0; g.ldc = c.ldx;
    g.ax = c0; g.ay = 0;
    g.bx = 0; g.by = c0;
    g.flags = GF_ROWS_INPLACE;
    return gemm_launch(GEMM_NT, c.mapX128, c.mapD128, g, c.stream);
  }
  const int n1 = split_point(n), n2 = n - n1;
  int rc = trsm_panel_rec(c, c0, n1);
  if (rc) return rc;
  GemmArgs g;
  g.M = c.m; g.N = n2; g.K = n1;
  g.alpha = -1.0; g.beta = 1.0;
  g.C = c.X + c0 + n1; g.ldc = c.ldx;
  g.ax = c0; g.ay = 0;
  g.bx = c0; g.by = c0 + n1;
  rc = gemm_launch(GEMM_NT, c.mapX128, c.mapL128, g, c.stream);
  if (rc) return rc;
  return trsm_panel_rec(c, c0 + n1, n2);
}

int trsm_right_lt(const double* L, int n, long ldl, const double* dinv, double* X, int m, long ldx,
                  cudaStream_t stream) {
  if (n <= 0 || m <= 0) return GPB_OK;
  if (!L || !dinv || !X || ldl < n || ldx < n) return GPB_ERR_BADARG;
  TrsmCtx c;
  c.X = X; c.ldx = ldx; c.m = m; c.stream = stream;
  int rc = make_tmap_f64(&c.mapX128, X, m, n, ldx, 32);
  if (rc) return rc;
  rc = make_tmap_f64(&c.mapL128, L, n, n, ldl, 32);
  if (rc) return rc;
  rc = make_tmap_f64(&c.mapD128, dinv, npad128(n), NB, NB, 32);
  if (rc) return rc;
  return trsm_panel_rec(c, 0, n);
}

int tri_diag_inverse(const double* L, int n, long ldl, double* dinv, cudaStream_t stream) {
  if (n <= 0) return GPB_OK;
  if (!L || !dinv || ldl < n) return GPB_ERR_BADARG;
  const int nblk = (n + NB - 1) / NB;
  return launch_diag_blocks(const_cast<double*>(L), ldl, n, dinv, nullptr, 0, nblk, 0, stream);
}

// ================================================================================================
// potri: T = L^-T in the upper triangle, then Kinv = T T^T
// ================================================================================================
// Base case: diagonal block j of the buffer <- transpose(dinv block j) (upper triangular, zeros below).
__global__ void __launch_bounds__(256) tinv_base_kernel(double* __restrict__ A, long lda, int n,
                                                        const double* __restrict__ dinv) {
  __shared__ double tile[32][33];
  const int j0 = blockIdx.z * NB;
  const int bx = blockIdx.x * 32, by = blockIdx.y * 32;  // output tile: rows by.., cols bx.. inside the block
  const double* D = dinv + static_cast<long>(j0) * NB;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  // read dinv[(bx + i)][by + tx] -> tile[i][tx]   (transposed source tile)
  for (int i = ty; i < 32; i += 8) tile[i][tx] = D[(bx + i) * NB + by + tx];
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const int r = by + i, c = bx + tx;  // output (r, c) = dinv[c][r], upper triangular
    if (j0 + r < n && j0 + c < n) {
      const double v = (c >= r) ? tile[tx][i] : 0.0;
      A[static_cast<long>(j0 + r) * lda + j0 + c] = v;
    }
  }
}

size_t potri_workspace_bytes(int n) {
  // P^T scratch: max over levels s of (#problems at the level) * s * s doubles.
  size_t best = 0;
  for (long s = NB; s < n; s *= 2) {
    long nprob = (n + 2 * s - 1) / (2 * s);
    best = std::max(best, static_cast<size_t>(nprob) * s * s);
  }
  return best * sizeof(double) + 256;
}

// T = L^-T into the upper triangle of A (diagonal 128-blocks are overwritten by T_jj with zeros below the
// diagonal; the strictly-lower off-diagonal blocks keep L).
int trtri_upper(double* A, int n, long lda, const double* dinv, void* workspace, size_t workspace_bytes,
                cudaStream_t stream) {
  if (n <= 0) return GPB_OK;
  if (!A || !dinv || lda < n) return GPB_ERR_BADARG;
  if (workspace_bytes < potri_workspace_bytes(n) || (n > NB && !workspace)) return GPB_ERR_BADARG;
  const int nblk = (n + NB - 1) / NB;
  {
    dim3 grid(NB / 32, NB / 32, nblk);
    tinv_base_kernel<<<grid, 256, 0, stream>>>(A, lda, n, dinv);
    count_launch();
    GPB_CUDA_CHECK(cudaGetLastError());
  }
  CUtensorMap mapA128, mapA16;
  int rc = make_tmap_f64(&mapA128, A, n, n, lda, 32);
  if (rc) return rc;
  rc = make_tmap_f64(&mapA16, A, n, n, lda, 16);
  if (rc) return rc;
  double* W = static_cast<double*>(workspace);

  for (long s = NB; s < n; s *= 2) {
    // problems p = 0.. : block [p*2s, p*2s + 2s): T11 = first s, T22 = next n2 = min(s, n - p*2s - s) (> 0)
    const int nfull = static_cast<int>(n / (2 * s));              // problems with n2 == s
    const long rem = n - static_cast<long>(nfull) * 2 * s;        // leftover rows after the full problems
    const int n2_last = rem > s ? static_cast<int>(rem - s) : 0;  // ragged problem (n2 < s) if any
    CUtensorMap mapW128;
    const int nprob = nfull + (n2_last > 0 ? 1 : 0);
    if (nprob == 0) continue;
    rc = make_tmap_f64(&mapW128, W, static_cast<long>(nprob) * s, s, s, 32);
    if (rc) return rc;
    for (int pass = 0; pass < 2; ++pass) {
      const int batch = pass == 0 ? nfull : (n2_last > 0 ? 1 : 0);
      if (batch == 0) continue;
      const int p0 = pass == 0 ? 0 : nfull;
      const int n2 = pass == 0 ? static_cast<int>(s) : n2_last;
      const int off = static_cast<int>(p0 * 2 * s);
      // (1) P^T[n2 x s] = T22^T L21        TN, A = T22 (k <= m: GF_KHI_M), B = L21
      GemmArgs g1;
      g1.M = n2; g1.N = static_cast<int>(s); g1.K = n2;
      g1.alpha = 1.0; g1.beta = 0.0;
      g1.C = W + static_cast<long>(p0) * s * s; g1.ldc = s; g1.c_batch = s * s;
      g1.ax = off + static_cast<int>(s); g1.ay = off + static_cast<int>(s);
      g1.bx = off; g1.by = off + static_cast<int>(s);
      g1.dax = g1.day = g1.dbx = g1.dby = static_cast<int>(2 * s);
      g1.flags = GF_KHI_M;
      g1.batch = batch;
      rc = GPB_ERR_UNSUPPORTED;
      if (const int oz = inverse_slices(n); oz > 0 && pass == 0 && s >= OZ_TRTRI_MIN_S) {
        // int8-sliced path (inverse_slices, see potri_lower): rows [a0, a0 + R) of P^T only involve rows 0 .. a0 + R
        // of T22 and L21; both operands are stored with the contraction index as the row, so the split transposes them
        rc = GPB_OK;
        for (int pb = 0; pb < batch && rc == GPB_OK; ++pb) {
          const long o2 = off + static_cast<long>(pb) * 2 * s;
          for (int a0 = 0; a0 < n2 && rc == GPB_OK; a0 += OZ_TRI_STRIP) {
            const int rows = std::min(OZ_TRI_STRIP, n2 - a0);
            OzEx x;
            x.m = rows; x.n = static_cast<int>(s); x.k = a0 + rows;
            x.A = A + (o2 + s) * lda + o2 + s + a0; x.lda = lda; x.a_trans = 1; x.a_tri = 1; x.a_row0 = 0; x.a_col0 = a0;
            x.B = A + (o2 + s) * lda + o2; x.ldb = lda; x.b_trans = 1;
            x.C = W + static_cast<long>(p0 + pb) * s * s + static_cast<long>(a0) * s; x.ldc = s;
            x.slices = oz; x.stream = stream;
            rc = gemm_ozaki_nt_ex(x);
          }
        }
      }
      if (rc == GPB_ERR_UNSUPPORTED) rc = gemm_launch(GEMM_TN, mapA16, mapA16, g1, stream);
      if (rc) return rc;
      // (2) T12[s x n2] = -T11 (P^T)^T     NT, A = T11 (k >= m: GF_KLO_M), B = P^T (n2 x s)
      GemmArgs g2;
      g2.M = static_cast<int>(s); g2.N = n2; g2.K = static_cast<int>(s);
      g2.alpha = -1.0; g2.beta = 0.0;
      g2.C = A + static_cast<long>(off) * lda + off + s; g2.ldc = lda; g2.c_batch = 2 * s * (lda + 1);
      g2.ax = off; g2.ay = off;
      g2.dax = g2.day = static_cast<int>(2 * s);
      g2.bx = 0; g2.by = static_cast<int>(p0 * s);
      g2.dbx = 0; g2.dby = static_cast<int>(s);
      g2.flags = GF_KLO_M;
      g2.batch = batch;
      rc = GPB_ERR_UNSUPPORTED;
      if (const int oz = inverse_slices(n); oz > 0 && pass == 0 && s >= OZ_TRTRI_MIN_S) {
        // int8-sliced path, per problem and per row strip of T11 (entries from the strip's first column on)
        rc = GPB_OK;
        for (int pb = 0; pb < batch && rc == GPB_OK; ++pb) {
          const long o2 = off + static_cast<long>(pb) * 2 * s;
          for (int i0 = 0; i0 < s && rc == GPB_OK; i0 += OZ_TRI_STRIP) {
            const int rows = std::min<long>(OZ_TRI_STRIP, s - i0);
            OzEx x;
            x.m = rows; x.n = n2; x.k = static_cast<int>(s) - i0;
            x.alpha = -1.0; x.beta = 0.0;
            x.A = A + (o2 + i0) * lda + o2 + i0; x.lda = lda; x.a_tri = 1; x.a_row0 = i0; x.a_col0 = i0;
            x.B = W + static_cast<long>(p0 + pb) * s * s + i0; x.ldb = s;
            x.C = A + (o2 + i0) * lda + o2 + s; x.ldc = lda;
            x.slices = oz; x.stream = stream;
            rc = gemm_ozaki_nt_ex(x);
          }
        }
      }
      if (rc == GPB_ERR_UNSUPPORTED) rc = gemm_launch(GEMM_NT, mapA128, mapW128, g2, stream);
      if (rc) return rc;
    }
  }
  return GPB_OK;
}

int potri_lower(double* A, int n, long lda, const double* dinv, double* kdiag_blocks, void* workspace,
                size_t workspace_bytes, cudaStream_t stream) {
  if (n <= 0) return GPB_OK;
  if (!kdiag_blocks) return GPB_ERR_BADARG;
  int rc = trtri_upper(A, n, lda, dinv, workspace, workspace_bytes, stream);
  if (rc) return rc;
  CUtensorMap mapA128;
  rc = make_tmap_f64(&mapA128, A, n, n, lda, 32);
  if (rc) return rc;
  // Kinv = T T^T: strictly-lower blocks in place, diagonal blocks to kdiag_blocks.
  // The inverse's products (the two trtri_upper hooks and this one) are int8-sliced at inverse_slices(n): 9 slices on
  // the default fused engine, one more than the factor's.  Ky^-1 feeds sums that cancel (the GPR gradient's
  // tr(Ky^-1 dK), the predictive variance), which amplify the products' norm-wise error.  Measured on B200 with the
  // inverse sliced at 8: N = 16384 variance gradient 1.4e-7 from the reference (tolerance 1e-7), N = 32768
  // Ky^-1 (Ky v) - v 1.5e-8 (tolerance 1e-8); at 9 slices 6e-10 and 1.3e-10 (DESIGN.md section 8).
  if (const int oz = inverse_slices(n); oz > 0 && n >= OZ_MIN_ROWS) {
    // int8-sliced path: row strip [i0, i0 + R) of T only has entries from column i0 on, so its product with the rows
    // 0 .. i0 + R runs over k in [i0, n) -- one independent sliced product per strip, no flop on the zero triangle
    rc = GPB_OK;
    for (int i0 = 0; i0 < n && rc == GPB_OK; i0 += OZ_TRI_STRIP) {
      const int rows = std::min(OZ_TRI_STRIP, n - i0);
      OzEx x;
      x.m = rows; x.n = i0 + rows; x.k = n - i0;
      x.A = A + static_cast<long>(i0) * lda + i0; x.lda = lda; x.a_tri = 1; x.a_row0 = i0; x.a_col0 = i0;
      x.B = A + i0; x.ldb = lda; x.b_tri = 1; x.b_row0 = 0; x.b_col0 = i0;
      x.C = A + static_cast<long>(i0) * lda; x.ldc = lda;
      x.lower = 1; x.gi0 = i0; x.Cdiag = kdiag_blocks;
      x.slices = oz; x.stream = stream;
      rc = gemm_ozaki_nt_ex(x);
    }
    if (rc != GPB_ERR_UNSUPPORTED) return rc;     // (a decline leaves T intact: the DMMA product below recomputes every block)
  }
  GemmArgs g;
  g.M = n; g.N = n; g.K = n;
  g.alpha = 1.0; g.beta = 0.0;
  g.C = A; g.ldc = lda;
  g.Cdiag = kdiag_blocks; g.ldd = NB;
  g.flags = GF_LOWER_TILES | GF_KLO_M | GF_DIAG_TO_WS;
  return gemm_launch(GEMM_NT, mapA128, mapA128, g, stream);
}

// out (full symmetric) <- blocked potri result
__global__ void __launch_bounds__(256) potri_assemble_kernel(const double* __restrict__ A, long lda, int n,
                                                             const double* __restrict__ kd, double* __restrict__ out,
                                                             long ldo) {
  __shared__ double tile[32][33];
  const int bi = blockIdx.y, bj = blockIdx.x;  // 32 x 32 tiles; only bj <= bi launched usefully
  if (bj > bi) return;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int r0 = bi * 32, c0 = bj * 32;
  const bool diag_blk = (r0 / NB) == (c0 / NB);
  for (int i = ty; i < 32; i += 8) {
    const int r = r0 + i, c = c0 + tx;
    double v = 0.0;
    if (r < n && c < n) v = diag_blk ? kd[static_cast<long>(r) * NB + (c - (c0 / NB) * NB)] : A[static_cast<long>(r) * lda + c];
    tile[i][tx] = v;
    if (r < n && c < n) out[static_cast<long>(r) * ldo + c] = v;
  }
  __syncthreads();
  if (bi != bj) {
    for (int i = ty; i < 32; i += 8) {
      const int r = c0 + i, c = r0 + tx;  // mirrored position
      if (r < n && c < n) out[static_cast<long>(r) * ldo + c] = tile[tx][i];
    }
  }
}

int potri_assemble(const double* A, int n, long lda, const double* kd, double* out, long ldo, cudaStream_t stream) {
  if (n <= 0) return GPB_OK;
  const int nt = (n + 31) / 32;
  dim3 grid(nt, nt);
  potri_assemble_kernel<<<grid, 256, 0, stream>>>(A, lda, n, kd, out, ldo);
  count_launch();
  GPB_CUDA_CHECK(cudaGetLastError());
  return GPB_OK;
}

}  // namespace gpb
