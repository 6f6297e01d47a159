// gpb_ozaki.cu -- FP64-equivalent C = beta C + alpha A B^T on the INT8 tensor path by integer slicing (Ozaki scheme):
// the split kernels, the driver of both product engines and the library engine.  DESIGN.md section 8; measurements in
// profiles/r02_ozaki_*.txt and profiles/r05_*.json.
//
// Two engines share the split and the workspace.  The default is this library's fused tcgen05 kernel
// (gpb_ozaki_mma.cu: products and recombination in one launch, GPB_I8MMA / gpb_i8mma_config).  The library engine
// described below (GPB_OZAKI / gpb_ozaki_config) takes precedence while switched on; it is the bitwise reference of the
// fused kernel.
//
// Every row of A (m x k) and B (n x k), both K-major, is scaled by a power of two 2^-e_i so that |a| <= 1/2 and cut into
// S signed 7-bit slices, a = 2^e sum_s q_s 2^(-7 (s + 1)), q_s in [-64, 64] (error-free: each remainder is exact in
// fp64).  A B^T = sum_{s,t} 2^(-7 (s + t + 2)) Q^A_s (Q^B_t)^T; the terms with s + t >= S are dropped (they are below
// 2^(-7 S) relative to the row/column scales).  The products of one weight class u = s + t are ONE int8 GEMM over a
// concatenated K: the slices of A are stored side by side in forward order, those of B in reverse order, so that
// [Q^A_0 | .. | Q^A_u] [Q^B_u | .. | Q^B_0]^T is a prefix of the A row times a suffix of the B row -- S GEMMs with
// K' = (u + 1) k, exact in int32 (64 * 64 * S * k < 2^31), instead of S (S + 1) / 2 separate products and as many int32
// matrices to recombine.  The int8 GEMMs are plain library calls (cuBLASLt, loaded with dlopen on first use so that
// the library keeps no link-time dependency); the split and the fp64 recombination are the two kernels below.  C is
// produced in strips of OZ_STRIP rows; with `lower` only the columns up to the strip's diagonal block are computed.
//
// Error model: |dC_ij| <= k 2^(-7 S + 1) max|A_i.| max|B_j.| -- norm-wise like a DGEMM for S = 8 (measured on
// covariance-conditioned operands: tools/ozaki_probe.py), weaker component-wise (DESIGN.md section 8 says why 8 slices
// are the default for the GPR path's products; GPB_I8MMA=0 returns them to the FP64 DMMA engine).
#include "gpb_common.cuh"
#include "gpb_ozaki.cuh"
#include <cublasLt.h>
#include <dlfcn.h>
#include <algorithm>
#include <cfloat>
#include <cstdlib>
#include <map>
#include <mutex>
#include <tuple>

namespace gpb {

constexpr int OZ_BITS = 7;
constexpr int OZ_MAX_SLICES = 10;
constexpr int OZ_STRIP = 2048;
constexpr size_t OZ_LT_WORKSPACE = 64u << 20;

// ------------------------------------------------------------------------------------------------------------------
// cuBLASLt through dlopen
// ------------------------------------------------------------------------------------------------------------------
struct LtApi {
  void* lib = nullptr;
  decltype(&cublasLtCreate) Create = nullptr;
  decltype(&cublasLtMatmulDescCreate) DescCreate = nullptr;
  decltype(&cublasLtMatmulDescDestroy) DescDestroy = nullptr;
  decltype(&cublasLtMatmulDescSetAttribute) DescSet = nullptr;
  decltype(&cublasLtMatrixLayoutCreate) LayoutCreate = nullptr;
  decltype(&cublasLtMatrixLayoutDestroy) LayoutDestroy = nullptr;
  decltype(&cublasLtMatmulPreferenceCreate) PrefCreate = nullptr;
  decltype(&cublasLtMatmulPreferenceDestroy) PrefDestroy = nullptr;
  decltype(&cublasLtMatmulPreferenceSetAttribute) PrefSet = nullptr;
  decltype(&cublasLtMatmulAlgoGetHeuristic) Heuristic = nullptr;
  decltype(&cublasLtMatmul) Matmul = nullptr;
  int status = 0;   // 0 = not tried, 1 = loaded, -1 = unavailable
};

struct OzState {
  cublasLtHandle_t handle = nullptr;
  char* ws = nullptr;
  size_t ws_bytes = 0;
  std::map<std::tuple<int, int, int>, cublasLtMatmulAlgo_t> algos;
};

static std::mutex g_oz_mutex;
static LtApi g_lt;
static std::map<std::pair<int, cudaStream_t>, OzState> g_oz_state;
static std::atomic<int> g_oz_slices{-1};   // -1 = read GPB_OZAKI on first use
static std::atomic<int> g_mma_slices{-1};  // -1 = read GPB_I8MMA on first use

static int lt_load() {
  if (g_lt.status) return g_lt.status > 0 ? GPB_OK : GPB_ERR_UNSUPPORTED;
  const char* names[] = {"libcublasLt.so.12", "libcublasLt.so.13", "libcublasLt.so"};
  for (const char* nm : names) {
    g_lt.lib = dlopen(nm, RTLD_NOW | RTLD_LOCAL);
    if (g_lt.lib) break;
  }
  if (!g_lt.lib) { g_lt.status = -1; return GPB_ERR_UNSUPPORTED; }
  bool ok = true;
#define GPB_LT_SYM(field, name)                                               \
  g_lt.field = reinterpret_cast<decltype(g_lt.field)>(dlsym(g_lt.lib, name)); \
  ok = ok && g_lt.field != nullptr
  GPB_LT_SYM(Create, "cublasLtCreate");
  GPB_LT_SYM(DescCreate, "cublasLtMatmulDescCreate");
  GPB_LT_SYM(DescDestroy, "cublasLtMatmulDescDestroy");
  GPB_LT_SYM(DescSet, "cublasLtMatmulDescSetAttribute");
  GPB_LT_SYM(LayoutCreate, "cublasLtMatrixLayoutCreate");
  GPB_LT_SYM(LayoutDestroy, "cublasLtMatrixLayoutDestroy");
  GPB_LT_SYM(PrefCreate, "cublasLtMatmulPreferenceCreate");
  GPB_LT_SYM(PrefDestroy, "cublasLtMatmulPreferenceDestroy");
  GPB_LT_SYM(PrefSet, "cublasLtMatmulPreferenceSetAttribute");
  GPB_LT_SYM(Heuristic, "cublasLtMatmulAlgoGetHeuristic");
  GPB_LT_SYM(Matmul, "cublasLtMatmul");
#undef GPB_LT_SYM
  g_lt.status = ok ? 1 : -1;
  return ok ? GPB_OK : GPB_ERR_UNSUPPORTED;
}

// C (rows_c x cols_c, column-major, int32) = op_T(A: kk x rows_c, ld lda) * (B: kk x cols_c, ld ldb), int8 operands.
static int lt_gemm_i8(OzState& st, int rows_c, int cols_c, int kk, const int8_t* A, long lda, const int8_t* B, long ldb,
                      int32_t* C, long ldc, void* lt_ws, cudaStream_t stream) {
  cublasLtMatmulDesc_t desc = nullptr;
  cublasLtMatrixLayout_t la = nullptr, lb = nullptr, lc = nullptr;
  int rc = GPB_OK;
  const cublasOperation_t opT = CUBLAS_OP_T, opN = CUBLAS_OP_N;
  if (g_lt.DescCreate(&desc, CUBLAS_COMPUTE_32I, CUDA_R_32I) != CUBLAS_STATUS_SUCCESS) return GPB_ERR_UNSUPPORTED;
  g_lt.DescSet(desc, CUBLASLT_MATMUL_DESC_TRANSA, &opT, sizeof(opT));
  g_lt.DescSet(desc, CUBLASLT_MATMUL_DESC_TRANSB, &opN, sizeof(opN));
  if (g_lt.LayoutCreate(&la, CUDA_R_8I, kk, rows_c, lda) != CUBLAS_STATUS_SUCCESS ||
      g_lt.LayoutCreate(&lb, CUDA_R_8I, kk, cols_c, ldb) != CUBLAS_STATUS_SUCCESS ||
      g_lt.LayoutCreate(&lc, CUDA_R_32I, rows_c, cols_c, ldc) != CUBLAS_STATUS_SUCCESS) {
    rc = GPB_ERR_UNSUPPORTED;
  }
  if (rc == GPB_OK) {
    const auto key = std::make_tuple(rows_c, cols_c, kk);
    auto it = st.algos.find(key);
    if (it == st.algos.end()) {
      cublasLtMatmulPreference_t pref = nullptr;
      cublasLtMatmulHeuristicResult_t res;
      int found = 0;
      size_t wsb = OZ_LT_WORKSPACE;
      if (g_lt.PrefCreate(&pref) != CUBLAS_STATUS_SUCCESS) rc = GPB_ERR_UNSUPPORTED;
      if (rc == GPB_OK) {
        g_lt.PrefSet(pref, CUBLASLT_MATMUL_PREF_MAX_WORKSPACE_BYTES, &wsb, sizeof(wsb));
        if (g_lt.Heuristic(st.handle, desc, la, lb, lc, lc, pref, 1, &res, &found) != CUBLAS_STATUS_SUCCESS || found < 1)
          rc = GPB_ERR_UNSUPPORTED;
        g_lt.PrefDestroy(pref);
      }
      if (rc == GPB_OK) it = st.algos.emplace(key, res.algo).first;
    }
    if (rc == GPB_OK) {
      const int32_t one = 1, zero = 0;
      if (g_lt.Matmul(st.handle, desc, &one, A, la, B, lb, &zero, C, lc, C, lc, &it->second, lt_ws, OZ_LT_WORKSPACE,
                      stream) != CUBLAS_STATUS_SUCCESS)
        rc = GPB_ERR_UNSUPPORTED;      // (library kernels are not counted in gpb::launch_count)
    }
  }
  if (la) g_lt.LayoutDestroy(la);
  if (lb) g_lt.LayoutDestroy(lb);
  if (lc) g_lt.LayoutDestroy(lc);
  if (desc) g_lt.DescDestroy(desc);
  return rc;
}

// ------------------------------------------------------------------------------------------------------------------
// split: one CTA per row
// ------------------------------------------------------------------------------------------------------------------
// tri != 0: the operand is upper triangular BY 128-BLOCKS inside a larger buffer whose other blocks hold unrelated data
// (the factor L): element (row, j) with global position (row0 + row, col0 + j) counts as zero when it lies left of the
// row's diagonal block.  jlo is the first column that is read.
__global__ void __launch_bounds__(256) oz_split_kernel(const double* __restrict__ A, long lda, int k, int S,
                                                       int8_t* __restrict__ fwd, int8_t* __restrict__ rev, long ld8,
                                                       double* __restrict__ scale, int tri, int row0, int col0) {
  __shared__ double red[8];
  __shared__ int bad_s;
  const long row = blockIdx.x;
  const double* a = A + row * lda;
  const int tid = threadIdx.x;
  const int jlo = tri ? max(0, ((row0 + static_cast<int>(row)) / NB) * NB - col0) : 0;   // multiple of 4 (col0 % 4 == 0)
  if (tid == 0) bad_s = 0;
  __syncthreads();
  double mx = 0.0;
  bool bad = false;
  for (int j = jlo + tid; j < k; j += 256) {
    const double v = fabs(a[j]);
    bad = bad || !(v <= DBL_MAX);       // NaN or Inf
    mx = fmax(mx, v);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((tid & 31) == 0) red[tid >> 5] = mx;
  if (bad) bad_s = 1;
  __syncthreads();
  mx = red[0];
#pragma unroll
  for (int w = 1; w < 8; ++w) mx = fmax(mx, red[w]);
  const bool row_bad = bad_s != 0;
  int e = 0;
  if (mx > 0.0 && !row_bad) e = ilogb(mx) + 2;                 // |a| 2^-e < 1/2
  e = max(-1000, min(1000, e));
  if (tid == 0) scale[row] = row_bad ? __longlong_as_double(0x7ff8000000000000LL) : ldexp(1.0, e);
  const double inv = ldexp(1.0, -e);
  const double radix = static_cast<double>(1 << OZ_BITS);
  int8_t* f = fwd ? fwd + row * ld8 : nullptr;
  int8_t* rv = rev ? rev + row * ld8 : nullptr;
  for (int j = tid * 4; j < k; j += 1024) {
    double r[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) r[q] = (row_bad || j < jlo) ? 0.0 : a[j + q] * inv;
    for (int s = 0; s < S; ++s) {
      char4 c;
      signed char qv[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        r[q] *= radix;
        const double t = rint(r[q]);
        r[q] -= t;
        qv[q] = static_cast<signed char>(static_cast<int>(t));
      }
      c.x = qv[0]; c.y = qv[1]; c.z = qv[2]; c.w = qv[3];
      if (f) *reinterpret_cast<char4*>(f + static_cast<long>(s) * k + j) = c;
      if (rv) *reinterpret_cast<char4*>(rv + static_cast<long>(S - 1 - s) * k + j) = c;
    }
  }
}

// Transposed operands (stored k x m, the logical operand is its transpose): column maxima first, then 128 x 32 tiles are
// sliced and transposed through shared memory so that the int8 rows are written in 128-byte runs.
__global__ void __launch_bounds__(256) oz_colmax_kernel(const double* __restrict__ src, long ld, int k, int m,
                                                        double* __restrict__ scale, int tri, int row0, int col0) {
  __shared__ double smx[8][32];
  __shared__ int sbad[8][32];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int col = blockIdx.x * 32 + tx;
  double mx = 0.0;
  int bad = 0;
  if (col < m) {
    for (int r = ty; r < k; r += 8) {
      if (tri && (col0 + col) < ((row0 + r) / NB) * NB) continue;
      const double v = fabs(src[static_cast<long>(r) * ld + col]);
      bad |= !(v <= DBL_MAX);
      mx = fmax(mx, v);
    }
  }
  smx[ty][tx] = mx;
  sbad[ty][tx] = bad;
  __syncthreads();
  if (ty == 0 && col < m) {
#pragma unroll
    for (int w = 1; w < 8; ++w) { mx = fmax(mx, smx[w][tx]); bad |= sbad[w][tx]; }
    int e = 0;
    if (mx > 0.0 && !bad) e = ilogb(mx) + 2;
    e = max(-1000, min(1000, e));
    scale[col] = bad ? __longlong_as_double(0x7ff8000000000000LL) : ldexp(1.0, e);
  }
}

__global__ void __launch_bounds__(256) oz_split_t_kernel(const double* __restrict__ src, long ld, int k, int m, int S,
                                                         int8_t* __restrict__ fwd, int8_t* __restrict__ rev, long ld8,
                                                         const double* __restrict__ scale, int tri, int row0, int col0) {
  __shared__ __align__(4) int8_t sm[OZ_MAX_SLICES][32][132];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int col = blockIdx.x * 32 + tx;
  const int r0 = blockIdx.y * 128;
  const double sc = col < m ? scale[col] : 1.0;
  const bool bad = !(sc == sc);
  const double inv = bad ? 0.0 : 1.0 / sc;                      // exact: sc is a power of two
  const double radix = static_cast<double>(1 << OZ_BITS);
  for (int t = 0; t < 16; ++t) {
    const int rl = ty + 8 * t, r = r0 + rl;
    double v = 0.0;
    if (!bad && col < m && r < k && !(tri && (col0 + col) < ((row0 + r) / NB) * NB))
      v = src[static_cast<long>(r) * ld + col] * inv;
    for (int s = 0; s < S; ++s) {
      v *= radix;
      const double q = rint(v);
      v -= q;
      sm[s][tx][rl] = static_cast<int8_t>(static_cast<int>(q));
    }
  }
  __syncthreads();
  const int w = threadIdx.x & 31;
  for (int rowid = threadIdx.x >> 5; rowid < S * 32; rowid += 8) {
    const int s = rowid >> 5, a = rowid & 31;
    const long c = static_cast<long>(blockIdx.x) * 32 + a;
    const int r = r0 + 4 * w;
    if (c < m && r < k) {
      const int32_t word = *reinterpret_cast<const int32_t*>(&sm[s][a][4 * w]);
      if (fwd) *reinterpret_cast<int32_t*>(fwd + c * ld8 + static_cast<long>(s) * k + r) = word;
      if (rev) *reinterpret_cast<int32_t*>(rev + c * ld8 + static_cast<long>(S - 1 - s) * k + r) = word;
    }
  }
}

// ------------------------------------------------------------------------------------------------------------------
// recombination: C = beta C + alpha sa_i sb_j 2^-14 sum_u P_u 2^(-7 u), four columns per thread
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) oz_recombine_kernel(const int32_t* __restrict__ P, long plane, long ldp, int S,
                                                           int rows, int cols, const double* __restrict__ sa,
                                                           const double* __restrict__ sb, double alpha, double beta,
                                                           double* __restrict__ C, long ldc, int lower, int gi0,
                                                           double* __restrict__ Cdiag) {
  const int j = (blockIdx.x * 256 + threadIdx.x) * 4;
  const int i = blockIdx.y;
  if (j >= cols || i >= rows) return;
  if (lower && (j >> 7) > ((gi0 + i) >> 7)) return;            // whole 4-group lies in one 128-block (j % 4 == 0)
  const bool to_diag = Cdiag != nullptr && (j >> 7) == ((gi0 + i) >> 7);   // gpb_potri_lower's layout: kd[row][col in block]
  const double down = 1.0 / static_cast<double>(1 << OZ_BITS);
  double t[4] = {0.0, 0.0, 0.0, 0.0};
  const int32_t* p = P + static_cast<long>(i) * ldp + j;
  for (int u = S - 1; u >= 0; --u) {                           // Horner from the smallest weight class up
    const int4 v = *reinterpret_cast<const int4*>(p + static_cast<long>(u) * plane);
    t[0] = t[0] * down + static_cast<double>(v.x);
    t[1] = t[1] * down + static_cast<double>(v.y);
    t[2] = t[2] * down + static_cast<double>(v.z);
    t[3] = t[3] * down + static_cast<double>(v.w);
  }
  const double si = alpha * sa[i] * (down * down);
  double* c = to_diag ? Cdiag + static_cast<long>(gi0 + i) * NB + (j & (NB - 1)) : C + static_cast<long>(i) * ldc + j;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    if (j + q < cols) {
      const double val = (si * sb[j + q]) * t[q];
      c[q] = beta == 0.0 ? val : beta * c[q] + val;
    }
  }
}

// ------------------------------------------------------------------------------------------------------------------
// driver
// ------------------------------------------------------------------------------------------------------------------
static inline size_t oz_align(size_t x) { return (x + 255) & ~static_cast<size_t>(255); }

int ozaki_slices() {
  int s = g_oz_slices.load(std::memory_order_relaxed);
  if (s < 0) {
    const char* e = getenv("GPB_OZAKI");
    s = e && *e ? atoi(e) : 0;
    if (s < 0 || s > OZ_MAX_SLICES) s = 0;
    if (s == 1) s = 8;
    g_oz_slices.store(s, std::memory_order_relaxed);
  }
  return s;
}

int i8mma_slices() {
  int s = g_mma_slices.load(std::memory_order_relaxed);
  if (s < 0) {
    const char* e = getenv("GPB_I8MMA");
    s = e && *e ? atoi(e) : OZ_MMA_DEFAULT_SLICES;
    s = (s < 0 || s == 1 || s > OZ_MMA_MAX_SLICES) ? OZ_MMA_DEFAULT_SLICES : s;
    g_mma_slices.store(s, std::memory_order_relaxed);
  }
  return s;
}

int sliced_slices() {
  const int oz = ozaki_slices();
  return oz > 0 ? oz : i8mma_slices();
}

int inverse_slices(int n) {
  if (n & 15) return 0;
  const int oz = ozaki_slices();
  if (oz > 0) return oz;
  return i8mma_slices() > 0 ? OZ_INV_SLICES : 0;
}

// switching a sliced engine off returns the workspaces (hundreds of MB at N = 32768, several GB for the library engine)
// of the current device
static void free_workspaces() {
  std::lock_guard<std::mutex> lock(g_oz_mutex);
  int dev = -1;
  if (cudaGetDevice(&dev) != cudaSuccess) return;
  for (auto& kv : g_oz_state) {
    if (kv.first.first != dev || !kv.second.ws) continue;
    cudaDeviceSynchronize();
    cudaFree(kv.second.ws);
    kv.second.ws = nullptr;
    kv.second.ws_bytes = 0;
  }
}

void ozaki_set_slices(int s) {
  s = (s < 0 || s > OZ_MAX_SLICES) ? 0 : (s == 1 ? 8 : s);     // 1 = "on" = 8 slices, as for GPB_OZAKI
  g_oz_slices.store(s, std::memory_order_relaxed);
  if (s == 0) free_workspaces();
}

void i8mma_set_slices(int s) {
  s = (s == 1 || s > OZ_MMA_MAX_SLICES) ? OZ_MMA_DEFAULT_SLICES : s;
  g_mma_slices.store(s, std::memory_order_relaxed);
  if (s == 0) free_workspaces();
}

int gemm_ozaki_nt(int m, int n, int k, double alpha, const double* A, long lda, const double* B, long ldb, double beta,
                  double* C, long ldc, int lower, int slices, cudaStream_t stream) {
  OzEx x;
  x.m = m; x.n = n; x.k = k; x.alpha = alpha; x.A = A; x.lda = lda; x.B = B; x.ldb = ldb; x.beta = beta;
  x.C = C; x.ldc = ldc; x.lower = lower; x.slices = slices; x.stream = stream;
  return gemm_ozaki_nt_ex(x);
}

int gemm_ozaki_nt_ex(const OzEx& x) {
  const int m = x.m, n = x.n, k = x.k, lower = x.lower, slices = x.slices;
  const double alpha = x.alpha, beta = x.beta;
  const double *A = x.A, *B = x.B;
  double* C = x.C;
  const long lda = x.lda, ldb = x.ldb, ldc = x.ldc;
  cudaStream_t stream = x.stream;
  if (m <= 0 || n <= 0) return GPB_OK;
  if (!A || !B || !C || k <= 0 || lda < (x.a_trans ? m : k) || ldb < (x.b_trans ? n : k) || ldc < n) return GPB_ERR_BADARG;
  if (slices < 2 || slices > OZ_MAX_SLICES) return GPB_ERR_BADARG;
  // shapes the int8 path takes (everything else stays on the DMMA engine)
  if ((k & 15) || (m & 3) || (n & 3) || (ldc & 1)) return GPB_ERR_UNSUPPORTED;
  if ((x.a_tri && (x.a_col0 & 3)) || (x.b_tri && (x.b_col0 & 3)) || (x.gi0 & 3)) return GPB_ERR_UNSUPPORTED;
  if (static_cast<long long>(k) * slices * 4096 >= (1LL << 31)) return GPB_ERR_UNSUPPORTED;
  if (lower && x.gi0 == 0 && x.Cdiag == nullptr && m != n) return GPB_ERR_BADARG;
  // the library engine while GPB_OZAKI / gpb_ozaki_config asks for it, this library's fused kernel otherwise
  const bool native = ozaki_slices() == 0;
  std::lock_guard<std::mutex> lock(g_oz_mutex);
  int rc = GPB_OK;
  int dev = 0;
  GPB_CUDA_CHECK(cudaGetDevice(&dev));
  OzState& st = g_oz_state[std::make_pair(dev, stream)];
  if (!native) {
    rc = lt_load();
    if (rc) return rc;
    if (!st.handle && g_lt.Create(&st.handle) != CUBLAS_STATUS_SUCCESS) return GPB_ERR_UNSUPPORTED;
  }

  const int S = slices;
  const bool same = (A == B && lda == ldb && m == n && !x.a_trans && !x.b_trans && x.a_tri == x.b_tri &&
                     x.a_row0 == x.b_row0 && x.a_col0 == x.b_col0);
  const long ld8 = static_cast<long>(S) * k;
  const int strip = OZ_STRIP;
  const long ldp = (static_cast<long>(n) + 15) & ~15L;
  const long plane = static_cast<long>(strip) * ldp;
  // workspace: the slices and the scales; the library engine adds its int32 class planes and its own workspace.  The
  // fused kernel reads B in the forward slice order, so for A A^T it reads A's slices twice instead of a second copy.
  size_t off = 0;
  const size_t o_a8 = off;   off += oz_align(static_cast<size_t>(m) * ld8);
  const size_t o_b8 = off;   off += (native && same) ? 0 : oz_align(static_cast<size_t>(n) * ld8);
  const size_t o_sa = off;   off += oz_align(static_cast<size_t>(m) * sizeof(double));
  const size_t o_sb = off;   off += oz_align(static_cast<size_t>(n) * sizeof(double));
  const size_t o_p = off;    off += native ? 0 : oz_align(static_cast<size_t>(S) * plane * sizeof(int32_t));
  const size_t o_lt = off;   off += native ? 0 : OZ_LT_WORKSPACE;
  if (off > st.ws_bytes) {
    // a stream being captured into a CUDA graph cannot allocate: such products stay on the DMMA engine
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    GPB_CUDA_CHECK(cudaStreamIsCapturing(stream, &cap));
    if (cap != cudaStreamCaptureStatusNone) return GPB_ERR_UNSUPPORTED;
    if (st.ws) {
      GPB_CUDA_CHECK(cudaStreamSynchronize(stream));
      GPB_CUDA_CHECK(cudaFree(st.ws));
      st.ws = nullptr;
      st.ws_bytes = 0;
    }
    GPB_CUDA_CHECK(cudaMalloc(&st.ws, off));
    st.ws_bytes = off;
  }
  int8_t* a8 = reinterpret_cast<int8_t*>(st.ws + o_a8);
  int8_t* b8 = (native && same) ? a8 : reinterpret_cast<int8_t*>(st.ws + o_b8);
  double* sa = reinterpret_cast<double*>(st.ws + o_sa);
  double* sb = same ? sa : reinterpret_cast<double*>(st.ws + o_sb);
  // B's slices: forward order for the fused kernel, reverse order for the library's concatenated-k products
  int8_t* b_fwd = native ? b8 : nullptr;
  int8_t* b_rev = native ? nullptr : b8;

  if (x.a_trans) {
    oz_colmax_kernel<<<(m + 31) / 32, 256, 0, stream>>>(A, lda, k, m, sa, x.a_tri, x.a_row0, x.a_col0);
    oz_split_t_kernel<<<dim3((m + 31) / 32, (k + 127) / 128), 256, 0, stream>>>(A, lda, k, m, S, a8, nullptr, ld8, sa, x.a_tri,
                                                                               x.a_row0, x.a_col0);
    count_launch(2);
  } else {
    oz_split_kernel<<<m, 256, 0, stream>>>(A, lda, k, S, a8, (same && !native) ? b8 : nullptr, ld8, sa, x.a_tri, x.a_row0,
                                           x.a_col0);
    count_launch();
  }
  if (x.b_trans) {
    oz_colmax_kernel<<<(n + 31) / 32, 256, 0, stream>>>(B, ldb, k, n, sb, x.b_tri, x.b_row0, x.b_col0);
    oz_split_t_kernel<<<dim3((n + 31) / 32, (k + 127) / 128), 256, 0, stream>>>(B, ldb, k, n, S, b_fwd, b_rev, ld8, sb, x.b_tri,
                                                                               x.b_row0, x.b_col0);
    count_launch(2);
  } else if (!same) {
    oz_split_kernel<<<n, 256, 0, stream>>>(B, ldb, k, S, b_fwd, b_rev, ld8, sb, x.b_tri, x.b_row0, x.b_col0);
    count_launch();
  }
  GPB_CUDA_CHECK(cudaGetLastError());

  if (native) return ozaki_mma_launch(x, a8, b8, sa, sb);

  void* lt_ws = st.ws + o_lt;
  int32_t* P = reinterpret_cast<int32_t*>(st.ws + o_p);
  for (int i0 = 0; i0 < m; i0 += strip) {
    const int rows = std::min(strip, m - i0);
    int cols = n;
    if (lower) cols = std::min(n, ((x.gi0 + i0 + rows + NB - 1) / NB) * NB);
    for (int u = 0; u < S; ++u) {
      const int kk = (u + 1) * k;
      rc = lt_gemm_i8(st, cols, rows, kk, b8 + static_cast<long>(S - 1 - u) * k, ld8, a8 + static_cast<long>(i0) * ld8, ld8,
                      P + static_cast<long>(u) * plane, ldp, lt_ws, stream);
      // "not taken, use the DMMA engine instead" is only a valid answer while C is untouched: once a strip has been
      // recombined into C (beta may be 1) a library failure is a hard error, not a fallback
      if (rc) return (rc == GPB_ERR_UNSUPPORTED && i0 > 0) ? GPB_ERR_DRIVER : rc;
    }
    dim3 grid((cols + 1023) / 1024, rows);
    oz_recombine_kernel<<<grid, 256, 0, stream>>>(P, plane, ldp, S, rows, cols, sa + i0, sb, alpha, beta,
                                                  C + static_cast<long>(i0) * ldc, ldc, lower, x.gi0 + i0, x.Cdiag);
    count_launch();
  }
  GPB_CUDA_CHECK(cudaGetLastError());
  return GPB_OK;
}

}  // namespace gpb
