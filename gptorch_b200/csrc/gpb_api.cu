// gpb_api.cu -- the extern "C" boundary of libgpb200.so (declared in include/gpb200.h).
#include "gpb_gemm.cuh"
#include "gpb_ozaki.cuh"
#include <map>
#include <mutex>
#include <utility>
#include <algorithm>
#include "../../include/gpb200.h"
#include "../../include/gpb200_posterior.h"
#include "../../include/gpb200_i8mma.h"

namespace gpb {
const char* last_error();
void set_last_error_msg(const char* msg);
int potrf_lower(double* A, int n, long lda, double* dinv, int* info, cudaStream_t stream);
int trsm_right_lt(const double* L, int n, long ldl, const double* dinv, double* X, int m, long ldx, cudaStream_t stream);
int tri_diag_inverse(const double* L, int n, long ldl, double* dinv, cudaStream_t stream);
int gemm_ozaki_nt(int m, int n, int k, double alpha, const double* A, long lda, const double* B, long ldb, double beta,
                  double* C, long ldc, int lower, int slices, cudaStream_t stream);
int ozaki_slices();
void ozaki_set_slices(int s);
int i8mma_slices();
void i8mma_set_slices(int s);
size_t potri_workspace_bytes(int n);
int potri_lower(double* A, int n, long lda, const double* dinv, double* kdiag_blocks, void* workspace,
                size_t workspace_bytes, cudaStream_t stream);
int potri_assemble(const double* A, int n, long lda, const double* kd, double* out, long ldo, cudaStream_t stream);
int trtri_upper(double* A, int n, long lda, const double* dinv, void* workspace, size_t workspace_bytes,
                cudaStream_t stream);
size_t trsv_workspace_bytes(int n);
int trsv_lower(const double* L, int n, long ldl, const double* dinv, double* B, int k, long ldb, int trans,
               void* workspace, size_t workspace_bytes, cudaStream_t stream);
size_t gemv_t_workspace_bytes(long rows, int cols);
int gemv_t(const double* A, long rows, int cols, long lda, const double* Y, int dy, long ldy, double beta, double* out,
           long ldo, void* workspace, size_t workspace_bytes, cudaStream_t stream);
int logdet_sumsq(const double* L, int n, long ldl, const double* V, int vrows, int k, long ldv, double* out,
                 cudaStream_t stream);
int rowdot(const double* A, long lda, const double* B, long ldb, long rows, int cols, double alpha, double beta,
           double* out, cudaStream_t stream);
int gemv_n(const double* A, long rows, int cols, long lda, const double* V, int dy, long ldv, double* out, long ldo,
           cudaStream_t stream);
int rows_scale_add_outer(double* A, long rows, int cols, long lda, const double* s, double scale, const double* G, int dy,
                         long ldg, const double* V, long ldv, cudaStream_t stream);
int tri_zero_upper(double* A, int n, long lda, cudaStream_t stream);
int add_diag(double* A, int n, long lda, const double* value, double host_value, cudaStream_t stream);
int kern_fwd(int kind, const double* X, int n1, long ldx, const double* X2, int n2, long ldx2, int D,
             const double* ell, int ell_len, const double* sigma2, const double* noise, int fill, double* K,
             long ldk, cudaStream_t stream);
size_t kern_bwd_workspace_bytes(int n1, int n2, int D);
int kern_bwd(int kind, const double* X, int n1, long ldx, const double* X2, int n2, long ldx2, int D,
             const double* ell, int ell_len, const double* sigma2, const double* G, long ldg, int g_transposed,
             double* g_ell, double* g_sigma2, double* gX2, void* workspace, size_t workspace_bytes,
             cudaStream_t stream);
int kern_bwd_mul(int kind, const double* X, int n1, long ldx, const double* X2, int n2, long ldx2, int D,
                 const double* ell, int ell_len, const double* sigma2, const double* G, long ldg, int g_transposed,
                 const double* Mul, long ldm, int symmetric, double* g_ell, double* g_sigma2, double* gX2,
                 void* workspace, size_t workspace_bytes, cudaStream_t stream);
int kern_sop_fwd(int n_terms, const int* term_len, const int* leaf_kind, const double* const* leaf_ell,
                 const int* leaf_ell_len, const double* const* leaf_sigma2, const double* X, int n1, long ldx,
                 const double* X2, int n2, long ldx2, int D, const double* noise, int fill, double* K, long ldk,
                 cudaStream_t stream);
int linear_kdiag(const double* X, int n, long ldx, int D, const double* v, double* out, cudaStream_t stream);
size_t gpr_grad_workspace_bytes(int n, int D);
int gpr_grad(int kind, const double* X, int n, long ldx, int D, const double* ell, int ell_len,
             const double* sigma2, const double* Kinv, long ldk, const double* kdiag_blocks, const double* a,
             int dy, long lda_a, double* g_ell, double* g_sigma2, double* g_noise, void* workspace,
             size_t workspace_bytes, double* gX, long ldgx, cudaStream_t stream);
int pred_gx(int kind, const double* Xs, int ns, long ldxs, const double* X, int n, long ldx, int D, const double* ell,
            int ell_len, const double* sigma2, const double* a, int dy, long lda, const double* g_mean, long ldgm,
            const double* g_var, const double* Q, long ldq, double* gXs, long ldgx, cudaStream_t stream);
}  // namespace gpb

using namespace gpb;
static inline cudaStream_t S(void* s) { return static_cast<cudaStream_t>(s); }

// FP64 tensor-pipe issue-rate probe: every warp issues independent DMMA.8x8x4 chains from registers, nothing else.
// This is the ceiling the GEMM engine is measured against (bench.py roofline.peak).
__global__ void __launch_bounds__(512) dmma_issue_probe_kernel(double* out, int iters) {
  double c[8][2];
  double a = threadIdx.x * 1e-9, b = 1.0 + threadIdx.x * 1e-9;
#pragma unroll
  for (int i = 0; i < 8; i++) { c[i][0] = i; c[i][1] = -i; }
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int i = 0; i < 8; i++) dmma884_ordered(c[i][0], c[i][1], a, b);
  }
  double s = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) s += c[i][0] + c[i][1];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

// ---- helpers of the streamed Kuf statistics (gpb_kuf_stats_fwd / _bwd) ------------------------------------------------
constexpr int KUF_SPLITS = 16;   // k-slices of the streamed Gram product: the M x M output alone has too few tiles for 148 SMs

// Phi[i][j] = sum_s slots[s][max(i,j)][min(i,j)]: sum the split-K slots (lower tiles valid) and mirror to a full matrix
__global__ void kuf_reduce_sym_kernel(const double* __restrict__ slots, int splits, int m, long ldm, long slot_stride,
                                      double* __restrict__ Phi, long ldphi) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
  if (j >= m) return;
  const int r = i > j ? i : j, c = i > j ? j : i;
  double s = 0.0;
  for (int q = 0; q < splits; ++q) s += slots[q * slot_stride + static_cast<long>(r) * ldm + c];
  Phi[static_cast<long>(i) * ldphi + j] = s;
}

__global__ void kuf_accumulate_kernel(double* __restrict__ dst, const double* __restrict__ src, long count) {
  const long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < count) dst[i] += src[i];
}

static inline size_t kuf_align(size_t b) { return (b + 255) / 256 * 256; }

// Two-stage software pipeline over the row chunks: the tensor-pipe-bound GEMM stage of chunk c runs on the caller's
// stream while the covariance build (forward) or the covariance backward (adjoint) of a neighbouring chunk runs on a
// high-priority side stream, double-buffered.  One side stream + event set per (device, caller stream).
struct KufAux {
  cudaStream_t side = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr, ready[2] = {nullptr, nullptr}, free_[2] = {nullptr, nullptr};
};

static int kuf_aux(cudaStream_t caller, KufAux** out) {
  static std::mutex mu;
  static std::map<std::pair<int, cudaStream_t>, KufAux> table;
  int dev = 0;
  GPB_CUDA_CHECK(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(mu);
  KufAux& a = table[std::make_pair(dev, caller)];
  if (a.side == nullptr) {
    int lo = 0, hi = 0;
    GPB_CUDA_CHECK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    GPB_CUDA_CHECK(cudaStreamCreateWithPriority(&a.side, cudaStreamNonBlocking, hi));
    cudaEvent_t* evs[] = {&a.fork, &a.join, &a.ready[0], &a.ready[1], &a.free_[0], &a.free_[1]};
    for (cudaEvent_t* e : evs) GPB_CUDA_CHECK(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
  }
  *out = &a;
  return GPB_OK;
}
static inline int kuf_k_per_split(int rows) {
  const int per = (rows + KUF_SPLITS - 1) / KUF_SPLITS;
  return std::max(16, (per + 15) / 16 * 16);
}

#pragma GCC visibility push(default)
extern "C" {

int gpb_version(void) { return 105; }
const char* gpb_last_error(void) { return last_error(); }
int gpb_block_size(void) { return NB; }
long gpb_launch_count(void) { return launch_count(); }
int gpb_dmma_issue_probe(int iters, double* scratch, size_t scratch_bytes, double* flop_out, void* stream) {
  int dev = 0, sms = 0;
  GPB_CUDA_CHECK(cudaGetDevice(&dev));
  GPB_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int blocks = 2 * sms, threads = 512;
  if (iters <= 0 || scratch == nullptr || scratch_bytes < sizeof(double) * blocks * threads) return GPB_ERR_BADARG;
  dmma_issue_probe_kernel<<<blocks, threads, 0, S(stream)>>>(scratch, iters);
  GPB_CUDA_CHECK(cudaGetLastError());
  count_launch();
  if (flop_out) *flop_out = (double)blocks * (threads / 32) * (double)iters * 8.0 * (8 * 8 * 4 * 2.0);
  return GPB_OK;
}
void gpb_reset_launch_count(void) { reset_launch_count(); }

int gpb_kern_fwd(int kind, const double* X, int n1, long ldx, const double* X2, int n2, long ldx2, int D,
                 const double* ell, int ell_len, const double* sigma2, const double* noise, int fill, double* K,
                 long ldk, void* stream) {
  return kern_fwd(kind, X, n1, ldx, X2, n2, ldx2, D, ell, ell_len, sigma2, noise, fill, K, ldk, S(stream));
}
size_t gpb_kern_bwd_workspace_bytes(int n1, int n2, int D) { return kern_bwd_workspace_bytes(n1, n2, D); }
int gpb_kern_bwd(int kind, const double* X, int n1, long ldx, const double* X2, int n2, long ldx2, int D,
                 const double* ell, int ell_len, const double* sigma2, const double* G, long ldg, int g_transposed,
                 double* g_ell, double* g_sigma2, double* gX2, void* workspace, size_t workspace_bytes,
                 void* stream) {
  return kern_bwd(kind, X, n1, ldx, X2, n2, ldx2, D, ell, ell_len, sigma2, G, ldg, g_transposed, g_ell, g_sigma2,
                  gX2, workspace, workspace_bytes, S(stream));
}
int gpb_kern_bwd_mul(int kind, const double* X, int n1, long ldx, const double* X2, int n2, long ldx2, int D,
                     const double* ell, int ell_len, const double* sigma2, const double* G, long ldg,
                     int g_transposed, const double* Mul, long ldm, int symmetric, double* g_ell, double* g_sigma2,
                     double* gX2, void* workspace, size_t workspace_bytes, void* stream) {
  return kern_bwd_mul(kind, X, n1, ldx, X2, n2, ldx2, D, ell, ell_len, sigma2, G, ldg, g_transposed, Mul, ldm,
                      symmetric, g_ell, g_sigma2, gX2, workspace, workspace_bytes, S(stream));
}
int gpb_kern_sop_fwd(int n_terms, const int* term_len, const int* leaf_kind, const double* const* leaf_ell,
                     const int* leaf_ell_len, const double* const* leaf_sigma2, const double* X, int n1, long ldx,
                     const double* X2, int n2, long ldx2, int D, const double* noise, int fill, double* K, long ldk,
                     void* stream) {
  return kern_sop_fwd(n_terms, term_len, leaf_kind, leaf_ell, leaf_ell_len, leaf_sigma2, X, n1, ldx, X2, n2, ldx2, D,
                      noise, fill, K, ldk, S(stream));
}
int gpb_linear_kdiag(const double* X, int n, long ldx, int D, const double* v, double* out, void* stream) {
  return linear_kdiag(X, n, ldx, D, v, out, S(stream));
}

int gpb_potrf_lower(double* A, int n, long lda, double* dinv, int* info, void* stream) {
  return potrf_lower(A, n, lda, dinv, info, S(stream));
}
int gpb_tri_diag_inverse(const double* L, int n, long ldl, double* dinv, void* stream) {
  return tri_diag_inverse(L, n, ldl, dinv, S(stream));
}
size_t gpb_potri_workspace_bytes(int n) { return potri_workspace_bytes(n); }
int gpb_potri_lower(double* A, int n, long lda, const double* dinv, double* kdiag_blocks, void* workspace,
                    size_t workspace_bytes, void* stream) {
  return potri_lower(A, n, lda, dinv, kdiag_blocks, workspace, workspace_bytes, S(stream));
}
int gpb_trtri_upper(double* A, int n, long lda, const double* dinv, void* workspace, size_t workspace_bytes,
                    void* stream) {
  return trtri_upper(A, n, lda, dinv, workspace, workspace_bytes, S(stream));
}
int gpb_potri_assemble(const double* A, int n, long lda, const double* kdiag_blocks, double* out, long ldo,
                       void* stream) {
  return potri_assemble(A, n, lda, kdiag_blocks, out, ldo, S(stream));
}
int gpb_tri_zero_upper(double* A, int n, long lda, void* stream) { return tri_zero_upper(A, n, lda, S(stream)); }
int gpb_add_diag(double* A, int n, long lda, const double* value, double host_value, void* stream) {
  return add_diag(A, n, lda, value, host_value, S(stream));
}

size_t gpb_trsv_workspace_bytes(int n) { return trsv_workspace_bytes(n); }
int gpb_trsv_lower(const double* L, int n, long ldl, const double* dinv, double* B, int k, long ldb, int trans,
                   void* workspace, size_t workspace_bytes, void* stream) {
  return trsv_lower(L, n, ldl, dinv, B, k, ldb, trans, workspace, workspace_bytes, S(stream));
}
int gpb_trsm_right_lt(const double* L, int n, long ldl, const double* dinv, double* X, int m, long ldx,
                      void* stream) {
  return trsm_right_lt(L, n, ldl, dinv, X, m, ldx, S(stream));
}
int gpb_logdet_sumsq(const double* L, int n, long ldl, const double* V, int vrows, int k, long ldv, double* out,
                     void* stream) {
  return logdet_sumsq(L, n, ldl, V, vrows, k, ldv, out, S(stream));
}

int gpb_rowdot(const double* A, long lda, const double* B, long ldb, long rows, int cols, double alpha, double beta,
               double* out, void* stream) {
  return rowdot(A, lda, B, ldb, rows, cols, alpha, beta, out, S(stream));
}
int gpb_gemv_n(const double* A, long rows, int cols, long lda, const double* V, int dy, long ldv, double* out, long ldo,
               void* stream) {
  return gemv_n(A, rows, cols, lda, V, dy, ldv, out, ldo, S(stream));
}
int gpb_rows_scale_add_outer(double* A, long rows, int cols, long lda, const double* s, double scale, const double* G,
                             int dy, long ldg, const double* V, long ldv, void* stream) {
  return rows_scale_add_outer(A, rows, cols, lda, s, scale, G, dy, ldg, V, ldv, S(stream));
}
size_t gpb_gemv_t_workspace_bytes(long rows, int cols) { return gemv_t_workspace_bytes(rows, cols); }
int gpb_gemv_t(const double* A, long rows, int cols, long lda, const double* Y, int dy, long ldy, double beta,
               double* out, long ldo, void* workspace, size_t workspace_bytes, void* stream) {
  return gemv_t(A, rows, cols, lda, Y, dy, ldy, beta, out, ldo, workspace, workspace_bytes, S(stream));
}

int gpb_gemm_ozaki_nt(int m, int n, int k, double alpha, const double* A, long lda, const double* B, long ldb, double beta,
                      double* C, long ldc, int lower, int slices, void* stream) {
  // on the fused engine the public entry takes the slice counts gpb_i8mma_config takes; more (the blocked inverse's
  // products, in narrower tiles) are internal
  if (ozaki_slices() == 0 && slices > OZ_MMA_MAX_SLICES && slices <= OZ_MMA_MAX_TILE_SLICES) return GPB_ERR_UNSUPPORTED;
  return gemm_ozaki_nt(m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, lower, slices, S(stream));
}
int gpb_ozaki_config(int slices) {
  const int prev = ozaki_slices();
  if (slices >= 0) ozaki_set_slices(slices);
  return prev;
}
int gpb_i8mma_config(int slices) {
  const int prev = i8mma_slices();
  if (slices >= 0) i8mma_set_slices(slices);
  return prev;
}

int gpb_gemm(int mode, int m, int n, int k, double alpha, const double* A, long lda, const double* B, long ldb,
             double beta, double* C, long ldc, int flags, void* stream) {
  if (mode < 0 || mode > 2 || m < 0 || n < 0 || k < 0) return GPB_ERR_BADARG;
  if (m == 0 || n == 0) return GPB_OK;
  if (!A || !B || !C) return GPB_ERR_BADARG;
  const GemmMode gm = static_cast<GemmMode>(mode);
  CUtensorMap mapA, mapB;
  // A is stored (m x k) for NT/NN and (k x m) for TN; B is (n x k) for NT and (k x n) for TN/NN.
  const long a_rows = gm == GEMM_TN ? k : m, a_cols = gm == GEMM_TN ? m : k;
  const long b_rows = gm == GEMM_NT ? n : k, b_cols = gm == GEMM_NT ? k : n;
  if (k > 0) {
    int rc = make_tmap_f64(&mapA, A, a_rows, a_cols, lda, gemm_box_rows_a(gm));
    if (rc) return rc;
    rc = make_tmap_f64(&mapB, B, b_rows, b_cols, ldb, gemm_box_rows_b(gm));
    if (rc) return rc;
  } else {
    // k == 0: C = beta * C; the maps are never dereferenced but must be valid objects
    int rc = make_tmap_f64(&mapA, C, m, n, ldc, 16);
    if (rc) return rc;
    mapB = mapA;
  }
  GemmArgs g;
  g.M = m; g.N = n; g.K = k;
  g.alpha = alpha; g.beta = beta;
  g.C = C; g.ldc = ldc;
  g.flags = static_cast<unsigned>(flags) & (GF_LOWER_TILES | GF_KLO_M | GF_KHI_M | GF_KLO_N | GF_KHI_N);
  if ((g.flags & GF_LOWER_TILES) && m != n) return GPB_ERR_BADARG;
  return gemm_launch(gm, mapA, mapB, g, S(stream));
}

int gpb_gemm_splitk(int mode, int m, int n, int k_total, int k_per_split, double alpha, const double* A, long lda,
                    const double* B, long ldb, double beta, double* C, long ldc, long c_split_stride, int lower_only,
                    void* stream) {
  if (mode < 0 || mode > 2 || m <= 0 || n <= 0 || k_total <= 0 || k_per_split <= 0) return GPB_ERR_BADARG;
  if (!A || !B || !C || (k_per_split % 16) != 0) return GPB_ERR_BADARG;
  const GemmMode gm = static_cast<GemmMode>(mode);
  const int splits = (k_total + k_per_split - 1) / k_per_split;
  CUtensorMap mapA, mapB;
  const long a_rows = gm == GEMM_TN ? k_total : m, a_cols = gm == GEMM_TN ? m : k_total;
  const long b_rows = gm == GEMM_NT ? n : k_total, b_cols = gm == GEMM_NT ? k_total : n;
  int rc = make_tmap_f64(&mapA, A, a_rows, a_cols, lda, gemm_box_rows_a(gm));
  if (rc) return rc;
  rc = make_tmap_f64(&mapB, B, b_rows, b_cols, ldb, gemm_box_rows_b(gm));
  if (rc) return rc;
  GemmArgs g;
  g.M = m; g.N = n; g.K = k_per_split;
  g.alpha = alpha; g.beta = beta;
  g.C = C; g.ldc = ldc; g.c_batch = c_split_stride;
  g.batch = splits;
  // the k index is the row index for MN-contiguous operands and the column index for K-contiguous ones
  if (gm == GEMM_TN) { g.day = k_per_split; g.dby = k_per_split; }
  else if (gm == GEMM_NT) { g.dax = k_per_split; g.dbx = k_per_split; }
  else { g.dax = k_per_split; g.dby = k_per_split; }
  g.flags = lower_only ? GF_LOWER_TILES : 0u;
  return gemm_launch(gm, mapA, mapB, g, S(stream));
}

// kern_bwd scratch of the input-gradient reduction K(Z, X_c): the largest over every chunk height up to chunk_rows (a
// short last chunk has fewer column blocks and may take more strips).  For a fixed number of 128-column blocks the size
// grows with the height, so the block-aligned heights and chunk_rows itself cover all cases.
static size_t kuf_gx_kb_bytes(int m, int chunk_rows, int D) {
  size_t b = 0;
  for (int r = 128;; r += 128) {
    const int h = std::min(r, chunk_rows);
    b = std::max(b, kern_bwd_workspace_bytes(m, h, D));
    if (h == chunk_rows) break;
  }
  return b;
}

// Workspace: [3 chunk x ldm buffers][split slots S x m x ldm][kern_bwd scratch][gemv_t scratch][small temporaries]
// and, with the input gradient, [kern_bwd scratch of the transposed reduction][chunk x D gradient, D + 1 temporaries]
size_t gpb_kuf_stats_workspace_bytes(int m, int D, int dy, int chunk_rows, int with_gx) {
  if (m <= 0 || D <= 0 || dy <= 0 || chunk_rows <= 0) return 0;
  const size_t ldm = static_cast<size_t>(m) + (m & 1);
  size_t b = 3 * kuf_align(static_cast<size_t>(chunk_rows) * ldm * 8);       // two pipeline buffers + one panel
  b += kuf_align(static_cast<size_t>(KUF_SPLITS) * m * ldm * 8);
  b += kuf_align(kern_bwd_workspace_bytes(chunk_rows, m, D));
  b += kuf_align(gemv_t_workspace_bytes(chunk_rows, m));
  b += kuf_align((static_cast<size_t>(D) + 1 + static_cast<size_t>(m) * D) * 8);
  if (with_gx) {
    b += kuf_align(kuf_gx_kb_bytes(m, chunk_rows, D));
    b += kuf_align((static_cast<size_t>(chunk_rows) * D + D + 1) * 8);
  }
  return b;
}

int gpb_kuf_stats_fwd(int kind, const double* X, long n, long ldx, const double* Y, int dy, long ldy, const double* Z,
                      int m, long ldz, int D, const double* ell, int ell_len, const double* sigma2, int chunk_rows,
                      double* Phi, long ldphi, double* psi, long ldpsi, double* kfu_cache, long ldcache,
                      void* workspace, size_t workspace_bytes, void* stream) {
  if (n < 0 || m <= 0 || D <= 0 || dy <= 0 || chunk_rows <= 0) return GPB_ERR_BADARG;
  if (!X || !Y || !Z || !ell || !sigma2 || !Phi || !psi || ldphi < m || ldpsi < dy) return GPB_ERR_BADARG;
  if (kfu_cache && (ldcache < m || (ldcache & 1) || (reinterpret_cast<uintptr_t>(kfu_cache) & 15))) return GPB_ERR_ALIGN;
  if (!workspace || workspace_bytes < gpb_kuf_stats_workspace_bytes(m, D, dy, chunk_rows, 0)) return GPB_ERR_BADARG;
  if (reinterpret_cast<uintptr_t>(workspace) & 15) return GPB_ERR_ALIGN;
  const long ldm = m + (m & 1);
  const size_t chunk_bytes = kuf_align(static_cast<size_t>(chunk_rows) * ldm * 8);
  char* w = static_cast<char*>(workspace);
  double* pbuf[2] = {reinterpret_cast<double*>(w), reinterpret_cast<double*>(w + chunk_bytes)};
  w += 3 * chunk_bytes;
  double* slots = reinterpret_cast<double*>(w);
  w += kuf_align(static_cast<size_t>(KUF_SPLITS) * m * ldm * 8);
  w += kuf_align(kern_bwd_workspace_bytes(chunk_rows, m, D));
  void* gemv_ws = w;
  const size_t gemv_bytes = gemv_t_workspace_bytes(chunk_rows, m);
  cudaStream_t st = S(stream);
  KufAux* aux = nullptr;
  if (int rc = kuf_aux(st, &aux)) return rc;
  const long slot_stride = static_cast<long>(m) * ldm;
  GPB_CUDA_CHECK(cudaMemsetAsync(slots, 0, static_cast<size_t>(KUF_SPLITS) * slot_stride * 8, st));
  for (int o = 0; o < dy; ++o)
    GPB_CUDA_CHECK(cudaMemset2DAsync(psi + o, ldpsi * 8, 0, 8, m, st));
  const int kper = kuf_k_per_split(static_cast<int>(std::min<long>(chunk_rows, std::max<long>(n, 1))));
  GPB_CUDA_CHECK(cudaEventRecord(aux->fork, st));
  GPB_CUDA_CHECK(cudaStreamWaitEvent(aux->side, aux->fork, 0));
  long c = 0;
  for (long s0 = 0; s0 < n; s0 += chunk_rows, ++c) {
    const int rows = static_cast<int>(std::min<long>(chunk_rows, n - s0));
    const int b = static_cast<int>(c & 1);
    double* P = kfu_cache ? kfu_cache + s0 * ldcache : pbuf[b];
    const long ldp = kfu_cache ? ldcache : ldm;
    // side stream: covariance panel of this chunk (its buffer must have been consumed by the Gram product of chunk c - 2)
    if (!kfu_cache && c >= 2) GPB_CUDA_CHECK(cudaStreamWaitEvent(aux->side, aux->free_[b], 0));
    int rc = gpb_kern_fwd(kind, X + s0 * ldx, rows, ldx, Z, m, ldz, D, ell, ell_len, sigma2, nullptr, 0, P, ldp, aux->side);
    if (rc) return rc;
    GPB_CUDA_CHECK(cudaEventRecord(aux->ready[b], aux->side));
    // caller's stream: Gram product and psi of this chunk
    GPB_CUDA_CHECK(cudaStreamWaitEvent(st, aux->ready[b], 0));
    rc = gpb_gemm_splitk(GEMM_TN, m, m, rows, kper, 1.0, P, ldp, P, ldp, 1.0, slots, ldm, slot_stride, 1, stream);
    if (rc) return rc;
    rc = gpb_gemv_t(P, rows, m, ldp, Y + s0 * ldy, dy, ldy, 1.0, psi, ldpsi, gemv_ws, gemv_bytes, stream);
    if (rc) return rc;
    GPB_CUDA_CHECK(cudaEventRecord(aux->free_[b], st));
  }
  dim3 grid((m + 255) / 256, m);
  kuf_reduce_sym_kernel<<<grid, 256, 0, st>>>(slots, KUF_SPLITS, m, ldm, slot_stride, Phi, ldphi);
  count_launch();
  GPB_CUDA_CHECK(cudaGetLastError());
  return GPB_OK;
}

int gpb_kuf_stats_bwd(int kind, const double* X, long n, long ldx, const double* Y, int dy, long ldy, const double* Z,
                      int m, long ldz, int D, const double* ell, int ell_len, const double* sigma2, int chunk_rows,
                      const double* R, long ldr, const double* W, long ldw, const double* kfu_cache, long ldcache,
                      double* g_ell, double* g_sigma2, double* gZ, void* workspace, size_t workspace_bytes,
                      void* stream, double* gX, long ldgx) {
  if (n < 0 || m <= 0 || D <= 0 || dy <= 0 || chunk_rows <= 0) return GPB_ERR_BADARG;
  if (!X || !Y || !Z || !ell || !sigma2 || !R || !W || !g_ell || !g_sigma2 || !gZ) return GPB_ERR_BADARG;
  if (gX && ldgx < D) return GPB_ERR_BADARG;
  if (ldr < m || (ldr & 1) || (reinterpret_cast<uintptr_t>(R) & 15)) return GPB_ERR_ALIGN;
  if (kfu_cache && (ldcache < m || (ldcache & 1) || (reinterpret_cast<uintptr_t>(kfu_cache) & 15))) return GPB_ERR_ALIGN;
  if (!workspace || workspace_bytes < gpb_kuf_stats_workspace_bytes(m, D, dy, chunk_rows, gX != nullptr))
    return GPB_ERR_BADARG;
  if (reinterpret_cast<uintptr_t>(workspace) & 15) return GPB_ERR_ALIGN;
  const long ldm = m + (m & 1);
  const size_t chunk_bytes = kuf_align(static_cast<size_t>(chunk_rows) * ldm * 8);
  char* w = static_cast<char*>(workspace);
  double* gbuf[2] = {reinterpret_cast<double*>(w), reinterpret_cast<double*>(w + chunk_bytes)};
  double* panel = reinterpret_cast<double*>(w + 2 * chunk_bytes);
  w += 3 * chunk_bytes;
  w += kuf_align(static_cast<size_t>(KUF_SPLITS) * m * ldm * 8);
  void* kb_ws = w;
  const size_t kb_bytes = kern_bwd_workspace_bytes(chunk_rows, m, D);
  w += kuf_align(kb_bytes);
  w += kuf_align(gemv_t_workspace_bytes(chunk_rows, m));
  double* t_ell = reinterpret_cast<double*>(w);
  double* t_s2 = t_ell + D;
  double* t_z = t_s2 + 1;
  w += kuf_align((static_cast<size_t>(D) + 1 + static_cast<size_t>(m) * D) * 8);
  // input gradient: the same G_c reduced with the roles of X and Z exchanged (G_c read transposed), whose column
  // gradient is dLoss/dX_c; its hyper-parameter sums are discarded
  void* xb_ws = w;
  const size_t xb_bytes = gX ? kuf_gx_kb_bytes(m, chunk_rows, D) : 0;
  double* x_g = reinterpret_cast<double*>(w + kuf_align(xb_bytes));
  double* x_ell = x_g + static_cast<size_t>(chunk_rows) * D;
  double* x_s2 = x_ell + D;
  cudaStream_t st = S(stream);
  KufAux* aux = nullptr;
  if (int rc = kuf_aux(st, &aux)) return rc;
  GPB_CUDA_CHECK(cudaMemsetAsync(g_ell, 0, static_cast<size_t>(ell_len) * 8, st));
  GPB_CUDA_CHECK(cudaMemsetAsync(g_sigma2, 0, 8, st));
  GPB_CUDA_CHECK(cudaMemsetAsync(gZ, 0, static_cast<size_t>(m) * D * 8, st));
  GPB_CUDA_CHECK(cudaEventRecord(aux->fork, st));
  GPB_CUDA_CHECK(cudaStreamWaitEvent(aux->side, aux->fork, 0));
  long c = 0;
  for (long s0 = 0; s0 < n; s0 += chunk_rows, ++c) {
    const int rows = static_cast<int>(std::min<long>(chunk_rows, n - s0));
    const int b = static_cast<int>(c & 1);
    double* G = gbuf[b];
    // caller's stream: dLoss/dKfu_c = Kfu_c R + Y_c W^T into buffer b (consumed by the reduction of chunk c - 2)
    if (c >= 2) GPB_CUDA_CHECK(cudaStreamWaitEvent(st, aux->free_[b], 0));
    const double* P;
    long ldp;
    if (kfu_cache) {
      P = kfu_cache + s0 * ldcache; ldp = ldcache;
    } else {
      int rc = gpb_kern_fwd(kind, X + s0 * ldx, rows, ldx, Z, m, ldz, D, ell, ell_len, sigma2, nullptr, 0, panel, ldm, stream);
      if (rc) return rc;
      P = panel; ldp = ldm;
    }
    int rc = gpb_gemm(GEMM_NN, rows, m, m, 1.0, P, ldp, R, ldr, 0.0, G, ldm, 0, stream);
    if (rc) return rc;
    // Y rows (dy values, stride ldy) may be odd-strided: the rank-dy update runs through the in-place row kernel
    rc = gpb_rows_scale_add_outer(G, rows, m, ldm, nullptr, 1.0, Y + s0 * ldy, dy, ldy, W, ldw, stream);
    if (rc) return rc;
    GPB_CUDA_CHECK(cudaEventRecord(aux->ready[b], st));
    // side stream: reduce it against dK/d(ell, sigma2, Z) while the next chunk's product runs
    GPB_CUDA_CHECK(cudaStreamWaitEvent(aux->side, aux->ready[b], 0));
    rc = gpb_kern_bwd(kind, X + s0 * ldx, rows, ldx, Z, m, ldz, D, ell, ell_len, sigma2, G, ldm, 0, t_ell, t_s2, t_z,
                      kb_ws, kb_bytes, aux->side);
    if (rc) return rc;
    kuf_accumulate_kernel<<<(ell_len + 255) / 256, 256, 0, aux->side>>>(g_ell, t_ell, ell_len);
    kuf_accumulate_kernel<<<1, 32, 0, aux->side>>>(g_sigma2, t_s2, 1);
    kuf_accumulate_kernel<<<(m * D + 255) / 256, 256, 0, aux->side>>>(gZ, t_z, static_cast<long>(m) * D);
    count_launch(3);
    GPB_CUDA_CHECK(cudaGetLastError());
    if (gX) {
      rc = gpb_kern_bwd(kind, Z, m, ldz, X + s0 * ldx, rows, ldx, D, ell, ell_len, sigma2, G, ldm, 1, x_ell, x_s2, x_g,
                        xb_ws, xb_bytes, aux->side);
      if (rc) return rc;
      GPB_CUDA_CHECK(cudaMemcpy2DAsync(gX + s0 * ldgx, ldgx * 8, x_g, static_cast<size_t>(D) * 8,
                                       static_cast<size_t>(D) * 8, rows, cudaMemcpyDeviceToDevice, aux->side));
    }
    GPB_CUDA_CHECK(cudaEventRecord(aux->free_[b], aux->side));
  }
  GPB_CUDA_CHECK(cudaEventRecord(aux->join, aux->side));
  GPB_CUDA_CHECK(cudaStreamWaitEvent(st, aux->join, 0));
  return GPB_OK;
}

size_t gpb_gpr_grad_workspace_bytes(int n, int D) { return gpr_grad_workspace_bytes(n, D); }
int gpb_gpr_grad(int kind, const double* X, int n, long ldx, int D, const double* ell, int ell_len,
                 const double* sigma2, const double* Kinv, long ldk, const double* kdiag_blocks, const double* a,
                 int dy, long lda_a, double* g_ell, double* g_sigma2, double* g_noise, void* workspace,
                 size_t workspace_bytes, void* stream, double* gX, long ldgx) {
  return gpr_grad(kind, X, n, ldx, D, ell, ell_len, sigma2, Kinv, ldk, kdiag_blocks, a, dy, lda_a, g_ell, g_sigma2,
                  g_noise, workspace, workspace_bytes, gX, ldgx, S(stream));
}

int gpb_pred_gx(int kind, const double* Xs, int ns, long ldxs, const double* X, int n, long ldx, int D,
                const double* ell, int ell_len, const double* sigma2, const double* a, int dy, long lda,
                const double* g_mean, long ldgm, const double* g_var, const double* Q, long ldq, double* gXs, long ldgx,
                void* stream) {
  return pred_gx(kind, Xs, ns, ldxs, X, n, ldx, D, ell, ell_len, sigma2, a, dy, lda, g_mean, ldgm, g_var, Q, ldq, gXs,
                 ldgx, S(stream));
}

}  // extern "C"
#pragma GCC visibility pop
