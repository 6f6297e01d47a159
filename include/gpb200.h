/* gpb200.h -- C ABI of libgpb200.so, the B200 (sm_100a) implementation of gptorch's dense-GP hot path.
 *
 * The reference (cics-nd/gptorch v0.3.2) has no FFI: its hot path is Python calling torch ops.  Each entry
 * point below names the reference call site it replaces (file:line under the reference tree); the
 * reference-side binding a maintainer would add is the ctypes stub in INTEGRATION.md.
 *
 * Conventions
 *   - every matrix is fp64, row-major, on the current CUDA device; `ld*` are leading dimensions in elements;
 *   - pointers are plain device pointers, `stream` is a cudaStream_t passed as void*;
 *   - hyper-parameters (length scales, variances) are DEVICE pointers so a call never synchronises;
 *   - the library never allocates or frees: workspaces are supplied by the caller (see *_workspace_bytes);
 *   - return value: 0 = launched, <0 = rejected (GPB_ERR_*); numerical status (LAPACK-style `info`) is
 *     written to a device int by the kernels and read by the caller when it chooses to synchronise;
 *   - matrices handed to the GEMM-based entry points (potrf/potri/trsm/gemm) need a 16-byte aligned base
 *     and an even leading dimension (TMA requirement); GPB_ERR_ALIGN is returned otherwise.
 */
#ifndef GPB200_H_
#define GPB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GPB_OK 0
#define GPB_ERR_BADARG (-1)
#define GPB_ERR_ALIGN (-2)
#define GPB_ERR_CUDA (-3)
#define GPB_ERR_DRIVER (-4)
#define GPB_ERR_UNSUPPORTED (-5)

/* Covariance families.  Reference: gptorch/kernels.py Rbf :215-222, Exp/Matern12 :182-194,
 * Matern32 :197-201, Matern52 :204-212, Linear :238-265. */
enum gpb_kernel_kind {
  GPB_KERN_RBF = 0,
  GPB_KERN_EXP = 1,      /* == Matern12 */
  GPB_KERN_MATERN32 = 2,
  GPB_KERN_MATERN52 = 3,
  GPB_KERN_LINEAR = 4,
  GPB_KERN_PERIODIC = 5, /* variance * cos(r), gptorch/kernels.py:228-235 */
  /* leaves of composite kernels only (gpb_kern_sop_fwd, gpb_kern_bwd_mul): gptorch/kernels.py:83-101 */
  GPB_KERN_CONSTANT = 6,
  GPB_KERN_WHITE = 7
};

/* Which part of a symmetric output to produce. */
enum gpb_fill { GPB_FILL_FULL = 0, GPB_FILL_LOWER = 1 };

int gpb_version(void);
/* Human-readable description of the last error on the calling thread (never NULL). */
const char* gpb_last_error(void);
/* ABI block size: diagonal-block workspaces (`dinv`, `kdiag_blocks`) are ceil(n/128)*128 rows of 128 doubles. */
int gpb_block_size(void);
/* Number of CUDA kernels this library has launched since load / the last reset (bench.py: gpu_launches). */
long gpb_launch_count(void);
void gpb_reset_launch_count(void);
/* Measurement aid (bench.py roofline.peak): one launch in which every warp of 2 CTAs x 16 warps per SM issues
 * independent DMMA.8x8x4 chains from registers for `iters` rounds of 8 -- the FP64 tensor-pipe issue ceiling the GEMM
 * engine is bounded by (torch's cuBLAS DGEMM is the other, lower, denominator).  `scratch`: device buffer of at least
 * 2 * SMs * 512 doubles; *flop_out (host, optional) receives the flop count of the launch; the caller times it with
 * CUDA events on `stream`.  No reference counterpart. */
int gpb_dmma_issue_probe(int iters, double* scratch, size_t scratch_bytes, double* flop_out, void* stream);

/* ---- covariance construction ---------------------------------------------------------------------------
 * K[i][j] = k(X[i,:], X2[j,:]).  Replaces Kernel.K(X, X2) (gptorch/kernels.py:189,198,205,220,258) with its
 * callees Stationary.squared_dist/dist (:149-172) and util.squared_distance (gptorch/util.py:73-88):
 * scaled squared distance by the expansion |a|^2+|b|^2-2ab (the a.b term on FP64 DMMA), clamp at 0, the
 * kernel non-linearity, times the variance.  X2 == NULL means X2 = X.
 *   ell:     device, length ell_len (1 = isotropic, D = ARD); for GPB_KERN_LINEAR it is the per-dimension
 *            variance vector v (ell_len == D) and `sigma2` is ignored (may be NULL).
 *   noise:   optional device scalar added to the diagonal when X2 == NULL (GPR._compute_kyy,
 *            gptorch/models/gpr.py:69-86, without the dense N x N diagonal temporary).
 *   fill:    GPB_FILL_LOWER skips tiles strictly above the diagonal (only valid when X2 == NULL). */
int gpb_kern_fwd(int kind, const double* X, int n1, long ldx, const double* X2, int n2, long ldx2, int D,
                 const double* ell, int ell_len, const double* sigma2, const double* noise, int fill,
                 double* K, long ldk, void* stream);

/* Bytes of scratch needed by gpb_kern_bwd for the given problem. */
size_t gpb_kern_bwd_workspace_bytes(int n1, int n2, int D);

/* Backward of gpb_kern_fwd for an upstream gradient G = dLoss/dK (n1 x n2, ldg).  Replaces torch autograd
 * through the composite ops of gptorch/kernels.py and gptorch/util.py:82-88 (gradient passes the r^2 clamp
 * unchanged; for Exp/Matern the sqrt clamp at 1e-40 zeroes it, gptorch/kernels.py:171-172).
 *   g_ell:    out, ell_len doubles: dLoss/d ell  (for LINEAR: dLoss/d v)
 *   g_sigma2: out, 1 double (ignored for LINEAR; may be NULL)
 *   gX2:      optional out, n2 x D (ld = D): dLoss/dX2 treating X as constant.  (The gradient w.r.t. the first
 *             argument is obtained by calling again with the arguments swapped and g_transposed = 1.)
 *   g_transposed: G is stored n2 x n1 (element (i,j) at G[j*ldg + i]). */
int gpb_kern_bwd(int kind, const double* X, int n1, long ldx, const double* X2, int n2, long ldx2, int D,
                 const double* ell, int ell_len, const double* sigma2, const double* G, long ldg,
                 int g_transposed, double* g_ell, double* g_sigma2, double* gX2, void* workspace,
                 size_t workspace_bytes, void* stream);

/* gpb_kern_bwd with an optional element-wise multiplier: the upstream gradient is G .* Mul (Mul: same shape, layout
 * and transposition flag as G; NULL = ones).  This is the backward of one leaf of a Product kernel
 * (gptorch/kernels.py:286-295: d(k1 k2)/d theta1 = k2 dk1/d theta1), with Mul = the product of the other leaves.
 * Also accepts GPB_KERN_CONSTANT and GPB_KERN_WHITE (only g_sigma2 is meaningful; `ell` may be any valid vector of
 * length ell_len).  `symmetric` != 0 declares X2 == X even when X2 is passed explicitly (White is the identity then). */
int gpb_kern_bwd_mul(int kind, const double* X, int n1, long ldx, const double* X2, int n2, long ldx2, int D,
                     const double* ell, int ell_len, const double* sigma2, const double* G, long ldg,
                     int g_transposed, const double* Mul, long ldm, int symmetric, double* g_ell, double* g_sigma2,
                     double* gX2, void* workspace, size_t workspace_bytes, void* stream);

/* Composite covariance in one pass: K = sum_t prod_{l in term t} k_l(X, X2) [+ noise I when X2 == NULL].
 * Replaces the Sum / Product combinators (gptorch/kernels.py:286-306) over leaf kernels of any family above --
 * every tree of + and * is a sum of products of leaves -- without the reference's N x N temporary per child.
 *   n_terms <= 8 terms; term t has term_len[t] consecutive leaves (<= 16 leaves in total); all arrays below are
 *   HOST arrays indexed by leaf:  leaf_kind, leaf_ell (device pointers; Linear: the variance vector; ignored for
 *   Constant / White), leaf_ell_len (1 or D), leaf_sigma2 (device pointers; ignored for Linear).
 *   noise / fill / K / ldk as in gpb_kern_fwd. */
int gpb_kern_sop_fwd(int n_terms, const int* term_len, const int* leaf_kind, const double* const* leaf_ell,
                     const int* leaf_ell_len, const double* const* leaf_sigma2, const double* X, int n1, long ldx,
                     const double* X2, int n2, long ldx2, int D, const double* noise, int fill, double* K, long ldk,
                     void* stream);

/* Kdiag for the non-stationary kernel (Linear.Kdiag, gptorch/kernels.py:264-265): out[i] = sum_d v_d x_id^2.
 * Stationary kernels return the variance broadcast (gptorch/kernels.py:174-179) and need no kernel. */
int gpb_linear_kdiag(const double* X, int n, long ldx, int D, const double* v, double* out, void* stream);

/* ---- Cholesky ------------------------------------------------------------------------------------------
 * In-place lower Cholesky of the symmetric matrix whose LOWER triangle is stored in A (n x n, lda).
 * Replaces torch.cholesky behind functions.cholesky (gptorch/functions.py:46-47).  The strictly upper
 * triangle of A is scratch afterwards (gpb_tri_zero_upper restores the reference's zero upper triangle).
 *   dinv:  out workspace, ceil(n/128)*128 x 128 doubles: inverses of the 128 x 128 diagonal blocks of L
 *          (used by the solves and by gpb_potri_lower).
 *   info:  device int, must be zeroed by the caller; set to the 1-based index of the first non-positive
 *          pivot (LAPACK potrf semantics: the factorisation "failed" and jit_op must add jitter,
 *          gptorch/functions.py:28-43). */
int gpb_potrf_lower(double* A, int n, long lda, double* dinv, int* info, void* stream);

/* Inverses of the diagonal 128-blocks of an existing lower factor L (for callers that did not run potrf). */
int gpb_tri_diag_inverse(const double* L, int n, long ldl, double* dinv, void* stream);

size_t gpb_potri_workspace_bytes(int n);
/* Given L (lower triangle of A, with `dinv` from potrf) compute (L L^T)^-1.  Replaces
 * functions.cholesky_inverse (gptorch/functions.py:50-54) and, inside the fused GPR backward, autograd's
 * CholeskyBackward0.  On return: strictly-lower 128-blocks of A hold the inverse; the diagonal 128-blocks are
 * in kdiag_blocks (ceil(n/128)*128 x 128, symmetric, full); the upper triangle of A is scratch. */
int gpb_potri_lower(double* A, int n, long lda, const double* dinv, double* kdiag_blocks, void* workspace,
                    size_t workspace_bytes, void* stream);
/* First half of gpb_potri_lower on its own: T = L^-T is written to the UPPER triangle of A (diagonal 128-blocks
 * become T_jj with zeros below the diagonal; strictly-lower off-diagonal blocks keep L).  Used for the
 * backward of functions.cholesky / trtrs (dL/dA = L^-T Phi(L^T dL) L^-1 becomes three GEMMs with T).
 * Workspace size: gpb_potri_workspace_bytes(n). */
int gpb_trtri_upper(double* A, int n, long lda, const double* dinv, void* workspace, size_t workspace_bytes,
                    void* stream);
/* Expand the blocked result of gpb_potri_lower into a full symmetric n x n matrix `out` (ldo). */
int gpb_potri_assemble(const double* A, int n, long lda, const double* kdiag_blocks, double* out, long ldo,
                       void* stream);

/* Zero the strictly upper triangle (torch.cholesky returns a clean lower factor). */
int gpb_tri_zero_upper(double* A, int n, long lda, void* stream);
/* A[i][i] += *value (value: device scalar) or += host_value when value == NULL (jitter, functions.py:36). */
int gpb_add_diag(double* A, int n, long lda, const double* value, double host_value, void* stream);

/* ---- triangular solves and log-determinant ---------------------------------------------------------------
 * B <- L^-1 B (trans = 0) or L^-T B (trans = 1), L lower n x n, B n x k row-major (ldb), in place.
 * Replaces functions.trtrs (gptorch/functions.py:71-76) -- without torch.triangular_solve's clone of L.
 * `dinv` are the diagonal-block inverses of L (from potrf or gpb_tri_diag_inverse).  One launch per group
 * of <= 4 right-hand sides streams L exactly once; `workspace` holds the per-block ready flags. */
size_t gpb_trsv_workspace_bytes(int n);
int gpb_trsv_lower(const double* L, int n, long ldl, const double* dinv, double* B, int k, long ldb, int trans,
                   void* workspace, size_t workspace_bytes, void* stream);
/* Right-side solve on a row-panel: X <- X L^-T, X m x n row-major (ldx), L lower n x n.  This is the layout
 * the sparse models use for A^T = Kfu L^-T (gptorch/models/sparse_gpr.py:132,360). */
int gpb_trsm_right_lt(const double* L, int n, long ldl, const double* dinv, double* X, int m, long ldx,
                      void* stream);

/* out[0] = sum_i log L[i][i], i < n  (functions.lt_log_determinant, gptorch/functions.py:61-68; n = 0 skips it);
 * out[1] = sum of squares of the vrows x k matrix V (ldv) if V != NULL (the -1/2 sum alpha^2 term of
 * gptorch/models/gpr.py:66, and sum Y^2 of gptorch/models/sparse_gpr.py:146).  Deterministic (fixed order). */
int gpb_logdet_sumsq(const double* L, int n, long ldl, const double* V, int vrows, int k, long ldv, double* out,
                     void* stream);

/* out[c][o] = beta * out[c][o] + sum_r A[r][c] * Y[r][o]:  A^T Y for a tall row panel A (rows x cols) and a few
 * right-hand sides (the "A @ err" statistic of gptorch/models/sparse_gpr.py:137 in row-panel layout).  HBM-bound:
 * A is read once; deterministic two-stage reduction. */
/* out[i] = alpha * sum_j A[i][j] B[i][j] + beta * out[i] for i < rows: the row-wise reductions of the sparse models'
 * predictive variance, sum(alpha ** 2, dim=1) / sum(gamma ** 2, dim=1) (gptorch/models/sparse_gpr.py:374-379,
 * :186-190) and Kdiag - colsum(A * A) (gptorch/models/gpr.py:109-113), in one pass without an [rows x cols] temporary. */
int gpb_rowdot(const double* A, long lda, const double* B, long ldb, long rows, int cols, double alpha, double beta,
               double* out, void* stream);
/* out[i][o] = sum_j A[i][j] V[j][o]: a row panel times a few vectors (the predictive mean alpha @ t of
 * gptorch/models/sparse_gpr.py:369, K(x*, X) @ a of gptorch/models/gpr.py:107) -- A is read once. */
int gpb_gemv_n(const double* A, long rows, int cols, long lda, const double* V, int dy, long ldv, double* out, long ldo,
               void* stream);
/* In place: A[i][j] = scale * s[i] * A[i][j] + sum_o G[i][o] V[j][o]  (s == NULL: 1; G == NULL: no outer product).  The
 * adjoint of the two reductions above in one pass: d/dA of sum_i s_i (row quadratic form) plus (A V) against G. */
int gpb_rows_scale_add_outer(double* A, long rows, int cols, long lda, const double* s, double scale, const double* G,
                             int dy, long ldg, const double* V, long ldv, void* stream);
size_t gpb_gemv_t_workspace_bytes(long rows, int cols);
int gpb_gemv_t(const double* A, long rows, int cols, long lda, const double* Y, int dy, long ldy, double beta,
               double* out, long ldo, void* workspace, size_t workspace_bytes, void* stream);

/* ---- GEMM ------------------------------------------------------------------------------------------------
 * C = alpha * op(A) op(B) + beta * C on the FP64 DMMA engine.  mode: 0 = A B^T (A: m x k, B: n x k),
 * 1 = A^T B (A: k x m, B: k x n), 2 = A B (A: m x k, B: k x n).  Replaces the `@` products of
 * gptorch/models/sparse_gpr.py:133,137,176,183,360-370.
 * flags (OR of GPB_GEMM_*): LOWER computes only the tiles that intersect the lower triangle (m == n, SYRK);
 * the K* flags declare a triangular operand so that all-zero k-chunks are skipped, per 128-row/column tile:
 *   KLO_M: terms with k <  first row of the tile vanish     KHI_M: terms with k >  last row of the tile vanish
 *   KLO_N: terms with k <  first column of the tile vanish  KHI_N: terms with k >  last column of the tile vanish
 * (the zero part of the operand must really hold zeros inside the partially covered 128-blocks). */
#define GPB_GEMM_LOWER 1
#define GPB_GEMM_KLO_M 2
#define GPB_GEMM_KHI_M 4
#define GPB_GEMM_KLO_N 8
#define GPB_GEMM_KHI_N 16
int gpb_gemm(int mode, int m, int n, int k, double alpha, const double* A, long lda, const double* B, long ldb,
             double beta, double* C, long ldc, int flags, void* stream);

/* EXPERIMENTAL (off by default; DESIGN.md section 8): C = beta C + alpha A B^T (A: m x k, B: n x k, row-major) computed on the
 * INT8 tensor path by integer slicing (Ozaki scheme): every row is cut into `slices` (2..10) signed 7-bit digits relative
 * to its own power-of-two scale, the digit products of one weight class run as one int8 GEMM over a concatenated k
 * (cuBLASLt, loaded with dlopen on first use), and a recombination kernel applies the scales in fp64.  8 slices match a
 * DGEMM norm-wise on covariance-conditioned operands (profiles/r02_ozaki_probe.txt).  lower != 0 (m == n): only the
 * 128-blocks on and below the diagonal are written.  Returns GPB_ERR_UNSUPPORTED (-5) for shapes the int8 path does not
 * take (k % 16, m % 4, n % 4, ldc odd) or when cuBLASLt cannot be loaded; callers then use gpb_gemm.
 * No counterpart in the reference (torch.matmul in fp64, gptorch/models/gpr.py:69-86 via torch.linalg). */
int gpb_gemm_ozaki_nt(int m, int n, int k, double alpha, const double* A, long lda, const double* B, long ldb, double beta,
                      double* C, long ldc, int lower, int slices, void* stream);
/* Number of slices the blocked Cholesky uses for its large trailing updates (0 = FP64 DMMA engine, the default; the initial
 * value comes from the environment variable GPB_OZAKI).  slices < 0 only queries.  Returns the previous value. */
int gpb_ozaki_config(int slices);

/* Split-K form: the k range is cut into ceil(k_total / k_per_split) slices (k_per_split a multiple of 16) that run
 * as independent CTAs; slice s accumulates into C + s * c_split_stride.  Used for the Gram products of the sparse
 * models, whose M x M output has far fewer tiles than the GPU has SMs (A A^T over N >> M rows,
 * gptorch/models/sparse_gpr.py:133); the caller sums the slices (deterministic, fixed order). */
int gpb_gemm_splitk(int mode, int m, int n, int k_total, int k_per_split, double alpha, const double* A, long lda,
                    const double* B, long ldb, double beta, double* C, long ldc, long c_split_stride, int lower_only,
                    void* stream);

/* ---- streamed Kuf statistics of the sparse models ---------------------------------------------------------------
 * Phi = Kuf Kfu (M x M, full symmetric) and psi = Kuf Y (M x dy) for Kfu = K(X, Z), accumulated over row chunks of X
 * without ever holding the N x M matrix: per chunk the covariance panel is built (gpb_kern_fwd), its Gram product is
 * accumulated by the split-K TN GEMM and psi by the transposed panel-vector kernel.  Replaces Kuf = K(Z, x) and the
 * products A @ A.t(), A @ err of VFE.log_likelihood (gptorch/models/sparse_gpr.py:126-137) in the form with the M x M
 * congruence applied afterwards (A A^T = L^-1 Phi L^-T); it is also the quantity a row-sharded run all-reduces.
 *   chunk_rows: rows of X per panel;  kfu_cache: optional N x ldcache buffer that receives every panel (NULL = the panels
 *   are rebuilt by the backward call);  workspace: gpb_kuf_stats_workspace_bytes(m, D, dy, chunk_rows).
 * The backward call reduces the gradient with respect to the panels, dLoss/dKfu_c = Kfu_c R + Y_c W^T with
 * R = dLoss/dPhi + (dLoss/dPhi)^T (M x M, symmetric) and W = dLoss/dpsi (M x dy), against dK/d(ell, sigma2, Z):
 *   g_ell (ell_len), g_sigma2 (1) and gZ (M x D, dense) are OVERWRITTEN with the sums over all chunks.
 *   gX (optional, n x D, row stride ldgx >= D): receives dLoss/dX, the gradient with respect to the rows of X (each
 *   chunk's panel gradient reduced with X and Z exchanged, G_c read transposed); NULL skips it.  A workspace for a call
 *   with gX is sized by gpb_kuf_stats_workspace_bytes(..., with_gx = 1); with_gx = 0 gives the size without it. */
size_t gpb_kuf_stats_workspace_bytes(int m, int D, int dy, int chunk_rows, int with_gx);
int gpb_kuf_stats_fwd(int kind, const double* X, long n, long ldx, const double* Y, int dy, long ldy, const double* Z,
                      int m, long ldz, int D, const double* ell, int ell_len, const double* sigma2, int chunk_rows,
                      double* Phi, long ldphi, double* psi, long ldpsi, double* kfu_cache, long ldcache,
                      void* workspace, size_t workspace_bytes, void* stream);
int gpb_kuf_stats_bwd(int kind, const double* X, long n, long ldx, const double* Y, int dy, long ldy, const double* Z,
                      int m, long ldz, int D, const double* ell, int ell_len, const double* sigma2, int chunk_rows,
                      const double* R, long ldr, const double* W, long ldw, const double* kfu_cache, long ldcache,
                      double* g_ell, double* g_sigma2, double* gZ, void* workspace, size_t workspace_bytes,
                      void* stream, double* gX, long ldgx);

/* ---- fused GPR gradient ------------------------------------------------------------------------------------
 * Given Kinv in the blocked form left by gpb_potri_lower and a = Ky^-1 (y - m) (n x dy, lda_a), reduce
 *    W = 1/2 (dy * Kinv - a a^T)            (dLoss/dKy, SURVEY 10; gptorch/models/gpr.py:47-67)
 * against dK/d(ell, sigma2) without materialising W or K:  g_ell[d] = sum_ij W_ij dK_ij/d ell_d,
 * g_sigma2 = sum_ij W_ij K_ij / sigma2, g_noise = tr W.  Replaces the autograd backward of
 * kernels.K + _compute_kyy + cholesky + trtrs.
 *   gX (optional, n x D, row stride ldgx >= D): receives dLoss/dX = sum_j 2 W_ij dK_ij/dx_i, the gradient with
 *   respect to the training inputs (deep kernel learning, learned input warps), from W formed on the fly as above --
 *   no N x N temporary and no extra workspace.  NULL skips it; the hyper-parameter reduction is the same either way. */
size_t gpb_gpr_grad_workspace_bytes(int n, int D);
int gpb_gpr_grad(int kind, const double* X, int n, long ldx, int D, const double* ell, int ell_len,
                 const double* sigma2, const double* Kinv, long ldk, const double* kdiag_blocks,
                 const double* a, int dy, long lda_a, double* g_ell, double* g_sigma2, double* g_noise,
                 void* workspace, size_t workspace_bytes, void* stream, double* gX, long ldgx);

#ifdef __cplusplus
}
#endif
#endif /* GPB200_H_ */
