// gpb_ozaki.cuh -- internal interface of the int8-sliced GEMM (gpb_ozaki.cu, gpb_ozaki_mma.cu).
#pragma once
#include "gpb_common.cuh"

namespace gpb {

// Extended arguments (internal callers: the triangular products of gpb_potri_lower).
struct OzEx {
  int m = 0, n = 0, k = 0;
  double alpha = 1.0, beta = 0.0;
  // operands: logical A is m x k, logical B is n x k.  *_trans = 0: stored like that (row-major, K-major);
  // *_trans = 1: stored as the k x m (k x n) row-major array whose transpose is meant (the split transposes on the fly).
  // *_tri / *_row0 / *_col0 refer to the STORED array: element (r, c) counts as zero when col0 + c lies left of the
  // 128-block of row0 + r (upper triangular by blocks inside a buffer whose other blocks hold unrelated data).
  const double* A = nullptr; long lda = 0; int a_trans = 0, a_tri = 0, a_row0 = 0, a_col0 = 0;
  const double* B = nullptr; long ldb = 0; int b_trans = 0, b_tri = 0, b_row0 = 0, b_col0 = 0;
  double* C = nullptr; long ldc = 0;
  int lower = 0;            // skip 128-blocks right of the diagonal; rows of C are global rows gi0 + i, columns global j
  int gi0 = 0;
  double* Cdiag = nullptr;  // diagonal 128-blocks go here ([row][NB] layout of gpb_potri_lower) instead of into C
  int slices = 8;
  cudaStream_t stream = nullptr;
};

// C = beta C + alpha A B^T on the INT8 tensor path; GPB_ERR_UNSUPPORTED for shapes it does not take (callers use the FP64
// DMMA engine for those).
int gemm_ozaki_nt_ex(const OzEx& x);
int gemm_ozaki_nt(int m, int n, int k, double alpha, const double* A, long lda, const double* B, long ldb, double beta,
                  double* C, long ldc, int lower, int slices, cudaStream_t stream);
// Engines.  GPB_OZAKI / gpb_ozaki_config: slices of the library engine (cuBLASLt int8 products, 0 = off, the default).
// GPB_I8MMA / gpb_i8mma_config: slices of the fused tcgen05 kernel (gpb_ozaki_mma.cu; 8 by default, 0 = FP64 DMMA).
// gemm_ozaki_nt_ex runs the library engine while ozaki_slices() > 0 and the fused kernel otherwise; the Cholesky's
// updates use sliced_slices() = ozaki_slices() if that is > 0, else i8mma_slices(); the inverse's use inverse_slices(n).
int ozaki_slices();
void ozaki_set_slices(int s);
int i8mma_slices();
void i8mma_set_slices(int s);
int sliced_slices();
// Slices of the blocked inverse's products (gpb_chol.cu) at order n: ozaki_slices() if that is > 0, else OZ_INV_SLICES
// while the fused engine is on, else 0 (FP64 DMMA); always 0 when n is not a multiple of 16, so that the inverse's
// products are either all sliced or none.  The inverse takes more slices than the factor: its consumers (tr(Ky^-1 dK),
// the predictive variance) cancel and amplify the products' norm-wise error, which shrinks 2^7 per slice (DESIGN.md
// section 8).
int inverse_slices(int n);
// OZ_MMA_MAX_SLICES: what gpb_gemm_ozaki_nt and gpb_i8mma_config take on the fused engine; the kernel itself takes up to
// OZ_MMA_MAX_TILE_SLICES (in narrower tiles, gpb_ozaki_mma.cu), which only the inverse's products use.
constexpr int OZ_MMA_MAX_SLICES = 8, OZ_MMA_DEFAULT_SLICES = 8, OZ_MMA_MAX_TILE_SLICES = 9, OZ_INV_SLICES = 9;
// The fused product (gpb_ozaki_mma.cu) on slices already split by gemm_ozaki_nt_ex: a8 (m rows) and b8 (n rows), both in
// forward slice order with row pitch slices * k bytes, row scales sa / sb.
int ozaki_mma_launch(const OzEx& x, const int8_t* a8, const int8_t* b8, const double* sa, const double* sb);
// thresholds of the hooks in gpb_chol.cu
constexpr int OZ_MIN_ROWS = 4096, OZ_MIN_COLS = 1024, OZ_MIN_K = 512, OZ_TRI_STRIP = 2048, OZ_TRTRI_MIN_S = 4096;

}  // namespace gpb
