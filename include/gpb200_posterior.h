/* gpb200_posterior.h -- entry points of libgpb200.so for predictions from a cached GPR posterior (GPR.posterior()).
 *
 * A companion of gpb200.h with the same conventions (fp64 row-major device matrices, leading dimensions in elements,
 * device hyper-parameters, `stream` a cudaStream_t passed as void*, 0 = launched, GPB_ERR_* = rejected).  The core ABI
 * of the training path stays in gpb200.h; what a cached posterior adds is declared here.  Available from
 * gpb_version() >= 102.
 */
#ifndef GPB200_POSTERIOR_H_
#define GPB200_POSTERIOR_H_

#include "gpb200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Test-input gradient of the cached posterior's predictions.  For the predictive mean = K(x*, X) a (ns x dy) and the
 * diagonal variance var = sigma2 - rowdot(K(x*, X), Q) with Q = K(x*, X) Ky^-1 (ns x n, ldq) and
 * a = Ky^-1 (y - m(X)) (n x dy, lda), write
 *    gXs[t][d] = sum_j W_tj dk(x*_t, x_j)/dx*_td,   W_tj = g_mean[t] . a[j] - 2 g_var[t] Q[t][j],
 * the gradient with respect to the test inputs x* (ns x D, ldxs) of a loss with upstream gradients g_mean (ns x dy,
 * ldgm) and g_var (ns), without forming W or dK.  Stationary families only (not GPB_KERN_LINEAR), D <= 160.  Each
 * test row's sum is formed in a fixed order: the result is bitwise reproducible.  Replaces the autograd backward of
 * K(x*, X) -> trtrs -> row sums of squares in GPR._predict (gptorch/models/gpr.py:88-117) for a fixed factor.
 * Arguments are validated before any CUDA call (GPB_ERR_BADARG / GPB_ERR_UNSUPPORTED). */
int gpb_pred_gx(int kind, const double* Xs, int ns, long ldxs, const double* X, int n, long ldx, int D,
                const double* ell, int ell_len, const double* sigma2, const double* a, int dy, long lda,
                const double* g_mean, long ldgm, const double* g_var, const double* Q, long ldq, double* gXs, long ldgx,
                void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GPB200_POSTERIOR_H_ */
