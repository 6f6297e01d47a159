"""torch.autograd.Function nodes over the native library.

The reference has no custom autograd nodes: gradients come from torch autograd through composite ops
(gptorch/functions.py:1-5 says otherwise but none exist).  Here every forward AND backward is a call (or a
short sequence of calls) into libgpb200.so; the backward formulas are the closed forms verified against the
reference's autograd in SURVEY.md section 10.
"""
import math

import torch
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from . import _native as nv

TRSV_MAX_RHS = 32  # up to this many right-hand sides use the streaming trsv kernel, beyond it the GEMM path


class Factor:
    """A lower Cholesky factor as the native library keeps it: an (n, ld) buffer whose lower triangle is L,
    plus the inverses of its 128x128 diagonal blocks."""

    __slots__ = ("buf", "ld", "n", "dinv")

    def __init__(self, buf, ld, n, dinv):
        self.buf, self.ld, self.n, self.dinv = buf, ld, n, dinv


def _dinv_of(L):
    """Diagonal-block inverses of a lower-triangular tensor, reusing the ones cached by functions.cholesky()."""
    dinv = getattr(L, "_gpb_dinv", None)
    if dinv is not None and dinv.shape[0] >= L.shape[0] and dinv.device == L.device:
        return dinv
    return nv.tri_diag_inverse(nv._c(L))


def _tinv(L, dinv):
    """T = L^-T as a dense upper-triangular tensor (n x n view of a TMA-aligned buffer)."""
    n = L.shape[0]
    buf, ld = nv.sym_buffer_from(L)
    nv.trtri_upper_(buf, ld, dinv)
    T = buf[:, :n]
    T.triu_()  # the strictly-lower off-diagonal blocks still hold L
    return T


# ------------------------------------------------------------------------------------------------------
# covariance
# ------------------------------------------------------------------------------------------------------
class KernelFn(Function):
    """K(X, X2) for the stationary kernels and Linear (gptorch/kernels.py:182-265); with `noise` (and X2 None)
    it is Ky = K(X) + noise I of GPR._compute_kyy (gptorch/models/gpr.py:69-86)."""

    @staticmethod
    def forward(ctx, kind, X, X2, ell, sigma2, noise=None):
        ctx.kind = kind
        ctx.save_for_backward(X, X2, ell, sigma2)
        return nv.kern_fwd(kind, X, X2, ell, sigma2, noise=noise if X2 is None else None)

    @staticmethod
    @once_differentiable
    def backward(ctx, G):
        X, X2, ell, sigma2 = ctx.saved_tensors
        kind = ctx.kind
        need_x, need_x2 = ctx.needs_input_grad[1], ctx.needs_input_grad[2]
        sym = X2 is None
        G = nv._c(G)
        g_ell, g_s2, g_col = nv.kern_bwd(kind, X, X2, ell, sigma2, G, need_x2 or (sym and need_x))
        gX = gX2 = None
        if need_x:
            _, _, g_row = nv.kern_bwd(kind, X if sym else X2, X, ell, sigma2, G, True, g_transposed=True)
            gX = g_row + g_col if sym else g_row
        if need_x2 and not sym:
            gX2 = g_col
        g_ell = g_ell.reshape(ell.shape) if ctx.needs_input_grad[3] else None
        g_s2 = g_s2.reshape(sigma2.shape) if (sigma2 is not None and ctx.needs_input_grad[4]) else None
        g_noise = G.diagonal().sum().reshape(1) if (len(ctx.needs_input_grad) > 5 and ctx.needs_input_grad[5]) else None
        return None, gX, gX2, g_ell, g_s2, g_noise


class LinearKdiagFn(Function):
    """Linear.Kdiag (gptorch/kernels.py:264-265): out[i] = sum_d v_d x_id^2 in one pass over X (gpb_linear_kdiag).
    The backward is an O(n D) element-wise product, left to torch."""

    @staticmethod
    def forward(ctx, X, v):
        ctx.save_for_backward(X, v)
        return nv.linear_kdiag(X, v)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        X, v = ctx.saved_tensors
        gX = (2.0 * g[:, None]) * X * v if ctx.needs_input_grad[0] else None
        gv = (g[:, None] * X * X).sum(0).reshape(v.shape) if ctx.needs_input_grad[1] else None
        return gX, gv


def _spec_terms(spec, params):
    """Resolve a composite spec -- terms of (kind, ell index or -1, sigma2 index or -1) -- against `params`."""
    return [[(k, params[ie] if ie >= 0 else None, params[isg] if isg >= 0 else None) for (k, ie, isg) in term]
            for term in spec]


def _composite_grads(spec, X, X2, params, G, need_x, need_x2):
    """Backward of K = sum_t prod_{l in t} k_l(X, X2) for an upstream gradient G: returns ([grad per param], gX, gX2).

    Leaf l of term t sees the upstream gradient G .* prod_{l' != l in t} k_l'; the product of the other leaves is
    formed by one composite forward pass (the only N x N temporary, and only for Product terms) and multiplied into
    G on the fly by gpb_kern_bwd_mul.  Sum terms (a single leaf) read G directly."""
    sym = X2 is None
    grads = [None] * len(params)
    gX = gX2 = None

    def add(i, g, like):
        if i < 0:
            return
        g = g.reshape(like.shape)
        grads[i] = g if grads[i] is None else grads[i] + g

    for term in spec:
        for li, (kind, ie, isg) in enumerate(term):
            others = [leaf for lj, leaf in enumerate(term) if lj != li]
            Mul = nv.kern_sop_fwd(_spec_terms([others], params), X, X2) if others else None
            ell = params[ie] if ie >= 0 else None
            s2 = params[isg] if isg >= 0 else None
            has_x = kind < nv.KERN_CONSTANT
            want_col = has_x and (need_x2 or (sym and need_x))
            g_ell, g_s2, g_col = nv.kern_bwd_mul(kind, X, X2, ell, s2, G, Mul, want_col, symmetric=sym)
            if ie >= 0:
                add(ie, g_ell, params[ie])
            if isg >= 0:
                add(isg, g_s2, params[isg])
            if has_x and need_x:
                _, _, g_row = nv.kern_bwd_mul(kind, X if sym else X2, X, ell, s2, G, Mul, True, g_transposed=True,
                                              symmetric=sym)
                contrib = g_row + g_col if sym else g_row
                gX = contrib if gX is None else gX + contrib
            if has_x and need_x2 and not sym:
                gX2 = g_col if gX2 is None else gX2 + g_col
    return grads, gX, gX2


class CompositeKernelFn(Function):
    """Sum / Product trees of leaf kernels (gptorch/kernels.py:286-306) in sum-of-products normal form, evaluated by
    ONE pass of gpb_kern_sop_fwd; with `noise` (and X2 None) it is Ky of GPR._compute_kyy."""

    @staticmethod
    def forward(ctx, spec, X, X2, noise, *params):
        ctx.spec = spec
        ctx.save_for_backward(X, X2, *params)
        return nv.kern_sop_fwd(_spec_terms(spec, params), X, X2, noise=noise if X2 is None else None)

    @staticmethod
    @once_differentiable
    def backward(ctx, G):
        X, X2, *params = ctx.saved_tensors
        G = nv._c(G)
        need = ctx.needs_input_grad
        grads, gX, gX2 = _composite_grads(ctx.spec, X, X2, params, G, need[1], need[2] and X2 is not None)
        g_noise = G.diagonal().sum().reshape(1) if need[3] else None
        grads = [g if need[4 + i] else None for i, g in enumerate(grads)]
        return (None, gX, gX2, g_noise) + tuple(grads)


# ------------------------------------------------------------------------------------------------------
# Cholesky and solves
# ------------------------------------------------------------------------------------------------------
def _raise_not_pd(info):
    raise torch.linalg.LinAlgError(
        "gpb_potrf_lower: the leading minor of order %d is not positive-definite (the input might not be "
        "positive-definite)." % info)


class CholeskyFn(Function):
    """Lower Cholesky (torch.cholesky at gptorch/functions.py:47).  Raises LinAlgError (a RuntimeError, which
    is what jit_op's retry loop catches, gptorch/functions.py:38) on a non-positive pivot."""

    @staticmethod
    def forward(ctx, A):
        n = A.shape[0]
        buf, ld = nv.sym_buffer_from(A)
        dinv, info = nv.potrf_(buf, ld)
        status = nv.read_info(info)  # the one host sync of a factorisation (SURVEY 7 "hard parts")
        if status != 0:
            _raise_not_pd(status)
        nv.tri_zero_upper_(buf, ld)
        L = buf[:, :n]
        ctx.save_for_backward(L, dinv)
        ctx.mark_non_differentiable(dinv)
        return L, dinv

    @staticmethod
    @once_differentiable
    def backward(ctx, gL, _g_dinv):
        L, dinv = ctx.saved_tensors
        T = _tinv(L, dinv)
        P = nv.gemm(nv.GEMM_TN, L, nv._c(gL), lower_only=True, flags=nv.GF_KLO_M)  # tril(L^T gL), L[k][m] = 0 for k < m
        P.tril_()
        P.diagonal().mul_(0.5)
        W1 = nv.gemm(nv.GEMM_NT, P, T, flags=nv.GF_KHI_M | nv.GF_KLO_N)   # Phi T^T (Phi lower, T upper)
        S = nv.gemm(nv.GEMM_NN, T, W1, flags=nv.GF_KLO_M)                 # T Phi T^T = L^-T Phi L^-1
        return 0.5 * (S + S.t())


class TrsvFn(Function):
    """x = L^-1 b (trans=False) or L^-T b (trans=True) for few right-hand sides (functions.trtrs with
    b = y - m, gptorch/models/gpr.py:62).  L is streamed once per group of 4 columns."""

    @staticmethod
    def forward(ctx, b, L, dinv, trans):
        x = nv._c(b).clone()
        nv.trsv_(nv._c(L), dinv, x, trans)
        ctx.trans = trans
        ctx.save_for_backward(L, dinv, x)
        return x

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        L, dinv, x = ctx.saved_tensors
        gb = nv._c(g).clone()
        nv.trsv_(nv._c(L), dinv, gb, not ctx.trans)
        gL = None
        if ctx.needs_input_grad[1]:
            if ctx.trans:   # x = L^-T b:  dL = -tril(x gb^T)
                gL = nv.gemm(nv.GEMM_NT, x, gb, alpha=-1.0)
            else:           # x = L^-1 b:  dL = -tril(gb x^T)
                gL = nv.gemm(nv.GEMM_NT, gb, x, alpha=-1.0)
            gL.tril_()
        return gb, gL, None, None


class TrsmRightFn(Function):
    """Out = X L^-T for a row panel X (m x n): the layout the sparse models use for A^T = Kfu L^-T
    (gptorch/models/sparse_gpr.py:132, :360 compute the transpose, L^-1 Kuf)."""

    @staticmethod
    def forward(ctx, X, L, dinv):
        m, n = X.shape
        T = None
        if m >= 2 * n and n >= 2 * nv.NB:
            # tall panel: one product with the dense inverse factor T = L^-T (upper, k <= n) writes every output
            # tile once with k up to n; the solve recursion would make log2(n/128) short-k passes over the panel
            T = _tinv(nv._gemm_operand(L.detach()), dinv)
            out = nv.gemm(nv.GEMM_NN, X, T, flags=nv.GF_KHI_N)
        else:
            buf, ld = nv._aligned_empty(m, n, X.device)
            buf[:, :n].copy_(X)
            nv.trsm_right_lt_(nv._gemm_operand(L), dinv, buf, ld)
            out = buf[:, :n]
        ctx.has_t = T is not None
        ctx.save_for_backward(L, dinv, out, T)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, G):
        L, dinv, out, T = ctx.saved_tensors
        if T is None:
            T = _tinv(L, dinv)
        G = nv._c(G)
        # T is upper triangular: (G T^T)[., n] only needs k >= n; -tril(T Q) only needs the lower part of Q
        gX = nv.gemm(nv.GEMM_NT, G, T, flags=nv.GF_KLO_N) if ctx.needs_input_grad[0] else None   # G L^-1 = G T^T
        gL = None
        if ctx.needs_input_grad[1]:
            Q = nv.gemm(nv.GEMM_TN, G, out, lower_only=True)             # tril(G^T Out)
            Q.tril_()
            gL = nv.gemm(nv.GEMM_NN, T, Q, alpha=-1.0, lower_only=True, flags=nv.GF_KLO_M)   # -L^-T G^T Out
            gL.tril_()
        return gX, gL, None


class TrsmLeftTFn(Function):
    """X = L^-T B for many right-hand sides (functions.trtrs with an upper-triangular matrix, lower=False,
    gptorch/functions.py:71-76), as one product with the dense upper-triangular T = L^-T; differentiable in B and L."""

    @staticmethod
    def forward(ctx, B, L, dinv):
        T = _tinv(nv._gemm_operand(L.detach()), dinv)
        X = nv.gemm(nv.GEMM_NN, T, nv._c(B), flags=nv.GF_KLO_M)      # T[m][k] = 0 for k < m
        ctx.save_for_backward(T, X)
        return X

    @staticmethod
    @once_differentiable
    def backward(ctx, G):
        T, X = ctx.saved_tensors
        gB = nv.gemm(nv.GEMM_TN, T, nv._c(G))                         # L^-1 G = T^T G
        gL = None
        if ctx.needs_input_grad[1]:                                   # X = L^-T B:  dL = -tril(X gB^T)
            gL = nv.gemm(nv.GEMM_NT, X, gB, alpha=-1.0, lower_only=True)
            gL.tril_()
        return gB if ctx.needs_input_grad[0] else None, gL, None


class CholeskyInverseFn(Function):
    """(L L^T)^-1 from a lower Cholesky factor (functions.cholesky_inverse, gptorch/functions.py:50-54): blocked
    trtri + lauum in place, assembled to a full symmetric matrix.  backward: with S = G + G^T,
    dL = -tril(Kinv S L^-T)."""

    @staticmethod
    def forward(ctx, L):
        buf, ld = nv.sym_buffer_from(L.detach())
        dinv = nv.tri_diag_inverse(buf)
        ctx.save_for_backward(L.detach(), dinv)
        kd = nv.potri_(buf, ld, dinv)
        Kinv = nv.potri_assemble(buf, ld, kd)
        ctx.kinv = Kinv
        return Kinv

    @staticmethod
    @once_differentiable
    def backward(ctx, G):
        L, dinv = ctx.saved_tensors
        Kinv, ctx.kinv = ctx.kinv, None
        if Kinv is None:
            raise RuntimeError("CholeskyInverseFn: the inverse was released by a previous backward pass")
        G = nv._c(G)
        S = nv._c(G + G.t())
        T = _tinv(nv._gemm_operand(L), dinv)
        M1 = nv.gemm(nv.GEMM_NN, Kinv, S)
        gL = nv.gemm(nv.GEMM_NN, M1, T, alpha=-1.0, flags=nv.GF_KHI_N)   # T[k][n] = 0 for k > n
        gL.tril_()
        return gL


class TriInvTFn(Function):
    """T = L^-T as a dense upper-triangular matrix, differentiable in L:  dL = -tril(T G^T T).  Used where the sparse
    models apply L^-1 . L^-T to M x M quantities instead of solving against tall panels."""

    @staticmethod
    def forward(ctx, L, dinv):
        T = _tinv(nv._gemm_operand(L.detach()), dinv)
        ctx.save_for_backward(T)
        return T

    @staticmethod
    @once_differentiable
    def backward(ctx, G):
        (T,) = ctx.saved_tensors
        Gu = torch.triu(nv._c(G))                                       # T is upper triangular: only those entries count
        M1 = nv.gemm(nv.GEMM_NT, T, Gu, flags=nv.GF_KLO_M | nv.GF_KLO_N)   # T G^T  (both upper: k >= row, k >= col)
        gL = nv.gemm(nv.GEMM_NN, M1, T, alpha=-1.0, flags=nv.GF_KHI_N)    # (T G^T) T
        gL.tril_()
        return gL, None


class SyrkFn(Function):
    """U U^T (full symmetric result from the lower tiles); backward dU = (G + G^T) U.  `upper`: U is upper triangular
    (U[i][k] = 0 for k < i), which halves the k-range."""

    @staticmethod
    def forward(ctx, U, upper=False):
        ctx.upper = bool(upper)
        ctx.save_for_backward(U)
        flags = (nv.GF_KLO_M | nv.GF_KLO_N) if upper else 0
        C = nv.gemm(nv.GEMM_NT, U, U, lower_only=True, flags=flags)
        return torch.tril(C) + torch.tril(C, -1).t()

    @staticmethod
    @once_differentiable
    def backward(ctx, G):
        (U,) = ctx.saved_tensors
        S = nv._c(G + G.t())
        gU = nv.gemm(nv.GEMM_NN, S, U)
        if ctx.upper:
            gU.triu_()
        return gU, None


class RowSumSqFn(Function):
    """sum(A ** 2, dim=1) for a row panel in one pass (gpb_rowdot): the variance reductions of the predictive equations,
    (A * A).sum(0) of gptorch/models/gpr.py:109-113 and sum(alpha ** 2, dim=1), sum(gamma ** 2, dim=1) of
    gptorch/models/sparse_gpr.py:186-190, :374-379 (panels are row-major here), without the [rows x cols] temporary."""

    @staticmethod
    def forward(ctx, A):
        A = nv._c(A)
        ctx.save_for_backward(A)
        return nv.rowdot(A, A)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        (A,) = ctx.saved_tensors
        return A * (2.0 * g)[:, None]


SVGP_SPLITS = 4


class SvgpMomentsFn(Function):
    """(Kfu m, diag(Kfu C Kfu^T)) for a row panel Kfu [B, M], a symmetric C [M, M] and m [M, dy]: the q(f) moments of
    SVGP._predict (gptorch/models/sparse_gpr.py:357-379) with the M x M algebra done first,
        mean_i = k_i^T Kuu^-1 m_u,     var_i - Kdiag_i = k_i^T C k_i,   C = Kuu^-1 (S - Kuu) Kuu^-1,
    i.e. ONE panel product Kfu C (2 B M^2 flop) instead of alpha = L^-1 Kuf, gamma = alpha beta and their adjoints
    (6 B M^2 per loss+grad in the reference order, 3 B M^2 here).  backward: dKfu = 2 g_var . (Kfu C) + g_mean m^T (in
    place on the saved product), dC = Kfu^T diag(g_var) Kfu (split-K Gram product), dm = Kfu^T g_mean."""

    @staticmethod
    def forward(ctx, Kfu, C, mvec):
        Kfu, C, mvec = nv._c(Kfu), nv._gemm_operand(C), nv._c(mvec)
        with nv.phase("svgp_panel_gemm"):
            KC = nv.gemm(nv.GEMM_NN, Kfu, C)
        with nv.phase("svgp_reduce"):
            q = nv.rowdot(KC, Kfu)
            mean = nv.gemv_n(Kfu, mvec)
        ctx.save_for_backward(Kfu, KC, mvec)
        ctx.used = False
        return mean, q

    @staticmethod
    @once_differentiable
    def backward(ctx, g_mean, g_q):
        if ctx.used:
            raise RuntimeError("SvgpMomentsFn: the saved panel product was consumed by a previous backward pass")
        ctx.used = True
        Kfu, KC, mvec = ctx.saved_tensors
        g_mean, g_q = nv._c(g_mean), nv._c(g_q).reshape(-1)
        b, m = Kfu.shape
        gC = gm = None
        if ctx.needs_input_grad[1]:
            with nv.phase("svgp_gram"):
                Ks = Kfu * g_q[:, None]
                ldm = m + (m & 1)
                kper = max(16, ((b + SVGP_SPLITS - 1) // SVGP_SPLITS + 15) // 16 * 16)
                C3 = torch.zeros((SVGP_SPLITS, m, ldm), dtype=torch.float64, device=Kfu.device)
                nv.gemm_splitk(nv.GEMM_TN, Ks, Kfu, kper, C3, beta=0.0, lower_only=True)
                del Ks
                gC = C3.sum(0)[:, :m]
                gC = torch.tril(gC) + torch.tril(gC, -1).t()
        if ctx.needs_input_grad[2]:
            gm = torch.zeros_like(mvec)
            nv.gemv_t(Kfu, g_mean, gm, beta=0.0)
        gK = None
        if ctx.needs_input_grad[0]:
            with nv.phase("svgp_reduce"):
                gK = nv.rows_scale_add_outer_(KC, s=g_q, scale=2.0, G=g_mean, V=mvec)   # consumes the saved product
        return gK, gC, gm


class LogDetFn(Function):
    """sum(log(diag(L)))  (functions.lt_log_determinant, gptorch/functions.py:61-68)."""

    @staticmethod
    def forward(ctx, L):
        ctx.save_for_backward(L)
        return nv.logdet_sumsq(nv._c(L))[0]

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        (L,) = ctx.saved_tensors
        return torch.diag_embed(g / L.diagonal())


class GemmFn(Function):
    """C = A B^T (NT), A^T B (TN) or A B (NN) on the DMMA engine, differentiable in A and B.

    `b_lower`: B is a square lower-triangular matrix (NN mode only: C = A B with B[k][n] = 0 for k < n).  The zero
    half of the k-range is skipped in forward and backward, and only the lower part of dB is formed.
    """

    @staticmethod
    def forward(ctx, mode, A, B, b_lower=False):
        ctx.mode, ctx.b_lower = mode, bool(b_lower) and mode == nv.GEMM_NN
        ctx.save_for_backward(A, B)
        return nv.gemm(mode, A, B, flags=nv.GF_KLO_N if ctx.b_lower else 0)

    @staticmethod
    @once_differentiable
    def backward(ctx, G):
        A, B = ctx.saved_tensors
        G = nv._c(G)
        need_a, need_b = ctx.needs_input_grad[1], ctx.needs_input_grad[2]
        gA = gB = None
        if ctx.mode == nv.GEMM_NT:      # C = A B^T
            if need_a: gA = nv.gemm(nv.GEMM_NN, G, B)
            if need_b: gB = nv.gemm(nv.GEMM_TN, G, A)
        elif ctx.mode == nv.GEMM_TN:    # C = A^T B
            if need_a: gA = nv.gemm(nv.GEMM_NT, B, G)
            if need_b: gB = nv.gemm(nv.GEMM_NN, A, G)
        elif ctx.b_lower:               # C = A B, B lower triangular
            if need_a: gA = nv.gemm(nv.GEMM_NT, G, B, flags=nv.GF_KHI_N)   # (G B^T)[., n]: B[n][k] = 0 for k > n
            if need_b:
                gB = nv.gemm(nv.GEMM_TN, A, G, lower_only=True)
                gB.tril_()
        else:                           # C = A B
            if need_a: gA = nv.gemm(nv.GEMM_NT, G, B)
            if need_b: gB = nv.gemm(nv.GEMM_TN, A, G)
        return None, gA, gB, None


# ------------------------------------------------------------------------------------------------------
# fused GPR log marginal likelihood
# ------------------------------------------------------------------------------------------------------
JITTER_TRIES = 10  # gptorch/functions.py:21
VFE_PANEL_CACHE_BYTES = 16 << 30   # keep the streamed panels (Kfu, or A^T in the reference order) for backward up to this size
VFE_SPLITS = 16    # k-slices of the streamed Gram products (fills the GPU when M x M has few tiles)


class GPRLogLikFn(Function):
    """GPR.log_likelihood (gptorch/models/gpr.py:47-67) as one node.

    forward : Ky = K(X) + noise I (lower tiles only) -> potrf (same jitter schedule as functions.jit_op,
              gptorch/functions.py:28-43) -> alpha = L^-1 resid -> -1/2 |alpha|^2 - dy sum log L_ii - const.
    backward: a = L^-T alpha ; Kinv = potri(L) in place ; W = 1/2 (dy Kinv - a a^T) reduced against
              dK/d(ell, sigma2) on the fly ; d/d noise = tr W ; d/d resid = -a.       (SURVEY 10)
              When X requires a gradient, a second pass reduces the same W against dK/dX (gpb_gpr_grad's gX).
    One N^2 buffer in total; N^3/3 + 2N^3/3 flops.
    """

    @staticmethod
    def forward(ctx, kind, X, resid, ell, sigma2, noise):
        n, dy = resid.shape
        X = nv._c(X)
        buf, ld = nv._aligned_empty(n, n, X.device)
        dinv = None
        for attempt in range(JITTER_TRIES + 1):
            with nv.phase("kern_fwd"):
                nv.kern_fwd(kind, X, None, ell, sigma2, noise=noise, lower=True, out=buf, ldk=ld)
            if attempt > 0:
                nv.add_diag_(buf, ld, 10.0 ** (-JITTER_TRIES + attempt - 1))
            with nv.phase("potrf"):
                dinv, info = nv.potrf_(buf, ld)
            if nv.read_info(info) == 0:
                break
        else:
            raise RuntimeError("Max tries exceeded.")
        with nv.phase("solve_logdet"):
            alpha = nv._c(resid).clone()
            nv.trsv_(buf, dinv, alpha, False)
            red = nv.logdet_sumsq(buf, alpha)
        loglik = (-0.5 * red[1] - dy * red[0] - 0.5 * dy * n * math.log(2.0 * math.pi)).reshape(1)
        ctx.kind, ctx.ld, ctx.used = kind, ld, False
        ctx.save_for_backward(X, ell, sigma2, buf, dinv, alpha)
        return loglik

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        if ctx.used:
            raise RuntimeError("GPRLogLikFn: the factor buffer was consumed by a previous backward pass")
        ctx.used = True
        X, ell, sigma2, buf, dinv, alpha = ctx.saved_tensors
        dy = alpha.shape[1]
        with nv.phase("solve_logdet"):
            a = alpha.clone()
            nv.trsv_(buf, dinv, a, True)                 # a = Ky^-1 resid
        with nv.phase("potri"):
            kd = nv.potri_(buf, ctx.ld, dinv)            # Kinv, in place (L is gone after this)
        gX = torch.empty_like(X) if ctx.needs_input_grad[1] else None
        with nv.phase("gpr_grad"):
            g_ell, g_s2, g_noise = nv.gpr_grad(ctx.kind, X, ell, sigma2, buf, ctx.ld, kd, a, gX=gX)
        g = g.reshape(())
        # the native reduction returns d(-loglik)/d theta; the node's output is +loglik
        out_ell = (-g) * g_ell.reshape(ell.shape) if ctx.needs_input_grad[3] else None
        out_s2 = (-g) * g_s2.reshape(sigma2.shape) if (sigma2 is not None and ctx.needs_input_grad[4]) else None
        out_noise = (-g) * g_noise.reshape(-1) if ctx.needs_input_grad[5] else None
        out_resid = (-g) * a if ctx.needs_input_grad[2] else None
        out_x = (-g) * gX if gX is not None else None
        return None, out_x, out_resid, out_ell, out_s2, out_noise


class GPRCompositeLogLikFn(Function):
    """GPR.log_likelihood with a composite kernel (BASELINE config #1: Linear + Rbf + Constant,
    examples/regression_1d.py:42) as one node: same N^3-flop structure as GPRLogLikFn -- potrf, blocked inverse --
    with W = 1/2 (dy Kinv - a a^T) assembled once (dense, symmetric) and reduced leaf by leaf by _composite_grads."""

    @staticmethod
    def forward(ctx, spec, X, resid, noise, *params):
        n, dy = resid.shape
        X = nv._c(X)
        buf, ld = nv._aligned_empty(n, n, X.device)
        terms = _spec_terms(spec, params)
        for attempt in range(JITTER_TRIES + 1):
            with nv.phase("kern_fwd"):
                nv.kern_sop_fwd(terms, X, None, noise=noise, lower=True, out=buf, ldk=ld)
            if attempt > 0:
                nv.add_diag_(buf, ld, 10.0 ** (-JITTER_TRIES + attempt - 1))
            with nv.phase("potrf"):
                dinv, info = nv.potrf_(buf, ld)
            if nv.read_info(info) == 0:
                break
        else:
            raise RuntimeError("Max tries exceeded.")
        with nv.phase("solve_logdet"):
            alpha = nv._c(resid).clone()
            nv.trsv_(buf, dinv, alpha, False)
            red = nv.logdet_sumsq(buf, alpha)
        loglik = (-0.5 * red[1] - dy * red[0] - 0.5 * dy * n * math.log(2.0 * math.pi)).reshape(1)
        ctx.spec, ctx.ld, ctx.used = spec, ld, False
        ctx.save_for_backward(X, buf, dinv, alpha, *params)
        return loglik

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        if ctx.used:
            raise RuntimeError("GPRCompositeLogLikFn: the factor buffer was consumed by a previous backward pass")
        ctx.used = True
        X, buf, dinv, alpha, *params = ctx.saved_tensors
        dy = alpha.shape[1]
        with nv.phase("solve_logdet"):
            a = alpha.clone()
            nv.trsv_(buf, dinv, a, True)
        with nv.phase("potri"):
            kd = nv.potri_(buf, ctx.ld, dinv)
            W = nv.potri_assemble(buf, ctx.ld, kd)                                   # full symmetric Ky^-1
        with nv.phase("gpr_grad"):
            nv.gemm(nv.GEMM_NT, a, a, alpha=-0.5, beta=0.5 * dy, C=W)                # W = 1/2 (dy Kinv - a a^T)
            grads, gX, _ = _composite_grads(ctx.spec, X, None, params, W, ctx.needs_input_grad[1], False)
            g_noise = W.diagonal().sum().reshape(1)
        g = g.reshape(())
        need = ctx.needs_input_grad
        out_x = (-g) * gX if gX is not None else None
        return (None, out_x, (-g) * a if need[2] else None, (-g) * g_noise if need[3] else None) + tuple(
            ((-g) * gr if (gr is not None and need[4 + i]) else None) for i, gr in enumerate(grads))


# ------------------------------------------------------------------------------------------------------
# cached GPR posterior: predictive mean and variance, differentiable in the test inputs only
# ------------------------------------------------------------------------------------------------------
class GPRPredFn(Function):
    """(mean [n*, dy], diagonal variance [n*, dy]) of GPR._predict (gptorch/models/gpr.py:88-117) against a cached
    a = Ky^-1 (y - m(X)) and the full symmetric Ky^-1, for a stationary kernel (the mean function is added outside).

    forward : K* = K(x*, X) (gpb_kern_fwd) ; mean = K* a (gpb_gemv_n) ; Q = K* Ky^-1 (one DMMA GEMM) ;
              var = sigma2 - rowdot(K*, Q).  Q is kept for the backward pass; K* is not.
    backward: dLoss/dK*_tj = W_tj = g_mean_t . a_j - 2 g_var_t Q_tj is reduced against dk(x*_t, x_j)/dx*_t on the fly
              by gpb_pred_gx -- no solve, no [n*, N] panel gradient.  Only x* receives a gradient: X, a, Ky^-1 and the
              hyper-parameters are constants of the posterior.
    """

    @staticmethod
    def forward(ctx, kind, x_new, X, a, Kinv, ell, sigma2):
        ns, dy = x_new.shape[0], a.shape[1]
        Ks = nv.kern_fwd(kind, x_new, X, ell, sigma2)
        mean = nv.gemv_n(Ks, a)
        Q = nv.gemm(nv.GEMM_NN, Ks, Kinv)
        var = nv._c(sigma2).reshape(1).repeat(ns)
        nv.rowdot(Ks, Q, alpha=-1.0, out=var, beta=1.0)
        ctx.kind = kind
        ctx.save_for_backward(x_new, X, a, Q, ell, sigma2)
        return mean, var[:, None].expand(ns, dy).contiguous()

    @staticmethod
    @once_differentiable
    def backward(ctx, g_mean, g_var):
        x_new, X, a, Q, ell, sigma2 = ctx.saved_tensors
        gx = None
        if ctx.needs_input_grad[1]:
            gx = nv.pred_gx(ctx.kind, x_new, X, ell, sigma2, a, g_mean, g_var.sum(1), Q)
        return None, gx, None, None, None, None, None


# ------------------------------------------------------------------------------------------------------
# VFE sufficient statistics, streamed over row chunks of X
# ------------------------------------------------------------------------------------------------------
def kuu_condition_estimate(L, T, iters=6):
    """Estimate of cond_2(Kuu) = lambda_max(L L^T) * lambda_max(T T^T) (T = L^-T) by two short power iterations on the
    native matrix-vector kernel.  Power iteration approaches each factor from below, so the result is a (slightly low)
    estimate; callers compare it with a threshold that leaves a safety margin."""
    m = L.shape[0]
    Lt, Tt = L.t().contiguous(), T.t().contiguous()
    out = []
    # Kuu is entrywise positive for the stationary families: its dominant (Perron) eigenvector is close to the start
    # vector and half the iterations suffice; the small end of the spectrum (T T^T) gets the full count
    for A, At, its in ((L, Lt, max(2, iters // 2)), (T, Tt, iters)):                 # v <- A (A^T v)
        v = torch.full((m, 1), 1.0 / math.sqrt(m), dtype=torch.float64, device=L.device)
        u = torch.empty_like(v)
        lam = None
        for _ in range(its):
            nv.gemv_t(A, v, u, beta=0.0)            # u = A^T v
            nv.gemv_t(At, u, v, beta=0.0)           # v = A u
            lam = torch.linalg.vector_norm(v)
            v = v / lam
        out.append(lam)
    return float((out[0] * out[1]).item())


class VfeStatsFn(Function):
    """(A A^T, A Y) with A = L^-1 Kuf (gptorch/models/sparse_gpr.py:127-137) without ever holding Kuf.

    Rows of X are processed in chunks.  Two forms, selected by `phi_form`:

    * reference order (phi_form False): Kfu_c = K(X_c, Z) -> At_c = Kfu_c L^-T -> AA += At_c^T At_c, AY += At_c^T Y_c --
      solve first, then the Gram product, exactly the reference's sequence of roundings; 5 N M^2 flop per loss+grad.
    * Phi form (phi_form True): Phi += Kfu_c^T Kfu_c, psi += Kfu_c^T Y_c over the stream, then the M x M congruence
      AA = L^-1 Phi L^-T, AY = L^-1 psi once -- 3 N M^2 flop per loss+grad (SURVEY 8d's algorithmic count), no solved
      panels to keep or rebuild for the backward pass.  The congruence amplifies the rounding of Phi by cond(Kuu)
      (normal-equations effect; the reference order only by its square root), so the caller enables it only when the
      estimated cond_2(Kuu) keeps the error far inside the parity tolerances (VFE._stats, settings.vfe_phi_form).

    backward re-streams the chunks: the gradient with respect to a panel is G_c = At_c (S L^-1) + Y_c (L^-T gAY)^T
    (reference order) or G_c = Kfu_c (L^-T S L^-1) + Y_c (L^-T gAY)^T (Phi form), S = gAA + gAA^T, reduced against
    dK/d(ell, sigma2, Z) by gpb_kern_bwd.  With torch.distributed initialised and `group` given, rows are this rank's
    shard and the M x M statistics / the streamed gradients are all-reduced (SURVEY 8e).
    """

    @staticmethod
    def forward(ctx, kind, X, Y, Z, ell, sigma2, L, chunk, group, phi_form=False):
        X, Y, Z = nv._c(X), nv._c(Y), nv._c(Z)
        Lc = nv._gemm_operand(L)
        dinv = _dinv_of(L)
        T = _tinv(Lc, dinv)
        n, m, dy = X.shape[0], Z.shape[0], Y.shape[1]
        ldm = m + (m & 1)
        # Keep the streamed panels for the backward pass when they fit a modest budget (N*M*8 bytes <= 16 GiB of the
        # 180 GB); otherwise the backward pass rebuilds them chunk by chunk (one more covariance build, plus the solve in
        # the reference order).
        keep = any(ctx.needs_input_grad) and n * ldm * 8 <= VFE_PANEL_CACHE_BYTES
        cache = []
        if phi_form:
            # ONE native call streams the chunks: panel build, split-K Gram product, psi (gpb_kuf_stats_fwd)
            with nv.phase("vfe_stats_fwd"):
                AAf, AYf, kfu = nv.kuf_stats_fwd(kind, X, Y, Z, ell, sigma2, chunk, cache=keep)
            cache = kfu
        else:
            # The M x M Gram output has only (M/128)^2/2 tiles, far fewer than the GPU has SMs, so the long k = rows
            # dimension is cut into VFE_SPLITS slices that accumulate into separate slots, summed at the end.
            kper = VfeStatsFn._k_per_split(min(chunk, n))
            AA3 = torch.zeros((VFE_SPLITS, m, ldm), dtype=torch.float64, device=X.device)
            AYf = torch.zeros((m, dy), dtype=torch.float64, device=X.device)
            for s in range(0, n, chunk):
                e = min(n, s + chunk)
                P = VfeStatsFn._panel(kind, X[s:e], Z, ell, sigma2, T)
                if keep:
                    cache.append(P)
                with nv.phase("vfe_gram"):
                    nv.gemm_splitk(nv.GEMM_TN, P, P, kper, AA3, beta=1.0, lower_only=True)
                    nv.gemv_t(P, Y[s:e], AYf, beta=1.0)
                del P
            AAf = AA3.sum(0)[:, :m]
            AAf = torch.tril(AAf) + torch.tril(AAf, -1).t()
        # sum_i k(x_i, x_i) = n * sigma2 for a stationary kernel (gptorch/kernels.py:174-179); sum Y^2
        scal = torch.stack([sigma2.reshape(()) * float(n), nv.logdet_sumsq(None, Y)[1]])
        if group is not None:
            AAf, AYf = AAf.contiguous(), AYf.contiguous()
            torch.distributed.all_reduce(AAf, group=group)
            torch.distributed.all_reduce(AYf, group=group)
            torch.distributed.all_reduce(scal, group=group)
        if phi_form:
            with nv.phase("vfe_congruence"):
                PhiT = nv.gemm(nv.GEMM_NN, AAf, T, flags=nv.GF_KHI_N)          # Phi L^-T  (T upper: k <= n)
                AAf = nv.gemm(nv.GEMM_TN, T, PhiT, flags=nv.GF_KHI_M)          # L^-1 Phi L^-T
                AAf = 0.5 * (AAf + AAf.t())
                AYf = nv.gemm(nv.GEMM_TN, T, AYf, flags=nv.GF_KHI_M)           # L^-1 psi
        ctx.kind, ctx.chunk, ctx.group, ctx.n_local, ctx.phi_form = kind, chunk, group, n, bool(phi_form)
        ctx.panels = cache if (keep and cache is not None and (phi_form or len(cache))) else None
        ctx.save_for_backward(X, Y, Z, ell, sigma2, T, AAf, AYf)
        return AAf, AYf, scal[0], scal[1]

    @staticmethod
    def _k_per_split(rows):
        per = (rows + VFE_SPLITS - 1) // VFE_SPLITS
        return max(16, (per + 15) // 16 * 16)

    @staticmethod
    def _panel(kind, Xc, Z, ell, sigma2, T):
        """One row chunk: Kfu_c = K(Xc, Z) (T None) or A_c^T = Kfu_c L^-T as ONE product with the dense upper-triangular
        T = L^-T (k <= n): every output tile is written once with k up to M, instead of the solve recursion's many
        short-k passes."""
        with nv.phase("vfe_kern_fwd"):
            Kfu = nv.kern_fwd(kind, Xc, Z, ell, sigma2)
        if T is None:
            return Kfu
        with nv.phase("vfe_trsm"):
            return nv.gemm(nv.GEMM_NN, Kfu, T, flags=nv.GF_KHI_N)

    @staticmethod
    @once_differentiable
    def backward(ctx, gAA, gAY, g_kd, _g_yy):
        X, Y, Z, ell, sigma2, T, AA, AY = ctx.saved_tensors
        kind, chunk, group, phi = ctx.kind, ctx.chunk, ctx.group, ctx.phi_form
        n = X.shape[0]
        S = nv._c(gAA + gAA.t())
        gAY = nv._c(gAY)
        R = nv.gemm(nv.GEMM_NT, S, T, flags=nv.GF_KLO_N)   # S L^-1 = S T^T
        if phi:
            R = nv.gemm(nv.GEMM_NN, T, R, flags=nv.GF_KLO_M)   # L^-T S L^-1  (T[m][k] = 0 for k < m)
        w = nv.gemm(nv.GEMM_NN, T, gAY)          # L^-T gAY   (m x dy)
        panels, ctx.panels = ctx.panels, None
        # dLoss/dX: each chunk's panel gradient reduced with X and Z exchanged.  The rows are this rank's own, so it is
        # not all-reduced; sum Kdiag = n sigma2 does not depend on X.
        gX = torch.empty_like(X) if ctx.needs_input_grad[1] else None
        if phi:
            with nv.phase("vfe_stats_bwd"):      # ONE native call re-streams the chunks (gpb_kuf_stats_bwd)
                g_ell, g_s2, gZ = nv.kuf_stats_bwd(kind, X, Y, Z, ell, sigma2, chunk, R, w, kfu=panels, gX=gX)
            del panels
        else:
            g_ell = torch.zeros_like(ell.reshape(-1))
            g_s2 = torch.zeros(1, dtype=torch.float64, device=X.device)
            gZ = torch.zeros_like(Z)
            for ci, s in enumerate(range(0, n, chunk)):
                e = min(n, s + chunk)
                if panels is not None:
                    P = panels[ci]
                    panels[ci] = None
                else:
                    P = VfeStatsFn._panel(kind, X[s:e], Z, ell, sigma2, T)
                with nv.phase("vfe_bwd_gemm"):
                    G = nv.gemm(nv.GEMM_NN, P, R)
                    nv.gemm(nv.GEMM_NT, Y[s:e], w, beta=1.0, C=G)
                del P
                with nv.phase("vfe_kern_bwd"):
                    ge, gs, gz = nv.kern_bwd(kind, X[s:e], Z, ell, sigma2, G, True)
                    if gX is not None:
                        gX[s:e] = nv.kern_bwd(kind, Z, X[s:e], ell, sigma2, G, True, g_transposed=True)[2]
                del G
                g_ell += ge
                g_s2 += gs
                gZ += gz
        g_s2 += g_kd * float(ctx.n_local)
        if group is not None:
            flat = torch.cat([g_ell, g_s2, gZ.reshape(-1)])
            torch.distributed.all_reduce(flat, group=group)
            g_ell, g_s2, gZ = flat[: g_ell.numel()], flat[g_ell.numel(): g_ell.numel() + 1], flat[g_ell.numel() + 1:].reshape(Z.shape)
        Q = nv.gemm(nv.GEMM_NN, S, AA)
        nv.gemm(nv.GEMM_NT, gAY, AY, beta=1.0, C=Q)
        gL = nv.gemm(nv.GEMM_NN, T, Q, alpha=-1.0, flags=nv.GF_KLO_M)
        gL.tril_()
        return (None, gX, None, gZ if ctx.needs_input_grad[3] else None,
                g_ell.reshape(ell.shape) if ctx.needs_input_grad[4] else None,
                g_s2.reshape(sigma2.shape) if (sigma2 is not None and ctx.needs_input_grad[5]) else None,
                gL if ctx.needs_input_grad[6] else None, None, None, None)
