"""Functional (non-autograd) wrappers over the C ABI: allocate outputs/workspaces with torch, pass raw pointers.

torch is used here for device memory and the current stream only; every computation happens in
libgpb200.so.  Shapes follow the reference: row-major fp64 2-D tensors (gptorch/util.py:11-12).
"""
import torch

from . import _lib
from ._lib import ptr, stream_ptr, call, query

NB = 128


class PhaseTimer:
    """Optional CUDA-event timing of named phases on the current stream (used by bench.py only).

    ``with phase("potrf"):`` records start/end events when a timer is installed; otherwise it is a no-op.
    """

    def __init__(self):
        self.records = []   # (name, start_event, end_event)

    def totals_ms(self):
        torch.cuda.synchronize()
        out = {}
        for name, e0, e1 in self.records:
            out[name] = out.get(name, 0.0) + e0.elapsed_time(e1)
        return out


_timer = None


def install_timer(timer):
    global _timer
    _timer = timer


class phase:
    def __init__(self, name):
        self.name = name

    def __enter__(self):
        if _timer is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e0.record()
        return self

    def __exit__(self, *exc):
        if _timer is not None:
            e1 = torch.cuda.Event(enable_timing=True)
            e1.record()
            _timer.records.append((self.name, self.e0, e1))
        return False


# ---------------------------------------------------------------------------------------------- factorisation status
_deferred_info = None   # device int32 [1]: max of the LAPACK-style `info` values seen while host reads are deferred


def read_info(info):
    """Status of a factorisation: normally ONE host read of the device int (the only sync of an evaluation).  While
    an evaluation is being captured into / replayed from a CUDA graph (gptorch_b200/model.py GraphedEvaluation) the
    host cannot read: the value is folded into a device accumulator that the replay returns with the loss, and the
    caller proceeds as if the factorisation had succeeded."""
    if _deferred_info is not None:
        torch.maximum(_deferred_info, info.reshape(-1)[:1], out=_deferred_info)
        return 0
    return int(info.item())


class deferred_info:
    """Context manager: route read_info() into `accumulator` (device int32 [1])."""

    def __init__(self, accumulator):
        self.acc = accumulator

    def __enter__(self):
        global _deferred_info
        self.prev, _deferred_info = _deferred_info, self.acc
        return self.acc

    def __exit__(self, *exc):
        global _deferred_info
        _deferred_info = self.prev
        return False


def launch_count():
    return _lib.load().gpb_launch_count()


def reset_launch_count():
    _lib.load().gpb_reset_launch_count()

def dmma_issue_peak_tflops(iters=20000, repeats=5):
    """FP64 DMMA issue-rate ceiling of the current device, measured live (gpb_dmma_issue_probe, CUDA events, best
    of `repeats` after one warm-up launch)."""
    import ctypes
    sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    scratch = torch.empty(2 * sms * 512, dtype=torch.float64, device="cuda")
    flop = ctypes.c_double(0.0)
    best = float("inf")
    for i in range(repeats + 1):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        call("gpb_dmma_issue_probe", int(iters), ptr(scratch), scratch.numel() * 8, ctypes.byref(flop), stream_ptr())
        e1.record()
        torch.cuda.synchronize()
        if i:
            best = min(best, e0.elapsed_time(e1))
    return flop.value / best / 1e9


KIND = {"Rbf": 0, "SquaredExponential": 0, "Exp": 1, "Matern12": 1, "Matern32": 2, "Matern52": 3, "Linear": 4,
        "Periodic": 5, "Constant": 6, "Bias": 6, "White": 7}
KERN_LINEAR, KERN_CONSTANT, KERN_WHITE = 4, 6, 7
SOP_MAX_TERMS, SOP_MAX_LEAVES = 8, 16      # gpb_kern_sop_fwd limits (include/gpb200.h)


def _c(t):
    """fp64 row-major view of t: 1-D/0-D tensors are made contiguous; a 2-D tensor is accepted as is when its
    rows are dense (stride(1) == 1) even if padded (stride(0) > shape[1]), otherwise it is copied."""
    if t.dtype != torch.float64:
        t = t.to(torch.float64)
    if t.dim() == 2 and t.stride(1) == 1 and t.stride(0) >= max(t.shape[1], 1) and t.shape[0] > 1:
        return t
    return t.contiguous()


def _npad(n):
    return (n + NB - 1) // NB * NB


def _aligned_empty(rows, cols, device):
    """rows x cols fp64 buffer whose leading dimension is even (TMA needs 16-byte row strides)."""
    ld = cols + (cols & 1)
    buf = torch.empty((rows, ld), dtype=torch.float64, device=device)
    return buf, ld


def _ws(nbytes, device):
    return torch.empty((max(int(nbytes), 8) + 7) // 8, dtype=torch.float64, device=device)


# ---------------------------------------------------------------------------------------------- covariance
def kern_fwd(kind, X, X2, ell, sigma2, noise=None, lower=False, out=None, ldk=None):
    """K(X, X2) [+ noise I].  ell: (1,) or (D,) tensor; sigma2: (1,) tensor (None for Linear)."""
    X = _c(X)
    n1, D = X.shape
    if X2 is not None:
        X2 = _c(X2)
        n2 = X2.shape[0]
        if X2.shape[1] != D:
            raise ValueError("X and X2 have different input dimensions")
    else:
        n2 = n1
    ell = _c(ell).reshape(-1)
    if kind == KERN_LINEAR and ell.numel() != D:
        raise ValueError("Linear kernel needs one variance per input dimension")
    if out is None:
        out, ldk = _aligned_empty(n1, n2, X.device)
    if n1 == 0 or n2 == 0:
        return out[:, :n2]
    call("gpb_kern_fwd", kind, ptr(X), n1, X.stride(0), ptr(X2), n2, X2.stride(0) if X2 is not None else 0, D,
         ptr(ell), ell.numel(), ptr(_c(sigma2).reshape(-1)) if sigma2 is not None else None,
         ptr(_c(noise).reshape(-1)) if noise is not None else None, 1 if lower else 0, ptr(out), ldk, stream_ptr())
    return out[:, :n2]


def kern_bwd(kind, X, X2, ell, sigma2, G, need_gx2, g_transposed=False):
    """Reduce G = dLoss/dK against dK/d(ell, sigma2[, X2]).  Returns (g_ell, g_sigma2, gX2 or None)."""
    X = _c(X)
    n1, D = X.shape
    X2c = _c(X2) if X2 is not None else X
    n2 = X2c.shape[0]
    ell = _c(ell).reshape(-1)
    G = _c(G)
    g_ell = torch.empty(ell.numel(), dtype=torch.float64, device=X.device)
    g_sig = torch.empty(1, dtype=torch.float64, device=X.device)
    gX2 = torch.empty((n2, D), dtype=torch.float64, device=X.device) if need_gx2 else None
    ws_bytes = query("gpb_kern_bwd_workspace_bytes", n1, n2, D)
    ws = _ws(ws_bytes, X.device)
    call("gpb_kern_bwd", kind, ptr(X), n1, X.stride(0), ptr(X2c), n2, X2c.stride(0), D, ptr(ell), ell.numel(),
         ptr(_c(sigma2).reshape(-1)) if sigma2 is not None else None, ptr(G), G.stride(0), 1 if g_transposed else 0,
         ptr(g_ell), ptr(g_sig), ptr(gX2), ptr(ws), ws.numel() * 8, stream_ptr())
    return g_ell, g_sig, gX2


def kern_bwd_mul(kind, X, X2, ell, sigma2, G, Mul, need_gx2, g_transposed=False, symmetric=False):
    """kern_bwd with the upstream gradient G .* Mul (Mul may be None); also handles Constant / White leaves.
    Returns (g_ell, g_sigma2, gX2 or None)."""
    X = _c(X)
    n1, D = X.shape
    X2c = _c(X2) if X2 is not None else X
    n2 = X2c.shape[0]
    if ell is None:
        ell = torch.ones(1, dtype=torch.float64, device=X.device)
    ell = _c(ell).reshape(-1)
    G = _c(G)
    Mul = _c(Mul) if Mul is not None else None
    g_ell = torch.empty(ell.numel(), dtype=torch.float64, device=X.device)
    g_sig = torch.empty(1, dtype=torch.float64, device=X.device)
    gX2 = torch.empty((n2, D), dtype=torch.float64, device=X.device) if need_gx2 else None
    ws = _ws(query("gpb_kern_bwd_workspace_bytes", n1, n2, D), X.device)
    call("gpb_kern_bwd_mul", kind, ptr(X), n1, X.stride(0), ptr(X2c), n2, X2c.stride(0), D, ptr(ell), ell.numel(),
         ptr(_c(sigma2).reshape(-1)) if sigma2 is not None else None, ptr(G), G.stride(0), 1 if g_transposed else 0,
         ptr(Mul), Mul.stride(0) if Mul is not None else 0, 1 if (symmetric or X2 is None) else 0,
         ptr(g_ell), ptr(g_sig), ptr(gX2), ptr(ws), ws.numel() * 8, stream_ptr())
    return g_ell, g_sig, gX2


def kern_sop_fwd(terms, X, X2, noise=None, lower=False, out=None, ldk=None):
    """K = sum over terms of the product of the term's leaves, in one pass.  terms: list of lists of
    (kind, ell or None, sigma2 or None) with device tensors."""
    import ctypes
    X = _c(X)
    n1, D = X.shape
    if X2 is not None:
        X2 = _c(X2)
        n2 = X2.shape[0]
        if X2.shape[1] != D:
            raise ValueError("X and X2 have different input dimensions")
    else:
        n2 = n1
    leaves = [leaf for term in terms for leaf in term]
    if not terms or len(terms) > SOP_MAX_TERMS or len(leaves) > SOP_MAX_LEAVES:
        raise ValueError("composite kernel: at most %d terms / %d leaves" % (SOP_MAX_TERMS, SOP_MAX_LEAVES))
    if out is None:
        out, ldk = _aligned_empty(n1, n2, X.device)
    if n1 == 0 or n2 == 0:
        return out[:, :n2]
    keep = []   # keep the contiguous parameter copies alive until the launch has been issued

    def dev_ptr(t):
        if t is None:
            return None
        t = _c(t).reshape(-1)
        keep.append(t)
        return ptr(t).value

    nl = len(leaves)
    term_len = (ctypes.c_int * len(terms))(*[len(t) for t in terms])
    kinds = (ctypes.c_int * nl)(*[int(k) for k, _, _ in leaves])
    ells = (ctypes.c_void_p * nl)(*[dev_ptr(e) for _, e, _ in leaves])
    ell_len = (ctypes.c_int * nl)(*[(e.numel() if e is not None else 0) for _, e, _ in leaves])
    sig = (ctypes.c_void_p * nl)(*[dev_ptr(s) for _, _, s in leaves])
    call("gpb_kern_sop_fwd", len(terms), term_len, kinds, ells, ell_len, sig, ptr(X), n1, X.stride(0), ptr(X2), n2,
         X2.stride(0) if X2 is not None else 0, D, ptr(_c(noise).reshape(-1)) if noise is not None else None,
         1 if lower else 0, ptr(out), ldk, stream_ptr())
    return out[:, :n2]


def linear_kdiag(X, v):
    X = _c(X)
    out = torch.empty(X.shape[0], dtype=torch.float64, device=X.device)
    if X.shape[0]:
        call("gpb_linear_kdiag", ptr(X), X.shape[0], X.stride(0), X.shape[1], ptr(_c(v).reshape(-1)), ptr(out),
             stream_ptr())
    return out


# ---------------------------------------------------------------------------------------------- Cholesky
def potrf_(A, lda):
    """In-place lower Cholesky of the n x n matrix in the (n, lda) buffer A.  Returns (dinv, info) where info
    is a device int32 tensor (0 = success, k = first non-positive pivot, LAPACK convention)."""
    n = A.shape[0]
    dinv = torch.empty((_npad(n), NB), dtype=torch.float64, device=A.device)
    info = torch.zeros(1, dtype=torch.int32, device=A.device)
    call("gpb_potrf_lower", ptr(A), n, lda, ptr(dinv), ptr(info), stream_ptr())
    return dinv, info


def tri_diag_inverse(L):
    n = L.shape[0]
    dinv = torch.empty((_npad(n), NB), dtype=torch.float64, device=L.device)
    call("gpb_tri_diag_inverse", ptr(L), n, L.stride(0), ptr(dinv), stream_ptr())
    return dinv


def potri_(A, lda, dinv):
    """In place: strictly-lower blocks of A <- (L L^T)^-1; returns the diagonal 128-blocks (npad x 128)."""
    n = A.shape[0]
    kd = torch.empty((_npad(n), NB), dtype=torch.float64, device=A.device)
    ws_bytes = query("gpb_potri_workspace_bytes", n)
    ws = _ws(ws_bytes, A.device)
    call("gpb_potri_lower", ptr(A), n, lda, ptr(dinv), ptr(kd), ptr(ws), ws.numel() * 8, stream_ptr())
    return kd


def trtri_upper_(A, lda, dinv):
    """In place: upper triangle of A <- L^-T (diagonal 128-blocks become clean upper-triangular blocks)."""
    n = A.shape[0]
    ws_bytes = query("gpb_potri_workspace_bytes", n)
    ws = _ws(ws_bytes, A.device)
    call("gpb_trtri_upper", ptr(A), n, lda, ptr(dinv), ptr(ws), ws.numel() * 8, stream_ptr())


def potri_assemble(A, lda, kd):
    n = A.shape[0]
    out, ldo = _aligned_empty(n, n, A.device)
    call("gpb_potri_assemble", ptr(A), n, lda, ptr(kd), ptr(out), ldo, stream_ptr())
    return out[:, :n]


def tri_zero_upper_(A, lda):
    call("gpb_tri_zero_upper", ptr(A), A.shape[0], lda, stream_ptr())


def add_diag_(A, lda, value):
    """A += value * I; value is a python float or a 1-element device tensor."""
    if isinstance(value, torch.Tensor):
        call("gpb_add_diag", ptr(A), A.shape[0], lda, ptr(_c(value).reshape(-1)), 0.0, stream_ptr())
    else:
        call("gpb_add_diag", ptr(A), A.shape[0], lda, None, float(value), stream_ptr())


def sym_buffer_from(x):
    """Copy a square matrix into a fresh TMA-aligned (n, ld) buffer; returns (buffer, ld)."""
    n = x.shape[0]
    buf, ld = _aligned_empty(n, n, x.device)
    buf[:, :n].copy_(x)
    return buf, ld


# ---------------------------------------------------------------------------------------------- solves
def trsv_(L, dinv, B, trans):
    """B <- L^-1 B (trans=False) or L^-T B (trans=True), in place; B is (n, k) contiguous."""
    n, k = B.shape
    ws_bytes = query("gpb_trsv_workspace_bytes", n)
    ws = _ws(ws_bytes, B.device)
    call("gpb_trsv_lower", ptr(L), n, L.stride(0), ptr(dinv), ptr(B), k, B.stride(0), 1 if trans else 0, ptr(ws),
         ws.numel() * 8, stream_ptr())
    return B


def trsm_right_lt_(L, dinv, X, ldx):
    """X <- X L^-T for the (m, n) panel stored in the (m, ldx) buffer X."""
    m = X.shape[0]
    n = L.shape[0]
    call("gpb_trsm_right_lt", ptr(L), n, L.stride(0), ptr(dinv), ptr(X), m, ldx, stream_ptr())
    return X


def logdet_sumsq(L, V=None):
    """Returns a 2-element device tensor: [sum log diag L (0 if L is None), sum V^2 (0 if V is None)]."""
    dev = L.device if L is not None else V.device
    out = torch.empty(2, dtype=torch.float64, device=dev)
    n = L.shape[0] if L is not None else 0
    if V is not None:
        V = _c(V)
        call("gpb_logdet_sumsq", ptr(L), n, L.stride(0) if L is not None else 0, ptr(V), V.shape[0], V.shape[1],
             V.stride(0), ptr(out), stream_ptr())
    else:
        call("gpb_logdet_sumsq", ptr(L), n, L.stride(0), None, 0, 0, 0, ptr(out), stream_ptr())
    return out


# ---------------------------------------------------------------------------------------------- GEMM
GEMM_NT, GEMM_TN, GEMM_NN = 0, 1, 2
GF_LOWER, GF_KLO_M, GF_KHI_M, GF_KLO_N, GF_KHI_N = 1, 2, 4, 8, 16   # include/gpb200.h GPB_GEMM_*


def _gemm_operand(t):
    """Return a contiguous fp64 tensor with even row stride and 16-byte aligned base (copying if needed)."""
    t = _c(t)
    if (t.stride(0) & 1) or (t.data_ptr() & 15):
        buf, ld = _aligned_empty(t.shape[0], t.shape[1], t.device)
        buf[:, : t.shape[1]].copy_(t)
        return buf[:, : t.shape[1]]
    return t


def gemm(mode, A, B, alpha=1.0, beta=0.0, C=None, lower_only=False, flags=0):
    """C = alpha op(A) op(B) + beta C on the DMMA engine.  mode: GEMM_NT (A B^T), GEMM_TN (A^T B), GEMM_NN.
    flags: OR of GF_* (triangular-operand k-range hints, lower tiles only)."""
    A = _gemm_operand(A)
    B = _gemm_operand(B)
    if mode == GEMM_NT:
        m, k = A.shape
        n = B.shape[0]
        kb = B.shape[1]
    elif mode == GEMM_TN:
        k, m = A.shape
        kb, n = B.shape
    else:
        m, k = A.shape
        kb, n = B.shape
    if k != kb:
        raise ValueError("gemm: inner dimensions differ (%d vs %d)" % (k, kb))
    if C is None:
        buf, ldc = _aligned_empty(m, n, A.device)
        C = buf[:, :n]
        if beta != 0.0:
            raise ValueError("beta != 0 needs an existing C")
    call("gpb_gemm", mode, m, n, k, float(alpha), ptr(A), A.stride(0), ptr(B), B.stride(0), float(beta), ptr(C),
         C.stride(0), int(flags) | (GF_LOWER if lower_only else 0), stream_ptr())
    return C


def gemm_ozaki_nt(A, B, slices=8, alpha=1.0, beta=0.0, C=None, lower_only=False):
    """C = alpha A B^T + beta C on the INT8 tensor path by integer slicing (gpb_gemm_ozaki_nt): the fused tcgen05 kernel,
    or the library engine while ozaki_config() is above 0; raises NativeLibraryError with status -5 for shapes that path
    does not take."""
    A = _gemm_operand(A)
    B = A if B is None else _gemm_operand(B)
    m, k = A.shape
    n = B.shape[0]
    if B.shape[1] != k:
        raise ValueError("gemm_ozaki_nt: inner dimensions differ")
    if C is None:
        buf, ldc = _aligned_empty(m, n, A.device)
        C = buf[:, :n]
        if beta != 0.0:
            raise ValueError("beta != 0 needs an existing C")
    call("gpb_gemm_ozaki_nt", m, n, k, float(alpha), ptr(A), A.stride(0), ptr(B), B.stride(0), float(beta), ptr(C),
         C.stride(0), 1 if lower_only else 0, int(slices), stream_ptr())
    return C


def ozaki_config(slices=-1):
    """Slices of the library (cuBLASLt) engine for the large products of the blocked Cholesky and inverse; 0 = off, the
    default.  Above 0 it takes precedence over i8mma_config.  Returns the previous value; slices < 0 only queries."""
    return query("gpb_ozaki_config", int(slices))


def i8mma_config(slices=-1):
    """Slices of the fused tcgen05 int8 engine for the large trailing updates of the blocked Cholesky (2..8; 8, the
    default; 0 = FP64 DMMA engine for the factor and the inverse).  While it is above 0 the blocked inverse's products
    run on the same engine at a fixed 9 slices.  Returns the previous value; slices < 0 only queries."""
    return query("gpb_i8mma_config", int(slices))


def gemv_t(A, Y, out, beta=1.0):
    """out (cols x dy) = beta * out + A^T Y for a tall row panel A (rows x cols) and few right-hand sides."""
    A, Y = _c(A), _c(Y)
    rows, cols = A.shape
    dy = Y.shape[1]
    ws = _ws(query("gpb_gemv_t_workspace_bytes", rows, cols), A.device)
    call("gpb_gemv_t", ptr(A), rows, cols, A.stride(0), ptr(Y), dy, Y.stride(0), float(beta), ptr(out), out.stride(0),
         ptr(ws), ws.numel() * 8, stream_ptr())
    return out


def rowdot(A, B, alpha=1.0, out=None, beta=0.0):
    """out[i] = alpha * sum_j A[i][j] B[i][j] + beta * out[i] in one pass over A and B (no [rows x cols] temporary)."""
    A, B = _c(A), _c(B)
    if A.shape != B.shape:
        raise ValueError("rowdot: shapes differ")
    rows, cols = A.shape
    if out is None:
        out = torch.empty(rows, dtype=torch.float64, device=A.device)
        beta = 0.0
    if rows:
        call("gpb_rowdot", ptr(A), A.stride(0), ptr(B), B.stride(0), rows, cols, float(alpha), float(beta), ptr(out),
             stream_ptr())
    return out


def gemv_n(A, V):
    """A @ V for a row panel A (rows x cols) and a few columns V (cols x dy); A is read once."""
    A, V = _c(A), _c(V)
    rows, cols = A.shape
    out = torch.empty((rows, V.shape[1]), dtype=torch.float64, device=A.device)
    if rows and V.shape[1]:
        call("gpb_gemv_n", ptr(A), rows, cols, A.stride(0), ptr(V), V.shape[1], V.stride(0), ptr(out), out.stride(0),
             stream_ptr())
    return out


def rows_scale_add_outer_(A, s=None, scale=1.0, G=None, V=None):
    """In place: A[i][j] = scale * s[i] * A[i][j] + sum_o G[i][o] V[j][o]."""
    rows, cols = A.shape
    if G is not None:
        G, V = _c(G), _c(V)
    if rows:
        call("gpb_rows_scale_add_outer", ptr(A), rows, cols, A.stride(0), ptr(_c(s).reshape(-1)) if s is not None else None,
             float(scale), ptr(G), G.shape[1] if G is not None else 0, G.stride(0) if G is not None else 0, ptr(V),
             V.stride(0) if V is not None else 0, stream_ptr())
    return A


def gemm_splitk(mode, A, B, k_per_split, C3, beta=1.0, alpha=1.0, lower_only=False):
    """Split-K GEMM: slice s of the k range accumulates into C3[s] (C3: [splits, m, ld] with ld even)."""
    A = _gemm_operand(A)
    B = _gemm_operand(B)
    if mode == GEMM_TN:
        k, m = A.shape
        n = B.shape[1]
    elif mode == GEMM_NT:
        m, k = A.shape
        n = B.shape[0]
    else:
        m, k = A.shape
        n = B.shape[1]
    splits = (k + k_per_split - 1) // k_per_split
    if C3.shape[0] < splits or C3.shape[1] != m or C3.shape[2] < n:
        raise ValueError("gemm_splitk: C3 must be [>= %d, %d, >= %d]" % (splits, m, n))
    call("gpb_gemm_splitk", mode, m, n, k, k_per_split, float(alpha), ptr(A), A.stride(0), ptr(B), B.stride(0),
         float(beta), ptr(C3), C3.stride(1), C3.stride(0), 1 if lower_only else 0, stream_ptr())
    return C3


# ---------------------------------------------------------------------------------------------- streamed Kuf statistics
def kuf_stats_fwd(kind, X, Y, Z, ell, sigma2, chunk, cache=False):
    """(Phi = Kuf Kfu [m, m], psi = Kuf Y [m, dy], panel cache or None) streamed over row chunks of X in ONE native call."""
    X, Y, Z = _c(X), _c(Y), _c(Z)
    n, D = X.shape
    m, dy = Z.shape[0], Y.shape[1]
    ell = _c(ell).reshape(-1)
    s2 = _c(sigma2).reshape(-1)
    chunk = int(max(1, min(chunk, max(n, 1))))
    ws = _ws(query("gpb_kuf_stats_workspace_bytes", m, D, dy, chunk, 0), X.device)
    Phi = _aligned_empty(m, m, X.device)[0]
    psi = torch.empty((m, dy), dtype=torch.float64, device=X.device)
    kfu = _aligned_empty(n, m, X.device)[0] if cache else None
    call("gpb_kuf_stats_fwd", kind, ptr(X), n, X.stride(0), ptr(Y), dy, Y.stride(0), ptr(Z), m, Z.stride(0), D, ptr(ell),
         ell.numel(), ptr(s2), chunk, ptr(Phi), Phi.stride(0), ptr(psi), psi.stride(0), ptr(kfu),
         kfu.stride(0) if kfu is not None else 0, ptr(ws), ws.numel() * 8, stream_ptr())
    return Phi[:, :m], psi, kfu


def kuf_stats_bwd(kind, X, Y, Z, ell, sigma2, chunk, R, W, kfu=None, gX=None):
    """(g_ell, g_sigma2, gZ): the gradient Kfu_c R + Y_c W^T of every panel reduced against dK/d(ell, sigma2, Z).
    gX (n x D, optional) receives the gradient with respect to X."""
    X, Y, Z = _c(X), _c(Y), _c(Z)
    n, D = X.shape
    m, dy = Z.shape[0], Y.shape[1]
    ell = _c(ell).reshape(-1)
    s2 = _c(sigma2).reshape(-1)
    R, W = _gemm_operand(R), _c(W)
    chunk = int(max(1, min(chunk, max(n, 1))))
    ws = _ws(query("gpb_kuf_stats_workspace_bytes", m, D, dy, chunk, 1 if gX is not None else 0), X.device)
    g_ell = torch.empty(ell.numel(), dtype=torch.float64, device=X.device)
    g_s2 = torch.empty(1, dtype=torch.float64, device=X.device)
    gZ = torch.empty((m, D), dtype=torch.float64, device=X.device)
    call("gpb_kuf_stats_bwd", kind, ptr(X), n, X.stride(0), ptr(Y), dy, Y.stride(0), ptr(Z), m, Z.stride(0), D, ptr(ell),
         ell.numel(), ptr(s2), chunk, ptr(R), R.stride(0), ptr(W), W.stride(0), ptr(kfu),
         kfu.stride(0) if kfu is not None else 0, ptr(g_ell), ptr(g_s2), ptr(gZ), ptr(ws), ws.numel() * 8, stream_ptr(),
         ptr(gX), gX.stride(0) if gX is not None else 0)
    return g_ell, g_s2, gZ


# ---------------------------------------------------------------------------------------------- fused GPR gradient
def gpr_grad(kind, X, ell, sigma2, Kinv, ldk, kd, a, gX=None):
    """Returns (g_ell, g_sigma2, g_noise): d loss / d (ell, sigma2, sigma_n^2) for the GPR loss.  gX (n x D, optional)
    receives d loss / dX."""
    X = _c(X)
    n, D = X.shape
    ell = _c(ell).reshape(-1)
    a = _c(a)
    g_ell = torch.empty(ell.numel(), dtype=torch.float64, device=X.device)
    g_sig = torch.zeros(1, dtype=torch.float64, device=X.device)
    g_noise = torch.empty(1, dtype=torch.float64, device=X.device)
    ws_bytes = query("gpb_gpr_grad_workspace_bytes", n, D)
    ws = _ws(ws_bytes, X.device)
    call("gpb_gpr_grad", kind, ptr(X), n, X.stride(0), D, ptr(ell), ell.numel(),
         ptr(_c(sigma2).reshape(-1)) if sigma2 is not None else None, ptr(Kinv), ldk, ptr(kd), ptr(a), a.shape[1],
         a.stride(0), ptr(g_ell), ptr(g_sig), ptr(g_noise), ptr(ws), ws.numel() * 8, stream_ptr(),
         ptr(gX), gX.stride(0) if gX is not None else 0)
    return g_ell, g_sig, g_noise


# ---------------------------------------------------------------------------------------------- cached GPR posterior
def pred_gx(kind, Xs, X, ell, sigma2, a, g_mean, g_var, Q):
    """d loss / d x* (ns x D) for mean = K(x*, X) a and var = sigma2 - rowdot(K(x*, X), Q), given the upstream
    gradients g_mean (ns x dy) and g_var (ns)."""
    Xs, X, a, g_mean, Q = _c(Xs), _c(X), _c(a), _c(g_mean), _c(Q)
    ns, D = Xs.shape
    ell = _c(ell).reshape(-1)
    g_var = _c(g_var).reshape(-1)
    gXs = torch.empty((ns, D), dtype=torch.float64, device=Xs.device)
    call("gpb_pred_gx", kind, ptr(Xs), ns, _ld(Xs), ptr(X), X.shape[0], _ld(X), D, ptr(ell), ell.numel(),
         ptr(_c(sigma2).reshape(-1)), ptr(a), a.shape[1], _ld(a), ptr(g_mean), _ld(g_mean), ptr(g_var), ptr(Q), _ld(Q),
         ptr(gXs), gXs.stride(0), stream_ptr())
    return gXs


def _ld(t):
    """Leading dimension of a row-major 2-D tensor: the row stride, or the row length for a single row (whose row stride
    torch leaves arbitrary, e.g. 0 for a broadcast gradient)."""
    return t.stride(0) if t.shape[0] > 1 else t.shape[1]
