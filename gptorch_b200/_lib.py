"""ctypes binding of libgpb200.so (the C ABI declared in include/gpb200.h).

This is the only place Python touches the native library.  Arguments are raw device pointers
(``tensor.data_ptr()``), sizes, leading dimensions and the current CUDA stream; no torch types cross the
boundary.  There is deliberately NO fallback: if the library is missing, or a tensor is not a CUDA fp64
tensor, the call raises.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GPB200_LIB", os.path.join(_HERE, "lib", "libgpb200.so"))

c_int, c_long, c_double, c_void_p, c_size_t = (
    ctypes.c_int,
    ctypes.c_long,
    ctypes.c_double,
    ctypes.c_void_p,
    ctypes.c_size_t,
)

# name -> (restype, argtypes); mirrors include/gpb200.h one to one.
SIGNATURES = {
    "gpb_version": (c_int, []),
    "gpb_last_error": (ctypes.c_char_p, []),
    "gpb_block_size": (c_int, []),
    "gpb_launch_count": (c_long, []),
    "gpb_reset_launch_count": (None, []),
    "gpb_dmma_issue_probe": (c_int, [c_int, c_void_p, c_size_t, ctypes.POINTER(c_double), c_void_p]),
    "gpb_kern_fwd": (c_int, [c_int, c_void_p, c_int, c_long, c_void_p, c_int, c_long, c_int, c_void_p, c_int,
                             c_void_p, c_void_p, c_int, c_void_p, c_long, c_void_p]),
    "gpb_kern_bwd_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "gpb_kern_bwd": (c_int, [c_int, c_void_p, c_int, c_long, c_void_p, c_int, c_long, c_int, c_void_p, c_int,
                             c_void_p, c_void_p, c_long, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t,
                             c_void_p]),
    "gpb_kern_bwd_mul": (c_int, [c_int, c_void_p, c_int, c_long, c_void_p, c_int, c_long, c_int, c_void_p, c_int,
                                 c_void_p, c_void_p, c_long, c_int, c_void_p, c_long, c_int, c_void_p, c_void_p,
                                 c_void_p, c_void_p, c_size_t, c_void_p]),
    "gpb_kern_sop_fwd": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_long,
                                 c_void_p, c_int, c_long, c_int, c_void_p, c_int, c_void_p, c_long, c_void_p]),
    "gpb_linear_kdiag": (c_int, [c_void_p, c_int, c_long, c_int, c_void_p, c_void_p, c_void_p]),
    "gpb_potrf_lower": (c_int, [c_void_p, c_int, c_long, c_void_p, c_void_p, c_void_p]),
    "gpb_tri_diag_inverse": (c_int, [c_void_p, c_int, c_long, c_void_p, c_void_p]),
    "gpb_potri_workspace_bytes": (c_size_t, [c_int]),
    "gpb_potri_lower": (c_int, [c_void_p, c_int, c_long, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "gpb_trtri_upper": (c_int, [c_void_p, c_int, c_long, c_void_p, c_void_p, c_size_t, c_void_p]),
    "gpb_potri_assemble": (c_int, [c_void_p, c_int, c_long, c_void_p, c_void_p, c_long, c_void_p]),
    "gpb_tri_zero_upper": (c_int, [c_void_p, c_int, c_long, c_void_p]),
    "gpb_add_diag": (c_int, [c_void_p, c_int, c_long, c_void_p, c_double, c_void_p]),
    "gpb_trsv_workspace_bytes": (c_size_t, [c_int]),
    "gpb_trsv_lower": (c_int, [c_void_p, c_int, c_long, c_void_p, c_void_p, c_int, c_long, c_int, c_void_p,
                               c_size_t, c_void_p]),
    "gpb_trsm_right_lt": (c_int, [c_void_p, c_int, c_long, c_void_p, c_void_p, c_int, c_long, c_void_p]),
    "gpb_logdet_sumsq": (c_int, [c_void_p, c_int, c_long, c_void_p, c_int, c_int, c_long, c_void_p, c_void_p]),
    "gpb_rowdot": (c_int, [c_void_p, c_long, c_void_p, c_long, c_long, c_int, c_double, c_double, c_void_p, c_void_p]),
    "gpb_gemv_n": (c_int, [c_void_p, c_long, c_int, c_long, c_void_p, c_int, c_long, c_void_p, c_long, c_void_p]),
    "gpb_rows_scale_add_outer": (c_int, [c_void_p, c_long, c_int, c_long, c_void_p, c_double, c_void_p, c_int, c_long,
                                         c_void_p, c_long, c_void_p]),
    "gpb_gemv_t_workspace_bytes": (c_size_t, [c_long, c_int]),
    "gpb_gemv_t": (c_int, [c_void_p, c_long, c_int, c_long, c_void_p, c_int, c_long, c_double, c_void_p, c_long, c_void_p,
                           c_size_t, c_void_p]),
    "gpb_gemm": (c_int, [c_int, c_int, c_int, c_int, c_double, c_void_p, c_long, c_void_p, c_long, c_double,
                         c_void_p, c_long, c_int, c_void_p]),
    "gpb_gemm_ozaki_nt": (c_int, [c_int, c_int, c_int, c_double, c_void_p, c_long, c_void_p, c_long, c_double, c_void_p, c_long,
                                  c_int, c_int, c_void_p]),
    "gpb_ozaki_config": (c_int, [c_int]),
    "gpb_gemm_splitk": (c_int, [c_int, c_int, c_int, c_int, c_int, c_double, c_void_p, c_long, c_void_p, c_long, c_double,
                                c_void_p, c_long, c_long, c_int, c_void_p]),
    "gpb_kuf_stats_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int, c_int]),
    "gpb_kuf_stats_fwd": (c_int, [c_int, c_void_p, c_long, c_long, c_void_p, c_int, c_long, c_void_p, c_int, c_long, c_int,
                                  c_void_p, c_int, c_void_p, c_int, c_void_p, c_long, c_void_p, c_long, c_void_p, c_long,
                                  c_void_p, c_size_t, c_void_p]),
    "gpb_kuf_stats_bwd": (c_int, [c_int, c_void_p, c_long, c_long, c_void_p, c_int, c_long, c_void_p, c_int, c_long, c_int,
                                  c_void_p, c_int, c_void_p, c_int, c_void_p, c_long, c_void_p, c_long, c_void_p, c_long,
                                  c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p, c_void_p, c_long]),
    "gpb_gpr_grad_workspace_bytes": (c_size_t, [c_int, c_int]),
    "gpb_gpr_grad": (c_int, [c_int, c_void_p, c_int, c_long, c_int, c_void_p, c_int, c_void_p, c_void_p, c_long,
                             c_void_p, c_void_p, c_int, c_long, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t,
                             c_void_p, c_void_p, c_long]),
}

# include/gpb200_posterior.h: entry points of a cached GPR posterior (gpb_version() >= 102), mirrored one to one.
POSTERIOR_SIGNATURES = {
    "gpb_pred_gx": (c_int, [c_int, c_void_p, c_int, c_long, c_void_p, c_int, c_long, c_int, c_void_p, c_int, c_void_p,
                            c_void_p, c_int, c_long, c_void_p, c_long, c_void_p, c_void_p, c_long, c_void_p, c_long,
                            c_void_p]),
}

# include/gpb200_i8mma.h: the switch of the fused int8-sliced engine (gpb_version() >= 103), mirrored one to one.
I8MMA_SIGNATURES = {
    "gpb_i8mma_config": (c_int, [c_int]),
}

_ERRORS = {-1: "bad argument", -2: "alignment (16-byte base, even leading dimension required)",
           -3: "CUDA runtime error", -4: "CUDA driver / tensor-map error", -5: "unsupported configuration"}

_lib = None


class NativeLibraryError(RuntimeError):
    """libgpb200.so is missing or rejected a call.  (A RuntimeError subclass, but raised for argument and
    environment problems only -- numerical failure of a factorisation is reported through ``info``.)"""


def load():
    """Load libgpb200.so and type every entry point.  Raises if the library is absent (no CPU fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeLibraryError(
            "libgpb200.so not found at %s -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C gptorch_b200/csrc`.  gptorch_b200 has no CPU or PyTorch fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in list(SIGNATURES.items()) + list(POSTERIOR_SIGNATURES.items()) + list(I8MMA_SIGNATURES.items()):
        fn = getattr(lib, name)  # AttributeError here means header and library disagree
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def is_loaded():
    return _lib is not None


def _check(rc, what):
    if rc != 0:
        lib = load()
        detail = lib.gpb_last_error().decode("utf-8", "replace")
        raise NativeLibraryError("%s failed: %s (rc=%d) %s" % (what, _ERRORS.get(rc, "unknown"), rc, detail))


def stream_ptr():
    """cudaStream_t of torch's current stream (the raw query: torch.cuda.current_stream() costs ~15 us per call)."""
    return ctypes.c_void_p(torch._C._cuda_getCurrentRawStream(torch.cuda.current_device()))


_keep = []   # tensors whose pointers were taken for the call being assembled (see ptr / call)


def ptr(t):
    """Device pointer of a CUDA fp64 tensor (or NULL for None).

    The tensor is kept alive until the entry point it is passed to has been issued: wrappers hand in temporaries such
    as ``ptr(_c(sigma2).reshape(-1))``, and a temporary freed before the launch could be handed out again by the
    caching allocator to the next conversion.  The tensor must live on the CURRENT device -- launches go to the current
    device's current stream."""
    if t is None:
        return None
    if not t.is_cuda:
        raise NativeLibraryError("gptorch_b200 kernels need CUDA tensors (got a %s tensor); there is no CPU path"
                                 % t.device.type)
    if t.dtype != torch.float64 and t.dtype != torch.int32:
        raise NativeLibraryError("expected float64, got %s" % t.dtype)
    if t.device.index != torch.cuda.current_device():
        raise NativeLibraryError("tensor on %s but the current CUDA device is cuda:%d -- run the call under "
                                 "torch.cuda.device(tensor.device)" % (t.device, torch.cuda.current_device()))
    _keep.append(t)
    return ctypes.c_void_p(t.data_ptr())


def call(name, *args):
    """Call an int-returning entry point and raise on a non-zero status."""
    lib = load()
    try:
        rc = getattr(lib, name)(*args)
    finally:
        _keep.clear()
    _check(rc, name)


def query(name, *args):
    """Call a size-returning entry point."""
    lib = load()
    return getattr(lib, name)(*args)
