"""The blocked inverse (gpb_potri_lower, gpb_trtri_upper) on the fused int8-sliced engine.  By default its three product
hooks (T22^T L21 and T11 P in the triangular inverse, the strip-wise T T^T) run the fused tcgen05 kernel at 9 slices, in
32-column tiles (csrc/gpb_ozaki_mma.cu).  The int32 class sums are exact and the epilogue repeats the library engine's
recombination, and both engines use the same strip decomposition, so the fused inverse is BIT FOR BIT the library
engine's at 9 slices (gpb_ozaki_config(9)): transposed-triangular and triangular operands, lower blocks with the diagonal
blocks sent to their own buffer, NaN rows, ragged orders.  Where the sliced path does not apply (order not a multiple
of 16, a stream being captured into a CUDA graph, gpb_i8mma_config(0)) the inverse is the FP64 DMMA engine's."""
import pytest
import torch

pytestmark = pytest.mark.gpu

INVERSE_SLICES = 9


@pytest.fixture()
def nv():
    from gptorch_b200 import _native
    prev = _native.i8mma_config(-1)
    yield _native
    _native.ozaki_config(0)
    _native.i8mma_config(prev)


def _engine(nv, name):
    """'native' = the default fused engine (factor 8 slices, inverse 9), 'library' = cuBLASLt products at the inverse's
    slice count, 'dmma' = the FP64 DMMA engine."""
    if name == "library":
        nv.ozaki_config(INVERSE_SLICES)
    else:
        nv.ozaki_config(0)
        nv.i8mma_config(8 if name == "native" else 0)


def _bits_equal(a, b):
    a, b = a.contiguous(), b.contiguous()
    na, nb = torch.isnan(a), torch.isnan(b)
    if not torch.equal(na, nb):
        return False
    return torch.equal(a.view(torch.int64)[~na], b.view(torch.int64)[~nb])


def _factor(nv, n, seed=31):
    """The DMMA engine's Cholesky factor of an Rbf covariance (one fixed input for every engine's inverse)."""
    _engine(nv, "dmma")
    g = torch.Generator().manual_seed(seed)
    X = torch.rand(n, 8, generator=g, dtype=torch.float64).cuda()
    ell = torch.ones(8, dtype=torch.float64, device="cuda")
    s2 = torch.ones(1, dtype=torch.float64, device="cuda")
    noise = torch.full((1,), 0.01, dtype=torch.float64, device="cuda")
    buf, ld = nv._aligned_empty(n, n, X.device)
    nv.kern_fwd(0, X, None, ell, s2, noise=noise, lower=True, out=buf, ldk=ld)
    dinv, info = nv.potrf_(buf, ld)
    assert int(info.item()) == 0
    return buf, ld, dinv


def _inverse(nv, eng, buf, ld, dinv):
    _engine(nv, eng)
    b = buf.clone()
    kd = nv.potri_(b, ld, dinv)
    K = nv.potri_assemble(b, ld, kd).clone()
    del b
    torch.cuda.empty_cache()
    return K


@pytest.fixture(scope="module")
def factors():
    from gptorch_b200 import _native
    cache = {}

    def get(n):
        if n not in cache:
            prev = _native.i8mma_config(-1)
            cache.clear()
            torch.cuda.empty_cache()
            cache[n] = _factor(_native, n)
            _native.i8mma_config(prev)
        return cache[n]
    yield get
    cache.clear()


@pytest.mark.parametrize("n", [8192, 12304, 16384])
def test_fused_inverse_is_bitwise_the_library_inverse(nv, factors, n):
    """8192 and 16384 cross both trtri hooks (levels s >= 4096) and every T T^T strip; 12304 = 16 * 769 is ragged
    against the 128-block (a 16-row last strip, a DMMA-only ragged trtri problem)."""
    buf, ld, dinv = factors(n)
    K = {eng: _inverse(nv, eng, buf, ld, dinv) for eng in ("library", "native")}
    assert _bits_equal(K["library"], K["native"])
    if n == 8192:
        K0 = _inverse(nv, "dmma", buf, ld, dinv)
        assert not torch.equal(K0, K["native"])                 # the inverse really is sliced by default
        assert float((K["native"] - K0).abs().max()) / float(K0.abs().max()) < 1e-12


@pytest.mark.parametrize("op", ["trtri", "potri"])
def test_nan_rows_of_the_factor_give_the_library_engines_nans_and_values(nv, factors, op):
    """A NaN in L21 of the top trtri level makes a row of the sliced operands NaN (its scale is NaN): through
    T22^T L21 (transposed triangular A, transposed B), T11 P (triangular A, plain B) and the lower-block T T^T strips with
    their diagonal blocks in kd, the fused engine reproduces the library engine's NaNs and every finite value."""
    n = 8192
    buf, ld, dinv = factors(n)
    out = {}
    for eng in ("library", "native"):
        _engine(nv, eng)
        b = buf.clone()
        b[6000, 100] = float("nan")
        if op == "trtri":
            nv.trtri_upper_(b, ld, dinv)
            out[eng] = torch.triu(b[:, :n]).clone()
        else:
            kd = nv.potri_(b, ld, dinv)
            out[eng] = nv.potri_assemble(b, ld, kd).clone()
        del b
        torch.cuda.empty_cache()
    assert _bits_equal(out["library"], out["native"])
    nan = torch.isnan(out["native"])
    assert bool(nan.any()) and not bool(nan.all())


def test_order_not_a_multiple_of_16_is_the_dmma_inverse(nv):
    n = 8200
    buf, ld, dinv = _factor(nv, n)
    K = {eng: _inverse(nv, eng, buf, ld, dinv) for eng in ("dmma", "native")}
    assert _bits_equal(K["dmma"], K["native"])


def test_inverse_captured_into_a_cuda_graph_is_the_dmma_inverse(nv, factors):
    """The sliced engine's workspace cannot be allocated while a stream is being captured: the captured inverse runs
    every product on the DMMA engine."""
    n = 8192
    buf, ld, dinv = factors(n)
    K0 = _inverse(nv, "dmma", buf, ld, dinv)       # (switching the fused engine off also returns its workspaces)
    _engine(nv, "native")
    b = buf.clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            kd = nv.potri_(b, ld, dinv)
    graph.replay()
    torch.cuda.synchronize()
    K1 = nv.potri_assemble(b, ld, kd)
    assert _bits_equal(K0, K1)


def test_dmma_switch_gives_the_dmma_inverse_on_every_call(nv, factors):
    """gpb_i8mma_config(0) returns the inverse to the DMMA engine after sliced inverses have run (no workspace or state
    of the sliced engine leaks into it)."""
    n = 8192
    buf, ld, dinv = factors(n)
    K0 = _inverse(nv, "dmma", buf, ld, dinv)
    _inverse(nv, "native", buf, ld, dinv)
    assert _bits_equal(K0, _inverse(nv, "dmma", buf, ld, dinv))
