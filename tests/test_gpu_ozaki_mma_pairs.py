"""The fused int8-sliced kernel (csrc/gpb_ozaki_mma.cu) runs in clusters of two CTAs that take neighbouring tiles of one
tile row and share their A slices.  The shapes here put the pair logic at its edges: an odd number of tiles in n (the
last pair's second tile lies past n), n smaller than one tile, lower-block output with m not a multiple of 128 (pairs
right of the diagonal skipped as a whole), and NaN rows in either operand.  Everywhere the result must be BIT FOR BIT
the library engine's (cuBLASLt products, gpb_ozaki_config > 0) at the same slice count."""
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture()
def nv():
    from gptorch_b200 import _native
    prev = _native.i8mma_config(-1)
    yield _native
    _native.ozaki_config(0)
    _native.i8mma_config(prev)


def _engine(nv, name, slices):
    if name == "library":
        nv.ozaki_config(slices)
    else:
        nv.ozaki_config(0)
        nv.i8mma_config(slices)


def _bits_equal(a, b):
    a, b = a.contiguous(), b.contiguous()
    na, nb = torch.isnan(a), torch.isnan(b)
    if not torch.equal(na, nb):
        return False
    return torch.equal(a.view(torch.int64)[~na], b.view(torch.int64)[~nb])


def _cov_like(m, k, g, shift=0.0):
    X = torch.rand(max(m, k), 8, generator=g, dtype=torch.float64)
    return torch.exp(-0.5 * torch.cdist(X[:m] + shift, X[:k]).pow(2)).cuda()


@pytest.mark.parametrize("slices", [2, 5, 8])
@pytest.mark.parametrize("m,n,k", [(300, 132, 272),      # 3 tiles of 64 in n: the last pair has a phantom tile
                                   (1100, 4, 48),        # n = 4
                                   (260, 40, 1040),      # n < 64
                                   (700, 332, 272)])     # 6 tiles in n, 2 ragged ones in m
def test_paired_product_is_bitwise_the_library_product(nv, slices, m, n, k):
    g = torch.Generator().manual_seed(3 * m + n + k)
    A = _cov_like(m, k, g) * torch.exp(2 * torch.randn(m, 1, generator=g, dtype=torch.float64)).cuda()
    B = _cov_like(n, k, g, 0.1) - 0.3
    A[m - 2, k // 2] = float("nan")                          # a NaN row of A: that row of C is NaN
    B[n - 1, 1] = float("nan")                               # a NaN row of B: that column of C is NaN
    C0 = torch.randn(m, n, generator=g, dtype=torch.float64).cuda()
    out = {}
    for eng in ("library", "native"):
        _engine(nv, eng, slices)
        out[eng] = (nv.gemm_ozaki_nt(A, B, slices=slices).clone(),
                    nv.gemm_ozaki_nt(A, B, slices=slices, alpha=-1.0, beta=0.5, C=C0.clone()).clone())
    for x, y in zip(out["library"], out["native"]):
        assert _bits_equal(x, y)
    C = out["native"][0]
    assert bool(torch.isnan(C[m - 2]).all()) and bool(torch.isnan(C[:, n - 1]).all())
    assert bool(torch.isfinite(C[: m - 2, : n - 1]).all())


@pytest.mark.parametrize("slices", [2, 5, 8])
@pytest.mark.parametrize("m,k", [(172, 272), (332, 48), (1000, 1040)])
def test_paired_lower_product_is_bitwise_the_library_product(nv, slices, m, k):
    """m = 172: 3 tiles of 64 columns, the second pair holds the last live tile and a phantom; m = 332 and 1000: pairs
    right of the diagonal block of a ragged last tile row are skipped, the upper blocks stay untouched."""
    g = torch.Generator().manual_seed(m + 7 * k)
    A = _cov_like(m, k, g)
    out = {}
    for eng in ("library", "native"):
        _engine(nv, eng, slices)
        C = torch.full((m, m), 7.0, dtype=torch.float64, device="cuda")
        nv.gemm_ozaki_nt(A, None, slices=slices, alpha=-1.0, beta=1.0, C=C, lower_only=True)
        out[eng] = C
    assert _bits_equal(out["library"], out["native"])
    blk = torch.arange(m, device="cuda") // 128
    assert bool((out["native"][blk[None, :] > blk[:, None]] == 7.0).all())


def test_paired_inverse_is_bitwise_the_library_inverse(nv):
    """The inverse's products (9 slices) run in 48-column tiles, so a pair of 96 columns can straddle two 128-blocks: its
    k range is the union of both tiles' ranges and it is skipped only when both tiles lie right of the diagonal block.
    N = 10000 = 16 * 625 crosses both trtri hooks and every T T^T strip, with a 16-row last strip."""
    n = 10000
    nv.i8mma_config(0)
    g = torch.Generator().manual_seed(41)
    X = torch.rand(n, 8, generator=g, dtype=torch.float64).cuda()
    ell = torch.ones(8, dtype=torch.float64, device="cuda")
    s2 = torch.ones(1, dtype=torch.float64, device="cuda")
    noise = torch.full((1,), 0.01, dtype=torch.float64, device="cuda")
    buf, ld = nv._aligned_empty(n, n, X.device)
    nv.kern_fwd(0, X, None, ell, s2, noise=noise, lower=True, out=buf, ldk=ld)
    dinv, info = nv.potrf_(buf, ld)                    # the DMMA engine's factor: one input for both inverses
    assert int(info.item()) == 0
    K = {}
    for eng in ("library", "native"):
        _engine(nv, eng, 9 if eng == "library" else 8)   # the fused engine at 8 slices takes the inverse at 9
        b = buf.clone()
        kd = nv.potri_(b, ld, dinv)
        K[eng] = nv.potri_assemble(b, ld, kd).clone()
        del b
        torch.cuda.empty_cache()
    assert _bits_equal(K["library"], K["native"])
