"""The fused tcgen05 int8-sliced engine (csrc/gpb_ozaki_mma.cu), the default for the large products of gpb_potrf_lower /
gpb_potri_lower.  Its int32 class sums are exact and its epilogue runs the library engine's recombination step by step,
so against the library engine (cuBLASLt products, gpb_ozaki_config > 0) at the same slice count it must agree BIT FOR
BIT: products over ragged shapes, lower-block output, alpha/beta, NaN rows, and the factor of the blocked Cholesky.  The
inverse's products stay on the FP64 DMMA engine by default (csrc/gpb_chol.cu, potri_lower, says why)."""
import numpy as np
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
    """'native' = the fused kernel, 'library' = cuBLASLt products, 'dmma' = the FP64 DMMA engine."""
    if name == "library":
        nv.ozaki_config(slices)
    else:
        nv.ozaki_config(0)
        nv.i8mma_config(slices if name == "native" else 0)


def _bits_equal(a, b):
    a, b = a.contiguous(), b.contiguous()
    na, nb = torch.isnan(a), torch.isnan(b)
    if not torch.equal(na, nb):
        return False
    return torch.equal(a.view(torch.int64)[~na], b.view(torch.int64)[~nb])


def _cov_like(m, k, g, shift=0.0):
    X = torch.rand(max(m, k), 8, generator=g, dtype=torch.float64)
    return torch.exp(-0.5 * torch.cdist(X[:m] + shift, X[:k]).pow(2)).cuda()


@pytest.mark.parametrize("slices", [7, 8])
@pytest.mark.parametrize("m,n,k", [(1028, 516, 272), (260, 1100, 48), (8, 4, 16), (2052, 1988, 1040)])
def test_fused_product_is_bitwise_the_library_product(nv, slices, m, n, k):
    g = torch.Generator().manual_seed(m + n + k)
    A = _cov_like(m, k, g) * torch.exp(2 * torch.randn(m, 1, generator=g, dtype=torch.float64)).cuda()
    B = _cov_like(n, k, g, 0.1) - 0.3
    A[3, 5] = float("nan")                                   # a NaN row stays NaN
    C0 = torch.randn(m, n, generator=g, dtype=torch.float64).cuda()
    out = {}
    for eng in ("library", "native"):
        _engine(nv, eng, slices)
        out[eng] = (nv.gemm_ozaki_nt(A, B, slices=slices).clone(),
                    nv.gemm_ozaki_nt(A, B, slices=slices, alpha=-1.0, beta=0.5, C=C0.clone()).clone())
    for x, y in zip(out["library"], out["native"]):
        assert _bits_equal(x, y)
    C = out["native"][0]
    assert bool(torch.isnan(C[3]).all()) and bool(torch.isfinite(C[4]).all())
    ref = A[4:] @ B.t()
    assert float((C[4:] - ref).abs().max()) <= 1e-12 * float(ref.abs().max())


@pytest.mark.parametrize("slices", [7, 8])
@pytest.mark.parametrize("m,k", [(1028, 272), (4100, 2048)])
def test_fused_lower_product_is_bitwise_the_library_product(nv, slices, m, k):
    g = torch.Generator().manual_seed(m * k)
    A = _cov_like(m, k, g)
    out = {}
    for eng in ("library", "native"):
        _engine(nv, eng, slices)
        C = torch.full((m, m), 7.0, dtype=torch.float64, device="cuda")
        nv.gemm_ozaki_nt(A, None, slices=slices, alpha=-1.0, beta=1.0, C=C, lower_only=True)
        out[eng] = C
    assert _bits_equal(out["library"], out["native"])
    blk = torch.arange(m, device="cuda") // 128
    assert bool((out["native"][blk[None, :] > blk[:, None]] == 7.0).all())       # upper blocks untouched


def test_fused_engine_declines_what_it_does_not_take(nv):
    from gptorch_b200._lib import NativeLibraryError
    _engine(nv, "native", 8)
    A = torch.rand(64, 64, dtype=torch.float64, device="cuda")
    with pytest.raises(NativeLibraryError, match="rc=-5"):
        nv.gemm_ozaki_nt(A, None, slices=9)                   # more classes than tensor memory holds
    with pytest.raises(NativeLibraryError, match="rc=-5"):
        nv.gemm_ozaki_nt(torch.rand(64, 100, dtype=torch.float64, device="cuda"), None, slices=8)


def _factor_and_inverse(nv, n, seed):
    g = torch.Generator().manual_seed(seed)
    X = torch.rand(n, 8, generator=g, dtype=torch.float64).cuda()
    ell = torch.ones(8, dtype=torch.float64, device="cuda")
    s2 = torch.ones(1, dtype=torch.float64, device="cuda")
    noise = torch.full((1,), 0.01, dtype=torch.float64, device="cuda")
    buf, ld = nv._aligned_empty(n, n, X.device)
    nv.kern_fwd(0, X, None, ell, s2, noise=noise, lower=True, out=buf, ldk=ld)
    dinv, info = nv.potrf_(buf, ld)
    assert int(info.item()) == 0
    L = torch.tril(buf[:, :n]).clone()
    kd = nv.potri_(buf, ld, dinv)
    K = nv.potri_assemble(buf, ld, kd).clone()
    del buf
    return L, K


@pytest.mark.parametrize("n", [8192, 16384])
def test_cholesky_factor_is_bitwise_that_of_the_library_engine(nv, n):
    """n = 8192 and 16384 cross the factor's hooks: look-ahead trailing updates (A A^T, lower blocks) and the panel update
    (plain NT).  The default inverse is the DMMA engine's on that factor."""
    res = {}
    for eng in ("library", "native"):
        _engine(nv, eng, 8)
        res[eng] = _factor_and_inverse(nv, n, 22)
        torch.cuda.empty_cache()
    assert _bits_equal(res["library"][0], res["native"][0])


def test_dmma_engine_is_still_reachable_and_differs(nv):
    """GPB_I8MMA=0 runs the FP64 DMMA engine: its factor is not the sliced one (the switch really switches), and the two
    agree to the sliced engine's accuracy."""
    res = {}
    for eng in ("dmma", "native"):
        _engine(nv, eng, 8)
        res[eng] = _factor_and_inverse(nv, 8192, 23)
    (L0, K0), (L1, K1) = res["dmma"], res["native"]
    assert not torch.equal(L0, L1)
    assert float((L1 - L0).abs().max()) / float(L0.abs().max()) < 5e-12
    assert float((K1 - K0).abs().max()) / float(K0.abs().max()) < 1e-11


@pytest.mark.parametrize("noise", [1e-6, 1e-5, 1e-4, 1e-2])
def test_ill_conditioned_gpr_takes_the_dmma_engines_jitter_decisions_and_accuracy(nv, noise):
    """GPR loss+grad at N = 8192 with long length scales, cond(Ky) up to ~1e10 at noise 1e-6.

    The fused engine takes the same jitter decisions (potrf info of the plain factorisation and of each jitter level) as
    the DMMA engine.  Accuracy is judged against the DMMA engine's own spread: the same model with its training points
    permuted has the same exact loss but another rounding path, so the DMMA engine's distances from the fp64 oracle over
    a few permutations say how far an FP64 evaluation of this problem lands.  Wherever the DMMA engine meets the reference
    tolerances (loss 1e-9, gradients 1e-7) on every permutation, the fused engine does too, and everywhere its distance
    stays within 10x the DMMA engine's largest plus 1e-10 (the sliced products' norm-wise error; measured on B200: at
    cond ~1e10 the loss is 8e-9 .. 1.1e-8 from the oracle against DMMA's 1e-10 .. 1.8e-9, at noise >= 1e-4 within 2x)."""
    from oracle import gp_oracle as O
    from gptorch_b200 import kernels, likelihoods
    from gptorch_b200.models import GPR
    n, d = 8192, 8
    X, Y, _ = O.synth_regression(n, d)
    ell = np.full(d, 2.5)
    variance = 1.5
    ref_loss, ref_grads = O.gpr_loss_and_grads("Rbf", X, Y, ell, variance, noise)
    ref_loss = float(ref_loss.sum())
    g = torch.Generator().manual_seed(0)
    perms = [torch.arange(n)] + [torch.randperm(n, generator=g) for _ in range(2)]
    infos, dist = {}, {}
    for eng in ("dmma", "native"):
        _engine(nv, eng, 8)
        Xc = X.cuda()
        ell_t = torch.tensor(ell, dtype=torch.float64, device="cuda")
        s2 = torch.tensor([variance], dtype=torch.float64, device="cuda")
        nz = torch.tensor([noise], dtype=torch.float64, device="cuda")
        infos[eng] = []
        for jit in (0.0, 1e-10, 1e-8, 1e-6):
            buf, ld = nv._aligned_empty(n, n, Xc.device)
            nv.kern_fwd(0, Xc, None, ell_t, s2, noise=nz, lower=True, out=buf, ldk=ld)
            if jit:
                nv.add_diag_(buf, ld, jit)
            _, info = nv.potrf_(buf, ld)
            infos[eng].append(int(info.item()))
            del buf
        dist[eng] = []
        for p in perms:
            model = GPR(X[p].numpy(), Y[p].numpy(), kernels.Rbf(d, ARD=True, length_scales=ell.copy(), variance=variance),
                        likelihood=likelihoods.Gaussian(variance=noise))
            loss = model.loss()
            loss.backward()
            e = {"loss": abs(float(loss.item()) - ref_loss) / abs(ref_loss)}
            for k, v in (("variance", model.kernel.variance), ("length_scales", model.kernel.length_scales),
                         ("noise", model.likelihood.variance)):
                r = ref_grads[k].numpy().ravel()
                e[k] = float(np.abs(v.grad.cpu().numpy().ravel() - r).max() / np.abs(r).max())
            dist[eng].append(e)
    assert infos["native"] == infos["dmma"]
    for k in dist["dmma"][0]:
        tol = 1e-9 if k == "loss" else 1e-7
        worst_dmma = max(e[k] for e in dist["dmma"])
        worst_native = max(e[k] for e in dist["native"])
        if worst_dmma <= tol:
            assert worst_native <= tol, (k, dist)
        assert worst_native <= 10.0 * worst_dmma + 1e-10, (k, dist)
