"""GPR.posterior(): predictions from a factorisation computed once, differentiable in the test inputs x* only -- what
Bayesian optimisation, sensitivity analysis and active learning differentiate.  Checked against the torch-CPU oracle's
autograd, against GPR.predict_f (values under no_grad, x* gradients with autograd), for reuse of the factorisation,
reproducibility, and an acquisition-function ascent end to end."""
import contextlib

import numpy as np
import pytest
import torch

from conftest import Cases, rel_err

VAL_TOL = 1e-9
GRAD_TOL = 1e-7

_COMP = Cases("composite_cases.npz")
_STATIONARY = ["Rbf", "Exp", "Matern32", "Matern52", "Periodic"]


def _kern(kind, d, ell, var, ard):
    from gptorch_b200 import kernels
    if kind == "Linear":
        return kernels.Linear(d, variance=np.full(d, var), ARD=True)
    ls = np.array(ell, dtype=np.float64).copy() if ard else float(np.mean(ell))
    return getattr(kernels, kind)(d, ARD=ard, length_scales=ls, variance=float(var))


def _ell(kind, d):
    # Periodic (cos r) is positive definite only while the scaled distances stay short
    return (4.0 if kind == "Periodic" else 1.0) * (0.4 * np.sqrt(d) + 0.05 * np.arange(d))


def _data(n, d, dy, seed=1234):
    from oracle import gp_oracle as O
    X, Y1, _ = O.synth_regression(n, d, seed=seed)
    Y = torch.cat([Y1 * (1.0 + 0.5 * k) + 0.05 * k for k in range(dy)], dim=1)
    return X, Y


def _test_points(X, ns, seed=5):
    """ns test inputs: rows 1, 4, 7, ... are training inputs (coincident points), the others are drawn from a box three
    times the data's, so that some predictive variances stay of the order of the kernel variance.  (A lone test point
    on a training input has a variance of the order of the noise, left after cancelling most of sigma2: its relative
    error measures that cancellation, not the prediction.)"""
    g = torch.Generator().manual_seed(seed)
    Xs = 3.0 * torch.rand(ns, X.shape[1], generator=g, dtype=torch.float64) - 1.0
    idx = torch.randint(0, X.shape[0], (ns,), generator=g)
    Xs[1::3] = X[idx[1::3]]
    return Xs


def _weights(ns, dy, seed=11):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(ns, dy, generator=g, dtype=torch.float64), torch.randn(ns, dy, generator=g, dtype=torch.float64)


def _model(kern, X, Y, noise):
    from gptorch_b200 import likelihoods
    from gptorch_b200.models import GPR
    return GPR(X.numpy(), Y.numpy(), kern, likelihood=likelihoods.Gaussian(variance=noise))


def _native(post, Xs, wm, wv):
    """(mean, var, d(sum(wm mean) + sum(wv var))/dx*) through a posterior (or a model: same call surface)."""
    x = Xs.clone().cuda().requires_grad_(True)
    mean, var = post.predict_f(x)
    (mean * wm.cuda() + var * wv.cuda()).sum().backward()
    return mean.detach().cpu(), var.detach().cpu(), x.grad.detach().cpu()


def _exact_r(A, B, ell):
    """Scaled distances as sums of squared differences (exact zero for coincident points), clamped like the reference."""
    As, Bs = A / ell, B / ell
    return torch.sqrt(torch.clamp(((As[:, None, :] - Bs[None, :, :]) ** 2).sum(-1), min=1e-40))


def _oracle(kind, X, Y, Xs, ell, var, noise, wm, wv):
    """The reference's predictive equations (oracle.gpr_predict) under the oracle's autograd.  For Exp the distances
    are formed exactly (the checker variant of test_gpu_input_grads): the reference's expanded distance carries
    round-off of 1e-8 at coincident points, which Exp's value and its 1/r derivative do not damp."""
    from oracle import gp_oracle as O
    Xp = Xs.clone().requires_grad_(True)
    if kind == "Exp":
        e = torch.as_tensor(np.atleast_1d(ell))
        L = O.chol(var * torch.exp(-_exact_r(X, X, e)) + noise * torch.eye(X.shape[0], dtype=torch.float64))
        A = O.tri_solve(var * torch.exp(-_exact_r(X, Xp, e)), L)
        mean = A.t() @ O.tri_solve(Y, L)
        v = (var - (A * A).sum(0))[:, None].expand_as(mean)
    else:
        h = O.Hyper(kind, None if kind == "Linear" else np.atleast_1d(ell),
                    np.full(X.shape[1], var) if kind == "Linear" else var, noise)
        mean, v = O.gpr_predict(h, X, Y, Xp)
    (mean * wm + v * wv).sum().backward()
    return mean.detach(), v.detach(), Xp.grad


def _check(got, want, prior_var=0.0):
    """Mean and x* gradient relative to their largest magnitude; the variance relative to the larger of its largest
    magnitude and the prior variance: sigma2 - k*^T Ky^-1 k* is a difference of terms of the size of sigma2, so its
    rounding is of that size even where the posterior variance is far smaller (test points inside dense data)."""
    assert rel_err(got[0].numpy(), want[0].numpy()) <= VAL_TOL
    dv = float(np.max(np.abs(got[1].numpy() - want[1].numpy())))
    assert dv / max(float(np.max(np.abs(want[1].numpy()))), prior_var, 1e-300) <= VAL_TOL
    assert rel_err(got[2].numpy(), want[2].numpy()) <= GRAD_TOL


_DIMS = [1, 8, 17, 40]
# every stationary family at every D; dy, N (ragged), n* (1 and ragged) and ARD rotate so that each meets every family
_CASES = [(kind, d, [1, 3, 9][(i + k) % 3], [300, 1000][(i + k) % 2], [1, 77, 200][(2 * i + k) % 3], (i + k) % 2 == 0)
          for k, kind in enumerate(_STATIONARY) for i, d in enumerate(_DIMS)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,d,dy,n,ns,ard", _CASES)
def test_posterior_matches_oracle(kind, d, dy, n, ns, ard):
    X, Y = _data(n, d, dy)
    ell = _ell(kind, d)
    var, noise = 1.3, 0.05
    post = _model(_kern(kind, d, ell, var, ard), X, Y, noise).posterior()
    assert post.Kinv is not None                                  # the fused node
    Xs = _test_points(X, ns)
    wm, wv = _weights(ns, dy)
    _check(_native(post, Xs, wm, wv), _oracle(kind, X, Y, Xs, ell if ard else [np.mean(ell)], var, noise, wm, wv), var)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,d,dy", [("Rbf", 8, 1), ("Matern52", 17, 3), ("Periodic", 3, 2), ("Linear", 5, 2)])
def test_posterior_agrees_with_predict_f(kind, d, dy):
    """Means agree with predict_f under no_grad to 1e-12, variances to 1e-10, and x* gradients with predict_f's
    autograd to 1e-9.  The variance is sigma2 - k*^T Ky^-1 k* through the explicit inverse here and sigma2 - |L^-1 k*|^2
    through a solve in predict_f; the two roundings differ by about cond(Ky) eps sigma2 (measured on a B200: 1.0e-12
    for Rbf and 2.1e-11 for Periodic, whose variances here are two orders below sigma2)."""
    X, Y = _data(777, d, dy)
    model = _model(_kern(kind, d, _ell(kind, d), 1.3, True), X, Y, 0.05)
    post = model.posterior()
    Xs = _test_points(X, 150)
    wm, wv = _weights(150, dy)
    with torch.no_grad():
        mean_m, var_m = model.predict_f(Xs.cuda())
        mean_p, var_p = post.predict_f(Xs.cuda())
    assert rel_err(mean_p.cpu().numpy(), mean_m.cpu().numpy()) <= 1e-12
    assert rel_err(var_p.cpu().numpy(), var_m.cpu().numpy()) <= 1e-10
    g_post = _native(post, Xs, wm, wv)[2]
    g_model = _native(model, Xs, wm, wv)[2]
    assert rel_err(g_post.numpy(), g_model.numpy()) <= 1e-9


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["Rbf", "Matern32"])
def test_posterior_does_not_refactorise_and_trains_nothing(kind, monkeypatch):
    from gptorch_b200 import _native as nv
    X, Y = _data(1000, 4, 2)
    model = _model(_kern(kind, 4, _ell(kind, 4), 1.3, True), X, Y, 0.05)
    post = model.posterior()
    Xs = _test_points(X, 64)
    wm, wv = _weights(64, 2)

    torch.cuda.synchronize()
    nv.reset_launch_count()
    _native(model, Xs, wm, wv)
    torch.cuda.synchronize()
    model_launches = nv.launch_count()
    model.zero_grad(set_to_none=True)

    def refuse(*args, **kwargs):
        raise AssertionError("the posterior refactorised")

    for name in ("potrf_", "potri_", "trsv_", "trsm_right_lt_", "trtri_upper_"):
        monkeypatch.setattr(nv, name, refuse)
    counts = []
    for _ in range(3):
        nv.reset_launch_count()
        _native(post, Xs, wm, wv)
        torch.cuda.synchronize()
        counts.append(nv.launch_count())
    assert counts[0] == counts[1] == counts[2] and 0 < counts[0] < model_launches
    assert all(p.grad is None for p in model.parameters())
    assert all(not p.requires_grad for m in (post.kernel, post.mean_function, post.likelihood) for p in m.parameters())


@pytest.mark.gpu
def test_posterior_is_a_snapshot():
    X, Y = _data(500, 3, 1)
    model = _model(_kern("Rbf", 3, _ell("Rbf", 3), 1.3, True), X, Y, 0.05)
    post = model.posterior()
    Xs = _test_points(X, 20).cuda()
    with torch.no_grad():
        before = post.predict_f(Xs)[0].clone()
        model.kernel.variance.data.add_(0.5)
        model.X.mul_(2.0)
        after = post.predict_f(Xs)[0]
        fresh = model.posterior().predict_f(Xs)[0]
    assert torch.equal(before, after)
    assert not torch.equal(before, fresh)


def _composite_oracle(name, Xs, wm, wv):
    from oracle import gp_oracle as O
    c = _COMP
    kinds = [str(k) for k in c.get(name, "kinds")]
    X, Y = torch.as_tensor(c.get(name, "X")), torch.as_tensor(c.get(name, "Y"))
    leaves = []
    for i, kind in enumerate(kinds):
        ell = torch.as_tensor(c.get(name, "leaf%d/ell" % i)) if c.has(name, "leaf%d/ell" % i) else None
        leaves.append((kind, ell, torch.as_tensor(c.get(name, "leaf%d/variance" % i))))
    expr = str(c.get(name, "expr"))
    Xp = Xs.clone().requires_grad_(True)
    with (O.exact_diagonal() if "Exp" in kinds else contextlib.nullcontext()):
        L = O.chol(O.cov_composite(expr, leaves, X) + float(c.get(name, "noise")) * torch.eye(X.shape[0],
                                                                                             dtype=torch.float64))
        A = O.tri_solve(O.cov_composite(expr, leaves, X, Xp), L)
        kdiag = O.cov_composite(expr, leaves, Xp).diagonal()
    mean = A.t() @ O.tri_solve(Y, L)
    v = (kdiag - (A * A).sum(0))[:, None].expand_as(mean)
    (mean * wm + v * wv).sum().backward()
    return mean.detach(), v.detach(), Xp.grad


@pytest.mark.gpu
@pytest.mark.parametrize("name", _COMP.names)
def test_composite_posterior_matches_oracle(name):
    from test_gpu_input_grads import _composite
    c = _COMP
    kern, kinds = _composite(name)
    X, Y = torch.as_tensor(c.get(name, "X")), torch.as_tensor(c.get(name, "Y"))
    post = _model(kern, X, Y, float(c.get(name, "noise"))).posterior()
    assert post.L is not None                                     # the composed path
    # test points away from the training inputs: Exp's expanded-distance round-off (DESIGN 6) stays out of the check
    Xs = _test_points(X, 40)[::3]
    wm, wv = _weights(Xs.shape[0], Y.shape[1])
    _check(_native(post, Xs, wm, wv), _composite_oracle(name, Xs, wm, wv))


@pytest.mark.gpu
def test_linear_posterior_matches_oracle():
    X, Y = _data(300, 4, 2)
    post = _model(_kern("Linear", 4, None, 0.7, True), X, Y, 0.05).posterior()
    assert post.L is not None
    Xs = _test_points(X, 50)
    wm, wv = _weights(50, 2)
    _check(_native(post, Xs, wm, wv), _oracle("Linear", X, Y, Xs, None, 0.7, 0.05, wm, wv))


@pytest.mark.gpu
@pytest.mark.parametrize("kind,d", [("Rbf", 8), ("Exp", 24), ("Periodic", 40)])
def test_posterior_gradient_is_reproducible(kind, d):
    X, Y = _data(1000, d, 3)
    post = _model(_kern(kind, d, _ell(kind, d), 1.3, True), X, Y, 0.05).posterior()
    Xs = _test_points(X, 300)
    wm, wv = _weights(300, 3)
    a, b = _native(post, Xs, wm, wv), _native(post, Xs, wm, wv)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])


@pytest.mark.gpu
def test_single_test_point_with_a_broadcast_gradient():
    """n* = 1, dy = 1 and loss = mean.sum() + var.sum(): the upstream gradients arrive as broadcast 1 x 1 tensors."""
    X, Y = _data(500, 4, 1)
    ell = _ell("Matern32", 4)
    post = _model(_kern("Matern32", 4, ell, 1.3, True), X, Y, 0.05).posterior()
    Xs = _test_points(X, 1)
    x = Xs.clone().cuda().requires_grad_(True)
    mean, var = post.predict_f(x)
    (mean.sum() + var.sum()).backward()
    one = torch.ones(1, 1, dtype=torch.float64)
    want = _oracle("Matern32", X, Y, Xs, ell, 1.3, 0.05, one, one)
    _check((mean.detach().cpu(), var.detach().cpu(), x.grad.cpu()), want, 1.3)


@pytest.mark.gpu
def test_posterior_shapes_predict_y_and_samples():
    X, Y = _data(400, 3, 2)
    model = _model(_kern("Matern52", 3, _ell("Matern52", 3), 1.3, True), X, Y, 0.05)
    post = model.posterior()
    Xs = _test_points(X, 30)
    m, v = post.predict_y(Xs.numpy())
    assert isinstance(m, np.ndarray) and m.shape == v.shape == (30, 2)
    with torch.no_grad():
        mm, vm = model.predict_y(Xs.cuda())
        mf, cf = post.predict_f(Xs.cuda(), diag=False)
        mfm, cfm = model.predict_f(Xs.cuda(), diag=False)
    assert rel_err(m, mm.cpu().numpy()) <= 1e-12 and rel_err(v, vm.cpu().numpy()) <= 1e-10
    assert cf.shape == (30, 30) and rel_err(cf.cpu().numpy(), cfm.cpu().numpy()) <= 1e-9
    x = Xs.clone().cuda().requires_grad_(True)
    s = post.predict_f_samples(x, n_samples=4)
    assert s.shape == (4, 30, 2)
    s.sum().backward()
    assert torch.isfinite(x.grad).all()
    assert all(p.grad is None for p in model.parameters())


@pytest.mark.gpu
def test_ucb_ascent_matches_predict_f_path():
    """A few Adam steps on an upper-confidence-bound acquisition over 16 candidate points with a fixed N = 8192 model:
    the posterior drives the candidates along the same path as predict_f with autograd."""
    n, d, ns, beta = 8192, 8, 16, 2.0
    X, Y = _data(n, d, 1)
    ell = 0.4 * np.sqrt(d) + 0.05 * np.arange(d)
    model = _model(_kern("Rbf", d, ell, 1.3, True), X, Y, 0.05)
    post = model.posterior()
    start = _test_points(X, ns, seed=3).cuda()

    def ascend(source):
        x = start.clone().requires_grad_(True)
        opt = torch.optim.Adam([x], lr=0.05)
        for _ in range(5):
            opt.zero_grad()
            mean, var = source.predict_f(x)
            (-(mean + beta * var.clamp_min(1e-30).sqrt())).sum().backward()
            opt.step()
        return x.detach().cpu()

    got, want = ascend(post), ascend(model)
    assert rel_err(got.numpy(), want.numpy()) <= 1e-9
    assert not torch.equal(got, start.cpu())


def test_posterior_validates_before_any_native_call(monkeypatch):
    """No GPU needed: a D mismatch is a ValueError raised before the library is touched, and a CPU tensor that reaches
    the library raises NativeLibraryError (there is no CPU path)."""
    from gptorch_b200 import _lib, _native as nv, kernels, likelihoods, mean_functions
    from gptorch_b200.models import GPR, GPRPosterior
    n, d = 50, 3
    X = torch.rand(n, d, dtype=torch.float64)
    kern = kernels.Rbf(d, ARD=True)
    post = GPRPosterior(kern, mean_functions.Zero(1), likelihoods.Gaussian(variance=0.1), X,
                        Kinv=torch.eye(n, dtype=torch.float64), a=torch.zeros(n, 1, dtype=torch.float64))
    def no_native(*args):
        raise AssertionError("native call before validation")

    with monkeypatch.context() as m:
        m.setattr(nv, "call", no_native)
        m.setattr(nv, "query", no_native)
        with pytest.raises(ValueError):
            post.predict_f(torch.rand(4, d + 1, dtype=torch.float64))
        with pytest.raises(ValueError):
            post.predict_f(np.random.rand(4, d - 1))
    with pytest.raises(_lib.NativeLibraryError):
        post.predict_f(torch.rand(4, d, dtype=torch.float64))
    model = GPR(X.numpy(), torch.rand(n, 1, dtype=torch.float64).numpy(), kern)
    model.cpu()
    with pytest.raises(_lib.NativeLibraryError):
        model.posterior()
