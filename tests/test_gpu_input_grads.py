"""Gradients with respect to the training inputs x through the fused nodes (GPR stationary, GPR Sum / Product, VFE):
against the torch-CPU oracle's autograd, against the step-by-step native path, and bitwise reproducibility.  What a
user of deep kernel learning or learned input warps relies on: log_likelihood(x=net(x_raw)) differentiates net."""
import contextlib

import numpy as np
import pytest
import torch

from conftest import Cases, rel_err

pytestmark = pytest.mark.gpu

LML_TOL = 1e-9
GRAD_TOL = 1e-7

_COMP = Cases("composite_cases.npz")


def _kern(kind, d, ell, var, ard):
    from gptorch_b200 import kernels
    if kind == "Linear":      # one variance per dimension (the native Linear leaf is ARD)
        return kernels.Linear(d, variance=np.full(d, var), ARD=True)
    ls = np.array(ell, dtype=np.float64).copy() if ard else float(np.mean(ell))
    return getattr(kernels, kind)(d, ARD=ard, length_scales=ls, variance=float(var))


def _native_gpr(kern, X, Y, noise, x=None, need_x=True):
    """(loss, gX or None, {param: grad}) of -GPR.log_likelihood(x) on cuda."""
    from gptorch_b200 import likelihoods
    from gptorch_b200.models import GPR
    model = GPR(X.numpy(), Y.numpy(), kern, likelihood=likelihoods.Gaussian(variance=noise))
    if x is None:
        x = X.clone().cuda()
    if need_x:
        x = x.detach().requires_grad_(True)
    loss = -model.log_likelihood(x=x)
    loss.sum().backward()
    grads = {n: p.grad.detach().clone() for n, p in model.named_parameters() if p.grad is not None}
    return loss.detach(), (x.grad.detach().clone() if need_x else None), grads


def _oracle_gpr(kind, X, Y, ell, var, noise, ard, exact=False):
    """-loglik and d/dX from the oracle (the reference's expanded-distance autograd)."""
    from oracle import gp_oracle as O
    d = X.shape[1]
    if kind == "Linear":
        h = O.Hyper(kind, None, np.full(d, var), noise)
    else:
        h = O.Hyper(kind, np.array(ell) if ard else np.array([np.mean(ell)]), var, noise)
    Xp = X.clone().requires_grad_(True)
    with (O.exact_diagonal() if exact else contextlib.nullcontext()):
        loss = -O.gpr_loglik(h, Xp, Y)
    loss.sum().backward()
    return loss.detach(), Xp.grad


def _oracle_exp_exact_distance(X, Y, ell, var, noise):
    """-loglik and d/dX for Exp with the scaled distances formed as sums of squared differences (exact zero for
    coincident points) instead of the reference's |x|^2 + |x'|^2 - 2 x.x'.  A checker variant, as O.exact_diagonal: for
    close pairs the expanded form's round-off (relative 1e-4 at a spacing of 1e-6) is multiplied by Exp's 1/r in dK/dx,
    so the reference's own input gradient is not accurate to GRAD_TOL there (DESIGN 6)."""
    from oracle import gp_oracle as O
    ell = np.atleast_1d(np.asarray(ell, dtype=np.float64))
    h = O.Hyper("Exp", ell, var, noise)
    Xp = X.clone().requires_grad_(True)
    Xs = Xp / h.ell
    r = torch.sqrt(torch.clamp(((Xs[:, None, :] - Xs[None, :, :]) ** 2).sum(-1), min=1e-40))
    n = X.shape[0]
    L = O.chol(h.variance * torch.exp(-r) + h.noise * torch.eye(n, dtype=torch.float64))
    alpha = O.tri_solve(Y, L)
    loss = 0.5 * alpha.pow(2).sum() + Y.shape[1] * O.tri_logdet(L) + 0.5 * Y.numel() * np.log(2 * np.pi)
    loss.backward()
    return loss.detach(), Xp.grad


def _ell(kind, d):
    # Periodic (cos r) is positive definite only while the scaled distances stay short
    return (4.0 if kind == "Periodic" else 1.0) * (0.4 * np.sqrt(d) + 0.05 * np.arange(d))


def _data(n, d, dy, seed=1234):
    from oracle import gp_oracle as O
    X, Y1, _ = O.synth_regression(n, d, seed=seed)
    Y = torch.cat([Y1 * (1.0 + 0.5 * k) + 0.05 * k for k in range(dy)], dim=1)
    return X, Y


_FAMILIES = ["Rbf", "Exp", "Matern32", "Matern52", "Periodic", "Linear"]
_DIMS = [1, 8, 17, 32, 40]
# every family at every D (so both the DMMA and the scalar reductions run for the hyper-parameters); dy, N and ARD
# rotate so that dy = 9 (> the DMMA path's 8-output chunk), ragged N and the isotropic form all meet every family
_GPR_CASES = [(kind, d, [1, 3, 9][(i + k) % 3], [300, 1000][(i + k) % 2], (i + k) % 2 == 0)
              for k, kind in enumerate(_FAMILIES) for i, d in enumerate(_DIMS)]


@pytest.mark.parametrize("kind,d,dy,n,ard", _GPR_CASES)
def test_gpr_input_gradient_matches_oracle(kind, d, dy, n, ard):
    X, Y = _data(n, d, dy)
    ell = _ell(kind, d)
    var, noise = 1.3, 0.05
    loss, gX, _ = _native_gpr(_kern(kind, d, ell, var, ard), X, Y, noise)
    if kind == "Exp":
        _, ref_gX = _oracle_exp_exact_distance(X, Y, ell if ard else [np.mean(ell)], var, noise)
        ref_loss, _ = _oracle_gpr(kind, X, Y, ell, var, noise, ard, exact=True)
    else:
        ref_loss, ref_gX = _oracle_gpr(kind, X, Y, ell, var, noise, ard)
    assert rel_err(loss.cpu().numpy(), ref_loss.numpy()) <= LML_TOL
    assert rel_err(gX.cpu().numpy(), ref_gX.numpy()) <= GRAD_TOL


@pytest.mark.parametrize("kind", ["Rbf", "Matern32", "Matern52"])
def test_gpr_input_gradient_with_duplicate_rows(kind):
    """Exactly coincident training rows (common in real data): the pair contributes nothing to either row's gradient
    (for Matern through the distance clamp), as in the reference.  (Exp on coincident pairs: the reference's distance
    is sqrt(round-off), whose derivative is the documented exception of DESIGN 6.)"""
    X, Y = _data(400, 3, 2)
    X[200:260] = X[0:60]             # 60 duplicated rows, with different targets
    ell = np.array([0.5, 0.7, 0.9])
    _, gX, _ = _native_gpr(_kern(kind, 3, ell, 1.1, True), X, Y, 0.05)
    _, ref_gX = _oracle_gpr(kind, X, Y, ell, 1.1, 0.05, True)
    assert torch.isfinite(gX).all()
    assert rel_err(gX.cpu().numpy(), ref_gX.numpy()) <= GRAD_TOL


def test_gpr_input_gradient_after_a_jitter_retry():
    """Ky singular without jitter (every point duplicated, noise 1e-30): the factorisation is retried with the
    reference's schedule, and the input gradient is that of the jittered loss.

    The jitter is a constant on the diagonal, so the loss and gX after the retry are BITWISE those of the same model
    whose noise already holds the jitter (1 + 1e-30 == 1: both build the same Ky, factorise it at the first attempt
    of the second model, and reduce the same W) -- equal losses also show that exactly one retry, at 1e-10, happened.

    Against the oracle's jitter_retry: after the retry cond(Ky) ~ 1e10, and one-ulp perturbations of Ky move the
    oracle's own gX by 4e-6 .. 7e-6 (max-norm relative; measured over random symmetric perturbations), so the
    comparison is made at 3e-5, not GRAD_TOL.  The oracle keeps the reference's values (expanded distances: the same
    Ky, jitter and W) but differentiates the distances exactly: on a coincident pair W is ~1e10 and the expanded
    form's derivative there is round-off instead of 0, whose product would swamp even that bound."""
    from oracle import gp_oracle as O
    x = np.linspace(0, 1, 30).reshape(-1, 1)
    x = np.concatenate([x, x])
    X = torch.as_tensor(x)
    Y = torch.sin(6 * X)
    ell, n = 0.02, X.shape[0]
    h = O.Hyper("Rbf", [ell], 1.0, 1e-30)
    with pytest.raises(RuntimeError):     # the un-jittered factorisation fails: at least one retry happens
        torch.linalg.cholesky(O.gpr_kyy(h, X))
    loss, gX, _ = _native_gpr(_kern("Rbf", 1, [ell], 1.0, True), X, Y, 1e-30)
    loss_f, gX_f, _ = _native_gpr(_kern("Rbf", 1, [ell], 1.0, True), X, Y, 1e-10)
    assert torch.equal(loss, loss_f)
    assert torch.equal(gX, gX_f)

    Xp = X.clone().requires_grad_(True)
    r2_val = O.scaled_r2(X, None, h.ell).detach()
    r2_dir = ((Xp[:, None, :] - Xp[None, :, :]) ** 2).sum(-1) / ell ** 2
    K = h.variance * torch.exp(-(r2_val + r2_dir - r2_dir.detach()) / 2.0) + h.noise * torch.eye(n, dtype=torch.float64)
    L = O.chol(K)
    alpha = O.tri_solve(Y, L)
    ref = 0.5 * alpha.pow(2).sum() + O.tri_logdet(L) + 0.5 * n * np.log(2 * np.pi)
    ref.backward()
    assert rel_err(loss.cpu().numpy(), ref.detach().numpy()) <= 1e-6
    assert rel_err(gX.cpu().numpy(), Xp.grad.numpy()) <= 3e-5


def _composite(name):
    from gptorch_b200 import kernels
    c = _COMP
    kinds = [str(k) for k in c.get(name, "kinds")]
    d = int(c.get(name, "d"))
    leaves = []
    for i, kind in enumerate(kinds):
        var = c.get(name, "leaf%d/variance" % i)
        if kind == "Linear":
            leaves.append(kernels.Linear(d, variance=var.copy(), ARD=True))
        elif kind in ("Constant", "White"):
            leaves.append(getattr(kernels, kind)(d, variance=float(var[0])))
        else:
            leaves.append(getattr(kernels, kind)(d, ARD=True, length_scales=c.get(name, "leaf%d/ell" % i).copy(),
                                                 variance=float(var[0])))
    kern = eval(str(c.get(name, "expr")), {"__builtins__": {}}, {"k%d" % i: k for i, k in enumerate(leaves)})
    return kern, kinds


def _oracle_composite_gx(name, exact):
    from oracle import gp_oracle as O
    c = _COMP
    kinds = [str(k) for k in c.get(name, "kinds")]
    X, Y = torch.as_tensor(c.get(name, "X")), torch.as_tensor(c.get(name, "Y"))
    leaves = []
    for i, kind in enumerate(kinds):
        ell = torch.as_tensor(c.get(name, "leaf%d/ell" % i)) if c.has(name, "leaf%d/ell" % i) else None
        leaves.append((kind, ell, torch.as_tensor(c.get(name, "leaf%d/variance" % i))))
    Xp = X.clone().requires_grad_(True)
    n = X.shape[0]
    with (O.exact_diagonal() if exact else contextlib.nullcontext()):
        K = O.cov_composite(str(c.get(name, "expr")), leaves, Xp)
    L = O.chol(K + float(c.get(name, "noise")) * torch.eye(n, dtype=torch.float64))
    alpha = O.tri_solve(Y, L)
    loss = 0.5 * alpha.pow(2).sum() + Y.shape[1] * O.tri_logdet(L) + 0.5 * Y.numel() * np.log(2 * np.pi)
    loss.backward()
    return Xp.grad


@pytest.mark.parametrize("name", _COMP.names)
def test_composite_gpr_input_gradient_matches_oracle(name):
    from gptorch_b200 import kernels
    c = _COMP
    kern, kinds = _composite(name)
    assert kernels.sum_of_products(kern) is not None          # the fused composite node
    X, Y = torch.as_tensor(c.get(name, "X")), torch.as_tensor(c.get(name, "Y"))
    _, gX, _ = _native_gpr(kern, X, Y, float(c.get(name, "noise")))
    ref = _oracle_composite_gx(name, exact="Exp" in kinds)
    assert rel_err(gX.cpu().numpy(), ref.numpy()) <= GRAD_TOL


def _vfe(X, Y, Z, d, ell, x):
    from gptorch_b200 import kernels, likelihoods
    from gptorch_b200.models import VFE
    model = VFE(X.numpy(), Y.numpy(), kernels.Matern52(d, ARD=True, length_scales=ell.copy(), variance=1.3),
                inducing_points=Z.numpy(), likelihood=likelihoods.Gaussian(variance=0.05))
    loss = -model.log_likelihood(x=x)
    loss.sum().backward()
    grads = {n: p.grad.detach().clone() for n, p in model.named_parameters() if p.grad is not None}
    return loss.detach(), grads


@pytest.mark.parametrize("chunk", [1000, 999, 64])
def test_vfe_input_gradient_both_forms_ragged_chunks_and_panel_cache(chunk, monkeypatch):
    from oracle import gp_oracle as O
    from gptorch_b200 import settings, _autograd as ag
    from gptorch_b200.models import sparse_gpr
    n, d, m, dy = 4321, 5, 37, 3
    X, Y = _data(n, d, dy)
    Z = O.synth_inducing(X, m, torch.Generator().manual_seed(7))
    ell = 0.5 + 0.1 * np.arange(d)
    h = O.Hyper("Matern52", ell, 1.3, 0.05)
    Xp = X.clone().requires_grad_(True)
    ref = -O.vfe_elbo(h, Xp, Y, Z)
    ref.backward()
    monkeypatch.setattr(sparse_gpr, "VFE_CHUNK_ROWS", chunk)
    for form in (True, False):
        for budget in (ag.VFE_PANEL_CACHE_BYTES, 0):
            monkeypatch.setattr(ag, "VFE_PANEL_CACHE_BYTES", budget)
            settings.vfe_phi_form = form
            try:
                x = X.clone().cuda().requires_grad_(True)
                loss, _ = _vfe(X, Y, Z, d, ell, x)
            finally:
                settings.vfe_phi_form = "auto"
            assert rel_err(loss.item(), ref.item()) <= LML_TOL, (form, budget)
            assert rel_err(x.grad.cpu().numpy(), Xp.grad.numpy()) <= GRAD_TOL, (form, budget)


def test_gpr_mid_size_matches_step_by_step_path_and_oracle():
    """N = 8192 (64 column blocks, many CTAs): the fused node's gX against the step-by-step native path (a kernel
    subclass that overrides K goes through KernelFn -> CholeskyFn -> trtrs, which differentiates x) and the oracle."""
    from gptorch_b200 import kernels

    class StepRbf(kernels.Rbf):
        def K(self, X, X2=None):
            return super().K(X, X2)

    n, d = 8192, 8
    X, Y = _data(n, d, 1)
    ell = 0.4 * np.sqrt(d) + 0.05 * np.arange(d)
    _, gX, _ = _native_gpr(_kern("Rbf", d, ell, 1.3, True), X, Y, 0.05)
    step = StepRbf(d, ARD=True, length_scales=ell.copy(), variance=1.3)
    _, gX_step, _ = _native_gpr(step, X, Y, 0.05)
    _, ref_gX = _oracle_gpr("Rbf", X, Y, ell, 1.3, 0.05, True)
    assert rel_err(gX.cpu().numpy(), gX_step.cpu().numpy()) <= GRAD_TOL
    assert rel_err(gX.cpu().numpy(), ref_gX.numpy()) <= GRAD_TOL


def _assert_same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        assert torch.equal(a[k], b[k]), k


@pytest.mark.parametrize("kind,d,dy", [("Rbf", 8, 1), ("Matern32", 24, 3), ("Periodic", 40, 9)])
def test_gpr_nothing_else_moves_and_gx_is_reproducible(kind, d, dy):
    """Loss and every hyper-parameter gradient are bitwise the same whether x requires a gradient or not, and gX is
    bitwise the same across runs (fixed-order reductions, no atomics)."""
    X, Y = _data(1000, d, dy)
    ell = _ell(kind, d)
    l0, _, g0 = _native_gpr(_kern(kind, d, ell, 1.3, True), X, Y, 0.05, need_x=False)
    l1, x1, g1 = _native_gpr(_kern(kind, d, ell, 1.3, True), X, Y, 0.05)
    l2, x2, g2 = _native_gpr(_kern(kind, d, ell, 1.3, True), X, Y, 0.05)
    assert torch.equal(l0, l1)
    _assert_same(g0, g1)
    _assert_same(g1, g2)
    assert torch.equal(x1, x2)


def test_composite_nothing_else_moves_and_gx_is_reproducible():
    name = _COMP.names[0]
    c = _COMP
    X, Y = torch.as_tensor(c.get(name, "X")), torch.as_tensor(c.get(name, "Y"))
    runs = [_native_gpr(_composite(name)[0], X, Y, float(c.get(name, "noise")), need_x=nx) for nx in (False, True, True)]
    assert torch.equal(runs[0][0], runs[1][0])
    _assert_same(runs[0][2], runs[1][2])
    _assert_same(runs[1][2], runs[2][2])
    assert torch.equal(runs[1][1], runs[2][1])


@pytest.mark.parametrize("form", [True, False])
def test_vfe_nothing_else_moves_and_gx_is_reproducible(form):
    from oracle import gp_oracle as O
    from gptorch_b200 import settings
    n, d, m = 3000, 4, 50
    X, Y = _data(n, d, 2)
    Z = O.synth_inducing(X, m, torch.Generator().manual_seed(7))
    ell = 0.5 + 0.1 * np.arange(d)
    settings.vfe_phi_form = form
    try:
        runs = []
        for nx in (False, True, True):
            x = X.clone().cuda().requires_grad_(nx)
            loss, grads = _vfe(X, Y, Z, d, ell, x)
            runs.append((loss, x.grad, grads))
    finally:
        settings.vfe_phi_form = "auto"
    assert torch.equal(runs[0][0], runs[1][0])
    _assert_same(runs[0][2], runs[1][2])
    _assert_same(runs[1][2], runs[2][2])
    assert torch.equal(runs[1][1], runs[2][1])


def test_deep_kernel_learning_end_to_end():
    """A small MLP feeds GPR.log_likelihood(x=net(x_raw)); its weight gradients match the same MLP on the CPU through
    the oracle."""
    from gptorch_b200 import likelihoods, kernels
    from gptorch_b200.models import GPR
    from oracle import gp_oracle as O
    torch.manual_seed(0)
    n = 600
    x_raw, Y = _data(n, 4, 1)
    net = torch.nn.Sequential(torch.nn.Linear(4, 16), torch.nn.Tanh(), torch.nn.Linear(16, 8)).double()
    net_gpu = torch.nn.Sequential(torch.nn.Linear(4, 16), torch.nn.Tanh(), torch.nn.Linear(16, 8)).double().cuda()
    net_gpu.load_state_dict(net.state_dict())
    ell = 1.0 + 0.1 * np.arange(8)
    feats0 = net(x_raw).detach()
    model = GPR(feats0.numpy(), Y.numpy(), kernels.Rbf(8, ARD=True, length_scales=ell.copy(), variance=1.2),
                likelihood=likelihoods.Gaussian(variance=0.05))
    loss = -model.log_likelihood(x=net_gpu(x_raw.cuda()))
    loss.sum().backward()
    h = O.Hyper("Rbf", ell, 1.2, 0.05)
    ref = -O.gpr_loglik(h, net(x_raw), Y)
    ref.sum().backward()
    assert rel_err(loss.item(), ref.item()) <= LML_TOL
    # all weights as one vector: the last layer's bias gradient is zero (a stationary kernel is shift-invariant)
    got = torch.cat([p.grad.reshape(-1).cpu() for p in net_gpu.parameters()])
    want = torch.cat([q.grad.reshape(-1) for q in net.parameters()])
    assert rel_err(got.numpy(), want.numpy()) <= GRAD_TOL
