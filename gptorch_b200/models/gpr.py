"""Exact GP regression (reference: gptorch/models/gpr.py)."""
import copy

import torch

from .. import _autograd as ag
from .. import _native as nv
from .. import kernels
from ..functions import cholesky, trtrs, mm, mm_nt
from ..likelihoods import Gaussian
from ..param import Param
from ..util import torch_dtype
from .base import GPModel, input_as_tensor


def _native_kind(kernel):
    """Index of the fused native kernel family, or None when the kernel has to be composed in torch."""
    if isinstance(kernel, kernels.Stationary) and kernel._kind is not None and type(kernel).K is kernels.Stationary.K:
        return kernel._kind
    return None


class GPR(GPModel):
    """Gaussian-process regression with a Gaussian likelihood."""

    def __init__(self, x, y, kernel, mean_function=None, likelihood=None, name="gpr"):
        super().__init__(x, y, kernel, likelihood, mean_function, name)

    def log_likelihood(self, x=None, y=None):
        """log p(y | x, theta), shape [1] (Rasmussen & Williams alg. 2.1; gptorch/models/gpr.py:47-67).

        With a stationary kernel and the Gaussian likelihood the whole evaluation is one fused native node
        (covariance build -> Cholesky -> solve -> log-det, analytic backward); Sum / Product trees of native leaves
        (and a bare Linear) use the composite form of the same node.  Kernels with user-defined leaves go through the
        reference's step-by-step form on the native primitives.
        """
        x = x if x is not None else self.X
        y = y if y is not None else self.Y
        if x.shape[0] != y.shape[0]:
            raise ValueError("X and Y must have same # data.")
        n, dy = y.shape
        resid = y - self.mean_function(x)
        kind = _native_kind(self.kernel)
        if kind is not None and isinstance(self.likelihood, Gaussian):
            return ag.GPRLogLikFn.apply(kind, x, resid, self.kernel.length_scales.transform(),
                                        self.kernel.variance.transform(), self.likelihood.variance.transform())
        terms = kernels.sum_of_products(self.kernel) if isinstance(self.likelihood, Gaussian) else None
        if terms is not None:
            spec, params = kernels.composite_spec(terms)
            return ag.GPRCompositeLogLikFn.apply(spec, x.to(torch.float64), resid, self.likelihood.variance.transform(),
                                                 *params)
        L = cholesky(self._compute_kyy(x=x))
        alpha = trtrs(resid, L)
        red_logdet = ag.LogDetFn.apply(L)
        const = -0.5 * dy * n * torch.log(torch.tensor(2.0 * torch.pi, dtype=alpha.dtype, device=alpha.device))
        return (-0.5 * alpha.pow(2).sum() - dy * red_logdet + const).reshape(1)

    def _compute_kyy(self, x=None):
        """K(x, x) + noise * I (gptorch/models/gpr.py:69-86)."""
        x = x if x is not None else self.X
        kind = _native_kind(self.kernel)
        noise = self.likelihood.variance.transform()
        if kind is not None:
            return ag.KernelFn.apply(kind, x.to(torch.float64), None, self.kernel.length_scales.transform(),
                                     self.kernel.variance.transform(), noise)
        terms = kernels.sum_of_products(self.kernel)
        if terms is not None:
            spec, params = kernels.composite_spec(terms)
            return ag.CompositeKernelFn.apply(spec, x.to(torch.float64), None, noise, *params)
        n = x.shape[0]
        return self.kernel.K(x) + noise * torch.eye(n, dtype=x.dtype, device=x.device)

    def _factor(self, x):
        """L = chol(Ky) and V = L^-1 (Y - m(x)).

        The reference re-factorises on every _predict call (gptorch/models/gpr.py:104).  Under torch.no_grad() the
        factor is cached and reused while parameters and data are unchanged (SURVEY 8f row 1, GPModel._memo); with
        autograd enabled it is recomputed so that predictions stay differentiable exactly as in the reference.
        """
        def compute():
            L = cholesky(self._compute_kyy(x=x))
            return L, trtrs(self.Y - self.mean_function(x), L)

        return self._memo("factor", x, compute)

    def _predict(self, x_new, diag=True, x=None):
        """p(f* | y): mean [n*, dy] and variance [n*, dy] (diag) or covariance [n*, n*]
        (gptorch/models/gpr.py:88-117)."""
        x = x if x is not None else self.X
        k_sy = self.kernel.K(x_new, x)                       # [n*, n]
        L, V = self._factor(x)
        At = trtrs(k_sy.t(), L).t()                          # (L^-1 k_ys)^T, solved on the row panel k_sy L^-T
        mean_f = mm(At, V) + self.mean_function(x_new)
        if diag:
            var_f = (self.kernel.Kdiag(x_new) - ag.RowSumSqFn.apply(At))[:, None].expand_as(mean_f)   # fused Kdiag - colsum(A^2)
        else:
            var_f = self.kernel.K(x_new) - mm_nt(At, At)
        return mean_f, var_f

    def posterior(self):
        """A GPRPosterior: p(f* | y) for the current parameters and data, factorised once.

        Its predictions differentiate with respect to the test inputs only, and repeated calls reuse the factorisation
        (predict_f with autograd enabled refactorises on every call).  It is a snapshot: changing a parameter or the
        data afterwards does not change it -- call posterior() again."""
        with torch.no_grad():
            X = self.X.detach().clone()
            kernel, mean_function, likelihood = (_frozen(m) for m in (self.kernel, self.mean_function, self.likelihood))
            L = cholesky(self._compute_kyy(x=X))
            V = trtrs(self.Y - self.mean_function(X), L)
            if _native_kind(kernel) is None:
                return GPRPosterior(kernel, mean_function, likelihood, X, L=L, V=V)
            dinv = ag._dinv_of(L)
            a = V.contiguous().clone()
            nv.trsv_(L, dinv, a, True)                               # a = Ky^-1 (y - m(X))
            kd = nv.potri_(L, L.stride(0), dinv)                     # blocked Ky^-1, in place over L
            Kinv = nv.potri_assemble(L, L.stride(0), kd)
            del L, kd
            return GPRPosterior(kernel, mean_function, likelihood, X, Kinv=Kinv, a=a)


def _frozen(module):
    """A copy of `module` whose parameters hold the same raw values and transforms and require no gradient."""
    snap = copy.deepcopy(module)
    for p, q in zip(module.parameters(), snap.parameters()):
        if isinstance(p, Param):
            q._transform, q.prior = p._transform, p.prior   # torch's Parameter deepcopy keeps neither
        q.requires_grad_(False)
    return snap


class GPRPosterior:
    """p(f* | y) of a GPR model with its factorisation computed once (GPR.posterior()).

    Holds a snapshot of the training inputs, of the kernel, mean function and likelihood (their parameters detached),
    and of the factorisation: for a stationary kernel with a native family, the full symmetric Ky^-1 and
    a = Ky^-1 (y - m(X)); for any other kernel (Sum / Product trees, Linear, user-defined), the Cholesky factor L and
    L^-1 (y - m(X)).  Changing the model's parameters or data afterwards does not change the posterior; call
    GPR.posterior() again for the new state.

    predict_f / predict_y / predict_f_samples have the shapes and the input conventions (numpy in, numpy out; tensors
    on any device) of the model's methods.  Their results differentiate with respect to the test inputs x* and
    nothing else: no parameter of the model receives a .grad from them.  A call costs O(n* N^2), not O(N^3).
    """

    def __init__(self, kernel, mean_function, likelihood, X, Kinv=None, a=None, L=None, V=None):
        if (Kinv is None) == (L is None) or (Kinv is None) != (a is None) or (L is None) != (V is None):
            raise ValueError("GPRPosterior needs either (Kinv, a) or (L, V)")
        self.kernel, self.mean_function, self.likelihood = kernel, mean_function, likelihood
        self.X = X
        self.Kinv, self.a, self.L, self.V = Kinv, a, L, V
        self._kind = _native_kind(kernel) if Kinv is not None else None
        if Kinv is not None and self._kind is None:
            raise ValueError("the cached Ky^-1 form needs a stationary kernel with a native family")

    @property
    def compute_device(self):
        return self.X.device

    def _check(self, x_new):
        if x_new.dim() != 2 or x_new.shape[1] != self.X.shape[1]:
            raise ValueError("test inputs must be [n*, %d], got %s" % (self.X.shape[1], tuple(x_new.shape)))
        return x_new if x_new.dtype == torch_dtype else x_new.to(torch_dtype)

    def _predict(self, x_new, diag=True):
        """(mean [n*, dy], variance [n*, dy]) if diag else (mean, covariance [n*, n*])."""
        x_new = self._check(x_new)
        X = self.X
        if self._kind is not None:
            ell, s2 = self.kernel.length_scales.transform(), self.kernel.variance.transform()
            if diag:
                mean_f, var_f = ag.GPRPredFn.apply(self._kind, x_new, X, self.a, self.Kinv, ell, s2)
            else:
                k_sy = ag.KernelFn.apply(self._kind, x_new, X, ell, s2)
                mean_f = mm(k_sy, self.a)
                var_f = ag.KernelFn.apply(self._kind, x_new, None, ell, s2) - mm_nt(mm(k_sy, self.Kinv), k_sy)
            return mean_f + self.mean_function(x_new), var_f
        k_sy = self.kernel.K(x_new, X)
        At = trtrs(k_sy.t(), self.L).t()
        mean_f = mm(At, self.V) + self.mean_function(x_new)
        if diag:
            var_f = (self.kernel.Kdiag(x_new) - ag.RowSumSqFn.apply(At))[:, None].expand_as(mean_f)
        else:
            var_f = self.kernel.K(x_new) - mm_nt(At, At)
        return mean_f, var_f

    @input_as_tensor
    def predict_f(self, input_new, diag=True):
        """p(f* | y) at the test inputs: (mean [n*, dy], variance [n*, dy]) if diag else (mean, covariance [n*, n*]).
        Differentiable with respect to input_new only; the posterior's parameters receive no gradient."""
        return self._predict(input_new, diag=diag)

    @input_as_tensor
    def predict_y(self, input_new, diag=True):
        """p(y* | y): predict_f plus the likelihood's noise.  Differentiable with respect to input_new only."""
        mean_f, cov_f = self._predict(input_new, diag=diag)
        if diag:
            return self.likelihood.predict_mean_variance(mean_f, cov_f)
        return self.likelihood.predict_mean_covariance(mean_f, cov_f)

    @input_as_tensor
    def predict_f_samples(self, input_new, n_samples=1):
        """[n_samples, n*, dy] draws from p(f* | y) (full covariance).  Differentiable with respect to input_new only."""
        mu, sigma = self._predict(input_new, diag=False)
        return GPModel._sample(self, mu, sigma, n_samples)
