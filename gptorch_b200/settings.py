"""Package-wide settings (reference: gptorch/settings.py:5-7)."""
import torch
from torch.distributions.transforms import ExpTransform

# Positive hyper-parameters are stored as logs and read through exp(), so gradients are w.r.t. the logs.
DefaultPositiveTransform = ExpTransform

_device = None


def default_device():
    """Device new parameters and data are created on: the current CUDA device when there is one.

    The reference builds everything on the CPU and moves with model.cuda(); this package computes only on
    the GPU, so it starts there.  Without CUDA (e.g. the CPU test tier) objects can still be constructed and
    inspected, but any numerical call raises.
    """
    if _device is not None:
        return _device
    if torch.cuda.is_available():
        return torch.device("cuda", torch.cuda.current_device())
    return torch.device("cpu")


def set_default_device(device):
    global _device
    _device = None if device is None else torch.device(device)


# Optimiser bridge (Model._loss_and_grad): capture one loss+gradient evaluation into a CUDA graph and replay it per
# optimiser step when the model says its evaluation is static (GPModel._graphable).  Small problems are launch- and
# host-bound: the reference's own example (N = 100) costs ~15 kernel launches and ~1 ms of Python per evaluation
# eagerly, ~0.1 ms replayed.  Set to False to force eager evaluation.
cuda_graphs = True
graph_max_rows = 4096      # larger evaluations are compute-bound (and use the look-ahead side stream): eager


# VFE sufficient statistics (gptorch_b200/_autograd.py VfeStatsFn): "auto" streams Phi = Kuf Kfu and applies L^-1 . L^-T
# once (3 N M^2 flop per loss+grad instead of the reference order's 5 N M^2) when the estimated cond_2(Kuu) is at most
# vfe_phi_cond_max -- the congruence amplifies rounding by cond(Kuu); measured against the reference the hyper-parameter
# gradients deviate by <= 200 * eps * cond (tests/test_gpu_models.py), i.e. <= 1e-8 at the default bound, an order of
# magnitude inside the 1e-7 tolerance.  False = always the reference's order of operations; True = always the Phi form.
vfe_phi_form = "auto"
vfe_phi_cond_max = 2.0e5

# SVGP data term (SvgpMomentsFn): "auto" forms C = Kuu^-1 (S - Kuu) Kuu^-1 first and evaluates the batch moments with one
# panel product (3 B M^2 flop per loss+grad instead of 6 B M^2) under the same conditioning gate as the VFE Phi form, for
# batches of at least 16 M rows with the Gaussian likelihood.  False = the reference's order; True = always.
svgp_quadratic_form = "auto"


def int8_sliced_products(slices=None):
    """Slices of the FP64-equivalent int8 products that run the large O(N^3) trailing updates of the Cholesky factor
    (DESIGN.md section 8): 8 by default, 2..8 allowed, 0 = the FP64 DMMA engine.  While it is above 0 the blocked
    inverse's products run sliced too, at a fixed 9 slices (its consumers cancel, so it keeps one more); 0 returns both
    to the FP64 DMMA engine.  With an argument it sets the value for the process (and returns the previous one); without, it only
    queries.  The environment variable GPB_I8MMA sets the initial value."""
    from . import _native
    return _native.i8mma_config(-1 if slices is None else int(slices))
