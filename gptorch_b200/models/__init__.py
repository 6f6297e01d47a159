"""Gaussian-process models (reference: gptorch/models/__init__.py): GPR (exact), VFE and SVGP (sparse)."""
from .base import GPModel
from .gpr import GPR, GPRPosterior
from .sparse_gpr import VFE, SVGP
from .dist_gpr import DistributedGPR
