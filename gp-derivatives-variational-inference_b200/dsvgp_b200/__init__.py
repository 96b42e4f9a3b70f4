"""dsvgp_b200 -- B200-native DSVGP minibatch train / predict hot path behind the reference's Python API.

Importing this package loads libdsvgp_b200.so (hand-written sm_100a CUDA kernels, C ABI in include/dsvgp_b200.h).
There is no CPU, PyTorch-eager or oracle fallback: a missing library raises at import, a non-CUDA tensor raises
at call time.
"""
from . import _lib, ops  # noqa: F401  (fails loudly if the extension is missing)
from .engine import ENGINE, NanError, NotPSDError
from .optim import FusedAdam
from .gp import (ApproximateGP, CholeskyVariationalDistribution, ConstantMean, DFreeDirectionalGradVariationalStrategy,
                 DirectionalGradVariationalStrategy, GaussianLikelihood, GradVariationalStrategy, MultivariateNormal, NGD, NaturalVariationalDistribution,
                 PredictiveDistribution, PredictiveLogLikelihood, RBFKernel, RBFKernelDirectionalGrad, RBFKernelGrad, ScaleKernel,
                 VariationalELBO, VariationalStrategy)

__all__ = ["ENGINE", "NanError", "NotPSDError", "ApproximateGP", "CholeskyVariationalDistribution", "ConstantMean",
           "DFreeDirectionalGradVariationalStrategy", "DirectionalGradVariationalStrategy", "FusedAdam", "GaussianLikelihood",
           "GradVariationalStrategy", "MultivariateNormal", "NGD", "NaturalVariationalDistribution", "PredictiveDistribution", "PredictiveLogLikelihood",
           "RBFKernel", "RBFKernelDirectionalGrad", "RBFKernelGrad", "ScaleKernel", "VariationalELBO", "VariationalStrategy"]
__version__ = "0.1.0"
