"""vittles_b200 - the sensitivity hot path of rgiordan/vittles, B200-native.

Same public names as ``vittles/__init__.py:1-8``; the arithmetic runs in
hand-written sm_100a CUDA kernels behind the C ABI of
``include/vittles_b200.h``.  There is no CPU fallback.
"""
from .sensitivity_lib import \
    HyperparameterSensitivityLinearApproximation, \
    ParametricSensitivityTaylorExpansion

from .sparse_hessian_lib import SparseBlockHessian
from .lr_cov_lib import LinearResponseCovariances
from .influence_lib import ObservationInfluence, AMIPResult, ApproximateCVResult
from . import influence_lib
from . import solver_lib
from . import bivariate_sensitivity_lib
from . import objectives
from . import ops
from . import patterns

__version__ = '0.1.0'
