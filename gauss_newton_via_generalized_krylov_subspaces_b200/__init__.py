"""B200-native Gauss-Newton-Krylov hot path with the reference's Python entry points.

    from gauss_newton_via_generalized_krylov_subspaces_b200 import (
        gauss_newton_krylow, gauss_newton, armijo_goldstein, BratuPdeProblem, RegressionResult)

The modules keep the reference's names (``gauss_newton_krylow``, ``krylow``, ``armijo_goldstein``,
``gauss_newton``, ``bratu_pde_problem``, ``rosenbrock_problem``, ``regression_result``, ``benchmark``);
``install_flat_names()`` registers them under those bare names so that the reference's own driver scripts
(``from gauss_newton_krylow import gauss_newton_krylow`` ...) run unchanged on the device path.

Importing the package needs neither a GPU nor the built library; calling a solver does (no CPU fallback).
"""
import importlib
import sys

_MODULES = ("regression_result", "armijo_goldstein", "krylow", "bratu_pde_problem", "rosenbrock_problem",
            "gauss_newton_krylow", "gauss_newton", "benchmark")

from .regression_result import RegressionResult  # noqa: E402
from .armijo_goldstein import StepLengthConvergenceError, armijo_goldstein  # noqa: E402
from .krylow import (GeneralizedKrylowSubspace, GeneralizedKrylowSubspaceBreakdown,  # noqa: E402
                     GeneralizedKrylowSubspaceSpansEntireSpace)
from .bratu_pde_problem import BratuPdeProblem, default_u  # noqa: E402
from .gauss_newton_krylow import gauss_newton_krylow, linear_least_squares  # noqa: E402
from .gauss_newton import cg_least_squares, gauss_newton  # noqa: E402
from .device import DeviceLinearOperator, DeviceVector, autograd_jacobian, get_runtime  # noqa: E402


def install_flat_names(overwrite=True):
    """Make ``import gauss_newton_krylow`` etc. resolve to this package's modules."""
    for name in _MODULES:
        if overwrite or name not in sys.modules:
            sys.modules[name] = importlib.import_module(f"{__name__}.{name}")


__all__ = ["RegressionResult", "StepLengthConvergenceError", "armijo_goldstein", "GeneralizedKrylowSubspace",
           "GeneralizedKrylowSubspaceBreakdown", "GeneralizedKrylowSubspaceSpansEntireSpace", "BratuPdeProblem",
           "default_u", "gauss_newton_krylow", "linear_least_squares", "cg_least_squares", "gauss_newton",
           "DeviceLinearOperator", "DeviceVector", "autograd_jacobian", "get_runtime", "install_flat_names"]
