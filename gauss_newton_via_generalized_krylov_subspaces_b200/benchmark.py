"""Experiment harness -- mirror of the reference's ``benchmark.py``: collects error / loss / nfev / cg_iter per
callback for any solver with the uniform signature ``method(res, x0, jac, args=, callback=, **kwargs)``."""
from typing import List

import numpy as np

from .armijo_goldstein import StepLengthConvergenceError


def ref_method(res, x0, jac, args, callback, **kwargs):
    """the comparison curve of the reference (benchmark.py:7-11): scipy.optimize.least_squares, a host algorithm.  A
    device-native Jacobian (the matrix-free stencil operator) is handed to scipy as the assembled CSR matrix."""
    import scipy.optimize

    def cb_scipy(intermediate_result):
        callback(intermediate_result.x, intermediate_result.nfev, None)

    def jac_host(x, *a):
        J = jac(x, *a)
        return J.tocsr() if hasattr(J, "_gnk_sparse_like") else J

    scipy.optimize.least_squares(res, x0, jac_host, callback=cb_scipy, args=args)


def reverse_accumulation(nfev_list: List[int]) -> List[int]:
    """callbacks report the accumulated count of residual evaluations; return the per-step counts."""
    return [b - a for a, b in zip([0] + list(nfev_list[:-1]), nfev_list)]


def benchmark_method(method, res, x0, jac, error, args=(), kwargs={}):
    # a device-native residual evaluates the loss without a host round trip of the residual vector
    if hasattr(res, "loss") and not args:
        loss = res.loss
    else:
        def loss(x):
            r = res(x, *args)
            if hasattr(r, "is_cuda"):  # device callables: a torch tensor, reduced where it lives
                return 0.5 * float((r.double() ** 2).sum())
            return 0.5 * np.sum(np.asarray(r) ** 2)

    error_list = [error(x0)]
    loss_list = [loss(x0)]
    nfev_list = []
    cg_iter_list = []

    def callback(x, nfev, cg_iter):
        error_list.append(error(x))
        loss_list.append(loss(x))
        if nfev is not None:
            nfev_list.append(nfev)
        if cg_iter is not None:
            cg_iter_list.append(cg_iter)

    try:
        method(res, x0, jac, args=args, callback=callback, **kwargs)
    except StepLengthConvergenceError as e:
        print("Warning:", e.message)

    return error_list, loss_list, reverse_accumulation(nfev_list), cg_iter_list
