"""CPU tests of the dense-Jacobian branch of gauss_newton for 256..4095 parameters (gnk_dense_qr_ls), driven through the
numpy mock of the C ABI (tests/mock_backend.py, with the numpy mirror of gnk_dense_qr_ls below attached), and a SASS
check of the kernels in the shipped library."""
import shutil
import subprocess
import types

import numpy as np
import pytest
import scipy.linalg

from golden_util import rel
from oracle import gnk_oracle as orc


def mock_dense_qr_ls(self, ctx, A, lda, n_rows, p, sign_a, out, stream):
    """numpy mirror of gnk_dense_qr_ls: the augmented panel [A | y] (p + 1 columns, stride lda) -> the result block of
    gnk_tsqr_ls, by numpy QR (like the mock's gnk_tsqr_ls); the panel is left holding R in its upper triangle (the CUDA
    kernel also stores its reflectors below it)"""
    import mock_backend
    from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib
    if not (_lib.GNK_DENSE_QR_MIN <= p <= _lib.GNK_DENSE_QR_MAX and p <= n_rows <= lda):
        return -2
    self.launches += 1
    panel = mock_backend.arr(A, lda * (p + 1)).reshape(p + 1, lda)
    M = panel[:, :n_rows].T.copy()
    M[:, :p] *= sign_a
    R = np.linalg.qr(M, mode="r")
    if R.shape[0] < p + 1:  # n_rows == p: a zero residual
        R = np.concatenate([R, np.zeros((p + 1 - R.shape[0], p + 1))])
    rr = min(n_rows, p + 1)
    panel[:, :n_rows] = 0.0
    panel[:, :rr] = R[:rr].T
    z = R[:p, p]
    try:
        d = scipy.linalg.solve_triangular(R[:p, :p], z)
    except Exception:  # exactly singular R: the CUDA kernel divides by zero and reports the zero diagonal
        d = np.full(p, np.inf)
    o = mock_backend.arr(out, 2 * p + 4)
    o[:p] = d
    o[p] = np.sum(z * z)
    o[p + 1] = R[p, p] ** 2
    o[p + 2] = np.sum(np.abs(np.diag(R)[:p]) <= 1e-8)
    o[p + 3] = np.sum(d * d)
    o[p + 4:2 * p + 4] = np.diag(R)[:p]
    return 0


@pytest.fixture()
def g():
    import mock_backend
    rt = mock_backend.install()
    rt.lib.gnk_dense_qr_ls = types.MethodType(mock_dense_qr_ls, rt.lib)
    import gauss_newton_via_generalized_krylov_subspaces_b200 as pkg
    yield pkg
    mock_backend.uninstall()


def _smooth_fit(n, p, seed):
    rs = np.random.RandomState(seed)
    A = rs.normal(size=(n, p)) / np.sqrt(n)
    B = rs.normal(size=(n, p)) / np.sqrt(p)
    xt = rs.normal(size=p)
    y = A @ xt + 0.1 * np.sin(B @ xt) + 1e-3 * rs.normal(size=n)
    res = lambda x: A @ x + 0.1 * np.sin(B @ x) - y  # noqa: E731
    jac = lambda x: A + (0.1 * np.cos(B @ x))[:, None] * B  # noqa: E731
    return res, jac, xt + 0.5 * rs.normal(size=p)


def _count_calls(rt, names):
    calls = {n: 0 for n in names}
    real = {n: getattr(rt.lib, n) for n in names}

    def wrap(name):
        def f(*a):
            calls[name] += 1
            return real[name](*a)
        return f

    for n in names:
        setattr(rt.lib, n, wrap(n))
    return calls, real


@pytest.mark.parametrize("order", ["C", "F"])
def test_host_gn_dense_300_parameters(g, order):
    """a dense 4000 x 300 Jacobian (C- or Fortran-ordered) takes gnk_dense_qr_ls every step and no CSR product: against
    oracle.gn, counters equal and iterates within 1e-10"""
    res, jac, x0 = _smooth_fit(4000, 300, 1)
    jac_o = (lambda x: np.asfortranarray(jac(x))) if order == "F" else jac
    ref_trace, our_trace = [], []
    ref = orc.gn(res, x0, jac, max_iter=5, callback=lambda x, **kw: ref_trace.append(np.array(x)))
    rt = g.get_runtime()
    calls, real = _count_calls(rt, ["gnk_dense_qr_ls", "gnk_tsqr_ls", "gnk_spmm_csr"])
    try:
        out = g.gauss_newton(res, x0.copy(), jac_o, max_iter=5, callback=lambda x, **kw: our_trace.append(np.array(x)))
    finally:
        for n, f in real.items():
            setattr(rt.lib, n, f)
    assert (out.nit, out.nrev, out.njev, bool(out.success)) == (ref["nit"], ref["nfev"], ref["njev"], ref["success"])
    assert len(our_trace) == len(ref_trace) and max(rel(a, b) for a, b in zip(our_trace, ref_trace)) < 1e-10
    assert calls == {"gnk_dense_qr_ls": out.njev, "gnk_tsqr_ls": 0, "gnk_spmm_csr": 0}


def test_host_gn_dense_255_parameters_keeps_the_tsqr_path(g):
    res, jac, x0 = _smooth_fit(2000, 255, 2)
    rt = g.get_runtime()
    calls, real = _count_calls(rt, ["gnk_dense_qr_ls", "gnk_tsqr_ls"])
    try:
        out = g.gauss_newton(res, x0.copy(), jac, max_iter=2, callback=lambda **kw: None)
    finally:
        for n, f in real.items():
            setattr(rt.lib, n, f)
    assert calls == {"gnk_dense_qr_ls": 0, "gnk_tsqr_ls": out.njev}


def test_host_gn_plugin_gets_the_users_dense_jacobian(g):
    """a step_length_control plug-in still receives the ndarray jac returned"""
    res, jac, x0 = _smooth_fit(1000, 300, 3)
    seen = []

    def plugin(res_, x, r, J, args, d):
        seen.append(type(J))
        return 1.0, res_(x + d, *args), 1

    g.gauss_newton(res, x0.copy(), jac, max_iter=2, step_length_control=plugin, callback=lambda **kw: None)
    assert seen == [np.ndarray]


def test_host_gn_dense_errors(g):
    from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib
    res, jac, x0 = _smooth_fit(4100, 4096, 1)
    with pytest.raises(_lib.GnkError, match="4095"):
        g.gauss_newton(res, x0, jac, max_iter=3)
    res, jac, x0 = _smooth_fit(200, 300, 1)
    with pytest.raises(np.linalg.LinAlgError, match="rank deficient"):
        g.gauss_newton(res, x0, jac, max_iter=3)
    res, jac, x0 = _smooth_fit(1000, 300, 1)

    def jac0(x):
        J = jac(x)
        J[:, 17] = 0.0
        return J

    with pytest.raises(np.linalg.LinAlgError, match="rank deficient"):
        g.gauss_newton(res, x0, jac0, max_iter=3)


def test_scalar_read_back_refuses_more_than_its_staging(g):
    from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib
    rt = g.get_runtime()
    t = rt.zeros(rt._pinned_np.shape[0] + 1)
    with pytest.raises(_lib.GnkError, match="staging"):
        rt.read(t)


def test_library_holds_the_dense_qr_kernels():
    """the shipped .so carries the blocked QR kernels, with V^T C, T^T W and the update on the FP64 tensor pipe"""
    import __graft_entry__
    __graft_entry__.build()
    from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib
    if not shutil.which("cuobjdump"):
        pytest.skip("cuobjdump is not installed")
    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    funcs = {f.split("\n", 1)[0].strip(): f for f in sass.split("Function : ")[1:]}

    def body(name):
        found = [b for n, b in funcs.items() if name in n]
        assert len(found) == 1, name
        return found[0]

    assert body("dqr_vtc_kernel").count("DMMA.8x8x4") >= 4 * 8   # 4 row tiles x 8 k-steps, unrolled
    assert body("dqr_tw_kernel").count("DMMA.8x8x4") >= 4 * 8
    assert body("dqr_update_kernel").count("DMMA.8x8x4") >= 8 * 8
    body("dqr_panel_kernel")
    body("dqr_solve_kernel")
