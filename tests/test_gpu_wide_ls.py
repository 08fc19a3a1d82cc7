"""Least squares on panels of 105..256 columns that the single-CTA QR cannot take (more than 2^22 doubles, or several
ranks): the blocked Householder TSQR of csrc/tsqr.cu (wide_tsqr_kernel), at the kernel level against LAPACK and at
the solver level against the oracle (LAPACK QR / lstsq) computed at test time."""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest
import scipy.linalg

from golden_util import rel
from oracle import gnk_oracle as orc

TOL = 1e-10
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def g():
    import gauss_newton_via_generalized_krylov_subspaces_b200 as pkg
    import gauss_newton_via_generalized_krylov_subspaces_b200.device as device
    device._runtime = None
    pkg.get_runtime()
    return pkg


def _raw_ls(g, A, y, sign, lda=None, y_off=0):
    """gnk_tsqr_ls on a host panel with column stride lda and y at an offset of y_off doubles; the 2k+4 result doubles"""
    from gauss_newton_via_generalized_krylov_subspaces_b200.gauss_newton_krylow import tsqr_solve
    rt = g.get_runtime()
    n, k = A.shape
    lda = lda or (n + 15) // 16 * 16
    dA = rt.zeros(lda * k)
    for j in range(k):
        rt.upload(np.ascontiguousarray(A[:, j]), dA[j * lda:j * lda + n])
    dy = rt.zeros(n + y_off)
    rt.upload(y, dy[y_off:y_off + n])
    out = rt.zeros(2 * 256 + 8)
    tsqr_solve(rt, dA, lda, n, k, dy[y_off:], sign, out)
    return rt.read(out, 2 * k + 4).copy()


def _panel(n, k, seed):
    rs = np.random.RandomState(seed)
    A = rs.normal(size=(n, k)) @ (np.eye(k) + 0.3 * rs.normal(size=(k, k)) / np.sqrt(k))
    return A, rs.normal(size=n)


def _check_block(v, A, y, sign, cond):
    n, k = A.shape
    xr = np.linalg.lstsq(sign * A, y, rcond=None)[0]
    assert rel(v[:k], xr) <= 1e-13 * max(cond, 10.0), (rel(v[:k], xr), cond)
    Ad = sign * (A @ v[:k])
    assert abs(v[k] - Ad @ Ad) <= 1e-10 * (Ad @ Ad)
    assert abs(v[k + 1] - np.sum((y - Ad) ** 2)) <= 1e-10 * (y @ y)
    assert v[k + 2] == 0
    assert abs(v[k + 3] - v[:k] @ v[:k]) <= 1e-12 * (v[:k] @ v[:k])
    rdiag = np.abs(np.diag(scipy.linalg.qr(sign * A, mode="r", check_finite=False)[0]))
    assert np.allclose(np.abs(v[k + 4:2 * k + 4]), rdiag, rtol=1e-10, atol=0)


@pytest.mark.gpu
@pytest.mark.parametrize("n,k,lda_pad,y_off", [(40000, 104, 0, 0), (16385, 255, 0, 0), (65536, 160, 0, 0),
                                               (1 << 20, 200, 0, 0), (40001, 129, 7, 1)])
def test_wide_tsqr_against_lapack(g, n, k, lda_pad, y_off):
    """panels above 2^22 doubles: every result entry against LAPACK; odd row counts, odd lda (8-byte aligned
    columns) and an 8-byte offset y; signs +-1 and 0.5"""
    A, y = _panel(n, k, n + k)
    cond = np.linalg.cond(A)
    lda = n + lda_pad if lda_pad else None
    for sign in (1.0, -1.0, 0.5):
        _check_block(_raw_ls(g, A, y, sign, lda=lda, y_off=y_off), A, y, sign, cond)


@pytest.mark.gpu
def test_wide_tsqr_graded_columns():
    """columns graded over eight decades (cond ~ 1e8): the forward error stays at eps * cond"""
    import gauss_newton_via_generalized_krylov_subspaces_b200 as g
    n, k = 40000, 150
    A, y = _panel(n, k, 7)
    A = A * np.logspace(0, -8, k)[None, :]
    cond = np.linalg.cond(A)
    v = _raw_ls(g, A, y, 1.0)
    xr = np.linalg.lstsq(A, y, rcond=None)[0]
    assert rel(v[:k], xr) <= 1e-13 * cond, (rel(v[:k], xr), cond)


@pytest.mark.gpu
def test_wide_tsqr_rank_deficient(g, capsys):
    """an exactly zero column and two equal columns: the count of |R_jj| <= 1e-8 equals LAPACK's, and the rank report
    of the solvers (_report_rank) raises scipy's LinAlgError exactly where solve_triangular would (an exactly zero
    pivot)"""
    from gauss_newton_via_generalized_krylov_subspaces_b200.gauss_newton_krylow import _report_rank
    n, k = 40000, 120
    for case in ("zero", "equal"):
        A, y = _panel(n, k, 3)
        if case == "zero":
            A[:, 50] = 0.0
        else:
            A[:, 70] = A[:, 20]
        rdiag = np.diag(scipy.linalg.qr(A, mode="r")[0])
        v = _raw_ls(g, A, y, 1.0)
        assert v[k + 2] == np.sum(np.abs(rdiag) <= 1e-8) == 1
        assert np.array_equal(v[k + 4:] == 0.0, rdiag == 0.0)
        capsys.readouterr()
        if np.any(rdiag == 0.0):
            with pytest.raises(np.linalg.LinAlgError):
                _report_rank(v, k)
        else:
            _report_rank(v, k)
        assert capsys.readouterr().out.count("A is rank deficient") == 1


@pytest.mark.gpu
def test_wide_tsqr_deterministic_and_scale_exact(g):
    """fixed reduction order: two calls give the same bits; a power-of-two scaling of the panel changes no rounding"""
    A, y = _panel(100000, 200, 5)
    v1, v2 = _raw_ls(g, A, y, -1.0), _raw_ls(g, A, y, -1.0)
    assert np.array_equal(v1, v2)
    v3 = _raw_ls(g, A * 2.0 ** 40, y * 2.0 ** 40, -1.0)
    assert np.array_equal(v1[:200], v3[:200])


def _bratu_trace(g, G, restart, max_iter):
    o = orc.BratuOracle(G, 5, 10)
    y, u0 = o.operator(o.u_true), o.start_vector(seed=42)
    idx = np.random.RandomState(0).choice(o.n, 64, replace=False)
    ref_trace, our_trace = [], []
    ref = orc.gnk(o.make_res(y), u0, o.make_jac(), restart=restart, max_iter=max_iter,
                  callback=lambda x, **kw: ref_trace.append(np.asarray(x)[idx].copy()))
    pb = g.BratuPdeProblem(G, 5, 10)
    out = g.gauss_newton_krylow(pb.make_res(y), u0, pb.make_jac(), krylow_restart=restart, max_iter=max_iter,
                                callback=lambda x, **kw: our_trace.append(np.asarray(x)[idx].copy()))
    assert len(our_trace) == len(ref_trace)
    dev = [float(np.max(np.abs(a - b)) / np.max(np.abs(b))) for a, b in zip(our_trace, ref_trace)]
    print(f"G={G} restart={restart}: deviation per iteration:", " ".join(f"{d:.1e}" for d in dev))
    return out, ref, dev


@pytest.mark.gpu
def test_bratu_257_no_restart_200_iterations(g):
    """Bratu 257^2 (65025 interior rows) without a restart: from outer iteration 104 on the panel has 105..200 columns
    and 6.8e6..1.3e7 doubles, which only the blocked TSQR takes.  Iterations 1..103 run on the existing paths and carry
    the early-iteration cancellation of DESIGN.md section 5 (1e-8); the wide-panel iterations are held to 1e-10."""
    out, ref, dev = _bratu_trace(g, 257, None, 200)
    assert (out.nit, out.nrev, out.njev, bool(out.success)) == (199, 200, 200, False)
    assert (out.nit, out.nrev, out.njev) == (ref["nit"], ref["nfev"], ref["njev"])
    assert max(dev[103:]) < TOL, max(dev[103:])
    assert max(dev[:103]) < 1e-8
    assert rel(out.x, ref["x"]) < 1e-9


@pytest.mark.gpu
def test_bratu_257_restart_after_wide_panels(g):
    """krylow_restart=130: panels of 105..130 columns on the blocked TSQR, then a restart (post-restart bar 1e-8)"""
    out, ref, dev = _bratu_trace(g, 257, 130, 140)
    assert (out.nit, out.nrev, out.njev) == (ref["nit"], ref["nfev"], ref["njev"]) == (139, 140, 140)
    assert max(dev[103:129]) < TOL, max(dev[103:129])
    assert max(dev) < 1e-8


def _smooth_fit(n, p, seed):
    rs = np.random.RandomState(seed)
    A = rs.normal(size=(n, p)) / np.sqrt(n)
    B = rs.normal(size=(n, p)) / np.sqrt(p)
    xt = rs.normal(size=p)
    y = A @ xt + 0.1 * np.sin(B @ xt) + 1e-3 * rs.normal(size=n)
    res = lambda x: A @ x + 0.1 * np.sin(B @ x) - y  # noqa: E731
    jac = lambda x: A + (0.1 * np.cos(B @ x))[:, None] * B  # noqa: E731
    return res, jac, xt + 0.5 * rs.normal(size=p), A


@pytest.mark.gpu
def test_gauss_newton_dense_jacobian_150_parameters(g):
    """gauss_newton with a host dense Jacobian of 40000 x 150 (6.0e6 doubles): every step's least squares on the blocked
    TSQR, against oracle.gn (LAPACK lstsq) -- counters equal, iterates within 1e-10.  max_iter=5 stops after the fourth
    step, whose Armijo decrease is still 3.5e-12 of ||r||^2; the fifth is at rounding level (||J d||^2 / ||r||^2 ~ 1e-20),
    where even two LAPACK builds take different numbers of trials."""
    res, jac, x0, A = _smooth_fit(40000, 150, 1)
    ref_trace, our_trace = [], []
    ref = orc.gn(res, x0, jac, max_iter=5, callback=lambda x, **kw: ref_trace.append(np.array(x)))
    out = g.gauss_newton(res, x0.copy(), jac, max_iter=5, callback=lambda x, **kw: our_trace.append(np.array(x)))
    assert (out.nit, out.nrev, out.njev) == (4, 5, 4)
    assert (out.nit, out.nrev, out.njev, bool(out.success)) == (ref["nit"], ref["nfev"], ref["njev"], ref["success"])
    dev = [rel(a, b) for a, b in zip(our_trace, ref_trace)]
    print("gauss_newton 40000 x 150, deviation per iteration:", " ".join(f"{d:.1e}" for d in dev))
    assert len(dev) == len(ref_trace) and max(dev) < TOL


def test_library_holds_the_wide_tsqr_kernels():
    """the shipped .so carries the blocked TSQR kernels, with their compact-WY products on the FP64 tensor pipe"""
    import __graft_entry__
    __graft_entry__.build()
    from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib
    if not shutil.which("cuobjdump"):
        pytest.skip("cuobjdump is not installed")
    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    funcs = {f.split("\n", 1)[0].strip(): f for f in sass.split("Function : ")[1:]}
    wide = [body for name, body in funcs.items() if "wide_tsqr_kernel" in name]
    assert len(wide) == 1
    assert wide[0].count("DMMA.8x8x4") >= 4 * 8   # G = U^T U, U^T C, T^T W and U W, unrolled
    assert any("wide_solve_kernel" in name for name in funcs)


def _gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.gpu
@pytest.mark.parametrize("nproc", [2, 4, 8])
def test_wide_tsqr_multi_gpu(nproc):
    """several ranks: each holds a row block of one global panel (some fewer rows than columns); every rank's result
    block equals the global lstsq and all ranks agree bit for bit (tests/wide_ls_worker.py)"""
    if _gpus() < nproc:
        pytest.skip(f"needs {nproc} GPUs")
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([ROOT, os.path.join(ROOT, "tests")]))
    cmd = [sys.executable, "-m", "torch.distributed.run", f"--nproc_per_node={nproc}",
           os.path.join(ROOT, "tests", "wide_ls_worker.py")]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=3000, cwd=ROOT)
    print(r.stdout[-4000:], r.stderr[-4000:])
    assert r.returncode == 0
    assert r.stdout.count("WIDE_LS_OK") == nproc



@pytest.mark.gpu
def test_linear_least_squares_keeps_its_range(g):
    """the host-array linear_least_squares keeps the range it always had above 104 columns (the single-CTA QR's
    2^22 doubles); the same panel goes through gnk_tsqr_ls on the device"""
    from gauss_newton_via_generalized_krylov_subspaces_b200._lib import GnkError
    A, y = _panel(40000, 110, 2)
    with pytest.raises(GnkError):
        g.linear_least_squares(A, y)
    _check_block(_raw_ls(g, A, y, 1.0), A, y, 1.0, np.linalg.cond(A))
    B, yb = A[:37000], y[:37000]                         # 37000 x 111 < 2^22 doubles: the single-CTA QR
    assert rel(g.linear_least_squares(B, yb), np.linalg.lstsq(B, yb, rcond=None)[0]) < 1e-12
