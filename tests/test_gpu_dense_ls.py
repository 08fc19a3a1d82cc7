"""Dense least squares of 256..4095 columns: the blocked Householder QR of csrc/dense_qr.cu (gnk_dense_qr_ls) at the
kernel level against LAPACK, and gauss_newton with dense Jacobians of that width -- host and device callables -- against
the oracle (LAPACK lstsq) computed at test time."""
import numpy as np
import pytest
import scipy.linalg

from golden_util import rel
from oracle import gnk_oracle as orc

TOL = 1e-10


@pytest.fixture(scope="module")
def g():
    import gauss_newton_via_generalized_krylov_subspaces_b200 as pkg
    import gauss_newton_via_generalized_krylov_subspaces_b200.device as device
    device._runtime = None
    pkg.get_runtime()
    return pkg


def _raw_dense(g, A, y, sign, lda=None):
    """gnk_dense_qr_ls on the panel [A | y] with column stride lda -> (rc, the 2p + 4 result doubles)"""
    import torch
    from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib
    rt = g.get_runtime()
    n, p = A.shape
    lda = lda or (n + 15) // 16 * 16
    M = np.zeros((p + 1, lda))
    M[:p, :n] = A.T
    M[p, :n] = y
    dA = torch.from_numpy(M.reshape(-1)).to(rt.device)
    out = rt.zeros(2 * p + 8)
    rc = rt.lib.gnk_dense_qr_ls(rt.ctx, dA.data_ptr(), lda, n, p, float(sign), out.data_ptr(), rt.stream)
    if rc != 0:
        raise _lib.GnkError(rt.lib.gnk_last_error().decode())
    return out[:2 * p + 4].cpu().numpy()


def _panel(n, p, seed):
    rs = np.random.RandomState(seed)
    A = rs.normal(size=(n, p)) @ (np.eye(p) + 0.3 * rs.normal(size=(p, p)) / np.sqrt(p))
    return A, rs.normal(size=n)


def _reference(A, y):
    """LAPACK on the panel once: the solution for sign 1, |diag R| and the condition number"""
    x = scipy.linalg.lstsq(A, y, lapack_driver="gelsy", check_finite=False)[0]
    R = scipy.linalg.qr(A, mode="r", check_finite=False)[0]
    s = np.linalg.svd(R[:A.shape[1]], compute_uv=False)
    return x, np.abs(np.diag(R)), s[0] / s[-1]


def _check_block(v, A, y, sign, ref):
    """the bounds of test_gpu_wide_ls._check_block, with the LAPACK side computed once for all signs"""
    x1, rdiag, cond = ref
    n, p = A.shape
    assert rel(v[:p], x1 / sign) <= 1e-13 * max(cond, 10.0), (rel(v[:p], x1 / sign), cond)
    Ad = sign * (A @ v[:p])
    assert abs(v[p] - Ad @ Ad) <= 1e-10 * (Ad @ Ad)
    assert abs(v[p + 1] - np.sum((y - Ad) ** 2)) <= 1e-10 * (y @ y)
    assert v[p + 2] == 0
    assert abs(v[p + 3] - v[:p] @ v[:p]) <= 1e-12 * (v[:p] @ v[:p])
    assert np.allclose(np.abs(v[p + 4:2 * p + 4]), abs(sign) * rdiag, rtol=1e-10, atol=0)


@pytest.mark.gpu
@pytest.mark.parametrize("n,p,lda_pad", [(256, 256, 0), (1000, 256, 0), (40001, 300, 2), (20000, 1000, 0),
                                         (65536, 511, 0), (8192, 4095, 0)])
def test_dense_qr_against_lapack(g, n, p, lda_pad):
    """every entry of the result block against LAPACK, signs 1, -1 and 0.5; a square panel, odd row counts, an odd lda,
    a partial last panel (300, 511, 1000, 4095 columns) and the widest panel"""
    A, y = _panel(n, p, n + p)
    ref = _reference(A, y)
    lda = n + lda_pad if lda_pad else None
    for sign in (1.0, -1.0, 0.5):
        _check_block(_raw_dense(g, A, y, sign, lda=lda), A, y, sign, ref)


@pytest.mark.gpu
def test_dense_qr_graded_columns(g):
    """columns graded over eight decades (cond ~ 1e8): the forward error stays at eps * cond"""
    n, p = 40000, 300
    A, y = _panel(n, p, 7)
    A = A * np.logspace(0, -8, p)[None, :]
    cond = np.linalg.cond(A)
    v = _raw_dense(g, A, y, 1.0)
    xr = np.linalg.lstsq(A, y, rcond=None)[0]
    assert rel(v[:p], xr) <= 1e-13 * cond, (rel(v[:p], xr), cond)


@pytest.mark.gpu
def test_dense_qr_rank_deficient(g):
    """an exactly zero column gives an exact zero on diag(R); a zero and a duplicated column each count once"""
    n, p = 20000, 300
    for case in ("zero", "equal"):
        A, y = _panel(n, p, 3)
        if case == "zero":
            A[:, 150] = 0.0
        else:
            A[:, 270] = A[:, 20]
        v = _raw_dense(g, A, y, 1.0)
        rdiag = np.diag(scipy.linalg.qr(A, mode="r")[0])
        assert v[p + 2] == np.sum(np.abs(rdiag) <= 1e-8) == 1
        if case == "zero":
            assert v[p + 4 + 150] == 0.0 and np.sum(v[p + 4:] == 0.0) == 1


@pytest.mark.gpu
def test_dense_qr_deterministic_and_scale_exact(g):
    """fixed reduction order: two calls give the same bits; a power-of-two scaling of the panel changes no rounding"""
    A, y = _panel(100000, 512, 5)
    v1, v2 = _raw_dense(g, A, y, -1.0), _raw_dense(g, A, y, -1.0)
    assert np.array_equal(v1, v2)
    v3 = _raw_dense(g, A * 2.0 ** 40, y * 2.0 ** 40, -1.0)
    assert np.array_equal(v1[:512], v3[:512])


@pytest.mark.gpu
def test_dense_qr_refuses_what_it_does_not_take(g):
    from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib
    for n, p in ((300, 255), (5000, 4096), (200, 300)):
        A, y = _panel(n, p, 1)
        with pytest.raises(_lib.GnkError):
            _raw_dense(g, A, y, 1.0)


def _smooth_fit(n, p, seed):
    rs = np.random.RandomState(seed)
    A = rs.normal(size=(n, p)) / np.sqrt(n)
    B = rs.normal(size=(n, p)) / np.sqrt(p)
    xt = rs.normal(size=p)
    y = A @ xt + 0.1 * np.sin(B @ xt) + 1e-3 * rs.normal(size=n)
    res = lambda x: A @ x + 0.1 * np.sin(B @ x) - y  # noqa: E731
    jac = lambda x: A + (0.1 * np.cos(B @ x))[:, None] * B  # noqa: E731
    return res, jac, xt + 0.5 * rs.normal(size=p), (A, B, y)


def _gn_against_oracle(g, res, jac, x0, max_iter=5, dev_res=None, dev_jac=None):
    ref_trace, our_trace = [], []
    ref = orc.gn(res, x0, jac, max_iter=max_iter, callback=lambda x, **kw: ref_trace.append(np.array(x)))
    if dev_res is None:
        out = g.gauss_newton(res, x0.copy(), jac, max_iter=max_iter,
                             callback=lambda x, **kw: our_trace.append(np.array(x)))
    else:
        import torch
        out = g.gauss_newton(dev_res, torch.from_numpy(x0.copy()).cuda(), dev_jac, max_iter=max_iter,
                             callback=lambda x, **kw: our_trace.append(x.cpu().numpy()))
    assert (out.nit, out.nrev, out.njev, bool(out.success)) == (ref["nit"], ref["nfev"], ref["njev"], ref["success"])
    dev = [rel(a, b) for a, b in zip(our_trace, ref_trace)]
    print(f"deviation per iteration ({len(dev)}):", " ".join(f"{d:.1e}" for d in dev))
    assert len(dev) == len(ref_trace) and max(dev) < TOL
    return out, ref


@pytest.mark.gpu
@pytest.mark.parametrize("n,p", [(40000, 300), (60000, 1000)])
def test_gauss_newton_dense_jacobian_host(g, n, p):
    """host callables with a dense ndarray Jacobian of 300 / 1000 columns: gnk_dense_qr_ls every step, against
    oracle.gn -- counters equal, iterates within 1e-10"""
    res, jac, x0, _ = _smooth_fit(n, p, 1)
    calls = []
    rt = g.get_runtime()
    real = rt.lib.gnk_dense_qr_ls

    def spy(*a):
        calls.append(a[4])
        return real(*a)

    rt.lib.gnk_dense_qr_ls = spy
    try:
        out, _ = _gn_against_oracle(g, res, jac, x0)
    finally:
        rt.lib.gnk_dense_qr_ls = real
    assert calls == [p] * out.njev


@pytest.mark.gpu
def test_gauss_newton_dense_jacobian_device_callables(g, monkeypatch):
    """torch res and a dense torch jac with 512 parameters against oracle.gn on the numpy twin: same counters, iterates
    within 1e-10, x comes back as a CUDA tensor, and no CSR form of J is ever built"""
    import torch
    import gauss_newton_via_generalized_krylov_subspaces_b200.device as device
    n, p = 40000, 512
    res, jac, x0, (A, B, y) = _smooth_fit(n, p, 2)
    At, Bt, yt = (torch.from_numpy(a).cuda() for a in (A, B, y))
    dres = lambda x: At @ x + 0.1 * torch.sin(Bt @ x) - yt  # noqa: E731
    djac = lambda x: At + (0.1 * torch.cos(Bt @ x))[:, None] * Bt  # noqa: E731

    def no_csr(*a, **k):
        raise AssertionError("a CSR form of the dense Jacobian was built")

    monkeypatch.setattr(device, "device_csr", no_csr)
    monkeypatch.setattr(device, "CsrPattern", no_csr)
    out, _ = _gn_against_oracle(g, res, jac, x0, dev_res=dres, dev_jac=djac)
    assert isinstance(out.x, torch.Tensor) and out.x.is_cuda


@pytest.mark.gpu
def test_dense_range_boundary(g):
    """p = 255 is still solved by gnk_tsqr_ls and p = 256 by gnk_dense_qr_ls; both steps match LAPACK lstsq"""
    rt = g.get_runtime()
    for p, used, other in ((255, "gnk_tsqr_ls", "gnk_dense_qr_ls"), (256, "gnk_dense_qr_ls", "gnk_tsqr_ls")):
        res, jac, x0, _ = _smooth_fit(20000, p, 4)
        calls = {used: 0, other: 0}
        real = {name: getattr(rt.lib, name) for name in calls}

        def wrap(name):
            def f(*a):
                calls[name] += 1
                return real[name](*a)
            return f

        for name in calls:
            setattr(rt.lib, name, wrap(name))
        try:
            _gn_against_oracle(g, res, jac, x0, max_iter=2)
        finally:
            for name in calls:
                setattr(rt.lib, name, real[name])
        assert calls[used] >= 1 and calls[other] == 0, (p, calls)


@pytest.mark.gpu
def test_gauss_newton_dense_errors(g):
    """p = 4096 is beyond the range (GnkError); fewer residuals than parameters, and a zero column, are rank deficient"""
    from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib
    res, jac, x0, _ = _smooth_fit(5000, 4096, 1)
    with pytest.raises(_lib.GnkError, match="4095"):
        g.gauss_newton(res, x0, jac, max_iter=3)
    res, jac, x0, _ = _smooth_fit(200, 300, 1)
    with pytest.raises(np.linalg.LinAlgError, match="rank deficient"):
        g.gauss_newton(res, x0, jac, max_iter=3)
    res, jac, x0, _ = _smooth_fit(20000, 300, 1)

    def jac0(x):
        J = jac(x)
        J[:, 17] = 0.0
        return J

    with pytest.raises(np.linalg.LinAlgError, match="rank deficient"):
        g.gauss_newton(res, x0, jac0, max_iter=3)
