"""Dense CUDA Jacobians without a CSR form (device.py: DenseDeviceJacobian, csrc/dense_jac.cu): gnk_dense_matmat and
gnk_dense_rmatvec against gnk_spmm_csr on the CSR of the same matrix, bit for bit; gauss_newton_krylow and
gauss_newton with strided device Jacobians against the same problems handed over as torch CSR and as host ndarrays;
a jac that refills one tensor in place; and Jacobians of 2^31 entries and more, which the CSR route refused."""
import numpy as np
import pytest
import scipy.sparse as sp

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def g():
    import gauss_newton_via_generalized_krylov_subspaces_b200 as pkg
    import gauss_newton_via_generalized_krylov_subspaces_b200.device as device
    device._runtime = None
    pkg.get_runtime()
    return pkg


def _lib_ptr():
    from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib
    from gauss_newton_via_generalized_krylov_subspaces_b200.device import ptr
    return _lib, ptr


def _bits(t):
    return t.cpu().numpy().view(np.int64)


# ------------------------------------------------------------------------------------------------
# 1. kernels: bit for bit the CSR kernel on the CSR of the same matrix
# ------------------------------------------------------------------------------------------------
def _matrix(rng, n, p):
    """exact zeros, -0.0 entries, a NaN, a zero row and a zero column, magnitudes over six decades"""
    A = rng.standard_normal((n, p)) * 10.0 ** rng.integers(-3, 4, (n, p))
    A[rng.random((n, p)) < 0.3] = 0.0
    A[rng.random((n, p)) < 0.05] = -0.0
    if n > 2 and p > 2:
        A[n // 2, :] = 0.0
        A[:, p // 3] = -0.0
        A[n - 1, p - 1] = np.nan
    return A


def _layouts(torch, A, dev):
    """row-major, column-major, a row-major view with a padded row stride, a transposed view (column-major, padded)"""
    n, p = A.shape
    t = torch.as_tensor(A, device=dev)
    padded = torch.full((n, p + 3), 7.0, dtype=torch.float64, device=dev)
    padded[:, :p] = t
    tpad = torch.full((p, n + 5), 7.0, dtype=torch.float64, device=dev)
    tpad[:, :n] = t.T
    return {"row": t.contiguous(), "col": t.T.contiguous().T, "row_view": padded[:, :p], "t_view": tpad[:, :n].T}


def _strides(J):
    return tuple(1 if n == 1 else s for n, s in zip(J.shape, J.stride()))


def _csr(g, A):
    import torch
    A = sp.csr_array(A)  # drops +0.0 and -0.0, keeps NaN, like torch's to_sparse_csr
    A.sort_indices()
    dev = g.get_runtime().device
    return [torch.as_tensor(a, device=dev) for a in (A.indptr.astype(np.int32), A.indices.astype(np.int32),
                                                     A.data.astype(np.float64))]


@gpu
@pytest.mark.parametrize("n,p", [(1, 1), (1, 37), (53, 1), (300, 300), (1001, 77), (45, 700), (517, 129)])
def test_dense_kernels_equal_the_csr_kernel_bitwise(g, n, p):
    import torch
    _lib, ptr = _lib_ptr()
    rt = g.get_runtime()
    rng = np.random.default_rng(n * 1000 + p)
    A = _matrix(rng, n, p)
    rp, ci, va = _csr(g, A)
    rpt, cit, vat = _csr(g, A.T)
    for k in (1, 7, 8, 9, 33, 64, 255):
        in_ld, in_off, out_ld, out_off = p + 5, 3, n + 7, 2
        V = torch.as_tensor(rng.standard_normal(in_ld * k + in_off), device=rt.device)
        ref = torch.full((out_ld * k + out_off,), 3.0, dtype=torch.float64, device=rt.device)
        for sign in (1.0, -1.0, 0.5):
            _lib.check(rt.lib.gnk_spmm_csr(rt.ctx, n, ptr(rp), ptr(ci), ptr(va), ptr(V), in_ld, in_off, k, sign,
                                           ptr(ref), out_ld, out_off, rt.stream), "gnk_spmm_csr")
            for name, J in _layouts(torch, A, rt.device).items():
                out = torch.full_like(ref, 3.0)
                rs, cs = _strides(J)
                _lib.check(rt.lib.gnk_dense_matmat(rt.ctx, n, p, ptr(J), rs, cs, ptr(V), in_ld, in_off, k, sign,
                                                   ptr(out), out_ld, out_off, rt.stream), "gnk_dense_matmat")
                assert np.array_equal(_bits(out), _bits(ref)), (name, k, sign)
    r = torch.as_tensor(rng.standard_normal(n), device=rt.device)
    for sign in (1.0, -1.0, 0.5):
        ref = torch.zeros(p, dtype=torch.float64, device=rt.device)
        _lib.check(rt.lib.gnk_spmm_csr(rt.ctx, p, ptr(rpt), ptr(cit), ptr(vat), ptr(r), 0, 0, 1, sign, ptr(ref), 0, 0,
                                       rt.stream), "gnk_spmm_csr(T)")
        for name, J in _layouts(torch, A, rt.device).items():
            out = torch.full_like(ref, 3.0)
            rs, cs = _strides(J)
            _lib.check(rt.lib.gnk_dense_rmatvec(rt.ctx, n, p, ptr(J), rs, cs, ptr(r), sign, ptr(out), rt.stream),
                       "gnk_dense_rmatvec")
            assert np.array_equal(_bits(out), _bits(ref)), (name, sign)


@gpu
def test_dense_kernels_refuse_bad_layouts(g):
    import torch
    _lib, ptr = _lib_ptr()
    rt = g.get_runtime()
    J = torch.zeros(8, 8, dtype=torch.float64, device=rt.device)
    v = torch.zeros(64, dtype=torch.float64, device=rt.device)
    assert rt.lib.gnk_dense_matmat(rt.ctx, 4, 4, ptr(J), 2, 2, ptr(v), 4, 0, 1, 1.0, ptr(v), 4, 0, rt.stream) != 0
    assert rt.lib.gnk_dense_rmatvec(rt.ctx, 2 ** 31, 1, ptr(J), 1, 1, ptr(v), 1.0, ptr(v), rt.stream) != 0
    assert rt.lib.gnk_dense_matmat(rt.ctx, 4, 4, ptr(J), 4, 1, ptr(v), 4, 0, 0, 1.0, ptr(v), 4, 0, rt.stream) != 0


# ------------------------------------------------------------------------------------------------
# 2. solvers: strided device J == the same J as torch CSR == the same J as host ndarrays, bit for bit
# ------------------------------------------------------------------------------------------------
def _fit(g, n, p, seed, decades=4.0):
    """r(x) = A x + 0.1 sin(B x) - y with graded columns (slow Krylov convergence), in torch on the device"""
    import torch
    dev = g.get_runtime().device
    rng = np.random.default_rng(seed)
    scale = 10.0 ** -np.linspace(0.0, decades, p)
    A = torch.as_tensor(rng.standard_normal((n, p)) * scale, device=dev)
    B = torch.as_tensor(rng.standard_normal((n, p)) / np.sqrt(p), device=dev)
    y = torch.as_tensor(rng.standard_normal(n), device=dev)
    res = lambda x: A @ x + 0.1 * torch.sin(B @ x) - y  # noqa: E731
    jac = lambda x: A + (0.1 * torch.cos(B @ x))[:, None] * B  # noqa: E731
    return res, jac, np.full(p, 0.5)


def _run(g, solver, res, jac, x0, capsys, **kw):
    import torch
    cbs = []
    cb = lambda x, nfev, cg_iter: cbs.append((np.array(x.cpu() if hasattr(x, "cpu") else np.asarray(x)), nfev))  # noqa
    try:
        out = solver(res, x0, jac, callback=cb, **kw)
        xf = out.x.cpu().numpy() if isinstance(out.x, torch.Tensor) else np.asarray(out.x)
        head = ("ok", out.nit, out.nrev, out.njev, bool(out.success))
    except Exception as e:  # noqa: BLE001  (an exception must be the same one on every path)
        head, xf = ("raised", type(e).__name__, str(e)), None
    return head, capsys.readouterr().out, cbs, xf


def _same(a, b):
    (ha, pa, ca, xa), (hb, pb, cb, xb) = a, b
    assert ha == hb and pa == pb
    assert [n for _, n in ca] == [n for _, n in cb]
    assert all(np.array_equal(u.view(np.int64), v.view(np.int64)) for (u, _), (v, _) in zip(ca, cb))
    assert (xa is None and xb is None) or np.array_equal(xa.view(np.int64), xb.view(np.int64))


def _three_ways(g, solver, res, jac, x0, capsys, host=True, csr=True, **kw):
    """(strided device J, device CSR J, host ndarray J) runs of one problem; asserts they agree bit for bit"""
    import torch
    dev = g.get_runtime().device
    x0d = torch.as_tensor(x0, device=dev)
    runs = [_run(g, solver, res, jac, x0d, capsys, **kw)]
    if csr:
        runs.append(_run(g, solver, res, lambda x: jac(x).to_sparse_csr(), x0d, capsys, **kw))
    if host:
        res_h = lambda x: res(torch.as_tensor(x, device=dev)).cpu().numpy()  # noqa: E731
        jac_h = lambda x: jac(torch.as_tensor(x, device=dev)).cpu().numpy()  # noqa: E731
        runs.append(_run(g, solver, res_h, jac_h, np.array(x0), capsys, **kw))
    for other in runs[1:]:
        _same(runs[0], other)
    return runs[0]


@gpu
@pytest.mark.parametrize("kw", [dict(max_iter=25), dict(max_iter=25, version="res_new"),
                                dict(max_iter=25, version="jac_old_res_old"),
                                dict(max_iter=25, version="jac_old_res_new"),
                                dict(max_iter=30, krylow_restart=10), dict(max_iter=25, ls_solver="cgls")])
def test_gnk_dense_device_jacobian_bitwise(g, capsys, kw):
    res, jac, x0 = _fit(g, 3000, 96, 1)
    head, _, cbs, _ = _three_ways(g, g.gauss_newton_krylow, res, jac, x0, capsys, **kw)
    assert head[0] == "ok" and len(cbs) >= 10


@gpu
def test_gnk_dense_device_jacobian_wide_panels_bitwise(g, capsys):
    """no restart and more than 104 iterations: the basis passes 104 columns and the least squares takes the wide
    Householder path"""
    res, jac, x0 = _fit(g, 2000, 160, 2, decades=6.0)
    head, _, cbs, _ = _three_ways(g, g.gauss_newton_krylow, res, jac, x0, capsys, max_iter=115, tol=1e-14)
    assert len(cbs) >= 106, head


@gpu
def test_gn_dense_device_jacobian_bitwise(g, capsys):
    """gauss_newton, 64 columns: the least squares by gnk_tsqr_ls, J d of the Armijo rule by gnk_dense_matmat, against
    the host ndarray run (a torch CSR J would take the CGLS branch instead)"""
    res, jac, x0 = _fit(g, 4000, 64, 3)
    head, _, cbs, _ = _three_ways(g, g.gauss_newton, res, jac, x0, capsys, csr=False, max_iter=12)
    assert head[0] == "ok" and len(cbs) >= 2


@gpu
def test_dense_device_jacobian_dtype_and_layout_copies(g, capsys):
    """float32 and non-unit-stride Jacobians get one contiguous float64 copy; the solve matches the CSR route"""
    import torch
    res, jac, x0 = _fit(g, 1500, 40, 4)
    for conv in (lambda J: J.float(), lambda J: torch.cat([J, J], 1)[:, ::2]):
        head, _, _, _ = _three_ways(g, g.gauss_newton_krylow, res, lambda x: conv(jac(x)), x0, capsys, host=False,
                                    max_iter=12)
        assert head[0] == "ok"
    from gauss_newton_via_generalized_krylov_subspaces_b200.device import DenseDeviceJacobian
    J = jac(torch.as_tensor(x0, device=g.get_runtime().device))
    d = DenseDeviceJacobian(g.get_runtime(), J.float())
    assert d.dense.dtype == torch.float64 and d.user.dtype == torch.float32 and (d.rs, d.cs) == (40, 1)
    d = DenseDeviceJacobian(g.get_runtime(), J.T.contiguous().T)
    assert d.dense.data_ptr() == d.user.data_ptr() and (d.rs, d.cs) == (1, 1500)


@gpu
def test_dense_device_jacobian_keeps_the_errors(g):
    import torch
    A = torch.as_tensor(np.array([[1.0, 2.0], [0.0, 1.0], [3.0, -1.0]]), device=g.get_runtime().device)
    x0 = torch.ones(2, dtype=torch.float64, device=A.device)
    with pytest.raises(ValueError, match=r"expected shape \(3, 2\)"):
        g.gauss_newton_krylow(lambda x: A @ x, x0, lambda x: A.T, callback=lambda **kw: None)
    with pytest.raises(ValueError, match="2-D"):
        g.gauss_newton_krylow(lambda x: A @ x, x0, lambda x: A[None], callback=lambda **kw: None)
    with pytest.raises(ValueError, match="cpu"):
        g.gauss_newton_krylow(lambda x: A @ x, x0, lambda x: A.cpu(), callback=lambda **kw: None)


# ------------------------------------------------------------------------------------------------
# 3. a jac that refills one tensor in place
# ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("version", ["jac_old_res_old", "jac_old_res_new"])
def test_in_place_refilled_jacobian_equals_fresh_tensors(g, capsys, version):
    import torch
    res, jac, x0 = _fit(g, 2500, 80, 5)
    buf = {}

    def jac_in_place(x):
        J = jac(x)
        if "J" not in buf:
            buf["J"] = torch.empty_like(J)
        buf["J"].copy_(J)
        return buf["J"]

    x0d = torch.as_tensor(x0, device=g.get_runtime().device)
    a = _run(g, g.gauss_newton_krylow, res, jac_in_place, x0d, capsys, max_iter=25, version=version)
    b = _run(g, g.gauss_newton_krylow, res, jac, x0d, capsys, max_iter=25, version=version)
    c = _run(g, g.gauss_newton_krylow, res, lambda x: jac(x).to_sparse_csr(), x0d, capsys, max_iter=25,
             version=version)
    _same(a, b)
    _same(a, c)
    assert a[0][0] == "ok" and len(a[2]) >= 10


# ------------------------------------------------------------------------------------------------
# 4. 2^31 entries and more on one B200
# ------------------------------------------------------------------------------------------------
def _free_gb(rt):
    import torch
    return torch.cuda.mem_get_info(rt.device)[0] / 1e9


@gpu
def test_gnk_dense_jacobian_past_2_31_entries(g):
    """A 1 049 600 x 2048 dense J (2.15e9 entries, 17.2 GB).  Before DenseDeviceJacobian the CSR route raised GnkError
    here (the int32 CSR kernels), after allocating a 25 GB CSR copy.  Checks: row blocks of J V_k bit-identical to
    gnk_spmm_csr on the CSR of those rows; J^T r exact on an integer-valued J and within 1e-12 of torch's fp64 product on
    a Gaussian J; a GNK solve through a restart, with a jac that refills the tensor in place, decreases the loss as the
    same problem does at 1/16 of the rows."""
    import torch
    _lib, ptr = _lib_ptr()
    rt = g.get_runtime()
    n, p = 1049600, 2048
    assert n * p >= 2 ** 31
    if _free_gb(rt) < 40:
        pytest.skip("needs about 40 GB of free device memory")
    gen = torch.Generator(device=rt.device).manual_seed(7)
    J = torch.empty(n, p, dtype=torch.float64, device=rt.device)
    # integer-valued J and r: every partial sum is an integer below 2^53, so J^T r is exact in any order
    J.copy_(torch.randint(-4, 5, (n, p), generator=gen, device=rt.device, dtype=torch.int8))
    r = torch.randint(-8, 9, (n,), generator=gen, device=rt.device).to(torch.float64)
    w = torch.empty(p, dtype=torch.float64, device=rt.device)
    _lib.check(rt.lib.gnk_dense_rmatvec(rt.ctx, n, p, ptr(J), p, 1, ptr(r), 1.0, ptr(w), rt.stream), "rmatvec")
    assert torch.equal(w, J.T @ r)
    J.normal_(generator=gen)
    r.normal_(generator=gen)
    _lib.check(rt.lib.gnk_dense_rmatvec(rt.ctx, n, p, ptr(J), p, 1, ptr(r), -1.0, ptr(w), rt.stream), "rmatvec")
    want = -(J.T @ r)
    assert float(torch.linalg.norm(w - want) / torch.linalg.norm(want)) < 1e-12
    # J V_k, k = 33: sampled row blocks (rows are independent) against the CSR kernel on those rows alone
    k = 33
    V = torch.randn(p * k, dtype=torch.float64, device=rt.device, generator=gen)
    JV = torch.empty(n * k, dtype=torch.float64, device=rt.device)
    _lib.check(rt.lib.gnk_dense_matmat(rt.ctx, n, p, ptr(J), p, 1, ptr(V), p, 0, k, 1.0, ptr(JV), n, 0, rt.stream),
               "matmat")
    for r0, m in ((0, 4096), (n // 2 - 777, 3001), (n - 2049, 2049)):
        A = J[r0:r0 + m].to_sparse_csr()
        rp, ci = A.crow_indices().to(torch.int32), A.col_indices().to(torch.int32)
        ref = torch.empty(m * k, dtype=torch.float64, device=rt.device)
        _lib.check(rt.lib.gnk_spmm_csr(rt.ctx, m, ptr(rp), ptr(ci), ptr(A.values()), ptr(V), p, 0, k, 1.0, ptr(ref),
                                       m, 0, rt.stream), "gnk_spmm_csr")
        assert torch.equal(JV.view(k, n)[:, r0:r0 + m], ref.view(k, m)), r0
    del JV, A, ref
    # A problem with a known solution x*: F(x) = J tanh(x) - y, y = J tanh(x*), columns of J graded over three decades.
    # It has to be nonlinear: for a linear F the first iteration after a restart has d = 0 exactly (x is already the
    # least-squares optimum over a span that contains x), and the Armijo rule must fail there.  The Jacobian
    # J diag(1 - tanh(x)^2) is refilled in place, by rescaling the columns of the one 17.2 GB tensor, and returned.
    J *= torch.logspace(0, -3, p, dtype=torch.float64, device=rt.device)
    x_true = torch.randn(p, dtype=torch.float64, device=rt.device, generator=gen)

    def solve(M):
        scale = torch.ones(p, dtype=torch.float64, device=rt.device)  # M = J diag(scale)

        def F(x):
            return M @ (torch.tanh(x) / scale)

        def jac(x):
            new = 1.0 - torch.tanh(x) ** 2
            M.mul_(new / scale)
            scale.copy_(new)
            return M

        y = F(x_true)
        x0 = torch.ones(p, dtype=torch.float64, device=rt.device)
        out = g.gauss_newton_krylow(lambda x: F(x) - y, x0, jac, krylow_restart=2, max_iter=6,
                                    callback=lambda **kw: None)
        l0, l1 = float(torch.sum((F(x0) - y) ** 2)), float(torch.sum((F(out.x) - y) ** 2))
        return l1 / l0, out

    small, out_small = solve(J[: n // 16].clone())
    big, out = solve(J)
    # five iterations, restarts after iterations 2 and 4; the loss ratios agree across row counts
    assert out.nit == out_small.nit == 5 and big < 0.5 and small < 0.5, (out.nit, out_small.nit, big, small)
    assert 0.25 < big / small < 4.0, (big, small)


@gpu
def test_gauss_newton_dense_jacobian_past_2_31_entries(g):
    """An 8.5 M x 255 dense J (2.17e9 entries): the least squares through the blocked Householder TSQR, J d by
    gnk_dense_matmat.  Before DenseDeviceJacobian the CSR route raised GnkError here."""
    import torch
    rt = g.get_runtime()
    n, p = 8_500_000, 255
    assert n * p >= 2 ** 31
    if _free_gb(rt) < 40:
        pytest.skip("needs about 40 GB of free device memory")
    gen = torch.Generator(device=rt.device).manual_seed(11)
    J = torch.randn(n, p, dtype=torch.float64, device=rt.device, generator=gen)
    x_true = torch.randn(p, dtype=torch.float64, device=rt.device, generator=gen)
    y = J @ x_true
    out = g.gauss_newton(lambda x: J @ x - y, torch.zeros(p, dtype=torch.float64, device=rt.device), lambda x: J,
                         max_iter=4, callback=lambda **kw: None)
    assert out.success
    assert float(torch.max(torch.abs(out.x - x_true))) < 1e-10
