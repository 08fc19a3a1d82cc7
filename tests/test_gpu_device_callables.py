"""Device callables: res / jac on CUDA tensors (selected by a CUDA-tensor x0), the device CSR pattern / transpose
(gnk_csr_pattern, gnk_csr_pattern_equal, gnk_csr_gather) and the column-blocked gnk_spmm_csr.

The solver-level tests run each problem twice -- as numpy / scipy host callables and as device callables wrapping the
same host functions -- and require the same counters, prints, callback data and final x bit for bit."""
import subprocess
from fractions import Fraction

import numpy as np
import pytest
import scipy.sparse as sp

from golden_util import Golden, Recorder, bound_for, check_trace  # noqa: E402
from oracle import gnk_oracle as orc  # noqa: E402

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def g():
    import gauss_newton_via_generalized_krylov_subspaces_b200 as pkg
    import gauss_newton_via_generalized_krylov_subspaces_b200.device as device
    device._runtime = None
    pkg.get_runtime()
    return pkg


def _t(g, a, dtype=None):
    import torch
    return torch.as_tensor(np.asarray(a), device=g.get_runtime().device, dtype=dtype)


def _torch_csr(g, A, index_dtype=None):
    import torch
    A = sp.csr_array(A)
    A.sort_indices()
    it = index_dtype or torch.int64
    return torch.sparse_csr_tensor(_t(g, A.indptr.astype(np.int64)).to(it), _t(g, A.indices.astype(np.int64)).to(it),
                                   _t(g, A.data.astype(np.float64)), size=A.shape)


def _random_csr(rng, n_rows, n_cols, density, long_row=None, empty_rows=(), empty_cols=()):
    A = sp.random(n_rows, n_cols, density=density, format="lil", random_state=rng,
                  data_rvs=lambda k: rng.standard_normal(k) * 10.0 ** rng.integers(-3, 4, k))
    if long_row is not None:
        A[long_row, :] = rng.standard_normal(n_cols)
    for r in empty_rows:
        A[r, :] = 0
    for c in empty_cols:
        A[:, c] = 0
    A = sp.csr_array(A.tocsr())
    A.eliminate_zeros()
    A.sort_indices()
    return A


# ------------------------------------------------------------------------------------------------
# 1. blocked SpMM: the fma chain of every (row, column), bit for bit
# ------------------------------------------------------------------------------------------------
def _fma_chain(A, x, sign):
    """sign * (fma(val[e], x[col[e]], acc) over the row from 0.0), each fma rounded once (Fraction -> float is
    correctly rounded)"""
    out = np.empty(A.shape[0])
    for r in range(A.shape[0]):
        acc = 0.0
        for e in range(A.indptr[r], A.indptr[r + 1]):
            acc = float(Fraction(A.data[e]) * Fraction(x[A.indices[e]]) + Fraction(acc))
        out[r] = sign * acc
    return out


def _spmm(g, A, V, k, sign, in_ld, in_off, out_ld, out_off):
    from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib
    from gauss_newton_via_generalized_krylov_subspaces_b200.device import ptr
    rt = g.get_runtime()
    n_rows, n_cols = A.shape
    rp, ci, va = _t(g, A.indptr.astype(np.int32)), _t(g, A.indices.astype(np.int32)), _t(g, A.data)
    din = rt.zeros(in_ld * k + in_off + n_cols)
    for j in range(k):
        rt.upload(V[j], din[j * in_ld + in_off:j * in_ld + in_off + n_cols])
    dout = rt.zeros(out_ld * k + out_off + n_rows)
    dout.fill_(float("nan"))
    _lib.check(rt.lib.gnk_spmm_csr(rt.ctx, n_rows, ptr(rp), ptr(ci), ptr(va), ptr(din), in_ld, in_off, k, sign,
                                   ptr(dout), out_ld, out_off, rt.stream), "gnk_spmm_csr")
    got = rt.download(dout)
    cols = [got[j * out_ld + out_off:j * out_ld + out_off + n_rows] for j in range(k)]
    gaps = [got[j * out_ld + out_off + n_rows:(j + 1) * out_ld + out_off] for j in range(k - 1)]
    assert all(np.all(np.isnan(a)) for a in gaps) and np.all(np.isnan(got[:out_off]))  # nothing else is written
    return cols


@gpu
def test_blocked_spmm_is_the_fma_chain_bit_for_bit(g):
    rng = np.random.default_rng(7)
    mats = {
        "random": _random_csr(rng, 301, 10_050, 0.002, long_row=17, empty_rows=(0, 5, 300)),
        "one_column": _random_csr(rng, 97, 1, 0.6),
        "one_row": _random_csr(rng, 1, 640, 0.5),
    }
    for name, A in mats.items():
        n_rows, n_cols = A.shape
        for k in (1, 7, 8, 9, 30, 56, 255):
            V = rng.standard_normal((k, n_cols))
            for sign in (1.0, -1.0, 0.5):
                in_ld, out_ld = n_cols + 3 + (k % 2), n_rows + 5
                cols = _spmm(g, A, V, k, sign, in_ld, 3, out_ld, 1)
                # every column of the k-column call equals the one-column call on the same data
                for j in range(k):
                    one = _spmm(g, A, V[j:j + 1], 1, sign, n_cols, 0, n_rows, 0)[0] if k > 1 and j in (0, k - 1) \
                        else None
                    if one is not None:
                        assert np.array_equal(cols[j].view(np.int64), one.view(np.int64)), (name, k, j)
                # ... and the exact fma chain (a few columns per call: the restatement is slow)
                for j in sorted({0, k // 2, k - 1}):
                    want = _fma_chain(A, V[j], sign)
                    assert np.array_equal(cols[j].view(np.int64), want.view(np.int64)), (name, k, j, sign)


@gpu
def test_blocked_spmm_bratu_k_columns_equal_k_single_calls(g):
    pb = g.BratuPdeProblem(1025, 5, 10)
    u = np.random.default_rng(3).standard_normal(pb.n if hasattr(pb, "n") else 1024 * 1024)
    A = sp.csr_array(pb.make_jac()(u).tocsr())
    A.sort_indices()
    k = 30
    V = np.random.default_rng(4).standard_normal((k, A.shape[1]))
    cols = _spmm(g, A, V, k, -1.0, A.shape[1] + 16, 0, A.shape[0] + 16, 0)
    for j in range(k):
        one = _spmm(g, A, V[j:j + 1], 1, -1.0, A.shape[1], 0, A.shape[0], 0)[0]
        assert np.array_equal(cols[j].view(np.int64), one.view(np.int64)), j


# ------------------------------------------------------------------------------------------------
# 2. pattern and gather against scipy's sorted transpose
# ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("index_dtype", ["int32", "int64"])
def test_pattern_and_gather_equal_scipy_transpose(g, index_dtype):
    import torch
    from gauss_newton_via_generalized_krylov_subspaces_b200.device import DeviceCsrJacobian
    rt = g.get_runtime()
    rng = np.random.default_rng(11)
    it = getattr(torch, index_dtype)
    cases = [_random_csr(rng, 500, 300, 0.02, long_row=3, empty_rows=(0, 10, 499), empty_cols=(0, 7, 299)),
             _random_csr(rng, 40, 2000, 0.01), sp.csr_array((0, 5)), sp.csr_array((5, 0)), sp.csr_array((6, 4)),
             _random_csr(rng, 3000, 1, 0.5)]
    for A in cases:
        op = DeviceCsrJacobian.from_tensor(rt, _torch_csr(g, A, it))
        AT = sp.csr_array(A.T)
        AT.sort_indices()
        assert np.array_equal(rt.download(op.rowptr).astype(np.int64), A.indptr)
        assert np.array_equal(rt.download(op.col).astype(np.int64), A.indices)
        assert np.array_equal(rt.download(op.rowptr_t).astype(np.int64), AT.indptr), A.shape
        assert np.array_equal(rt.download(op.col_t).astype(np.int64), AT.indices), A.shape
        assert np.array_equal(rt.download(op.val_t).view(np.int64), AT.data.view(np.int64)), A.shape


@gpu
@pytest.mark.parametrize("defect,rowptr,col,match", [
    ("unsorted", [0, 2, 4], [0, 1, 2, 1], "row 1: column indices not sorted"),
    ("duplicate", [0, 2, 4], [0, 1, 2, 2], "row 1: duplicate column index"),
    ("out_of_range", [0, 2, 3], [0, 1, 3, 0], "row 1: column index out of range"),
    ("negative_col", [0, 2, 3], [0, -1, 1, 0], "row 0: column index out of range"),
    ("rowptr_decreasing", [0, 3, 2], [0, 1, 2], "row 1: row pointer decreases"),
    ("rowptr_start", [1, 2, 3], [0, 1, 2], "row 0: rowptr\\[0\\] is not 0"),
    ("rowptr_end", [0, 1, 2], [0, 1, 2], "row 2: rowptr\\[n_rows\\] is not nnz"),
])
@pytest.mark.parametrize("index_dtype", ["int32", "int64"])
def test_invalid_patterns_raise_value_errors_naming_the_row(g, defect, rowptr, col, match, index_dtype):
    import torch
    from gauss_newton_via_generalized_krylov_subspaces_b200.device import CsrPattern
    rt = g.get_runtime()
    it = getattr(torch, index_dtype)
    with pytest.raises(ValueError, match=match):
        CsrPattern(rt, 2, 3, _t(g, rowptr).to(it), _t(g, col).to(it))
    # the context is still usable afterwards
    CsrPattern(rt, 2, 3, _t(g, [0, 2, 3]).to(it), _t(g, [0, 2, 1]).to(it))


# ------------------------------------------------------------------------------------------------
# 3. pattern cache
# ------------------------------------------------------------------------------------------------
def _rosenbrock_pair(g, index_dtype=None, fresh=True, mutate=None):
    """host (res, jac) of the chained Rosenbrock problem and device wrappers around the SAME host functions"""
    import torch
    from gauss_newton_via_generalized_krylov_subspaces_b200 import rosenbrock_problem as rp
    res_h = lambda x: rp.res(x)  # noqa: E731  (not rp.res itself: that one has a native device twin)
    jac_h = lambda x: rp.jac(x)  # noqa: E731
    held = {}

    def res_d(x):
        return _t(g, rp.res(x.cpu().numpy()))

    def jac_d(x):
        J = _torch_csr(g, rp.jac(x.cpu().numpy()), index_dtype)
        if fresh or "J" not in held:
            held["J"] = J
            return J
        crow, col = held["J"].crow_indices(), held["J"].col_indices()
        if mutate is not None:
            mutate(crow, col, J)
        else:
            crow.copy_(J.crow_indices())
            col.copy_(J.col_indices())
        return torch.sparse_csr_tensor(crow, col, J.values(), size=J.shape)

    return res_h, jac_h, res_d, jac_d


def _probe(g, res_d, jac_d, x0):
    from gauss_newton_via_generalized_krylov_subspaces_b200.gauss_newton_krylow import resolve_problem
    prob = resolve_problem(res_d, jac_d, _t(g, x0), ())
    x = prob.new_sol()
    prob.upload_x(_t(g, x0), x)
    prob.evaluate(x)  # the first residual fixes the residual-space layout
    return prob, x


@gpu
def test_pattern_cache_builds_once_per_pattern(g):
    x0 = Golden("rosenbrock")["x0_i"]
    for fresh in (False, True):  # the same index tensors every call / fresh tensors with the same contents
        _, _, res_d, jac_d = _rosenbrock_pair(g, fresh=fresh)
        prob, x = _probe(g, res_d, jac_d, x0)
        for _ in range(4):
            prob.jacobian(x)
        assert prob.pattern_builds == 1, fresh


def _alternating_pattern_jac(g, in_place):
    """J of the chained Rosenbrock problem with one explicit zero stored at (0, 2) on odd calls and at (0, 3) on even
    calls: the same matrix on two patterns of the same size.  in_place: written into the same index tensors."""
    import torch
    from gauss_newton_via_generalized_krylov_subspaces_b200 import rosenbrock_problem as rp
    state = {"n": 0, "bufs": None}

    def jac(x):
        state["n"] += 1
        J = sp.coo_array(rp.jac(x.cpu().numpy()))
        extra = 2 if state["n"] % 2 else 3
        J = sp.coo_array((np.append(J.data, 0.0), (np.append(J.row, 0), np.append(J.col, extra))), shape=J.shape)
        T = _torch_csr(g, J.tocsr())
        if not in_place:
            return T
        if state["bufs"] is None:
            state["bufs"] = (T.crow_indices().clone(), T.col_indices().clone())
        crow, col = state["bufs"]
        crow.copy_(T.crow_indices())
        col.copy_(T.col_indices())
        return torch.sparse_csr_tensor(crow, col, T.values(), size=T.shape)

    return jac


@gpu
def test_in_place_index_rewrites_rebuild_and_keep_the_solve_bitwise(g):
    """a jac that refills the same index tensors with a changed pattern: the cache compares contents, so every change
    rebuilds, and the run equals the one that hands over fresh tensors bit for bit"""
    from gauss_newton_via_generalized_krylov_subspaces_b200 import rosenbrock_problem as rp
    x0 = Golden("rosenbrock")["x0_i"]
    res_d = lambda x: _t(g, rp.res(x.cpu().numpy()))  # noqa: E731
    prob, x = _probe(g, res_d, _alternating_pattern_jac(g, True), x0)
    for _ in range(4):
        prob.jacobian(x)
    assert prob.pattern_builds == 4
    outs = [g.gauss_newton_krylow(res_d, _t(g, x0), _alternating_pattern_jac(g, in_place), callback=lambda **kw: None)
            for in_place in (True, False)]
    a, b = outs
    assert (a.nit, a.nrev, a.njev) == (b.nit, b.nrev, b.njev) == (48, 49, 48)
    assert np.array_equal(a.x.cpu().numpy().view(np.int64), b.x.cpu().numpy().view(np.int64))


# ------------------------------------------------------------------------------------------------
# 4. solver layer: host callables and device callables around the same host functions, bitwise
# ------------------------------------------------------------------------------------------------
def _both(g, solver, res_h, jac_h, res_d, jac_d, x0, capsys, **kw):
    runs = []
    for res, jac, x in ((res_h, jac_h, np.asarray(x0, dtype=np.float64)), (res_d, jac_d, _t(g, x0))):
        cbs = []
        out = solver(res, x, jac, callback=lambda x, nfev, cg_iter: cbs.append(
            (np.array(np.asarray(x.cpu()) if hasattr(x, "cpu") else np.asarray(x)), nfev, cg_iter)), **kw)
        printed = capsys.readouterr().out
        xf = out.x.cpu().numpy() if hasattr(out.x, "cpu") else np.asarray(out.x)
        runs.append((out, cbs, printed, xf))
    (oh, ch, ph, xh), (od, cd, pd, xd) = runs
    assert (oh.nit, oh.nrev, oh.njev, bool(oh.success)) == (od.nit, od.nrev, od.njev, bool(od.success))
    assert ph == pd
    assert [(n, c) for _, n, c in ch] == [(n, c) for _, n, c in cd]
    assert all(np.array_equal(a.view(np.int64), b.view(np.int64)) for (a, _, _), (b, _, _) in zip(ch, cd))
    assert np.array_equal(xh.view(np.int64), xd.view(np.int64))
    import torch
    assert isinstance(od.x, torch.Tensor) and od.x.is_cuda and od.x.shape == (len(x0),)
    return oh, od


def _bratu_pair(g, G, lam=10):
    gd = Golden(f"bratu_g{G}") if G == 101 else None
    o = orc.BratuOracle(G, 5, lam)
    y = gd["y"] if gd is not None else o.operator(o.u_true)
    u0 = gd["u0"] if gd is not None else o.start_vector(seed=42)
    pb = g.BratuPdeProblem(G, 5, lam)
    res, jac = pb.make_res(y), pb.make_jac()
    res_h = lambda x: res(x)  # noqa: E731  (wrapped: the Bratu callables themselves run natively)
    jac_h = lambda x: jac(x).tocsr()  # noqa: E731
    res_d = lambda x: _t(g, res(x.cpu().numpy()))  # noqa: E731
    jac_d = lambda x: _torch_csr(g, jac(x.cpu().numpy()).tocsr())  # noqa: E731
    return res_h, jac_h, res_d, jac_d, u0


@gpu
@pytest.mark.parametrize("kw", [dict(max_iter=30), dict(max_iter=30, version="res_new"),
                                dict(max_iter=25, version="jac_old_res_old"),
                                dict(max_iter=25, version="jac_old_res_new"),
                                dict(max_iter=40, krylow_restart=30)])
def test_bratu_g101_gnk_device_callables_bitwise(g, capsys, kw):
    res_h, jac_h, res_d, jac_d, u0 = _bratu_pair(g, 101)
    _both(g, g.gauss_newton_krylow, res_h, jac_h, res_d, jac_d, u0, capsys, **kw)


@gpu
def test_bratu_g257_wide_panels_device_callables_bitwise(g, capsys):
    res_h, jac_h, res_d, jac_d, u0 = _bratu_pair(g, 257)
    oh, od = _both(g, g.gauss_newton_krylow, res_h, jac_h, res_d, jac_d, u0, capsys, max_iter=130)
    assert od.nit >= 105 or od.success


@gpu
@pytest.mark.parametrize("tag", ["i", "ii", "iii"])
def test_rosenbrock_device_callables_bitwise(g, capsys, tag):
    x0 = Golden("rosenbrock")["x0_" + tag]
    res_h, jac_h, res_d, jac_d = _rosenbrock_pair(g)
    for kw in ({}, dict(version="res_new")):
        _both(g, g.gauss_newton_krylow, res_h, jac_h, res_d, jac_d, x0, capsys, **kw)
    _both(g, g.gauss_newton, res_h, jac_h, res_d, jac_d, x0, capsys)


@gpu
@pytest.mark.parametrize("precond", [False, True])
def test_gauss_newton_sparse_device_callables_bitwise(g, capsys, precond):
    res_h, jac_h, res_d, jac_d, u0 = _bratu_pair(g, 101)
    oh, od = _both(g, g.gauss_newton, res_h, jac_h, res_d, jac_d, u0, capsys, cg_preconditioner=precond)
    assert od.success


@gpu
def test_rosenbrock_3d_dense_device_callables_bitwise(g, capsys):
    def res2(x):
        return 2 ** 0.5 * np.concatenate([10 * (x[1:] - x[:-1] ** 2), 1 - x[:-1]])

    def jac2(x):
        b1 = 10 * sp.eye(1, 2, k=1) - 20 * sp.diags(x[:-1], shape=(1, 2))
        return 2 ** 0.5 * sp.block_array([[b1], [-sp.eye(1, 2, k=0)]]).todense()

    oh, od = _both(g, g.gauss_newton, res2, jac2, lambda x: _t(g, res2(x.cpu().numpy())),
                   lambda x: _t(g, np.asarray(jac2(x.cpu().numpy()))), np.array([-1.0, 1.0]), capsys)
    assert (od.nit, od.nrev, od.njev) == (19, 71, 19)


@gpu
def test_powell_step_length_plugins_device_callables(g, capsys):
    import torch

    def pres(x, tau):
        if isinstance(x, torch.Tensor):
            return _t(g, pres(x.cpu().numpy(), tau))
        return np.array([x[0] + 1, tau * x[0] ** 2 + x[0] - 1])

    def pjac(x, tau):
        if isinstance(x, torch.Tensor):
            return _t(g, pjac(x.cpu().numpy(), tau).astype(np.float64))
        return np.array([[1], [2 * tau * x[0] + 1]])

    seen = []

    def no_step_length_control(res, x, res_ev, jac_ev, args, descent_direction, *_):
        seen.append(type(x).__name__ + type(res_ev).__name__ + type(jac_ev).__name__ + type(descent_direction).__name__)
        return 1, res(x + descent_direction, *args), 1

    state = dict(it=2)

    def too_small_steps(res, x, res_ev, jac_ev, args, descent_direction, *_):
        step_length = -1 / float(descent_direction[0]) * 2 ** -state["it"]
        state["it"] += 1
        return step_length, res(x + step_length * descent_direction, *args), 1

    for tau in (-5, 5):
        for ctl in (g.armijo_goldstein, too_small_steps, no_step_length_control):
            if tau == 5 and ctl is too_small_steps:
                continue
            outs = []
            for x0 in (np.array([1.0]), _t(g, [1.0])):
                state["it"] = 2
                xs = []
                cb = lambda x, nfev, cg_iter: xs.append(float(x[0]))  # noqa: E731
                try:
                    out = g.gauss_newton(pres, x0, pjac, args=(tau,), max_iter=19, callback=cb,
                                         step_length_control=ctl)
                    outs.append((out.nit, out.nrev, bool(out.success), xs))
                except g.StepLengthConvergenceError:
                    outs.append(("raised", xs))
            assert outs[0] == outs[1], (tau, ctl.__name__)
            capsys.readouterr()
    assert "TensorTensorTensorTensor" in seen and "ndarrayndarrayndarrayndarray" in seen


@gpu
def test_cg_least_squares_device_tensors_bitwise(g):
    import torch
    rng = np.random.default_rng(5)
    A = _random_csr(rng, 400, 150, 0.05, long_row=2)
    y = rng.standard_normal(400)
    x0 = rng.standard_normal(150)
    for pre in (False, True):
        xh, ih = g.cg_least_squares(A, y, preconditioner=pre)
        xd, id_ = g.cg_least_squares(_torch_csr(g, A), _t(g, y), preconditioner=pre)
        assert ih == id_ and np.array_equal(xh.view(np.int64), xd.cpu().numpy().view(np.int64))
        assert isinstance(xd, torch.Tensor) and xd.is_cuda
    xh, ih = g.cg_least_squares(A, y, x0=x0)
    xd, id_ = g.cg_least_squares(_torch_csr(g, A, torch.int32), _t(g, y), x0=_t(g, x0))
    assert ih == id_ and np.array_equal(xh, xd.cpu().numpy())
    # COO with duplicates (summed), dense (exact zeros dropped), and -1 * J.T
    Acoo = sp.coo_array(A)
    rows = np.concatenate([Acoo.row, Acoo.row[:50]])
    cols = np.concatenate([Acoo.col, Acoo.col[:50]])
    vals = np.concatenate([Acoo.data * 0.5, Acoo.data[:50] * 0.5])
    vals[50:len(Acoo.data)] = Acoo.data[50:]
    Ad = sp.coo_array((vals, (rows, cols)), shape=A.shape)
    tcoo = torch.sparse_coo_tensor(_t(g, np.stack([rows, cols])), _t(g, vals), size=A.shape)
    xh, ih = g.cg_least_squares(Ad, y)
    xd, id_ = g.cg_least_squares(tcoo, _t(g, y))
    assert ih == id_ and np.array_equal(xh, xd.cpu().numpy())
    D = A.toarray()
    D[0, 0] = -0.0
    xh, ih = g.cg_least_squares(D, y)
    xd, id_ = g.cg_least_squares(_t(g, D), _t(g, y))
    assert ih == id_ and np.array_equal(xh, xd.cpu().numpy())
    pb = g.BratuPdeProblem(41, 5, 10)
    J = pb.make_jac()(np.random.default_rng(1).standard_normal(40 * 40) * 0.1)
    yb = rng.standard_normal(40 * 40)
    xh, ih = g.cg_least_squares(-1 * J.T, yb)
    xd, id_ = g.cg_least_squares(_torch_csr(g, -1 * sp.csr_array(J.tocsr()).T), _t(g, yb))
    assert ih == id_ and np.array_equal(xh, xd.cpu().numpy())


@gpu
def test_linear_least_squares_device_tensors_bitwise(g, capsys):
    import torch
    rng = np.random.default_rng(9)
    for n, k in ((300, 20), (5000, 120)):
        A = rng.standard_normal((n, k))
        A[:, 3] = A[:, 2] + 1e-12 * rng.standard_normal(n)  # a pivot below 1e-8: the reference's print
        y = rng.standard_normal(n)
        xh = g.linear_least_squares(A, y)
        ph = capsys.readouterr().out
        xd = g.linear_least_squares(_t(g, A), _t(g, y))
        assert capsys.readouterr().out == ph and "rank deficient" in ph
        assert isinstance(xd, torch.Tensor) and xd.is_cuda
        assert np.array_equal(xh.view(np.int64), xd.cpu().numpy().view(np.int64))


# ------------------------------------------------------------------------------------------------
# 5. a pure-torch Bratu problem against the reference's goldens
# ------------------------------------------------------------------------------------------------
def _torch_bratu(g, G, y):
    from torch_bratu import TorchBratu
    return TorchBratu(g.BratuPdeProblem(G, 5, 10), orc.BratuOracle(G, 5, 10), y, g.get_runtime().device)


@gpu
@pytest.mark.parametrize("rname,kw", [
    ("gnk_res_old", dict(max_iter=100)),
    ("gnk_res_new", dict(max_iter=100, version="res_new")),
    ("gnk_jac_old_res_old", dict(max_iter=25, version="jac_old_res_old")),
    ("gnk_jac_old_res_new", dict(max_iter=25, version="jac_old_res_new")),
    ("gnk_restart30", dict(max_iter=100, krylow_restart=30)),
])
def test_pure_torch_bratu_g101_against_goldens(g, rname, kw):
    gd = Golden("bratu_g101")
    tb = _torch_bratu(g, 101, gd["y"])
    gr = gd.run(rname)
    o = orc.BratuOracle(101, 5, 10)
    rec = Recorder(gr["sample_idx"], lambda x: float(np.linalg.norm(o.u_true - x)))
    out = g.gauss_newton_krylow(tb.res, _t(g, gd["u0"]), tb.jac,
                                callback=lambda x, nfev, cg_iter: rec(x.cpu().numpy(), nfev, cg_iter), **kw)
    n = len(gr["xnorm"])
    restart = kw.get("krylow_restart")
    check_trace(rec, gr, 1e-10, upto=n if restart is None else min(n, restart))
    check_trace(rec, gr, 1e-10 if restart is None else 1e-8)
    assert (out.nit, out.nrev, out.njev, bool(out.success)) == (
        int(gr["nit"]), int(gr["nfev"]), int(gr["njev"]), bool(gr["success"]))


@gpu
def test_pure_torch_bratu_1024_restart30_against_goldens(g):
    gd = Golden("bratu_g1025")
    o = orc.BratuOracle(1025, 5, 10)
    y = o.operator(o.u_true)
    u0 = o.start_vector(seed=42)
    tb = _torch_bratu(g, 1025, y)
    gr = gd.run("gnk_restart30")
    bound = bound_for("bratu_g1025", "gnk_restart30")
    rec = Recorder(gr["sample_idx"], lambda x: float(np.linalg.norm(o.u_true - x)))
    out = g.gauss_newton_krylow(tb.res, _t(g, u0), tb.jac, krylow_restart=30, max_iter=100,
                                callback=lambda x, nfev, cg_iter: rec(x.cpu().numpy(), nfev, cg_iter))
    check_trace(rec, gr, bound)
    assert (out.nit, out.nrev, out.njev, bool(out.success)) == (
        int(gr["nit"]), int(gr["nfev"]), int(gr["njev"]), bool(gr["success"]))


# ------------------------------------------------------------------------------------------------
# 6. contract checks
# ------------------------------------------------------------------------------------------------
@gpu
def test_device_callables_contract(g):
    import torch
    rt = g.get_runtime()
    A = _t(g, np.array([[1.0, 2.0], [0.0, 1.0], [3.0, -1.0]]))
    b = _t(g, np.array([1.0, 2.0, 0.5]))

    def res(x, scale):
        assert isinstance(x, torch.Tensor) and x.is_cuda and x.dtype == torch.float64 and x.shape == (2,)
        return scale * (A @ x - b)

    def jac(x, scale):
        return (scale * A).to_sparse_csr()

    kept = []
    # two iterations: the basis then spans R^2 and x is the least-squares solution (a third trial could not decrease)
    out = g.gauss_newton_krylow(res, _t(g, [1.0, 1.0]), jac, args=(2.0,), max_iter=3,
                                callback=lambda x, nfev, cg_iter: kept.append(x))
    assert isinstance(out.x, torch.Tensor) and out.x.device == rt.device and out.x.shape == (2,)
    assert len(kept) >= 2 and all(isinstance(k, torch.Tensor) and k.is_cuda for k in kept)
    assert not torch.equal(kept[0], kept[-1]) or len(kept) == 1  # the callback's copies are its own
    want = np.linalg.lstsq(A.cpu().numpy(), b.cpu().numpy(), rcond=None)[0]
    assert np.allclose(out.x.cpu().numpy(), want, atol=1e-8)
    # float32 results are converted, like np.asarray(..., float64) on the host path
    out32 = g.gauss_newton(lambda x, s: res(x, s).float(), _t(g, [1.0, 1.0]), jac, args=(2.0,), max_iter=2,
                           callback=lambda **kw: None)
    assert out32.x.dtype == torch.float64
    # the benchmark harness works unchanged
    from gauss_newton_via_generalized_krylov_subspaces_b200.benchmark import benchmark_method
    err, loss, nfev, cg = benchmark_method(g.gauss_newton_krylow, res, _t(g, [1.0, 1.0]), jac,
                                           lambda x: float(torch.linalg.norm(x - _t(g, want))), args=(2.0,),
                                           kwargs=dict(max_iter=3))
    assert len(err) == len(loss) and loss[-1] < loss[0] and all(isinstance(v, float) for v in loss)
    # a CPU tensor keeps the host path (host callables)
    outc = g.gauss_newton_krylow(lambda x: np.asarray(A.cpu()) @ np.asarray(x) - np.asarray(b.cpu()),
                                 torch.tensor([1.0, 1.0], dtype=torch.float64),
                                 lambda x: np.asarray(A.cpu()), max_iter=3, callback=lambda **kw: None)
    assert isinstance(outc.x, np.ndarray)


@gpu
def test_device_callables_errors(g):
    import torch
    rt = g.get_runtime()
    A = _t(g, np.array([[1.0, 2.0], [0.0, 1.0], [3.0, -1.0]]))
    good_res = lambda x: A @ x  # noqa: E731
    good_jac = lambda x: A  # noqa: E731
    x0 = _t(g, [1.0, 1.0])
    with pytest.raises(ValueError, match="cpu"):
        g.gauss_newton_krylow(lambda x: (A @ x).cpu(), x0, good_jac, callback=lambda **kw: None)
    with pytest.raises(TypeError, match="ndarray"):
        g.gauss_newton_krylow(lambda x: (A @ x).cpu().numpy(), x0, good_jac, callback=lambda **kw: None)
    calls = {"n": 0}

    def res_len(x):
        calls["n"] += 1
        return A @ x if calls["n"] == 1 else torch.cat([A @ x, A @ x])

    with pytest.raises(ValueError, match="expected 3 values"):
        g.gauss_newton_krylow(res_len, x0, good_jac, callback=lambda **kw: None)
    with pytest.raises(ValueError, match="1-D"):
        g.gauss_newton(lambda x: (A @ x)[:, None], x0, good_jac, callback=lambda **kw: None)
    with pytest.raises(ValueError, match=r"expected shape \(3, 2\)"):
        g.gauss_newton_krylow(good_res, x0, lambda x: A.T, callback=lambda **kw: None)
    with pytest.raises(ValueError, match="cpu"):
        g.gauss_newton(good_res, x0, lambda x: A.cpu(), callback=lambda **kw: None)
    # dimensions at or above 2^31 are refused before anything is allocated for them
    big = torch.sparse_coo_tensor(_t(g, [[5], [0]]), _t(g, [1.0]), size=(2 ** 31, 1))
    free0 = torch.cuda.mem_get_info(rt.device)[0]
    from gauss_newton_via_generalized_krylov_subspaces_b200._lib import GnkError
    with pytest.raises(GnkError, match="2\\^31"):
        g.cg_least_squares(big, _t(g, np.zeros(4)))
    assert torch.cuda.mem_get_info(rt.device)[0] >= free0 - (64 << 20)


def test_library_holds_the_device_callable_kernels():
    """CPU: the sm_100a SASS of the shipped library carries the blocked SpMM and the pattern / gather kernels"""
    import __graft_entry__
    __graft_entry__.build()
    from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib
    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    for name in ("spmm_csr_kernelILi8E", "spmm_csr_kernelILi1E", "spmm_csr_kernelILi7E", "pattern_check_kernel",
                 "transpose_cols_kernel", "pattern_equal_kernel", "gather_kernel", "DeviceRadixSort"):
        assert name in sass, name
    for name in ("gnk_csr_pattern", "gnk_csr_pattern_equal", "gnk_csr_gather"):
        assert name in _lib.SIGNATURES
