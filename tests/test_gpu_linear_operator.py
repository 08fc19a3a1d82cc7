"""Matrix-free Jacobians on the B200: scipy LinearOperators with host x0 (the basis mirrored to the host, J V_k uploaded)
and DeviceLinearOperator / autograd_jacobian with a CUDA-tensor x0 (J V_k formed by the user's torch code on a view
of the basis), against the reference's goldens and the oracle with the criteria the CSR paths are held to."""
import numpy as np
import pytest
from scipy.sparse.linalg import LinearOperator, aslinearoperator

from golden_util import Golden, Recorder, check_trace  # noqa: E402
from oracle import gnk_oracle as orc  # noqa: E402

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def g():
    import gauss_newton_via_generalized_krylov_subspaces_b200 as pkg
    import gauss_newton_via_generalized_krylov_subspaces_b200.device as device
    device._runtime = None
    pkg.get_runtime()
    return pkg


def _t(g, a):
    import torch
    return torch.as_tensor(np.asarray(a), device=g.get_runtime().device)


def _torch_bratu(g, G, y):
    from torch_bratu import TorchBratu
    return TorchBratu(g.BratuPdeProblem(G, 5, 10), orc.BratuOracle(G, 5, 10), y, g.get_runtime().device)


class Counting(LinearOperator):
    def __init__(self, A, log):
        super().__init__(np.float64, A.shape)
        self.A, self.log = A, log

    def _matvec(self, v):
        return self.A @ v

    def _matmat(self, X):
        self.log["matmat"].append(X.shape[1])
        return self.A @ X

    def _rmatvec(self, u):
        self.log["rmatvec"] += 1
        return self.A.T @ u


def _golden_check(out, rec, gr, restart):
    n = len(gr["xnorm"])
    check_trace(rec, gr, 1e-10, upto=n if restart is None else min(n, restart))
    check_trace(rec, gr, 1e-10 if restart is None else 1e-8)
    assert (out.nit, out.nrev, out.njev, bool(out.success)) == (
        int(gr["nit"]), int(gr["nfev"]), int(gr["njev"]), bool(gr["success"]))


# ------------------------------------------------------------------------------------------------
# host LinearOperators
# ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("rname,kw", [("gnk_res_old", dict(max_iter=100)),
                                      ("gnk_res_new", dict(max_iter=100, version="res_new")),
                                      ("gnk_restart30", dict(max_iter=100, krylow_restart=30))])
def test_bratu_g101_host_operator_against_goldens(g, rname, kw):
    gd = Golden("bratu_g101")
    gr = gd.run(rname)
    o = orc.BratuOracle(101, 5, 10)
    rec = Recorder(gr["sample_idx"], o.make_error())
    jac = lambda x, _j=o.make_jac(): aslinearoperator(_j(x).tocsr())  # noqa: E731
    out = g.gauss_newton_krylow(o.make_res(gd["y"]), gd["u0"], jac, callback=rec, **kw)
    _golden_check(out, rec, gr, kw.get("krylow_restart"))
    assert isinstance(out.x, np.ndarray)


@gpu
def test_bratu_g41_host_operator_wide_basis(g):
    """no restart, 311 iterations: the mirror grows past 255 columns and the panel goes to gnk_basis_ls_wide"""
    o = orc.BratuOracle(41, 5, 10)
    y, u0 = o.operator(o.u_true), o.start_vector(seed=42)
    idx = np.random.RandomState(0).choice(o.n, 64, replace=False)
    rtrace, trace = [], []
    ref = orc.gnk(o.make_res(y), u0, o.make_jac(), restart=None, max_iter=700,
                  callback=lambda x, **kw: rtrace.append(np.asarray(x)[idx].copy()))
    assert (ref["nit"], ref["nfev"], ref["njev"], ref["success"]) == (311, 312, 311, True)
    jac = lambda x, _j=o.make_jac(): aslinearoperator(_j(x).tocsr())  # noqa: E731
    out = g.gauss_newton_krylow(o.make_res(y), u0, jac, max_iter=700, max_basis_columns=400,
                                callback=lambda x, **kw: trace.append(np.asarray(x)[idx].copy()))
    assert (out.nit, out.nrev, out.njev, out.success) == (311, 312, 311, True)
    dev = np.array([np.max(np.abs(a - b)) / np.max(np.abs(b)) for a, b in zip(trace, rtrace)])
    print(f"G=41 host operator, wide: max deviation through 255 {dev[:255].max():.2e}, 256..311 {dev[255:].max():.2e}")
    assert dev.max() < 1e-10


@gpu
def test_host_operator_call_counts(g):
    gd = Golden("bratu_g101")
    o = orc.BratuOracle(101, 5, 10)
    log, olog, trace = dict(matmat=[], rmatvec=0), dict(matmat=[], rmatvec=0), []
    J = o.make_jac()
    out = g.gauss_newton_krylow(o.make_res(gd["y"]), gd["u0"], lambda x: Counting(J(x).tocsr(), log), max_iter=30,
                                krylow_restart=12, callback=lambda **k: None)
    ref = orc.gnk(o.make_res(gd["y"]), gd["u0"], lambda x: Counting(J(x).tocsr(), olog), restart=12, max_iter=30,
                  trace=trace)
    assert out.nit == ref["nit"]
    assert log["matmat"] == olog["matmat"] == [t["k"] for t in trace]
    assert log["rmatvec"] == olog["rmatvec"] > 0


# ------------------------------------------------------------------------------------------------
# device operators
# ------------------------------------------------------------------------------------------------
def _csr_operator(g, tb, log=None):
    """jac(x) -> DeviceLinearOperator over the torch CSR Jacobian of TorchBratu"""

    def jac(x):
        J = tb.jac(x)

        def matvec(v):
            return J @ v

        def matmat(V):
            if log is not None:
                log["matmat"].append(V.shape[1])
            return J @ V

        def rmatvec(u):
            if log is not None:
                log["rmatvec"] += 1
            return J.t() @ u

        return g.DeviceLinearOperator(J.shape, matvec=matvec, rmatvec=rmatvec, matmat=matmat if log else None)

    return jac


@gpu
@pytest.mark.parametrize("kind", ["csr_operator", "autograd"])
@pytest.mark.parametrize("rname,kw", [("gnk_res_old", dict(max_iter=100)),
                                      ("gnk_res_new", dict(max_iter=100, version="res_new")),
                                      ("gnk_jac_old_res_old", dict(max_iter=25, version="jac_old_res_old")),
                                      ("gnk_jac_old_res_new", dict(max_iter=25, version="jac_old_res_new")),
                                      ("gnk_restart30", dict(max_iter=100, krylow_restart=30))])
def test_bratu_g101_device_operator_against_goldens(g, kind, rname, kw):
    import torch
    gd = Golden("bratu_g101")
    tb = _torch_bratu(g, 101, gd["y"])
    gr = gd.run(rname)
    o = orc.BratuOracle(101, 5, 10)
    rec = Recorder(gr["sample_idx"], o.make_error())
    jac = _csr_operator(g, tb) if kind == "csr_operator" else g.autograd_jacobian(tb.res)
    kept = []

    def cb(x, nfev, cg_iter):
        kept.append(isinstance(x, torch.Tensor) and x.is_cuda)
        rec(x.cpu().numpy(), nfev, cg_iter)

    out = g.gauss_newton_krylow(tb.res, _t(g, gd["u0"]), jac, callback=cb, **kw)
    _golden_check(out, rec, gr, kw.get("krylow_restart"))
    assert all(kept) and isinstance(out.x, torch.Tensor) and out.x.is_cuda and out.x.dtype == torch.float64


@gpu
@pytest.mark.parametrize("version", ["res_old", "jac_old_res_new"])
def test_device_operator_call_counts(g, version):
    gd = Golden("bratu_g101")
    tb = _torch_bratu(g, 101, gd["y"])
    o = orc.BratuOracle(101, 5, 10)
    log, olog, trace = dict(matmat=[], rmatvec=0), dict(matmat=[], rmatvec=0), []
    out = g.gauss_newton_krylow(tb.res, _t(g, gd["u0"]), _csr_operator(g, tb, log), max_iter=30, krylow_restart=12,
                                version=version, callback=lambda **k: None)
    J = o.make_jac()
    ref = orc.gnk(o.make_res(gd["y"]), gd["u0"], lambda x: Counting(J(x).tocsr(), olog), restart=12, max_iter=30,
                  version=version, trace=trace)
    assert out.nit == ref["nit"] and tb.jac_calls == ref["njev"]
    assert log["matmat"] == olog["matmat"] == [t["k"] for t in trace]
    assert log["rmatvec"] == olog["rmatvec"] > 0


@gpu
def test_in_place_refill_equals_fresh_operators(g):
    """jac refills ONE preallocated state in place at every call; with jac_old_res_old the expansion needs J_old,
    whose -J_old^T r is formed before jac is called at the new point: the result equals fresh operators bit for bit"""
    import torch
    gd = Golden("bratu_g101")
    tb = _torch_bratu(g, 101, gd["y"])
    state = {}

    def jac_in_place(x):
        J = tb.jac(x)
        if "J" not in state:
            state["J"] = J
        else:
            state["J"].values().copy_(J.values())
        S = state["J"]
        return g.DeviceLinearOperator(S.shape, matvec=lambda v: S @ v, rmatvec=lambda u: S.t() @ u)

    outs = []
    for jac in (_csr_operator(g, tb), jac_in_place):
        xs = []
        out = g.gauss_newton_krylow(tb.res, _t(g, gd["u0"]), jac, max_iter=25, version="jac_old_res_old",
                                    callback=lambda x, nfev, cg_iter: xs.append((x.cpu().numpy(), nfev)))
        outs.append(((out.nit, out.nrev, out.njev, bool(out.success)), xs, out.x.cpu().numpy()))
    (ca, xa, fa), (cb_, xb, fb) = outs
    assert ca == cb_ and [n for _, n in xa] == [n for _, n in xb]
    assert all(np.array_equal(a, b) for (a, _), (b, _) in zip(xa, xb)) and np.array_equal(fa, fb)
    assert isinstance(state["J"], torch.Tensor)


@gpu
def test_device_operator_errors(g):
    import torch
    rt = g.get_runtime()
    A = _t(g, np.array([[1.0, 2.0], [0.0, 1.0], [3.0, -1.0]]))
    res = lambda x: A @ x - 1.0  # noqa: E731
    x0 = _t(g, [1.0, 1.0])

    def op(matvec=lambda v: A @ v, rmatvec=lambda u: A.T @ u, shape=(3, 2)):
        return lambda x: g.DeviceLinearOperator(shape, matvec=matvec, rmatvec=rmatvec)

    with pytest.raises(ValueError, match=f"expected a tensor on {rt.device}, got one on cpu"):
        g.gauss_newton_krylow(res, x0, op(matvec=lambda v: (A @ v).cpu()), callback=lambda **k: None)
    with pytest.raises(ValueError, match=f"expected a tensor on {rt.device}, got one on cpu"):
        g.gauss_newton_krylow(res, x0, op(rmatvec=lambda u: (A.T @ u).cpu()), callback=lambda **k: None)
    with pytest.raises(ValueError, match=r"expected shape \(2,\), got \(1,\)"):
        g.gauss_newton_krylow(res, x0, op(rmatvec=lambda u: (A.T @ u)[:1]), callback=lambda **k: None)
    with pytest.raises(ValueError, match=r"expected shape \(3,\), got \(4,\)"):
        g.gauss_newton_krylow(res, x0, op(matvec=lambda v: torch.cat([A @ v, A[:1] @ v])), callback=lambda **k: None)
    with pytest.raises(ValueError, match=r"shape \(3, 2\) \(n_res, p\), got \(2, 3\)"):
        g.gauss_newton_krylow(res, x0, op(shape=(2, 3)), callback=lambda **k: None)
    with pytest.raises(TypeError, match="DeviceLinearOperator.*gauss_newton_krylow"):
        g.gauss_newton(res, x0, op(), callback=lambda **k: None)
    # float32 products are converted
    out = g.gauss_newton_krylow(res, x0, op(matvec=lambda v: (A @ v).float()), max_iter=3, callback=lambda **k: None)
    assert out.x.dtype == torch.float64 and out.x.is_cuda
