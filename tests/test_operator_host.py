"""Matrix-free Jacobians on the CPU: scipy LinearOperators in gauss_newton_krylow and GeneralizedKrylowSubspace.update,
driven through the numpy mock of the C ABI (tests/mock_backend.py), against the oracle run on the SAME operator; the
argument checks of DeviceLinearOperator and autograd_jacobian on CPU tensors; the refusals of gauss_newton and
cg_least_squares; and the refusal of a multi-rank process group."""
import os
import socket
import sys

import numpy as np
import pytest
import scipy.sparse as sp
from scipy.sparse.linalg import LinearOperator, aslinearoperator

from golden_util import Golden, rel
from oracle import gnk_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture()
def g():
    import mock_backend
    mock_backend.install()
    import gauss_newton_via_generalized_krylov_subspaces_b200 as pkg
    yield pkg
    mock_backend.uninstall()


class Hand(LinearOperator):
    """a LinearOperator written by hand: only _matvec / _rmatvec, over any matrix-like A"""

    def __init__(self, A):
        super().__init__(np.float64, A.shape)
        self.A = A

    def _matvec(self, v):
        return self.A @ v

    def _rmatvec(self, u):
        return self.A.T @ u


class Counting(Hand):
    """records the width of every J @ V_k and the number of J^T u products"""

    def __init__(self, A, log):
        super().__init__(A)
        self.log = log

    def _matmat(self, X):
        self.log["matmat"].append(X.shape[1])
        return self.A @ X

    def _rmatvec(self, u):
        self.log["rmatvec"] += 1
        return self.A.T @ u


def _bratu(G=34, lam=10):
    gd = Golden(f"bratu_g{G}") if G in (34, 101) else Golden("bratu_g25_linear")
    o = orc.BratuOracle(G, 5, lam)
    return o.make_res(gd["y"]), gd["u0"], (lambda x, _j=o.make_jac(): _j(x).tocsr())


def _fit():
    """a random nonlinear least-squares fit: res(x) = A x + 0.1 (B x)^2 - y, J = A + 0.2 diag(B x) B, with a zero
    residual at the solution (with noise in y, the last Armijo tests of a run compare losses that differ in rounding
    only, and two correct implementations may count a trial more or less)"""
    rs = np.random.RandomState(3)
    A, B = rs.normal(size=(60, 20)), rs.normal(size=(60, 20)) / 5
    xt = rs.normal(size=20)
    y = A @ xt + 0.1 * (B @ xt) ** 2
    res = lambda x: A @ x + 0.1 * (B @ x) ** 2 - y  # noqa: E731
    jac = lambda x: A + 0.2 * (B @ x)[:, None] * B  # noqa: E731
    return res, xt + 0.3 * rs.normal(size=20), jac


def _run(g, res, x0, jac, capsys, **kw):
    xs = []
    out = g.gauss_newton_krylow(res, x0, jac, callback=lambda x, nfev, cg_iter: xs.append((np.array(x), nfev)), **kw)
    return out, xs, capsys.readouterr().out


def _oracle_kw(kw):
    ok = dict(restart=kw.get("krylow_restart"), max_iter=kw.get("max_iter", 100), version=kw.get("version", "res_old"),
              reorth=kw.get("reorth_passes", 1))
    if kw.get("ls_solver") == "cgls":
        ok["ls"] = lambda A, y, log: orc.cgls(A, y, rtol=kw.get("cg_rtol", 1e-4), preconditioner=True)[0]
    return ok


def _check_against_oracle(g, capsys, res, x0, jac_csr, wrap, **kw):
    """the operator run against the oracle on the same operator (counters, iterates within 1e-12, nfev per callback)
    and against the package's CSR run of the same Jacobian (the same printed messages)"""
    jac = lambda x: wrap(jac_csr(x))  # noqa: E731
    out, xs, printed = _run(g, res, x0, jac, capsys, **kw)
    xo = []
    ref = orc.gnk(res, x0, jac, callback=lambda x, nfev, cg_iter: xo.append((x.copy(), nfev)), **_oracle_kw(kw))
    assert (out.nit, out.nrev, out.njev, bool(out.success)) == (ref["nit"], ref["nfev"], ref["njev"], ref["success"])
    assert [n for _, n in xs] == [n for _, n in xo]
    tol = 1e-6 if kw.get("ls_solver") == "cgls" else 1e-12
    assert max(rel(a, b) for (a, _), (b, _) in zip(xs, xo)) < tol
    assert rel(out.x, ref["x"]) < tol
    csr, _, printed_csr = _run(g, res, x0, jac_csr, capsys, **kw)
    assert printed == printed_csr
    assert (csr.nit, csr.nrev, csr.njev) == (out.nit, out.nrev, out.njev)
    return out, printed


@pytest.mark.parametrize("wrap", [aslinearoperator, Hand], ids=["aslinearoperator", "hand_written"])
@pytest.mark.parametrize("kw", [dict(max_iter=30), dict(max_iter=30, version="res_new"),
                                dict(max_iter=25, version="jac_old_res_old"),
                                dict(max_iter=25, version="jac_old_res_new"),
                                dict(max_iter=40, krylow_restart=7), dict(max_iter=30, reorth_passes=2),
                                dict(max_iter=20, krylow_restart=9, ls_solver="cgls", cg_rtol=1e-12)],
                         ids=["res_old", "res_new", "jac_old_res_old", "jac_old_res_new", "restart7", "cgs2", "cgls"])
def test_bratu_operator_against_oracle(g, capsys, wrap, kw):
    res, x0, jac = _bratu()
    _check_against_oracle(g, capsys, res, x0, jac, wrap, **kw)


@pytest.mark.parametrize("wrap", [aslinearoperator, Hand], ids=["aslinearoperator", "hand_written"])
@pytest.mark.parametrize("version", ["res_old", "res_new", "jac_old_res_old", "jac_old_res_new"])
def test_nonlinear_fit_operator_against_oracle(g, capsys, wrap, version):
    res, x0, jac = _fit()
    out, printed = _check_against_oracle(g, capsys, res, x0, jac, wrap, max_iter=40, version=version)
    assert out.nit >= 20  # the basis reached the whole 20-dimensional space on the way


def test_breakdown_with_the_host_mirror(g, capsys):
    """compare_linear_small (G = 25, LAMBDA = 0) breaks down at iteration 2: the deferred flag retracts the column that
    the next J @ V_k already saw, and the mirror follows the retraction"""
    res, x0, jac = _bratu(25, 0)
    outs = []
    for wrap in (aslinearoperator, Hand, None):
        try:
            out, xs, printed = _run(g, res, x0, (lambda x: wrap(jac(x))) if wrap else jac, capsys, max_iter=12)
            outs.append(((out.nit, out.nrev, out.njev, bool(out.success)), xs, printed))
        except g.StepLengthConvergenceError as e:
            outs.append((("step", str(e)), [], capsys.readouterr().out))
    assert "Generalized krylow subspace breakdown at iteration = 2, basis.shape = (576, 2)" in outs[-1][2]
    for got in outs[:2]:
        assert got[0] == outs[-1][0] and got[2] == outs[-1][2]
        assert [n for _, n in got[1]] == [n for _, n in outs[-1][1]]
        assert all(rel(a, b) < 1e-12 for (a, _), (b, _) in zip(got[1], outs[-1][1]))


@pytest.mark.parametrize("kw", [dict(max_iter=30), dict(max_iter=40, krylow_restart=7),
                                dict(max_iter=25, version="jac_old_res_new")], ids=["no_restart", "restart7", "jac_old"])
def test_call_counts_and_basis_downloads(g, capsys, kw):
    """one J @ V_k per outer iteration with the oracle's k, one J^T u per expansion, and 8 p bytes of basis download
    per appended column plus one column per restart"""
    res, x0, jac = _bratu()
    p = x0.shape[0]
    log, olog = dict(matmat=[], rmatvec=0), dict(matmat=[], rmatvec=0)
    rt = g.get_runtime()
    real = rt.download
    basis_bytes = [0]

    def download(t):
        if t.dim() == 2:  # only the basis mirror downloads 2-D blocks (columns of V_k)
            basis_bytes[0] += 8 * t.numel()
        return real(t)

    rt.download = download
    try:
        out, _, _ = _run(g, res, x0, lambda x: Counting(jac(x), log), capsys, **kw)
    finally:
        rt.download = real
    trace = []
    ref = orc.gnk(res, x0, lambda x: Counting(jac(x), olog), trace=trace, **_oracle_kw(kw))
    assert out.nit == ref["nit"]
    ks = [t["k"] for t in trace]
    assert log["matmat"] == olog["matmat"] == ks
    assert log["rmatvec"] == olog["rmatvec"] > 0
    new_cols = sum(k - prev if k >= prev else k for prev, k in zip([0] + ks[:-1], ks))
    assert basis_bytes[0] == 8 * p * new_cols
    if "krylow_restart" in kw:
        assert new_cols > max(ks) * 2  # the column 0 of every restart was downloaded again


def test_writes_and_shapes_are_refused(g):
    res, x0, jac = _bratu()

    class Writes(Hand):
        def _matmat(self, X):
            X[0, 0] = 1.0
            return self.A @ X

    with pytest.raises(ValueError, match="read-only"):
        g.gauss_newton_krylow(res, x0, lambda x: Writes(jac(x)), max_iter=5, callback=lambda **k: None)
    p = x0.shape[0]
    with pytest.raises(ValueError, match=rf"expected a LinearOperator of shape \({p}, {p}\).*got \({p}, {p + 1}\)"):
        g.gauss_newton_krylow(res, x0, lambda x: aslinearoperator(sp.hstack([jac(x), sp.csr_array((p, 1))])),
                              max_iter=5, callback=lambda **k: None)


def test_standalone_update_with_an_operator(g):
    rs = np.random.RandomState(1)
    A = sp.random(70, 40, density=0.2, random_state=rs, format="csr")
    x0, r = rs.normal(size=40), rs.normal(size=70)
    bases = []
    for J in (A, aslinearoperator(A), Hand(A)):
        kr = g.GeneralizedKrylowSubspace()
        kr.start(x0)
        kr.update(J, r)
        kr.update(J, 2 * r + 1)
        bases.append(kr.basis)
    assert bases[0].shape == (40, 3)
    assert rel(bases[1], bases[0]) < 1e-14 and rel(bases[2], bases[0]) < 1e-14
    kr = g.GeneralizedKrylowSubspace()
    kr.start(x0)
    with pytest.raises(ValueError, match=r"shape \(70, 40\)"):
        kr.update(aslinearoperator(A.T), r)


def test_gauss_newton_and_cg_least_squares_refuse_operators(g):
    res, x0, jac = _fit()
    with pytest.raises(TypeError, match="MatrixLinearOperator.*gauss_newton_krylow"):
        g.gauss_newton(res, x0, lambda x: aslinearoperator(jac(x)), callback=lambda **k: None)
    with pytest.raises(TypeError, match="Hand"):
        g.gauss_newton(res, x0, lambda x: Hand(jac(x)), callback=lambda **k: None)
    with pytest.raises(TypeError, match="cg_least_squares"):
        g.cg_least_squares(aslinearoperator(jac(x0)), res(x0))
    import torch
    op = g.DeviceLinearOperator((60, 20), matvec=lambda v: v, rmatvec=lambda u: u)
    with pytest.raises(TypeError, match="DeviceLinearOperator"):
        g.cg_least_squares(op, torch.zeros(60, dtype=torch.float64))


# ------------------------------------------------------------------------------------------------
# DeviceLinearOperator / autograd_jacobian: argument checks and products on CPU tensors (the solver path is on the GPU)
# ------------------------------------------------------------------------------------------------
def test_device_linear_operator_checks():
    import torch
    from gauss_newton_via_generalized_krylov_subspaces_b200 import DeviceLinearOperator
    A = torch.arange(12, dtype=torch.float64).reshape(4, 3)
    V = torch.ones(3, 2, dtype=torch.float64)
    op = DeviceLinearOperator((4, 3), matvec=lambda v: A @ v, rmatvec=lambda u: A.T @ u)
    assert torch.equal(op.matmat(V), A @ V) and torch.equal(op.rmatvec(torch.ones(4, dtype=torch.float64)), A.sum(0))
    assert op.matvec(V[:, 0]).dtype == torch.float64
    only_mm = DeviceLinearOperator((4, 3), matmat=lambda X: (A @ X).float(), rmatvec=lambda u: A.T @ u)
    assert only_mm.matvec(V[:, 0]).dtype == torch.float64 and torch.equal(only_mm.matvec(V[:, 0]), A @ V[:, 0])
    with pytest.raises(TypeError, match="rmatvec is required"):
        DeviceLinearOperator((4, 3), matvec=lambda v: A @ v)
    with pytest.raises(TypeError, match="matvec, matmat"):
        DeviceLinearOperator((4, 3), rmatvec=lambda u: A.T @ u)
    with pytest.raises(ValueError, match="shape must be"):
        DeviceLinearOperator((4, 3, 1), matvec=lambda v: v, rmatvec=lambda u: u)
    bad = DeviceLinearOperator((4, 3), matvec=lambda v: (A @ v)[:3], rmatvec=lambda u: (A.T @ u)[:, None])
    with pytest.raises(ValueError, match=r"matvec: expected shape \(4,\), got \(3,\)"):
        bad.matmat(V)  # the default matmat goes through matvec
    with pytest.raises(ValueError, match=r"matmat: expected shape \(4, 2\), got \(3, 2\)"):
        DeviceLinearOperator((4, 3), matmat=lambda X: (A @ X)[:3], rmatvec=lambda u: u).matmat(V)
    with pytest.raises(ValueError, match=r"expected shape \(3,\), got \(3, 1\)"):
        bad.rmatvec(torch.ones(4, dtype=torch.float64))
    with pytest.raises(ValueError, match=r"matvec: v: expected shape \(3,\), got \(4,\)"):
        op.matvec(torch.ones(4, dtype=torch.float64))
    with pytest.raises(TypeError, match="ndarray"):
        DeviceLinearOperator((4, 3), matvec=lambda v: (A @ v).numpy(), rmatvec=lambda u: u).matvec(V[:, 0])
    with pytest.raises(TypeError, match="floating-point"):
        DeviceLinearOperator((4, 3), matvec=lambda v: (A @ v).long(), rmatvec=lambda u: u).matvec(V[:, 0])


def test_autograd_jacobian_products_on_cpu():
    """J V by vmap over jvp and J^T u by vjp, on the pure-torch Bratu residual, against the assembled Jacobian"""
    import torch
    from torch_bratu import TorchBratu
    from gauss_newton_via_generalized_krylov_subspaces_b200 import BratuPdeProblem, autograd_jacobian
    o = orc.BratuOracle(21, 5, 10)
    tb = TorchBratu(BratuPdeProblem(21, 5, 10), o, o.operator(o.u_true), "cpu")
    u = o.start_vector()
    op = autograd_jacobian(lambda x, s: s * tb.res(x))(torch.from_numpy(u), 2.0)
    J = 2.0 * o.make_jac()(u).tocsr().toarray()
    assert op.shape == (o.n, o.n)
    V = torch.from_numpy(np.random.RandomState(0).normal(size=(o.n, 5)))
    r = torch.from_numpy(np.random.RandomState(1).normal(size=o.n))
    assert rel(op.matmat(V).numpy(), J @ V.numpy()) < 1e-13
    assert rel(op.matvec(V[:, 1]).numpy(), J @ V[:, 1].numpy()) < 1e-13
    assert rel(op.rmatvec(r).numpy(), J.T @ r.numpy()) < 1e-13


# ------------------------------------------------------------------------------------------------
# several ranks: operators belong to replicated problems, which a multi-rank process group refuses
# ------------------------------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _rank_worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import mock_backend
    mock_backend.install()
    import gauss_newton_via_generalized_krylov_subspaces_b200 as g
    from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib
    res, x0, jac = _fit()
    msgs = []
    for call in (lambda: g.gauss_newton_krylow(res, x0, lambda x: aslinearoperator(jac(x)), callback=lambda **k: None),
                 lambda: g.GeneralizedKrylowSubspace().start(x0)):
        try:
            call()
            msgs.append("")
        except _lib.GnkError as e:
            msgs.append(str(e))
    np.save(os.path.join(out_dir, f"r{rank}.npy"), np.array(msgs))
    dist.barrier()
    dist.destroy_process_group()


def test_operators_refuse_a_multi_rank_process_group(tmp_path):
    import torch.multiprocessing as mp
    mp.spawn(_rank_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    for r in range(2):
        msgs = np.load(os.path.join(tmp_path, f"r{r}.npy"))
        assert len(msgs) == 2 and all("not row-sharded" in m for m in msgs), msgs
