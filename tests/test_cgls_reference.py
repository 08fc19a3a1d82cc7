"""cg_least_squares without a GPU: the high-precision CG reference that tests/test_gpu_cgls.py holds the device loop to,
and the host routing of a transposed Bratu Jacobian (through tests/mock_backend.py, which mirrors gnk_cgls_x0).

The reference restates scipy's ``cg`` exactly as ``oracle.gnk_oracle.pcg`` does (x0 = 0 or the given x0, r = b - M x0,
stopping test ||r_j|| < rtol ||b|| at the top of iteration j, maxiter = 10 p) but runs without the stopping test and
records ||r_j|| and x_j for every j, in float64 and in np.longdouble.  From the longdouble history one can pick
thresholds at which the iteration count is determined with a known margin; from the float64-vs-longdouble gap of x_j a
per-iteration tolerance for the iterate (the ``sensitivity_bound`` idea of tests/golden_util.py).
"""
import numpy as np
import pytest
import scipy.sparse as sp

from golden_util import rel
from oracle import gnk_oracle as orc

LD = np.longdouble
LD_OK = np.finfo(LD).eps < 1e-18  # x86-64: 80-bit extended, eps 1.08e-19
SEP = 1.001                        # min_{i<j} ||r_i|| / ||r_j|| that makes j a threshold candidate


# ------------------------------------------------------------------------------------------------
# reference
# ------------------------------------------------------------------------------------------------
def csr_matvec(A, x, dtype):
    """A @ x with every product and sum in ``dtype`` (row by row in index order); rows without entries give 0
    (np.add.reduceat would return the next row's first product for them)"""
    out = np.zeros(A.shape[0], dtype=dtype)
    if A.nnz:
        prod = A.data.astype(dtype) * np.asarray(x, dtype=dtype)[A.indices]
        full = np.diff(A.indptr) > 0
        out[full] = np.add.reduceat(prod, A.indptr[:-1][full])
    return out


class NormalEq:
    """A^T A v, A^T y and the Jacobi diagonal diag(A^T A) of an assembled matrix, in ``dtype``"""

    def __init__(self, A, dtype):
        A = sp.csr_array(A, dtype=np.float64)
        A.sum_duplicates()
        A.sort_indices()
        self.A, self.AT, self.dtype = A, sp.csr_array(A.T), dtype
        self.AT.sort_indices()

    def mv(self, v):
        if self.dtype == np.float64:  # scipy's csr_matvec: the same order, compiled
            return self.AT @ (self.A @ v)
        return csr_matvec(self.AT, csr_matvec(self.A, v, self.dtype), self.dtype)

    def rmv(self, y):
        return self.AT @ y if self.dtype == np.float64 else csr_matvec(self.AT, y, self.dtype)

    def diag(self):
        sq = sp.csr_array((np.ones(self.AT.nnz), self.AT.indices, self.AT.indptr), shape=self.AT.shape)
        sq.data = self.AT.data.astype(self.dtype) ** 2
        return csr_matvec(sq, np.ones(self.AT.shape[1]), self.dtype)


def pcg_history(ne, b, minv, nmax, x0=None, keep=None, stop=0.0):
    """oracle.pcg (scipy cg) for nmax iterations without the stopping test (or until ||r_j|| < stop).  Returns (rn, xs):
    rn[j] = ||r_j|| at the top of iteration j (j = 0 .. nmax), xs[j] = x_j as float64 for j in ``keep`` (every j if
    keep is None)."""
    dt = ne.dtype
    if x0 is None:
        x = np.zeros(b.shape[0], dtype=dt)
        r = b.copy()
    else:
        x = np.asarray(x0, dtype=np.float64).astype(dt)
        r = b - ne.mv(x)
    rn = np.zeros(nmax + 1)
    xs = {}
    p = rho_prev = None
    for it in range(nmax + 1):
        rn[it] = float(np.sqrt(np.dot(r, r)))
        if keep is None or it in keep:
            xs[it] = x.astype(np.float64)
        if it == nmax or not rn[it] > stop:  # r = 0 exactly (or lost): nothing beyond is defined
            rn = rn[:it + 1]
            break
        z = r if minv is None else minv * r
        rho = np.dot(r, z)
        p = z.copy() if it == 0 else p * (rho / rho_prev) + z
        q = ne.mv(p)
        a = rho / np.dot(p, q)
        x = x + a * p
        r = r - a * q
        rho_prev = rho
    return rn, xs


def first_below(rn, atol):
    """(j, margin): the count scipy's cg returns for this atol (the first j with rn[j] < atol; None past the history)
    and how far atol is from both sides of the decision, min(atol / rn[j], min_{i<j} rn[i] / atol) - 1"""
    below = np.nonzero(rn < atol)[0]
    if below.size == 0:
        return None, 0.0
    j = int(below[0])
    hi = float(np.min(rn[:j])) / atol if j else np.inf
    return j, min(atol / rn[j], hi) - 1.0


def separated(rn):
    """{j: atol_j} for every j >= 1 with min_{i<j} rn[i] / rn[j] >= SEP; atol_j = sqrt(min_{i<j} rn[i] * rn[j]) sits
    in the middle (geometrically) of the gap, so the count for atol_j is exactly j"""
    out = {}
    run = np.minimum.accumulate(rn)
    for j in range(1, rn.shape[0]):
        m = run[j - 1]
        if m / rn[j] >= SEP:
            out[j] = float(np.sqrt(m * rn[j]))
    return out


class CgReference:
    """cg_least_squares(A, y, x0, rtol, preconditioner) of the reference (gauss_newton.py:11-60) as histories.

    ``passes``: one history per CG run (the unpreconditioned one first when preconditioner=False).  ``hi`` is the
    longdouble arm when ``longdouble`` (and the host has it), else float64; ``lo`` is always float64.  ``dev[k][j]`` =
    max_{i<=j} |rn_lo - rn_hi| / rn_hi of pass k."""

    def __init__(self, A, y, preconditioner, x0=None, nmax=None, longdouble=True, stop_rtol=0.0):
        self.A = sp.csr_array(A)
        self.p = self.A.shape[1]
        self.maxiter = 10 * self.p
        self.nmax = self.maxiter if nmax is None else min(nmax, self.maxiter)
        self.x0 = x0
        self.y = np.asarray(y, dtype=np.float64)
        self.precise = bool(longdouble and LD_OK)
        self.ne = {"lo": NormalEq(self.A, np.float64), "hi": NormalEq(self.A, LD if self.precise else np.float64)}
        self.b = {k: ne.rmv(self.y) for k, ne in self.ne.items()}
        self.bn = float(np.sqrt(np.dot(self.b["hi"], self.b["hi"])))
        self.minv = ([None] if not preconditioner else []) + [1.0 / self.ne["hi"].diag()]
        self.minv_lo = ([None] if not preconditioner else []) + [1.0 / self.ne["lo"].diag()]
        self.rn = {"hi": [], "lo": []}
        stop = stop_rtol * self.bn
        for mi, ml in zip(self.minv, self.minv_lo):
            self.rn["hi"].append(pcg_history(self.ne["hi"], self.b["hi"], mi, self.nmax, x0, keep=(), stop=stop)[0])
            self.rn["lo"].append(pcg_history(self.ne["lo"], self.b["lo"], ml, self.nmax, x0, keep=(), stop=stop)[0]
                                 if self.precise else self.rn["hi"][-1])
        self.dev = []
        for lo, hi in zip(self.rn["lo"], self.rn["hi"]):
            n = min(lo.shape[0], hi.shape[0])
            d = np.maximum.accumulate(np.abs(lo[:n] - hi[:n]) / hi[:n])
            self.dev.append(np.concatenate([d, np.full(hi.shape[0] - n, np.inf)]))

    def counts(self, atol):
        """[(j, margin, dev_j)] per pass for this atol"""
        out = []
        for k, rn in enumerate(self.rn["hi"]):
            j, mg = first_below(rn, atol)
            out.append((j, mg, None if j is None else float(self.dev[k][j])))
        return out

    def iterate(self, j):
        """(x_j of the last pass in the precise arm, its per-entry tolerance max(1e-12, 10 |x_j(fp64) - x_j(hi)| /
        |x_j|), both max-norm relative)"""
        xh = pcg_history(self.ne["hi"], self.b["hi"], self.minv[-1], j, self.x0, keep={j})[1][j]
        if not self.precise:
            return xh, None
        xl = pcg_history(self.ne["lo"], self.b["lo"], self.minv_lo[-1], j, self.x0, keep={j})[1][j]
        return xh, max(1e-12, 10.0 * rel(xl, xh))

    def thresholds(self, targets, min_margin=None, default_rtol=1e-4):
        """rtol values at which every pass's count is decided with margin >= max(min_margin, 100 x dev): for each target
        count (of the LAST pass) the nearest separated j at or above it, plus ``default_rtol`` itself when it is.
        Returns [(rtol, total count, last-pass count)]."""
        cand = separated(self.rn["hi"][-1])
        picks, seen = [], set()

        def ok(atol):
            cs = self.counts(atol)
            if any(j is None for j, _, _ in cs):
                return None
            need = [max(min_margin or 0.0, 100.0 * d) for _, _, d in cs]
            if all(mg >= nd for (_, mg, _), nd in zip(cs, need)):
                return cs
            return None

        for t in targets:
            for j in sorted(cand):
                if j < t:
                    continue
                cs = ok(cand[j])
                if cs is not None:
                    if j not in seen:
                        seen.add(j)
                        picks.append((cand[j] / self.bn, sum(c[0] for c in cs), cs[-1][0]))
                    break
        cs = ok(default_rtol * self.bn)
        if cs is not None and cs[-1][0] not in seen:
            picks.append((default_rtol, sum(c[0] for c in cs), cs[-1][0]))
        return picks


# ------------------------------------------------------------------------------------------------
# the matrices of the device tests (built on the host, deterministic)
# ------------------------------------------------------------------------------------------------
def random_sparse(n_res, p, seed, per_row=6, empty_rows=0, long_col=False):
    """n_res x p CSR with ~per_row entries a row, a strong entry in every column (no empty column: diag(A^T A) > 0),
    ``empty_rows`` rows without entries and, with ``long_col``, one column that is full but for those rows (a row of
    A^T with ~n_res entries)"""
    rs = np.random.RandomState(seed)
    empty = rs.choice(n_res, size=empty_rows, replace=False)
    live = np.setdiff1d(np.arange(n_res), empty)
    rows = [rs.choice(live, size=n_res * per_row), live[rs.permutation(np.arange(p) % live.shape[0])]]
    cols = [rs.randint(0, p, size=n_res * per_row), np.arange(p)]
    vals = [rs.normal(size=n_res * per_row), 4.0 + rs.rand(p)]
    if long_col:
        rows.append(live)
        cols.append(np.full(live.shape[0], p // 3))
        vals.append(0.05 * rs.normal(size=live.shape[0]))
    A = sp.coo_array((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(n_res, p)).tocsr()
    A.sort_indices()
    return sp.csr_array(A)


def graded_maxiter_problem():
    """40 x 20, singular values 1 .. 1e-6, rtol 1e-18 (below what float64 can reach, so that no rounding order stops
    early): scipy's cg runs into maxiter = 200 in both passes.  (With singular values down to 1e-8 the end point depends
    on rounding so much that one ulp of y moves ||A^T(y - A x)|| by 14x; here the spread is ~4x.)"""
    rs = np.random.RandomState(0)
    p, n = 20, 40
    U, _ = np.linalg.qr(rs.normal(size=(n, p)))
    V, _ = np.linalg.qr(rs.normal(size=(p, p)))
    A = sp.csr_array((U * np.logspace(0, -6, p)) @ V.T)
    return A, rs.normal(size=n), 1e-18


# ------------------------------------------------------------------------------------------------
# CPU tests of the reference itself
# ------------------------------------------------------------------------------------------------
def test_csr_matvec_handles_empty_rows_and_longdouble():
    A = random_sparse(300, 120, 3, empty_rows=17, long_col=True)
    assert np.sum(np.diff(A.indptr) == 0) == 17
    x = np.random.RandomState(4).normal(size=120)
    assert rel(csr_matvec(A, x, np.float64), A @ x) < 1e-14
    got = csr_matvec(A, x, LD)
    assert got.dtype == LD and np.all(got[np.diff(A.indptr) == 0] == 0)
    assert rel(got.astype(np.float64), A @ x) < 1e-14


@pytest.mark.parametrize("precond", [True, False])
def test_history_reproduces_the_oracle_cg(precond):
    """the float64 arm with the stopping test applied afterwards is oracle.cgls, iteration for iteration"""
    o = orc.BratuOracle(12, 5, 10)
    u = 0.2 * np.random.RandomState(1).normal(size=o.n)
    y = np.random.RandomState(2).normal(size=o.n)
    A = (-1 * o.make_jac()(u).tocsr())
    ref = CgReference(A, y, precond, longdouble=False)
    for rtol in (1e-2, 1e-4, 1e-8):
        x_orc, it_orc = orc.cgls(A, y, rtol=rtol, preconditioner=precond)
        cs = [first_below(rn, rtol * ref.bn)[0] for rn in ref.rn["lo"]]
        assert sum(cs) == it_orc
        xl = pcg_history(ref.ne["lo"], ref.b["lo"], ref.minv_lo[-1], cs[-1], keep={cs[-1]})[1][cs[-1]]
        assert rel(xl, x_orc) < 1e-13


@pytest.mark.skipif(not LD_OK, reason="np.longdouble is not wider than float64 here")
def test_longdouble_arm_separates_thresholds_on_bratu():
    """Bratu G = 41: nearly every iteration of the first 400 is a separated threshold, each with a margin far above
    the float64 rounding of ||r_j|| (what makes exact iteration counts testable)"""
    o = orc.BratuOracle(41, 5, 10)
    rs = np.random.RandomState(1)
    u = 0.2 * rs.normal(size=o.n)
    y = rs.normal(size=o.n)
    ref = CgReference(-1 * o.make_jac()(u).tocsr(), y, True, nmax=400)
    sep = separated(ref.rn["hi"][0])
    assert len(sep) >= 380, len(sep)
    picks = ref.thresholds([1, 2, 3, 50])
    assert [c for _, c, _ in picks][:4] == [1, 2, 3, 50] and picks[-1][0] == 1e-4
    x, tol = ref.iterate(50)
    assert 1e-12 <= tol < 1e-6


def test_the_graded_problem_runs_into_maxiter():
    A, y, rtol = graded_maxiter_problem()
    assert orc.cgls(A, y, rtol=rtol, preconditioner=True)[1] == 200
    assert orc.cgls(A, y, rtol=rtol, preconditioner=False)[1] == 400


# ------------------------------------------------------------------------------------------------
# host routing of J.T through the mock library
# ------------------------------------------------------------------------------------------------
@pytest.fixture()
def g():
    import mock_backend
    mock_backend.install()
    import gauss_newton_via_generalized_krylov_subspaces_b200 as pkg
    yield pkg
    mock_backend.uninstall()


@pytest.mark.parametrize("scale,transposed", [(-1.0, False), (2.5, False), (-1.0, True), (2.0, True)])
@pytest.mark.parametrize("precond", [True, False])
def test_cg_least_squares_on_a_scaled_or_transposed_bratu_jacobian(g, scale, transposed, precond):
    """cg_least_squares(s * J [.T], y) solves with exactly that operator: J is not symmetric (ALPHA d/dx1), so J.T
    solved as J misses by O(1)"""
    o = orc.BratuOracle(41, 5, 10)
    pb = g.BratuPdeProblem(41, 5, 10)
    rs = np.random.RandomState(1)
    u = 0.2 * rs.normal(size=o.n)
    y = rs.normal(size=o.n)
    J = pb.make_jac()(u)
    A = scale * (J.T if transposed else J)
    Ar = scale * o.make_jac()(u).tocsr()
    Ar = sp.csr_array(Ar.T) if transposed else Ar
    assert abs(sp.csr_array(A.tocsr()) - Ar).max() == 0.0
    xr, itr = orc.cgls(Ar, y, preconditioner=precond)
    x, it = g.cg_least_squares(A, y, preconditioner=precond)
    assert it == itr
    assert rel(x, xr) < 1e-12


def test_transposed_stencil_operator_is_refused_on_several_ranks_and_by_linop(g, monkeypatch):
    pb = g.BratuPdeProblem(12, 5, 10)
    J = pb.make_jac()(np.zeros(pb.n))
    from gauss_newton_via_generalized_krylov_subspaces_b200._lib import GnkError
    with pytest.raises(GnkError, match="J.T"):
        J.T.linop(1.0)
    J.linop(1.0)  # untransposed: fine
    rt = g.get_runtime()
    monkeypatch.setattr(rt, "world", 2)
    with pytest.raises(GnkError, match="transposed Bratu Jacobian"):
        g.cg_least_squares(-1 * J.T, np.ones(pb.n))


def test_gauss_newton_with_a_jac_callable_returning_a_transposed_operator(g):
    """a foreign jac that returns J.T (here: of a residual whose true Jacobian is J.T) reaches the CG solve as the
    assembled CSR of J.T, so the trace is the oracle's on the same callables"""
    o = orc.BratuOracle(12, 5, 0)
    pb = g.BratuPdeProblem(12, 5, 0)
    JT = sp.csr_array(o.make_jac()(None).tocsr().T)
    xs = np.random.RandomState(3).normal(size=o.n)
    y = JT @ xs
    res = lambda u: JT @ u - y  # noqa: E731
    jac_dev = lambda u: pb.make_jac()(u).T  # noqa: E731
    jac_ref = lambda u: JT  # noqa: E731
    cg_dev, cg_ref = [], []
    out = g.gauss_newton(res, np.zeros(o.n), jac_dev, max_iter=4, callback=lambda **kw: cg_dev.append(kw["cg_iter"]))
    ref = orc.gn(res, np.zeros(o.n), jac_ref, max_iter=4, callback=lambda **kw: cg_ref.append(kw["cg_iter"]))
    assert cg_dev == cg_ref and len(cg_ref) >= 2
    assert rel(out.x, ref["x"]) < 1e-12
