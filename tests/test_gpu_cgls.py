"""gnk_cgls / gnk_cgls_x0 (csrc/cgls.cu, the inner solve of gauss_newton and every cg_least_squares call) held to
scipy's cg iteration by iteration, and the CSR kernels it runs on (-m gpu).

Iteration counts are compared EXACTLY: the thresholds are chosen from the reference's own residual history
(tests/test_cgls_reference.py) where ||r_j|| drops by at least 0.1 % below every earlier residual, with a margin of at
least 100x the float64-vs-longdouble deviation of ||r_j|| (grids up to G = 45 and p <= 5000; beyond that the float64
history and a margin of 1e-2).  The iterate is compared with the longdouble x_j at 10x the float64-vs-longdouble gap of
x_j, never below 1e-12.  The pipelined loop (stopping test read one iteration late) must give bit-identical results to
the synchronous one (GNK_CG_PIPELINE=0, read once per process, hence the subprocess).
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp

pytestmark = pytest.mark.gpu

from golden_util import rel  # noqa: E402
from oracle import gnk_oracle as orc  # noqa: E402
from test_cgls_reference import CgReference, graded_maxiter_problem, random_sparse  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


@pytest.fixture(scope="module")
def g():
    return _package()


def _package():
    import gauss_newton_via_generalized_krylov_subspaces_b200 as pkg
    import gauss_newton_via_generalized_krylov_subspaces_b200.device as device
    if os.environ.get("GNK_TEST_MOCK"):  # debugging aid for the test code itself
        import mock_backend
        mock_backend.install()
        return pkg
    device._runtime = None
    pkg.get_runtime()  # raises without CUDA + the built library: no fallback
    return pkg


# ------------------------------------------------------------------------------------------------
# operators: the device object handed to cg_least_squares and the assembled matrix of the reference
# ------------------------------------------------------------------------------------------------
def bratu_case(g, G, lam, op, seed=1):
    """op: a scale s (A = s J) or "sT" (A = s J.T).  J(u) = -(L + 5 d/dx1 + lam diag(e^u)), u = 0.2 N(0, 1); the
    reference matrix is the oracle's assembly with the device's own e^u"""
    rs = np.random.RandomState(seed)
    o = orc.BratuOracle(G, 5, lam)
    pb = g.BratuPdeProblem(G, 5, lam)
    u = 0.2 * rs.normal(size=o.n)
    y = rs.normal(size=o.n)
    J = pb.make_jac()(u)
    expu = None if J.expu is None else pb.dev.download_global(J.expu)
    tr = isinstance(op, str)
    s = float(op[:-1]) if tr else float(op)
    Jr = orc.StencilJacobian(o, expu).tocsr()
    if tr:
        return s * J.T, sp.csr_array(s * Jr.T), y
    return s * J, sp.csr_array(s * Jr), y


def csr_matrix(name):
    """the generic-Jacobian operators: chained Rosenbrock (3 entries a row) and random sparse matrices with empty rows,
    a full column (a row of A^T with >= 1e4 entries) and p not a multiple of 128"""
    if name == "rosenbrock":
        x = 1 + 0.1 * np.random.RandomState(7).normal(size=1000)
        return sp.csr_array(-1 * orc.rosenbrock_jac(x))
    if name == "tall":
        return random_sparse(3 * 3371, 3371, 11, empty_rows=40, long_col=True)
    if name == "square":
        return random_sparse(1000, 1000, 12, empty_rows=9)
    if name == "wide":
        return random_sparse(700, 1000, 13, per_row=9, empty_rows=5)
    raise KeyError(name)


def csr_case(name, seed=2):
    A = csr_matrix(name)
    rs = np.random.RandomState(seed)
    y = A @ rs.normal(size=A.shape[1]) if name == "wide" else rs.normal(size=A.shape[0])  # wide: y in the range
    return A, A, y


def _check_counts(g, A_dev, A_ref, y, precond, precise, x0=None, extra_targets=()):
    ref = CgReference(A_ref, y, precond, x0=x0, longdouble=precise, stop_rtol=1e-5)
    default = ref.counts(1e-4 * ref.bn)[-1][0]
    assert default is not None and default > 4
    picks = ref.thresholds([1, 2, 3, default // 2, *extra_targets], min_margin=None if ref.precise else 1e-2)
    assert len(picks) >= 3, picks
    done = []
    for rtol, total, jlast in picks:
        x, it = g.cg_least_squares(A_dev, y, x0=x0, cg_rtol=rtol, preconditioner=precond)
        assert it == total, (rtol, it, total)
        if ref.precise:
            xr, tol = ref.iterate(jlast)
            assert rel(x, xr) <= tol, (jlast, rel(x, xr), tol)
        done.append(total)
    return done


# ------------------------------------------------------------------------------------------------
# exact iteration counts
# ------------------------------------------------------------------------------------------------
BRATU_OPS = [-1.0, 2.5, -0.5, "-1T", "2T"]


# the full matrix on the grids of the longdouble arm; on the larger ones (float64 arm, up to 5000 iterations a case)
# every operator once, lambda alternating
BRATU_CASES = [(G, lam, op) for G in (12, 41) for lam in (10, 0) for op in BRATU_OPS] + \
    [(G, lam, op) for G in (130, 131) for lam, op in zip((10, 0, 10, 0, 10), BRATU_OPS)]


@pytest.mark.parametrize("precond", [True, False])
@pytest.mark.parametrize("G,lam,op", BRATU_CASES)
def test_cgls_bratu_exact_counts(g, G, lam, op, precond):
    """matrix-free stencil operator s J (|s| != 1 runs the s^2 rescale of the Jacobi diagonal) and s J.T (assembled)"""
    A, Ar, y = bratu_case(g, G, lam, op)
    done = _check_counts(g, A, Ar, y, precond, precise=G <= 45)
    if precond:
        assert done[0] <= 3  # the first iterations are separated on every grid


@pytest.mark.parametrize("precond", [True, False])
@pytest.mark.parametrize("name", ["rosenbrock", "tall", "square", "wide"])
def test_cgls_csr_exact_counts(g, name, precond):
    A, Ar, y = csr_case(name)
    _check_counts(g, A, Ar, y, precond, precise=True)


@pytest.mark.parametrize("fmt", ["coo_duplicates", "csr_unsorted", "dense"])
def test_cgls_input_formats_give_the_csr_result(g, fmt):
    """COO with duplicate entries, CSR with unsorted indices and a dense ndarray reach the device as the same CSR:
    the result is bitwise the canonical CSR's"""
    A, _, y = csr_case("square")
    rs = np.random.RandomState(5)
    if fmt == "coo_duplicates":
        c = A.tocoo()
        half = rs.rand(c.nnz) < 0.5
        part = np.where(half, 0.5, 1.0)  # a split into two entries whose sum is exact
        Ain = sp.coo_array((np.concatenate([c.data * part, (c.data * part)[half]]),
                            (np.concatenate([c.row, c.row[half]]), np.concatenate([c.col, c.col[half]]))),
                           shape=A.shape)
        assert Ain.nnz > A.nnz and abs(Ain.tocsr() - A).max() == 0.0
    elif fmt == "csr_unsorted":
        Ain = sp.csr_array(A, copy=True)
        for i in range(A.shape[0]):
            s, e = Ain.indptr[i], Ain.indptr[i + 1]
            perm = s + rs.permutation(e - s)
            Ain.indices[s:e], Ain.data[s:e] = Ain.indices[perm], Ain.data[perm]
        Ain.has_sorted_indices = False
        assert not np.all(np.diff(Ain.indices[Ain.indptr[0]:Ain.indptr[1]]) > 0) or Ain.indptr[1] - Ain.indptr[0] < 2
    else:
        Ain = A.toarray()
    for precond in (True, False):
        x0, it0 = g.cg_least_squares(A, y, preconditioner=precond)
        x1, it1 = g.cg_least_squares(Ain, y, preconditioner=precond)
        assert it1 == it0 and np.array_equal(x1, x0)


# ------------------------------------------------------------------------------------------------
# initial guess and the edge exits
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precond", [True, False])
@pytest.mark.parametrize("case", ["bratu41", "bratu41T", "square"])
def test_cgls_random_x0_exact_counts(g, case, precond):
    if case.startswith("bratu"):
        A, Ar, y = bratu_case(g, 41, 10, "-1T" if case.endswith("T") else -1.0)
    else:
        A, Ar, y = csr_case(case)
    x0 = 0.1 * np.random.RandomState(9).normal(size=Ar.shape[1])
    _check_counts(g, A, Ar, y, precond, precise=True, x0=x0)


@pytest.mark.parametrize("precond", [True, False])
def test_cgls_x0_at_the_solution_and_zero_right_hand_side(g, precond):
    A, _, _ = csr_case("square")
    xs = np.random.RandomState(3).normal(size=A.shape[1])
    x, it = g.cg_least_squares(A, A @ xs, x0=xs, preconditioner=precond)
    assert it == 0 and np.array_equal(x, xs)
    Ab, _, _ = bratu_case(g, 41, 10, -1.0)
    xb = np.random.RandomState(4).normal(size=Ab.shape[1])
    x, it = g.cg_least_squares(Ab, Ab @ xb, x0=xb, preconditioner=precond)
    assert it == 0 and np.array_equal(x, xb)
    # A^T y = 0 exactly (y lives on the rows without entries), x0 != 0: scipy returns b = 0 and no iteration
    empty = np.diff(A.indptr) == 0
    y = np.where(empty, 1.0 + np.arange(A.shape[0]), 0.0)
    assert empty.sum() > 0 and not np.any(A.T @ y)
    x, it = g.cg_least_squares(A, y, x0=xs, preconditioner=precond)
    assert it == 0 and np.all(x == 0)
    assert orc.cgls(A, y, preconditioner=precond, x0=xs)[1] == 0


@pytest.mark.parametrize("precond", [True, False])
def test_cgls_maxiter_exit(g, precond):
    """40 x 20, singular values 1 .. 1e-6, rtol 1e-18: every pass runs into maxiter = 10 p; the pipelined loop must
    report 10 p per pass (its tail check looks at the last queued test) and a finite x whose normal residual is within
    10x of the reference's -- the worst of the reference itself and of the reference on y moved by one ulp (random
    signs), since after 200 iterations at this conditioning the end point is set by rounding"""
    A, y, rtol = graded_maxiter_problem()
    passes = 1 if precond else 2
    nres = lambda v: np.linalg.norm(A.T @ (y - A @ v))  # noqa: E731
    xr, itr = orc.cgls(A, y, rtol=rtol, preconditioner=precond)
    assert itr == 200 * passes  # the reference runs into maxiter
    worst = nres(xr)
    for s in range(3):
        yp = y * (1 + np.random.RandomState(s).choice([-1.0, 1.0], size=y.shape[0]) * np.finfo(float).eps / 2)
        worst = max(worst, nres(orc.cgls(A, yp, rtol=rtol, preconditioner=precond)[0]))
    x, it = g.cg_least_squares(A, y, cg_rtol=rtol, preconditioner=precond)
    assert it == 200 * passes
    assert np.all(np.isfinite(x))
    assert nres(x) <= 10 * worst, (nres(x), nres(xr), worst)
    # a threshold decided at j = maxiter - 1 (the tail check's done_at = it - 1), where the history separates it
    ref = CgReference(A, y, precond)
    picks = [p for p in ref.thresholds([199]) if p[2] == 199]
    for rtol_j, total, _ in picks:
        assert g.cg_least_squares(A, y, cg_rtol=rtol_j, preconditioner=precond)[1] == total
    print(f"[maxiter] precond={precond}: |A^T(y - A x)| = {nres(x):.2e}, reference {nres(xr):.2e} (worst {worst:.2e}); "
          f"threshold at j = 199 {'tested' if picks else 'not separated'}")


# ------------------------------------------------------------------------------------------------
# pipelined == synchronous
# ------------------------------------------------------------------------------------------------
def equivalence_runs(g):
    """the operators above at several tolerances, with and without x0 and preconditioner: {name: x} and {name_it: n}"""
    out = {}
    cases = [("b41", bratu_case(g, 41, 10, -1.0)), ("b41s", bratu_case(g, 41, 0, 2.5)),
             ("b130", bratu_case(g, 130, 10, -0.5)), ("b41T", bratu_case(g, 41, 10, "-1T")),
             ("rosen", csr_case("rosenbrock")), ("tall", csr_case("tall")), ("wide", csr_case("wide"))]
    for name, (A, Ar, y) in cases:
        x0 = 0.1 * np.random.RandomState(9).normal(size=Ar.shape[1])
        for precond in (True, False):
            for rtol in (1e-1, 1e-2, 1e-4, 1e-8):
                for with_x0 in (False, True):
                    key = f"{name}_{int(precond)}_{rtol:g}_{int(with_x0)}"
                    x, it = g.cg_least_squares(A, y, x0=x0 if with_x0 else None, cg_rtol=rtol, preconditioner=precond)
                    out[key], out[key + "_it"] = x, np.array(it)
    A, y, rtol = graded_maxiter_problem()
    for precond in (True, False):
        x, it = g.cg_least_squares(A, y, cg_rtol=rtol, preconditioner=precond)
        out[f"maxiter_{int(precond)}"], out[f"maxiter_{int(precond)}_it"] = x, np.array(it)
    return out


def test_cgls_pipelined_equals_synchronous_and_repeats_bitwise(g, tmp_path):
    a = equivalence_runs(g)
    b = equivalence_runs(g)
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    out = tmp_path / "sync.npz"
    env = dict(os.environ, GNK_CG_PIPELINE="0")
    code = ("import sys; sys.path[:0] = [{h!r}, {r!r}]; import numpy as np; import test_gpu_cgls as t; "
            "np.savez({o!r}, **t.equivalence_runs(t._package()))").format(h=HERE, r=ROOT, o=str(out))
    proc = subprocess.run([sys.executable, "-c", code], env=env, cwd=ROOT, capture_output=True, text=True,
                          timeout=600)
    assert proc.returncode == 0, proc.stdout[-3000:] + proc.stderr[-3000:]
    s = np.load(out)
    assert sorted(s.files) == sorted(a)
    diff = [k for k in a if not np.array_equal(a[k], s[k])]
    assert not diff, diff[:10]


# ------------------------------------------------------------------------------------------------
# the CSR kernels directly
# ------------------------------------------------------------------------------------------------
def _kernel_matrices():
    long_col = random_sparse(12001, 500, 21, per_row=1, long_col=True)  # its transpose has a row of 12001 entries
    return {"rosenbrock": csr_matrix("rosenbrock"), "tall": csr_matrix("tall"), "square": csr_matrix("square"),
            "wide": csr_matrix("wide"), "longrow": sp.csr_array(long_col.T)}


@pytest.mark.parametrize("name", ["rosenbrock", "tall", "square", "wide", "longrow"])
def test_spmm_csr_and_row_sumsq(g, name):
    from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib
    from gauss_newton_via_generalized_krylov_subspaces_b200.device import CsrJacobian, ptr
    rt = g.get_runtime()
    A = _kernel_matrices()[name]
    if name == "longrow":
        assert np.max(np.diff(A.indptr)) >= 10 ** 4
    op = CsrJacobian(rt, A, True)
    rs = np.random.RandomState(17)
    for M, rp, ci, va in ((A, op.rowptr, op.col, op.val), (sp.csr_array(A.T), op.rowptr_t, op.col_t, op.val_t)):
        n_rows, n_cols = M.shape
        absM = abs(M)
        for k, sign, in_off, out_off in ((1, 1.0, 0, 0), (3, -1.0, 5, 3), (33, 0.5, 17, 129)):
            in_ld, out_ld = n_cols + in_off + 7, n_rows + out_off + 3
            V = rs.normal(size=(k, n_cols))
            din = rt.zeros(in_ld * k)
            for j in range(k):
                rt.upload(V[j], din[j * in_ld + in_off:j * in_ld + in_off + n_cols])
            dout = rt.zeros(out_ld * k)
            dout.fill_(float("nan"))
            _lib.check(rt.lib.gnk_spmm_csr(rt.ctx, n_rows, ptr(rp), ptr(ci), ptr(va), ptr(din), in_ld, in_off, k, sign,
                                           ptr(dout), out_ld, out_off, rt.stream), "gnk_spmm_csr")
            got = rt.download(dout).reshape(k, out_ld)
            for j in range(k):
                want = sign * (M @ V[j])
                scale = abs(sign) * (absM @ np.abs(V[j]))
                gj = got[j, out_off:out_off + n_rows]
                assert np.all(np.abs(gj - want) <= 1e-14 * scale), (name, k, j, float(np.max(np.abs(gj - want))))
                empty = np.diff(M.indptr) == 0
                assert np.all(gj[empty] == 0)
                # entries outside [out_off, out_off + n_rows) of the column are not written
                assert np.all(np.isnan(got[j, :out_off])) and np.all(np.isnan(got[j, out_off + n_rows:]))
    ss = rt.zeros(A.shape[1] + 16)
    _lib.check(rt.lib.gnk_csr_row_sumsq(rt.ctx, A.shape[1], ptr(op.rowptr_t), ptr(op.val_t), ptr(ss), rt.stream),
               "gnk_csr_row_sumsq")
    want = np.asarray(A.multiply(A).sum(axis=0)).reshape(-1)
    assert rel(rt.download(ss[:A.shape[1]]), want) < 1e-14
