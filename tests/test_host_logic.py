"""CPU tests of everything that is not a CUDA kernel: the C-ABI library's exported surface, the slab partition, and
the Python host logic (solver control flow, buffer rotation, counters, messages) driven through the numpy mock of
the C ABI (tests/mock_backend.py -- test infrastructure, injected explicitly; the product has no CPU path).
"""
import os
import re
import subprocess

import numpy as np
import pytest

from golden_util import Golden, Recorder, check_trace, rel

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "gauss_newton_via_generalized_krylov_subspaces_b200")


# ------------------------------------------------------------------------------------------------
# the shared library: loads, exports every symbol include/gnk_b200.h declares, and nothing computes without a GPU
# ------------------------------------------------------------------------------------------------
def _header_functions():
    text = open(os.path.join(ROOT, "include", "gnk_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(gnk_[a-z0-9_]+)\s*\(", text)))


def test_library_builds_and_exports_the_header_surface():
    import __graft_entry__
    __graft_entry__.build()
    from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib
    lib = _lib.load()
    declared = _header_functions()
    assert len(declared) >= 25
    nm = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r"\bT (gnk_[a-z0-9_]+)", nm))
    assert set(declared) <= exported, sorted(set(declared) - exported)
    assert set(declared) == set(_lib.SIGNATURES), (set(declared) ^ set(_lib.SIGNATURES))
    assert lib.gnk_abi_version() == 1
    # sm_100a code is in the fat binary
    out = subprocess.run(["cuobjdump", "--list-elf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out


def test_library_holds_the_sm100a_kernels_of_the_hot_path():
    """the shipped .so carries the kernels bench.py and smoke() are supposed to launch: the FP64 tensor-pipe
    instructions (DMMA) of the Gram passes, the stencil, Gram-Schmidt and least-squares kernels -- no stub library"""
    import __graft_entry__
    __graft_entry__.build()
    from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib
    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    for name in ("cholqr_gram_kernel", "cholqr_gram2_kernel", "cholqr_refine_kernel", "cholqr_factor1_kernel",
                 "cholqr_factor2_kernel", "tsqr_quad_kernel", "apply_kernel", "residual_kernel", "combine_kernel",
                 "dots_kernel", "update_kernel", "normalize_kernel", "normalize_halo_kernel", "stencil_gram_kernel",
                 "gram_wide_kernel", "gram_pcg_kernel", "wide_factor1_kernel", "wide_refine_kernel",
                 "wide_factor2_kernel", "cg_precond_kernel", "cg_step_kernel"):
        assert name in sass, name
    assert "UTMALDG" in sass                       # the TMA-staged row slots of the fused stencil + Gram sweep
    assert "SYNCS" in sass                         # ... and their mbarriers
    assert sass.count("DMMA.8x8x4") > 500          # Gram passes (and the quad reductions of the Householder leaf)
    assert "LDG.E.EF.128" in sass or "LDG.E.128" in sass


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    import gauss_newton_via_generalized_krylov_subspaces_b200 as g
    import gauss_newton_via_generalized_krylov_subspaces_b200.device as device
    device._runtime = None
    pb = g.BratuPdeProblem(11, 5, 10)
    with pytest.raises(Exception) as ei:
        pb.pde_operator(np.zeros(100))
    assert "no CPU fallback" in str(ei.value) or "CUDA" in str(ei.value)
    with pytest.raises(Exception):
        g.gauss_newton_krylow(lambda x: x, np.ones(3), lambda x: np.eye(3), callback=lambda **k: None)


def test_product_never_imports_the_oracle():
    for dirpath, _, files in os.walk(PKG):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in text.replace("the oracle", "").replace("CPU oracle", "") or f == "__init__.py", f
                assert "mock_backend" not in text, f


# ------------------------------------------------------------------------------------------------
# slab partition (pure integer logic)
# ------------------------------------------------------------------------------------------------
def test_slab_partition():
    from gauss_newton_via_generalized_krylov_subspaces_b200 import partition as P
    for m in (1, 2, 7, 33, 100, 1024, 4096, 8192):
        for world in (1, 2, 3, 4, 8):
            bounds = [P.slab_bounds(m, world, r) for r in range(world)]
            assert bounds[0][0] == 0 and bounds[-1][1] == m
            assert all(bounds[i][1] == bounds[i + 1][0] for i in range(world - 1))
            sizes = [b - a for a, b in bounds]
            assert max(sizes) - min(sizes) <= 1
            assert sum(P.all_counts(m, world)) == m * m
    # the tensor-pipe least squares must be taken by all ranks or by none (different collectives)
    assert P.tensor_ls_on_every_rank(4096, 8) and P.tensor_ls_on_every_rank(1024, 8) and P.tensor_ls_on_every_rank(128, 1)
    assert not P.tensor_ls_on_every_rank(1001, 2)      # 501 * 1001 is odd
    assert not P.tensor_ls_on_every_rank(181, 2)       # 91 * 181 = 16471 >= 16384 > 90 * 181
    assert not P.tensor_ls_on_every_rank(33, 3)
    f = P.stencil_layout_fields(4096, 8, 3)
    assert (f["rows"], f["off"], f["n_own"], f["has_lo"], f["has_hi"]) == (512, 8192, 512 * 4096, 1, 1)
    assert f["ld"] % 16 == 0 and f["ld"] >= (512 + 4) * 4096
    with pytest.raises(ValueError):
        P.stencil_layout_fields(8, 8, 0)   # 1-row slabs are thinner than the halo
    x = np.arange(7 * 7, dtype=np.float64)
    f = P.stencil_layout_fields(7, 3, 1)   # rows [3,5)
    col = np.full(f["ld"], -1.0)
    P.stored_column_from_global(x, f, col[:(f["rows"] + 4) * 7])
    assert np.array_equal(col[:(f["rows"] + 4) * 7], x[7:49])   # rows 1..6
    f = P.stencil_layout_fields(7, 3, 0)   # rows [0,3): two zero halo rows in front
    col = np.full(f["ld"], -1.0)
    P.stored_column_from_global(x, f, col[:(f["rows"] + 4) * 7])
    assert np.all(col[:14] == 0) and np.array_equal(col[14:49], x[:35])


# ------------------------------------------------------------------------------------------------
# host logic through the mock
# ------------------------------------------------------------------------------------------------
@pytest.fixture()
def g():
    import mock_backend
    mock_backend.install()
    import gauss_newton_via_generalized_krylov_subspaces_b200 as pkg
    yield pkg
    mock_backend.uninstall()


def test_host_gnk_bratu(g, capsys):
    gd = Golden("bratu_g101")
    pb = g.BratuPdeProblem(101, 5, 10)
    assert rel(pb.pde_operator(pb.u_true), gd["y"]) < 1e-14
    res, jac, err = pb.make_res(gd["y"]), pb.make_jac(), pb.make_error()
    for rname, kw, tol in (("gnk_res_old", dict(max_iter=30), 1e-12),
                           ("gnk_jac_old_res_new", dict(max_iter=25, version="jac_old_res_new"), 1e-12),
                           ("gnk_restart7_res_new", dict(max_iter=40, krylow_restart=7, version="res_new"), 1e-8)):
        gr = gd.run(rname)
        rec = Recorder(gr["sample_idx"], err)
        out = g.gauss_newton_krylow(res, gd["u0"], jac, callback=rec, **kw)
        check_trace(rec, gr, tol, upto=len(rec.xnorm))
        assert out.nrev == out.nit + 1 and out.njev == out.nit + 1 and not out.success
    assert "reached maximal iteration bound" in capsys.readouterr().out


def test_host_gnk_least_squares_refusal_falls_back_to_householder(g):
    """gnk_tsqr_ls may refuse a panel (CholeskyQR2 on a numerically rank deficient Gram matrix: d = 0 and
    out[k+2] = -1, include/gnk_b200.h).  The solver must re-issue the SAME solve with the Householder path pinned,
    not count the wasted trial, and end on the same trajectory."""
    import ctypes as C
    gd = Golden("bratu_g101")
    pb = g.BratuPdeProblem(101, 5, 10)
    res, jac = pb.make_res(gd["y"]), pb.make_jac()
    base = g.gauss_newton_krylow(res, gd["u0"], jac, callback=lambda **kw: None, max_iter=12)

    lib = g.get_runtime().lib
    real = lib.gnk_tsqr_ls
    calls = {"refused": 0, "householder": 0}

    def refusing(ctx, A, lda, n_rows, k, y, sign_a, out, stream):
        if getattr(lib, "ls_method", 0) == 0 and k in (3, 4, 9):
            calls["refused"] += 1
            o = np.ctypeslib.as_array(C.cast(out, C.POINTER(C.c_double)), shape=(2 * k + 4,))
            o[:] = 0.0
            o[k + 2] = -1.0
            o[k + 4:] = 1.0
            return 0
        if getattr(lib, "ls_method", 0) == 1:
            calls["householder"] += 1
        return real(ctx, A, lda, n_rows, k, y, sign_a, out, stream)

    lib.gnk_tsqr_ls = refusing
    try:
        seen = []
        out = g.gauss_newton_krylow(res, gd["u0"], jac, callback=lambda x, nfev, cg_iter: seen.append(nfev),
                                    max_iter=12)
    finally:
        lib.gnk_tsqr_ls = real
    assert calls == {"refused": 3, "householder": 3}
    assert getattr(lib, "ls_method", 0) == 0                       # the pin is released after the call
    assert out.nit == base.nit and out.nrev == base.nrev and seen == list(range(2, 13))
    assert np.array_equal(out.x, base.x)
    # the public linear_least_squares mirror falls back the same way
    rs = np.random.RandomState(0)
    A, y = rs.normal(size=(50, 3)), rs.normal(size=50)
    lib.gnk_tsqr_ls = refusing
    try:
        x = g.linear_least_squares(A, y)
    finally:
        lib.gnk_tsqr_ls = real
    assert rel(x, np.linalg.lstsq(A, y, rcond=None)[0]) < 1e-13


def test_host_gnk_deferred_breakdown_flag(g, capsys, monkeypatch):
    """The Krylov breakdown flag (krylow.py:66) is read with the NEXT iteration's scalar block instead of right away
    (one host synchronisation less per outer iteration).  compare_linear_small (grid_nodes=25, LAMBDA=0) breaks down
    at iteration 2: the speculatively appended column must be retracted, the message printed before the next
    callback, and the run must be identical to the one with the synchronous read (GNK_DEFER_BREAKDOWN=0)."""
    gd = Golden("bratu_g25_linear")
    pb = g.BratuPdeProblem(25, 5, 0)
    res, jac = pb.make_res(gd["y"]), pb.make_jac()
    gr = gd.run("gnk_res_old")
    runs = {}
    for mode in ("1", "0"):
        monkeypatch.setenv("GNK_DEFER_BREAKDOWN", mode)
        events = []
        rec = Recorder(gr["sample_idx"])

        def cb(x, nfev, cg_iter):
            events.append(("cb", nfev))
            rec(x, nfev, cg_iter)

        reads = {"n": 0}
        rt = g.get_runtime()
        real_read = rt.read_i32

        def counting(t):
            reads["n"] += 1
            return real_read(t)

        rt.read_i32 = counting
        try:
            out = g.gauss_newton_krylow(res, gd["u0"], jac, callback=cb, max_iter=100)
            outcome = ("ok", out.nit, out.nrev, bool(out.success))
        except g.StepLengthConvergenceError:
            outcome = ("step",)
        finally:
            rt.read_i32 = real_read
        text = capsys.readouterr().out
        assert "Generalized krylow subspace breakdown at iteration = 2, basis.shape = (576, 2)" in text
        runs[mode] = (outcome, [e[1] for e in events], np.array(rec.xs), reads["n"])
        check_trace(rec, gr, 1e-10, upto=2)
    assert runs["1"][0] == runs["0"][0] and runs["1"][1] == runs["0"][1]
    assert np.array_equal(runs["1"][2], runs["0"][2])
    assert runs["1"][3] < runs["0"][3]          # fewer flag read-backs in deferred mode


def test_host_gn_and_foreign_callables(g):
    from gauss_newton_via_generalized_krylov_subspaces_b200 import rosenbrock_problem as rp
    gd = Golden("rosenbrock")
    for tag, rname, kw in (("i", "gnk_res_new", dict(version="res_new")), ("iii", "gnk_res_old", {})):
        gr = gd.run(f"{tag}_{rname}")
        rec = Recorder(gr["sample_idx"], rp.error)
        out = g.gauss_newton_krylow(rp.res, gd["x0_" + tag], rp.jac, callback=rec, **kw)
        check_trace(rec, gr, 1e-10)
        assert (out.nit, out.nrev, out.success) == (int(gr["nit"]), int(gr["nfev"]), True)
    gr = gd.run("i_gn")
    rec = Recorder(gr["sample_idx"], rp.error)
    out = g.gauss_newton(rp.res, gd["x0_i"], rp.jac, callback=rec)
    assert (out.nit, out.nrev, out.njev) == (5, 6, 5) and list(rec.cg) == list(gr["cg_iter"])


def test_host_gn_dense_rank_deficient_jacobian_is_reported(g):
    """advisor: a dense Jacobian with a zero column must not hand inf/NaN to the line search"""
    res = lambda x: np.array([x[0] - 1.0, 2.0 * x[0] + 1.0, x[0]])
    jac = lambda x: np.array([[1.0, 0.0], [2.0, 0.0], [1.0, 0.0]])
    with pytest.raises(np.linalg.LinAlgError, match="rank deficient"):
        g.gauss_newton(res, np.array([1.0, 2.0]), jac, callback=lambda **k: None)


def test_host_step_length_plugins_and_errors(g):
    def pres(x, tau):
        return np.array([x[0] + 1, tau * x[0] ** 2 + x[0] - 1])

    def pjac(x, tau):
        return np.array([[1], [2 * tau * x[0] + 1]])

    def no_step_length_control(res, x, res_ev, jac_ev, args, descent_direction, *_):
        return 1, res(x + descent_direction, *args), 1

    gd = Golden("powell")
    xs = []
    out = g.gauss_newton(pres, np.array([1.0]), pjac, args=(-5,), max_iter=19, step_length_control=no_step_length_control,
                         callback=lambda x, nfev, cg_iter: xs.append(float(np.asarray(x)[0])))
    gr = gd.run("tau-5_no_step_length_control")
    assert (out.nit, out.nrev, out.success) == (18, 19, False)
    assert np.max(np.abs(np.array(xs) - gr["xs"][:, 0])) < 1e-12
    with pytest.raises(g.StepLengthConvergenceError) as ei:
        g.gauss_newton(pres, np.array([1.0]), pjac, args=(-5,), max_iter=19, callback=lambda **k: None)
    assert "Norm of descent_direction" in ei.value.message
    with pytest.raises(TypeError):
        g.gauss_newton(pres, np.array([1.0]), pjac, args=(5,))       # default callback is called with keywords
    with pytest.raises(ValueError):
        g.gauss_newton_krylow(pres, np.zeros(1), pjac, args=(5,), callback=lambda **k: None)


def test_flat_module_names(g):
    import sys
    g.install_flat_names()
    import gauss_newton_krylow as m1
    import krylow as m2
    from bratu_pde_problem import BratuPdeProblem
    from regression_result import RegressionResult
    assert m1.gauss_newton_krylow is g.gauss_newton_krylow and m2.GeneralizedKrylowSubspace is g.GeneralizedKrylowSubspace
    assert BratuPdeProblem is g.BratuPdeProblem
    r = RegressionResult("gauss newton", np.ones(2), True, 3, 2, 2)
    assert "converged successfuly" in str(r) and r.nrev == 3
    for name in ("gauss_newton_krylow", "krylow", "bratu_pde_problem", "regression_result", "armijo_goldstein",
                 "gauss_newton", "rosenbrock_problem", "benchmark"):
        sys.modules.pop(name, None)


def test_benchmark_harness(g):
    from gauss_newton_via_generalized_krylov_subspaces_b200.benchmark import benchmark_method, reverse_accumulation
    assert reverse_accumulation([2, 3, 7]) == [2, 1, 4] and reverse_accumulation([]) == []
    gd = Golden("bratu_g34")
    pb = g.BratuPdeProblem(34, 5, 10)
    res, jac, err = pb.make_res(gd["y"]), pb.make_jac(), pb.make_error()
    e, l, nf, cg = benchmark_method(g.gauss_newton_krylow, res, gd["u0"], jac, err, kwargs=dict(max_iter=6))
    gr = gd.run("gnk_res_old")
    assert len(e) == 6 and nf == [2, 1, 1, 1, 1] and cg == []
    assert np.allclose(e[1:], gr["err"][:5], rtol=1e-10) and np.allclose(l[1:], gr["loss"][:5], rtol=1e-10)


def test_host_gnk_with_cgls_inner_solve(g):
    """BASELINE config 5 at toy size: GNK whose projected least squares is solved by CGLS (the reference never runs
    this combination; the oracle is the reference's cg_least_squares patched in for linear_least_squares, SURVEY 8c)."""
    from oracle import gnk_oracle as orc
    gd = Golden("bratu_g34")
    pb = g.BratuPdeProblem(34, 5, 10)
    res, jac, err = pb.make_res(gd["y"]), pb.make_jac(), pb.make_error()
    o = orc.BratuOracle(34, 5, 10)
    ls = lambda A, y, log: orc.cgls(A, y, rtol=1e-10, preconditioner=True)[0]  # noqa: E731
    ref = orc.gnk(o.make_res(gd["y"]), gd["u0"], o.make_jac(), restart=20, max_iter=31, ls=ls)
    out = g.gauss_newton_krylow(res, gd["u0"], jac, krylow_restart=20, max_iter=31, callback=lambda **k: None,
                                ls_solver="cgls", cg_rtol=1e-10)
    assert (out.nit, out.nrev, out.njev) == (ref["nit"], ref["nfev"], ref["njev"])
    assert rel(out.x, ref["x"]) < 1e-6
    qr = g.gauss_newton_krylow(res, gd["u0"], jac, krylow_restart=20, max_iter=31, callback=lambda **k: None)
    assert rel(out.x, qr.x) < 1e-6   # tight CG tolerance reproduces the QR solve
    with pytest.raises(ValueError):
        g.gauss_newton_krylow(res, gd["u0"], jac, max_iter=3, callback=lambda **k: None, ls_solver="nope")


def test_device_side_error_and_loss_in_callbacks(g):
    """SURVEY 8f(1): error(x) / loss(x) of the benchmark harness evaluated on the callback's DeviceVector in place."""
    gd = Golden("bratu_g34")
    pb = g.BratuPdeProblem(34, 5, 10)
    res, jac, err = pb.make_res(gd["y"]), pb.make_jac(), pb.make_error()
    seen = []

    def cb(x, nfev, cg_iter):
        assert isinstance(x, g.DeviceVector) and x._t is not None
        e_dev, l_dev = err(x), res.loss(x)
        assert x._host is None                      # nothing was copied to the host for that
        xh = np.asarray(x)
        seen.append((e_dev, np.linalg.norm(pb.u_true - xh), l_dev, 0.5 * np.sum(res(xh) ** 2)))

    g.gauss_newton_krylow(res, gd["u0"], jac, callback=cb, max_iter=6)
    a = np.array(seen)
    gr = gd.run("gnk_res_old")
    assert np.allclose(a[:, 0], a[:, 1], rtol=1e-13) and np.allclose(a[:, 2], a[:, 3], rtol=1e-12)
    assert np.allclose(a[:, 0], gr["err"][:5], rtol=1e-10) and np.allclose(a[:, 2], gr["loss"][:5], rtol=1e-10)


def test_callback_that_keeps_x_gets_a_snapshot(g):
    """Ownership hand-off of the callback's DeviceVector (device.DeviceVector.settle): a callback that KEEPS x -- in a
    list, behind a wrapper, in a closure -- must later still read the iterate of that iteration, although the solver
    reuses the device buffer; a callback that drops x costs no download.  No reference counts are inspected."""
    gd = Golden("bratu_g34")
    pb = g.BratuPdeProblem(34, 5, 10)
    res, jac = pb.make_res(gd["y"]), pb.make_jac()
    kept, copies = [], []

    def keeps(x, nfev, cg_iter):
        kept.append(x)                           # no copy: the DeviceVector itself

    def wrapped(**kw):                           # an extra frame / an extra reference while the callback runs
        holder = [kw["x"]]
        keeps(**kw)
        del holder

    g.gauss_newton_krylow(res, gd["u0"], jac, callback=wrapped, max_iter=8)
    g.gauss_newton_krylow(res, gd["u0"], jac, callback=lambda x, nfev, cg_iter: copies.append(np.array(x)), max_iter=8)
    assert len(kept) == len(copies) == 7
    for a, b in zip(kept, copies):
        assert isinstance(a, g.DeviceVector) and a._host is not None     # snapshot taken when the callback returned
        assert np.array_equal(np.asarray(a), b)
    # a callback that ignores x: nothing is downloaded
    rt = g.get_runtime()
    n_down = [0]
    real = pb.dev.download_global
    pb.dev.download_global = lambda col: (n_down.__setitem__(0, n_down[0] + 1), real(col))[1]
    g.gauss_newton_krylow(res, gd["u0"], jac, callback=lambda **kw: None, max_iter=8, x_on_device=True)
    assert n_down[0] == 0
    # same contract in the full-space solver (gauss_newton.py:125-127 hands the SAME array every time; here each
    # callback gets its own lazy vector)
    kept2 = []
    out = g.gauss_newton(res, gd["u0"], jac, callback=lambda x, nfev, cg_iter: kept2.append(x), max_iter=4)
    assert all(v._host is not None for v in kept2) and np.array_equal(np.asarray(kept2[-1]), out.x)


def test_device_vector_as_x0_of_a_foreign_problem(g):
    """a DeviceVector is an ordinary array-like for every problem but the one that made it (advisor, round 1: it used
    to be materialised by np.asarray and then dereferenced as a NULL device pointer)"""
    from gauss_newton_via_generalized_krylov_subspaces_b200 import rosenbrock_problem as rp
    pb = g.BratuPdeProblem(34, 5, 10)
    x0 = np.full(1089, 2.0)
    x0[2] = 1.99
    dv = pb.dev.resident(x0)                       # lives on the device, made by ANOTHER problem
    p = 1089

    def res(x):
        return np.concatenate([10 * (x[1:] - x[:-1] ** 2), 1 - x[:-1]])

    def jac(x):
        import scipy.sparse as sp
        b1 = 10 * sp.eye(p - 1, p, k=1) - 20 * sp.diags(x[:-1], shape=(p - 1, p))
        return sp.vstack([b1, -sp.eye(p - 1, p)]).tocsr()

    a = g.gauss_newton_krylow(res, dv, jac, callback=lambda **k: None, max_iter=6)
    b = g.gauss_newton_krylow(res, x0, jac, callback=lambda **k: None, max_iter=6)
    assert np.array_equal(a.x, b.x) and a.nit == b.nit


def test_cg_least_squares_with_initial_guess(g):
    """cg_least_squares(A, y, x0=...) -- the reference forwards x0 to scipy's cg (gauss_newton.py:14,46,56); golden
    from the unmodified reference (oracle/gen_golden.py cgx0): same iteration counts, same solution."""
    from oracle import gnk_oracle as orc
    import scipy.sparse as sp
    z = np.load(os.path.join(ROOT, "tests", "golden", "cg_x0.npz"))
    from gauss_newton_via_generalized_krylov_subspaces_b200 import rosenbrock_problem as rp
    o = orc.BratuOracle(34, 5, 10)
    A = -1 * o.make_jac()(z["bratu/u"])
    pb = g.BratuPdeProblem(34, 5, 10)
    Ad = -1 * pb.make_jac()(z["bratu/u"])
    Ar = sp.csr_array(-1 * rp.jac(z["rosen/x"]))
    rr = rp.res(z["rosen/x"])
    for pre in (True, False):
        # the oracle restatement against the reference
        x, it = orc.cgls(A, z["bratu/y"], preconditioner=pre, x0=z["bratu/x0"])
        assert it == int(z[f"bratu/it_pre{int(pre)}"]) and rel(x, z[f"bratu/x_pre{int(pre)}"]) < 1e-10
        x, it = orc.cgls(Ar, rr, preconditioner=pre, x0=z["rosen/x0"])
        assert it == int(z[f"rosen/it_pre{int(pre)}"]) and rel(x, z[f"rosen/x_pre{int(pre)}"]) < 1e-10
        # the package's entry point (host logic through the mock; the CUDA path is tests/test_gpu_kernels.py)
        x, it = g.cg_least_squares(Ad, z["bratu/y"], x0=z["bratu/x0"], preconditioner=pre)
        assert abs(it - int(z[f"bratu/it_pre{int(pre)}"])) <= 2 and rel(x, z[f"bratu/x_pre{int(pre)}"]) < 1e-6
        x, it = g.cg_least_squares(Ar, rr, x0=z["rosen/x0"], preconditioner=pre)
        assert abs(it - int(z[f"rosen/it_pre{int(pre)}"])) <= 1 and rel(x, z[f"rosen/x_pre{int(pre)}"]) < 1e-6


def test_reference_modules_pin_the_oracle():
    """The oracle port reproduces a run of the unmodified reference, stored by oracle/gen_golden.py in
    tests/golden/bratu_g34.npz (grid_nodes=34, i.e. odd m = 33; 39 iterations, restart after 12): same operator and
    start vector bit for bit, same counters and nfev sequence, iterates within 1e-11 up to the restart and 1e-9 after
    it (a restart amplifies last-bit differences, see tests/test_gpu_solvers.py).  Where oracle/_ref has been
    assembled (oracle/make_ref.sh), its files must also match their SHA-256 sums and a run of the imported reference
    must agree with the oracle."""
    from oracle import ref_loader, gnk_oracle as orc
    gd = Golden("bratu_g34")
    gr = gd.run("gnk_res_old")
    o = orc.BratuOracle(34, 5, 10)
    assert np.array_equal(o.operator(o.u_true), gd["y"]) and np.array_equal(o.start_vector(seed=42), gd["u0"])
    rec = Recorder(gr["sample_idx"], o.make_error())
    po = orc.gnk(o.make_res(gd["y"]), gd["u0"], o.make_jac(), restart=12, max_iter=40, callback=rec)
    check_trace(rec, gr, np.where(np.arange(len(gr["xnorm"])) < 12, 1e-11, 1e-9))
    assert (po["nit"], po["nfev"], po["njev"], po["success"]) == (
        int(gr["nit"]), int(gr["nfev"]), int(gr["njev"]), bool(gr["success"])) == (39, 40, 40, False)
    assert rel(po["x"], gr["x_final"]) < 1e-9
    if not ref_loader.available():
        return
    import hashlib
    sums = dict(line.split()[::-1] for line in open(os.path.join(ref_loader.REF_DIR, "SHA256SUMS")))
    for name, digest in sums.items():
        assert hashlib.sha256(open(os.path.join(ref_loader.REF_DIR, name), "rb").read()).hexdigest() == digest
        if os.path.isdir("/root/reference"):
            assert open(os.path.join(ref_loader.REF_DIR, name), "rb").read() == open(f"/root/reference/{name}", "rb").read()
    ref = ref_loader.load_reference()
    import sys
    assert "krylow" not in sys.modules or "_ref" not in getattr(sys.modules["krylow"], "__file__", "")
    pb = ref.bratu_pde_problem.BratuPdeProblem(34, 5, 10)
    y = pb.pde_operator(pb.u_true)
    np.random.seed(42)
    u0 = pb.u_true + 0.1 * np.random.normal(loc=0, scale=1, size=pb.u_true.shape[0])
    xs = []
    out = ref.gauss_newton_krylow.gauss_newton_krylow(pb.make_res(y), u0, pb.make_jac(), max_iter=15,
                                                      callback=lambda x, nfev, cg_iter: xs.append(x.copy()))
    o = orc.BratuOracle(34, 5, 10)
    assert np.array_equal(o.operator(o.u_true), y) and np.array_equal(o.start_vector(seed=42), u0)
    xo = []
    po = orc.gnk(o.make_res(y), u0, o.make_jac(), max_iter=15, callback=lambda x, nfev, cg_iter: xo.append(x.copy()))
    assert (po["nit"], po["nfev"], po["njev"]) == (out.nit, out.nrev, out.njev)
    assert max(rel(a, b) for a, b in zip(xo, xs)) < 1e-11


def test_speculative_expansion_changes_nothing(g, monkeypatch, capsys):
    """The basis expansion enqueued behind the first Armijo trial (GNK_SPECULATE, default on) against the expansion
    after the trial was judged: same iterates bit for bit, same counters, same messages -- on a run with accepted first
    trials (Bratu), on one with REJECTED first trials (the speculated expansion must be dropped and redone), with
    restarts, with a breakdown (the deferred flag travels through the second slot) and for every `version`."""
    from gauss_newton_via_generalized_krylov_subspaces_b200 import rosenbrock_problem as rp
    gd = Golden("bratu_g34")
    pb = g.BratuPdeProblem(34, 5, 10)
    res, jac = pb.make_res(gd["y"]), pb.make_jac()
    lin = g.BratuPdeProblem(25, 5, 0)
    gl = Golden("bratu_g25_linear")
    lres, ljac = lin.make_res(gl["y"]), lin.make_jac()

    def runs():
        out = []
        for version in ("res_old", "res_new", "jac_old_res_old", "jac_old_res_new"):
            xs = []
            o = g.gauss_newton_krylow(res, gd["u0"], jac, callback=lambda x, nfev, cg_iter: xs.append((np.array(x), nfev)),
                                      max_iter=18, krylow_restart=7, version=version)
            out.append((o.x, o.nit, o.nrev, o.njev, o.success, xs))
        # a start far from the valley: several trials per iteration are rejected (Armijo halving)
        x0 = np.full(1000, -1.5)
        xs = []
        o = g.gauss_newton_krylow(rp.res, x0, rp.jac, callback=lambda x, nfev, cg_iter: xs.append((np.array(x), nfev)),
                                  max_iter=12)
        assert o.nrev > o.nit + 1                      # halving happened
        out.append((o.x, o.nit, o.nrev, o.njev, o.success, xs))
        # breakdown at iteration 2 of the linear problem
        xs = []
        try:
            o = g.gauss_newton_krylow(lres, gl["u0"], ljac, callback=lambda x, nfev, cg_iter: xs.append((np.array(x), nfev)),
                                      max_iter=6)
            out.append((o.x, o.nit, o.nrev, o.njev, o.success, xs))
        except g.StepLengthConvergenceError:
            out.append((None, None, None, None, None, xs))
        return out, capsys.readouterr().out

    monkeypatch.setenv("GNK_SPECULATE", "1")
    a, msg_a = runs()
    monkeypatch.setenv("GNK_SPECULATE", "0")
    b, msg_b = runs()
    assert msg_a == msg_b and "breakdown" in msg_a
    for ra, rb in zip(a, b):
        assert ra[1:5] == rb[1:5]
        assert (ra[0] is None and rb[0] is None) or np.array_equal(ra[0], rb[0])
        assert len(ra[5]) == len(rb[5])
        for (xa, na), (xb, nb) in zip(ra[5], rb[5]):
            assert na == nb and np.array_equal(xa, xb)
