"""Krylov bases of 256..4095 columns (gauss_newton_krylow(max_basis_columns=...)): the wide streaming kernels
(gnk_combine_step, gnk_cgs_dots, gnk_cgs_update at k >= 256), the wide projected least squares (gnk_basis_ls_wide),
solver runs past 255 iterations without a restart against the oracle, and a basis that reaches the whole space."""
import ctypes as C
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

from golden_util import rel
from oracle import gnk_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def g():
    import gauss_newton_via_generalized_krylov_subspaces_b200 as pkg
    import gauss_newton_via_generalized_krylov_subspaces_b200.device as device
    device._runtime = None
    pkg.get_runtime()
    return pkg


def _flat(g, n, ld):
    from gauss_newton_via_generalized_krylov_subspaces_b200.device import make_layout
    from gauss_newton_via_generalized_krylov_subspaces_b200.partition import flat_layout_fields
    return make_layout(dict(flat_layout_fields(n), ld=ld))


def _dev(rt, a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(rt.device)


# ---- streaming kernels -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [256, 257, 300, 1000, 4095])
def test_wide_streaming_kernels_against_numpy(g, k):
    """x = V(c + s d) with c_out / cprev2, h = V^T w and w - V h with its statistics, against numpy (relative 1e-13 of
    the sum of magnitudes), bitwise repeatable, one launch per call; odd n exercises the tail element"""
    from gauss_newton_via_generalized_krylov_subspaces_b200.device import ptr
    rt, lib = g.get_runtime(), g.get_runtime().lib
    n, ld = 20001, 20002
    rs = np.random.RandomState(k)
    Vh = rs.normal(size=(k, ld))
    c, d, w0 = rs.normal(size=k), rs.normal(size=k), rs.normal(size=ld)
    s = 0.375
    V = _dev(rt, Vh).reshape(-1)
    lay = _flat(g, n, ld)
    dc, dd = _dev(rt, c), _dev(rt, d)
    outs = []
    for _ in range(2):
        x, cout, cp = rt.zeros(ld), rt.zeros(k + 1) - 1.0, rt.zeros(1)
        h, w, st = rt.zeros(k), _dev(rt, w0), rt.zeros(2)
        l0 = rt.launches()
        _lib_check(g, lib.gnk_combine_step(rt.ctx, C.byref(lay), ptr(V), k, ptr(dc), ptr(dd), s, ptr(x), ptr(cout),
                                           ptr(cp), rt.stream))
        _lib_check(g, lib.gnk_cgs_dots(rt.ctx, C.byref(lay), ptr(V), k, ptr(w), ptr(h), rt.stream))
        _lib_check(g, lib.gnk_cgs_update(rt.ctx, C.byref(lay), ptr(V), k, ptr(h), ptr(w), ptr(st), rt.stream))
        assert rt.launches() - l0 == 3
        rt.sync()
        outs.append([t.cpu().numpy().copy() for t in (x, cout, cp, h, w, st)])
    for a, b in zip(*outs):
        assert np.array_equal(a.view(np.int64), b.view(np.int64))
    x, cout, cp, h, w, st = outs[0]
    coef = c + s * d
    assert np.max(np.abs(cout[:k] - coef) / (np.abs(c) + np.abs(s * d))) <= 4.5e-16 and cout[k] == 0.0
    assert abs(cp[0] - c @ c) <= 1e-14 * (c @ c)
    assert np.all(np.abs(x - coef @ Vh) <= 1e-13 * (np.abs(coef) @ np.abs(Vh)))
    Vo = Vh[:, :n]
    assert np.all(np.abs(h - Vo @ w0[:n]) <= 1e-13 * (np.abs(Vo) @ np.abs(w0[:n])))
    wr = w0[:n] - h @ Vo
    assert np.all(np.abs(w[:n] - wr) <= 1e-13 * (np.abs(w0[:n]) + np.abs(h) @ np.abs(Vo)))
    assert np.array_equal(w[n:], w0[n:])
    assert abs(st[0] - wr @ wr) <= 1e-12 * (wr @ wr) and st[1] == np.max(np.abs(w[:n]))


def _lib_check(g, rc, what="call"):
    g._lib.check(rc, what)


def test_wide_kernels_reduce_like_the_narrow_ones(g):
    """per entry the wide kernels do the arithmetic of the 255-column kernels: h over the first 255 columns of a
    300-column basis, x and w with zero coefficients past column 255, and the 255-column calls themselves launch once"""
    from gauss_newton_via_generalized_krylov_subspaces_b200.device import ptr
    rt, lib = g.get_runtime(), g.get_runtime().lib
    n = ld = 1 << 18
    rs = np.random.RandomState(7)
    V = _dev(rt, rs.normal(size=(300, ld))).reshape(-1)
    w0 = _dev(rt, rs.normal(size=ld))
    coef = np.zeros(300)
    coef[:255] = rs.normal(size=255)
    dc = _dev(rt, coef)
    lay = _flat(g, n, ld)
    res = {}
    for k in (255, 300):
        x, h, w, st = rt.zeros(ld), rt.zeros(k), w0.clone(), rt.zeros(2)
        l0 = rt.launches()
        _lib_check(g, lib.gnk_combine(rt.ctx, C.byref(lay), ptr(V), k, ptr(dc), None, 0.0, ptr(x), rt.stream))
        _lib_check(g, lib.gnk_cgs_dots(rt.ctx, C.byref(lay), ptr(V), k, ptr(w0), ptr(h), rt.stream))
        _lib_check(g, lib.gnk_cgs_update(rt.ctx, C.byref(lay), ptr(V), k, ptr(dc), ptr(w), ptr(st), rt.stream))
        assert rt.launches() - l0 == 3
        res[k] = (x, h[:255], w, st)
    for a, b in zip(res[255], res[300]):
        assert bool((a == b).all())


# ---- wide least squares ------------------------------------------------------------------------------------------
def _graded_panel(rt, n, k, cond, seed):
    """A = H [S W^T; 0] with H three Householder reflectors, W orthogonal, singular values graded from 1 to 1/cond;
    y = A x + r with r orthogonal to range(A), |r| = 1e-3 |A x|.  Returns A, y (device) and the exact solution x."""
    import torch
    gen = torch.Generator(device=rt.device).manual_seed(seed)
    W, _ = torch.linalg.qr(torch.randn(k, k, generator=gen, device=rt.device, dtype=torch.float64))
    sv = torch.logspace(0, -np.log10(cond), k, device=rt.device, dtype=torch.float64)
    A = torch.zeros(n, k, device=rt.device, dtype=torch.float64)
    A[:k] = sv[:, None] * W.T
    x = torch.randn(k, generator=gen, device=rt.device, dtype=torch.float64)
    y = torch.zeros(n, device=rt.device, dtype=torch.float64)
    y[:k] = A[:k] @ x
    if n > k:
        r = torch.randn(n - k, generator=gen, device=rt.device, dtype=torch.float64)
        y[k:] = r * (1e-3 * torch.linalg.norm(y[:k]) / torch.linalg.norm(r))
    for _ in range(3):
        v = torch.randn(n, generator=gen, device=rt.device, dtype=torch.float64)
        v /= torch.linalg.norm(v)
        A -= 2.0 * torch.outer(v, v @ A)
        y -= 2.0 * v * (v @ y)
    return A, y, x


def _ls_wide(g, A, y, sign, lda=None):
    """gnk_basis_ls_wide on the panel [A | y] (column stride lda) -> the 2k + 4 result doubles"""
    from gauss_newton_via_generalized_krylov_subspaces_b200.device import ptr
    rt = g.get_runtime()
    n, k = A.shape
    lda = lda or (n + 15) // 16 * 16
    P = rt.zeros(lda * (k + 1))
    P.view(k + 1, lda)[:k, :n].copy_(A.T)
    P.view(k + 1, lda)[k, :n].copy_(y)
    out = rt.zeros(2 * k + 4)
    _lib_check(g, rt.lib.gnk_basis_ls_wide(rt.ctx, ptr(P), lda, n, k, float(sign), ptr(out), rt.stream))
    return rt.read(out, 2 * k + 4).copy()


@pytest.mark.parametrize("k", [256, 511, 1024, 4095])
@pytest.mark.parametrize("rows", ["k+1", "3k", "2^17"])
@pytest.mark.parametrize("cond", [10.0, 1e5])
def test_basis_ls_wide_graded(g, k, rows, cond):
    """the result block against the exact solution of a panel with known SVD (and numpy.linalg.lstsq where the panel is
    small), forward error within 1e-13 max(cond, 10) as for the narrower panels"""
    n = {"k+1": k + 1, "3k": 3 * k, "2^17": 1 << 17}[rows]
    rt = g.get_runtime()
    A, y, x = _graded_panel(rt, n, k, cond, seed=k + n)
    v = _ls_wide(g, A, y, -1.0)
    xr = -x.cpu().numpy()
    assert rel(v[:k], xr) <= 1e-13 * max(cond, 10.0), (rel(v[:k], xr), cond)
    if n * k <= 3 * 1024 * 1024:
        An, yn = A.cpu().numpy(), y.cpu().numpy()
        assert rel(v[:k], np.linalg.lstsq(-An, yn, rcond=None)[0]) <= 1e-13 * max(cond, 10.0)
    Ad = -(A @ A.new_tensor(v[:k]))
    ad2, r2 = float(Ad @ Ad), float(((y - Ad) ** 2).sum())
    assert abs(v[k] - ad2) <= 1e-10 * ad2 and abs(v[k + 1] - r2) <= 1e-8 * ad2 + 1e-6 * r2
    assert v[k + 2] == 0 and abs(v[k + 3] - v[:k] @ v[:k]) <= 1e-12 * (v[:k] @ v[:k])
    assert np.all(np.abs(v[k + 4:]) >= 0.5 / cond)


def test_basis_ls_wide_rank_deficiency_scaling_and_refusal(g, capsys):
    """exactly repeated columns are counted (and printed by the solver's report), a 2^40 scaling of the panel changes
    no bit, repeated calls give the same bits, and one rank refuses fewer than k + 1 rows"""
    from gauss_newton_via_generalized_krylov_subspaces_b200.gauss_newton_krylow import _report_rank
    rt = g.get_runtime()
    k, n = 300, 5000
    A, y, _ = _graded_panel(rt, n, k, 100.0, seed=3)
    A[:, 17] = A[:, 5]
    A[:, 200] = A[:, 5]
    v = _ls_wide(g, A, y, 1.0)
    assert v[k + 2] == 2
    try:
        _report_rank(v, k)
    except np.linalg.LinAlgError:  # an exactly zero pivot: printed first, then raised as scipy would
        pass
    assert capsys.readouterr().out.count("A is rank deficient") == 2
    A, y, _ = _graded_panel(rt, n, k, 1e3, seed=4)
    v1, v2 = _ls_wide(g, A, y, -1.0), _ls_wide(g, A, y, -1.0)
    assert np.array_equal(v1.view(np.int64), v2.view(np.int64))
    big = _ls_wide(g, A * 2.0 ** 40, y * 2.0 ** 40, -1.0)
    assert np.array_equal(big[:k], v1[:k])
    assert np.array_equal(big[k:k + 2], v1[k:k + 2] * 2.0 ** 80) and big[k + 2] == v1[k + 2]
    assert np.array_equal(big[k + 4:], v1[k + 4:] * 2.0 ** 40)
    with pytest.raises(g._lib.GnkError, match="fewer residuals"):
        _ls_wide(g, A[:k], y[:k], -1.0)
    with pytest.raises(g._lib.GnkError, match="k out of range"):
        _ls_wide(g, A[:, :255], y, -1.0)


def test_narrow_fused_paths_decline_wide_panels(g):
    """the fused trial/projection kernel (k <= 32), the fused stencil-Gram kernel (k <= 32) and the tensor-pipe Gram
    paths (<= 56 columns) are gated to narrow panels: a 300-column call is declined (1) or refused (< 0) without a
    launch, and the solver never makes it (test_bratu_g41_without_restart_past_255_columns profiles the run)"""
    import torch
    from gauss_newton_via_generalized_krylov_subspaces_b200.device import ptr
    rt, lib = g.get_runtime(), g.get_runtime().lib
    pb = g.BratuPdeProblem(257, 5, 10)
    d = pb.dev
    k = 300
    V = torch.randn((k + 1) * d.ld, dtype=torch.float64, device=rt.device)
    c, dd = rt.zeros(k + 1), rt.zeros(k + 1)
    x, w, F, expu = d.new_col(), d.new_col(), d.new_col(), d.new_col() + 1.0
    h, c_out, cp = rt.zeros(k + 1), rt.zeros(k + 1), rt.zeros(1)
    n = d.lay.n_own
    JV, out = rt.zeros(n * (k + 1)), rt.zeros(2 * k + 8)
    l0 = rt.launches()
    assert lib.gnk_bratu_trial_project(rt.ctx, C.byref(d.lay), C.byref(d.prm), ptr(V), k, ptr(c), ptr(dd), 1.0,
                                       ptr(x), ptr(c_out), ptr(cp), ptr(F), ptr(w), ptr(h), rt.stream) == 1
    assert lib.gnk_stencil_gram_ls(rt.ctx, C.byref(d.lay), C.byref(d.prm), ptr(expu), ptr(V), d.ld, k + 1, k, ptr(F),
                                   -1.0, ptr(JV), n, -1.0, ptr(out), rt.stream) < 0
    assert lib.gnk_gram_cgls(rt.ctx, ptr(JV), n, n, k, ptr(F), -1.0, 1e-4, ptr(out), rt.stream) < 0
    assert lib.gnk_tsqr_ls(rt.ctx, ptr(JV), n, n, k, ptr(F), -1.0, ptr(out), rt.stream) < 0
    assert rt.launches() == l0
    rt.sync()
    assert not x.any() and not w.any() and not h.any()


# ---- solver level --------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _oracle(version="res_old", reorth=1, cgls=False, G=41):
    o = orc.BratuOracle(G, 5, 10)
    y, u0 = o.operator(o.u_true), o.start_vector(seed=42)
    idx = np.random.RandomState(0).choice(o.n, 64, replace=False)
    trace = []
    kw = {}
    if cgls:
        kw["ls"] = lambda A, yy, log: orc.cgls(A, yy, rtol=1e-4, preconditioner=True)[0]
    ref = orc.gnk(o.make_res(y), u0, o.make_jac(), restart=None, max_iter=700, version=version, reorth=reorth,
                  callback=lambda x, **kw_: trace.append(np.asarray(x)[idx].copy()), **kw)
    return o, y, u0, idx, ref, trace


def test_bratu_g41_without_restart_past_255_columns(g):
    """the oracle converges with a basis of 311 columns: the same counts, the per-iteration deviation below 1e-10, the
    least squares of iterations 256.. on gnk_basis_ls_wide; without the keyword the run stops at column 256"""
    o, y, u0, idx, ref, rtrace = _oracle()
    assert (ref["nit"], ref["nfev"], ref["njev"], ref["success"]) == (311, 312, 311, True)
    pb = g.BratuPdeProblem(41, 5, 10)
    rt = g.get_runtime()
    trace = []
    rt.begin_profile()
    out = g.gauss_newton_krylow(pb.make_res(y), u0, pb.make_jac(), max_iter=700, max_basis_columns=700,
                                callback=lambda x, **kw: trace.append(np.asarray(x)[idx].copy()))
    prof = rt.end_profile()
    assert (out.nit, out.nrev, out.njev, out.success) == (311, 312, 311, True)
    dev = np.array([np.max(np.abs(a - b)) / np.max(np.abs(b)) for a, b in zip(trace, rtrace)])
    print(f"G=41 wide: max deviation through 255 {dev[:255].max():.2e}, 256..311 {dev[255:].max():.2e}")
    assert dev[:255].max() < 1e-10
    assert dev[255:].max() < 1e-10
    assert prof["ls_wide"]["launches"] == 311 - 255  # iterations 256 .. 311 have k = iteration columns
    assert not {"spmm+ls", "trial_project", "gram_cgls"} & set(prof) or prof.get("spmm+ls", {}).get("launches", 0) < 256
    with pytest.raises(g._lib.GnkError, match="wider than 255 columns"):
        g.gauss_newton_krylow(pb.make_res(y), u0, pb.make_jac(), max_iter=700, callback=lambda **kw: None)


@pytest.mark.parametrize("variant", ["res_new", "reorth2", "cgls", "host_csr", "torch_dense"])
def test_bratu_g41_wide_variants(g, variant):
    """one wide run per variant: counts equal to the oracle's (the CG-based run within 2 %).  res_new converges at
    iteration 218 on G = 41, so it runs on G = 46, where the oracle needs 273 iterations"""
    import torch
    version = "res_new" if variant == "res_new" else "res_old"
    reorth = 2 if variant == "reorth2" else 1
    G = 46 if variant == "res_new" else 41
    o, y, u0, idx, ref, _ = _oracle(version, reorth, variant == "cgls", G)
    pb = g.BratuPdeProblem(G, 5, 10)
    res, jac, x0 = pb.make_res(y), pb.make_jac(), u0
    kw = dict(version=version, reorth_passes=reorth)
    if variant == "cgls":
        kw["ls_solver"] = "cgls"
    if variant == "host_csr":
        res, jac = o.make_res(y), (lambda x, _j=o.make_jac(): _j(x).tocsr())
    if variant == "torch_dense":
        ores, ojac = o.make_res(y), o.make_jac()
        res = lambda x: torch.from_numpy(ores(x.cpu().numpy())).cuda()  # noqa: E731
        jac = lambda x: torch.from_numpy(ojac(x.cpu().numpy()).tocsr().toarray()).cuda()  # noqa: E731
        x0 = torch.from_numpy(u0).cuda()
    out = g.gauss_newton_krylow(res, x0, jac, max_iter=700, max_basis_columns=700, callback=lambda **k: None, **kw)
    got = (out.nit, out.nrev, out.njev, out.success)
    want = (ref["nit"], ref["nfev"], ref["njev"], ref["success"])
    print(f"G={G} wide {variant}: {got} oracle {want}")
    assert out.nit >= 256 and out.success == ref["success"]
    if variant == "cgls":
        assert abs(out.nit - ref["nit"]) <= 0.02 * ref["nit"] and abs(out.nrev - ref["nfev"]) <= 0.02 * ref["nfev"]
    else:
        assert got == want
    x = out.x.cpu().numpy() if hasattr(out.x, "cpu") else np.asarray(out.x)
    assert rel(x, ref["x"]) < 1e-6


def test_standalone_basis_reaches_the_whole_space(g):
    """n = 300 with random dense Jacobians and residuals: 299 updates, then GeneralizedKrylowSubspaceSpansEntireSpace;
    with two Gram-Schmidt passes V^T V stays at the identity to rounding level"""
    from gauss_newton_via_generalized_krylov_subspaces_b200.krylow import GeneralizedKrylowSubspaceSpansEntireSpace
    rs = np.random.RandomState(5)
    ks = g.GeneralizedKrylowSubspace(max_columns=300, reorth_passes=2)
    ks.start(rs.normal(size=300))
    for _ in range(299):
        ks.update(rs.normal(size=(400, 300)), rs.normal(size=400))
    assert ks.k == 300
    with pytest.raises(GeneralizedKrylowSubspaceSpansEntireSpace):
        ks.update(rs.normal(size=(400, 300)), rs.normal(size=400))
    V = ks.basis
    assert V.shape == (300, 300) and np.max(np.abs(V.T @ V - np.eye(300))) < 1e-12
    x = ks.x(np.arange(300.0))
    assert rel(x, V @ np.arange(300.0)) < 1e-13


def _gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.parametrize("nproc", [2, 8])
def test_wide_basis_multi_gpu(nproc):
    """several ranks: the sharded wide least squares (slabs with fewer rows than k + 1 included) and the G = 41 run with
    the oracle's counts, bit-identical on every rank (tests/wide_basis_worker.py)"""
    if _gpus() < nproc:
        pytest.skip(f"needs {nproc} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--standalone", f"--nproc-per-node={nproc}",
           os.path.join(ROOT, "tests", "wide_basis_worker.py")]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=1800, cwd=ROOT)
    print(p.stdout[-4000:], p.stderr[-4000:])
    assert p.returncode == 0 and "WIDE_BASIS_OK" in p.stdout
