"""gnk_bratu_trial_project (-m gpu): the speculative Armijo trial point, -J(x)^T F and V_k^T w in one pass over the
basis must be bit-identical to the four calls it replaces (gnk_combine_step, gnk_bratu_residual's e^x,
gnk_stencil_apply transposed, gnk_cgs_dots), and a solve that takes it must follow today's trajectory bit for bit.
"""
import ctypes as C
import hashlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import gnk_oracle as orc  # noqa: E402


@pytest.fixture(scope="module")
def g():
    import gauss_newton_via_generalized_krylov_subspaces_b200 as pkg
    import gauss_newton_via_generalized_krylov_subspaces_b200.device as device
    device._runtime = None
    pkg.get_runtime()
    return pkg


_CASES = {}


def _case(g, G, lam):
    """problem, basis of 34 stored columns (halo rows included, all random), F, c, d -- one per (G, lam)"""
    key = (G, lam)
    if key not in _CASES:
        import torch
        pb = g.BratuPdeProblem(G, 5, lam)
        d = pb.dev
        gen = torch.Generator(device=d.rt.device).manual_seed(G)
        ncol = 34
        V = torch.randn(ncol * d.ld, dtype=torch.float64, device=d.rt.device, generator=gen) / np.sqrt(30.0)
        F = torch.randn(d.ld, dtype=torch.float64, device=d.rt.device, generator=gen) * 1e3
        c = torch.zeros(256, dtype=torch.float64, device=d.rt.device)
        dd = torch.zeros(256, dtype=torch.float64, device=d.rt.device)
        c[:ncol] = torch.randn(ncol, dtype=torch.float64, device=d.rt.device, generator=gen)
        dd[:ncol] = torch.randn(ncol, dtype=torch.float64, device=d.rt.device, generator=gen)
        _CASES[key] = (pb, V, F, c, dd)
    return _CASES[key]


def _separate(g, pb, V, F, c, dd, k, s):
    from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib
    from gauss_newton_via_generalized_krylov_subspaces_b200.device import ptr
    d = pb.dev
    rt, lay = d.rt, C.byref(d.lay)
    x, w, expu = d.new_col(), d.new_col(), d.new_col()
    h, c_out, cprev2 = rt.zeros(256), rt.zeros(256), rt.zeros(1)
    _lib.check(rt.lib.gnk_combine_step(rt.ctx, lay, ptr(V), k, ptr(c), ptr(dd), s, ptr(x), ptr(c_out), ptr(cprev2),
                                       rt.stream))
    _lib.check(rt.lib.gnk_bratu_residual(rt.ctx, lay, C.byref(d.prm), ptr(x), ptr(d.zero_col()), ptr(d.new_col()),
                                         ptr(expu), 1, ptr(rt.zeros(1)), rt.stream))
    _lib.check(rt.lib.gnk_stencil_apply(rt.ctx, lay, C.byref(d.prm), ptr(expu), ptr(F), d.ld, 1, 1.0, 1, ptr(w), d.ld,
                                        d.fields["off"], rt.stream))
    _lib.check(rt.lib.gnk_cgs_dots(rt.ctx, lay, ptr(V), k, ptr(w), ptr(h), rt.stream))
    return x, w, h, c_out, cprev2


def _fused(g, pb, V, F, c, dd, k, s):
    from gauss_newton_via_generalized_krylov_subspaces_b200.device import ptr
    d = pb.dev
    rt = d.rt
    x, w = d.new_col(), d.new_col()
    h, c_out, cprev2 = rt.zeros(256), rt.zeros(256), rt.zeros(1)
    rc = rt.lib.gnk_bratu_trial_project(rt.ctx, C.byref(d.lay), C.byref(d.prm), ptr(V), k, ptr(c), ptr(dd), s,
                                        ptr(x), ptr(c_out), ptr(cprev2), ptr(F), ptr(w), ptr(h), rt.stream)
    return rc, (x, w, h, c_out, cprev2)


def _np(ts):
    return [t.cpu().numpy() for t in ts]


# G = 129 / 257: dots' grid of 8 and 32 CTAs; 2049: its cap of 4 CTAs per SM
@pytest.mark.parametrize("G", [129, 257, 2049])
@pytest.mark.parametrize("lam", [10, 0])
@pytest.mark.parametrize("k", [1, 2, 7, 8, 9, 16, 23, 30, 32])
@pytest.mark.parametrize("s", [1.0, 0.5])
def test_trial_project_is_bit_identical_to_the_separate_kernels(g, G, lam, k, s):
    pb, V, F, c, dd = _case(g, G, lam)
    ref = _np(_separate(g, pb, V, F, c, dd, k, s))   # columns >= k of V and entries >= k of c, d hold data
    rc, out = _fused(g, pb, V, F, c, dd, k, s)
    assert rc == 0
    out = _np(out)
    names = ("x", "w", "h", "c_out", "cprev2")
    for name, a, b in zip(names, out, ref):
        assert np.array_equal(a, b), (name, float(np.max(np.abs(a - b))))
    assert np.all(out[2][k:] == 0.0) and np.all(out[3][k + 1:] == 0.0)
    rc2, again = _fused(g, pb, V, F, c, dd, k, s)
    assert rc2 == 0
    for name, a, b in zip(names, _np(again), out):
        assert np.array_equal(a, b), name


def test_trial_project_declines_what_it_does_not_take(g):
    pb, V, F, c, dd = _case(g, 257, 10)
    rc, (x, w, h, _, _) = _fused(g, pb, V, F, c, dd, 33, 1.0)
    assert rc == 1 and not x.any() and not w.any() and not h.any()
    odd = g.BratuPdeProblem(130, 5, 10)   # m = 129
    d = odd.dev
    Vo = d.rt.zeros(4 * d.ld) + 1.0
    rc, (x, w, h, _, _) = _fused(g, odd, Vo, d.new_col(), c, dd, 3, 1.0)
    assert rc == 1 and not x.any() and not w.any() and not h.any()


# ------------------------------------------------------------------------------------------------
# solver level: the fused pass changes no bit of the trajectory
# ------------------------------------------------------------------------------------------------
def _solve(g, G, max_iter, restart, monkeypatch, speculate, version="res_old"):
    monkeypatch.setenv("GNK_SPECULATE", "1" if speculate else "0")
    o = orc.BratuOracle(G, 5, 10)
    y = o.operator(o.u_true)
    u0 = o.start_vector(seed=42)
    pb = g.BratuPdeProblem(G, 5, 10)
    digests = []

    def cb(x, nfev, cg_iter):
        digests.append((hashlib.sha256(np.ascontiguousarray(np.asarray(x)).tobytes()).hexdigest(), nfev))

    rt = g.get_runtime()
    rt.begin_profile()
    out = g.gauss_newton_krylow(pb.make_res(y), u0, pb.make_jac(), krylow_restart=restart, max_iter=max_iter,
                                callback=cb, version=version)
    prof = rt.end_profile()
    return out, digests, prof


@pytest.mark.parametrize("G,max_iter,restart", [(1025, 100, 30), (4097, 31, None)])
def test_solve_with_the_fused_trial_matches_the_unspeculated_sequence(g, monkeypatch, G, max_iter, restart):
    out, digests, prof = _solve(g, G, max_iter, restart, monkeypatch, speculate=True)
    ref, ref_digests, ref_prof = _solve(g, G, max_iter, restart, monkeypatch, speculate=False)
    assert "trial_project" not in ref_prof
    speculated = sum(1 for it in range(1, out.nit + 1) if it + 1 < max_iter and (restart is None or it % restart))
    assert prof["trial_project"]["launches"] >= speculated > 0
    assert prof["cgs_dots"]["launches"] < ref_prof["cgs_dots"]["launches"]
    assert len(digests) == len(ref_digests) and digests == ref_digests
    assert (out.nit, out.nrev, out.njev, out.success) == (ref.nit, ref.nrev, ref.njev, ref.success)
    assert np.array_equal(out.x, ref.x)


def test_res_new_keeps_the_separate_kernels(g, monkeypatch):
    out, _, prof = _solve(g, 1025, 10, None, monkeypatch, speculate=True, version="res_new")
    assert "trial_project" not in prof and prof["cgs_dots"]["launches"] >= out.nit - 1
