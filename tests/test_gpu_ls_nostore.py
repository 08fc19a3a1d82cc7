"""The fused least squares without the J V_k store (-m gpu): gnk_stencil_gram_ls with d_JV = NULL recomputes J V_k in
its refinement pass (stencil_refine_kernel) instead of reading it back.

Everything up to the refinement (Gram matrix, first factor, refinement decision) is bit-identical to the storing call;
d is the refinement of the same d0 with g summed in another order, so it agrees to rounding.
"""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from golden_util import Recorder, rel  # noqa: E402
from oracle import gnk_oracle as orc  # noqa: E402


@pytest.fixture(scope="module")
def g():
    import gauss_newton_via_generalized_krylov_subspaces_b200 as pkg
    import gauss_newton_via_generalized_krylov_subspaces_b200.device as device
    device._runtime = None
    pkg.get_runtime()  # raises without CUDA + the built library: no fallback
    return pkg


def _panel(g, G, k, lam, dup=False):
    from gauss_newton_via_generalized_krylov_subspaces_b200 import device
    pb = g.BratuPdeProblem(G, 5, lam)
    d = pb.dev
    n, ld = d.fields["n_own"], d.ld
    assert pb.m % 8 == 0 and n >= 16384
    rs = np.random.RandomState(G * 100 + k)
    cap = k + 2
    V = d.rt.zeros(cap * ld)
    for j in range(cap):
        d.upload_x(rs.normal(size=pb.n), V[j * ld:(j + 1) * ld])
    if dup:  # two equal basis columns: the Gram matrix is singular
        V[ld:2 * ld].copy_(V[:ld])
    u, r = d.new_col(), d.new_col()
    d.upload_x(0.3 * rs.normal(size=pb.n), u)
    d.upload_x(rs.normal(size=pb.n), r)
    E = None
    if lam != 0:
        E = d.new_col()
        d.residual_into(u, d.zero_col(), d.new_col(), E, d.scal_tmp, depth=0)
    ldjv = (n + 15) // 16 * 16

    def fused(JV, out):
        return d.rt.lib.gnk_stencil_gram_ls(d.rt.ctx, C.byref(d.lay), C.byref(d.prm), device.ptr(E), device.ptr(V), ld,
                                            cap, k, device.ptr(r), -1.0, device.ptr(JV), ldjv, -1.0, device.ptr(out),
                                            d.rt.stream)
    return d, V, r, E, ldjv, fused


@pytest.mark.parametrize("G,k,lam", [(129, 7, 10.0), (137, 8, 10.0), (201, 15, 10.0), (257, 16, 3.0), (265, 23, 10.0),
                                      (513, 24, 10.0), (521, 31, 10.0), (1025, 30, 10.0), (193, 12, 0.0),
                                      (145, 30, 0.0)])
def test_store_free_matches_storing_call_and_lstsq(g, G, k, lam):
    """1..4 column blocks; row counts that are not a multiple of the strip height; row lengths with partial 64-point
    tiles (m = 136, 200, 264, 520, 144); lam = 0 (no e^u plane)"""
    d, V, r, E, ldjv, fused = _panel(g, G, k, lam)
    rt, n, off = d.rt, d.fields["n_own"], d.fields["off"]
    JV = rt.zeros(k * ldjv)
    a, b = rt.zeros(256), rt.zeros(256)
    assert fused(JV, a) == 0
    assert fused(None, b) == 0
    va, vb = rt.read(a, 2 * k + 4), rt.read(b, 2 * k + 4)
    JVa = rt.zeros(k * ldjv)
    d.apply(E, V, d.ld, k, -1.0, 0, JVa, ldjv, 0)
    assert np.array_equal(rt.download(JVa), rt.download(JV))
    JVh = rt.download(JV).reshape(k, ldjv)[:, :n].T
    dref = np.linalg.lstsq(-JVh, rt.download(r[off:off + n]), rcond=None)[0]
    cond = np.linalg.cond(JVh)
    assert va[k + 2] == 0 and vb[k + 2] == 0
    # the diagonal of R is R1's, written before the refinement: same bits
    assert np.array_equal(vb[k + 4:2 * k + 4], va[k + 4:2 * k + 4])
    assert rel(vb[:k], dref) < 1e-13 * max(cond, 10.0) and rel(vb[:k], va[:k]) < 1e-13 * max(cond, 10.0)
    assert np.allclose(vb[k:k + 4], va[k:k + 4], rtol=1e-9, atol=0)            # |A d|^2, resid^2, ndef, |d|^2
    # run-to-run deterministic
    b2 = rt.zeros(256)
    assert fused(None, b2) == 0
    assert np.array_equal(rt.read(b2, 2 * k + 4), vb)


def test_store_free_refuses_singular_panel_and_householder_takes_over(g):
    """two equal basis columns: the store-free call refuses (out[k+2] = -1, d = 0) like the storing call; the host's
    fallback -- J V from gnk_stencil_apply, then the Householder TSQR -- gives the Householder result"""
    from gauss_newton_via_generalized_krylov_subspaces_b200.gauss_newton_krylow import tsqr_solve
    k = 9
    d, V, r, E, ldjv, fused = _panel(g, 257, k, 10.0, dup=True)
    rt, n, off = d.rt, d.fields["n_own"], d.fields["off"]
    JVs = rt.zeros(k * ldjv)
    a, b = rt.zeros(256), rt.zeros(256)
    assert fused(JVs, a) == 0 and fused(None, b) == 0
    va, vb = rt.read(a, 2 * k + 4), rt.read(b, 2 * k + 4)
    assert va[k + 2] == -1 and vb[k + 2] == -1
    assert np.array_equal(vb[:k], np.zeros(k))
    JV = rt.zeros(k * ldjv)
    d.apply(E, V, d.ld, k, -1.0, 0, JV, ldjv, 0)
    assert np.array_equal(rt.download(JV), rt.download(JVs))
    tsqr_solve(rt, JV, ldjv, n, k, r[off:], -1.0, b, householder=True)
    ref = rt.zeros(256)
    tsqr_solve(rt, JVs, ldjv, n, k, r[off:], -1.0, ref, householder=True)
    vb, vr = rt.read(b, 2 * k + 4), rt.read(ref, 2 * k + 4)
    assert np.array_equal(vb, vr) and vb[k + 2] != -1


def test_bratu_257_k30_matches_oracle(g):
    """Bratu 257^2 (65536 unknowns: every panel from k = 7 on takes the store-free fused path), 30 outer iterations,
    k = 1..30: counts and nfev sequence equal to the oracle's, iterates within 1e-9 relative"""
    G, alpha, lam = 257, 5, 10
    o = orc.BratuOracle(G, alpha, lam)
    y = o.operator(o.u_true)
    u0 = o.start_vector(seed=7)
    idx = np.arange(0, len(u0), 97)
    rec_o = Recorder(idx)
    ref = orc.gnk(o.make_res(y), u0, o.make_jac(), max_iter=31, callback=rec_o)
    pb = g.BratuPdeProblem(G, alpha, lam)
    rec = Recorder(idx)
    out = g.gauss_newton_krylow(pb.make_res(y), u0, pb.make_jac(), max_iter=31, callback=rec)
    assert (out.nit, out.nrev, bool(out.success)) == (ref["nit"], ref["nfev"], bool(ref["success"]))
    assert rec.nfev == rec_o.nfev and len(rec.xs) == len(rec_o.xs)
    xs, xo = np.array(rec.xs), np.array(rec_o.xs)
    assert np.max(np.abs(xs - xo) / np.max(np.abs(xo), axis=1, keepdims=True)) < 1e-9
    assert rel(out.x, ref["x"]) < 1e-9
