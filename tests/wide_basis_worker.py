"""torchrun worker for Krylov bases past 255 columns on several ranks (launched by tests/test_gpu_wide_basis.py):

    python -m torch.distributed.run --nproc-per-node 2 tests/wide_basis_worker.py

Kernel level: every rank holds a row block of one global panel [A | y] of 256..1024 columns (rank 0 fewer rows than
k + 1, so its slab goes through the zero-padded scratch panel); gnk_basis_ls_wide must equal the global lstsq and give
the same bits on all ranks.  Solver level: Bratu G = 41 without a restart (the oracle converges with 311 columns) with
max_basis_columns=700: the oracle's counts, and the same x on every rank.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    import torch
    import torch.distributed as dist

    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    import gauss_newton_via_generalized_krylov_subspaces_b200 as g
    from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib
    from gauss_newton_via_generalized_krylov_subspaces_b200.device import ptr
    from golden_util import rel
    from oracle import gnk_oracle as orc

    rt = g.get_runtime()
    assert rt.world == world

    def gather_equal(x):
        t = torch.from_numpy(np.ascontiguousarray(x)).cuda()
        ts = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(ts, t)
        return all(torch.equal(ts[0], u) for u in ts[1:])

    for k in (256, 300, 1024):
        rs = np.random.RandomState(k)
        rows = [100] + [3000 + 77 * r for r in range(1, world)]  # rank 0: fewer rows than k + 1
        n = sum(rows)
        A = rs.normal(size=(n, k)) @ (np.eye(k) + 0.3 * rs.normal(size=(k, k)) / np.sqrt(k))
        y = rs.normal(size=n)
        r0, nl = sum(rows[:rank]), rows[rank]
        lda = nl + 1
        P = rt.zeros(lda * (k + 1))
        P.view(k + 1, lda)[:k, :nl].copy_(torch.from_numpy(A[r0:r0 + nl].T.copy()))
        P.view(k + 1, lda)[k, :nl].copy_(torch.from_numpy(y[r0:r0 + nl]))
        out = rt.zeros(2 * k + 4)
        _lib.check(rt.lib.gnk_basis_ls_wide(rt.ctx, ptr(P), lda, nl, k, -1.0, ptr(out), rt.stream), "gnk_basis_ls_wide")
        v = rt.read(out, 2 * k + 4).copy()
        xr = np.linalg.lstsq(-A, y, rcond=None)[0]
        cond = np.linalg.cond(A)
        assert rel(v[:k], xr) <= 1e-13 * max(cond, 10.0), (k, rel(v[:k], xr), cond)
        Ad = -(A @ v[:k])
        assert abs(v[k] - Ad @ Ad) <= 1e-10 * (Ad @ Ad)
        assert abs(v[k + 1] - np.sum((y - Ad) ** 2)) <= 1e-10 * (y @ y)
        assert v[k + 2] == 0
        assert gather_equal(v), f"result blocks differ between ranks (k={k})"
        if rank == 0:
            print(f"[wide-basis] N={world} k={k}: rel(d) {rel(v[:k], xr):.1e}, cond {cond:.1f}", flush=True)

    G = 41
    o = orc.BratuOracle(G, 5, 10)
    yb, u0 = o.operator(o.u_true), o.start_vector(seed=42)
    pb = g.BratuPdeProblem(G, 5, 10)
    res = g.gauss_newton_krylow(pb.make_res(yb), u0, pb.make_jac(), max_iter=700, max_basis_columns=700,
                                callback=lambda **kw: None)
    assert (res.nit, res.nrev, res.njev, res.success) == (311, 312, 311, True), (res.nit, res.nrev, res.njev)
    x = np.asarray(res.x)
    assert gather_equal(x)
    ref = orc.gnk(o.make_res(yb), u0, o.make_jac(), restart=None, max_iter=700) if rank == 0 else None
    if rank == 0:
        assert (ref["nit"], ref["nfev"], ref["njev"]) == (311, 312, 311)
        print(f"[wide-basis] N={world} G=41 no restart: rel(x, oracle) {rel(x, ref['x']):.1e}", flush=True)
        assert rel(x, ref["x"]) < 1e-8
    print("WIDE_BASIS_OK", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
