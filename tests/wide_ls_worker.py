"""torchrun worker for the multi-rank blocked TSQR (launched by tests/test_gpu_wide_ls.py):

    python -m torch.distributed.run --nproc-per-node 2 tests/wide_ls_worker.py

Kernel level: every rank holds a row block of one global panel of 105..256 columns (rank 0 fewer rows than columns),
the result block must equal the global lstsq and be bit-identical on all ranks.  Solver level: Bratu G = 41 without a
restart for 256 iterations (panels up to 256 columns on slabs of a few grid rows) against the oracle.
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
    from gauss_newton_via_generalized_krylov_subspaces_b200.gauss_newton_krylow import tsqr_solve
    from golden_util import rel
    from oracle import gnk_oracle as orc

    rt = g.get_runtime()
    assert rt.world == world

    def gather_equal(x):
        t = torch.from_numpy(np.ascontiguousarray(x)).cuda()
        ts = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(ts, t)
        return all(torch.equal(ts[0], u) for u in ts[1:])

    for k in (104, 200, 255):
        rs = np.random.RandomState(k)
        rows = [100] + [30000 + 777 * r for r in range(1, world)]  # rank 0: fewer rows than columns
        n = sum(rows)
        A = rs.normal(size=(n, k)) @ (np.eye(k) + 0.3 * rs.normal(size=(k, k)) / np.sqrt(k))
        y = rs.normal(size=n)
        r0 = sum(rows[:rank])
        Al, yl = A[r0:r0 + rows[rank]], y[r0:r0 + rows[rank]]
        nl = rows[rank]
        lda = nl + 1
        dA = rt.zeros(lda * k)
        for j in range(k):
            rt.upload(np.ascontiguousarray(Al[:, j]), dA[j * lda:j * lda + nl])
        dy = rt.zeros(nl)
        rt.upload(yl, dy)
        out = rt.zeros(2 * 256 + 8)
        tsqr_solve(rt, dA, lda, nl, k, dy, -1.0, out)
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
            print(f"[wide-ls] N={world} k={k}: rel(d) {rel(v[:k], xr):.1e}, cond {cond:.1f}", flush=True)

    # ---- solver level: Bratu G = 41 without a restart, panels up to 256 columns ------------------
    G = 41
    o = orc.BratuOracle(G, 5, 10)
    yb, u0 = o.operator(o.u_true), o.start_vector(seed=42)
    idx = np.random.RandomState(0).choice(o.n, 64, replace=False)
    ref_trace, our_trace = [], []
    ref = orc.gnk(o.make_res(yb), u0, o.make_jac(), restart=None, max_iter=256,
                  callback=lambda x, **kw: ref_trace.append(np.asarray(x)[idx].copy()))
    pb = g.BratuPdeProblem(G, 5, 10)
    res = g.gauss_newton_krylow(pb.make_res(yb), u0, pb.make_jac(), krylow_restart=None, max_iter=256,
                                callback=lambda x, **kw: our_trace.append(np.asarray(x)[idx].copy()))
    assert (res.nit, res.nrev, res.njev) == (ref["nit"], ref["nfev"], ref["njev"]) == (255, 256, 256)
    dev = [float(np.max(np.abs(a - b)) / np.max(np.abs(b))) for a, b in zip(our_trace, ref_trace)]
    assert len(dev) == 255 and max(dev) < 1e-10, max(dev)
    assert gather_equal(np.asarray(res.x))
    if rank == 0:
        print(f"[wide-ls] N={world} G=41 no restart: max deviation {max(dev):.1e}", flush=True)
    print("WIDE_LS_OK", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
