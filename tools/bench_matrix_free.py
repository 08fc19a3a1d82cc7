"""Matrix-free Jacobians in gauss_newton_krylow: Bratu 1024^2, krylow_restart=30, 100 outer iterations, five ways --
the native BratuPdeProblem, torch device callables returning the CSR Jacobian, a DeviceLinearOperator over the same CSR
tensor, autograd_jacobian of the torch residual (J V_k by vmap over jvp, J^T r by vjp), and a scipy LinearOperator
over the host CSR matrix.  Prints one JSON document: it/s per way; from a profiled run of its own, a CUDA-event split
into the user's products, the copy into the J V_k panel and the library's kernels; basis bytes downloaded per
iteration by the host path; and the card's name, power limit and SM clocks read in the same run.

    python tools/bench_matrix_free.py [--grid 1025] [--iters 100] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import numpy as np  # noqa: E402
import torch  # noqa: E402
from scipy.sparse.linalg import aslinearoperator  # noqa: E402

import gauss_newton_via_generalized_krylov_subspaces_b200 as g  # noqa: E402
from oracle import gnk_oracle as orc  # noqa: E402
from torch_bratu import TorchBratu  # noqa: E402

# marks recorded inside an operator Jacobian's products (device.py), nested in the solver's "spmm" / "spmv_t" marks
USER = ("op_matmat", "op_rmatvec")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def timed(rt, fn, profile):
    if profile:
        rt.begin_profile()
    rt.sync()
    t0 = time.perf_counter()
    out = fn()
    rt.sync()
    dt = time.perf_counter() - t0
    prof = rt.end_profile() if profile else None
    return out, dt, prof


def split(prof, nit):
    """ms per iteration: the user's products, the panel copy, the library's kernels (every other mark)"""
    ms = {k: v["ms"] for k, v in prof.items()}
    user = sum(ms.get(k, 0.0) for k in USER)
    panel = ms.get("panel_copy", 0.0)
    # the operator marks are counted twice in the sum, once on their own and once inside "spmm" / "spmv_t"; without
    # them (CSR products, the native stencil) every mark is a library kernel
    library = sum(ms.values()) - 2.0 * (user + panel)
    return dict(user_products_ms_per_it=user / nit, panel_copy_ms_per_it=panel / nit,
                library_kernels_ms_per_it=library / nit, marks_ms={k: round(v, 3) for k, v in sorted(ms.items())},
                marks_launches={k: v["launches"] for k, v in sorted(prof.items())})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grid", type=int, default=1025)
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    rt = g.get_runtime()
    G, it = a.grid, a.iters
    o = orc.BratuOracle(G, 5, 10)
    y = o.operator(o.u_true)
    u0 = o.start_vector(seed=42)
    pb = g.BratuPdeProblem(G, 5, 10)
    tb = TorchBratu(pb, o, y, rt.device)
    res_n, jac_n = pb.make_res(y), pb.make_jac()
    u0_d = torch.as_tensor(u0, device=rt.device)

    def jac_op(x):
        J = tb.jac(x)
        return g.DeviceLinearOperator(J.shape, matvec=lambda v: J @ v, matmat=lambda V: J @ V,
                                      rmatvec=lambda u: J.t() @ u)

    ways = {
        "native": (res_n, jac_n, u0),
        "device_callables_csr": (tb.res, tb.jac, u0_d),
        "device_linear_operator_csr": (tb.res, jac_op, u0_d),
        "autograd_jacobian": (tb.res, g.autograd_jacobian(tb.res), u0_d),
        "host_linear_operator": (lambda x: res_n(x), lambda x: aslinearoperator(jac_n(x).tocsr()), u0),
    }
    kw = dict(krylow_restart=30, max_iter=it + 1, tol=0.0, callback=lambda **k: None)
    result = dict(card=card(), card_fields="name, power.limit, clocks.sm, clocks.max.sm", grid=G,
                  unknowns=(G - 1) ** 2, krylow_restart=30, iterations=it, runs={})
    xs = {}
    for name, (res, jac, x0) in ways.items():
        g.gauss_newton_krylow(res, x0, jac, **dict(kw, max_iter=4))  # warm-up: modules, cub / cuSPARSE work sizes
        out, dt, _ = timed(rt, lambda: g.gauss_newton_krylow(res, x0, jac, **kw), False)
        xs[name] = out.x.cpu().numpy() if hasattr(out.x, "cpu") else np.asarray(out.x)
        run = dict(seconds=dt, it_per_s=out.nit / dt, nit=out.nit, nfev=out.nrev)
        downloads = {"basis": 0, "all": 0, "calls": 0}
        real = rt.download

        def counting(t):
            downloads["all"] += t.numel() * t.element_size()
            downloads["calls"] += 1
            if t.dim() == 2:  # only the host basis mirror downloads 2-D blocks
                downloads["basis"] += t.numel() * t.element_size()
            return real(t)

        rt.download = counting
        try:
            outp, dtp, prof = timed(rt, lambda: g.gauss_newton_krylow(res, x0, jac, **kw), True)
        finally:
            rt.download = real
        run.update(profiled_seconds=dtp, **split(prof, outp.nit))
        if name == "host_linear_operator":
            run.update(basis_download_bytes_per_it=downloads["basis"] / outp.nit,
                       all_download_bytes_per_it=downloads["all"] / outp.nit,
                       downloads_per_it=downloads["calls"] / outp.nit,
                       basis_bytes_per_new_column=8 * (G - 1) ** 2)
        result["runs"][name] = run
        print(name, f"{run['it_per_s']:.1f} it/s", flush=True)
    ref = xs["native"]
    result["max_rel_dev_of_x_vs_native"] = {k: float(np.max(np.abs(v - ref)) / np.max(np.abs(ref)))
                                             for k, v in xs.items()}
    js = json.dumps(result, indent=1)
    print(js)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(js + "\n")


if __name__ == "__main__":
    main()
