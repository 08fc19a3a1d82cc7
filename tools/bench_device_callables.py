"""Bratu 1024^2, krylow_restart=30, 100 outer iterations, three ways: the native BratuPdeProblem, torch device
callables (residual in torch ops, CSR Jacobian with a fixed pattern and new values per call), and the same problem as
scipy host callables.  Also gauss_newton (CGLS) on the device callables, per CG iteration.  Prints one JSON document
(it/s, per-kernel-class times from CUDA events, card name and power limit read in the same run).

    python tools/bench_device_callables.py [--grid 1025] [--iters 100] [--out FILE]
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

import gauss_newton_via_generalized_krylov_subspaces_b200 as g  # noqa: E402
from oracle import gnk_oracle as orc  # noqa: E402
from torch_bratu import TorchBratu  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
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
    res_h = lambda x: res_n(x)  # noqa: E731  (wrapped: host-callable path)
    jac_h = lambda x: jac_n(x).tocsr()  # noqa: E731
    u0_d = torch.as_tensor(u0, device=rt.device)
    kw = dict(krylow_restart=30, max_iter=it + 1, tol=0.0, callback=lambda **k: None)
    ways = {"native": (res_n, jac_n, u0), "device_callables": (tb.res, tb.jac, u0_d), "host_callables": (res_h, jac_h, u0)}
    result = dict(card=card(), grid=G, unknowns=(G - 1) ** 2, krylow_restart=30, iterations=it, runs={})
    for name, (res, jac, x0) in ways.items():
        g.gauss_newton_krylow(res, x0, jac, **dict(kw, max_iter=4))  # warm-up: modules, cub temp sizes
        out, dt, _ = timed(rt, lambda: g.gauss_newton_krylow(res, x0, jac, **kw), False)
        result["runs"][name] = dict(seconds=dt, it_per_s=out.nit / dt, nit=out.nit, nfev=out.nrev)
        if name != "host_callables":  # per-kernel-class CUDA-event times, in a run of their own
            _, dtp, prof = timed(rt, lambda: g.gauss_newton_krylow(res, x0, jac, **kw), True)
            result["runs"][name].update(profiled_seconds=dtp,
                                        kernels_ms={k: round(v["ms"], 3) for k, v in sorted(prof.items())})
        print(name, f"{out.nit / dt:.1f} it/s", flush=True)
    # where the device-callable Jacobian's time goes: pattern compare (one int read back) and the J^T gather
    from gauss_newton_via_generalized_krylov_subspaces_b200.device import DeviceCallableProblem
    prob = DeviceCallableProblem(tb.res, tb.jac, u0_d, ())
    x = prob.new_sol()
    prob.upload_x(u0_d, x)
    prob.evaluate(x)
    J = tb.jac(u0_d)
    prob.jacobian(x)
    reps = 50
    rt.sync()
    t0 = time.perf_counter()
    for _ in range(reps):
        prob.pattern.matches(J.shape[0], J.shape[1], J.crow_indices(), J.col_indices(), prob._flag)
    rt.sync()
    t_cmp = (time.perf_counter() - t0) / reps
    from gauss_newton_via_generalized_krylov_subspaces_b200.device import CsrPattern, DeviceCsrJacobian
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        DeviceCsrJacobian(rt, prob.pattern, J.values(), True)
    e1.record()
    rt.sync()
    t_gather = e0.elapsed_time(e1) / reps / 1e3
    t0 = time.perf_counter()
    for _ in range(5):
        CsrPattern(rt, J.shape[0], J.shape[1], J.crow_indices(), J.col_indices())
    t_pattern = (time.perf_counter() - t0) / 5
    result["jacobian_ms"] = dict(pattern_compare_incl_readback=1e3 * t_cmp, gather_values_t=1e3 * t_gather,
                                 pattern_build=1e3 * t_pattern, nnz=int(J._nnz()))
    # gauss_newton (CGLS) on the device callables: time per CG iteration
    cgs = []
    g.gauss_newton(tb.res, u0_d, tb.jac, max_iter=2, callback=lambda **k: None)
    out, dt, _ = timed(rt, lambda: g.gauss_newton(tb.res, u0_d, tb.jac, max_iter=5,
                                                    callback=lambda x, nfev, cg_iter: cgs.append(cg_iter)), False)
    result["gauss_newton_device_callables"] = dict(seconds=dt, nit=out.nit, cg_iterations=int(sum(cgs)),
                                                   ms_per_cg_iteration=1e3 * dt / max(1, sum(cgs)))
    js = json.dumps(result, indent=1)
    print(js)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(js + "\n")


if __name__ == "__main__":
    main()
