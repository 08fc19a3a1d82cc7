"""Dense device Jacobians in gauss_newton_krylow: used as they arrive (gnk_dense_matmat / gnk_dense_rmatvec) against the
same matrices handed over as torch CSR (the route every dense device Jacobian took before: CSR copy, pattern compare,
J^T gather, gnk_spmm_csr).  Shapes 2^17 x 4096, 2^20 x 1024 and 1 049 600 x 2048 (2.15e9 entries, which the CSR route
refuses).  The problem is linear, r(x) = J x - y with columns graded over three decades; jac returns the same tensor
at every call.  A solve converges to rounding level within a few dozen iterations (after which the Armijo rule can no
longer find a decrease), so the it/s come from --repeat solves of --iters iterations each from the same start.  Prints one JSON document: GNK it/s both ways,
per-iteration J V_k and J^T r times (CUDA events, a profiled run of its own), what the CSR route spends on
conversion / pattern compare / gather per Jacobian, and the kernels alone with their HBM and FP64-pipe fractions.
Card, SM clock and power limit are read in the same run.

    python tools/bench_dense_jacobian.py [--iters 6] [--repeat 5] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT]

import torch  # noqa: E402

import gauss_newton_via_generalized_krylov_subspaces_b200 as g  # noqa: E402
from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib  # noqa: E402
from gauss_newton_via_generalized_krylov_subspaces_b200.device import (DeviceCallableProblem,  # noqa: E402
                                                                       DeviceCsrJacobian, ptr)

HBM_TBS = 7.7          # HGX B200 data sheet, per GPU
FP64_DFMA_TFLOPS = 34.2  # DFMA peak measured on this project's B200s (profiles/r01_fp64_peak.json)
SHAPES = [(1 << 17, 4096), (1 << 20, 1024), (1049600, 2048)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def event_ms(fn, reps):
    fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


def gnk(rt, J, y, x0, jac, iters, repeat, profile):
    """repeat solves of iters outer iterations -> (iterations, seconds, per-class CUDA-event ms or None)"""
    kw = dict(max_iter=iters + 1, tol=0.0, callback=lambda **k: None)
    res = lambda x: J @ x - y  # noqa: E731
    if profile:
        rt.begin_profile()
    rt.sync()
    t0 = time.perf_counter()
    nit = sum(g.gauss_newton_krylow(res, x0, jac, **kw).nit for _ in range(repeat))
    rt.sync()
    dt = time.perf_counter() - t0
    prof = rt.end_profile() if profile else None
    return nit, dt, prof


def kernels(rt, J, n, p, reps):
    """gnk_dense_matmat at k = 1, 8, 30, 64, 255 and gnk_dense_rmatvec alone (CUDA events, J resident in HBM)"""
    out = {}
    for k in (1, 8, 30, 64, 255):
        V = torch.randn(p * k, dtype=torch.float64, device=rt.device)
        JV = torch.empty(n * k, dtype=torch.float64, device=rt.device)
        ms = event_ms(lambda: rt.lib.gnk_dense_matmat(rt.ctx, n, p, ptr(J), p, 1, ptr(V), p, 0, k, 1.0, ptr(JV), n, 0,
                                                      rt.stream), reps)
        nbytes, flops = 8.0 * (n * p + p * k + n * k), 2.0 * n * p * k
        out[f"matmat_k{k}"] = dict(ms=ms, hbm_fraction=nbytes / (ms * 1e-3) / (HBM_TBS * 1e12),
                                   fp64_fraction=flops / (ms * 1e-3) / (FP64_DFMA_TFLOPS * 1e12))
        del V, JV
    r = torch.randn(n, dtype=torch.float64, device=rt.device)
    w = torch.empty(p, dtype=torch.float64, device=rt.device)
    ms = event_ms(lambda: rt.lib.gnk_dense_rmatvec(rt.ctx, n, p, ptr(J), p, 1, ptr(r), -1.0, ptr(w), rt.stream), reps)
    out["rmatvec"] = dict(ms=ms, hbm_fraction=8.0 * (n * p + n + p) / (ms * 1e-3) / (HBM_TBS * 1e12))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=6)
    ap.add_argument("--repeat", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    rt = g.get_runtime()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    result = dict(card_name_power_limit_sm_clock_max_sm_clock=card(), iterations_per_solve=a.iters, solves=a.repeat,
                  peaks=dict(hbm_tbs=HBM_TBS, fp64_dfma_tflops=FP64_DFMA_TFLOPS), shapes={})
    for n, p in SHAPES:
        torch.cuda.empty_cache()
        gen = torch.Generator(device=rt.device).manual_seed(1)
        J = torch.randn(n, p, dtype=torch.float64, device=rt.device, generator=gen)
        J *= torch.logspace(0, -3, p, dtype=torch.float64, device=rt.device)
        y = J @ torch.randn(p, dtype=torch.float64, device=rt.device, generator=gen)
        x0 = torch.ones(p, dtype=torch.float64, device=rt.device)
        row = dict(entries=n * p, gib=8.0 * n * p / 2 ** 30)
        ways = {"dense": lambda x: J, "csr": lambda x: J.to_sparse_csr()}
        for name, jac in ways.items():
            try:
                gnk(rt, J, y, x0, jac, a.iters, 1, False)  # warm-up: modules, cub temp sizes
                nit, dt, _ = gnk(rt, J, y, x0, jac, a.iters, a.repeat, False)
                nitp, _, prof = gnk(rt, J, y, x0, jac, a.iters, a.repeat, True)
                per_it = {k: v["ms"] / nitp for k, v in sorted(prof.items())}
                row[name] = dict(seconds=dt, it_per_s=nit / dt, nit=nit, profiled_ms_per_iteration=per_it)
            except (_lib.GnkError, torch.OutOfMemoryError) as e:
                row[name] = dict(refused=str(e).splitlines()[0])
            except g.StepLengthConvergenceError as e:
                row[name] = dict(error=str(e).splitlines()[0])
            torch.cuda.empty_cache()
            print(n, p, name, row[name].get("it_per_s", "refused"), flush=True)
        # what the CSR route spends per Jacobian besides the products
        try:
            t_conv = event_ms(lambda: J.to_sparse_csr(), 3)
            A = J.to_sparse_csr()
            if A._nnz() < (1 << 31) - 1:
                prob = DeviceCallableProblem(lambda x: J @ x - y, ways["csr"], x0, ())
                x = prob.new_sol()
                prob.upload_x(x0, x)
                prob.evaluate(x)
                prob.jacobian(x)
                rt.sync()
                t0 = time.perf_counter()
                for _ in range(5):
                    prob.pattern.matches(n, p, A.crow_indices(), A.col_indices(), prob._flag)
                t_cmp = (time.perf_counter() - t0) / 5 * 1e3
                t_gather = event_ms(lambda: DeviceCsrJacobian(rt, prob.pattern, A.values(), False), 3)
                op = DeviceCsrJacobian(rt, prob.pattern, A.values(), False)
                r = torch.randn(n, dtype=torch.float64, device=rt.device)
                w = torch.empty(prob.p_glob, dtype=torch.float64, device=rt.device)
                t_csr_t = event_ms(lambda: op.neg_rmatvec(r, w), 5)
                row["csr_route_ms"] = dict(to_sparse_csr=t_conv, pattern_compare_incl_readback=t_cmp,
                                           gather_values_t=t_gather, spmm_csr_transpose_product=t_csr_t)
                del prob, op, x, r, w
            else:
                row["csr_route_ms"] = dict(to_sparse_csr=t_conv, note="nnz >= 2^31: the int32 CSR kernels refuse it")
            del A
        except torch.OutOfMemoryError as e:
            row["csr_route_ms"] = dict(error=str(e).splitlines()[0])
        torch.cuda.empty_cache()
        row["kernels"] = kernels(rt, J, n, p, 5)
        result["shapes"][f"{n}x{p}"] = row
        del J, y, x0
        if a.out:  # what is measured so far survives a later failure
            with open(a.out, "w") as f:
                json.dump(result, f, indent=1)
    result["card_after"] = card()
    js = json.dumps(result, indent=1)
    print(js)
    if a.out:
        with open(a.out, "w") as f:
            f.write(js + "\n")


if __name__ == "__main__":
    main()
