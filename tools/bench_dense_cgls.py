"""cg_least_squares with a dense CUDA A: the dense operator (gnk_linop kind 2, A read in place) against the same matrix
handed over as A.to_sparse_csr() (the route a dense A took before: CSR copy, device transpose pattern, A^T gather,
gnk_spmm_csr).  Shapes 2^20 x 256, 2^20 x 1024, 2^22 x 512 (2^31 entries: the CSR route refuses it) and 8192 x 8192,
every one far above the 126 MB L2.  A is Gaussian (seeded), y Gaussian, preconditioner on.

Per shape and route: the set-up (operator construction: for CSR the conversion, pattern and gather; for dense none),
ms per CG iteration ((t(rtol_b) - t(rtol_a)) / (count_b - count_a) over two full solves, wall clock around work that
ends in a device synchronise, so set-up, A^T y and the Jacobi diagonal cancel), and the memory a solve adds (torch's
peak over the call, the CSR conversion included, plus the library's own scratch growth).  Then the two kernels of a
dense iteration, timed inside the CG loop by torch.profiler in a run of its own: dense_matvec_kernel (A p) and
dense_rmatvec_kernel (A^T t), each as a share of the HBM bound 8 n p bytes / 7.7 TB/s; and the same kernels alone with
CUDA events, next to the 2-column dense_matmat_kernel pass (k = 2) that k = 1 took before.  Card and power limit are
read in the same run.

    python tools/bench_dense_cgls.py [--out FILE]
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
from gauss_newton_via_generalized_krylov_subspaces_b200.device import (DenseDeviceJacobian,  # noqa: E402
                                                                       DeviceCsrJacobian, ptr)

HBM_TBS = 7.7  # HGX B200 data sheet, per GPU
SHAPES = [(1 << 20, 256), (1 << 20, 1024), (1 << 22, 512), (8192, 8192)]
RTOLS = {(8192, 8192): (1e-1, 1e-2)}  # a square Gaussian A converges slowly; the tall ones in a few iterations
RTOLS_TALL = (1e-2, 1e-10)


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


def solve(rt, make, y, rtol):
    """one cg_least_squares call on make() (for the CSR route the conversion is part of the call) -> (count, seconds,
    torch peak growth in bytes)"""
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats(rt.device)
    before = torch.cuda.memory_allocated(rt.device)
    t0 = time.perf_counter()
    x, it = g.cg_least_squares(make(), y, cg_rtol=rtol)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    grown = torch.cuda.max_memory_allocated(rt.device) - before
    del x
    return it, dt, grown


def route(rt, A, y, rtols, csr):
    """set-up time, ms per CG iteration and memory of one route"""
    make = A.to_sparse_csr if csr else (lambda: A)
    torch.cuda.empty_cache()
    free0 = torch.cuda.mem_get_info(rt.device)[0]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    op = DeviceCsrJacobian.from_tensor(rt, make(), "A") if csr else DenseDeviceJacobian(rt, A)
    torch.cuda.synchronize()
    setup_ms = (time.perf_counter() - t0) * 1e3
    del op
    solve(rt, make, y, rtols[0])  # warm-up: modules, scratch
    counts, secs, peak = [], [], 0
    for rtol in rtols:
        it, dt, grown = solve(rt, make, y, rtol)
        counts.append(it)
        secs.append(dt)
        peak = max(peak, grown)
    torch.cuda.empty_cache()
    lib_scratch = max(0, free0 - torch.cuda.mem_get_info(rt.device)[0])
    per_it = (secs[1] - secs[0]) / (counts[1] - counts[0]) * 1e3 if counts[1] > counts[0] else None
    return dict(setup_ms=setup_ms, cg_rtols=list(rtols), cg_iterations=counts, solve_seconds=secs,
                ms_per_cg_iteration=per_it, torch_peak_growth_bytes=peak, library_scratch_growth_bytes=lib_scratch)


def in_loop_kernels(rt, A, y, rtol, hbm_ms):
    """torch.profiler over one dense solve: mean device time of the two product kernels inside the CG loop"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        g.cg_least_squares(A, y, cg_rtol=rtol)
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        for name in ("dense_matvec_kernel", "dense_rmatvec_kernel", "dense_col_sumsq_kernel"):
            if name in ev.key:
                us = getattr(ev, "device_time_total", None)
                if us is None:
                    us = ev.cuda_time_total
                d = out.setdefault(name, dict(launches=0, us_total=0.0))
                d["launches"] += ev.count
                d["us_total"] += us
    for d in out.values():
        d["ms_mean"] = d["us_total"] / d["launches"] / 1e3
        d["hbm_share"] = hbm_ms / d["ms_mean"]
    return out


def alone_kernels(rt, A, n, p, hbm_ms):
    """the same kernels alone (CUDA events over 5 launches, A resident in HBM), and the k = 2 pass of
    dense_matmat_kernel that served k = 1 before the one-column kernel"""
    rs, cs = A.stride()
    out = {}
    v = torch.randn(2 * p, dtype=torch.float64, device=rt.device)
    t = torch.empty(2 * n, dtype=torch.float64, device=rt.device)
    for k in (1, 2):
        ms = event_ms(lambda: rt.lib.gnk_dense_matmat(rt.ctx, n, p, ptr(A), rs, cs, ptr(v), p, 0, k, 1.0, ptr(t), n, 0,
                                                      rt.stream), 5)
        out[f"matmat_k{k}"] = dict(ms=ms, hbm_share=hbm_ms / ms)
    w = torch.empty(p, dtype=torch.float64, device=rt.device)
    ms = event_ms(lambda: rt.lib.gnk_dense_rmatvec(rt.ctx, n, p, ptr(A), rs, cs, ptr(t), 1.0, ptr(w), rt.stream), 5)
    out["rmatvec"] = dict(ms=ms, hbm_share=hbm_ms / ms)
    ms = event_ms(lambda: rt.lib.gnk_dense_col_sumsq(rt.ctx, n, p, ptr(A), rs, cs, ptr(w), rt.stream), 3)
    out["col_sumsq"] = dict(ms=ms, hbm_share=hbm_ms / ms)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    rt = g.get_runtime()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    result = dict(card_name_power_limit_sm_clock_max_sm_clock=card(), peaks=dict(hbm_tbs=HBM_TBS),
                  hbm_bound="8 n p bytes / 7.7 TB/s", shapes={})
    for n, p in SHAPES:
        torch.cuda.empty_cache()
        gen = torch.Generator(device=rt.device).manual_seed(1)
        A = torch.empty(n, p, dtype=torch.float64, device=rt.device)
        for r0 in range(0, n, 1 << 17):
            A[r0:r0 + (1 << 17)].normal_(generator=gen)
        y = torch.randn(n, dtype=torch.float64, device=rt.device, generator=gen)
        hbm_ms = 8.0 * n * p / (HBM_TBS * 1e12) * 1e3
        rtols = RTOLS.get((n, p), RTOLS_TALL)
        row = dict(entries=n * p, gib=8.0 * n * p / 2 ** 30, hbm_bound_ms=hbm_ms)
        for name in ("dense", "csr"):
            try:
                row[name] = route(rt, A, y, rtols, name == "csr")
            except (_lib.GnkError, torch.OutOfMemoryError) as e:
                row[name] = dict(refused=str(e).splitlines()[0])
            torch.cuda.empty_cache()
            print(n, p, name, row[name], flush=True)
        if "cg_iterations" in row["csr"]:
            row["same_counts"] = row["csr"]["cg_iterations"] == row["dense"]["cg_iterations"]
        row["in_cg_loop"] = in_loop_kernels(rt, A, y, rtols[1], hbm_ms)
        row["alone"] = alone_kernels(rt, A, n, p, hbm_ms)
        result["shapes"][f"{n}x{p}"] = row
        del A, y
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
