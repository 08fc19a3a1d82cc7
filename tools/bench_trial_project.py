#!/usr/bin/env python
"""The fused trial pass (gnk_bratu_trial_project) against the calls it replaces, at the north-star size.

    python tools/bench_trial_project.py [--m 4096] [--ks 1-32] [--out results/trial_project.json]

For every k: CUDA-event time of the fused pass and of combine + -J^T r + dots (gnk_combine_step,
gnk_stencil_apply transposed on the e^x the residual kernel stored, gnk_cgs_dots -- the residual itself runs in both
sequences and is not timed), algorithmic GB/s over the measured HBM peak (MEASURED_PEAKS.json), and whether x, w, h
and the coordinate outputs are bit-identical.  The basis (k x 134 MB) is far larger than L2.  The card's name, power
limit and maximum SM clock are read (nvidia-smi --query-gpu, read only) in the same run and written beside the numbers.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        name, power, clock = (s.strip() for s in q[0].split(","))
        return dict(name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:  # the numbers stay valid, only their label is missing
        return dict(error=str(e))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--m", type=int, default=4096)
    ap.add_argument("--ks", default="1-32")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if "-" in a.ks:
        lo, hi = (int(v) for v in a.ks.split("-"))
        ks = list(range(lo, hi + 1))
    else:
        ks = [int(v) for v in a.ks.split(",")]
    import torch
    import gauss_newton_via_generalized_krylov_subspaces_b200 as g
    from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib
    from gauss_newton_via_generalized_krylov_subspaces_b200.device import ptr

    info = gpu_info()
    rt = g.get_runtime()
    lib = rt.lib
    try:
        peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        peak = 6650.0
    pb = g.BratuPdeProblem(a.m + 1, 5, 10)
    d = pb.dev
    n, ld, off = d.fields["n_own"], d.ld, d.fields["off"]
    kmax = max(ks)
    gen = torch.Generator(device=rt.device).manual_seed(0)
    V = torch.randn(kmax * ld, dtype=torch.float64, device=rt.device, generator=gen) / np.sqrt(kmax)
    u, y, F, E = (d.new_col() for _ in range(4))
    u[off:off + n] = torch.randn(n, dtype=torch.float64, device=rt.device, generator=gen) * 1e-2
    y[off:off + n] = torch.randn(n, dtype=torch.float64, device=rt.device, generator=gen)
    st = rt.zeros(2)
    d.residual_into(u, y, F, E, st, depth=1)   # F: a residual with its depth-1 halo rows, as in the solver
    cc = torch.randn(256, dtype=torch.float64, device=rt.device, generator=gen)
    dd = torch.randn(256, dtype=torch.float64, device=rt.device, generator=gen) * 1e-2
    lay, prm = C.byref(d.lay), C.byref(d.prm)
    bufs = {tag: dict(x=d.new_col(), w=d.new_col(), h=rt.zeros(256), c_out=rt.zeros(256), cprev2=rt.zeros(1))
            for tag in ("sep", "fused")}
    expu = d.new_col()

    def separate(k):
        b = bufs["sep"]
        _lib.check(lib.gnk_combine_step(rt.ctx, lay, ptr(V), k, ptr(cc), ptr(dd), 1.0, ptr(b["x"]), ptr(b["c_out"]),
                                        ptr(b["cprev2"]), rt.stream))
        _lib.check(lib.gnk_stencil_apply(rt.ctx, lay, prm, ptr(expu), ptr(F), ld, 1, 1.0, 1, ptr(b["w"]), ld, off,
                                         rt.stream))
        _lib.check(lib.gnk_cgs_dots(rt.ctx, lay, ptr(V), k, ptr(b["w"]), ptr(b["h"]), rt.stream))

    def fused(k):
        b = bufs["fused"]
        _lib.check(lib.gnk_bratu_trial_project(rt.ctx, lay, prm, ptr(V), k, ptr(cc), ptr(dd), 1.0, ptr(b["x"]),
                                               ptr(b["c_out"]), ptr(b["cprev2"]), ptr(F), ptr(b["w"]), ptr(b["h"]),
                                               rt.stream))

    def timeit(fn):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        e = [torch.cuda.Event(enable_timing=True) for _ in range(a.reps + 1)]
        e[0].record()
        for i in range(a.reps):
            fn()
            e[i + 1].record()
        torch.cuda.synchronize()
        t = sorted(e[i].elapsed_time(e[i + 1]) for i in range(a.reps))
        return t[len(t) // 2]

    rows = []
    for k in ks:
        # the e^x of the separate sequence comes from the residual kernel at the separate x, as in the solver
        b = bufs["sep"]
        _lib.check(lib.gnk_combine_step(rt.ctx, lay, ptr(V), k, ptr(cc), ptr(dd), 1.0, ptr(b["x"]), ptr(b["c_out"]),
                                        ptr(b["cprev2"]), rt.stream))
        d.residual_into(b["x"], y, d.scratch_col(), expu, st, depth=1)
        ms_sep = timeit(lambda: separate(k))
        ms_fused = timeit(lambda: fused(k))
        same = all(torch.equal(bufs["sep"][key], bufs["fused"][key]) for key in ("x", "w", "h", "c_out", "cprev2"))
        b_sep = 8.0 * n * (k + 1) + 24.0 * n + 8.0 * n * (k + 1)
        b_fused = 8.0 * n * (k + 3)
        g_sep, g_fused = b_sep / ms_sep / 1e6, b_fused / ms_fused / 1e6
        rows.append(dict(k=k, ms_separate=round(ms_sep, 4), ms_fused=round(ms_fused, 4),
                         speedup=round(ms_sep / ms_fused, 3), gbs_separate=round(g_sep, 1),
                         gbs_fused=round(g_fused, 1), frac_separate=round(g_sep / peak, 3),
                         frac_fused=round(g_fused / peak, 3), bit_identical=bool(same)))
        print(f"k={k:2d}  separate {ms_sep:8.4f} ms ({g_sep / peak:5.3f})  fused {ms_fused:8.4f} ms "
              f"({g_fused / peak:5.3f})  x{ms_sep / ms_fused:5.2f}  bit-identical={same}", flush=True)
    res = dict(gpu=info, m=a.m, n=n, peak_gbs=peak, reps=a.reps, statistic="median of reps, CUDA events",
               bytes_separate="8n(k+1) combine + 24n -J^T r + 8n(k+1) dots", bytes_fused="8n(k+3)",
               total_ms_separate_k1_30=round(sum(r["ms_separate"] for r in rows if r["k"] <= 30), 3),
               total_ms_fused_k1_30=round(sum(r["ms_fused"] for r in rows if r["k"] <= 30), 3), rows=rows)
    print(json.dumps({k_: v for k_, v in res.items() if k_ != "rows"}))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        json.dump(res, open(a.out, "w"), indent=1)
    if not all(r["bit_identical"] for r in rows):
        sys.exit(1)


if __name__ == "__main__":
    main()
