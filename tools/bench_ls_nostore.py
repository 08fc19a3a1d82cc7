#!/usr/bin/env python
"""The fused least squares of one outer iteration (gnk_stencil_gram_ls) with and without the J V_k store.

    python tools/bench_ls_nostore.py [--m 4096] [--ks 7-30] [--reps 15] [--out profiles/ls_nostore.json]

Storing: the sweep writes J V_k and the refinement pass reads it back (cholqr_refine_kernel).  Store-free (d_JV NULL):
the refinement pass streams V_k again and re-applies the stencil (stencil_refine_kernel).  For every k: CUDA events
around the whole call chain (sweep, first factor, refinement, second factor), the two modes alternating, median of
--reps each; the basis (k x 134 MB at m = 4096) is far larger than L2.  Checks that both modes take the refinement
form, that the diagonal of R (from the first factor) is bit-identical and how far d moves.  The summary weights every
k of the range equally, as a restarted solve visits them.  The card's name, power limit and SM clocks are read
(nvidia-smi --query-gpu, read only) in the same run and written beside the numbers.
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
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout
        name, power, clock_max, clock_now = (s.strip() for s in q.strip().splitlines()[0].split(","))
        return dict(name=name, power_limit=power, max_sm_clock=clock_max, sm_clock_after_timing=clock_now)
    except Exception as e:  # the numbers stay valid, only their label is missing
        return dict(error=str(e))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--m", type=int, default=4096)
    ap.add_argument("--ks", default="7-30")
    ap.add_argument("--reps", type=int, default=15)
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

    rt = g.get_runtime()
    lib = rt.lib
    pb = g.BratuPdeProblem(a.m + 1, 5, 10)
    d = pb.dev
    n, ld, off = d.fields["n_own"], d.ld, d.fields["off"]
    kmax = max(ks)
    gen = torch.Generator(device=rt.device).manual_seed(0)
    V = torch.randn(kmax * ld, dtype=torch.float64, device=rt.device, generator=gen) / np.sqrt(n)
    Vm = V.view(kmax, ld)
    Vm[:, :off] = 0.0          # Dirichlet halo rows, as the solver stores the basis
    Vm[:, off + n:] = 0.0
    u, r = d.new_col(), d.new_col()
    u[off:off + n] = 0.3 * torch.randn(n, dtype=torch.float64, device=rt.device, generator=gen)
    r[off:off + n] = torch.randn(n, dtype=torch.float64, device=rt.device, generator=gen)
    E = d.new_col()
    d.residual_into(u, d.zero_col(), d.new_col(), E, d.scal_tmp, depth=0)
    ldjv = (n + 15) // 16 * 16
    JV = rt.zeros(kmax * ldjv)
    lay, prm = C.byref(d.lay), C.byref(d.prm)
    outs = {"store": rt.zeros(256), "free": rt.zeros(256)}

    def call(mode, k):
        jv = ptr(JV) if mode == "store" else None
        _lib.check(lib.gnk_stencil_gram_ls(rt.ctx, lay, prm, ptr(E), ptr(V), ld, kmax, k, ptr(r), -1.0, jv, ldjv, -1.0,
                                           ptr(outs[mode]), rt.stream), "gnk_stencil_gram_ls")

    def once(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1)

    rows = []
    for k in ks:
        for mode in ("store", "free"):
            for _ in range(2):
                call(mode, k)
        torch.cuda.synchronize()
        t = {"store": [], "free": []}
        for _ in range(a.reps):
            for mode in ("store", "free"):
                t[mode].append(once(lambda: call(mode, k)))
        vs, vf = rt.read(outs["store"], 2 * k + 4), rt.read(outs["free"], 2 * k + 4)
        ms_s, ms_f = float(np.median(t["store"])), float(np.median(t["free"]))
        rows.append(dict(k=k, ms_store=round(ms_s, 4), ms_free=round(ms_f, 4), speedup=round(ms_s / ms_f, 3),
                         spread_store=round(float(np.max(t["store"]) - np.min(t["store"])), 4),
                         spread_free=round(float(np.max(t["free"]) - np.min(t["free"])), 4),
                         refine_form=bool(vs[k + 2] == 0 and vf[k + 2] == 0),
                         diag_r_bit_identical=bool(np.array_equal(vs[k + 4:2 * k + 4], vf[k + 4:2 * k + 4])),
                         d_max_rel_diff=float(np.max(np.abs(vs[:k] - vf[:k])) / np.max(np.abs(vs[:k])))))
        print(json.dumps(rows[-1]), flush=True)
    info = gpu_info()
    tot_s, tot_f = sum(x["ms_store"] for x in rows), sum(x["ms_free"] for x in rows)
    res = dict(gpu=info, m=a.m, n=n, reps=a.reps, ks=ks, rows=rows, sum_ms_store=round(tot_s, 3),
               sum_ms_free=round(tot_f, 3), weighted_gain=round(1.0 - tot_f / tot_s, 4))
    print(json.dumps({key: v for key, v in res.items() if key != "rows"}))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
