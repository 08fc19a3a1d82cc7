"""Krylov bases past 255 columns on one GPU (gauss_newton_krylow(max_basis_columns=...)):

  1. Bratu 1024^2 without a restart for 400 iterations (--iters): iterations per second (profiler off), then ms per
     class (J V_k, least squares, combine, dots, update) against k from a profiled run of its own.  A run of 1000
     iterations spends minutes in the least squares alone (0.66 s per call at k = 1000, section 3).
  2. The wide streaming kernels alone at n = 2^20, k = 256 .. 4095: time and share of the HBM bound (8 n k bytes).
  3. gnk_basis_ls_wide against torch.linalg.lstsq on the same 2^20 x k panels.

    python tools/bench_wide_basis.py --out profiles/r09_wide_basis_1gpu.json
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_BPS = 7.7e12  # HGX B200 data sheet, one GPU


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = f"nvidia-smi unavailable: {e}"
    return q


def bucket(k):
    for lo, hi in ((1, 255), (256, 511), (512, 767), (768, 1023)):
        if lo <= k <= hi:
            return f"{lo}-{hi}"
    return ">=1024"


def solve_bench(g, iters, reps):
    from oracle import gnk_oracle as orc
    G = 1025
    o = orc.BratuOracle(G, 5, 10)
    y, u0 = o.operator(o.u_true), o.start_vector(seed=42)
    pb = g.BratuPdeProblem(G, 5, 10)
    rt = g.get_runtime()
    kw = dict(max_iter=iters, max_basis_columns=iters, callback=lambda **k: None, x_on_device=True)
    times, nit = [], None
    for _ in range(reps):
        rt.sync()
        t0 = time.perf_counter()
        out = g.gauss_newton_krylow(pb.make_res(y), u0, pb.make_jac(), **kw)
        rt.sync()
        times.append(time.perf_counter() - t0)
        nit = out.nit
    n = pb.p_glob if hasattr(pb, "p_glob") else (G - 1) ** 2
    rt.begin_profile()
    g.gauss_newton_krylow(pb.make_res(y), u0, pb.make_jac(), **kw)
    rt.sync()
    recs = rt.prof
    per = {}
    for name, lst in recs.items():
        for e0, e1, nb in lst:
            ms = e0.elapsed_time(e1)
            # the marks carry their algorithmic bytes: combine / dots / ls 8n(k+1), update 8n(k+2), spmm 8n(2k+1)
            kk = {"combine": nb / (8 * n) - 1, "cgs_dots": nb / (8 * n) - 1, "ls_wide": nb / (8 * n) - 1,
                  "tsqr": nb / (8 * n) - 1, "cgs_update": nb / (8 * n) - 2, "spmm": (nb / (8 * n) - 1) / 2}.get(name)
            key = bucket(int(round(kk))) if kk is not None else "all"
            d = per.setdefault(name, {}).setdefault(key, dict(calls=0, ms=0.0, bytes=0.0))
            d["calls"] += 1
            d["ms"] += ms
            d["bytes"] += nb
    rt.prof = None
    for name, byk in per.items():
        for d in byk.values():
            d["ms_per_call"] = d["ms"] / d["calls"]
            d["hbm_share"] = d["bytes"] / (d["ms"] * 1e-3) / HBM_BPS if d["ms"] > 0 else None
    return dict(grid=f"{G - 1}^2", unknowns=n, max_iter=iters, nit=nit, seconds=times,
                it_per_s=[nit / t for t in times], profile_ms_by_class_and_k=per)


def stream_bench(g, ks, n, reps):
    import torch
    from gauss_newton_via_generalized_krylov_subspaces_b200.device import make_layout, ptr
    from gauss_newton_via_generalized_krylov_subspaces_b200.partition import flat_layout_fields
    rt, lib = g.get_runtime(), g.get_runtime().lib
    lay = make_layout(dict(flat_layout_fields(n), ld=n))
    V = torch.randn(max(ks) * n, dtype=torch.float64, device=rt.device)  # > 126 MB of L2 at every k
    out = []
    for k in ks:
        c, d = torch.randn(k + 1, dtype=torch.float64, device=rt.device), torch.randn(k, dtype=torch.float64,
                                                                                        device=rt.device)
        x, w, h, st, cout = (rt.zeros(n), torch.randn(n, dtype=torch.float64, device=rt.device), rt.zeros(k),
                             rt.zeros(2), rt.zeros(k + 1))
        calls = {
            "combine": lambda: lib.gnk_combine_step(rt.ctx, C.byref(lay), ptr(V), k, ptr(c), ptr(d), 0.5, ptr(x),
                                                    ptr(cout), None, rt.stream),
            "cgs_dots": lambda: lib.gnk_cgs_dots(rt.ctx, C.byref(lay), ptr(V), k, ptr(w), ptr(h), rt.stream),
            "cgs_update": lambda: lib.gnk_cgs_update(rt.ctx, C.byref(lay), ptr(V), k, ptr(h), ptr(w), ptr(st),
                                                     rt.stream),
        }
        row = dict(k=k, n=n)
        for name, fn in calls.items():
            assert fn() == 0
            rt.sync()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            rt.sync()
            ms = e0.elapsed_time(e1) / reps
            nbytes = 8.0 * n * k
            row[name] = dict(ms=ms, hbm_share=nbytes / (ms * 1e-3) / HBM_BPS)
        out.append(row)
        print(json.dumps(row), flush=True)
    return out


def ls_bench(g, ks, n, reps):
    import torch
    from gauss_newton_via_generalized_krylov_subspaces_b200.device import ptr
    rt = g.get_runtime()
    out = []
    for k in ks:
        A = torch.randn(n, k, dtype=torch.float64, device=rt.device)
        y = torch.randn(n, dtype=torch.float64, device=rt.device)
        P0 = torch.cat([A, y[:, None]], dim=1).T.contiguous().reshape(-1)
        P = torch.empty_like(P0)
        res = rt.zeros(2 * k + 4)

        def ours():
            P.copy_(P0)
            assert rt.lib.gnk_basis_ls_wide(rt.ctx, ptr(P), n, n, k, -1.0, ptr(res), rt.stream) == 0

        def theirs():
            return torch.linalg.lstsq(-A, y[:, None]).solution

        row = dict(k=k, n=n)
        for name, fn in (("gnk_basis_ls_wide", ours), ("torch.linalg.lstsq", theirs)):
            fn()
            rt.sync()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            rt.sync()
            row[name + "_ms"] = e0.elapsed_time(e1) / reps
        ours()
        d = rt.read(res, k).copy()
        ref = theirs().reshape(-1).cpu().numpy()
        row["rel_diff_vs_torch"] = float(np.max(np.abs(d - ref)) / np.max(np.abs(ref)))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            P.copy_(P0)
        e1.record()
        rt.sync()
        row["panel_copy_ms"] = e0.elapsed_time(e1) / reps
        out.append(row)
        print(json.dumps(row), flush=True)
        del A, P0, P
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--iters", default="400")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--stream-ks", default="256,512,1024,2048,4095")
    ap.add_argument("--ls-ks", default="256,512,1000")
    a = ap.parse_args()
    import gauss_newton_via_generalized_krylov_subspaces_b200 as g
    g.get_runtime()
    result = dict(gpu=gpu_info(), note="HBM share against the 7.7 TB/s data-sheet figure; L2 is exceeded at every size")
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)

    def save():  # after every section: a run cut short keeps what it measured
        with open(a.out, "w") as f:
            json.dump(result, f, indent=1)

    result["streaming_kernels"] = stream_bench(g, [int(k) for k in a.stream_ks.split(",")], 1 << 20, 5)
    save()
    result["least_squares"] = ls_bench(g, [int(k) for k in a.ls_ks.split(",")], 1 << 20, 3)
    save()
    result["bratu_1024_no_restart"] = []
    for it in [int(i) for i in a.iters.split(",")]:
        r = solve_bench(g, it, a.reps)
        print(json.dumps({kk: v for kk, v in r.items() if kk != "profile_ms_by_class_and_k"}), flush=True)
        result["bratu_1024_no_restart"].append(r)
        save()
    result["gpu_after"] = gpu_info()
    save()


if __name__ == "__main__":
    main()
