"""Device time of gnk_tsqr_ls on wide panels (105..256 columns): the blocked Householder TSQR (tsqr.cu:
wide_tsqr_kernel) at 2^20 and 2^24 rows, the single-CTA QR (dense_qr_ls_kernel) just below its 2^22-double limit, and
end-to-end GNK runs without a restart that reach the wide panels.  Prints one JSON object; card name and power limit
are read in the same run.

    python tools/bench_wide_householder.py [--skip-e2e] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import gauss_newton_via_generalized_krylov_subspaces_b200 as g  # noqa: E402
from gauss_newton_via_generalized_krylov_subspaces_b200.gauss_newton_krylow import tsqr_solve  # noqa: E402

DMMA_PEAK = 37.2e12   # profiles/r01_fp64_peak.json
HBM_COPY = 6549e9     # bytes/s


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def time_ls(rt, n, c, reps):
    k = c - 1
    A = torch.randn(k * n, dtype=torch.float64, device=rt.device)
    y = torch.randn(n, dtype=torch.float64, device=rt.device)
    out = rt.zeros(2 * 256 + 8)
    tsqr_solve(rt, A, n, n, k, y, -1.0, out)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        tsqr_solve(rt, A, n, n, k, y, -1.0, out)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    flops = 2.0 * n * c * c - 2.0 * c ** 3 / 3.0
    nbytes = 8.0 * n * c
    v = rt.read(out, 2 * k + 4)
    del A, y
    return {"n": n, "c": c, "ms": round(ms, 3), "tflops": round(flops / ms / 1e9, 2),
            "frac_dmma_peak": round(flops / (ms * 1e-3) / DMMA_PEAK, 3),
            "frac_hbm_copy": round(nbytes / (ms * 1e-3) / HBM_COPY, 4), "rank_count": float(v[k + 2])}


def e2e(G, max_iter):
    pb = g.BratuPdeProblem(G, 5, 10)
    y = pb.pde_operator(pb.u_true)
    u0 = pb.u_true + 0.1 * np.random.RandomState(42).normal(size=pb.n)
    res, jac = pb.make_res(y), pb.make_jac()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = g.gauss_newton_krylow(res, u0, jac, krylow_restart=None, max_iter=max_iter, callback=lambda **kw: None)
    torch.cuda.synchronize()
    s = time.perf_counter() - t0
    return {"G": G, "max_iter": max_iter, "nit": int(out.nit), "seconds": round(s, 2),
            "iterations_per_s": round(out.nit / s, 2)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    rt = g.get_runtime()
    result = {"card": card(), "wide_tsqr": [], "single_cta": [], "e2e": []}
    for n, reps in ((1 << 20, 5), (1 << 24, 2)):
        for c in (105, 160, 256):
            result["wide_tsqr"].append(time_ls(rt, n, c, reps))
            print(json.dumps(result["wide_tsqr"][-1]), flush=True)
    for c in (105, 160, 256):  # the single-CTA kernel at its largest panel: n * c <= 2^22
        result["single_cta"].append(time_ls(rt, (1 << 22) // c, c, 3))
        print(json.dumps(result["single_cta"][-1]), flush=True)
    if not a.skip_e2e:
        for G, it in ((1025, 200), (4097, 150)):
            result["e2e"].append(e2e(G, it))
            print(json.dumps(result["e2e"][-1]), flush=True)
    print(json.dumps(result))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
