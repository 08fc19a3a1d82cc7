"""Device time of gnk_dense_qr_ls (dense_qr.cu: blocked Householder QR of 256..4095 columns) on random panels resident
in HBM, its split into panel factorisation and trailing update (a separate torch.profiler pass), torch.linalg.lstsq
(cuSOLVER, driver gels) on the same panel as a yardstick, and one gauss_newton run on a dense fit with 1000 parameters
against the oracle on the host.  Prints one JSON object; card name, power limit and max SM clock are read in the same
run.

    python tools/bench_dense_ls.py [--reps R] [--skip-e2e] [--out FILE]
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
from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib  # noqa: E402

DMMA_PEAK = 37.2e12   # profiles/r01_fp64_peak.json
SHAPES = ((1 << 17, 256), (1 << 17, 1024), (1 << 17, 2048), (1 << 15, 4095), (1 << 20, 512))


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def call(rt, work, n, p, out):
    _lib.check(rt.lib.gnk_dense_qr_ls(rt.ctx, work.data_ptr(), n, n, p, -1.0, out.data_ptr(), rt.stream),
               "gnk_dense_qr_ls")


def time_dense(rt, n, p, reps):
    c = p + 1
    gen = torch.Generator(device=rt.device).manual_seed(n + p)
    panel = torch.randn(c * n, dtype=torch.float64, device=rt.device, generator=gen)
    work = torch.empty_like(panel)
    out = rt.zeros(2 * p + 8)
    work.copy_(panel)
    call(rt, work, n, p, out)  # warm-up (workspace, module load)
    times = []
    for _ in range(reps):
        work.copy_(panel)  # the call works in place: restore the panel outside the events
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        call(rt, work, n, p, out)
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    ms = float(np.median(times))
    v = out[:2 * p + 4].cpu().numpy()

    # where the time goes: one profiled call, kernel time by kernel
    work.copy_(panel)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        call(rt, work, n, p, out)
        torch.cuda.synchronize()
    split = {}
    for ev in prof.key_averages():
        for key in ("dqr_panel_kernel", "dqr_vtc_kernel", "dqr_tw_kernel", "dqr_update_kernel", "dqr_solve_kernel",
                    "dqr_scale_kernel"):
            if key in ev.key:
                split[key] = split.get(key, 0.0) + ev.device_time_total / 1e3  # us -> ms
    split = {k: round(t, 3) for k, t in split.items()}

    # yardstick: cuSOLVER least squares (QR, driver gels) on the same panel
    A = panel[:p * n].view(p, n).T
    y = panel[p * n:].view(n, 1)
    torch.linalg.lstsq(-A, y, driver="gels")
    torch.cuda.synchronize()
    lt = []
    for _ in range(max(2, reps // 2)):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        sol = torch.linalg.lstsq(-A, y, driver="gels").solution
        e1.record()
        torch.cuda.synchronize()
        lt.append(e0.elapsed_time(e1))
    lms = float(np.median(lt))
    agree = float(torch.linalg.norm(sol[:, 0] - torch.from_numpy(v[:p]).to(rt.device)) / torch.linalg.norm(sol))
    flops = 2.0 * n * c * c - 2.0 * c ** 3 / 3.0
    del panel, work, A, y, sol
    torch.cuda.empty_cache()
    return {"n": n, "p": p, "ms": round(ms, 3), "ms_all": [round(t, 3) for t in times],
            "tflops": round(flops / ms / 1e9, 2), "frac_dmma_peak": round(flops / (ms * 1e-3) / DMMA_PEAK, 3),
            "kernel_ms": split, "rank_count": float(v[p + 2]),
            "torch_lstsq_gels_ms": round(lms, 3), "speedup_vs_gels": round(lms / ms, 2),
            "rel_diff_vs_gels": agree}


def e2e(n, p, max_iter):
    from oracle import gnk_oracle as orc
    rs = np.random.RandomState(1)
    A = rs.normal(size=(n, p)) / np.sqrt(n)
    B = rs.normal(size=(n, p)) / np.sqrt(p)
    xt = rs.normal(size=p)
    y = A @ xt + 0.1 * np.sin(B @ xt) + 1e-3 * rs.normal(size=n)
    res = lambda x: A @ x + 0.1 * np.sin(B @ x) - y  # noqa: E731
    jac = lambda x: A + (0.1 * np.cos(B @ x))[:, None] * B  # noqa: E731
    x0 = xt + 0.5 * rs.normal(size=p)
    t0 = time.perf_counter()
    out = g.gauss_newton(res, x0.copy(), jac, max_iter=max_iter, callback=lambda **kw: None)
    torch.cuda.synchronize()
    s = time.perf_counter() - t0
    t0 = time.perf_counter()
    ref = orc.gn(res, x0.copy(), jac, max_iter=max_iter)
    so = time.perf_counter() - t0
    # the same run with device callables: x, F and J stay on the GPU
    At, Bt, yt = (torch.from_numpy(a).cuda() for a in (A, B, y))
    dres = lambda x: At @ x + 0.1 * torch.sin(Bt @ x) - yt  # noqa: E731
    djac = lambda x: At + (0.1 * torch.cos(Bt @ x))[:, None] * Bt  # noqa: E731
    g.gauss_newton(dres, torch.from_numpy(x0.copy()).cuda(), djac, max_iter=2, callback=lambda **kw: None)  # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    outd = g.gauss_newton(dres, torch.from_numpy(x0.copy()).cuda(), djac, max_iter=max_iter,
                          callback=lambda **kw: None)
    torch.cuda.synchronize()
    sd = time.perf_counter() - t0
    return {"n": n, "p": p, "max_iter": max_iter, "nit": int(out.nit), "oracle_nit": int(ref["nit"]),
            "s_per_iter_host_callables": round(s / out.nit, 4), "s_per_iter_device_callables": round(sd / outd.nit, 4),
            "s_per_iter_oracle_host": round(so / ref["nit"], 4),
            "rel_diff_vs_oracle": float(np.linalg.norm(out.x - ref["x"]) / np.linalg.norm(ref["x"]))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    rt = g.get_runtime()
    result = {"card": card(), "card_fields": "name, power.limit, clocks.max.sm",
              "flops": "2 n c^2 - 2 c^3 / 3, c = p + 1", "dmma_peak_tflops": DMMA_PEAK / 1e12, "dense_qr": [],
              "e2e": []}
    for n, p in SHAPES:
        result["dense_qr"].append(time_dense(rt, n, p, a.reps))
        print(json.dumps(result["dense_qr"][-1]), flush=True)
    if not a.skip_e2e:
        result["e2e"].append(e2e(50000, 1000, 5))
        print(json.dumps(result["e2e"][-1]), flush=True)
    print(json.dumps(result))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
