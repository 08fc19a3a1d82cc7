#!/usr/bin/env python
"""bench.py -- GN-Krylov outer iterations/s (and time-to-tolerance) on the Bratu problem (BASELINE.json metric).

A "step" is one complete GNK solve of a named workload (`--workload`, default = the north-star one):

  bratu_4096_k30         Bratu grid_nodes=4097 (n = 4096^2 = 16.7M unknowns), ALPHA=5, LAMBDA=10, u0 = u_true + 0.1 N(0,1)
                         (numpy legacy seed 42, drawn on the host), Krylov dimension <= 30 realised as
                         krylow_restart=None, max_iter=31 -> 30 outer iterations, k = 1..30 (SURVEY 8c': every decision
                         of this run is robust; it is the first 30 iterations of the reference's restart-30 run)
  bratu_1024_restart30   BASELINE config 3: grid_nodes=1025, krylow_restart=30, max_iter=100 -> 99 iterations
  bratu_8192_k50_cgls    BASELINE config 5: grid_nodes=8193 (67M unknowns), krylow_restart=50, projected least squares
                         by CGLS (cg_rtol 1e-4), max_iter=101 -> 100 iterations; meant for 8 GPUs
  bratu_8192_k50_qr      the same run with the reference's own projected least squares (QR): panels of 33..51 columns
                         take the wide tensor-pipe path (gnk_cholqr_wide_try)

  value     iterations/s with u0 and y resident in HBM and the result left in HBM
  e2e       the same through the public API with HOST buffers: make_res(y) + gauss_newton_krylow(res, u0, jac) -> host
            ndarray, i.e. H2D of y and u0 (pinned) and D2H of x inside the timed region
  roofline  the dominant kernel class of the step: algorithmic bytes / CUDA-event time, vs MEASURED_PEAKS.json
  parity    an extra (untimed) solve with a recording callback, compared with the reference's golden trace
            (tests/golden/*.npz, written by oracle/gen_golden.py from the unmodified reference): counts, per-iteration
            deviation of 64 sampled entries, final loss -- emitted at every N
  workloads (extra key) the other configs measured next to the headline: config 3 at N = 1, config 5 at N = 8
  time_to_tolerance  (N = 1) wall seconds until the solver's own stop test (tol = 1e-8) fires on the converging
            configuration of the reference, compare_without_scaling (bratu_pde_test.py:76-103: grid_resolution = 1)
  cpu_baseline   the reference itself (oracle/_ref, built by oracle/make_ref.sh from /root/reference; the oracle port
            if that is absent) on the host cores, bounded sample of the same workload

`--impl reference` times the reference's own CPU implementation on the host cores on the SAME workload: ONE full solve
(k = 1..30 for the headline workload), whatever --steps/--warmup say -- a solve takes minutes, and a truncated sample
would not be matched work.  `--ref-budget-s` bounds it: when the budget is exhausted the solve is cut at the current
outer iteration and the line says so.

`--dump-outputs DIR` writes what the last timed step of the headline workload returned to DIR (see dump_outputs).

Multi-GPU (torchrun, one rank per GPU): the grid rows are partitioned into slabs, scaling is strong.
"""
import argparse
import contextlib
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "gnk_outer_iterations_per_second"
UNIT = "it/s"

WORKLOADS = {
    "bratu_4096_k30": dict(grid_nodes=4097, restart=None, iters=30, ls="qr", cg_rtol=None,
                           golden=("bratu_g4097", "gnk_k30", "bratu_g4097_sens")),
    "bratu_1024_restart30": dict(grid_nodes=1025, restart=30, iters=99, ls="qr", cg_rtol=None,
                                 golden=("bratu_g1025", "gnk_restart30", "bratu_g1025_sens")),
    "bratu_8192_k50_cgls": dict(grid_nodes=8193, restart=50, iters=100, ls="cgls", cg_rtol=1e-4, golden=None),
    "bratu_8192_k50_qr": dict(grid_nodes=8193, restart=50, iters=100, ls="qr", cg_rtol=None, golden=None),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="bratu_4096_k30", choices=sorted(WORKLOADS) + ["custom"])
    ap.add_argument("--grid-nodes", type=int, default=None, help="custom workload: grid_nodes")
    ap.add_argument("--iters", type=int, default=None, help="custom workload: outer iterations per step")
    ap.add_argument("--restart", type=int, default=None, help="custom workload: krylow_restart")
    ap.add_argument("--ls", default=None, choices=["qr", "cgls"], help="custom workload: projected least squares")
    ap.add_argument("--reorth", type=int, default=1, help="Gram-Schmidt passes (1 = reference, 2 = CGS2)")
    ap.add_argument("--cpu-sample-iters", type=int, default=3,
                    help="outer iterations of the cpu_baseline sample inside the GPU arm (k = 1..3 at 4096^2: ~25 s)")
    ap.add_argument("--ref-budget-s", type=float, default=640.0,
                    help="--impl reference: wall-clock budget of the one full solve (cut at an iteration boundary)")
    ap.add_argument("--extras", default="auto", help="'auto', 'none', or a comma list of extra workloads to attach")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-ttt", action="store_true", help="skip the time-to-tolerance workloads")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result of the headline workload's last timed step to DIR/*.npy (see dump_outputs)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if a.dump_outputs is not None and a.impl != "ours":
        ap.error("--dump-outputs writes the result of the GPU path (--impl ours)")
    if a.grid_nodes is not None or a.iters is not None or a.restart is not None or a.ls is not None:
        a.workload = "custom"
    return a


def workload_spec(a, name=None):
    name = name or a.workload
    if name == "custom":
        return dict(grid_nodes=a.grid_nodes or 4097, restart=a.restart, iters=a.iters or 30, ls=a.ls or "qr",
                    cg_rtol=1e-4 if a.ls == "cgls" else None, golden=None)
    return dict(WORKLOADS[name])


def workload_config(a, spec, name, world):
    G = spec["grid_nodes"]
    label = name if name != "custom" else f"bratu_{G - 1}x{G - 1}_gnk_k{spec['iters']}"
    cfg = dict(workload=label, grid_nodes=G, unknowns=(G - 1) ** 2, ALPHA=5, LAMBDA=10,
               krylow_restart=spec["restart"], max_iter=spec["iters"] + 1, version="res_old", tol=1e-8,
               cgs_passes=a.reorth, projected_least_squares=spec["ls"],
               l2="inputs (basis 0.13-4 GB) exceed the 126 MB L2; no explicit flush",
               parallelism=f"row_slabs_x{world}")
    if spec["cg_rtol"] is not None:
        cfg["cg_rtol"] = spec["cg_rtol"]
    return cfg


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference itself (oracle/_ref) -- or the oracle port when it has not been built
# ------------------------------------------------------------------------------------------------
class _Budget(Exception):
    pass


def cpu_problem(G, grid_resolution=None):
    """(kind, solve, res, u0, jac, error) for the CPU arm; built once, outside every timed region"""
    from oracle import ref_loader
    ref = ref_loader.load_reference()
    if ref is not None:
        kw = {} if grid_resolution is None else dict(grid_resolution=grid_resolution)
        pb = ref.bratu_pde_problem.BratuPdeProblem(G, 5, 10, **kw)
        y = pb.pde_operator(pb.u_true)
        np.random.seed(42)
        u0 = pb.u_true + 0.1 * np.random.normal(loc=0, scale=1, size=pb.u_true.shape[0])

        def solve(res, x0, jac, restart, max_iter, callback):
            out = ref.gauss_newton_krylow.gauss_newton_krylow(res, x0, jac, krylow_restart=restart, max_iter=max_iter,
                                                              callback=callback)
            return out.nit, out.success

        return "reference", solve, pb.make_res(y), u0, pb.make_jac(), pb.make_error()
    from oracle import gnk_oracle as orc
    o = orc.BratuOracle(G, 5, 10) if grid_resolution is None else orc.BratuOracle(G, 5, 10, h=grid_resolution)
    y = o.operator(o.u_true)
    u0 = o.start_vector(seed=42)

    def solve(res, x0, jac, restart, max_iter, callback):
        out = orc.gnk(res, x0, jac, restart=restart, max_iter=max_iter, callback=callback)
        return out["nit"], out["success"]

    return "port", solve, o.make_res(y), u0, o.make_jac(), (lambda x: float(np.linalg.norm(o.u_true - x)))


def cpu_solve(problem, restart, iters, budget_s=None):
    """-> (iterations completed, seconds, finished).  With a budget the solve is cut at the first callback after it."""
    kind, solve, res, u0, jac, _ = problem
    done = [0, 0.0]
    t0 = time.perf_counter()

    def cb(x=None, nfev=None, cg_iter=None):
        done[0] += 1
        done[1] = time.perf_counter() - t0
        if budget_s is not None and done[1] > budget_s:
            raise _Budget()

    try:
        with contextlib.redirect_stdout(sys.stderr):
            nit, _ = solve(res, u0, jac, restart, iters + 1, cb)
        return nit, time.perf_counter() - t0, True
    except _Budget:
        return done[0], done[1], False


# time-to-tolerance workloads: the reference's converging configuration compare_without_scaling (bratu_pde_test.py:76-103:
# grid_nodes=101, grid_resolution=1, default version: 82 iterations) and the same set-up on larger grids with
# version="res_new", which converges within max_iter=100 there (65 / 66 iterations; goldens by oracle/gen_golden.py ttt)
TTT = (("bratu_g101_grid_resolution1_res_old", 101, "res_old"),
       ("bratu_g513_grid_resolution1_res_new", 513, "res_new"),
       ("bratu_g1025_grid_resolution1_res_new", 1025, "res_new"))


def time_to_tolerance_cpu(max_grid=513):
    out = []
    from oracle import ref_loader
    ref = ref_loader.load_reference()
    for name, G, version in TTT:
        if G > max_grid:
            continue
        kind, solve, res, u0, jac, err = cpu_problem(G, grid_resolution=1)
        xs = []
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(sys.stderr):
            if ref is not None:
                o = ref.gauss_newton_krylow.gauss_newton_krylow(res, u0, jac, max_iter=100, version=version,
                                                                callback=lambda x, nfev, cg_iter: xs.append(x))
                nit, success = o.nit, o.success
            else:
                from oracle import gnk_oracle as orc
                o = orc.gnk(res, u0, jac, max_iter=100, version=version,
                            callback=lambda x=None, nfev=None, cg_iter=None: xs.append(x))
                nit, success = o["nit"], o["success"]
        dt = time.perf_counter() - t0
        out.append(dict(workload=name, tol=1e-8, nit=int(nit), success=bool(success), seconds=dt,
                        error=float(err(xs[-1])), kind=kind, impl="reference", cores=os.cpu_count()))
    return out


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    spec = workload_spec(a)
    cores = os.cpu_count()
    cfg = workload_config(a, spec, a.workload, world)
    G = spec["grid_nodes"]
    if G > 5000:
        # SURVEY 8d: the reference needs ~24 GB at 4096^2 and materialises Q and hstack copies; 8192^2 with 50 columns
        # does not fit the host.  Extrapolated linearly in n from the 4096^2 run is all that can be said.
        line = dict(metric=METRIC, value=None, unit=UNIT, n_gpus=a.gpus, steps=0, warmup=0, ms_per_step=None,
                    higher_is_better=True, scaling="strong", vs_baseline=None, dtype="f64", data="synthetic",
                    impl="reference", config=cfg, gpu_launches=0,
                    unavailable="the reference's CPU path at 8192^2 / 50 columns exceeds host RAM (SURVEY 8d)")
        print(json.dumps(line), flush=True)
        return
    problem = cpu_problem(G)
    if spec["ls"] != "qr":
        raise SystemExit("the reference arm times the reference's own QR path; CGLS workloads have no CPU arm")
    nit, dt, finished = cpu_solve(problem, spec["restart"], spec["iters"], budget_s=a.ref_budget_s)
    val = nit / dt
    if finished:
        sample = (f"ONE full solve of the workload ({nit} outer iterations), {dt:.1f} s; --steps/--warmup are ignored "
                  "for this arm (a solve takes minutes)")
    else:
        sample = (f"the full solve was cut after {nit} of {spec['iters']} outer iterations when the {a.ref_budget_s:.0f} s "
                  f"budget ran out ({dt:.1f} s); CPU cost per iteration grows with k, so this flatters the CPU")
    line = dict(metric=METRIC, value=val, unit=UNIT, n_gpus=a.gpus, steps=1, warmup=0, ms_per_step=1e3 * dt,
                higher_is_better=True, scaling="strong", vs_baseline=None, dtype="f64", data="synthetic",
                impl="reference", config=cfg,
                cpu_baseline=dict(value=val, unit=UNIT, cores=cores, kind=problem[0], sample=sample,
                                  matched_work=bool(finished)),
                e2e=dict(value=val, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0,
                result=dict(nit=int(nit), finished=bool(finished)))
    if not a.no_ttt:
        line["time_to_tolerance"] = time_to_tolerance_cpu()
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# clocks during the timed region
# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.reasons, self.max_sm = index, False, [], set(), None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_sm = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                     nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
            while not self.stop_flag:
                self.sm.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(0.05)
        except Exception as e:  # clocks are diagnostics; never fail the bench on NVML
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    def summary(self):
        return dict(sm_mhz=float(np.median(self.sm)) if self.sm else None, sm_max_mhz=self.max_sm,
                    reasons=sorted(self.reasons))


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
DUMP_MAX_X = 1 << 22  # float64 entries of x written by --dump-outputs (32 MiB)


def dump_outputs(dump_dir, out, rank):
    """What the caller of the timed solve receives, so that two builds can be compared output for output:
      x.npy       the solution (float64); above DUMP_MAX_X entries, the entries at a fixed sample of indices
                  (numpy default_rng(0), drawn without replacement, in increasing order)
      counts.npy  [nit, nfev (RegressionResult.nrev), njev, success] as float64
    The inputs of a workload do not change from run to run (u0 from seed 42), so neither does the sample."""
    x = np.asarray(out.x, dtype=np.float64)  # every rank takes part in gathering the sharded solution
    if rank != 0:
        return
    if x.size > DUMP_MAX_X:
        x = x[np.sort(np.random.default_rng(0).choice(x.size, DUMP_MAX_X, replace=False))]
    os.makedirs(dump_dir, exist_ok=True)
    np.save(os.path.join(dump_dir, "x.npy"), x)
    np.save(os.path.join(dump_dir, "counts.npy"),
            np.array([out.nit, out.nrev, out.njev, float(out.success)], dtype=np.float64))


class Harness:
    def __init__(self, a):
        import torch
        import torch.distributed as dist

        self.a, self.torch, self.dist = a, torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        import gauss_newton_via_generalized_krylov_subspaces_b200 as g
        self.g = g
        self.rt = g.get_runtime()
        try:
            self.peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            self.peaks = {}

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, v):
        t = self.torch.tensor([v], dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    # --------------------------------------------------------------------------------------------
    def measure(self, name, steps, warmup, e2e=True, parity=True, sample_clocks=False, dump_dir=None):
        a, g, rt, torch = self.a, self.g, self.rt, self.torch
        spec = workload_spec(a, name)
        G = spec["grid_nodes"]
        n = (G - 1) ** 2
        pb = g.BratuPdeProblem(G, 5, 10)
        u_true = pb.u_true
        y = pb.pde_operator(u_true)
        u0 = u_true + 0.1 * np.random.RandomState(42).normal(loc=0, scale=1, size=n)
        kw = dict(krylow_restart=spec["restart"], max_iter=spec["iters"] + 1, callback=lambda **k: None,
                  reorth_passes=a.reorth)
        if spec["ls"] == "cgls":
            kw.update(ls_solver="cgls", cg_rtol=spec["cg_rtol"])

        # ---- device-resident leg ---------------------------------------------------------------
        res = pb.make_res(y)
        res.y_col  # upload y once
        jac = pb.make_jac()
        x0_dev = pb.dev.resident(u0)

        def step_resident():
            return g.gauss_newton_krylow(res, x0_dev, jac, x_on_device=True, **kw)

        for _ in range(warmup):
            out = step_resident()
        self.barrier()
        sampler = None
        if sample_clocks:
            sampler = ClockSampler(self.local)
            sampler.start()
        l0 = rt.launches()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        its = 0
        for _ in range(steps):
            out = step_resident()
            its += out.nit
        e1.record()
        self.barrier()
        if sampler is not None:
            sampler.stop_flag = True
        ms = self.max_over_ranks(e0.elapsed_time(e1))
        launches = rt.launches() - l0
        value = its / (ms * 1e-3)
        m = dict(value=value, ms_per_step=ms / steps, steps=steps, warmup=warmup, gpu_launches=int(launches),
                 result=dict(nit=int(out.nit), nfev=int(out.nrev), success=bool(out.success)),
                 clocks=sampler.summary() if sampler is not None else None)
        if dump_dir is not None:
            dump_outputs(dump_dir, out, self.rank)
        del out

        # ---- per-kernel roofline pass (events around every kernel class; not part of the headline timing) ----
        rt.begin_profile()
        step_resident()
        prof = rt.end_profile()
        m["kernels"], m["roofline"] = self.roofline(prof, pb, spec)

        # ---- end-to-end leg: host buffers in, host ndarray out -----------------------------------
        if e2e:
            y_pin = torch.empty(n, dtype=torch.float64, pin_memory=True)
            u0_pin = torch.empty(n, dtype=torch.float64, pin_memory=True)
            y_pin.numpy()[:] = y
            u0_pin.numpy()[:] = u0

            def step_e2e():
                r = pb.make_res(y_pin.numpy())
                j = pb.make_jac()
                return g.gauss_newton_krylow(r, u0_pin.numpy(), j, **kw)

            o = None
            for _ in range(warmup):
                o = step_e2e()
            self.barrier()
            t0 = time.perf_counter()
            its_e = 0
            for _ in range(steps):
                del o  # give the previous result's pinned buffer back before the next solve allocates its own
                o = step_e2e()
                its_e += o.nit
            self.barrier()
            dt = self.max_over_ranks(time.perf_counter() - t0)
            h2d = 2 * 8 * pb.dev.h2d_doubles_per_vector()
            d2h = 8 * pb.dev.d2h_doubles_per_vector()
            m["e2e"] = dict(value=its_e / dt, unit=UNIT, h2d_bytes_per_step=int(h2d), d2h_bytes_per_step=int(d2h),
                            ms_per_step=1e3 * dt / steps, final_loss=float(0.5 * np.sum(pb.make_res(y)(o.x) ** 2)),
                            bytes_note="per rank: its slab (+ halo rows) of y and u0 in, its slab of x out" if self.world > 1
                            else "y and u0 in, x out")
            del o

        # ---- parity against the reference's golden trace (untimed) --------------------------------
        if parity and spec["golden"] is not None:
            m["parity"] = self.parity(pb, res, jac, x0_dev, y, kw, spec)
        return m

    # --------------------------------------------------------------------------------------------
    def parity(self, pb, res, jac, x0_dev, y, kw, spec):
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from golden_util import Golden, bound_for
        gname, rname, sname = spec["golden"]
        try:
            gr = Golden(gname).run(rname)
            full_bound = bound_for(gname, rname)
        except Exception as e:
            return dict(available=False, why=f"golden fixture missing: {e}")
        idx = gr["sample_idx"]
        xs, nfevs = [], []

        def cb(x, nfev, cg_iter):
            xs.append(np.asarray(x)[idx].copy())
            nfevs.append(int(nfev))

        kw2 = dict(kw, callback=cb)
        out = self.g.gauss_newton_krylow(res, x0_dev, jac, **kw2)
        nref = len(gr["xs"])
        ncmp = min(len(xs), nref)
        X = np.array(xs[:ncmp])
        scale = np.max(np.abs(gr["xs"][:ncmp]), axis=1, keepdims=True)
        dev = np.max(np.abs(X - gr["xs"][:ncmp]) / scale, axis=1)
        bound = full_bound[:ncmp]
        loss = res.loss(out.x)
        gl = float(gr["loss"][-1]) if np.isfinite(gr["loss"][-1]) else None
        restart = spec["restart"]
        first_cycle = ncmp if restart is None else min(ncmp, restart)
        p = dict(golden=f"tests/golden/{gname}.npz:{rname}", iterations_compared=int(ncmp),
                 callbacks=len(xs), golden_callbacks=int(nref),
                 nfev_sequence_equal=bool(nfevs[:ncmp] == [int(v) for v in gr["nfev_cb"][:ncmp]]),
                 nit=int(out.nit), golden_nit=int(gr["nit"]), nfev=int(out.nrev), golden_nfev=int(gr["nfev"]),
                 max_dev=float(dev.max()), max_dev_first_cycle=float(dev[:first_cycle].max()),
                 max_dev_tail=float(dev[min(12, ncmp - 1):first_cycle].max()) if first_cycle > 12 else None,
                 max_dev_over_bound=float(np.max(dev / bound)), within_bound=bool(np.all(dev <= bound)),
                 dev_per_iteration=[float(f"{v:.3e}") for v in dev],
                 bound_per_iteration=[float(f"{v:.3e}") for v in bound],
                 bound="per iteration max(1e-10, 10 x the largest deviation the reference shows against itself at that "
                       "iteration (+-1) under ONE-ulp changes of u0 (3 draws) and of its own projected least-squares "
                       "solutions) (tests/golden_util.py:sensitivity_bound; fixtures by oracle/gen_golden.py)",
                 final_loss=float(loss), golden_final_loss=gl,
                 final_loss_dev=None if gl is None else float(abs(loss - gl) / gl))
        return p

    # --------------------------------------------------------------------------------------------
    def roofline(self, prof, pb, spec):
        peak = float(self.peaks.get("hbm_gbs", 6650.0))
        peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in self.peaks else "6650 GB/s (of fallback)"
        kernels = {}
        for name, p in prof.items():
            gbs = p["bytes"] / (p["ms"] * 1e-3) / 1e9 if p["ms"] > 0 else 0.0
            kernels[name] = dict(launches=p["launches"], ms=round(p["ms"], 3), achieved_gbs=round(gbs, 1),
                                 frac=round(gbs / peak, 3), bytes_per_launch=p["bytes"] / max(p["launches"], 1))
        # measured DRAM traffic per algorithmic byte from the committed ncu --set full captures (profiles/)
        dram = {}
        for fn in ("r02_dram_traffic.json", "r01_dram_traffic.json"):
            try:
                d = json.load(open(os.path.join(ROOT, "profiles", fn)))
                for k_, v_ in d.items():
                    dram.setdefault(k_, dict(v_, source=fn) if isinstance(v_, dict) else v_)
            except Exception:
                pass
        ncu_name = {"spmm+ls": "stencil_gram_ls"}
        ncu_name.update(tsqr="cholqr", spmm="apply_kernel", combine="combine_kernel",
                        cgs_dots="dots_kernel", cgs_update="update_kernel", residual="residual_kernel",
                        spmv_t="apply_kernel", normalize="normalize_kernel")
        for name in kernels:
            ent = dram.get(ncu_name.get(name, ""), {})
            ratio = ent.get("ratio") if isinstance(ent, dict) else None
            kernels[name]["traffic_per_launch"] = None if ratio is None else ratio * kernels[name]["bytes_per_launch"]
            kernels[name]["traffic_source"] = ent.get("source") if isinstance(ent, dict) and ratio is not None else None
        top = max(prof, key=lambda k_: prof[k_]["ms"]) if prof else None
        roofline = None
        if top:
            total = sum(p["ms"] for p in prof.values())
            roofline = dict(bound="hbm", kernel=top, achieved=kernels[top]["achieved_gbs"], peak=peak, unit="GB/s",
                            frac=kernels[top]["frac"], traffic=kernels[top]["traffic_per_launch"], peak_source=peak_src,
                            share_of_step=round(prof[top]["ms"] / total, 3),
                            traffic_source="dram__bytes_read+write per algorithmic byte (ncu --set full, profiles/"
                                           f"{kernels[top]['traffic_source']}) x this run's bytes per launch",
                            whole_step=dict(bytes=sum(p["bytes"] for p in prof.values()), ms=round(total, 3),
                                            achieved=round(sum(p["bytes"] for p in prof.values()) / (total * 1e-3) / 1e9, 1),
                                            frac=round(sum(p["bytes"] for p in prof.values()) / (total * 1e-3) / 1e9 / peak, 3)))
        return kernels, roofline

    # --------------------------------------------------------------------------------------------
    def time_to_tolerance(self):
        """wall seconds until the solver's own stop test fires (tol = 1e-8), host buffers in and out"""
        g = self.g
        out = []
        for name, G, version in TTT:
            pb = g.BratuPdeProblem(G, 5, 10, grid_resolution=1)
            y = pb.pde_operator(pb.u_true)
            u0 = pb.u_true + 0.1 * np.random.RandomState(42).normal(loc=0, scale=1, size=pb.n)
            err = pb.make_error()
            best, o = None, None
            for _ in range(4):
                self.torch.cuda.synchronize()
                t0 = time.perf_counter()
                o = g.gauss_newton_krylow(pb.make_res(y), u0, pb.make_jac(), callback=lambda **k: None, version=version,
                                          max_iter=100)
                dt = time.perf_counter() - t0
                best = dt if best is None else min(best, dt)
            out.append(dict(workload=name, tol=1e-8, nit=int(o.nit), success=bool(o.success), seconds=best,
                            error=float(err(o.x)), impl="ours", note="best of 4 (the first includes one-time allocations)"))
        return out


def run_ours(a):
    h = Harness(a)
    rank, world = h.rank, h.world
    name = a.workload
    head = h.measure(name, a.steps, a.warmup, e2e=not a.no_e2e, parity=not a.no_parity, sample_clocks=True,
                     dump_dir=a.dump_outputs)

    extras = {}
    if a.extras == "auto":
        want = []
        if name == "bratu_4096_k30":
            if world == 1:
                want.append("bratu_1024_restart30")
            if world == 8:
                want.append("bratu_8192_k50_cgls")
                want.append("bratu_8192_k50_qr")
    elif a.extras == "none":
        want = []
    else:
        want = [w for w in a.extras.split(",") if w]
    for w in want:
        try:
            e = h.measure(w, a.steps, a.warmup, e2e=not a.no_e2e, parity=not a.no_parity)
        except Exception as exc:  # an extra workload must never cost the headline line (raised alike on every rank)
            extras[w] = dict(error=f"{type(exc).__name__}: {exc}")
            continue
        e["config"] = workload_config(a, workload_spec(a, w), w, world)
        e["metric"], e["unit"] = METRIC, UNIT
        if w.startswith("bratu_8192"):
            e["cpu_reference"] = ("not runnable: the reference's CPU path at 8192^2 / 50 columns exceeds host RAM (SURVEY "
                                  "8d: 24 GB at 4096^2 / 30 columns); extrapolated linearly in n and k from the measured "
                                  "4096^2 run it would be ~0.01 it/s")
        extras[w] = e

    ttt = None
    if world == 1 and not a.no_ttt:
        ttt = h.time_to_tolerance()

    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        spec = workload_spec(a)
        problem = cpu_problem(spec["grid_nodes"])
        nit_c, dt_c, _ = cpu_solve(problem, spec["restart"], min(a.cpu_sample_iters, spec["iters"]))
        cpu = dict(value=nit_c / dt_c, unit=UNIT, cores=os.cpu_count(), kind=problem[0],
                   sample=f"first {nit_c} outer iterations (k=1..{nit_c}) of the same workload, {dt_c:.1f} s; CPU cost per "
                          "iteration grows with k, so this flatters the CPU (the full matched solve is what "
                          "`bench.py --impl reference` times)")
        if ttt is not None:
            ttt += time_to_tolerance_cpu()

    if rank == 0:
        cfg = workload_config(a, workload_spec(a), name, world)
        line = dict(metric=METRIC, value=head["value"], unit=UNIT, n_gpus=world, steps=a.steps, warmup=a.warmup,
                    ms_per_step=head["ms_per_step"], higher_is_better=True, scaling="strong", vs_baseline=None,
                    dtype="f64", data="synthetic", config=cfg, clocks=head["clocks"], e2e=head.get("e2e"),
                    gpu_launches=head["gpu_launches"], roofline=head["roofline"], kernels=head["kernels"],
                    cpu_baseline=cpu, result=head["result"], parity=head.get("parity"), workloads=extras or None,
                    time_to_tolerance=ttt)
        print(json.dumps(line), flush=True)
    if world > 1:
        h.dist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    # the contract is ONE JSON line on stdout: the solvers' own prints (the reference's "reached maximal iteration
    # bound" warning etc.) go to stderr
    # -- at the file-descriptor level, so that prints from C libraries (e.g. NCCL's version banner) go there too
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    with contextlib.redirect_stdout(sys.stderr):
        _emit = print

        def print(*a, **k):  # noqa: A001  (the JSON line)
            k.setdefault("file", real_stdout)
            _emit(*a, **k)

        globals()["print"] = print
        if args.impl == "reference":
            run_reference(args)
        else:
            run_ours(args)
