"""Gauss-Newton on generalized Krylov subspaces -- B200 mirror of the reference's ``gauss_newton_krylow.py``.

Same signature, same iteration logic and the same counters as gauss_newton_krylow.py:39-145; the host keeps
only the control flow.  Per outer iteration the device runs (all fp64, see csrc/):

    J V_k            stencil / CSR SpMM                       (:86)
    min|-JV d - r|   Householder TSQR of [-JV | r]            (:89, linear_least_squares :16-36)
    Armijo trials    x = V_k(c + s d) ; fused residual+norm   (:91-93, armijo_goldstein.py:47-72)
    c += s d ; stop test on s^2|d|^2 <= tol^2 |c_prev|^2      (:96-104)
    J(x_new)         e^x is a by-product of the accepted trial (:107)
    basis expansion  -J^T r, Gram-Schmidt vs V_k, normalise, append in place   (:110-124, krylow.py:55-73)
    restart          V <- [x/|x|]                              (:135-136)

and the host reads one small block of scalars per Armijo trial plus the breakdown flag.
"""
from __future__ import annotations

import ctypes as C
import os
import weakref
from typing import Any, Callable, Optional, Tuple

import numpy as np

from . import _lib
from .armijo_goldstein import armijo_device
from .bratu_pde_problem import BratuDeviceProblem
from .device import (DeviceCallableProblem, DeviceVector, HostCallableProblem, get_runtime, is_cuda_tensor,
                     make_layout, ptr)
from .krylow import (GeneralizedKrylowSubspace, GeneralizedKrylowSubspaceBreakdown,
                     GeneralizedKrylowSubspaceSpansEntireSpace, MAX_COLUMNS)
from .partition import flat_layout_fields, round_up, tensor_ls_on_every_rank
from .regression_result import RegressionResult
from .rosenbrock_problem import RosenbrockDeviceProblem

_NB = _lib.GNK_MAX_BASIS
_TSQR_MAX = _lib.GNK_TSQR_MAX
_DENSE_QR_MAX = 1 << 22  # doubles of the single-CTA wide-panel QR (csrc/tsqr.cu: run_dense_qr)
# layout of the per-iteration scalar block (device, one D2H read per Armijo trial)
_SC_LOSS = 2 * _NB + 8   # 2 doubles: sum(F^2) [, max|F|]
_SC_CPREV = _SC_LOSS + 2  # sum(c_prev^2)
_SC_FLAG = _SC_CPREV + 2   # int32 in a double slot: the deferred Krylov breakdown flag (krylow.dev_update)
_SC_FLAG2 = _SC_CPREV + 3  # second slot: an expansion writes its flag to the slot that is NOT pending, committing it flips
_BLK = _SC_CPREV + 6
_VERSIONS = ("res_old", "res_new", "jac_old_res_old", "jac_old_res_new")


def resolve_problem(res, jac, x0, args, native_rosenbrock=False):
    if is_cuda_tensor(x0):  # a CUDA-tensor x0: res / jac take and return CUDA tensors
        return DeviceCallableProblem(res, jac, x0, args)
    if BratuDeviceProblem.match(res, jac) and not args:
        return BratuDeviceProblem(res, jac)
    if native_rosenbrock and RosenbrockDeviceProblem.match(res, jac, args) \
            and os.environ.get("GNK_NATIVE_ROSENBROCK", "1") != "0":
        return RosenbrockDeviceProblem(x0)
    return HostCallableProblem(res, jac, x0, args)


def require_single_rank_unless_sharded(rt, prob, who):
    """Only the Bratu problem is row-sharded over the ranks of a process group.  Every other problem (foreign
    callables, the chained Rosenbrock problem, stand-alone least squares) holds FULL vectors on every rank, while the
    library's reductions sum over all ranks once a communicator is attached -- norms would come out sqrt(world) too
    large and the Armijo test would compare against world * g.  SURVEY 8e asks for "replicas only" there: run those
    problems in processes without a process group (or with world_size 1)."""
    if rt.world > 1 and not getattr(prob, "distributed", False):
        raise _lib.GnkError(
            f"{who}: this problem is not row-sharded (only BratuPdeProblem is), but the process group has "
            f"{rt.world} ranks and the library would sum its reductions over all of them.  Run replicated problems "
            "in single-rank processes (no torch.distributed process group).")


def tsqr_solve(rt, A, lda, n_rows, k, y, sign, out, householder=False, method=None):
    """gnk_tsqr_ls.  Large panels are factored on the FP64 tensor pipe (csrc/cholqr.cu: Gram matrix + Cholesky, then
    one refinement step or the second CholeskyQR2 pass), which refuses numerically rank deficient panels by writing
    d = 0 and out[k+2] = -1 (``ls_refused``); the caller then comes back with ``householder=True``, which pins the
    Householder TSQR for this call.  ``method``: 0 automatic, 1 Householder, 2 CholeskyQR2 without the refinement form
    (gnk_tsqr_ls_method)."""
    if method is None:
        method = 1 if householder else 0
    prev = rt.lib.gnk_tsqr_ls_method(rt.ctx, method) if method else 0  # returns the previous setting (>= 0)
    if prev < 0:
        _lib.check(prev, "gnk_tsqr_ls_method")
    try:
        _lib.check(rt.lib.gnk_tsqr_ls(rt.ctx, ptr(A), lda, n_rows, k, ptr(y), float(sign), ptr(out), rt.stream),
                   "gnk_tsqr_ls")
    finally:
        if method:
            rt.lib.gnk_tsqr_ls_method(rt.ctx, prev)


def ls_refused(vals, k):
    return vals[k + 2] < 0


class _LeastSquaresRefused(Exception):
    pass


class _DeferredBreakdown(Exception):
    pass


def _report_rank(vals, k):
    """the prints of gauss_newton_krylow.py:32-34, and scipy's solve_triangular error for an exactly singular R (:35)"""
    for _ in range(int(vals[k + 2])):
        print("A is rank deficient")
    diag = vals[k + 4:2 * k + 4]
    zero = np.nonzero(diag == 0.0)[0]
    if zero.size:
        raise np.linalg.LinAlgError(f"singular matrix: resolution failed at diagonal {int(zero[0])}")


def cgls_dense(rt, JV, ldjv, n_rows, k, y, sign, rtol, out):
    """Projected least squares by CGLS instead of QR (BASELINE config 5: "Krylov dim 50 with CGLS inner solve"):
    min || sign*JV d - y || via CG on the normal equations with the Jacobi preconditioner 1/diag(A^T A), i.e. the
    reference's ``cg_least_squares(A, y, cg_rtol, preconditioner=True)`` (gauss_newton.py:11-60 / scipy cg) applied to
    the dense n x k matrix A = sign*JV.  The n-sized work (A p = JV p, A^T t = JV^T t, column norms) runs in the same
    combine / dots / norm kernels as the Krylov path, row-sharded with one k-sized all-reduce per product; the
    k-sized CG recurrences run on the host.  Fills ``out`` like ``gnk_tsqr_ls`` (d, ||JV d||^2, -, 0, ||d||^2).
    Returns the number of CG iterations."""
    lib = rt.lib
    lay = make_layout(dict(flat_layout_fields(n_rows), ld=ldjv))
    h = rt.zeros(_NB)
    pdev = rt.zeros(_NB)
    t = rt.empty(ldjv)
    stats = rt.zeros(2 * k)
    stage = rt.pinned(_NB)
    stage_np = stage.numpy()

    def at_times(vec):  # A^T vec = sign * JV^T vec
        _lib.check(lib.gnk_cgs_dots(rt.ctx, C.byref(lay), ptr(JV), k, ptr(vec), ptr(h), rt.stream), "gnk_cgs_dots")
        if not rt.fused_reductions:
            rt.allreduce(h, k, 0)
        return sign * rt.read(h, k)

    def a_times(pv):  # t = JV pv (the sign is applied by the caller)
        stage_np[:k] = pv
        pdev[:k].copy_(stage[:k], non_blocking=True)
        _lib.check(lib.gnk_combine(rt.ctx, C.byref(lay), ptr(JV), k, ptr(pdev), None, 0.0, ptr(t), rt.stream),
                   "gnk_combine")

    for j in range(k):
        _lib.check(lib.gnk_norm_stats(rt.ctx, C.byref(lay), ptr(JV, j * ldjv), ptr(stats, 2 * j), rt.stream),
                   "gnk_norm_stats")
    rt.allreduce(stats, 2 * k, 0)
    minv = 1.0 / (sign * sign * rt.read(stats, 2 * k)[0::2])
    b = at_times(y)
    bn = float(np.linalg.norm(b))
    x = np.zeros(k)
    its = 0
    if bn != 0.0:
        atol = rtol * bn
        r = b.copy()
        rho_prev, pv = None, None
        for it in range(10 * k):
            if np.linalg.norm(r) < atol:
                break
            z = minv * r
            rho = float(np.dot(r, z))
            pv = z.copy() if it == 0 else z + (rho / rho_prev) * pv
            a_times(pv)
            q = sign * at_times(t)  # A^T (A p) = sign^2 JV^T JV p
            alpha = rho / float(np.dot(pv, q))
            x += alpha * pv
            r -= alpha * q
            rho_prev = rho
            its += 1
    a_times(x)
    _lib.check(lib.gnk_norm_stats(rt.ctx, C.byref(lay), ptr(t), ptr(stats), rt.stream), "gnk_norm_stats")
    rt.allreduce(stats, 1, 0)
    g = float(rt.read(stats, 1)[0])
    stage_np[:k] = x
    stage_np[k:k + 4] = (g, 0.0, 0.0, float(np.dot(x, x)))
    out[:k + 4].copy_(stage[:k + 4], non_blocking=True)
    rt.sync()
    return its


def linear_least_squares(A, y):
    """Least squares solution of ||y - A x|| by Householder TSQR on the device (reference :16-36: economic QR,
    a print per |r_kk| <= 1e-8, triangular solve).  A: (n, k) ndarray, y: (n,) ndarray -> x: (k,) ndarray; or A: dense
    (n, k) CUDA tensor, y: CUDA tensor -> x: CUDA tensor."""
    rt = get_runtime()
    require_single_rank_unless_sharded(rt, None, "linear_least_squares")
    on_device = is_cuda_tensor(A)
    if on_device:
        from .device import _require_on_device
        _require_on_device(rt, A, "linear_least_squares: A")
        _require_on_device(rt, y, "linear_least_squares: y")
        if A.dim() != 2 or A.layout != rt.torch.strided:
            raise ValueError(f"linear_least_squares: A must be a dense 2-D tensor, got shape {tuple(A.shape)} "
                             f"and layout {A.layout}")
        y = y.reshape(-1)
        if y.shape[0] != A.shape[0]:
            raise ValueError(f"linear_least_squares: y must have {A.shape[0]} entries, got {y.shape[0]}")
    else:
        A = np.asarray(A, dtype=np.float64)
        y = np.asarray(y, dtype=np.float64).reshape(-1)
    n, k = A.shape
    if k + 1 > _NB:
        raise _lib.GnkError(f"linear_least_squares supports at most {_NB - 1} columns")
    # The host-array entry keeps the single-CTA QR's range for panels wider than 104 columns, as it always had; the
    # blocked TSQR for larger wide panels serves the device-resident panels of gauss_newton_krylow and gauss_newton.
    if k + 1 > _TSQR_MAX and n * (k + 1) > _DENSE_QR_MAX:
        raise _lib.GnkError(f"linear_least_squares with more than {_TSQR_MAX - 1} columns is limited to panels of "
                            "2^22 doubles")
    lda = round_up(max(n, 1), 16)
    dA = rt.zeros(lda * k)
    dy = rt.zeros(lda)
    if on_device:
        dA.view(k, lda)[:, :n].copy_(A.T)
        dy[:n].copy_(y)
    else:
        for j in range(k):
            rt.upload(np.ascontiguousarray(A[:, j]), dA[j * lda:j * lda + n])
        rt.upload(y, dy[:n])
    out = rt.zeros(2 * _NB + 8)
    tsqr_solve(rt, dA, lda, n, k, dy, 1.0, out)
    vals = rt.read(out, 2 * k + 4)
    if ls_refused(vals, k):
        tsqr_solve(rt, dA, lda, n, k, dy, 1.0, out, householder=True)
        vals = rt.read(out, 2 * k + 4)
    _report_rank(vals, k)
    return out[:k].clone() if on_device else vals[:k].copy()


def gauss_newton_krylow(
    res: Callable,
    x0,
    jac: Callable,
    krylow_restart: Optional[int] = None,
    args: Tuple = (),
    tol: float = 1e-8,
    max_iter=100,
    callback: Callable = lambda: None,
    version: str = "res_old",
    reorth_passes: int = 1,
    x_on_device: bool = False,
    ls_solver: str = "qr",
    cg_rtol: float = 1e-4,
) -> RegressionResult:
    """
    Parameters
    ----------
    res: The residual function, called as res(x, *args).
    x0: Initial guess of the regression parameters.
    jac: Jacobian of residual function, called as jac(x, *args).
    krylow_restart: If the basis gets larger than krylow_restart it is reset; None = never.
    args: Additional arguments passed to res and jac.
    tol: Tolerance for termination by the change of the parameters x.
    max_iter: Maximum number of iterations.
    callback: Called as callback(x=, nfev=, cg_iter=None) once per iteration; x converts lazily to ndarray.
    version: One of ['res_old','res_new','jac_old_res_old','jac_old_res_new'] (see reference :61).
    reorth_passes: 1 = the reference's single classical Gram-Schmidt pass (krylow.py:64); 2 = CGS2.
    ls_solver: "qr" = Householder TSQR (the reference's QR); "cgls" = Jacobi-preconditioned CG on the normal equations
        of the projected problem with tolerance ``cg_rtol`` (BASELINE config 5).
    x_on_device: leave the solution in HBM (RegressionResult.x is then a lazy DeviceVector).  x0 may likewise be a
        DeviceVector made by ``BratuPdeProblem.dev.resident(u0)``.

    Returns
    -------
    RegressionResult
    """
    rt = get_runtime()
    lib = rt.lib
    success = False
    # a start vector already in HBM is used in place only by the problem that made it (BratuPdeProblem.dev.resident);
    # for every other problem a DeviceVector is an ordinary array-like and is read through its host copy
    x0_resident = (isinstance(x0, DeviceVector) and x0._t is not None and BratuDeviceProblem.match(res, jac)
                   and not args and getattr(x0._owner, "pb", None) is res.pb)
    if x0_resident or is_cuda_tensor(x0):
        x0_host = x0 if not x0_resident else None  # a CUDA tensor stays on the device (DeviceCallableProblem.upload_x)
    else:
        x0_host = np.asarray(x0, dtype=np.float64).reshape(-1)
    prob = resolve_problem(res, jac, x0 if x0_resident else x0_host, args, native_rosenbrock=True)
    require_single_rank_unless_sharded(rt, prob, "gauss_newton_krylow")
    if krylow_restart is None:
        krylow_restart = max_iter

    krylow = GeneralizedKrylowSubspace(prob, capacity=min(max_iter, krylow_restart) + 1, reorth_passes=reorth_passes)
    krylow._setup(prob.p_glob, prob.sol_fields, prob.sol, prob, krylow.capacity)
    ld = krylow.ld
    sol_lay = prob.sol

    blk = rt.zeros(_BLK)            # [d(k) | g | resid2 | ndef | dnorm2 | diagR(k) ... | loss(2) | cprev2]
    loss_slot = blk[_SC_LOSS:_SC_LOSS + 2]
    # coordinates: the current point's c and the trial's c + s d, which gnk_combine_step leaves on the device (with the
    # next column's zero entry appended, :124); accepting a trial swaps the two -- no k-sized kernel is launched
    cbuf = [rt.zeros(_NB), rt.zeros(_NB)]
    c, c_next = cbuf
    one = rt.pinned(1)

    def set_c0(value):
        c.zero_()
        one[0] = value
        c[:1].copy_(one, non_blocking=True)

    if x0_resident:
        x_start = x0._t
    else:
        x_start = prob.new_sol()
        prob.upload_x(x0_host, x_start)
    set_c0(krylow.dev_start(x_start))

    x_trial = prob.new_sol()
    krylow.dev_combine(c, None, 0.0, x_trial)
    is_bratu = isinstance(prob, BratuDeviceProblem)
    native = is_bratu or getattr(prob, "device_native", False)  # res / jac have device twins: no host evaluation
    user_code = getattr(prob, "user_code", False)  # device callables: native, but evaluated only where the reference does
    if not native:  # residual-space size of a foreign callable is known after its first evaluation
        r0 = np.asarray(res(prob.download_global(x_trial), *args), dtype=np.float64).reshape(-1)
        prob._ensure_res_layout(r0.shape[0])
    elif user_code:
        r0 = prob.evaluate(x_trial)
    F_cur, F_trial = prob.new_res(), prob.new_res()
    res_off = prob.res_fields["off"]
    n_res_own = prob.res_fields["n_own"]
    ldjv = round_up(max(n_res_own, 1), 16)
    use_aux = is_bratu and prob.pb.LAMBDA != 0
    aux = [prob.new_sol() for _ in range(3)] if use_aux else [None, None, None]  # e^x: J_cur, trial, spare
    hx = prob.d.halo_exchange if (is_bratu and prob.distributed) else None
    # Several ranks must take the SAME least-squares path (the tensor-pipe path and the Householder TSQR issue
    # different collectives).  The library decides per call from its local slab (>= 16384 owned rows, even count), which
    # uneven slabs can split; only the host knows every rank's slab, so it pins the Householder path for the solve
    # unless all slabs qualify.
    ls_method = 0
    if is_bratu and prob.distributed and not tensor_ls_on_every_rank(prob.sol_fields["m"], rt.world):
        ls_method = 1

    if user_code:
        F_cur[:n_res_own].copy_(r0)
        prob.sumsq(F_cur, loss_slot, prob.res_lay)
    elif native:
        prob.residual(x_trial, F_cur, loss_slot, aux=None)
    else:
        rt.upload(r0, F_cur[:n_res_own])
        prob.sumsq(F_cur, loss_slot, prob.res_lay)
    nfev = 1
    prev_loss = float(rt.read(loss_slot, 1)[0])
    jac_ev = prob.jacobian(x_start, aux=None)  # note: at x0 itself (reference :78), not at V c
    if use_aux:
        aux[0] = jac_ev.expu
    njev = 1

    JV = None
    jv_cap = 0
    # pending: the last basis expansion left its breakdown flag unread (see below); fslot: the slot that holds it.  A new
    # expansion always writes the OTHER slot, so neither a device copy nor a race with the read-back is needed.
    state = {"pending": False, "fslot": _SC_FLAG}

    def other_slot():
        return _SC_FLAG2 if state["fslot"] == _SC_FLAG else _SC_FLAG

    defer_ok = ls_solver == "qr" and os.environ.get("GNK_DEFER_BREAKDOWN", "1") != "0"

    for iter in range(1, max_iter):
        # One host synchronisation per outer iteration: the breakdown flag of the previous basis expansion is not read
        # back when it is written (krylow.dev_update, deferred_flag) but arrives with the scalar block of this
        # iteration's first Armijo trial.  If it was set, the speculatively appended column is retracted and the
        # iteration is redone with the unchanged basis (breakdowns are rare: only the degenerate linear problems).
        for attempt in (0, 1):
            k = krylow.k
            state["rank_reported"] = False
            if k > jv_cap:
                jv_cap = min(MAX_COLUMNS, max(krylow.cap, k))
                JV = rt.empty(jv_cap * ldjv)
            # projected operator and projected least squares  (:86-89)
            ls_done = False
            # Bratu + QR: one TMA-staged kernel applies the stencil, stores J V_k and forms the Gram matrix of the
            # panel in the same sweep (gnk_stencil_gram_ls); it answers 1 when the panel does not qualify
            if (is_bratu and ls_solver == "qr" and ls_method == 0 and not jac_ev.transposed
                    and jac_ev.scale == 1.0):
                # algorithmic bytes (SURVEY 8d): the SpMM's 16nk + 8n plus the least-squares panel once, 8n(k+1)
                with rt.mark("spmm+ls", 8.0 * n_res_own * (3 * k + 2)) as mk:
                    rc = lib.gnk_stencil_gram_ls(rt.ctx, C.byref(sol_lay), C.byref(prob.d.prm), ptr(jac_ev.expu),
                                                 ptr(krylow.V), ld, krylow.cap, k, ptr(F_cur), -1.0, ptr(JV), ldjv,
                                                 -1.0, ptr(blk), rt.stream)
                    mk.cancel = rc != 0
                if rc == 0:
                    ls_done = True
                elif rc != 1:
                    _lib.check(rc, "gnk_stencil_gram_ls")
            if not ls_done:
                with rt.mark("spmm", 8.0 * n_res_own * (2 * k + 1)):
                    jac_ev.matmat(krylow.V, ld, k, JV, ldjv)
            if ls_done:
                pass
            elif ls_solver == "qr":
                with rt.mark("tsqr", 8.0 * n_res_own * (k + 1)):
                    tsqr_solve(rt, JV, ldjv, n_res_own, k, F_cur[res_off:], -1.0, blk, method=ls_method)
            elif ls_solver == "cgls":
                # CG on the k x k normal equations formed once on the tensor pipe, recurrence in one kernel
                # (gnk_gram_cgls); panels it does not take (odd row counts, > 55 columns) run the reference-shaped loop
                # over the n x k panel (cgls_dense)
                if k + 1 <= 56 and n_res_own % 2 == 0 and ldjv % 2 == 0:
                    with rt.mark("gram_cgls", 8.0 * n_res_own * (k + 1)):
                        _lib.check(lib.gnk_gram_cgls(rt.ctx, ptr(JV), ldjv, n_res_own, k, ptr(F_cur, res_off), -1.0,
                                                     float(cg_rtol), ptr(blk), rt.stream), "gnk_gram_cgls")
                else:
                    cgls_dense(rt, JV, ldjv, n_res_own, k, F_cur[res_off:], -1.0, cg_rtol, blk)
            else:
                raise ValueError("ls_solver must be 'qr' or 'cgls'")
            # Speculative basis expansion: everything the expansion needs -- J at the trial point (e^x is a by-product
            # of the trial's residual kernel), the residuals -- exists once the FIRST trial has been enqueued, and in
            # every Bratu / Rosenbrock run measured that trial is accepted.  So -J^T r, the Gram-Schmidt pass and the
            # normalisation are enqueued BEHIND the trial and BEFORE the host reads the trial's loss: the device keeps
            # working while the host waits for the scalars, judges the trial, runs the callback and enqueues the next
            # iteration's least squares.  A rejected first trial simply does not commit the expansion (it is redone
            # after the accepted trial; w, h, column k and the flag slot are overwritten).  Only with device-native
            # residual / Jacobian (no host evaluation in between) and when the breakdown flag may be read late.  Never
            # with the user's device callables: jac would be called at a trial point the reference may reject.
            spec_ok = (native and not user_code and defer_ok and iter + 1 < max_iter and iter % krylow_restart != 0
                       and version in _VERSIONS and krylow.k < prob.p_glob
                       and os.environ.get("GNK_SPECULATE", "1") != "0")
            state["spec"] = None

            def expansion_operands(jac_new):
                if version == "res_old":
                    return jac_new, F_cur
                if version == "res_new":
                    return jac_new, F_trial
                if version == "jac_old_res_old":
                    return jac_ev, F_cur
                return jac_ev, F_trial

            # Armijo-Goldstein in coordinate space  (:91-93)
            def trial_loss(s):
                krylow.dev_combine(c, blk, s, x_trial, c_out=c_next, cprev2=ptr(blk, _SC_CPREV))
                with rt.mark("residual", 32.0 * n_res_own):
                    prob.residual(x_trial, F_trial, loss_slot, aux=aux[1])
                if spec_ok and state["spec"] is None:
                    pending_read = rt.read_begin(blk, _BLK)   # the scalars of this trial are complete here ...
                    jac_new = prob.jacobian(x_trial, aux=aux[1])
                    krylow.dev_expand_enqueue(*expansion_operands(jac_new), hx, ptr(blk, other_slot()))
                    state["spec"] = jac_new
                    state["vals"] = rt.read_end(pending_read)   # ... and are read while the expansion runs
                else:
                    if state["spec"] is not None:
                        state["spec"] = False  # a later trial: the speculation belonged to a rejected one
                    state["vals"] = rt.read(blk, _BLK)
                if state["pending"] and state["vals"][state["fslot"]:state["fslot"] + 1].view(np.int32)[0] != 0:
                    raise _DeferredBreakdown()
                if ls_solver == "qr" and ls_refused(state["vals"], k):
                    raise _LeastSquaresRefused()
                if ls_solver == "qr" and not state["rank_reported"]:
                    # the reference prints / raises inside linear_least_squares (:32-35), i.e. before any trial is
                    # judged: an exactly singular R must surface as LinAlgError, not as 100 rejected NaN trials
                    state["rank_reported"] = True
                    _report_rank(state["vals"], k)
                return float(state["vals"][_SC_LOSS])

            def line_search():
                return armijo_device(trial_loss, prev_loss, lambda: float(state["vals"][k]),
                                     lambda: float(np.sqrt(state["vals"][k + 3])))

            try:
                step_length, nfev_delta = line_search()
            except _DeferredBreakdown:
                state["pending"] = False
                krylow.retract()
                print(f"Generalized krylow subspace breakdown at iteration = {iter - 1}, "
                      f"basis.shape = ({prob.p_glob}, {krylow.k})")
                continue
            except _LeastSquaresRefused:
                # CholeskyQR2 met a numerically rank deficient panel (d = 0 was written, the trial above evaluated the
                # unchanged iterate and is not counted): same panel again through the Householder TSQR
                with rt.mark("tsqr", 8.0 * n_res_own * (k + 1)):
                    tsqr_solve(rt, JV, ldjv, n_res_own, k, F_cur[res_off:], -1.0, blk, householder=True)
                state["rank_reported"] = False
                step_length, nfev_delta = line_search()
            state["pending"] = False
            break
        nfev += nfev_delta
        vals = state["vals"]
        squared_sum_d = float(vals[k + 3])
        squared_sum_x_prev = float(vals[_SC_CPREV])

        # c += s d  (:98): the accepted trial's coordinates are already on the device
        c, c_next = c_next, c

        if user_code:
            callback(x=prob.x_out(x_trial), nfev=nfev, cg_iter=None)
        else:
            xv = DeviceVector(prob, x_trial, prob.p_glob)
            callback(x=xv, nfev=nfev, cg_iter=None)
            xref = weakref.ref(xv)
            del xv                      # if the callback kept x, the weak reference is still alive ...
            DeviceVector.settle(xref)   # ... and x takes its host snapshot before the buffer is reused

        if step_length**2 * squared_sum_d <= tol**2 * squared_sum_x_prev:
            success = True
            break

        jac_ev_old = jac_ev
        speculated = state["spec"] is not None and state["spec"] is not False
        # device callables, jac_old_*: -J_old^T r is formed before jac is called at the new point, so that a jac which
        # refills the tensor it returned last time cannot change J_old under the expansion (same bits, earlier)
        w_ready = (user_code and not speculated and version in ("jac_old_res_old", "jac_old_res_new")
                   and krylow.k < prob.p_glob)
        if w_ready:
            krylow.dev_rmatvec(jac_ev_old, F_cur if version == "jac_old_res_old" else F_trial)
            jac_ev_old = None
        jac_ev = state["spec"] if speculated else prob.jacobian(x_trial, aux=aux[1])  # e^x came out of the trial
        njev += 1

        # defer the breakdown read-back unless this iteration is the last one or ends with a restart (the message
        # of :127 must appear before either)
        defer = defer_ok and iter + 1 < max_iter and iter % krylow_restart != 0
        new_slot = other_slot()
        dflag = ptr(blk, new_slot) if defer else None
        try:
            if speculated:
                # the expansion was enqueued behind the accepted trial; its flag sits in the other slot, which becomes
                # the one the next iteration inspects
                krylow.commit()
            elif version == "res_old":
                krylow.dev_update(jac_ev, F_cur, hx, dflag)
            elif version == "res_new":
                krylow.dev_update(jac_ev, F_trial, hx, dflag)
            elif version == "jac_old_res_old":
                krylow.dev_update(jac_ev_old, F_cur, hx, dflag)
            elif version == "jac_old_res_new":
                krylow.dev_update(jac_ev_old, F_trial, hx, dflag)
            else:
                raise ValueError(
                    "Variable version must be in ['res_old','res_new','jac_old_res_old','jac_old_res_new']"
                )
            state["pending"] = defer
            if defer:
                state["fslot"] = new_slot
        except GeneralizedKrylowSubspaceBreakdown:
            print(
                f"Generalized krylow subspace breakdown at iteration = {iter}, basis.shape = ({prob.p_glob}, {krylow.k})"
            )
        except GeneralizedKrylowSubspaceSpansEntireSpace:
            print(
                f"Warning: The genearlized krylow subspace is now identical to the whole parameter space at iteration = {iter}"
            )

        # the trial becomes the current point
        F_cur, F_trial = F_trial, F_cur
        prev_loss = float(vals[_SC_LOSS])
        if use_aux:
            aux[0], aux[1], aux[2] = aux[1], aux[2], aux[0]
        del jac_ev_old

        if iter % krylow_restart == 0:  # (:135-136)  x = V c equals the accepted trial point bit for bit
            set_c0(krylow.dev_start(x_trial))

    if not success:
        print("Warning: The gauss_newton_krylow algorithm reached maximal iteration bound before terminating!")

    krylow.dev_combine(c, None, 0.0, x_trial)
    if user_code:
        x_final = prob.x_out(x_trial)
    else:
        x_final = DeviceVector(prob, x_trial, prob.p_glob) if x_on_device else prob.download_global(x_trial)
    return RegressionResult("gauss newton krylow", x_final, success, nfev, njev, iter)
