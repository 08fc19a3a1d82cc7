"""Classical Gauss-Newton in the full space -- B200 mirror of the reference's ``gauss_newton.py``.

Sparse (or matrix-free stencil) Jacobians take the CGLS route of gauss_newton.py:11-60,111-114 -- conjugate
gradients on the normal equations with the Jacobi preconditioner, built from the same SpMV / SpMV-transpose
kernels as the Krylov path (``gnk_cgls``); dense Jacobians (the 2x2 / 2x1 problems of
rosenbrock_3d_test.py and powell_divergence_test.py, up to dense fits of 4095 parameters) take a Householder
least-squares solve on the device in place of ``scipy.linalg.lstsq`` (:116): ``gnk_tsqr_ls`` up to 255 columns, the
blocked QR ``gnk_dense_qr_ls`` for 256..4095 columns, which takes J as it comes (one copy into a column-major panel,
no CSR form) and hands ||J d||^2 = ||R d||^2 to the Armijo rule.  ``step_length_control`` stays a plug-in point: the default
``armijo_goldstein`` runs device-native; a user function is called with host objects exactly like the
reference does (:118-120).
"""
from __future__ import annotations

import ctypes as C
import weakref
from typing import Callable, Tuple

import numpy as np

from . import _lib
from .armijo_goldstein import armijo_device, armijo_goldstein
from .bratu_pde_problem import BratuDeviceProblem, StencilJacobian
from .device import (_INT32_LIMIT, CsrJacobian, DenseDeviceJacobian, DenseJacobian, DeviceCsrJacobian,
                     DeviceLinearOperator, DeviceVector, _require_on_device, get_runtime, is_cuda_tensor, make_layout, ptr)
from .gauss_newton_krylow import _report_rank, require_single_rank_unless_sharded, resolve_problem, tsqr_solve
from .partition import flat_layout_fields, round_up
from .regression_result import RegressionResult

_NB = _lib.GNK_MAX_BASIS


def _cgls(rt, linop, y, rtol, preconditioner, x_out, vlen, x0=None):
    work = rt.zeros(7 * vlen)
    iters = C.c_int64(0)
    _lib.check(rt.lib.gnk_cgls_x0(rt.ctx, C.byref(linop), ptr(y), ptr(x0), float(rtol), int(bool(preconditioner)),
                                  ptr(x_out), ptr(work), C.byref(iters), rt.stream), "gnk_cgls")
    return int(iters.value)


def _device_operator(rt, A, what="cg_least_squares: A"):
    """a CUDA A -> DenseDeviceJacobian (strided) or DeviceCsrJacobian (sparse CSR / COO)"""
    if A.layout != rt.torch.strided:
        return DeviceCsrJacobian.from_tensor(rt, A, what)
    _require_on_device(rt, A, what)
    if A.dim() != 2:
        raise ValueError(f"{what}: expected a 2-D Jacobian, got shape {tuple(A.shape)}")
    if max(A.shape) >= _INT32_LIMIT:
        raise _lib.GnkError(f"{what}: a {A.shape[0]} x {A.shape[1]} matrix does not fit the dense kernels (n_res and p "
                            "must stay below 2^31 - 1; their product may be larger)")
    return DenseDeviceJacobian(rt, A)


def _refuse_operator(who, J):
    """matrix-free operators serve gauss_newton_krylow only: these solvers need J's entries (the reference fails here
    too, in scipy.linalg.lstsq(-1 * J, r) and in the A.T @ A of its Jacobi preconditioner)"""
    raise TypeError(f"{who}: got a {type(J).__name__}, a matrix-free operator; {who} needs the Jacobian's entries "
                    "(a dense array or a sparse matrix).  Matrix-free Jacobians are taken by gauss_newton_krylow.")


def cg_least_squares(A, y, x0=None, cg_rtol=1e-4, preconditioner=True):
    """Iterative solver for min ||y - A x|| via CG on the normal equations (reference :11-60), on the device.

    A: scipy sparse matrix / ndarray / device stencil operator, y: ndarray -- or A: CUDA tensor (torch sparse CSR / COO,
    or dense), y (and x0): CUDA tensors, and x comes back as a CUDA tensor.  A dense CUDA A is read in place (one
    contiguous float64 copy if it is of another dtype or has no unit stride), with no CSR form and no limit on its number
    of entries; the result is the one its CSR form gives, bit for bit.  Returns (x, cg_iter) where cg_iter
    sums the unpreconditioned and the preconditioned run when ``preconditioner`` is False (reference quirk)."""
    from scipy.sparse.linalg import LinearOperator
    if isinstance(A, (LinearOperator, DeviceLinearOperator)):
        _refuse_operator("cg_least_squares", A)
    rt = get_runtime()
    if is_cuda_tensor(A):
        require_single_rank_unless_sharded(rt, None, "cg_least_squares")
        op = _device_operator(rt, A)
        _require_on_device(rt, y, "cg_least_squares: y")
        y = y.reshape(-1)
        if y.shape[0] != op.n_res:
            raise ValueError(f"cg_least_squares: y must have {op.n_res} entries, got {y.shape[0]}")
        vlen = round_up(max(op.p, op.n_res), 16)
        dy = rt.zeros(vlen)
        dy[:op.n_res].copy_(y)
        x = rt.zeros(vlen)
        dx0 = None
        if x0 is not None:
            _require_on_device(rt, x0, "cg_least_squares: x0")
            if x0.numel() != op.p:
                raise ValueError(f"cg_least_squares: x0 must have {op.p} entries, got {x0.numel()}")
            dx0 = rt.zeros(vlen)
            dx0[:op.p].copy_(x0.reshape(-1))
        it = _cgls(rt, op.linop(1.0), dy, cg_rtol, preconditioner, x, vlen, dx0)
        return x[:op.p].clone(), it
    if isinstance(A, StencilJacobian) and A.transposed:
        # the device stencil operator has no transpose of its own (J is not symmetric: ALPHA d/dx1), and the Jacobi
        # diagonal of A = J^T needs the row sums of J^2, not the column sums the stencil kernel forms.  The assembled
        # CSR of J^T is exact on both counts; it exists on one rank only.
        if rt.world > 1:
            raise _lib.GnkError(
                f"cg_least_squares: a transposed Bratu Jacobian (J.T) is not supported with {rt.world} ranks; pass J, "
                "or solve in a single-rank process")
        A = CsrJacobian(rt, A.tocsr(), True)
    if isinstance(A, StencilJacobian):
        d = A.pb.dev
        ycol = d.new_col()
        d.upload_x(y, ycol)
        x = d.new_col()
        x0col = None
        if x0 is not None:  # the initial guess scipy's cg is given (:46,:56); both runs start from it
            x0col = d.new_col()
            d.upload_x(x0, x0col)
        it = _cgls(rt, A.linop(1.0), ycol, cg_rtol, preconditioner, x, d.ld, x0col)
        return d.download_global(x), it
    require_single_rank_unless_sharded(rt, None, "cg_least_squares")
    import scipy.sparse as sp
    op = A if isinstance(A, CsrJacobian) else CsrJacobian(rt, A, isinstance(A, (sp.sparray, sp.spmatrix)))
    y = np.asarray(y, dtype=np.float64).reshape(-1)
    vlen = round_up(max(op.p, op.n_res), 16)
    dy = rt.zeros(vlen)
    rt.upload(y, dy[:op.n_res])
    x = rt.zeros(vlen)
    dx0 = None
    if x0 is not None:
        dx0 = rt.zeros(vlen)
        rt.upload(np.asarray(x0, dtype=np.float64).reshape(-1), dx0[:op.p])
    it = _cgls(rt, op.linop(1.0), dy, cg_rtol, preconditioner, x, vlen, dx0)
    return rt.download(x[:op.p]), it


def gauss_newton(
    res: Callable,
    x0,
    jac: Callable,
    args: Tuple = (),
    tol: float = 1e-8,
    max_iter=100,
    step_length_control: Callable = armijo_goldstein,
    callback: Callable = lambda: None,
    cg_preconditioner: bool = False,
) -> RegressionResult:
    """
    Gauss Newton algorithm for minimizing ||res(theta)|| with respect to theta (reference :63-138).

    res: residual function res(x, *args); x0: initial guess; jac: jac(x, *args) returning ndarray or sparse
    (sparse -> CGLS, dense -> direct least squares: Householder QR on the device for up to 4095 parameters; a dense J
    with fewer rows than columns or an exactly singular R factor raises LinAlgError); step_length_control: plug-in, default Armijo-Goldstein;
    callback(x=, nfev=, cg_iter=) once per iteration.
    """
    rt = get_runtime()
    lib = rt.lib
    x0_host = x0 if is_cuda_tensor(x0) else np.asarray(x0, dtype=np.float64).reshape(-1)
    prob = resolve_problem(res, jac, x0_host, args)
    user_dev = getattr(prob, "user_code", False)  # device callables: x, F and J stay in HBM
    is_bratu = isinstance(prob, BratuDeviceProblem)
    require_single_rank_unless_sharded(rt, prob, "gauss_newton")
    # Several ranks (Bratu only: row slabs, as in gauss_newton_krylow): the CG solve exchanges one halo row per operator
    # application and all-reduces its dot products inside gnk_cgls; out here the step d gets its two halo rows from the
    # neighbours once per iteration, so that J d and the trial points x + s d -- formed on the WHOLE stored column -- are
    # valid on the halo rows without further exchanges, and the k-independent scalars are summed over the ranks.
    dist = is_bratu and prob.distributed
    success = False
    cg_iter = None
    sol = prob.sol_fields
    p, off, ld = sol["n_own"], sol["off"], sol["ld"]

    # entries of a solution vector that x + s d runs over: the owned part, or the stored rows incl. halos when sharded
    ax_n, ax_off = (p + 2 * off, 0) if dist else (p, off)

    def reduce(slot, count, op=0):
        if dist:
            rt.allreduce(scal[slot:slot + count], count, op)

    x = prob.new_sol()
    prob.upload_x(x0_host, x)
    x_trial = prob.new_sol()
    d = prob.new_sol()
    scal = rt.zeros(16)  # [0:2] loss, [2:4] sum (J d)^2, [4] sum x^2, [5] sum d^2
    use_aux = is_bratu and prob.pb.LAMBDA != 0
    aux_cur = prob.new_sol() if use_aux else None
    aux_trial = prob.new_sol() if use_aux else None
    native_armijo = step_length_control is armijo_goldstein

    if is_bratu:
        F, F_trial = prob.new_res(), prob.new_res()
        prob.residual(x, F, scal, aux=aux_cur)
        r_host = None
    elif user_dev:
        r0 = prob.evaluate(x)
        F, F_trial = prob.new_res(), prob.new_res()
        F[:prob.n_res].copy_(r0)
        prob.sumsq(F, scal, prob.res_lay)
        r_host = None
    else:
        r_host = np.asarray(res(x0_host.copy(), *args), dtype=np.float64).reshape(-1)
        prob._ensure_res_layout(r_host.shape[0])
        F, F_trial = prob.new_res(), prob.new_res()
        rt.upload(r_host, F[:prob.n_res])
        prob.sumsq(F, scal, prob.res_lay)
    res_lay, res_fields = prob.res_lay, prob.res_fields
    n_res, res_off, ldr = res_fields["n_own"], res_fields["off"], res_fields["ld"]
    Jd = rt.zeros(ldr)
    nfev = 1
    njev = 0
    prev_loss = float(rt.read(scal, 1)[0])
    dense_qr = not is_bratu and p >= _lib.GNK_DENSE_QR_MIN  # a dense J takes gnk_dense_qr_ls (no CSR form)
    blk = rt.zeros(2 * max(_NB, p + 1) + 8)
    state = {}

    for iter in range(1, max_iter):
        x_host = None
        if is_bratu:
            jac_ev = prob.jacobian(x, aux=aux_cur)
            sparse_like = True
        elif user_dev:
            jac_ev = prob.jacobian(x, dense_panel=dense_qr)
            sparse_like = jac_ev.is_sparse
        else:
            x_host = prob.download_global(x)
            jac_ev = prob.jacobian_host(x_host, dense_panel=dense_qr)
            sparse_like = jac_ev.is_sparse
        njev += 1
        if getattr(jac_ev, "matrix_free", False):
            _refuse_operator("gauss_newton", jac_ev.user)
        panel_qr = dense_qr and not sparse_like
        if panel_qr and not isinstance(jac_ev, DenseJacobian):  # a dense object with a tocsr method of its own
            jac_ev = DenseJacobian(rt, host=jac_ev.host)

        if sparse_like:
            cg_iter = _cgls(rt, jac_ev.linop(-1.0), F, 1e-4, cg_preconditioner, d, ld if is_bratu else
                            round_up(max(p, n_res), 16))
        else:
            # dense J: min ||-J d - r|| by Householder QR (reference: scipy.linalg.lstsq, full-rank case)
            if p > _lib.GNK_DENSE_QR_MAX:
                raise _lib.GnkError(f"dense Jacobians are supported up to {_lib.GNK_DENSE_QR_MAX} columns")
            lda = round_up(max(n_res, 1), 16)
            if panel_qr:
                if n_res < p:
                    raise np.linalg.LinAlgError(
                        f"gauss_newton: the dense Jacobian is rank deficient ({n_res} residuals for {p} parameters); the "
                        "reference's scipy.linalg.lstsq would return the minimum-norm step here, which the device QR "
                        "does not implement")
                # the augmented panel [J | r], column-major; gnk_dense_qr_ls factors it in place
                dA = rt.empty(lda * (p + 1))
                panel = dA.view(p + 1, lda)
                jac_ev.fill_panel(panel)
                panel[p, :n_res].copy_(F[res_off:res_off + n_res])
                _lib.check(lib.gnk_dense_qr_ls(rt.ctx, ptr(dA), lda, n_res, p, -1.0, ptr(blk), rt.stream),
                           "gnk_dense_qr_ls")
            else:
                dA = rt.zeros(lda * p)
                if user_dev:
                    dA.view(p, lda)[:, :n_res].copy_(jac_ev.dense.T)
                else:
                    dense = np.asfortranarray(np.asarray(jac_ev.host, dtype=np.float64))
                    for j in range(p):
                        rt.upload(np.ascontiguousarray(dense[:, j]), dA[j * lda:j * lda + n_res])
                tsqr_solve(rt, dA, lda, n_res, p, F[res_off:], -1.0, blk, householder=True)
            # scipy.linalg.lstsq (:126) is SVD-based and returns the minimum-norm step for a rank-deficient J; the QR here
            # has no such branch, and an exactly singular R would hand inf/NaN to 100 Armijo trials.  Say so instead.
            ls_vals = rt.read(blk, 2 * p + 4)
            if np.any(ls_vals[p + 4:2 * p + 4] == 0.0) or not np.all(np.isfinite(ls_vals[:p])):
                raise np.linalg.LinAlgError(
                    "gauss_newton: the dense Jacobian is rank deficient (a zero on the diagonal of its R factor); the "
                    "reference's scipy.linalg.lstsq would return the minimum-norm step here, which the device QR does "
                    "not implement")
            d[off:off + p].copy_(blk[:p])

        if dist:
            prob.d.halo_exchange(d, 2)

        if native_armijo:
            # g = sum((J d)^2), then trials x + s d  (armijo_goldstein.py:49-62)
            if panel_qr:  # ||J d||^2 = ||R d||^2 from the least-squares block: no J d product
                scal[2:3].copy_(blk[p:p + 1])
            else:
                jac_ev.matmat(d, ld, 1, Jd, ldr) if not is_bratu else prob.d.apply(
                    jac_ev.expu, d, ld, 1, -jac_ev.scale, 0, Jd, ldr, res_off)
                prob.sumsq(Jd, scal[2:4], res_lay) if not is_bratu else _lib.check(
                    lib.gnk_norm_stats(rt.ctx, C.byref(res_lay), ptr(Jd), ptr(scal, 2), rt.stream), "gnk_norm_stats")
                reduce(2, 2, 2)
            _lib.check(lib.gnk_dot(rt.ctx, p, ptr(d, off), ptr(d, off), ptr(scal, 5), rt.stream), "gnk_dot")
            reduce(5, 1)

            def trial_loss(s):
                _lib.check(lib.gnk_axpby(rt.ctx, ax_n, 1.0, ptr(x, ax_off), float(s), ptr(d, ax_off),
                                         ptr(x_trial, ax_off), rt.stream), "gnk_axpby")
                if is_bratu or user_dev:
                    prob.residual(x_trial, F_trial, scal, aux=aux_trial)
                else:
                    state["r_host"] = prob.residual_host(prob.download_global(x_trial), F_trial, scal)
                state["vals"] = rt.read(scal, 8)
                return float(state["vals"][0])

            step_length, nfev_delta = armijo_device(trial_loss, prev_loss, lambda: float(state["vals"][2]),
                                                    lambda: float(np.sqrt(state["vals"][5])))
            squared_sum_d = float(state["vals"][5])
            new_loss = float(state["vals"][0])
            r_host = state.get("r_host")
        else:
            # user plug-in: called with host objects like the reference (:118-120); with device callables, with the
            # objects res and jac take and return (CUDA tensors, the user's Jacobian)
            if user_dev:
                step_length, r_new, nfev_delta = step_length_control(
                    res, prob.x_out(x), F[:n_res].clone(), jac_ev.user, args, prob.x_out(d))
                _require_on_device(rt, r_new, "step_length_control: residual")
                if r_new.numel() != n_res:
                    raise ValueError(f"step_length_control: expected a residual of {n_res} values, got {r_new.numel()}")
                F_trial[:n_res].copy_(r_new.reshape(-1))
            else:
                if x_host is None:
                    x_host = prob.download_global(x)
                if r_host is None:
                    r_host = prob.download_global(F)
                d_host = prob.download_global(d)
                host_J = jac_ev if is_bratu else jac_ev.host
                step_length, r_new, nfev_delta = step_length_control(res, x_host, r_host, host_J, args, d_host)
                r_host = np.asarray(r_new, dtype=np.float64).reshape(-1)
                prob.upload_x(r_host, F_trial) if is_bratu else rt.upload(r_host, F_trial[:n_res])
            _lib.check(lib.gnk_norm_stats(rt.ctx, C.byref(res_lay), ptr(F_trial), ptr(scal), rt.stream), "gnk_norm_stats")
            reduce(0, 2, 2)
            _lib.check(lib.gnk_dot(rt.ctx, p, ptr(d, off), ptr(d, off), ptr(scal, 5), rt.stream), "gnk_dot")
            reduce(5, 1)
            _lib.check(lib.gnk_axpby(rt.ctx, ax_n, 1.0, ptr(x, ax_off), float(step_length), ptr(d, ax_off),
                                     ptr(x_trial, ax_off), rt.stream), "gnk_axpby")
            v = rt.read(scal, 8)
            squared_sum_d = float(v[5])
            new_loss = float(v[0])
            if use_aux:  # e^x at the accepted point for the next Jacobian
                prob.residual(x_trial, F_trial, scal, aux=aux_trial)
        nfev += nfev_delta

        _lib.check(lib.gnk_dot(rt.ctx, p, ptr(x, off), ptr(x, off), ptr(scal, 4), rt.stream), "gnk_dot")
        reduce(4, 1)
        squared_sum_x_prev = float(rt.read(scal, 8)[4])

        # x += s d  (the accepted trial point is exactly that)
        x, x_trial = x_trial, x
        F, F_trial = F_trial, F
        aux_cur, aux_trial = aux_trial, aux_cur
        prev_loss = new_loss

        if user_dev:
            callback(x=prob.x_out(x), nfev=nfev, cg_iter=cg_iter)
        else:
            xv = DeviceVector(prob, x, prob.p_glob)
            callback(x=xv, nfev=nfev, cg_iter=cg_iter)
            xref = weakref.ref(xv)
            del xv
            DeviceVector.settle(xref)  # a callback that kept x gets its host snapshot before the buffer is reused

        if step_length**2 * squared_sum_d <= tol**2 * squared_sum_x_prev:
            success = True
            break

    if not success:
        print("Warning: The gauss_newton algorithm reached maximal iteration bound before terminating!")

    return RegressionResult("gauss newton", prob.x_out(x) if user_dev else prob.download_global(x), success, nfev,
                            njev, iter)
