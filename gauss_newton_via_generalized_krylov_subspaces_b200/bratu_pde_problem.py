"""Bratu PDE problem -- call-compatible mirror of the reference's ``bratu_pde_problem.py``.

    -Lap(u) + ALPHA du/dx1 + LAMBDA e^u = f   on [lb, ub]^2, zero Dirichlet, 5-point Laplacian,
    forward difference in x1 (the slow index), h = (ub-lb)/grid_nodes   (bratu_pde_problem.py:20-74)

``make_res`` / ``make_jac`` / ``make_error`` return callables that (a) accept and return host ndarrays
exactly like the reference's lambdas (:85-99) -- computed by the CUDA stencil kernels -- and (b) carry a
device implementation that ``gauss_newton_krylow`` / ``gauss_newton`` recognise, in which case the
vectors never leave HBM.  Nothing is assembled: J(u) = -(L + ALPHA D + LAMBDA diag(e^u)) is the three
stencil constants plus the n-vector e^u (:88-96).  The scipy matrices ``laplace1d``, ``laplace2d``,
``partial_diff_x`` that the reference exposes (used by bratu_pde_test.py:211-219) are built lazily on
first access, only for callers that want them.
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, Optional

import numpy as np

from . import _lib
from .device import DeviceVector, NodeSharedBuffers, SharedBuffersUnavailable, get_runtime, make_layout, ptr
from .partition import HALO, all_counts, stencil_layout_fields


def default_u(x1, x2):
    return np.exp(-10 * (x1**2 + x2**2))


class BratuPdeProblem:
    """Notice that n = p = (grid_nodes-1)**2."""

    grid_nodes: int

    def __init__(self, grid_nodes: int, ALPHA: float, LAMBDA: float, lower_bound: float = -3.0,
                 upper_bound: float = 3.0, grid_resolution: Optional[float] = None,
                 u: Callable = default_u):
        self.grid_nodes = grid_nodes
        self.ALPHA = ALPHA
        self.LAMBDA = LAMBDA
        self.lower_bound = lower_bound
        self.upper_bound = upper_bound
        if grid_resolution is None:
            self.grid_resolution = (upper_bound - lower_bound) / grid_nodes
        else:
            self.grid_resolution = grid_resolution
        self.u = u
        self.m = grid_nodes - 1
        self.n = self.m * self.m
        self._cache = {}
        self._dev = None

    # ---- host-side attributes of the reference, built on demand ----------------------------------
    def _lazy(self, key, build):
        if key not in self._cache:
            self._cache[key] = build()
        return self._cache[key]

    @property
    def laplace1d(self):
        import scipy.sparse as sp
        g = self.grid_nodes
        return self._lazy("laplace1d", lambda: sp.diags_array(
            (-np.ones(g - 2), 2 * np.ones(g - 1), -np.ones(g - 2)), offsets=(-1, 0, 1)))

    @property
    def laplace2d(self):
        import scipy.sparse as sp

        def build():
            eye = sp.eye(self.m)
            return (sp.kron(self.laplace1d, eye) + sp.kron(eye, self.laplace1d)) * self.grid_resolution**-2
        return self._lazy("laplace2d", build)

    @property
    def partial_diff_x(self):
        import scipy.sparse as sp

        def build():
            g = self.grid_nodes
            d1 = sp.diags_array((-np.ones(g - 1), np.ones(g - 2)), offsets=(0, 1))
            return sp.kron(d1, sp.eye(self.m)) * self.grid_resolution**-1
        return self._lazy("partial_diff_x", build)

    @property
    def grid(self):
        t = np.linspace(self.lower_bound, self.upper_bound, self.grid_nodes + 1)[1:-1]
        return self._lazy("grid", lambda: np.meshgrid(t, t))

    @property
    def u_true(self):
        return self._lazy("u_true", lambda: self.u(*self.grid).flatten("F"))

    # ---- device side ------------------------------------------------------------------------------
    @property
    def dev(self) -> "BratuDevice":
        if self._dev is None:
            self._dev = BratuDevice(self)
        return self._dev

    def pde_operator(self, u):
        """P(u) = L u + ALPHA D u + LAMBDA e^u (bratu_pde_problem.py:76-83), evaluated by the stencil kernel."""
        d = self.dev
        x = d.new_col()
        d.upload_x(u, x)
        F = d.new_col()
        d.residual_into(x, d.zero_col(), F, None, d.scal_tmp, depth=0)
        return np.negative(d.download_global(F))  # a private array (with several ranks the download is a shared view)

    def make_res(self, y):
        return BratuResidual(self, y)

    def make_jac(self):
        return BratuJacobianFactory(self)

    def make_error(self):
        return BratuError(self)


class BratuDevice:
    """Device state of one BratuPdeProblem on this rank: slab layout, stencil constants, buffers."""

    def __init__(self, pb: BratuPdeProblem):
        rt = get_runtime()
        self.rt = rt
        self.pb = pb
        self.fields = stencil_layout_fields(pb.m, rt.world, rt.rank)
        self.lay = make_layout(self.fields)
        # the same host-computed constants as the reference: h**-2, ALPHA * h**-1 (:58,:67,:81)
        self.prm = _lib.Bratu(pb.grid_resolution**-2, pb.ALPHA * pb.grid_resolution**-1, float(pb.LAMBDA))
        self.ld = self.fields["ld"]
        self.counts = all_counts(pb.m, rt.world)
        self.scal_tmp = rt.zeros(8)
        self._zero = None
        self._host_stage = None
        self._shared = None

    def new_col(self):
        return self.rt.zeros(self.ld)

    def zero_col(self):
        if self._zero is None:
            self._zero = self.rt.zeros(self.ld)
        return self._zero

    def scratch_col(self):
        """a stored column whose contents nobody relies on (halo rows stay zero: only owned rows are written)"""
        if self._host_stage is None:
            self._host_stage = self.rt.zeros(self.ld)
        return self._host_stage

    def upload_x(self, x_global, out):
        """global host vector -> stored column (owned rows + the 2 halo rows each side)."""
        x_global = np.asarray(x_global, dtype=np.float64).reshape(-1)
        if x_global.shape[0] != self.pb.n:
            raise ValueError(f"expected a vector of length {self.pb.n}, got {x_global.shape[0]}")
        f = self.fields
        if self.rt.world == 1:
            self.rt.upload(x_global, out[f["off"]:f["off"] + f["n_own"]])
        else:
            # the rows [i0 - HALO, i1 + HALO) that lie inside the domain are ONE contiguous piece of the caller's
            # vector: it goes to the device straight from the caller's buffer (asynchronous DMA when that is pinned),
            # no pageable staging copy; halo rows outside the domain are the Dirichlet zeros
            lo, hi, dst0 = self._h2d_range()
            out[:dst0].zero_()
            out[dst0 + (hi - lo) * f["m"]:].zero_()
            self.rt.upload(x_global[lo * f["m"]:hi * f["m"]], out[dst0:dst0 + (hi - lo) * f["m"]])

    def _h2d_range(self):
        f = self.fields
        lo = max(f["i0"] - HALO, 0)
        hi = min(f["i1"] + HALO, self.pb.m)
        return lo, hi, (lo - (f["i0"] - HALO)) * f["m"]

    def h2d_doubles_per_vector(self):
        """doubles that upload_x moves host -> device on this rank (bench.py: e2e.h2d_bytes_per_step)"""
        if self.rt.world == 1:
            return self.fields["n_own"]
        lo, hi, _ = self._h2d_range()
        return (hi - lo) * self.fields["m"]

    def d2h_doubles_per_vector(self):
        """doubles that download_global moves device -> host on this rank: its own slab (the whole vector on the
        fallback path without node-shared buffers)"""
        return self.pb.n if self._shared is False else self.fields["n_own"]

    def resident(self, x_global):
        """upload a global host vector once; the returned DeviceVector can be passed to the solvers as x0"""
        col = self.new_col()
        self.upload_x(x_global, col)
        return DeviceVector(self, col, self.pb.n)

    def download_global(self, col):
        f = self.fields
        rt = self.rt
        if rt.world == 1:
            return rt.download(col[f["off"]:f["off"] + f["n_own"]])
        # Every rank copies only ITS slab device -> host, into a host buffer that all ranks of the node map
        # (device.NodeSharedBuffers); after the closing collective each rank holds the whole vector as an ndarray over
        # that buffer.  (Round 1 all-gathered the full vector onto every GPU and copied it N times.)
        if self._shared is None:
            self._shared = NodeSharedBuffers(rt, self.pb.n)
        if self._shared is not False:
            try:
                host, finish = self._shared.acquire()
            except SharedBuffersUnavailable:   # all ranks together (the failure is broadcast): /dev/shm is too small
                self._shared = False
            else:
                start = sum(self.counts[:rt.rank])
                host[start:start + f["n_own"]].copy_(col[f["off"]:f["off"] + f["n_own"]], non_blocking=True)
                return finish()
        return rt.download(self.allgather_device(col))   # fallback: all-gather on the devices, full copy per rank

    def allgather_device(self, col):
        """the global vector on EVERY rank's GPU (owned parts all-gathered over NVLink) -- for device-side consumers"""
        rt = self.rt
        full = rt.empty(self.pb.n)
        counts = (C.c_int64 * rt.world)(*self.counts)
        _lib.check(rt.lib.gnk_comm_allgather_owned(rt.ctx, C.byref(self.lay), ptr(col), ptr(full), counts, rt.stream),
                   "gnk_comm_allgather_owned")
        return full

    def residual_into(self, x, y, F, expu, loss_slot, depth=1):
        rt = self.rt
        _lib.check(rt.lib.gnk_bratu_residual(rt.ctx, C.byref(self.lay), C.byref(self.prm), ptr(x), ptr(y), ptr(F),
                                             ptr(expu), depth, ptr(loss_slot), rt.stream), "gnk_bratu_residual")
        if not rt.fused_reductions:  # else the kernel's last CTA has already summed over the ranks (peer mailboxes)
            rt.allreduce(loss_slot, 1, 0)

    def apply(self, expu, inp, in_ld, k, sign, transpose, out, out_ld, out_off):
        rt = self.rt
        _lib.check(rt.lib.gnk_stencil_apply(rt.ctx, C.byref(self.lay), C.byref(self.prm), ptr(expu), ptr(inp), in_ld, k,
                                            sign, transpose, ptr(out), out_ld, out_off, rt.stream), "gnk_stencil_apply")

    def halo_exchange(self, col, depth, offset=0):
        rt = self.rt
        if rt.world > 1:
            _lib.check(rt.lib.gnk_comm_halo_exchange(rt.ctx, C.byref(self.lay), ptr(col, offset), depth, rt.stream),
                       "gnk_comm_halo_exchange")


class StencilJacobian:
    """J(u) = -(L + ALPHA D + LAMBDA diag(e^u)) held as e^u on the device (None when LAMBDA == 0).

    Supports what the reference does with the scipy matrix it returns: ``J @ v``, ``J.T @ v``, ``-1 * J``,
    ``.shape`` -- all evaluated by the stencil kernel -- plus ``tocsr()`` for callers that really want
    the assembled matrix."""

    _gnk_sparse_like = True

    def __init__(self, pb, expu, transposed=False, scale=1.0):
        self.pb = pb
        self.expu = expu
        self.transposed = transposed
        self.scale = scale
        self.shape = (pb.n, pb.n)

    @property
    def T(self):
        return StencilJacobian(self.pb, self.expu, not self.transposed, self.scale)

    def __rmul__(self, s):
        return StencilJacobian(self.pb, self.expu, self.transposed, self.scale * s)

    __mul__ = __rmul__

    def __neg__(self):
        return self.__rmul__(-1.0)

    def __matmul__(self, v):
        d = self.pb.dev
        if isinstance(v, DeviceVector):
            v = v.materialize()
        v = np.asarray(v, dtype=np.float64)
        cols = v.reshape(self.pb.n, -1)
        outs = []
        x = d.new_col()
        o = d.new_col()
        for j in range(cols.shape[1]):
            d.upload_x(np.ascontiguousarray(cols[:, j]), x)
            d.apply(self.expu, x, d.ld, 1, -self.scale, int(self.transposed), o, d.ld, d.fields["off"])
            outs.append(d.download_global(o))
        return outs[0] if v.ndim == 1 else np.stack(outs, axis=1)

    # device-native protocol used by the solvers
    def matmat(self, V, ldv, k, JV, ldjv):
        self.pb.dev.apply(self.expu, V, ldv, k, -self.scale, int(self.transposed), JV, ldjv, 0)

    def neg_rmatvec(self, r, w):
        d = self.pb.dev
        d.apply(self.expu, r, d.ld, 1, self.scale, int(not self.transposed), w, d.ld, d.fields["off"])

    def linop(self, sign):
        # gnk_linop carries no transpose flag and gnk_stencil_normal_diag gives diag(J^T J) only: a transposed operator
        # would be solved as J.  Callers route J.T through CsrJacobian(rt, J.T.tocsr(), True) instead
        if self.transposed:
            raise _lib.GnkError("StencilJacobian.linop: the device CG operator cannot represent J.T; assemble it "
                                "(CsrJacobian of .tocsr())")
        d = self.pb.dev
        op = _lib.LinOp()
        op.kind = 0
        op.sign = -self.scale * sign
        op.lay = d.lay
        op.prm = d.prm
        op.d_expu = ptr(self.expu)
        return op

    def tocsr(self):
        import scipy.sparse as sp
        pb = self.pb
        J = pb.laplace2d + pb.ALPHA * pb.partial_diff_x
        if self.expu is not None:
            J = J + pb.LAMBDA * sp.diags(pb.dev.download_global(self.expu))
        J = sp.csr_array(-self.scale * J)
        return sp.csr_array(J.T) if self.transposed else J


class BratuResidual:
    """``res`` of the reference: u -> y - pde_operator(u)   (bratu_pde_problem.py:85-86)."""

    def __init__(self, pb: BratuPdeProblem, y):
        self.pb = pb
        self.y_host = np.asarray(y, dtype=np.float64).reshape(-1)
        self._y = None

    @property
    def y_col(self):
        if self._y is None:
            d = self.pb.dev
            self._y = d.new_col()
            d.upload_x(self.y_host, self._y)
        return self._y

    def __call__(self, u, *args):
        d = self.pb.dev
        x = d.new_col()
        d.upload_x(u.materialize() if isinstance(u, DeviceVector) else u, x)
        F = d.new_col()
        d.residual_into(x, self.y_col, F, None, d.scal_tmp, depth=0)
        return d.download_global(F)

    def loss(self, u):
        """0.5 * sum(res(u)**2) (benchmark.py:32-33) without moving the residual to the host; a DeviceVector that is
        still in HBM (the ``x`` handed to a solver callback) is used in place, nothing crosses PCIe but one scalar."""
        d = self.pb.dev
        if isinstance(u, DeviceVector) and u._t is not None and u._t.numel() == d.ld \
                and d in (u._owner, getattr(u._owner, "d", None)):
            x = u._t
        else:
            x = d.new_col()
            d.upload_x(u.materialize() if isinstance(u, DeviceVector) else u, x)
        d.residual_into(x, self.y_col, d.scratch_col(), None, d.scal_tmp, depth=0)
        return 0.5 * float(d.rt.read(d.scal_tmp, 1)[0])


class BratuJacobianFactory:
    """``jac`` of the reference: u -> -(L + ALPHA D + LAMBDA diag(e^u))   (bratu_pde_problem.py:88-96)."""

    def __init__(self, pb: BratuPdeProblem):
        self.pb = pb

    def __call__(self, u, *args):
        pb = self.pb
        if pb.LAMBDA == 0:
            return StencilJacobian(pb, None)
        d = pb.dev
        x = d.new_col()
        d.upload_x(u.materialize() if isinstance(u, DeviceVector) else u, x)
        expu = d.new_col()
        d.residual_into(x, d.zero_col(), d.new_col(), expu, d.scal_tmp, depth=0)
        return StencilJacobian(pb, expu)


class BratuError:
    """``error`` of the reference: u -> ||u_true - u||_2   (bratu_pde_problem.py:98-99).  For a DeviceVector that is
    still in HBM the difference and the norm are formed on the device (SURVEY 8f: the benchmark harness calls this
    once per callback; at 4096^2 the host path would move 134 MB per call)."""

    def __init__(self, pb):
        self.pb = pb
        self._ut = None

    def __call__(self, u):
        d = self.pb._dev
        if isinstance(u, DeviceVector) and u._t is not None and d is not None and u._t.numel() == d.ld:
            rt = d.rt
            if self._ut is None:
                self._ut = d.new_col()
                d.upload_x(self.pb.u_true, self._ut)
            f = d.fields
            diff = d.scratch_col()
            _lib.check(rt.lib.gnk_axpby(rt.ctx, f["n_own"], 1.0, ptr(self._ut, f["off"]), -1.0, ptr(u._t, f["off"]),
                                        ptr(diff, f["off"]), rt.stream), "gnk_axpby")
            _lib.check(rt.lib.gnk_norm_stats(rt.ctx, C.byref(d.lay), ptr(diff), ptr(d.scal_tmp), rt.stream),
                       "gnk_norm_stats")
            rt.allreduce(d.scal_tmp, 1, 0)
            return float(np.sqrt(rt.read(d.scal_tmp, 1)[0]))
        if isinstance(u, DeviceVector):
            u = u.materialize()
        return np.linalg.norm(self.pb.u_true - u)


class BratuDeviceProblem:
    """Problem adapter used by the solvers when ``res`` and ``jac`` both come from one BratuPdeProblem:
    vectors stay in HBM in the slab layout, the Jacobian is e^u, everything is one kernel call."""

    def __init__(self, res: BratuResidual, jac: BratuJacobianFactory):
        self.pb = res.pb
        self.d = self.pb.dev
        self.rt = self.d.rt
        self.res = res
        self.p_glob = self.pb.n
        self.sol_fields = self.res_fields = self.d.fields
        self.sol = self.res_lay = self.d.lay
        self.n_res = self.d.fields["n_own"]
        self.distributed = self.rt.world > 1

    @staticmethod
    def match(res, jac):
        return isinstance(res, BratuResidual) and isinstance(jac, BratuJacobianFactory) and res.pb is jac.pb

    def new_sol(self):
        return self.d.new_col()

    new_res = new_sol

    def upload_x(self, x_host, out):
        self.d.upload_x(x_host, out)

    def download_global(self, t):
        return self.d.download_global(t)

    def residual(self, x, F, loss_slot, aux=None):
        """F = res(x) on owned rows + 1 halo row each side; aux (optional) receives e^x."""
        self.d.residual_into(x, self.res.y_col, F, aux if self.pb.LAMBDA != 0 else None, loss_slot, depth=1)

    def jacobian(self, x, aux=None):
        """J(x).  aux = e^x if a residual evaluation at the same x already produced it."""
        if self.pb.LAMBDA == 0:
            return StencilJacobian(self.pb, None)
        if aux is None:
            aux = self.d.new_col()
            self.d.residual_into(x, self.d.zero_col(), self.d.new_col(), aux, self.d.scal_tmp, depth=0)
        return StencilJacobian(self.pb, aux)
