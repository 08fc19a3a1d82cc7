"""Generalized Krylov subspace state -- mirror of the reference's ``krylow.py`` on the device.

The orthonormal basis V_k lives in HBM as a pre-allocated block of ``capacity`` stored columns (column j
is one contiguous slab-layout vector), so appending a column writes n doubles instead of copying the
whole basis (the reference's ``np.hstack``, krylow.py:73).  Public methods keep the reference's
signatures and host-ndarray semantics (``start``, ``x``, ``evaluate``, ``update``, ``basis``); the
solvers use the ``dev_*`` methods, which never leave the device.
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np

from . import _lib
from .device import CsrJacobian, HostCallableProblem, get_runtime, make_layout, ptr
from .partition import flat_layout_fields

MAX_COLUMNS = _lib.GNK_MAX_BASIS - 1  # the TSQR panel carries one extra right-hand-side column


class GeneralizedKrylowSubspaceBreakdown(Exception):
    pass


class GeneralizedKrylowSubspaceSpansEntireSpace(Exception):
    pass


class _FlatOwner:
    """download helper for the stand-alone (flat layout) use of the class"""

    def __init__(self, rt, n):
        self.rt, self.n = rt, n

    def download_global(self, t):
        return self.rt.download(t[:self.n])


class GeneralizedKrylowSubspace:
    """
    Attributes
    ----------
    basis: The basis of the generalized Krylov subspace as an (n, k) host ndarray (downloaded on access).
    """

    def __init__(self, problem=None, capacity=None, reorth_passes=1):
        self.problem = problem
        self.capacity = capacity
        self.reorth_passes = int(reorth_passes)
        self.k = 0
        self.V = None
        self._ready = False

    # ---------------------------------------------------------------------------------------------
    def _setup(self, n_glob, fields, lay, owner, capacity):
        rt = get_runtime()
        self.rt = rt
        self.n_glob = int(n_glob)
        self.fields, self.lay, self.owner = fields, lay, owner
        self.ld = fields["ld"]
        cap = min(self.n_glob, capacity if capacity is not None else 32)
        self.cap = max(1, min(cap, MAX_COLUMNS))
        # no zero-fill of the basis storage (4 GB at 4096^2, k <= 30: 0.7 ms per solve): every column is written in full
        # -- owned rows and halo rows -- by the normalisation kernel before anything reads it, and columns >= k are
        # never part of any arithmetic (the fused least-squares kernel gives its padding lanes weight 0 on finite data)
        self.V = rt.empty(self.cap * self.ld)
        self.w = rt.zeros(self.ld)          # its halo rows stay zero: they become the new column's Dirichlet rows
        self.h = rt.zeros(_lib.GNK_MAX_BASIS)
        self.stats = rt.zeros(2)
        self.flag = rt.zeros(1, dtype=rt.torch.int32)
        self._ready = True

    def _grow(self):
        if self.cap >= MAX_COLUMNS:
            raise _lib.GnkError(f"Krylov basis wider than {MAX_COLUMNS} columns is not supported; pass krylow_restart")
        new_cap = min(MAX_COLUMNS, max(self.cap * 2, 2), self.n_glob)
        V = self.rt.empty(new_cap * self.ld)
        V[:self.k * self.ld].copy_(self.V[:self.k * self.ld])
        self.V, self.cap = V, new_cap

    def col(self, j):
        return self.V[j * self.ld:(j + 1) * self.ld]

    # ---- device-native operations -----------------------------------------------------------------
    def dev_start(self, x):
        """V = [x/||x||], returns ||x||   (krylow.py:30-39).  x: stored column with valid halos."""
        rt, lib = self.rt, self.rt.lib
        _lib.check(lib.gnk_norm_stats(rt.ctx, C.byref(self.lay), ptr(x), ptr(self.stats), rt.stream), "gnk_norm_stats")
        rt.allreduce(self.stats, 2, 2)
        _lib.check(lib.gnk_normalize(rt.ctx, C.byref(self.lay), ptr(x), ptr(self.stats), 1e-8, ptr(self.V),
                                     ptr(self.flag), rt.stream), "gnk_normalize")
        ss = rt.read(self.stats, 2)
        if ss[1] <= 1e-8:
            raise ValueError("x0 is not allowed to be 0 in the gauss_newton_krylow algorithm")
        self.k = 1
        return math.sqrt(ss[0])

    def dev_combine(self, c, d, s, out, c_out=None, cprev2=None):
        """out = V_k (c + s d) over the whole stored column (krylow.py:41-42); optionally the coordinates c + s d (with
        the next column's zero entry appended) and sum(c^2) are left on the device (gnk_combine_step)."""
        rt = self.rt
        with rt.mark("combine", 8.0 * self.fields["n_own"] * (self.k + 1)):
            _lib.check(rt.lib.gnk_combine_step(rt.ctx, C.byref(self.lay), ptr(self.V), self.k, ptr(c), ptr(d), float(s),
                                               ptr(out), ptr(c_out), cprev2 if cprev2 is not None else ptr(None),
                                               rt.stream), "gnk_combine")

    def dev_rmatvec(self, jac_op, r):
        """w = -J^T r alone, for a following expansion called with ``jac_op=None``"""
        with self.rt.mark("spmv_t", 24.0 * self.fields["n_own"]):
            jac_op.neg_rmatvec(r, self.w)

    def dev_expand_enqueue(self, jac_op, r, halo_exchange=None, flag_ptr=None):
        """Enqueue the basis expansion with -J^T r orthogonalised against V_k (krylow.py:55-73) WITHOUT committing it:
        the normalised vector lands in column k of the storage, the breakdown flag of krylow.py:66 in ``flag_ptr`` (a
        device int32; default: this object's own flag), and ``k`` is unchanged until ``commit()``.  Nothing is read
        back, so the caller may enqueue it speculatively (gauss_newton_krylow does, before it knows whether the Armijo
        trial is accepted) -- an expansion that is not committed leaves no trace: w, h, the statistics, column k and the
        flag are all overwritten by the next one.  ``jac_op=None``: w already holds -J^T r (``dev_rmatvec``)."""
        if self.k == self.n_glob:
            raise GeneralizedKrylowSubspaceSpansEntireSpace
        rt, lib = self.rt, self.rt.lib
        if self.k == self.cap:
            self._grow()
        n = self.fields["n_own"]
        if jac_op is not None:
            self.dev_rmatvec(jac_op, r)
        for ipass in range(self.reorth_passes):
            with rt.mark("cgs_dots", 8.0 * n * (self.k + 1)):
                _lib.check(lib.gnk_cgs_dots(rt.ctx, C.byref(self.lay), ptr(self.V), self.k, ptr(self.w),
                                            ptr(self.h), rt.stream), "gnk_cgs_dots")
            if not rt.fused_reductions:  # else summed over the ranks inside the kernel (peer mailboxes)
                rt.allreduce(self.h, self.k, 0)
            with rt.mark("cgs_update", 8.0 * n * (self.k + 2)):
                _lib.check(lib.gnk_cgs_update(rt.ctx, C.byref(self.lay), ptr(self.V), self.k, ptr(self.h),
                                              ptr(self.w), ptr(self.stats), rt.stream), "gnk_cgs_update")
        if not rt.fused_reductions:
            rt.allreduce(self.stats, 2, 2)
        new = self.col(self.k)
        fp = ptr(self.flag) if flag_ptr is None else flag_ptr
        with rt.mark("normalize", 16.0 * n):
            if halo_exchange is not None:
                # the one halo exchange of an outer iteration rides in the normalisation kernel (border threads push
                # into the neighbours' mailboxes, 32 CTAs receive).  A breakdown leaves column k unwritten on every rank
                # alike: it is decided from the all-reduced statistics, so nobody pushes and nobody waits
                _lib.check(lib.gnk_normalize_halo(rt.ctx, C.byref(self.lay), ptr(self.w), ptr(self.stats), 1e-8,
                                                  ptr(new), fp, rt.stream), "gnk_normalize_halo")
            else:
                _lib.check(lib.gnk_normalize(rt.ctx, C.byref(self.lay), ptr(self.w), ptr(self.stats), 1e-8, ptr(new),
                                             fp, rt.stream), "gnk_normalize")

    def commit(self):
        """make the column written by the last ``dev_expand_enqueue`` part of the basis"""
        self.k += 1

    def dev_update(self, jac_op, r, halo_exchange=None, deferred_flag=None):
        """Expand the basis with -J^T r orthogonalised against V_k (krylow.py:55-73).  Raises the same
        exceptions as the reference; on Breakdown the basis is left unchanged.
        ``deferred_flag`` (a device pointer to an int32): the breakdown flag of krylow.py:66 is written there and NOT
        read back; the column is appended speculatively and the caller inspects the flag with its next read-back
        (one host synchronisation less per outer iteration) and calls ``retract()`` if it was set."""
        self.dev_expand_enqueue(jac_op, r, halo_exchange, deferred_flag)
        if deferred_flag is None and int(self.rt.read_i32(self.flag)[0]) != 0:
            raise GeneralizedKrylowSubspaceBreakdown(
                "Normal residual is allready inside generalized Krylow Subspcae, there for gauss newton krylow "
                "algorithm has to proceed without enlarging the subspace.")
        self.commit()

    def retract(self):
        """undo a speculative append whose deferred breakdown flag turned out to be set (the column was not written)"""
        self.k -= 1

    # ---- the reference's public interface (host ndarrays) -------------------------------------------
    @property
    def basis(self):
        cols = [self.owner.download_global(self.col(j)) for j in range(self.k)]
        return np.stack(cols, axis=1)

    def start(self, x0):
        x0 = np.asarray(x0, dtype=np.float64).reshape(-1)
        if self.problem is not None:
            pb = self.problem
            self._setup(pb.p_glob, pb.sol_fields, pb.sol, pb, self.capacity)
            x = pb.new_sol()
            pb.upload_x(x0, x)
        else:
            rt = get_runtime()
            from .gauss_newton_krylow import require_single_rank_unless_sharded
            require_single_rank_unless_sharded(rt, None, "GeneralizedKrylowSubspace.start")
            f = flat_layout_fields(x0.shape[0])
            self._setup(x0.shape[0], f, make_layout(f), _FlatOwner(rt, x0.shape[0]), self.capacity)
            x = rt.zeros(self.ld)
            rt.upload(x0, x[:x0.shape[0]])
        return np.array([self.dev_start(x)])

    def x(self, x_coordinate):
        rt = self.rt
        c = rt.zeros(_lib.GNK_MAX_BASIS)
        rt.upload(np.asarray(x_coordinate, dtype=np.float64), c[:self.k])
        out = rt.zeros(self.ld)
        self.dev_combine(c, None, 0.0, out)
        return self.owner.download_global(out)

    def evaluate(self, function, x_coordinate, *args):
        """For evaluating functions such as res or jac on the generalized krylow subspace."""
        return function(self.x(x_coordinate), *args)

    def update(self, jac_ev, res_ev):
        rt = self.rt
        if hasattr(jac_ev, "neg_rmatvec"):
            op = jac_ev
            r = self.problem.new_res()
            self.problem.upload_x(np.asarray(res_ev, dtype=np.float64), r)
            if getattr(self.problem, "distributed", False):
                self.problem.d.halo_exchange(r, 1)
            hx = self.problem.d.halo_exchange if getattr(self.problem, "distributed", False) else None
        else:
            import scipy.sparse as sp
            op = CsrJacobian(rt, jac_ev, isinstance(jac_ev, (sp.sparray, sp.spmatrix)))
            res_ev = np.asarray(res_ev, dtype=np.float64).reshape(-1)
            r = rt.zeros(flat_layout_fields(res_ev.shape[0])["ld"])
            rt.upload(res_ev, r[:res_ev.shape[0]])
            hx = None
        self.dev_update(op, r, hx)
