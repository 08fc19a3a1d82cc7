"""Device runtime of the host mirror: one process per GPU, torch for device memory / streams /
torch.distributed plumbing, every arithmetic step in libgnk_b200.so (no CPU fallback).
"""
from __future__ import annotations

import atexit
import ctypes as C
import mmap
import os
import sys
import time
import weakref

import numpy as np

from . import _lib
from .partition import flat_layout_fields

_runtime = None


class Runtime:
    fused_reductions = False
    def __init__(self):
        import torch

        if not torch.cuda.is_available():
            raise _lib.GnkError("no CUDA device visible: this package runs its solvers on a B200 only "
                                "(there is no CPU fallback)")
        self.torch = torch
        self.lib = _lib.load()
        ndev = torch.cuda.device_count()
        self.device_index = int(os.environ.get("LOCAL_RANK", "0")) % max(ndev, 1)
        torch.cuda.set_device(self.device_index)
        self.device = torch.device("cuda", self.device_index)
        ctx = C.c_void_p()
        _lib.check(self.lib.gnk_create(C.byref(ctx), self.device_index), "gnk_create")
        self.ctx = ctx
        self.rank, self.world = 0, 1
        self.fused_reductions = False  # gnk_bratu_residual / gnk_cgs_dots / gnk_cgs_update reduce over the ranks themselves
        # the largest read: the 2p + 4 result block of gnk_dense_qr_ls at p = GNK_DENSE_QR_MAX
        self._pinned = torch.empty(2 * (_lib.GNK_DENSE_QR_MAX + 1) + 8, dtype=torch.float64, pin_memory=True)
        self._pinned_np = self._pinned.numpy()
        self._pinned_ptr = self._pinned.data_ptr()
        self._pinned2 = torch.empty(1024, dtype=torch.float64, pin_memory=True)
        self._pinned2_np = self._pinned2.numpy()
        self._pinned2_ptr = self._pinned2.data_ptr()
        self._pinned_i = torch.empty(16, dtype=torch.int32, pin_memory=True)
        self._raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)
        self._attach_comm_if_distributed()

    # -- multi-GPU ---------------------------------------------------------------------------------
    def _attach_comm_if_distributed(self):
        dist = self.torch.distributed
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
            return
        self.rank, self.world = dist.get_rank(), dist.get_world_size()
        buf = (C.c_char * 128)()
        if self.rank == 0:
            _lib.check(self.lib.gnk_comm_unique_id(buf), "gnk_comm_unique_id")
        box = [bytes(buf)]
        dist.broadcast_object_list(box, src=0)
        idbuf = (C.c_char * 128).from_buffer_copy(box[0])
        _lib.check(self.lib.gnk_comm_init(self.ctx, idbuf, self.rank, self.world), "gnk_comm_init")
        self._attach_peer_mailboxes(dist)

    def _attach_peer_mailboxes(self, dist):
        """One-node runs: map every rank's mailbox with CUDA IPC so that the small all-gathers and the halo rows go
        over NVLink as plain stores from single kernels (comm.cu).  Any failure leaves the NCCL path in use; all
        ranks take the same decision.  GNK_P2P=0 disables it."""
        lib = self.lib
        if os.environ.get("GNK_P2P", "1") == "0" or not hasattr(lib, "gnk_comm_p2p_export") or self.world > 16:
            return
        h = (C.c_char * 64)()
        rc = lib.gnk_comm_p2p_export(self.ctx, h)
        box = [None] * self.world
        dist.all_gather_object(box, (int(rc), bytes(h)))
        if any(r != 0 for r, _ in box):
            return
        allh = (C.c_char * (64 * self.world)).from_buffer_copy(b"".join(b for _, b in box))
        rc = lib.gnk_comm_p2p_attach(self.ctx, allh)
        ok = [None] * self.world
        dist.all_gather_object(ok, int(rc))
        if any(r != 0 for r in ok):  # e.g. no peer access between some pair of devices: everybody stays on NCCL
            lib.gnk_comm_p2p_disable(self.ctx)
        self.fused_reductions = bool(lib.gnk_comm_fused_reductions(self.ctx))

    # -- helpers -----------------------------------------------------------------------------------
    @property
    def stream(self):
        """torch's current stream on this device as a cudaStream_t (a plain int: every prototype declares c_void_p).
        Asked for at every launch, so it goes through the raw-handle query (0.2 us) rather than
        torch.cuda.current_stream() (3-4 us: a third of the host time per outer iteration in the launch-latency regime)."""
        raw = self._raw_stream
        if raw is not None:
            return raw(self.device_index)
        return self.torch.cuda.current_stream().cuda_stream

    def zeros(self, n, dtype=None):
        return self.torch.zeros(int(n), dtype=dtype or self.torch.float64, device=self.device)

    def empty(self, n, dtype=None):
        return self.torch.empty(int(n), dtype=dtype or self.torch.float64, device=self.device)

    def sync(self):
        self.torch.cuda.current_stream().synchronize()

    # -- optional per-kernel timing (bench.py roofline): CUDA events on the launching stream ---------
    prof = None

    def begin_profile(self):
        self.prof = {}

    def end_profile(self):
        """-> {name: dict(launches, ms, bytes)}; algorithmic bytes as stated in DESIGN.md"""
        self.sync()
        out = {}
        for name, recs in (self.prof or {}).items():
            ms = sum(a.elapsed_time(b) for a, b, _ in recs)
            out[name] = dict(launches=len(recs), ms=ms, bytes=float(sum(nb for _, _, nb in recs)))
        self.prof = None
        return out

    def mark(self, name, nbytes):
        """``with rt.mark("spmm", bytes): launch`` -- a no-op unless profiling is on"""
        if self.prof is None:
            return _NO_MARK
        return _Mark(self, name, nbytes)

    def pinned(self, n, dtype=None):
        return self.torch.empty(int(n), dtype=dtype or self.torch.float64, pin_memory=True)

    def read(self, t, count=None):
        """small device tensor -> numpy: gnk_scalars_fetch + gnk_scalars_wait (one async copy into pinned memory behind
        everything enqueued on the current stream so far, then a wait for that copy)."""
        n = t.numel() if count is None else count
        if n > self._pinned_np.shape[0]:
            raise _lib.GnkError(f"scalar read-back of {n} doubles exceeds the {self._pinned_np.shape[0]}-double staging buffer")
        lib, ctx = self.lib, self.ctx
        if lib.gnk_scalars_fetch(ctx, t.data_ptr(), n, self._pinned_ptr, self.stream) or lib.gnk_scalars_wait(ctx):
            _lib.check(-1, "scalar read-back")
        return self._pinned_np[:n].copy()

    def read_begin(self, t, count):
        """enqueue the read-back of ``t[:count]`` behind the work queued so far; ``read_end`` returns the values.
        Kernels enqueued between the two calls keep the device busy while the host waits for the scalars
        (gauss_newton_krylow's speculative basis expansion).  At most one such read is in flight (its own pinned
        block, so a plain ``read`` in between does not disturb it)."""
        if self.lib.gnk_scalars_fetch(self.ctx, t.data_ptr(), count, self._pinned2_ptr, self.stream):
            _lib.check(-1, "gnk_scalars_fetch")
        return count

    def read_end(self, count):
        if self.lib.gnk_scalars_wait(self.ctx):
            _lib.check(-1, "gnk_scalars_wait")
        return self._pinned2_np[:count].copy()

    def read_i32(self, t):
        self._pinned_i[:t.numel()].copy_(t, non_blocking=True)
        self.sync()
        return self._pinned_i[:t.numel()].numpy().copy()

    def upload(self, host, out):
        """host ndarray -> device tensor slice (direct DMA when the ndarray is pinned)."""
        src = self.torch.from_numpy(np.ascontiguousarray(host, dtype=np.float64))
        out.copy_(src, non_blocking=True)

    def download(self, t):
        """device tensor -> new host ndarray (through a pinned staging buffer it owns)."""
        h = self.pinned(t.numel(), t.dtype)
        h.copy_(t, non_blocking=True)
        self.sync()
        return h.numpy()

    def host_register(self, addr, nbytes):
        """page-lock host memory this process did not allocate through torch (a /dev/shm mapping), so that copies to
        and from it are asynchronous DMA"""
        rc = self.torch.cuda.cudart().cudaHostRegister(int(addr), int(nbytes), 0)
        if int(rc) != 0:
            raise _lib.GnkError(f"cudaHostRegister failed (cudaError {int(rc)})")

    def launches(self):
        return int(self.lib.gnk_launch_count(self.ctx))

    def allreduce(self, t, count, op=0):
        if self.world > 1:
            _lib.check(self.lib.gnk_comm_allreduce(self.ctx, ptr(t), int(count), int(op), self.stream), "allreduce")


class _Mark:
    __slots__ = ("rt", "name", "nbytes", "e0", "cancel")

    def __init__(self, rt, name, nbytes):
        self.rt, self.name, self.nbytes, self.cancel = rt, name, nbytes, False

    def __enter__(self):
        if self.rt.prof is not None:
            self.e0 = self.rt.torch.cuda.Event(enable_timing=True)
            self.e0.record()
        return self

    def __exit__(self, *exc):
        if self.rt.prof is not None and not self.cancel:
            e1 = self.rt.torch.cuda.Event(enable_timing=True)
            e1.record()
            self.rt.prof.setdefault(self.name, []).append((self.e0, e1, self.nbytes))
        return False


class _NoMark:
    """what ``rt.mark`` hands out while no profile is being taken: one shared object, nothing recorded"""
    __slots__ = ("cancel",)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


_NO_MARK = _NoMark()


class SharedBuffersUnavailable(RuntimeError):
    """raised on EVERY rank together when /dev/shm cannot hold another result buffer"""


class NodeSharedBuffers:
    """Host result buffers shared by the ranks of ONE node (files in /dev/shm mapped by every rank, page-locked with
    cudaHostRegister): a rank copies only ITS slab device -> host, and every rank still sees the whole vector -- the
    N-fold all-gather + N full-vector D2H copies of round 1 become one slab copy per rank.

    All ranks call ``acquire()`` together.  A buffer is handed out again only when NO rank holds an array over it any
    more: every rank tests its own weak reference, the flags are max-reduced over the ranks (one tiny collective), so
    all ranks pick the same buffer or grow the pool together."""

    def __init__(self, rt, n_doubles):
        self.rt, self.n = rt, int(n_doubles)
        box = [f"gnk_b200_{os.getpid()}_{time.monotonic_ns()}"]
        rt.torch.distributed.broadcast_object_list(box, src=0)
        self.token = box[0]
        self.bufs = []      # [mmap, host tensor over it, weakref to the ctypes owner of the array handed out | None]
        self.flags = rt.zeros(16)
        atexit.register(self.close)

    def _path(self, i):
        return f"/dev/shm/{self.token}_{i}"

    def _grow(self):
        rt, i = self.rt, len(self.bufs)
        if i >= 16:
            raise _lib.GnkError("more than 16 full-vector results are alive at once; copy or drop some")
        nbytes = 8 * self.n
        ok = [True]
        if rt.rank == 0:
            try:
                fd0 = os.open(self._path(i), os.O_RDWR | os.O_CREAT | os.O_EXCL, 0o600)
                try:
                    os.posix_fallocate(fd0, 0, nbytes)  # reserve the pages now: a full /dev/shm must not end in SIGBUS
                finally:
                    os.close(fd0)
            except OSError:
                ok[0] = False
                try:
                    os.unlink(self._path(i))
                except OSError:
                    pass
        rt.torch.distributed.broadcast_object_list(ok, src=0)
        if not ok[0]:
            raise SharedBuffersUnavailable(f"/dev/shm cannot hold a {nbytes >> 20} MiB result buffer")
        fd = os.open(self._path(i), os.O_RDWR)
        try:
            mm = mmap.mmap(fd, nbytes)
        finally:
            os.close(fd)
        host = rt.torch.frombuffer(mm, dtype=rt.torch.float64, count=self.n)
        rt.host_register(host.data_ptr(), nbytes)
        self.bufs.append([mm, host, None])
        return i

    def acquire(self):
        """-> (host tensor over the whole buffer, finish) ; ``finish()`` (collective, after this rank's copy has been
        enqueued) waits until every rank's part is in host memory and returns the ndarray to hand out"""
        rt = self.rt
        nb = len(self.bufs)
        pick = None
        if nb:
            busy = [1.0 if (b[2] is not None and b[2]() is not None) else 0.0 for b in self.bufs]
            stage = rt.pinned(16)
            stage.zero_()
            stage[:nb] = rt.torch.tensor(busy, dtype=rt.torch.float64)
            self.flags.copy_(stage, non_blocking=True)
            rt.allreduce(self.flags, nb, 1)
            vals = rt.read(self.flags, nb)
            free = np.nonzero(vals == 0.0)[0]
            if free.size:
                pick = int(free[0])
        if pick is None:
            pick = self._grow()
        mm, host, _ = self.bufs[pick]

        def finish():
            rt.sync()                      # this rank's slab is in host memory
            rt.allreduce(self.flags, 1, 1)   # ... and so is everybody else's (any collective is a barrier)
            rt.read(self.flags, 1)
            owner = (C.c_double * self.n).from_buffer(mm)
            self.bufs[pick][2] = weakref.ref(owner)
            out = np.frombuffer(owner, dtype=np.float64)
            out.flags.writeable = False  # the memory is shared by all ranks: in-place edits would hit every rank
            return out

        return host, finish

    def close(self):
        for i, (mm, host, _) in enumerate(self.bufs):
            try:
                self.rt.torch.cuda.cudart().cudaHostUnregister(host.data_ptr())
            except Exception:
                pass
            if self.rt.rank == 0:
                try:
                    os.unlink(self._path(i))
                except OSError:
                    pass
        self.bufs = []


def ptr(t, offset=0):
    """device pointer of a torch tensor (+ element offset) as a plain int, None -> NULL (every prototype in _lib.py
    declares c_void_p, which takes both; building a c_void_p object per argument cost ~25 us per outer iteration)"""
    if t is None:
        return None
    if offset:
        return t.data_ptr() + offset * t.element_size()
    return t.data_ptr()


def get_runtime() -> Runtime:
    global _runtime
    if _runtime is None:
        _runtime = Runtime()
    return _runtime


def make_layout(fields) -> _lib.Layout:
    return _lib.Layout(fields["n_own"], fields["off"], fields["ld"], fields["m"], fields["rows"], fields["halo"],
                       fields["has_lo"], fields["has_hi"], 0)


class DeviceVector:
    """A vector that lives in HBM, handed to callbacks and returned by device-native ``res``.

    It converts to a host ``ndarray`` lazily (``np.asarray(v)``, arithmetic with ndarrays, indexing,
    ``.copy()``), so a callback that ignores ``x`` costs no PCIe traffic, while reference-style
    callbacks (``error(x)``, ``x.copy()``) keep working unchanged.
    """

    __array_priority__ = 0.0

    def __init__(self, owner, tensor, n_global):
        self._owner = owner        # object with .download_global(tensor) -> ndarray
        self._t = tensor           # stored column (device)
        self._host = None
        self.shape = (int(n_global),)
        self.ndim = 1
        self.dtype = np.dtype(np.float64)
        self.size = int(n_global)

    def materialize(self):
        if self._host is None:
            self._host = self._owner.download_global(self._t)
            self._t = None
        return self._host

    def release_or_snapshot(self):
        """Ownership hand-off after a callback returned.  The solver calls this as ``ref = weakref.ref(xv); del xv;
        DeviceVector.settle(ref)``: if the weak reference is dead nobody kept the vector and nothing happens; if it is
        alive the callback (or a wrapper, a debugger, a list ...) holds it, and the host snapshot is taken NOW, because
        the device buffer is about to be overwritten.  No reference counts are inspected."""
        if self._host is None:
            self.materialize()

    @staticmethod
    def settle(ref):
        v = ref()
        if v is not None:
            v.release_or_snapshot()

    def __array__(self, dtype=None, copy=None):
        a = self.materialize()
        if dtype is not None and np.dtype(dtype) != a.dtype:
            return a.astype(dtype)
        return a

    def __len__(self):
        return self.shape[0]

    def __getitem__(self, i):
        return self.materialize()[i]

    def __iter__(self):
        return iter(self.materialize())

    def copy(self):
        return self.materialize().copy()

    def __neg__(self):
        return -self.materialize()

    def __add__(self, o):
        return self.materialize() + o

    def __sub__(self, o):
        return self.materialize() - o

    def __mul__(self, o):
        return self.materialize() * o

    def __pow__(self, o):
        return self.materialize() ** o

    def __repr__(self):
        return f"DeviceVector(n={self.shape[0]}, {'host' if self._host is not None else 'device'})"


# --------------------------------------------------------------------------------------------------
# generic problem: foreign Python callables res / jac (the reference's callback protocol, SURVEY A13).
# The callables themselves run on the host -- they are the user's code -- and their outputs are
# uploaded; every solver operation (J V_k, J^T r, Gram-Schmidt, least squares, line-search
# reductions) runs on the device through the CSR kernels.
# --------------------------------------------------------------------------------------------------
class CsrJacobian:
    def __init__(self, rt, host_J, is_sparse):
        import scipy.sparse as sp

        self.rt = rt
        self.host = host_J
        self.is_sparse = is_sparse
        A = host_J.tocsr() if hasattr(host_J, "tocsr") else sp.csr_array(np.asarray(host_J, dtype=np.float64))
        if max(int(A.nnz), *(int(v) for v in A.shape)) >= _INT32_LIMIT:  # the int32 casts below would wrap silently
            raise _lib.GnkError(f"jac: a {A.shape[0]} x {A.shape[1]} Jacobian with {A.nnz} non-zeros does not fit the "
                                "int32 indices of the CSR kernels (every dimension and nnz must stay below 2^31 - 1)")
        A = sp.csr_array(A)
        A.sort_indices()
        AT = sp.csr_array(A.T)
        AT.sort_indices()
        self.n_res, self.p = A.shape
        t = rt.torch
        dev = rt.device

        def up(a, dt):
            return t.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(dev)

        self.rowptr, self.col, self.val = up(A.indptr, np.int32), up(A.indices, np.int32), up(A.data, np.float64)
        self.rowptr_t, self.col_t, self.val_t = up(AT.indptr, np.int32), up(AT.indices, np.int32), up(AT.data, np.float64)

    def matmat(self, V, ldv, k, JV, ldjv):
        rt = self.rt
        _lib.check(rt.lib.gnk_spmm_csr(rt.ctx, self.n_res, ptr(self.rowptr), ptr(self.col), ptr(self.val), ptr(V), ldv,
                                       0, k, 1.0, ptr(JV), ldjv, 0, rt.stream), "gnk_spmm_csr")

    def neg_rmatvec(self, r, w):
        rt = self.rt
        _lib.check(rt.lib.gnk_spmm_csr(rt.ctx, self.p, ptr(self.rowptr_t), ptr(self.col_t), ptr(self.val_t), ptr(r), 0,
                                       0, 1, -1.0, ptr(w), 0, 0, rt.stream), "gnk_spmm_csr(T)")

    def linop(self, sign):
        op = _lib.LinOp()
        op.kind = 1
        op.sign = sign
        op.n_res, op.p = self.n_res, self.p
        op.d_rowptr, op.d_col, op.d_val = ptr(self.rowptr), ptr(self.col), ptr(self.val)
        op.d_rowptr_t, op.d_col_t, op.d_val_t = ptr(self.rowptr_t), ptr(self.col_t), ptr(self.val_t)
        return op


class DenseJacobian:
    """A dense Jacobian that gauss_newton solves with gnk_dense_qr_ls (p >= GNK_DENSE_QR_MIN columns): kept as the user
    returned it -- ``host`` the ndarray / np.matrix, or ``user`` = ``dense`` the strided CUDA tensor -- with no CSR form.
    The least-squares call gets it as one column-major panel (``fill_panel``)."""

    is_sparse = False

    def __init__(self, rt, host=None, dense=None):
        self.rt, self.host, self.dense, self.user = rt, host, dense, dense
        if dense is not None:
            self.n_res, self.p = (int(v) for v in dense.shape)
        else:
            self.n_res, self.p = np.shape(host)

    def fill_panel(self, panel):
        """panel: (p + 1, lda) view of the column-major least-squares panel; rows :p, entries :n_res get J^T"""
        n, p = self.n_res, self.p
        if self.dense is not None:
            panel[:p, :n].copy_(self.dense.T)  # one device-to-device copy (transpose, and a cast if not float64)
            return
        torch = self.rt.torch
        a = np.asarray(self.host, dtype=np.float64)
        if a.flags.f_contiguous:  # J^T is C-ordered already: upload it straight into the panel rows
            panel[:p, :n].copy_(torch.from_numpy(a.T))
        else:  # one upload of J, transposed on the device
            panel[:p, :n].copy_(torch.from_numpy(np.ascontiguousarray(a)).to(panel.device).T)


class HostCallableProblem:
    """res / jac are arbitrary Python callables returning host objects."""

    distributed = False

    def __init__(self, res, jac, x0, args):
        self.rt = get_runtime()
        self.res, self.jac, self.args = res, jac, tuple(args)
        self.p_glob = int(np.asarray(x0).shape[0])
        self.sol_fields = flat_layout_fields(self.p_glob)
        self.sol = make_layout(self.sol_fields)
        self.n_res = None
        self.res_fields = None
        self.last_res_host = None

    # residual-space layout is known after the first residual evaluation
    def _ensure_res_layout(self, n_res):
        if self.n_res is None:
            self.n_res = int(n_res)
            self.res_fields = flat_layout_fields(self.n_res)
            self.res_lay = make_layout(self.res_fields)

    def probe(self, x0_host):
        r = np.asarray(self.res(np.array(x0_host, dtype=np.float64), *self.args), dtype=np.float64).reshape(-1)
        self._ensure_res_layout(r.shape[0])
        return r

    def new_sol(self):
        return self.rt.zeros(self.sol_fields["ld"])

    def new_res(self):
        return self.rt.zeros(self.res_fields["ld"])

    def upload_x(self, x_host, out):
        self.rt.upload(np.asarray(x_host, dtype=np.float64).reshape(-1), out[:self.p_glob])

    def download_global(self, t):
        return self.rt.download(t[:self.p_glob])

    def residual_host(self, x_host, F, loss_slot):
        r = np.asarray(self.res(x_host, *self.args), dtype=np.float64).reshape(-1)
        self._ensure_res_layout(r.shape[0])
        self.rt.upload(r, F[:self.n_res])
        self.sumsq(F, loss_slot, self.res_lay)
        self.last_res_host = r
        return r

    def residual(self, x, F, loss_slot, aux=None):
        self.residual_host(self.download_global(x), F, loss_slot)

    def sumsq(self, vec, slot2, lay):
        rt = self.rt
        _lib.check(rt.lib.gnk_norm_stats(rt.ctx, C.byref(lay), ptr(vec), ptr(slot2), rt.stream), "gnk_norm_stats")

    def jacobian_host(self, x_host, dense_panel=False):
        """jac at x_host as a CsrJacobian; with ``dense_panel`` a dense J of p >= GNK_DENSE_QR_MIN columns comes back as a
        DenseJacobian instead (gauss_newton's blocked QR branch, which needs no CSR form)"""
        import scipy.sparse as sp

        J = self.jac(x_host, *self.args)
        sparse = isinstance(J, (sp.sparray, sp.spmatrix)) or hasattr(J, "_gnk_sparse_like")
        if dense_panel and not sparse and not hasattr(J, "tocsr") and self.p_glob >= _lib.GNK_DENSE_QR_MIN:
            if np.ndim(J) != 2 or np.shape(J)[1] != self.p_glob:
                raise ValueError(f"jac: expected a 2-D Jacobian with {self.p_glob} columns, got shape {np.shape(J)}")
            return DenseJacobian(self.rt, host=J)
        return CsrJacobian(self.rt, J, sparse)

    def jacobian(self, x, aux=None):
        return self.jacobian_host(self.download_global(x))


# --------------------------------------------------------------------------------------------------
# device callables: res / jac take and return CUDA tensors (selected by a CUDA-tensor x0).  The callables are still
# the user's code, but x, F and J never leave HBM: the residual is copied device to device; a dense Jacobian is used
# as it arrives (DenseDeviceJacobian), a sparse one's index pattern and its transpose are built on the device
# (gnk_csr_pattern) and cached while the pattern stays the same.
# --------------------------------------------------------------------------------------------------
_INT32_LIMIT = (1 << 31) - 1  # sizes and nnz stay below: int32 indices, and n + 1 row pointers


def is_cuda_tensor(x):
    torch = sys.modules.get("torch")
    return torch is not None and isinstance(x, torch.Tensor) and x.is_cuda


def _require_on_device(rt, t, what):
    if not isinstance(t, rt.torch.Tensor):
        raise TypeError(f"{what}: expected a torch.Tensor on {rt.device}, got {type(t).__name__}")
    if t.device != rt.device:
        raise ValueError(f"{what}: expected a tensor on {rt.device}, got one on {t.device}")


def device_csr(rt, J, shape=None, what="jac"):
    """A CUDA matrix (torch sparse CSR / COO, or a strided (n_res, p) tensor) -> (rowptr, col, val, is_sparse): the
    canonical CSR of J (COO coalesced, dense without its exact zeros, as scipy.sparse.csr_array(dense)) with int32 or
    int64 indices and float64 values."""
    torch = rt.torch
    _require_on_device(rt, J, what)
    if J.dim() != 2:
        raise ValueError(f"{what}: expected a 2-D Jacobian, got shape {tuple(J.shape)}")
    if shape is not None and tuple(J.shape) != tuple(shape):
        raise ValueError(f"{what}: expected shape {tuple(shape)} (n_res, p), got {tuple(J.shape)}")
    n_rows, n_cols = (int(v) for v in J.shape)
    nnz = J._nnz() if J.layout in (torch.sparse_csr, torch.sparse_coo) else 0
    if max(n_rows, n_cols, nnz) >= _INT32_LIMIT:
        raise _lib.GnkError(f"{what}: a {n_rows} x {n_cols} Jacobian with {nnz} stored entries does not fit the int32 "
                            "indices of the CSR kernels (every dimension and nnz must stay below 2^31 - 1)")
    if J.layout == torch.sparse_csr:
        A = J
    elif J.layout == torch.sparse_coo:
        A = J.coalesce().to_sparse_csr()
    elif J.layout == torch.strided:
        A = J.to_sparse_csr()
    else:
        raise TypeError(f"{what}: expected a sparse_csr, sparse_coo or strided tensor, got layout {J.layout}")
    if A._nnz() >= _INT32_LIMIT:
        raise _lib.GnkError(f"{what}: {A._nnz()} non-zeros do not fit the int32 indices of the CSR kernels")
    rowptr, col = A.crow_indices().contiguous(), A.col_indices().contiguous()
    if col.dtype != rowptr.dtype:
        col = col.to(rowptr.dtype)
    val = A.values().to(torch.float64).contiguous()
    return rowptr, col, val, J.layout != torch.strided


class CsrPattern:
    """The index pattern of a CSR matrix on the device, as int32 (rowptr, col), with the sorted pattern of its transpose
    (rowptr_t, col_t) and perm: transpose position -> non-zero of A (gnk_csr_pattern).  Immutable: a Jacobian built on
    it keeps it alive, and a changed pattern gets a new object."""

    def __init__(self, rt, n_rows, n_cols, rowptr, col):
        t = rt.torch
        self.rt = rt
        self.n_rows, self.n_cols, self.nnz = int(n_rows), int(n_cols), int(col.numel())
        i32 = t.int32
        self.rowptr = t.empty(self.n_rows + 1, dtype=i32, device=rt.device)
        self.rowptr_t = t.empty(self.n_cols + 1, dtype=i32, device=rt.device)
        self.col, self.col_t, self.perm = (t.empty(self.nnz, dtype=i32, device=rt.device) for _ in range(3))
        rc = rt.lib.gnk_csr_pattern(rt.ctx, self.n_rows, self.n_cols, self.nnz, ptr(rowptr), ptr(col),
                                    rowptr.element_size(), ptr(self.rowptr), ptr(self.col), ptr(self.rowptr_t),
                                    ptr(self.col_t), ptr(self.perm), rt.stream)
        if rc == _lib.GNK_PATTERN_INVALID:
            raise ValueError(rt.lib.gnk_last_error().decode())
        _lib.check(rc, "gnk_csr_pattern")

    def matches(self, n_rows, n_cols, rowptr, col, flag):
        """same shape and the same index arrays (one device compare, one int read back)"""
        if (int(n_rows), int(n_cols), int(col.numel())) != (self.n_rows, self.n_cols, self.nnz):
            return False
        rt = self.rt
        _lib.check(rt.lib.gnk_csr_pattern_equal(rt.ctx, self.n_rows, self.nnz, ptr(rowptr), ptr(col),
                                                rowptr.element_size(), ptr(self.rowptr), ptr(self.col), ptr(flag),
                                                rt.stream), "gnk_csr_pattern_equal")
        return int(rt.read_i32(flag)[0]) == 0


class DeviceCsrJacobian:
    """J on the device as CSR of J and of J^T over a CsrPattern; J^T's values by one gather (gnk_csr_gather).  Same
    interface as CsrJacobian.  ``user`` is the object the user's jac returned (handed to a step-length plug-in)."""

    transposed = False
    scale = 1.0

    def __init__(self, rt, pattern, val, is_sparse, user=None):
        self.rt, self.pattern, self.val = rt, pattern, val
        self.is_sparse, self.user = is_sparse, user
        self.n_res, self.p = pattern.n_rows, pattern.n_cols
        self.rowptr, self.col, self.rowptr_t, self.col_t = pattern.rowptr, pattern.col, pattern.rowptr_t, pattern.col_t
        self.val_t = rt.torch.empty_like(val)
        _lib.check(rt.lib.gnk_csr_gather(rt.ctx, pattern.nnz, ptr(pattern.perm), ptr(val), ptr(self.val_t), rt.stream),
                   "gnk_csr_gather")

    @classmethod
    def from_tensor(cls, rt, J, what="A"):
        rowptr, col, val, is_sparse = device_csr(rt, J, what=what)
        return cls(rt, CsrPattern(rt, J.shape[0], J.shape[1], rowptr, col), val, is_sparse, J)

    matmat = CsrJacobian.matmat
    neg_rmatvec = CsrJacobian.neg_rmatvec
    linop = CsrJacobian.linop


class DenseDeviceJacobian:
    """A strided CUDA Jacobian used as it arrives: J V_k and -J^T r by gnk_dense_matmat / gnk_dense_rmatvec, which give
    the bits gnk_spmm_csr gives on the CSR of the same matrix -- with no CSR form, no pattern and no copy of J^T, and
    no int32 limit on the number of entries.  ``user`` is the tensor jac returned (handed to a step-length plug-in),
    ``dense`` the float64 tensor the kernels read: ``user`` itself, or one contiguous float64 copy when ``user`` is of
    another dtype or has neither stride equal to 1.  The solvers read ``dense`` until the next jac call returns, so a jac
    may refill one tensor in place (gauss_newton_krylow forms -J_old^T r of the jac_old_* versions before that call)."""

    is_sparse = False

    def __init__(self, rt, J):
        torch = rt.torch
        self.rt, self.user = rt, J
        self.n_res, self.p = (int(v) for v in J.shape)
        if J.dtype != torch.float64:
            J = J.to(torch.float64)  # keeps a dense layout's strides, makes any other layout contiguous
        if not self._strides(J):
            J = J.contiguous()
        self.dense = J
        self.rs, self.cs = self._strides(J)

    def _strides(self, J):
        """(row stride, column stride) with the stride of a dimension of size 1 taken as 1, or None if neither is 1"""
        rs, cs = (1 if n == 1 else int(s) for n, s in zip(J.shape, J.stride()))
        return (rs, cs) if 1 in (rs, cs) else None

    def matmat(self, V, ldv, k, JV, ldjv):
        rt = self.rt
        _lib.check(rt.lib.gnk_dense_matmat(rt.ctx, self.n_res, self.p, ptr(self.dense), self.rs, self.cs, ptr(V), ldv, 0,
                                           k, 1.0, ptr(JV), ldjv, 0, rt.stream), "gnk_dense_matmat")

    def neg_rmatvec(self, r, w):
        rt = self.rt
        _lib.check(rt.lib.gnk_dense_rmatvec(rt.ctx, self.n_res, self.p, ptr(self.dense), self.rs, self.cs, ptr(r), -1.0,
                                            ptr(w), rt.stream), "gnk_dense_rmatvec")

    def linop(self, sign):
        """the kind-2 gnk_linop of sign * J for gnk_cgls: the matrix read in place, no CSR pair"""
        op = _lib.LinOp()
        op.kind = 2
        op.sign = sign
        op.n_res, op.p = self.n_res, self.p
        op.d_dense, op.row_stride, op.col_stride = ptr(self.dense), self.rs, self.cs
        return op


class DeviceCallableProblem:
    """res / jac are Python callables on CUDA tensors: res(x, *args) -> 1-D tensor of n_res values, jac(x, *args) ->
    torch sparse CSR / COO or strided (n_res, p) tensor.  x is a fresh float64 tensor of length p at every call."""

    distributed = False
    device_native = True  # x and F stay in HBM
    user_code = True      # ... but res / jac are the user's: they are evaluated only where the reference evaluates them

    def __init__(self, res, jac, x0, args):
        self.rt = rt = get_runtime()
        _require_on_device(rt, x0, "x0")
        self.res, self.jac, self.args = res, jac, tuple(args)
        self.p_glob = int(x0.numel())
        if self.p_glob >= _INT32_LIMIT:
            raise _lib.GnkError(f"x0 has {self.p_glob} entries; the CSR kernels index with int32")
        self.sol_fields = flat_layout_fields(self.p_glob)
        self.sol = make_layout(self.sol_fields)
        self.n_res = None
        self.res_fields = None
        self.pattern = None
        self.pattern_builds = 0   # gnk_csr_pattern calls: once per distinct sparsity pattern of jac
        self._flag = rt.torch.zeros(1, dtype=rt.torch.int32, device=rt.device)

    def _ensure_res_layout(self, n_res):
        if self.n_res is None:
            if n_res >= _INT32_LIMIT:
                raise _lib.GnkError(f"res returned {n_res} values; the CSR kernels index with int32")
            self.n_res = int(n_res)
            self.res_fields = flat_layout_fields(self.n_res)
            self.res_lay = make_layout(self.res_fields)

    def new_sol(self):
        return self.rt.zeros(self.sol_fields["ld"])

    def new_res(self):
        return self.rt.zeros(self.res_fields["ld"])

    def upload_x(self, x, out):
        out[:self.p_glob].copy_(x.reshape(-1))

    def download_global(self, t):
        return self.rt.download(t[:self.p_glob])

    def x_out(self, t):
        """the iterate as the user sees it: a CUDA tensor of its own"""
        return t[:self.p_glob].clone()

    def evaluate(self, x):
        """res at the stored column x -> 1-D CUDA tensor (fixes the residual-space layout at the first call)"""
        r = self.res(self.x_out(x), *self.args)
        _require_on_device(self.rt, r, "res")
        if r.dim() != 1:
            raise ValueError(f"res: expected a 1-D tensor, got shape {tuple(r.shape)}")
        if self.n_res is not None and r.shape[0] != self.n_res:
            raise ValueError(f"res: expected {self.n_res} values (the length of its first result), got {r.shape[0]}")
        self._ensure_res_layout(r.shape[0])
        return r

    def residual(self, x, F, loss_slot, aux=None):
        F[:self.n_res].copy_(self.evaluate(x))
        self.sumsq(F, loss_slot, self.res_lay)

    def sumsq(self, vec, slot2, lay):
        rt = self.rt
        _lib.check(rt.lib.gnk_norm_stats(rt.ctx, C.byref(lay), ptr(vec), ptr(slot2), rt.stream), "gnk_norm_stats")

    def jacobian(self, x, aux=None, dense_panel=False):
        """jac at x: a strided J as a DenseDeviceJacobian -- or, with ``dense_panel`` and p >= GNK_DENSE_QR_MIN, as a
        DenseJacobian (gauss_newton's blocked QR branch) -- and a sparse J as a DeviceCsrJacobian"""
        J = self.jac(self.x_out(x), *self.args)
        torch = self.rt.torch
        if isinstance(J, torch.Tensor) and J.layout == torch.strided:
            _require_on_device(self.rt, J, "jac")
            panel = dense_panel and self.p_glob >= _lib.GNK_DENSE_QR_MIN
            if tuple(J.shape) != (self.n_res, self.p_glob):
                if J.dim() != 2 and not panel:
                    raise ValueError(f"jac: expected a 2-D Jacobian, got shape {tuple(J.shape)}")
                raise ValueError(f"jac: expected shape {(self.n_res, self.p_glob)} (n_res, p), got {tuple(J.shape)}")
            if panel:
                return DenseJacobian(self.rt, dense=J)
            return DenseDeviceJacobian(self.rt, J)
        rowptr, col, val, is_sparse = device_csr(self.rt, J, (self.n_res, self.p_glob))
        pat = self.pattern
        if pat is None or not pat.matches(self.n_res, self.p_glob, rowptr, col, self._flag):
            pat = CsrPattern(self.rt, self.n_res, self.p_glob, rowptr, col)
            self.pattern = pat
            self.pattern_builds += 1
        return DeviceCsrJacobian(self.rt, pat, val, is_sparse, J)
