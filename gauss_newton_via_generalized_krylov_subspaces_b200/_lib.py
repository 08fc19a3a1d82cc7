"""ctypes binding of libgnk_b200.so (include/gnk_b200.h).

The shared object is built in-tree by ``__graft_entry__.build()`` / ``make -C csrc``.  There is no
CPU fallback: if the library is missing, or no CUDA device is visible, every solver entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgnk_b200.so")

GNK_MAX_BASIS = 256
GNK_MAX_BASIS_WIDE = 4096  # streaming kernels and gnk_basis_ls_wide: bases of up to 4095 columns
GNK_TSQR_MAX = 104  # include/gnk_b200.h
GNK_DENSE_QR_MIN, GNK_DENSE_QR_MAX = 256, 4095  # gnk_dense_qr_ls: dense least squares of 256..4095 columns
GNK_PATTERN_INVALID = 3  # gnk_csr_pattern: the index pattern is not canonical CSR


class Layout(C.Structure):
    """gnk_layout"""
    _fields_ = [("n_own", C.c_int64), ("off", C.c_int64), ("ld", C.c_int64), ("m", C.c_int32),
                ("rows", C.c_int32), ("halo", C.c_int32), ("has_lo", C.c_int32), ("has_hi", C.c_int32),
                ("pad_", C.c_int32)]


class Bratu(C.Structure):
    """gnk_bratu"""
    _fields_ = [("c_lap", C.c_double), ("c_adv", C.c_double), ("lam", C.c_double)]


class LinOp(C.Structure):
    """gnk_linop"""
    _fields_ = [("kind", C.c_int32), ("pad_", C.c_int32), ("sign", C.c_double), ("lay", Layout), ("prm", Bratu),
                ("d_expu", C.c_void_p), ("n_res", C.c_int64), ("p", C.c_int64), ("d_rowptr", C.c_void_p),
                ("d_col", C.c_void_p), ("d_val", C.c_void_p), ("d_rowptr_t", C.c_void_p), ("d_col_t", C.c_void_p),
                ("d_val_t", C.c_void_p), ("d_dense", C.c_void_p), ("row_stride", C.c_int64), ("col_stride", C.c_int64)]


_P = C.c_void_p
_I = C.c_int
_L = C.c_int64
_D = C.c_double
_LP = C.POINTER(Layout)
_BP = C.POINTER(Bratu)

# name -> (restype, argtypes); kept in one table so tests can check the exported symbols against the header
SIGNATURES = {
    "gnk_abi_version": (_I, []),
    "gnk_last_error": (C.c_char_p, []),
    "gnk_create": (_I, [C.POINTER(_P), _I]),
    "gnk_destroy": (_I, [_P]),
    "gnk_sm_count": (_I, [_P]),
    "gnk_launch_count": (_L, [_P]),
    "gnk_scalars_fetch": (_I, [_P, _P, _I, _P, _P]),
    "gnk_scalars_wait": (_I, [_P]),
    "gnk_bratu_residual": (_I, [_P, _LP, _BP, _P, _P, _P, _P, _I, _P, _P]),
    "gnk_stencil_apply": (_I, [_P, _LP, _BP, _P, _P, _L, _I, _D, _I, _P, _L, _L, _P]),
    "gnk_stencil_normal_diag": (_I, [_P, _LP, _BP, _P, _P, _P]),
    "gnk_combine": (_I, [_P, _LP, _P, _I, _P, _P, _D, _P, _P]),
    "gnk_combine_step": (_I, [_P, _LP, _P, _I, _P, _P, _D, _P, _P, _P, _P]),
    "gnk_norm_stats": (_I, [_P, _LP, _P, _P, _P]),
    "gnk_normalize": (_I, [_P, _LP, _P, _P, _D, _P, _P, _P]),
    "gnk_normalize_halo": (_I, [_P, _LP, _P, _P, _D, _P, _P, _P]),
    "gnk_cgs_dots": (_I, [_P, _LP, _P, _I, _P, _P, _P]),
    "gnk_bratu_trial_project": (_I, [_P, _LP, _BP, _P, _I, _P, _P, _D, _P, _P, _P, _P, _P, _P, _P]),
    "gnk_cgs_update": (_I, [_P, _LP, _P, _I, _P, _P, _P, _P]),
    "gnk_tsqr_ls": (_I, [_P, _P, _L, _L, _I, _P, _D, _P, _P]),
    "gnk_dense_qr_ls": (_I, [_P, _P, _L, _L, _I, _D, _P, _P]),
    "gnk_basis_ls_wide": (_I, [_P, _P, _L, _L, _I, _D, _P, _P]),
    "gnk_stencil_gram_ls": (_I, [_P, _LP, _BP, _P, _P, _L, _I, _I, _P, _D, _P, _L, _D, _P, _P]),
    "gnk_tsqr_ls_method": (_I, [_P, _I]),
    "gnk_gram_cgls": (_I, [_P, _P, _L, _L, _I, _P, _D, _D, _P, _P]),
    "gnk_spmm_csr": (_I, [_P, _L, _P, _P, _P, _P, _L, _L, _I, _D, _P, _L, _L, _P]),
    "gnk_csr_row_sumsq": (_I, [_P, _L, _P, _P, _P, _P]),
    "gnk_csr_pattern": (_I, [_P, _L, _L, _L, _P, _P, _I, _P, _P, _P, _P, _P, _P]),
    "gnk_csr_pattern_equal": (_I, [_P, _L, _L, _P, _P, _I, _P, _P, _P]),
    "gnk_csr_gather": (_I, [_P, _L, _P, _P, _P, _P]),
    "gnk_dense_matmat": (_I, [_P, _L, _L, _P, _L, _L, _P, _L, _L, _I, _D, _P, _L, _L, _P]),
    "gnk_dense_rmatvec": (_I, [_P, _L, _L, _P, _L, _L, _P, _D, _P, _P]),
    "gnk_dense_col_sumsq": (_I, [_P, _L, _L, _P, _L, _L, _P, _P]),
    "gnk_axpby": (_I, [_P, _L, _D, _P, _D, _P, _P, _P]),
    "gnk_dot": (_I, [_P, _L, _P, _P, _P, _P]),
    "gnk_cgls": (_I, [_P, C.POINTER(LinOp), _P, _D, _I, _P, _P, C.POINTER(_L), _P]),
    "gnk_cgls_x0": (_I, [_P, C.POINTER(LinOp), _P, _P, _D, _I, _P, _P, C.POINTER(_L), _P]),
    "gnk_rosenbrock_residual": (_I, [_P, _L, _D, _P, _P, _P]),
    "gnk_rosenbrock_jacobian": (_I, [_P, _L, _D, _P, _P, _P, _P]),
    "gnk_comm_unique_id": (_I, [_P]),
    "gnk_comm_init": (_I, [_P, _P, _I, _I]),
    "gnk_comm_size": (_I, [_P]),
    "gnk_comm_p2p_export": (_I, [_P, _P]),
    "gnk_comm_p2p_attach": (_I, [_P, _P]),
    "gnk_comm_p2p_enabled": (_I, [_P]),
    "gnk_comm_p2p_disable": (_I, [_P]),
    "gnk_comm_fused_reductions": (_I, [_P]),
    "gnk_comm_allreduce": (_I, [_P, _P, _I, _I, _P]),
    "gnk_comm_halo_exchange": (_I, [_P, _LP, _P, _I, _P]),
    "gnk_comm_allgather_owned": (_I, [_P, _LP, _P, _P, C.POINTER(_L), _P]),
}


class GnkError(RuntimeError):
    pass


_lib = None


def load():
    """Load libgnk_b200.so and declare every prototype.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GnkError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  This package has no CPU fallback.")
    nccl = _find_nccl()
    if nccl and "GNK_NCCL_LIB" not in os.environ:
        os.environ["GNK_NCCL_LIB"] = nccl
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.gnk_abi_version() != 1:
        raise GnkError("libgnk_b200.so ABI version mismatch")
    _lib = lib
    return lib


def _find_nccl():
    try:
        import nvidia.nccl  # torch-bundled wheel
        for base in list(getattr(nvidia.nccl, "__path__", [])):
            p = os.path.join(base, "lib", "libnccl.so.2")
            if os.path.exists(p):
                return p
    except Exception:
        pass
    return None


def check(rc, what=""):
    if rc != 0:
        msg = load().gnk_last_error()
        raise GnkError(f"{what} failed (rc={rc}): {msg.decode() if msg else '?'}")
