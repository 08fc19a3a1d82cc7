"""CPU checks for dense Jacobians: host Jacobians whose CSR form would overflow the int32 indices are refused before
anything is uploaded, and the shipped library carries the dense J V_k / J^T r kernels (FP64 FMA chains, no DMMA)."""
import re
import subprocess

import pytest


class _HugeCsr:
    """what scipy would hand CsrJacobian for a 2^20 x 2^12 matrix with 2^31 + 5 non-zeros, without the arrays"""
    shape = (1 << 20, 1 << 12)
    nnz = (1 << 31) + 5

    def tocsr(self):
        return self


def test_host_jacobian_with_2_31_nonzeros_is_refused_before_upload():
    from gauss_newton_via_generalized_krylov_subspaces_b200._lib import GnkError
    from gauss_newton_via_generalized_krylov_subspaces_b200.device import CsrJacobian

    class NoRuntime:
        def __getattr__(self, name):
            raise AssertionError(f"the runtime was used ({name}) before the size check")

    with pytest.raises(GnkError, match=r"2\^31"):
        CsrJacobian(NoRuntime(), _HugeCsr(), True)
    tall = _HugeCsr()
    tall.shape, tall.nnz = ((1 << 31), 1), 3
    with pytest.raises(GnkError, match=r"2\^31"):
        CsrJacobian(NoRuntime(), tall, True)


def _functions(sass):
    """{mangled kernel name: its SASS} from cuobjdump -sass output"""
    parts = re.split(r"\n\s*Function : (\S+)\n", sass)
    return dict(zip(parts[1::2], parts[2::2]))


def test_library_holds_the_dense_jacobian_kernels():
    import __graft_entry__
    __graft_entry__.build()
    from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib
    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    funcs = _functions(sass)
    matmat = [f for f in funcs if "dense_matmat_kernel" in f]
    rmatvec = [f for f in funcs if "dense_rmatvec_kernel" in f]
    assert len(matmat) == 10 and len(rmatvec) == 2
    for f in matmat + rmatvec:
        body = funcs[f]
        assert "DFMA" in body and "DMMA" not in body, f
        assert "LDGSTS" in body, f  # cp.async staging
    for name in ("gnk_dense_matmat", "gnk_dense_rmatvec"):
        assert name in _lib.SIGNATURES
