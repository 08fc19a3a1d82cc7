"""Krylov bases past 255 columns (gauss_newton_krylow(max_basis_columns=...), GeneralizedKrylowSubspace(max_columns=...))
on the CPU: argument checks, the default cap and its error, the scalar-block layout, the host control flow of a wide
solve through the numpy stand-in of the library, and the library's exports and SASS."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle import gnk_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_max_columns_is_checked_before_any_device_work():
    import gauss_newton_via_generalized_krylov_subspaces_b200 as g
    from gauss_newton_via_generalized_krylov_subspaces_b200.krylow import resolve_max_columns
    assert resolve_max_columns(None) == 255
    assert resolve_max_columns(1) == 1 and resolve_max_columns(np.int64(4095)) == 4095
    for bad in (0, -1, 4096, 300.0, "300", True, [300]):
        with pytest.raises(ValueError):
            resolve_max_columns(bad)
        with pytest.raises(ValueError):
            g.gauss_newton_krylow(lambda x: x, np.ones(3), lambda x: np.eye(3), max_basis_columns=bad)
        with pytest.raises(ValueError):
            g.GeneralizedKrylowSubspace(max_columns=bad)


def test_growing_past_the_cap_raises_the_message_of_the_default():
    from gauss_newton_via_generalized_krylov_subspaces_b200 import GeneralizedKrylowSubspace, _lib
    ks = GeneralizedKrylowSubspace()
    ks.cap = 255
    with pytest.raises(_lib.GnkError, match="^Krylov basis wider than 255 columns is not supported; pass krylow_restart$"):
        ks._grow()
    ks = GeneralizedKrylowSubspace(max_columns=700)
    ks.cap = 700
    with pytest.raises(_lib.GnkError, match="wider than 700 columns"):
        ks._grow()


def test_scalar_block_layout():
    from gauss_newton_via_generalized_krylov_subspaces_b200.gauss_newton_krylow import scalar_layout
    # the default cap (and every narrower one) keeps the offsets of a GNK_MAX_BASIS = 256 block
    for cap in (1, 100, 255):
        assert scalar_layout(cap) == (520, 522, 524, 525, 528)
    # a wide cap: the result block (2k + 4 doubles) of the widest panel stays below the loss slot
    for cap in (256, 700, 4095):
        loss, cprev, flag, flag2, total = scalar_layout(cap)
        assert loss >= 2 * cap + 4 and (cprev, flag, flag2, total) == (loss + 2, loss + 4, loss + 5, loss + 8)
    assert scalar_layout(4095)[4] <= 2 * 4096 + 16  # Runtime's pinned read-back buffers


def test_wide_entry_in_header_signatures_and_exports():
    from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib
    header = open(os.path.join(ROOT, "include", "gnk_b200.h")).read()
    assert "int gnk_basis_ls_wide(gnk_ctx* ctx, double* d_P, int64_t ldp, int64_t n_rows, int k, double sign_a, " \
           "double* d_out,\n                      void* stream);" in header
    assert "#define GNK_MAX_BASIS_WIDE 4096" in header and "#define GNK_MAX_BASIS 256" in header
    assert _lib.GNK_MAX_BASIS_WIDE == 4096 and _lib.GNK_MAX_BASIS == 256
    assert "gnk_basis_ls_wide" in _lib.SIGNATURES
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip("library not built")
    nm = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    assert " T gnk_basis_ls_wide" in nm


def test_library_holds_the_wide_kernels():
    """the shipped .so carries the wide streaming kernels (128-bit streaming loads, no DMMA) and the kernels of the
    sharded wide least squares"""
    import __graft_entry__
    __graft_entry__.build()
    from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib
    if not shutil.which("cuobjdump"):
        pytest.skip("cuobjdump is not installed")
    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    funcs = {f.split("\n", 1)[0].strip(): f for f in sass.split("Function : ")[1:]}
    for kern in ("combine_wide_kernel", "dots_wide_kernel", "update_wide_kernel"):
        body = [b for name, b in funcs.items() if kern in name]
        assert len(body) == 1, kern
        assert "LDG.E.EF.128" in body[0] or "LDG.E.128.STRONG" in body[0] or ".128" in body[0], kern
        assert "DFMA" in body[0] and "DMMA" not in body[0], kern
    for kern in ("wls_pack_kernel", "wls_rho_kernel", "wls_stack_kernel", "wls_pad_kernel"):
        assert any(kern in name for name in funcs), kern


# ---- host control flow of a wide solve, through the numpy stand-in ----------------------------------------------
@pytest.fixture()
def g():
    import mock_backend
    rt = mock_backend.install()
    lib = rt.lib
    # the read-back buffers of the product's Runtime (2 * GNK_MAX_BASIS_WIDE + 16 doubles): the stand-in's are narrower
    for name in ("_pinned", "_pinned2"):
        buf = rt.torch.empty(2 * 4096 + 16, dtype=rt.torch.float64)
        setattr(rt, name, buf)
        setattr(rt, name + "_np", buf.numpy())
        setattr(rt, name + "_ptr", buf.data_ptr())

    def basis_ls_wide(ctx, P, ldp, n_rows, k, sign_a, out, stream):  # the panel [JV | r]: r is column k
        assert k >= 256 and n_rows >= k + 1
        return lib.gnk_tsqr_ls(ctx, P, ldp, n_rows, k, int(P) + 8 * k * int(ldp), sign_a, out, stream)

    lib.gnk_basis_ls_wide = basis_ls_wide
    import gauss_newton_via_generalized_krylov_subspaces_b200 as pkg
    yield pkg
    mock_backend.uninstall()


def test_host_wide_basis_bratu_g41(g, capsys):
    """Bratu G = 41 without a restart: the oracle converges with a basis of 311 columns.  The default cap stops at column
    256 with today's error; max_basis_columns=700 runs to the oracle's counts."""
    o = orc.BratuOracle(41, 5, 10)
    y, u0 = o.operator(o.u_true), o.start_vector(seed=42)
    pb = g.BratuPdeProblem(41, 5, 10)
    cb = dict(callback=lambda **kw: None)
    with pytest.raises(g._lib.GnkError, match="wider than 255 columns"):
        g.gauss_newton_krylow(pb.make_res(y), u0, pb.make_jac(), max_iter=700, **cb)
    out = g.gauss_newton_krylow(pb.make_res(y), u0, pb.make_jac(), max_iter=700, max_basis_columns=700, **cb)
    assert (out.nit, out.nrev, out.njev, out.success) == (311, 312, 311, True)
    x = np.asarray(out.x)
    assert np.max(np.abs(x - o.u_true)) / np.max(np.abs(o.u_true)) < 1e-5  # the oracle: 1.07e-6
    with pytest.raises(g._lib.GnkError, match="wider than 300 columns"):
        g.gauss_newton_krylow(pb.make_res(y), u0, pb.make_jac(), max_iter=700, max_basis_columns=300, **cb)
