"""cg_least_squares with a dense CUDA A (gnk_linop kind 2: csrc/cgls.cu on the dense_jac.cu kernels): bit for bit the
result of the same matrix handed over as torch CSR, with no CSR form built; a matrix of more than 2^31 entries against
a float64 restatement of scipy's cg on cuBLAS products, with no copy of A; gnk_dense_col_sumsq against
gnk_csr_row_sumsq; and, without a GPU, the library surface (SASS, exports, the gnk_linop layout)."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def g():
    import gauss_newton_via_generalized_krylov_subspaces_b200 as pkg
    import gauss_newton_via_generalized_krylov_subspaces_b200.device as device
    device._runtime = None
    pkg.get_runtime()
    return pkg


def _bits(t):
    return t.detach().cpu().numpy().view(np.int64)


def _matrix(rng, n, p, zeros=True):
    """Gaussian entries over four decades; with ``zeros``: exact zeros, -0.0 entries and an empty row (row 1)"""
    A = rng.standard_normal((n, p)) * 10.0 ** rng.integers(-2, 2, (n, p))
    if zeros:
        A[rng.random((n, p)) < 0.3] = 0.0
        A[rng.random((n, p)) < 0.05] = -0.0
        A[1, :] = 0.0
    return A


def _layouts(torch, A, dev):
    """one matrix in every layout the dense operator reads in place, plus the two inputs that take one copy"""
    n, p = A.shape
    t = torch.as_tensor(A, device=dev)
    pad = torch.full((n, p + 3), 7.0, dtype=torch.float64, device=dev)
    pad[:, :p] = t
    tall = torch.full((n + 9, p), 7.0, dtype=torch.float64, device=dev)
    tall[4:4 + n] = t
    tpad = torch.full((p, n + 5), 7.0, dtype=torch.float64, device=dev)
    tpad[:, :n] = t.T
    wide = torch.full((n, 2 * p), 7.0, dtype=torch.float64, device=dev)
    wide[:, ::2] = t
    return {"row": t.contiguous(), "col": t.T.contiguous().T, "t_view": tpad[:, :n].T,
            "padded": pad[:, :p], "row_slice": tall[4:4 + n], "float32": t.float(), "step2": wide[:, ::2]}


def _both(g, A, y, **kw):
    """(dense x, dense count, CSR x, CSR count) of cg_least_squares on A and on A.to_sparse_csr()"""
    xd, itd = g.cg_least_squares(A, y, **kw)
    xc, itc = g.cg_least_squares(A.to_sparse_csr(), y, **kw)
    return xd, itd, xc, itc


def _cases(g):
    """name -> (A, y, kwargs): shapes x layouts, zeros / -0.0 / empty row, scaled operators, solver settings"""
    import torch
    dev = g.get_runtime().device
    rng = np.random.default_rng(11)
    out = {}
    for shape in ((20000, 300), (500, 500), (200, 700), (150000, 40)):
        A = _matrix(rng, *shape)
        y = torch.as_tensor(rng.standard_normal(shape[0]), device=dev)
        for name, At in _layouts(torch, A, dev).items():
            out[f"{shape[0]}x{shape[1]}-{name}"] = (At, y, {})
    A = torch.as_tensor(_matrix(rng, 3000, 120), device=dev)
    y = torch.as_tensor(rng.standard_normal(3000), device=dev)
    x0 = torch.as_tensor(rng.standard_normal(120), device=dev)
    out["neg"] = (-1 * A, y, {})
    yt = torch.as_tensor(rng.standard_normal(120), device=dev)
    out["scaled_transpose"] = (2.5 * A[2:].T, yt, {})  # without the empty row, which would be an empty column
    for pre in (True, False):
        out[f"precond_{pre}"] = (A, y, dict(preconditioner=pre))
        out[f"x0_random_precond_{pre}"] = (A.T.contiguous().T, y, dict(x0=x0, preconditioner=pre))
    x_true = torch.as_tensor(rng.standard_normal(120), device=dev)
    out["x0_exact"] = (A, A @ x_true, dict(x0=x_true))
    e1 = torch.zeros(3000, dtype=torch.float64, device=dev)
    e1[1] = 1.0  # row 1 of A is empty: A^T y = 0 exactly
    out["ATy_zero"] = (A, e1, dict(x0=x0))
    out["rtol_1e-9"] = (A, y, dict(cg_rtol=1e-9))
    # maxiter: singular values 1 .. 1e-6 and a tolerance below what float64 reaches (tests/test_cgls_reference.py)
    rs = np.random.RandomState(0)
    U, _ = np.linalg.qr(rs.normal(size=(40, 20)))
    V, _ = np.linalg.qr(rs.normal(size=(20, 20)))
    G = torch.as_tensor((U * np.logspace(0, -6, 20)) @ V.T, device=dev)
    yg = torch.as_tensor(rs.normal(size=40), device=dev)
    for pre in (True, False):
        out[f"maxiter_precond_{pre}"] = (G, yg, dict(cg_rtol=1e-18, preconditioner=pre))
    # an empty column (diag(A^T A) = 0) or one NaN: NaN iterates, the solve runs to maxiter = 10 p
    S = _matrix(rng, 60, 12)
    S[:, 5] = 0.0
    out["empty_column"] = (torch.as_tensor(S, device=dev), torch.as_tensor(rng.standard_normal(60), device=dev), {})
    S = _matrix(rng, 60, 12)
    S[7, 3] = np.nan
    out["nan"] = (torch.as_tensor(S, device=dev), torch.as_tensor(rng.standard_normal(60), device=dev),
                  dict(preconditioner=False))
    return out


CASE_NAMES = ([f"{n}x{p}-{lay}" for n, p in ((20000, 300), (500, 500), (200, 700), (150000, 40))
               for lay in ("row", "col", "t_view", "padded", "row_slice", "float32", "step2")]
              + ["neg", "scaled_transpose", "precond_True", "precond_False", "x0_random_precond_True",
                 "x0_random_precond_False", "x0_exact", "ATy_zero", "rtol_1e-9", "maxiter_precond_True",
                 "maxiter_precond_False", "empty_column", "nan"])


@pytest.fixture(scope="module")
def cases(g):
    out = _cases(g)
    assert sorted(out) == sorted(CASE_NAMES)
    return out


# ------------------------------------------------------------------------------------------------
# 1. bit for bit the CSR route, and no CSR built on the way
# ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", CASE_NAMES)
def test_dense_cg_least_squares_equals_the_csr_route_bitwise(g, cases, name):
    import torch
    A, y, kw = cases[name]
    xd, itd, xc, itc = _both(g, A, y, **kw)
    assert isinstance(xd, torch.Tensor) and xd.is_cuda and xd.shape == (A.shape[1],)
    assert itd == itc, (itd, itc)
    assert np.array_equal(_bits(xd), _bits(xc))
    p = A.shape[1]
    if name == "x0_exact":
        assert itd == 0 and torch.equal(xd, kw["x0"])
    elif name == "ATy_zero":
        assert itd == 0 and not torch.any(xd)
    elif name.startswith("maxiter"):
        assert itd == (10 * p if kw["preconditioner"] else 20 * p)
    elif name == "empty_column":
        assert itd == 10 * p and torch.isnan(xd).all()
    elif name == "nan":
        assert itd == 20 * p and torch.isnan(xd).all()
    else:
        assert 0 < itd < 10 * p and torch.isfinite(xd).all()


@gpu
def test_dense_cg_least_squares_builds_no_csr(g, cases, monkeypatch):
    import gauss_newton_via_generalized_krylov_subspaces_b200.device as device
    ref = {name: g.cg_least_squares(*cases[name][:2], **cases[name][2]) for name in CASE_NAMES}

    def refuse(*a, **k):
        raise AssertionError("a CSR form was built for a dense A")

    monkeypatch.setattr(device, "device_csr", refuse)
    monkeypatch.setattr(device, "CsrPattern", refuse)
    for name in CASE_NAMES:
        A, y, kw = cases[name]
        x, it = g.cg_least_squares(A, y, **kw)
        assert it == ref[name][1] and np.array_equal(_bits(x), _bits(ref[name][0])), name
    with pytest.raises(AssertionError, match="CSR form"):  # the patch is live: a sparse A still takes the CSR route
        g.cg_least_squares(cases["neg"][0].to_sparse_csr(), cases["neg"][1])


@gpu
def test_dense_cg_least_squares_keeps_the_errors(g):
    import torch
    dev = g.get_runtime().device
    A = torch.ones(5, 3, dtype=torch.float64, device=dev)
    y = torch.ones(5, dtype=torch.float64, device=dev)
    with pytest.raises(ValueError, match="y must have 5 entries, got 4"):
        g.cg_least_squares(A, y[:4])
    with pytest.raises(ValueError, match="x0 must have 3 entries, got 2"):
        g.cg_least_squares(A, y, x0=y[:2])
    with pytest.raises(ValueError, match="2-D"):
        g.cg_least_squares(A[None], y)
    with pytest.raises(TypeError, match="torch.Tensor"):
        g.cg_least_squares(A, y.cpu().numpy())
    with pytest.raises(ValueError, match="cpu"):
        g.cg_least_squares(A, y.cpu())


# ------------------------------------------------------------------------------------------------
# 2. more than 2^31 entries
# ------------------------------------------------------------------------------------------------
def _cg_reference(A, y, nmax, chunk):
    """scipy's cg on A^T A x = A^T y with the Jacobi preconditioner, x0 = 0, restated in float64 torch (cuBLAS
    products), without the stopping test: -> (||r_j|| for j = 0 .. nmax, [x_j])"""
    import torch
    b = A.T @ y
    diag = torch.zeros(A.shape[1], dtype=torch.float64, device=A.device)
    for r0 in range(0, A.shape[0], chunk):
        diag += (A[r0:r0 + chunk] ** 2).sum(0)
    minv = 1.0 / diag
    x = torch.zeros_like(b)
    r = b.clone()
    rn, xs = [], []
    p = rho_prev = None
    for it in range(nmax + 1):
        rn.append(float(torch.linalg.norm(r)))
        xs.append(x.clone())
        if it == nmax:
            break
        z = minv * r
        rho = torch.dot(r, z)
        p = z.clone() if it == 0 else p * (rho / rho_prev) + z
        q = A.T @ (A @ p)
        a = rho / torch.dot(p, q)
        x = x + a * p
        r = r - a * q
        rho_prev = rho
    return np.array(rn), xs, float(torch.linalg.norm(b))


@gpu
def test_dense_cg_least_squares_past_2_31_entries(g):
    """A seeded Gaussian 2 100 000 x 1100 A (2.31e9 entries, 18.5 GB), which the CSR route refused: the iteration count
    equals that of scipy's cg restated on cuBLAS products at a tolerance the residuals clear by 0.1 % or more, x agrees
    within 1e-10, and the call allocates no more than its work vectors (A is never copied)."""
    import torch
    rt = g.get_runtime()
    n, p, chunk = 2_100_000, 1100, 131072
    assert n * p >= 2 ** 31
    if torch.cuda.mem_get_info(rt.device)[0] < 30e9:
        pytest.skip("needs about 30 GB of free device memory")
    gen = torch.Generator(device=rt.device).manual_seed(3)
    A = torch.empty(n, p, dtype=torch.float64, device=rt.device)
    for r0 in range(0, n, chunk):
        A[r0:r0 + chunk].normal_(generator=gen)
    A *= torch.logspace(0, -1, p, dtype=torch.float64, device=rt.device)
    y = torch.randn(n, dtype=torch.float64, device=rt.device, generator=gen)
    rn, xs, bn = _cg_reference(A, y, 12, chunk)
    # the latest j whose residual lies 0.1 % or more below every earlier one, above rounding level; rtol halfway (in log)
    cand = [j for j in range(1, rn.shape[0]) if rn[:j].min() / rn[j] >= 1.001 and rn[j] > 1e-11 * bn]
    assert cand
    j = cand[-1]
    rtol = float(np.sqrt(rn[:j].min() * rn[j])) / bn
    vlen = -(-max(n, p) // 16) * 16
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats(rt.device)
    before = torch.cuda.memory_allocated(rt.device)
    x, it = g.cg_least_squares(A, y, cg_rtol=rtol)
    grown = torch.cuda.max_memory_allocated(rt.device) - before
    assert grown < 8 * 8 * vlen + (64 << 20), grown
    assert it == j, (it, j, rn.tolist())
    err = float(torch.linalg.norm(x - xs[j]) / torch.linalg.norm(xs[j]))
    assert err < 1e-10, err


# ------------------------------------------------------------------------------------------------
# 3. the kernels: gnk_dense_col_sumsq, the one-column product, kind 2 through gnk_cgls_x0
# ------------------------------------------------------------------------------------------------
def _strides(J):
    return tuple(1 if n == 1 else s for n, s in zip(J.shape, J.stride()))


def _csr32(torch, A):
    S = A.to_sparse_csr()
    return S.crow_indices().to(torch.int32), S.col_indices().to(torch.int32), S.values().contiguous()


@gpu
@pytest.mark.parametrize("n,p", [(1, 1), (1, 37), (53, 1), (300, 300), (1001, 77), (45, 700), (129, 33)])
def test_col_sumsq_equals_csr_row_sumsq_of_the_transpose_bitwise(g, n, p):
    import torch
    from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib
    from gauss_newton_via_generalized_krylov_subspaces_b200.device import ptr
    rt = g.get_runtime()
    rng = np.random.default_rng(n * 7 + p)
    A = _matrix(rng, n, p, zeros=n > 2)
    if n > 2 and p > 2:
        A[:, p // 2] = -0.0
        A[n - 2, 1] = np.nan
    t = torch.as_tensor(A, device=rt.device)
    rp, _, va = _csr32(torch, t.T)
    ref = torch.full((p,), 3.0, dtype=torch.float64, device=rt.device)
    _lib.check(rt.lib.gnk_csr_row_sumsq(rt.ctx, p, ptr(rp), ptr(va), ptr(ref), rt.stream), "gnk_csr_row_sumsq")
    for name, J in _layouts(torch, A, rt.device).items():
        if J.dtype != torch.float64 or _strides(J).count(1) == 0:
            continue
        rs, cs = _strides(J)
        out = torch.full_like(ref, 5.0)
        _lib.check(rt.lib.gnk_dense_col_sumsq(rt.ctx, n, p, ptr(J), rs, cs, ptr(out), rt.stream), "gnk_dense_col_sumsq")
        assert np.array_equal(_bits(out), _bits(ref)), name
    assert rt.lib.gnk_dense_col_sumsq(rt.ctx, n, p, ptr(t), 2, 2, ptr(ref), rt.stream) != 0


@gpu
@pytest.mark.parametrize("n,p", [(150001, 37), (120000, 64)])
def test_one_column_product_of_many_rows_equals_the_csr_kernel_bitwise(g, n, p):
    """k = 1 takes dense_matvec_kernel; at 3 x 148 row tiles of 256 and more it runs 256 chains per CTA (the
    shapes of tests/test_gpu_dense_jacobian.py take the 32-row tiles)"""
    import torch
    from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib
    from gauss_newton_via_generalized_krylov_subspaces_b200.device import ptr
    rt = g.get_runtime()
    rng = np.random.default_rng(p)
    A = _matrix(rng, n, p)
    A[n - 1, p - 1] = np.nan
    rp, ci, va = _csr32(torch, torch.as_tensor(A, device=rt.device))
    v = torch.as_tensor(rng.standard_normal(p + 2), device=rt.device)
    ref = torch.full((n + 3,), 3.0, dtype=torch.float64, device=rt.device)
    _lib.check(rt.lib.gnk_spmm_csr(rt.ctx, n, ptr(rp), ptr(ci), ptr(va), ptr(v), 0, 2, 1, -0.5, ptr(ref), 0, 3,
                                   rt.stream), "gnk_spmm_csr")
    for name, J in _layouts(torch, A, rt.device).items():
        if J.dtype != torch.float64 or _strides(J).count(1) == 0:
            continue
        rs, cs = _strides(J)
        out = torch.full_like(ref, 3.0)
        _lib.check(rt.lib.gnk_dense_matmat(rt.ctx, n, p, ptr(J), rs, cs, ptr(v), 0, 2, 1, -0.5, ptr(out), 0, 3,
                                           rt.stream), "gnk_dense_matmat")
        assert np.array_equal(_bits(out), _bits(ref)), name


@gpu
def test_kind_2_through_gnk_cgls_x0(g):
    import torch
    from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib
    from gauss_newton_via_generalized_krylov_subspaces_b200.device import DenseDeviceJacobian, DeviceCsrJacobian, ptr
    rt = g.get_runtime()
    rng = np.random.default_rng(4)
    n, p = 2000, 90
    A = torch.as_tensor(_matrix(rng, n, p), device=rt.device).T.contiguous().T
    vlen = -(-max(n, p) // 16) * 16
    y = torch.zeros(vlen, dtype=torch.float64, device=rt.device)
    y[:n] = torch.as_tensor(rng.standard_normal(n), device=rt.device)
    x0 = torch.zeros(vlen, dtype=torch.float64, device=rt.device)
    x0[:p] = torch.as_tensor(rng.standard_normal(p), device=rt.device)
    dense, csr = DenseDeviceJacobian(rt, A), DeviceCsrJacobian.from_tensor(rt, A)
    assert dense.dense.data_ptr() == A.data_ptr()
    got = []
    for op in (dense.linop(-1.5), csr.linop(-1.5)):
        for pre in (0, 1):
            x = torch.full((vlen,), 9.0, dtype=torch.float64, device=rt.device)
            work = torch.full((7 * vlen,), 9.0, dtype=torch.float64, device=rt.device)
            iters = C.c_int64(-1)
            _lib.check(rt.lib.gnk_cgls_x0(rt.ctx, C.byref(op), ptr(y), ptr(x0), 1e-6, pre, ptr(x), ptr(work),
                                          C.byref(iters), rt.stream), "gnk_cgls_x0")
            got.append((iters.value, _bits(x[:p])))
    assert got[0][0] > got[1][0] > 0  # preconditioner = 0 adds the iterations of the discarded first run
    for (ia, xa), (ib, xb) in zip(got[:2], got[2:]):
        assert ia == ib and np.array_equal(xa, xb)
    bad = dense.linop(1.0)
    bad.col_stride, bad.row_stride = 2, 2
    x = torch.zeros(vlen, dtype=torch.float64, device=rt.device)
    work = torch.zeros(7 * vlen, dtype=torch.float64, device=rt.device)
    iters = C.c_int64(0)
    assert rt.lib.gnk_cgls_x0(rt.ctx, C.byref(bad), ptr(y), None, 1e-6, 1, ptr(x), ptr(work), C.byref(iters),
                              rt.stream) != 0


# ------------------------------------------------------------------------------------------------
# 4. without a GPU: the shipped library and the header
# ------------------------------------------------------------------------------------------------
def _functions(sass):
    parts = re.split(r"\n\s*Function : (\S+)\n", sass)
    return dict(zip(parts[1::2], parts[2::2]))


def test_library_holds_the_dense_cg_kernels():
    import __graft_entry__
    __graft_entry__.build()
    from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib
    funcs = _functions(subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True,
                                      check=True).stdout)
    sumsq = [f for f in funcs if "dense_col_sumsq_kernel" in f]
    matvec = [f for f in funcs if "dense_matvec_kernel" in f]
    assert len(sumsq) == 2 and len(matvec) == 4
    for f in sumsq + matvec:
        assert "DFMA" in funcs[f] and "DMMA" not in funcs[f] and "LDGSTS" in funcs[f], f
    log = os.path.join(ROOT, "gauss_newton_via_generalized_krylov_subspaces_b200", "csrc", "build",
                       "dense_jac.ptxas.log")
    if os.path.exists(log):  # ptxas -v of the last build: no spills anywhere in dense_jac.cu
        text = open(log).read()
        assert "dense_col_sumsq_kernel" in text and "dense_matvec_kernel" in text
        assert all(m == "0" for m in re.findall(r"(\d+) bytes spill stores", text))


def test_header_declares_and_library_exports_col_sumsq():
    import __graft_entry__
    __graft_entry__.build()
    from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib
    header = open(os.path.join(ROOT, "include", "gnk_b200.h")).read()
    assert re.search(r"int gnk_dense_col_sumsq\(gnk_ctx\* ctx, int64_t n_rows, int64_t n_cols, const double\* d_J,",
                     header)
    nm = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    assert re.search(r"\bT gnk_dense_col_sumsq\b", nm)
    assert "gnk_dense_col_sumsq" in _lib.SIGNATURES


def test_linop_ctypes_layout_matches_the_header(tmp_path):
    from gauss_newton_via_generalized_krylov_subspaces_b200 import _lib
    src = tmp_path / "probe.cpp"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "gnk_b200.h"\n'
                   'int main() { printf("%zu %zu %zu %zu %zu\\n", sizeof(gnk_linop), offsetof(gnk_linop, d_val_t), '
                   'offsetof(gnk_linop, d_dense), offsetof(gnk_linop, row_stride), offsetof(gnk_linop, col_stride)); '
                   'return 0; }\n')
    exe = tmp_path / "probe"
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    subprocess.run([nvcc, "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    L = _lib.LinOp
    assert got == [C.sizeof(L), L.d_val_t.offset, L.d_dense.offset, L.row_stride.offset, L.col_stride.offset]
    assert L.d_dense.offset == L.d_val_t.offset + 8  # the new fields follow the kind-1 fields
