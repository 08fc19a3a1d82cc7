/* gnk_b200.h -- C ABI of the B200 (sm_100a) Gauss-Newton-Krylov hot path.
 *
 * The reference (mariusbaehr/gauss_newton_via_generalized_krylov_subspaces) is pure Python and has
 * no FFI layer; its operator API for this path is the Python callable protocol of
 * gauss_newton_krylow.py:39-49 / krylow.py:16-73 / armijo_goldstein.py:16-25 / gauss_newton.py:11-73 /
 * bratu_pde_problem.py:76-96.  Every entry point below names the reference expression it replaces.
 * The thin Python host (gauss_newton_via_generalized_krylov_subspaces_b200/*.py) binds these with
 * ctypes; INTEGRATION.md shows the stub.
 *
 * Conventions
 *   - all numeric data is IEEE fp64; indices int32 (CSR) / int64 (sizes)
 *   - every pointer named d_* is a DEVICE pointer owned by the caller (a torch allocation in the
 *     Python host); the library never frees or reallocates caller memory
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing synchronises
 *     unless stated
 *   - return value: 0 = ok, <0 = failure (gnk_last_error() gives the text).  No exceptions cross.
 *   - scalar results are written to caller-provided DEVICE slots so that the host reads one small
 *     block per outer iteration
 *
 * Vector layout (gnk_layout).  A "stored column" has `ld` doubles.  The rank's owned unknowns are
 * the n_own doubles starting at `off`.  For the Bratu stencil the column is a slab of `rows` owned
 * grid rows of `m` doubles each, preceded and followed by `halo` (=2) rows that mirror the
 * neighbouring ranks' rows (zeros at the domain boundary = the Dirichlet condition), so
 * off = halo*m, n_own = rows*m, ld >= (rows+2*halo)*m.  Generic (CSR) problems use m = 0,
 * halo = 0, off = 0.
 */
#ifndef GNK_B200_H
#define GNK_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GNK_B200_ABI_VERSION 1
#define GNK_MAX_BASIS 256 /* k <= 255 basis columns (+1 rhs column in the least-squares panel) */
#define GNK_TSQR_MAX 104  /* widest panel of the tiled Householder TSQR; wider panels (runs without a restart) take
                             the single-CTA Householder QR on one rank while n_rows * (k+1) <= 2^22 doubles (it needs
                             n_rows >= k+1), and the blocked Householder TSQR spread over the SMs otherwise (several
                             ranks, or larger panels) */

typedef struct gnk_ctx gnk_ctx;

typedef struct {
  int64_t n_own;  /* owned unknowns on this rank                                  */
  int64_t off;    /* index of the first owned double inside a stored column       */
  int64_t ld;     /* stored column length = stride between basis columns          */
  int32_t m;      /* doubles per grid row (0: not a stencil layout)               */
  int32_t rows;   /* owned grid rows                                              */
  int32_t halo;   /* stored halo depth in grid rows                               */
  int32_t has_lo; /* 1: a neighbour rank owns the rows before ours; 0: boundary   */
  int32_t has_hi; /* 1: a neighbour rank owns the rows after ours;  0: boundary   */
  int32_t pad_;
} gnk_layout;

/* constants of bratu_pde_problem.py:58,67,81-82: c_lap = h**-2, c_adv = ALPHA*h**-1, lam = LAMBDA */
typedef struct {
  double c_lap;
  double c_adv;
  double lam;
} gnk_bratu;

/* ---- lifecycle ------------------------------------------------------------------------------ */
int gnk_abi_version(void);
const char* gnk_last_error(void);
int gnk_create(gnk_ctx** out, int device);
int gnk_destroy(gnk_ctx* ctx);
int gnk_sm_count(gnk_ctx* ctx);
/* number of kernels this library has launched on this context since creation (bench: gpu_launches) */
int64_t gnk_launch_count(gnk_ctx* ctx);
/* The one host read-back of an outer iteration: the scalar block [d | ||JVd||^2 | ... | loss | flags] that
 * gauss_newton_krylow.py:88-100 consumes on the host (armijo_goldstein.py:47-72 judges the trial with it).
 * gnk_scalars_fetch enqueues the copy of `count` doubles to h_dst (page-locked host memory) behind the work queued on
 * `stream` so far, on the context's own copy stream; gnk_scalars_wait blocks until the last fetch has landed.  Kernels
 * enqueued on `stream` between the two calls overlap the host's wait (the speculative basis expansion, krylow.py:55-73). */
int gnk_scalars_fetch(gnk_ctx* ctx, const double* d_src, int count, double* h_dst, void* stream);
int gnk_scalars_wait(gnk_ctx* ctx);

/* ---- Bratu residual / Jacobian (bratu_pde_problem.py:76-96) ----------------------------------- */
/* F = y - (L u + alpha D u + lam e^u) on owned rows and `depth` (0|1) halo rows each side,
 * d_expu = e^u on the same rows (the only u-dependent part of J; pass NULL to skip, e.g. Armijo
 * trials), *d_loss = sum over OWNED rows of F^2 (armijo_goldstein.py:49,57).  Halo rows outside the
 * domain get F = 0.  u, y, F, expu all use the stored-column layout.  lam == 0 skips exp (:77-78). */
int gnk_bratu_residual(gnk_ctx* ctx, const gnk_layout* lay, const gnk_bratu* prm, const double* d_u,
                       const double* d_y, double* d_F, double* d_expu, int depth, double* d_loss,
                       void* stream);
/* out[:, j] = sign * Op * in[:, j], j < k, Op = P = L + alpha D + lam diag(e^u) (transpose == 0) or
 * P^T (transpose != 0).  sign = -1, transpose = 0 gives J @ V_k (gauss_newton_krylow.py:86);
 * sign = +1, transpose = 1 gives -J^T r (krylow.py:62).  `in` columns are stored columns (stride
 * in_ld, halo rows valid); out column j starts at d_out + j*out_ld + out_off and receives the n_own
 * owned values.  d_expu (stored-column layout) may be NULL when lam == 0. */
int gnk_stencil_apply(gnk_ctx* ctx, const gnk_layout* lay, const gnk_bratu* prm, const double* d_expu,
                      const double* d_in, int64_t in_ld, int k, double sign, int transpose,
                      double* d_out, int64_t out_ld, int64_t out_off, void* stream);
/* d_out[off + i] = diag(J^T J)_i (squared column norms of J), the Jacobi preconditioner that
 * gauss_newton.py:50-52 obtains from an A.T @ A SpGEMM. */
int gnk_stencil_normal_diag(gnk_ctx* ctx, const gnk_layout* lay, const gnk_bratu* prm,
                            const double* d_expu, double* d_out, void* stream);

/* ---- Krylov basis (krylow.py:30-73) ----------------------------------------------------------- */
/* x = V_k (c + s d) over the whole stored column (krylow.py:41-42, armijo_goldstein.py:56).
 * d_d may be NULL (x = V_k c).  c, d are device vectors of length k. */
int gnk_combine(gnk_ctx* ctx, const gnk_layout* lay, const double* d_V, int k, const double* d_c,
                const double* d_d, double s, double* d_x, void* stream);
/* gnk_combine that also leaves the coordinate bookkeeping of the outer iteration on the device (gauss_newton_krylow.py
 * :96-98,124), so that no k-sized kernel has to be launched for it: d_c_out[j] = c[j] + s d[j] for j < k and
 * d_c_out[k] = 0 (the trial's x_coordinate with the entry of the next basis column appended; GNK_MAX_BASIS doubles,
 * must not alias d_c; may be NULL), *d_cprev2 = sum_j c[j]^2 (may be NULL). */
int gnk_combine_step(gnk_ctx* ctx, const gnk_layout* lay, const double* d_V, int k, const double* d_c,
                     const double* d_d, double s, double* d_x, double* d_c_out, double* d_cprev2, void* stream);
/* d_stats[0] = sum of squares, d_stats[1] = max |.| over the owned part of a stored column
 * (krylow.py:31,36,66,71). */
int gnk_norm_stats(gnk_ctx* ctx, const gnk_layout* lay, const double* d_x, double* d_stats, void* stream);
/* out = x / sqrt(d_stats[0]) over the whole stored column (krylow.py:37,71) unless
 * d_stats[1] <= atol, in which case nothing is written and *d_flag = 1 (breakdown, krylow.py:66-69 /
 * x0 == 0, krylow.py:31-34); otherwise *d_flag = 0. */
int gnk_normalize(gnk_ctx* ctx, const gnk_layout* lay, const double* d_x, const double* d_stats,
                  double atol, double* d_out, int32_t* d_flag, void* stream);
/* gnk_normalize followed by the exchange of the new column's `halo` rows with the neighbouring ranks (the one halo
 * exchange of an outer iteration: every other vector inherits valid halos from the basis, DESIGN.md section 2).  With
 * the peer mailboxes attached both happen in ONE kernel: the CTAs that write the first / last owned rows also store
 * them into the neighbours' mailboxes over NVLink, and the CTA that arrives last exchanges the flags and fills this
 * rank's halo rows.  Single rank / no mailboxes: gnk_normalize (+ gnk_comm_halo_exchange). */
int gnk_normalize_halo(gnk_ctx* ctx, const gnk_layout* lay, const double* d_x, const double* d_stats, double atol,
                       double* d_out, int32_t* d_flag, void* stream);
/* h = V_k^T w over owned entries (first half of krylow.py:64). */
int gnk_cgs_dots(gnk_ctx* ctx, const gnk_layout* lay, const double* d_V, int k, const double* d_w,
                 double* d_h, void* stream);
/* w -= V_k h over owned entries (second half of krylow.py:64); d_stats as gnk_norm_stats of the
 * updated w (may be NULL). */
int gnk_cgs_update(gnk_ctx* ctx, const gnk_layout* lay, const double* d_V, int k, const double* d_h,
                   double* d_w, double* d_stats, void* stream);

/* ---- projected least squares (gauss_newton_krylow.py:16-36, :89) ------------------------------- */
/* Householder TSQR of the n_rows x (k+1) panel [sign_a*A | y] (A column-major, stride lda) and
 * solution of min || sign_a*A d - y ||_2.  Results (device): d_out[0..k) = d, d_out[k] = ||R d||^2
 * (= ||A d||^2, armijo_goldstein.py:50), d_out[k+1] = squared LS residual, d_out[k+2] = number of
 * |R_jj| <= 1e-8 (the "A is rank deficient" prints of :32-34), d_out[k+3] = ||d||^2,
 * d_out[k+4 .. 2k+4) = diag(R).  With a communicator attached the R factors of all ranks are
 * gathered and reduced identically on every rank.
 * Large panels (3 <= k+1 <= 32, >= 16384 rows, even row count, 16-byte aligned, sign_a = +-1) are solved on the FP64
 * tensor pipe instead (cholqr.cu): Gram matrix of the panel by DMMAs + Cholesky, then either one step of iterative
 * refinement of the normal-equation solution (one more HBM-bound pass; chosen on the device when every Cholesky pivot
 * ratio is >= 1e-10, i.e. cond <~ 1e5) or, on request (gnk_tsqr_ls_method 2), the second pass of CholeskyQR2
 * (R = R2 R1).  Same result block (diag(R) > 0; in the refinement form d_out[k] = (A^T y)^T d, which equals ||A d||^2 at
 * the least-squares solution with an error of second order in the remaining gradient, and d_out[k+1] = ||y - A d0||^2
 * of the normal-equation solution d0).  That path REFUSES panels whose Gram matrix is numerically rank
 * deficient (pivot ratio < 1e-12, e.g. a consistent system) or whose refinement step is not small: it then writes
 * d = 0 and d_out[k+2] = -1, and the caller re-issues the call after gnk_tsqr_ls_method(ctx, 1).
 * Panels of 33 <= k+1 <= 56 columns under the same conditions (krylow_restart up to 55; method 0 only) take the same
 * scheme with a wider Gram sweep (5..7 column blocks), a dense Cholesky in one CTA and the refinement form
 * (gram_cgls.cu: gnk_cholqr_wide_try), with the same result block and the same refusal convention.
 * Panels of GNK_TSQR_MAX < k+1 <= GNK_MAX_BASIS columns: one rank and n_rows * (k+1) <= 2^22 doubles take a single-CTA
 * unblocked Householder QR (n_rows >= k+1 required); several ranks or larger panels take a blocked Householder TSQR
 * (row-block leaves with compact-WY updates on the FP64 tensor pipe, pairwise tree, all-gather of the ranks' triangles,
 * reduced in rank order on every rank).  Any lda >= n_rows, 8-byte aligned A and y, ranks with fewer rows than columns. */
int gnk_tsqr_ls(gnk_ctx* ctx, const double* d_A, int64_t lda, int64_t n_rows, int k,
                const double* d_y, double sign_a, double* d_out, void* stream);

/* Least squares on a dense panel of GNK_DENSE_QR_MIN <= p <= GNK_DENSE_QR_MAX columns: the dense-Jacobian branch of
 * gauss_newton, scipy.linalg.lstsq(-J, r) (gauss_newton.py:116), for Jacobians wider than gnk_tsqr_ls takes.
 * d_A holds the augmented n_rows x (p+1) panel [A | y], column-major with stride lda (columns 0..p-1 = A, column p = y);
 * the call solves min || sign_a*A d - y ||_2 by blocked Householder QR of [sign_a*A | y] (LAPACK dgeqrf form: panels of
 * 32 columns factored over the SMs, compact-WY trailing updates with mma.m8n8k4.f64 on the FP64 tensor pipe, y updated
 * with the other trailing columns).  IN PLACE: the panel is overwritten (sign_a*A's R factor in the upper triangle,
 * the Householder vectors below it, Q^T y in column p); callers pass a scratch copy.  Result block (device, 2p+4
 * doubles) exactly as gnk_tsqr_ls: d_out[0..p) = d, d_out[p] = ||R d||^2, d_out[p+1] = squared LS residual,
 * d_out[p+2] = number of |R_jj| <= 1e-8, d_out[p+3] = ||d||^2, d_out[p+4 .. 2p+4) = diag(R).  Needs n_rows >= p,
 * lda >= n_rows and 8-byte aligned columns.  Every reduction has a fixed order: repeated calls give the same bits and a
 * power-of-two scaling of A and y changes no rounding.  One rank (the communicator is not used).  Scratch belongs to
 * the context. */
#define GNK_DENSE_QR_MIN 256
#define GNK_DENSE_QR_MAX 4095
int gnk_dense_qr_ls(gnk_ctx* ctx, double* d_A, int64_t lda, int64_t n_rows, int p, double sign_a, double* d_out,
                    void* stream);

/* Projected operator AND projected least squares of one GNK outer iteration in one call, for the Bratu stencil
 * (gauss_newton_krylow.py:86 `JV = jac_ev @ krylow.basis` followed by :89 `linear_least_squares(-1 * JV, res_ev)`):
 *   JV[:, j] = sign * (M V[:, j]), j < k   -- written (owned rows, column stride ldjv), bit-identical to gnk_stencil_apply
 *   d_out    = the result block of gnk_tsqr_ls(JV, ldjv, n_own, k, r, sign_a)
 * with the least-squares panel READ ONCE: a TMA-staged, warp-specialised kernel streams V_k through shared memory
 * (cp.async.bulk.tensor row slots, mbarrier ring), applies the stencil, stores J V and accumulates the Gram matrix of
 * [J V | r] with FP64 tensor-core MMAs in the same sweep; the refinement (or second CholeskyQR2) pass then reads J V
 * once more.  d_V: v_cols >= k stored columns (stride ldv, halo rows valid), d_r: the residual as a stored column,
 * d_expu as in gnk_stencil_apply.  Returns 1 -- nothing launched -- when the panel does not qualify (fewer than 16384
 * owned unknowns, more than 32 panel columns, m not a multiple of 8, Householder path pinned, GNK_LS_FUSED=0, ...): the
 * caller then issues gnk_stencil_apply + gnk_tsqr_ls.  Refusal (d_out[k+2] = -1) as for gnk_tsqr_ls; J V is valid then. */
int gnk_stencil_gram_ls(gnk_ctx* ctx, const gnk_layout* lay, const gnk_bratu* prm, const double* d_expu,
                        const double* d_V, int64_t ldv, int v_cols, int k, const double* d_r, double sign,
                        double* d_JV, int64_t ldjv, double sign_a, double* d_out, void* stream);

/* Factorisation used by gnk_tsqr_ls: 0 = automatic (tensor-pipe path where eligible, Householder TSQR otherwise; the
 * default -- GNK_LS_CHOLQR=0 in the environment disables the tensor-pipe path), 1 = Householder TSQR only,
 * 2 = as 0 but always the second CholeskyQR2 pass, never the refinement form.  Returns the previous setting, or a
 * negative status. */
int gnk_tsqr_ls_method(gnk_ctx* ctx, int method);

/* ---- generic sparse Jacobians (rosenbrock_problem.py:14-19, foreign callables) ----------------- */
/* out[:, j] = sign * A * in[:, j] for a CSR matrix with n_rows rows; in columns start at
 * d_in + j*in_ld + in_off, out columns at d_out + j*out_ld + out_off.  Each entry is sign * (the fma chain over the
 * row in index order, from 0.0), whatever k; the matrix is read once per block of 8 columns.  The transpose
 * product is the same call on the CSR of A^T (gnk_csr_pattern + gnk_csr_gather, or uploaded by the host). */
int gnk_spmm_csr(gnk_ctx* ctx, int64_t n_rows, const int32_t* d_rowptr, const int32_t* d_col,
                 const double* d_val, const double* d_in, int64_t in_ld, int64_t in_off, int k,
                 double sign, double* d_out, int64_t out_ld, int64_t out_off, void* stream);
/* out[i] = sum_j val_ij^2 per CSR row (on the CSR of A^T: diag(A^T A), gauss_newton.py:50-52). */
int gnk_csr_row_sumsq(gnk_ctx* ctx, int64_t n_rows, const int32_t* d_rowptr, const double* d_val,
                      double* d_out, void* stream);

/* Returned by gnk_csr_pattern for an index pattern that is not canonical CSR; gnk_last_error names the first
 * defective row and the defect. */
#define GNK_PATTERN_INVALID 3
/* Validates a CSR index pattern (n_rows x n_cols, nnz non-zeros; int32 or int64 indices, index_bytes = 4 / 8):
 * rowptr[0] = 0, non-decreasing, rowptr[n_rows] = nnz, 0 <= col < n_cols, strictly increasing within a row.  Then
 * writes its int32 copy (rowptr32: n_rows + 1, col32: nnz) and the sorted transpose pattern (rowptr_t: n_cols + 1,
 * col_t: nnz) with perm[e] = the non-zero of A at transpose position e -- a stable radix sort of the non-zeros by
 * column, i.e. scipy's sorted csr_array(A.T).  Replaces the host transpose sp.csr_array(A.T) for Jacobians that live
 * on the device (device.py: DeviceCsrJacobian).  n_rows, n_cols and nnz must be below 2^31 - 1.  Scratch belongs to
 * the context.  Synchronises the stream. */
int gnk_csr_pattern(gnk_ctx* ctx, int64_t n_rows, int64_t n_cols, int64_t nnz, const void* d_rowptr,
                    const void* d_col, int index_bytes, int32_t* d_rowptr32, int32_t* d_col32,
                    int32_t* d_rowptr_t, int32_t* d_col_t, int32_t* d_perm, void* stream);
/* *d_differ = 1 if the candidate pattern (int32 / int64) differs from the int32 copy made by gnk_csr_pattern, else 0
 * (same n_rows and nnz assumed).  Lets a Jacobian with a fixed pattern and new values skip the transpose rebuild. */
int gnk_csr_pattern_equal(gnk_ctx* ctx, int64_t n_rows, int64_t nnz, const void* d_rowptr, const void* d_col,
                          int index_bytes, const int32_t* d_rowptr32, const int32_t* d_col32, int32_t* d_differ,
                          void* stream);
/* out[e] = in[perm[e]] for n doubles: the values of A^T on the pattern of gnk_csr_pattern (replaces the value half of
 * sp.csr_array(A.T) per Jacobian). */
int gnk_csr_gather(gnk_ctx* ctx, int64_t n, const int32_t* d_perm, const double* d_in, double* d_out, void* stream);

/* ---- dense Jacobians (strided CUDA tensors from device callables, used without a CSR form) ---------- */
/* J is n_rows x n_cols (both below 2^31 - 1; n_rows * n_cols may exceed 2^31), entry (i, c) at
 * d_J[i * row_stride + c * col_stride], one of the two strides 1 (row-major or column-major; the other is any
 * stride >= 0).  Every output is sign * (the fma chain from 0.0 over the entries != 0.0 of the row / column of J in
 * ascending index order): bit for bit what gnk_spmm_csr gives on the CSR of J / on the sorted CSR of J^T, which drop
 * exact zeros (+0.0 and -0.0) and keep NaN.  One launch, no synchronisation.
 * gnk_dense_matmat: out[:, j] = sign * J @ in[:, j] for j < k, with in / out columns as in gnk_spmm_csr (d_in + j*in_ld
 * + in_off, d_out + j*out_ld + out_off).  A CTA stages tiles of J and of the basis through shared memory and keeps a
 * register tile of outputs; one pass carries up to 2 / 4 / 16 / 32 basis columns for k <= 2 / 4 / 16 / 32, passes of
 * 64 columns above (k <= 255: at most 4, adjacent in the grid so that J is read from HBM about once).  k = 1 takes a
 * kernel of its own: one chain per row, fed by a four-stage cp.async ring. */
int gnk_dense_matmat(gnk_ctx* ctx, int64_t n_rows, int64_t n_cols, const double* d_J, int64_t row_stride,
                     int64_t col_stride, const double* d_in, int64_t in_ld, int64_t in_off, int k, double sign,
                     double* d_out, int64_t out_ld, int64_t out_off, void* stream);
/* gnk_dense_rmatvec: out[c] = sign * (J^T r)[c], c < n_cols; one sequential chain of n_rows steps per column. */
int gnk_dense_rmatvec(gnk_ctx* ctx, int64_t n_rows, int64_t n_cols, const double* d_J, int64_t row_stride,
                      int64_t col_stride, const double* d_r, double sign, double* d_out, void* stream);
/* gnk_dense_col_sumsq: out[c] = sum_i J[i, c]^2, c < n_cols: the Jacobi diagonal diag(J^T J), bit for bit
 * gnk_csr_row_sumsq on the sorted CSR of J^T (one fma(a, a, acc) chain per column from 0.0, rows ascending). */
int gnk_dense_col_sumsq(gnk_ctx* ctx, int64_t n_rows, int64_t n_cols, const double* d_J, int64_t row_stride,
                        int64_t col_stride, double* d_out, void* stream);

/* ---- small vector algebra used by the full-space solver (gauss_newton.py:123-129) -------------- */
/* out = a*x + b*y over n doubles (x, y, out may alias). */
int gnk_axpby(gnk_ctx* ctx, int64_t n, double a, const double* d_x, double b, const double* d_y,
              double* d_out, void* stream);
int gnk_dot(gnk_ctx* ctx, int64_t n, const double* d_x, const double* d_y, double* d_out, void* stream);

/* ---- CGLS (gauss_newton.py:11-60 on top of scipy.sparse.linalg.cg) ------------------------------ */
typedef struct {
  int32_t kind;      /* 0 = Bratu stencil (A = sign*P), 1 = CSR pair, 2 = dense                     */
  int32_t pad_;
  double sign;       /* A = sign * Op                                                               */
  /* kind 0 */
  gnk_layout lay;
  gnk_bratu prm;
  const double* d_expu;
  /* kind 1: A (n_res x p) as CSR and A^T as CSR; kind 2 uses n_res and p as well */
  int64_t n_res, p;
  const int32_t *d_rowptr, *d_col;
  const double* d_val;
  const int32_t *d_rowptr_t, *d_col_t;
  const double* d_val_t;
  /* kind 2: A dense, read in place, A[i, j] at d_dense[i * row_stride + j * col_stride] with one stride 1 (the
   * layouts of gnk_dense_matmat).  Read only when kind == 2, so a caller that builds the struct without these fields
   * for kind 0 or 1 stays valid. */
  const double* d_dense;
  int64_t row_stride, col_stride;
} gnk_linop;
/* Solves A^T A x = A^T y by Jacobi-preconditioned CG exactly as the reference does, including its
 * quirk (preconditioner == 0 first runs an unpreconditioned CG whose result is discarded and whose
 * iterations are added to *iters).  d_y: residual vector (stencil: stored column, halo >= 1 valid;
 * CSR, dense: n_res doubles).  d_x: result (stencil: stored column; CSR, dense: p doubles).  d_work: at least
 * 7 stored columns (stencil) / 7 * roundup16(max(p, n_res)) doubles (CSR, dense).  A dense operator takes
 * gnk_dense_matmat (k = 1) for A p, gnk_dense_rmatvec for A^T t and gnk_dense_col_sumsq for the Jacobi diagonal: the
 * bits of the CSR pair of the same matrix, without its copy and with no limit on n_res * p; one rank only.
 * Synchronises the stream. */
int gnk_cgls(gnk_ctx* ctx, const gnk_linop* op, const double* d_y, double rtol, int preconditioner,
             double* d_x, double* d_work, int64_t* iters, void* stream);
/* The same with the initial guess that cg_least_squares forwards to scipy's cg (gauss_newton.py:14,46,56: `x0=x0`):
 * both runs start from d_x0 (same layout as d_x, must not alias it; NULL = zero start = gnk_cgls) with
 * r = A^T y - A^T A x0, while the stopping threshold stays rtol * ||A^T y||. */
int gnk_cgls_x0(gnk_ctx* ctx, const gnk_linop* op, const double* d_y, const double* d_x0, double rtol,
                int preconditioner, double* d_x, double* d_work, int64_t* iters, void* stream);

/* The projected least squares of GNK solved by CGLS (BASELINE config 5, "Krylov dim 50 with CGLS inner solve"):
 * cg_least_squares(sign_a * A, y, cg_rtol = rtol, preconditioner = True) of gauss_newton.py:11-60 for the DENSE n_rows x k
 * panel A (column-major, stride lda, k <= 55).  scipy's cg touches A through p -> A^T (A p) (16 n k bytes per CG iteration);
 * here G = A^T A, A^T y and y^T y are formed once (one sweep over the panel on the FP64 tensor pipe, up to 7 column
 * blocks) and the whole recurrence -- x0 = 0, M = 1 / diag(A^T A), stop when |r| < rtol |A^T y| tested at the top of
 * each iteration, at most 10 k iterations -- runs in one single-CTA kernel on the k x k system.  Result block as
 * gnk_tsqr_ls (d, d^T G d = ||A d||^2, ||y - A d||^2, 0, ||d||^2, sqrt(diag G)); d_out[2k+4] = CG iterations taken.
 * With a communicator attached the ranks' Gram matrices are summed in rank order before the iteration. */
int gnk_gram_cgls(gnk_ctx* ctx, const double* d_A, int64_t lda, int64_t n_rows, int k, const double* d_y,
                  double sign_a, double rtol, double* d_out, void* stream);

/* ---- chained Rosenbrock problem on the device (rosenbrock_problem.py:8-19; SURVEY 8f.3) -------------- */
/* F = sqrt2 * [10 (x[1:] - x[:-1]^2) ; 1 - x[:-1]]  (2p-2 values), numpy's rounding order (res, :8-12). */
int gnk_rosenbrock_residual(gnk_ctx* ctx, int64_t p, double sqrt2, const double* d_x, double* d_F, void* stream);
/* values of J(x) (jac, :14-19) in CSR form, 3(p-1) doubles: row i < p-1: (i, -20 sqrt2 x_i), (i+1, 10 sqrt2); row
 * p-1+i: (i, -sqrt2) -- and of J^T in CSR form (row pointer 0, 2, 5, ..., 3j-1, ..., 3(p-1)); the index arrays are
 * fixed and supplied by the host to gnk_spmm_csr. */
int gnk_rosenbrock_jacobian(gnk_ctx* ctx, int64_t p, double sqrt2, const double* d_x, double* d_val,
                            double* d_val_t, void* stream);

/* ---- multi-GPU plumbing (row slabs; SURVEY 8e) -------------------------------------------------- */
/* NCCL is owned by the library: rank 0 calls gnk_comm_unique_id, the 128 bytes travel by any
 * out-of-band channel (the Python host broadcasts them with torch.distributed), every rank calls
 * gnk_comm_init. */
int gnk_comm_unique_id(void* out128);
int gnk_comm_init(gnk_ctx* ctx, const void* id128, int rank, int nranks);
int gnk_comm_size(gnk_ctx* ctx);
/* Peer-memory collectives for the ranks of one NVLink/NVSwitch node (optional, after gnk_comm_init): every rank
 * exports a mailbox in its HBM as a 64-byte CUDA IPC handle, the host gathers the nranks handles (rank order, any
 * out-of-band channel) and attaches them.  From then on gnk_comm_allreduce, the TSQR triangle gather and
 * gnk_comm_halo_exchange are single kernels that store into the peers' mailboxes over NVLink and spin on flags there
 * instead of NCCL calls (same fixed rank-ordered reductions, bitwise identical results).  If either call fails the
 * NCCL path stays in use. */
int gnk_comm_p2p_export(gnk_ctx* ctx, void* out_handle64);
int gnk_comm_p2p_attach(gnk_ctx* ctx, const void* handles /* nranks x 64 bytes */);
int gnk_comm_p2p_enabled(gnk_ctx* ctx);
int gnk_comm_p2p_disable(gnk_ctx* ctx); /* back to the NCCL path (all ranks must call it together) */
/* 1 if, with the mailboxes attached, gnk_bratu_residual (*d_loss), gnk_cgs_dots (d_h) and gnk_cgs_update (d_stats)
 * deliver the value reduced over ALL ranks: the last CTA of those kernels runs the mailbox protocol itself (one kernel
 * for the compute step and its collective), so the host must not call gnk_comm_allreduce on their results.
 * GNK_P2P_FUSED=0 at attach time keeps the reductions as separate single-CTA kernels. */
int gnk_comm_fused_reductions(gnk_ctx* ctx);
/* in-place fixed-order sum (op 0) / max (op 1) of `count` <= 256 doubles over all ranks:
 * all-gather followed by the same rank-ordered reduction everywhere (bitwise identical results). */
int gnk_comm_allreduce(gnk_ctx* ctx, double* d_buf, int count, int op, void* stream);
/* fill the `depth` halo rows of one stored column from the neighbouring ranks' owned rows */
int gnk_comm_halo_exchange(gnk_ctx* ctx, const gnk_layout* lay, double* d_col, int depth, void* stream);
/* d_full (sum of all ranks' n_own, rank order) <- every rank's owned part of a stored column */
int gnk_comm_allgather_owned(gnk_ctx* ctx, const gnk_layout* lay, const double* d_col, double* d_full,
                             const int64_t* counts, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GNK_B200_H */
