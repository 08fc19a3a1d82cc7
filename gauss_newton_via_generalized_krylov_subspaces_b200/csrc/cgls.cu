// cgls.cu -- cg_least_squares (gauss_newton.py:11-60): conjugate gradients on A^T A x = A^T y with the
// Jacobi preconditioner 1/diag(A^T A), following scipy 1.18.1 sparse.linalg.cg step by step
// (_isolve/iterative.py:383-430: x0 = 0, r = b, stop when ||r||_2 < rtol*||b||_2 tested at the top of each
// iteration, maxiter = 10 p).  The reference's quirk is kept: preconditioner == 0 first runs an
// unpreconditioned CG whose solution is thrown away (gauss_newton.py:45-48) and then ALWAYS runs the
// preconditioned one (:50-58); the reported iteration count is the sum.
// A = sign*P for the Bratu stencil (matrix free; A p and A^T t are the same SpMV / SpMV-transpose kernels the
// Krylov path uses), a CSR pair for generic Jacobians, or a dense matrix read in place (the dense_jac.cu kernels, which
// give the bits of the CSR pair of the same matrix).  All scalars (rho, p.q, alpha, beta) stay on the
// device; the host reads one double (||r||^2) per iteration for the stopping test -- one iteration LATE: iteration i + 1
// is queued before the test of iteration i is looked at, and the two kernels that change the CG state (direction, step)
// repeat the test on the device and do nothing once it has fired, so the device never waits for the host and the result
// is the one scipy's loop produces.
#include <math.h>
#include <stdlib.h>

#include "common.cuh"

int gnk_comm_allgather_doubles(gnk_ctx* ctx, const double* d_send, double* d_recv, int64_t count, void* stream);

namespace {
constexpr int TPB = 256;
// (rr, rho) of iteration i live in slot pair S_RR + 8 (i & 1) .. so that the late read of iteration i cannot see i + 1's
enum { S_RR = 0, S_RHO = 1, S_RHO_PREV = 2, S_PQ = 3, S_BB = 4, S_ALT = 8 };

// z = minv * r (or r), rr = r.r, rho = r.z
__global__ void __launch_bounds__(TPB) cg_precond_kernel(int64_t n, const double* __restrict__ r,
                                                          const double* __restrict__ minv, double* __restrict__ z,
                                                          double* __restrict__ partials, unsigned int* ticket,
                                                          double* __restrict__ scal) {
  __shared__ double sh[32];
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  double rr = 0.0, rho = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const double ri = r[i];
    const double zi = minv ? ri * minv[i] : ri;
    z[i] = zi;
    rr = fma(ri, ri, rr);
    rho = fma(ri, zi, rho);
  }
  rr = block_sum(rr, sh);
  rho = block_sum(rho, sh);
  if (threadIdx.x == 0) {
    partials[2 * blockIdx.x] = rr;
    partials[2 * blockIdx.x + 1] = rho;
  }
  if (grid_arrive_last(ticket)) {
    double a = 0.0, b = 0.0;
    for (int i = threadIdx.x; i < (int)gridDim.x; i += blockDim.x) {
      a += __ldcg(partials + 2 * i);
      b += __ldcg(partials + 2 * i + 1);
    }
    a = block_sum(a, sh);
    b = block_sum(b, sh);
    if (threadIdx.x == 0) {
      scal[S_RR] = a;
      scal[S_RHO] = b;
    }
  }
}

// p = z + (rho/rho_prev) p   (first: p = z)
// rrho = (rr, rho) of this iteration; a no-op once the stopping test sqrt(rr) < atol has fired (the host learns one
// iteration later and stops queueing)
__global__ void __launch_bounds__(TPB) cg_direction_kernel(int64_t n, const double* __restrict__ z,
                                                            double* __restrict__ p, const double* __restrict__ scal,
                                                            const double* __restrict__ rrho, double atol, int first) {
  if (sqrt(rrho[0]) < atol) return;
  const double beta = first ? 0.0 : rrho[1] / scal[S_RHO_PREV];
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    p[i] = first ? z[i] : fma(beta, p[i], z[i]);
}

// x += alpha p, r -= alpha q, alpha = rho / p.q ; afterwards rho_prev <- rho
__global__ void __launch_bounds__(TPB) cg_step_kernel(int64_t n, const double* __restrict__ p,
                                                       const double* __restrict__ q, double* __restrict__ x,
                                                       double* __restrict__ r, double* __restrict__ scal,
                                                       const double* __restrict__ rrho, double atol) {
  if (sqrt(rrho[0]) < atol) return;
  const double rho = rrho[1];
  const double alpha = rho / scal[S_PQ];
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    x[i] = fma(alpha, p[i], x[i]);
    r[i] = fma(-alpha, q[i], r[i]);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) scal[S_RHO_PREV] = rho;  // S_RHO_PREV is read by no thread here
}

__global__ void __launch_bounds__(TPB) reciprocal_kernel(int64_t n, const double* __restrict__ a,
                                                          double* __restrict__ out) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = 1.0 / a[i];
}

struct Cg {
  gnk_ctx* ctx;
  const gnk_linop* op;
  cudaStream_t st;
  int64_t np;      // solution-space length handled by the vector kernels
  int64_t sol_off; // offset of the owned part inside a solution-space vector
  int grid;
  double* scal;

  int apply(const double* in, double* out, int transpose) {
    if (op->kind == 0) {
      if (ctx->nranks > 1) {
        int rc = gnk_comm_halo_exchange(ctx, &op->lay, const_cast<double*>(in), 1, st);
        if (rc) return rc;
      }
      return gnk_stencil_apply(ctx, &op->lay, &op->prm, op->d_expu, in, op->lay.ld, 1, op->sign, transpose, out,
                               op->lay.ld, op->lay.off, st);
    }
    if (op->kind == 2) {
      if (!transpose)
        return gnk_dense_matmat(ctx, op->n_res, op->p, op->d_dense, op->row_stride, op->col_stride, in, 0, 0, 1,
                                op->sign, out, 0, 0, st);
      return gnk_dense_rmatvec(ctx, op->n_res, op->p, op->d_dense, op->row_stride, op->col_stride, in, op->sign, out,
                               st);
    }
    if (!transpose)
      return gnk_spmm_csr(ctx, op->n_res, op->d_rowptr, op->d_col, op->d_val, in, 0, 0, 1, op->sign, out, 0, 0, st);
    return gnk_spmm_csr(ctx, op->p, op->d_rowptr_t, op->d_col_t, op->d_val_t, in, 0, 0, 1, op->sign, out, 0, 0, st);
  }
  int reduce(double* d, int count) {
    if (ctx->nranks == 1) return 0;
    return gnk_comm_allreduce(ctx, d, count, 0, st);
  }
  // late read of the stopping test: copy rrho[0] on the context's copy stream behind the work queued so far (slot s of
  // two); wait(s) blocks until that copy has landed
  int fetch(const double* rrho, int s) {
    if (int rc = gnk_ensure_fetch_stream(ctx)) return rc;
    for (int e = 0; e < 4; ++e)
      if (!ctx->cg_event[e]) GNK_CUDA(cudaEventCreateWithFlags(&ctx->cg_event[e], cudaEventDisableTiming));
    GNK_CUDA(cudaEventRecord(ctx->cg_event[s], st));
    GNK_CUDA(cudaStreamWaitEvent(ctx->fetch_stream, ctx->cg_event[s], 0));
    GNK_CUDA(cudaMemcpyAsync(ctx->h_pinned + 8 + s, rrho, sizeof(double), cudaMemcpyDeviceToHost, ctx->fetch_stream));
    GNK_CUDA(cudaEventRecord(ctx->cg_event[2 + s], ctx->fetch_stream));
    return 0;
  }
  int wait(int s, double* host) {
    GNK_CUDA(cudaEventSynchronize(ctx->cg_event[2 + s]));
    *host = ctx->h_pinned[8 + s];
    return 0;
  }
  int read(int slot, int count, double* host) {
    GNK_CUDA(cudaMemcpyAsync(ctx->h_pinned, scal + slot, sizeof(double) * count, cudaMemcpyDeviceToHost, st));
    GNK_CUDA(cudaStreamSynchronize(st));
    for (int i = 0; i < count; ++i) host[i] = ctx->h_pinned[i];
    return 0;
  }
};

}  // namespace

extern "C" int gnk_cgls_x0(gnk_ctx* ctx, const gnk_linop* op, const double* d_y, const double* d_x0, double rtol,
                           int preconditioner, double* d_x, double* d_work, int64_t* iters, void* stream) {
  GNK_REQUIRE(ctx && op && d_y && d_x && d_work && iters, "gnk_cgls: null argument");
  GNK_REQUIRE(d_x0 != d_x, "gnk_cgls: x0 and x must not alias (x0 is read again by the second run)");
  GNK_REQUIRE(op->kind == 0 || op->kind == 1 || op->kind == 2, "gnk_cgls: unknown operator kind");
  GNK_REQUIRE(op->kind != 2 || ctx->nranks == 1, "gnk_cgls: a dense operator runs on one rank");
  Cg cg;
  cg.ctx = ctx;
  cg.op = op;
  cg.st = (cudaStream_t)stream;
  cg.scal = ctx->d_partials + PART_SCAL;
  int64_t vlen, p_glob;  // stride between work vectors, global unknown count (for maxiter)
  if (op->kind == 0) {
    cg.np = op->lay.n_own;
    cg.sol_off = op->lay.off;
    vlen = op->lay.ld;
    p_glob = (int64_t)op->lay.m * op->lay.m;
  } else {
    cg.np = op->p;
    cg.sol_off = 0;
    vlen = (op->p > op->n_res ? op->p : op->n_res);
    vlen = (vlen + 15) / 16 * 16;
    p_glob = op->p;
  }
  int64_t g = ceil_div(cg.np, TPB);
  if (g > (int64_t)ctx->sm_count * 8) g = (int64_t)ctx->sm_count * 8;
  if (g < 1) g = 1;
  cg.grid = (int)g;
  double* b = d_work;
  double* r = d_work + vlen;
  double* z = d_work + 2 * vlen;
  double* pv = d_work + 3 * vlen;
  double* q = d_work + 4 * vlen;
  double* t = d_work + 5 * vlen;     // residual-space temporary A p
  double* dinv = d_work + 6 * vlen;  // Jacobi preconditioner 1/diag(A^T A)
  const int64_t o = cg.sol_off, n = cg.np;
  cudaStream_t st = cg.st;
  double* part = ctx->d_partials + PART_CG;
  // zero the work vectors (halo rows of stencil columns must be zero / defined)
  GNK_CUDA(cudaMemsetAsync(d_work, 0, sizeof(double) * 7 * vlen, st));
  // b = A^T y
  if (int rc = cg.apply(d_y, b, 1)) return rc;
  if (int rc = gnk_dot(ctx, n, b + o, b + o, cg.scal + S_BB, st)) return rc;
  if (int rc = cg.reduce(cg.scal + S_BB, 1)) return rc;
  double bb;
  if (int rc = cg.read(S_BB, 1, &bb)) return rc;
  *iters = 0;
  const double bn = sqrt(bb);
  if (bn == 0.0) {  // scipy returns the zero vector b itself (postprocess(b)), whatever x0 was
    GNK_CUDA(cudaMemcpyAsync(d_x + o, b + o, sizeof(double) * n, cudaMemcpyDeviceToDevice, st));
    return 0;
  }
  const double atol = rtol * bn;
  const int64_t maxiter = 10 * p_glob;
  for (int pass = (preconditioner ? 1 : 0); pass < 2; ++pass) {
    const bool use_m = (pass == 1);
    if (use_m) {
      if (op->kind == 0) {
        if (int rc = gnk_stencil_normal_diag(ctx, &op->lay, &op->prm, op->d_expu, dinv, st)) return rc;
        // diag((sign P)^T (sign P)) = sign^2 diag(P^T P)
        if (op->sign * op->sign != 1.0)
          if (int rc = gnk_axpby(ctx, n, op->sign * op->sign, dinv + o, 0.0, nullptr, dinv + o, st)) return rc;
      } else {
        if (op->kind == 1) {
          if (int rc = gnk_csr_row_sumsq(ctx, op->p, op->d_rowptr_t, op->d_val_t, dinv, st)) return rc;
        } else {
          if (int rc = gnk_dense_col_sumsq(ctx, op->n_res, op->p, op->d_dense, op->row_stride, op->col_stride, dinv, st))
            return rc;
        }
        if (op->sign * op->sign != 1.0)
          if (int rc = gnk_axpby(ctx, n, op->sign * op->sign, dinv, 0.0, nullptr, dinv, st)) return rc;
      }
      reciprocal_kernel<<<cg.grid, TPB, 0, st>>>(n, dinv + o, dinv + o);
      GNK_LAUNCH_CHECK(ctx);
    }
    if (d_x0) {
      // scipy's cg with an initial guess: x = x0, r = b - A^T A x0; the tolerance stays relative to |b|
      GNK_CUDA(cudaMemcpyAsync(d_x + o, d_x0 + o, sizeof(double) * n, cudaMemcpyDeviceToDevice, st));
      if (int rc = cg.apply(d_x, t, 0)) return rc;
      if (int rc = cg.apply(t, q, 1)) return rc;
      if (int rc = gnk_axpby(ctx, n, 1.0, b + o, -1.0, q + o, r + o, st)) return rc;
    } else {
      GNK_CUDA(cudaMemsetAsync(d_x + o, 0, sizeof(double) * n, st));
      GNK_CUDA(cudaMemcpyAsync(r + o, b + o, sizeof(double) * n, cudaMemcpyDeviceToDevice, st));
    }
    static const bool pipelined = !(getenv("GNK_CG_PIPELINE") && atoi(getenv("GNK_CG_PIPELINE")) == 0);
    int64_t done_at = -1;  // the first iteration whose stopping test fired
    int64_t it = 0;
    for (; it < maxiter; ++it) {
      const int s = (int)(it & 1);
      double* rrho = cg.scal + S_RR + S_ALT * s;
      cg_precond_kernel<<<cg.grid, TPB, 0, st>>>(n, r + o, use_m ? dinv + o : nullptr, z + o, part,
                                                 ctx->d_tickets + TK_CG, rrho);
      GNK_LAUNCH_CHECK(ctx);
      if (int rc = cg.reduce(rrho, 2)) return rc;
      if (int rc = cg.fetch(rrho, s)) return rc;                 // ||r||^2 of iteration `it`, looked at one iteration later
      if (!pipelined) {  // GNK_CG_PIPELINE=0: look at it now (the device idles while the host waits and re-queues)
        double rr_now;
        if (int rc = cg.wait(s, &rr_now)) return rc;
        if (sqrt(rr_now) < atol) {
          done_at = it;
          break;
        }
      } else if (it > 0) {
        double rr_prev;
        if (int rc = cg.wait(1 - s, &rr_prev)) return rc;
        if (sqrt(rr_prev) < atol) {  // iteration it - 1 had converged: its direction / step kernels did nothing
          done_at = it - 1;
          break;
        }
      }
      cg_direction_kernel<<<cg.grid, TPB, 0, st>>>(n, z + o, pv + o, cg.scal, rrho, atol, it == 0 ? 1 : 0);
      GNK_LAUNCH_CHECK(ctx);
      if (int rc = cg.apply(pv, t, 0)) return rc;
      if (int rc = cg.apply(t, q, 1)) return rc;
      if (int rc = gnk_dot(ctx, n, pv + o, q + o, cg.scal + S_PQ, st)) return rc;
      if (int rc = cg.reduce(cg.scal + S_PQ, 1)) return rc;
      cg_step_kernel<<<cg.grid, TPB, 0, st>>>(n, pv + o, q + o, d_x + o, r + o, cg.scal, rrho, atol);
      GNK_LAUNCH_CHECK(ctx);
    }
    if (pipelined && done_at < 0 && it > 0) {  // ran into maxiter: the test of the last queued iteration has not been looked at yet
      double rr_last;
      if (int rc = cg.wait((int)((it - 1) & 1), &rr_last)) return rc;
      if (sqrt(rr_last) < atol) done_at = it - 1;
    }
    *iters += (done_at >= 0) ? done_at : it;
  }
  GNK_CUDA(cudaStreamSynchronize(st));
  return 0;
}

extern "C" int gnk_cgls(gnk_ctx* ctx, const gnk_linop* op, const double* d_y, double rtol, int preconditioner,
                        double* d_x, double* d_work, int64_t* iters, void* stream) {
  return gnk_cgls_x0(ctx, op, d_y, nullptr, rtol, preconditioner, d_x, d_work, iters, stream);
}
