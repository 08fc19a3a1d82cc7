// csr.cu -- generic sparse Jacobians: the chained Rosenbrock problem (rosenbrock_problem.py:14-19) and every Jacobian
// a user callable returns, host (scipy / numpy, uploaded) or device (torch CSR / COO / dense CUDA tensors).
//   gnk_spmm_csr           out[:, j] = sign * A * in[:, j]   (J @ V_k, gauss_newton_krylow.py:86; with the CSR of A^T:
//                                                            -J^T r, krylow.py:62)
//   gnk_csr_row_sumsq      per-row sum of squares (on the CSR of A^T: diag(A^T A), gauss_newton.py:50-52)
//   gnk_csr_pattern        validates a CSR index pattern, keeps int32 copies and builds the sorted transpose pattern
//                          plus the permutation transpose position -> source non-zero
//   gnk_csr_pattern_equal  does a candidate index pattern equal the cached one (one device int)
//   gnk_csr_gather         out[e] = in[perm[e]]: the values of A^T for a new A on a cached pattern
// Summation order: one thread walks one row in index order, which is scipy's csr_matvec order; the products of a
// Jacobian with the Krylov basis are sign * (fma chain from 0.0) per (row, column).  At the sizes where a user problem
// pays off on the GPU (millions of rows) that product is bandwidth-bound on the matrix, so a thread owns a block of CB
// basis columns and reads col[e] / val[e] once per block: 12 nnz ceil(k / CB) bytes of matrix traffic instead of 12 nnz k.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>

#include "common.cuh"

namespace {
constexpr int TPB = 128;
constexpr int SPMM_CB = 8;

// columns [blockIdx.y * CB, blockIdx.y * CB + CB) of out; the fma chain of every column is the one-column chain
template <int CB>
__global__ void __launch_bounds__(TPB) spmm_csr_kernel(int64_t n_rows, const int32_t* __restrict__ rowptr,
                                                        const int32_t* __restrict__ col,
                                                        const double* __restrict__ val, const double* __restrict__ in,
                                                        int64_t in_ld, int64_t in_off, int j0, double sign,
                                                        double* __restrict__ out, int64_t out_ld, int64_t out_off) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n_rows) return;
  const int64_t jb = j0 + (int64_t)blockIdx.y * CB;
  const double* x = in + jb * in_ld + in_off;
  double acc[CB];
#pragma unroll
  for (int j = 0; j < CB; ++j) acc[j] = 0.0;
  const int e1 = rowptr[row + 1];
  for (int e = rowptr[row]; e < e1; ++e) {
    const double v = val[e];
    const int64_t c = col[e];
#pragma unroll
    for (int j = 0; j < CB; ++j) acc[j] = fma(v, x[c + j * in_ld], acc[j]);
  }
  double* o = out + jb * out_ld + out_off + row;
#pragma unroll
  for (int j = 0; j < CB; ++j) o[j * out_ld] = sign * acc[j];
}

template <int CB>
cudaError_t launch_spmm(int64_t n_rows, const int32_t* rowptr, const int32_t* col, const double* val, const double* in,
                        int64_t in_ld, int64_t in_off, int j0, int nblk, double sign, double* out, int64_t out_ld,
                        int64_t out_off, cudaStream_t st) {
  dim3 grid((unsigned)ceil_div(n_rows, TPB), nblk);
  spmm_csr_kernel<CB><<<grid, TPB, 0, st>>>(n_rows, rowptr, col, val, in, in_ld, in_off, j0, sign, out, out_ld,
                                            out_off);
  return cudaGetLastError();
}

__global__ void __launch_bounds__(TPB) row_sumsq_kernel(int64_t n_rows, const int32_t* __restrict__ rowptr,
                                                         const double* __restrict__ val, double* __restrict__ out) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n_rows) return;
  double acc = 0.0;
  const int e1 = rowptr[row + 1];
  for (int e = rowptr[row]; e < e1; ++e) acc = fma(val[e], val[e], acc);
  out[row] = acc;
}

// ---- pattern ---------------------------------------------------------------------------------------------------
// defects, in the order a row reports them; the first defect is the smallest (row, kind) key
enum PatternDefect { PD_START = 0, PD_ROWPTR = 1, PD_RANGE = 2, PD_ORDER = 3, PD_DUP = 4, PD_END = 5 };

// one thread per row (and thread 0 for rowptr[0] / rowptr[n]): validates, writes the int32 copies, the row of every
// non-zero, the identity permutation the sort starts from, and the column histogram
template <typename I>
__global__ void __launch_bounds__(TPB) pattern_check_kernel(int64_t n_rows, int64_t n_cols, int64_t nnz,
                                                             const I* __restrict__ rowptr, const I* __restrict__ col,
                                                             int32_t* __restrict__ rowptr32,
                                                             int32_t* __restrict__ col32, int32_t* __restrict__ row_of,
                                                             int32_t* __restrict__ iota, int32_t* __restrict__ hist,
                                                             unsigned long long* __restrict__ defect) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row == 0) {
    if ((int64_t)rowptr[0] != 0) atomicMin(defect, 8ull * 0 + PD_START);
    if ((int64_t)rowptr[n_rows] != nnz) atomicMin(defect, 8ull * (unsigned long long)n_rows + PD_END);
    rowptr32[n_rows] = (int32_t)nnz;
  }
  if (row >= n_rows) return;
  const int64_t a = rowptr[row], b = rowptr[row + 1];
  rowptr32[row] = (int32_t)a;
  if (a < 0 || b < a || b > nnz) {
    atomicMin(defect, 8ull * (unsigned long long)row + PD_ROWPTR);
    return;
  }
  int64_t prev = -1;
  for (int64_t e = a; e < b; ++e) {
    const int64_t c = col[e];
    if (c < 0 || c >= n_cols) {
      atomicMin(defect, 8ull * (unsigned long long)row + PD_RANGE);
      return;
    }
    if (c <= prev) {
      atomicMin(defect, 8ull * (unsigned long long)row + (c == prev ? PD_DUP : PD_ORDER));
      return;
    }
    prev = c;
    col32[e] = (int32_t)c;
    row_of[e] = (int32_t)row;
    iota[e] = (int32_t)e;
    atomicAdd(hist + c, 1);
  }
}

__global__ void __launch_bounds__(TPB) transpose_cols_kernel(int64_t nnz, const int32_t* __restrict__ perm,
                                                              const int32_t* __restrict__ row_of,
                                                              int32_t* __restrict__ col_t) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nnz) col_t[i] = row_of[perm[i]];
}

template <typename I>
__global__ void __launch_bounds__(TPB) pattern_equal_kernel(int64_t n_rows, int64_t nnz, const I* __restrict__ rowptr,
                                                             const I* __restrict__ col,
                                                             const int32_t* __restrict__ rowptr32,
                                                             const int32_t* __restrict__ col32,
                                                             int32_t* __restrict__ differ) {
  const int64_t n = n_rows + 1 > nnz ? n_rows + 1 : nnz;
  bool d = false;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    if (i <= n_rows && (int64_t)rowptr[i] != (int64_t)rowptr32[i]) d = true;
    if (i < nnz && (int64_t)col[i] != (int64_t)col32[i]) d = true;
  }
  if (d) *differ = 1;  // every writer stores the same value
}

__global__ void __launch_bounds__(TPB) gather_kernel(int64_t n, const int32_t* __restrict__ perm,
                                                      const double* __restrict__ in, double* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = in[perm[i]];
}

// scratch of gnk_csr_pattern, owned by the context and grown on demand
int pattern_scratch(gnk_ctx* ctx, size_t bytes) {
  if (bytes <= ctx->pattern_bytes) return 0;
  if (ctx->d_pattern) GNK_CUDA(cudaFree(ctx->d_pattern));
  ctx->d_pattern = nullptr;
  ctx->pattern_bytes = 0;
  GNK_CUDA(cudaMalloc(&ctx->d_pattern, bytes));
  ctx->pattern_bytes = bytes;
  return 0;
}

size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

template <typename I>
int csr_pattern(gnk_ctx* ctx, int64_t n_rows, int64_t n_cols, int64_t nnz, const I* rowptr, const I* col,
                int32_t* rowptr32, int32_t* col32, int32_t* rowptr_t, int32_t* col_t, int32_t* perm,
                cudaStream_t st) {
  int end_bit = 1;
  while (end_bit < 31 && (int64_t(1) << end_bit) < n_cols) ++end_bit;
  size_t sort_bytes = 0, scan_bytes = 0;
  GNK_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (const unsigned*)nullptr, (unsigned*)nullptr,
                                           (const int32_t*)nullptr, (int32_t*)nullptr, (int)nnz, 0, end_bit, st));
  GNK_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (const int32_t*)nullptr, (int32_t*)nullptr,
                                         (int)(n_cols + 1), st));
  // layout: defect word | row_of | iota | sorted keys | histogram | cub temp
  const size_t o_row = 256, o_iota = o_row + align256(4 * (size_t)nnz), o_keys = o_iota + align256(4 * (size_t)nnz),
               o_hist = o_keys + align256(4 * (size_t)nnz), o_tmp = o_hist + align256(4 * (size_t)(n_cols + 1));
  const size_t total = o_tmp + align256(sort_bytes > scan_bytes ? sort_bytes : scan_bytes);
  if (int rc = pattern_scratch(ctx, total)) return rc;
  char* s = static_cast<char*>(ctx->d_pattern);
  auto* defect = reinterpret_cast<unsigned long long*>(s);
  auto* row_of = reinterpret_cast<int32_t*>(s + o_row);
  auto* iota = reinterpret_cast<int32_t*>(s + o_iota);
  auto* keys = reinterpret_cast<unsigned*>(s + o_keys);
  auto* hist = reinterpret_cast<int32_t*>(s + o_hist);
  void* tmp = s + o_tmp;

  GNK_CUDA(cudaMemsetAsync(defect, 0xff, sizeof(unsigned long long), st));
  GNK_CUDA(cudaMemsetAsync(hist, 0, 4 * (size_t)(n_cols + 1), st));
  pattern_check_kernel<I><<<(unsigned)ceil_div(n_rows > 0 ? n_rows : 1, TPB), TPB, 0, st>>>(
      n_rows, n_cols, nnz, rowptr, col, rowptr32, col32, row_of, iota, hist, defect);
  GNK_LAUNCH_CHECK(ctx);
  unsigned long long h_defect = 0;
  GNK_CUDA(cudaMemcpyAsync(&h_defect, defect, sizeof(h_defect), cudaMemcpyDeviceToHost, st));
  GNK_CUDA(cudaStreamSynchronize(st));
  if (h_defect != ~0ull) {
    const long long row = (long long)(h_defect >> 3);
    static const char* what[] = {"rowptr[0] is not 0",
                                 "row pointer decreases or leaves [0, nnz] (rowptr[row + 1] < rowptr[row])",
                                 "column index out of range [0, n_cols)", "column indices not sorted within the row",
                                 "duplicate column index within the row", "rowptr[n_rows] is not nnz"};
    char buf[256];
    snprintf(buf, sizeof buf, "invalid CSR pattern (%lld x %lld, nnz %lld): row %lld: %s", (long long)n_rows,
             (long long)n_cols, (long long)nnz, row, what[h_defect & 7]);
    gnk_set_error(buf);
    return GNK_PATTERN_INVALID;
  }
  if (nnz > 0) {
    // stable: within a column the non-zeros keep their row order, i.e. scipy's sorted transpose
    GNK_CUDA(cub::DeviceRadixSort::SortPairs(tmp, sort_bytes, reinterpret_cast<const unsigned*>(col32), keys, iota,
                                             perm, (int)nnz, 0, end_bit, st));
    ctx->launches++;
    transpose_cols_kernel<<<(unsigned)ceil_div(nnz, TPB), TPB, 0, st>>>(nnz, perm, row_of, col_t);
    GNK_LAUNCH_CHECK(ctx);
  }
  GNK_CUDA(cub::DeviceScan::ExclusiveSum(tmp, scan_bytes, hist, rowptr_t, (int)(n_cols + 1), st));
  ctx->launches++;
  GNK_CUDA(cudaStreamSynchronize(st));
  return 0;
}
}  // namespace

extern "C" {

int gnk_spmm_csr(gnk_ctx* ctx, int64_t n_rows, const int32_t* d_rowptr, const int32_t* d_col, const double* d_val,
                 const double* d_in, int64_t in_ld, int64_t in_off, int k, double sign, double* d_out, int64_t out_ld,
                 int64_t out_off, void* stream) {
  GNK_REQUIRE(ctx && d_rowptr && d_in && d_out, "gnk_spmm_csr: null argument");
  GNK_REQUIRE(k >= 1 && k <= 65535 * SPMM_CB && n_rows >= 0, "gnk_spmm_csr: bad sizes");
  if (n_rows == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const int full = k / SPMM_CB, tail = k % SPMM_CB;
  cudaError_t e = cudaSuccess;
  if (full) {
    e = launch_spmm<SPMM_CB>(n_rows, d_rowptr, d_col, d_val, d_in, in_ld, in_off, 0, full, sign, d_out, out_ld,
                             out_off, st);
    ctx->launches++;
  }
  if (tail && e == cudaSuccess) {
    const int j0 = full * SPMM_CB;
    switch (tail) {
#define GNK_SPMM_TAIL(W)                                                                                           \
  case W:                                                                                                          \
    e = launch_spmm<W>(n_rows, d_rowptr, d_col, d_val, d_in, in_ld, in_off, j0, 1, sign, d_out, out_ld, out_off, st); \
    break;
      GNK_SPMM_TAIL(1) GNK_SPMM_TAIL(2) GNK_SPMM_TAIL(3) GNK_SPMM_TAIL(4) GNK_SPMM_TAIL(5) GNK_SPMM_TAIL(6)
      GNK_SPMM_TAIL(7)
#undef GNK_SPMM_TAIL
    }
    ctx->launches++;
  }
  if (e != cudaSuccess) return gnk_fail("kernel launch", e, __FILE__, __LINE__);
  return 0;
}

int gnk_csr_row_sumsq(gnk_ctx* ctx, int64_t n_rows, const int32_t* d_rowptr, const double* d_val, double* d_out,
                      void* stream) {
  GNK_REQUIRE(ctx && d_rowptr && d_out && n_rows >= 0, "gnk_csr_row_sumsq: bad argument");
  if (n_rows == 0) return 0;
  row_sumsq_kernel<<<(unsigned)ceil_div(n_rows, TPB), TPB, 0, (cudaStream_t)stream>>>(n_rows, d_rowptr, d_val, d_out);
  GNK_LAUNCH_CHECK(ctx);
  return 0;
}

int gnk_csr_pattern(gnk_ctx* ctx, int64_t n_rows, int64_t n_cols, int64_t nnz, const void* d_rowptr, const void* d_col,
                    int index_bytes, int32_t* d_rowptr32, int32_t* d_col32, int32_t* d_rowptr_t, int32_t* d_col_t,
                    int32_t* d_perm, void* stream) {
  GNK_REQUIRE(ctx && d_rowptr && d_rowptr32 && d_rowptr_t, "gnk_csr_pattern: null argument");
  GNK_REQUIRE(nnz == 0 || (d_col && d_col32 && d_col_t && d_perm), "gnk_csr_pattern: null argument");
  GNK_REQUIRE(n_rows >= 0 && n_cols >= 0 && nnz >= 0 && n_rows < INT32_MAX && n_cols < INT32_MAX && nnz < INT32_MAX,
              "gnk_csr_pattern: sizes must be below 2^31 - 1 (int32 indices; the transpose row pointer has n_cols + 1 "
              "entries)");
  GNK_REQUIRE(index_bytes == 4 || index_bytes == 8, "gnk_csr_pattern: indices must be int32 or int64");
  cudaStream_t st = (cudaStream_t)stream;
  if (index_bytes == 4)
    return csr_pattern<int32_t>(ctx, n_rows, n_cols, nnz, (const int32_t*)d_rowptr, (const int32_t*)d_col, d_rowptr32,
                                d_col32, d_rowptr_t, d_col_t, d_perm, st);
  return csr_pattern<int64_t>(ctx, n_rows, n_cols, nnz, (const int64_t*)d_rowptr, (const int64_t*)d_col, d_rowptr32,
                              d_col32, d_rowptr_t, d_col_t, d_perm, st);
}

int gnk_csr_pattern_equal(gnk_ctx* ctx, int64_t n_rows, int64_t nnz, const void* d_rowptr, const void* d_col,
                          int index_bytes, const int32_t* d_rowptr32, const int32_t* d_col32, int32_t* d_differ,
                          void* stream) {
  GNK_REQUIRE(ctx && d_rowptr && d_rowptr32 && d_differ && (nnz == 0 || (d_col && d_col32)),
              "gnk_csr_pattern_equal: null argument");
  GNK_REQUIRE(n_rows >= 0 && nnz >= 0 && (index_bytes == 4 || index_bytes == 8), "gnk_csr_pattern_equal: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  GNK_CUDA(cudaMemsetAsync(d_differ, 0, sizeof(int32_t), st));
  const int64_t n = n_rows + 1 > nnz ? n_rows + 1 : nnz;
  const unsigned grid = (unsigned)std::min<int64_t>(ceil_div(n, TPB), 8 * (int64_t)ctx->sm_count);
  if (index_bytes == 4)
    pattern_equal_kernel<int32_t><<<grid, TPB, 0, st>>>(n_rows, nnz, (const int32_t*)d_rowptr, (const int32_t*)d_col,
                                                        d_rowptr32, d_col32, d_differ);
  else
    pattern_equal_kernel<int64_t><<<grid, TPB, 0, st>>>(n_rows, nnz, (const int64_t*)d_rowptr, (const int64_t*)d_col,
                                                        d_rowptr32, d_col32, d_differ);
  GNK_LAUNCH_CHECK(ctx);
  return 0;
}

int gnk_csr_gather(gnk_ctx* ctx, int64_t n, const int32_t* d_perm, const double* d_in, double* d_out, void* stream) {
  GNK_REQUIRE(ctx && n >= 0 && (n == 0 || (d_perm && d_in && d_out)), "gnk_csr_gather: bad argument");
  if (n == 0) return 0;
  gather_kernel<<<(unsigned)ceil_div(n, TPB), TPB, 0, (cudaStream_t)stream>>>(n, d_perm, d_in, d_out);
  GNK_LAUNCH_CHECK(ctx);
  return 0;
}

}  // extern "C"
