// microbench_spmm_csr.cu -- the column-blocked gnk_spmm_csr of libgnk_b200.so against the one-thread-per-row kernel it
// replaced (held below as old_spmm_kernel, grid.y = k: the matrix is read once per column), side by side:
//   * matrices: the 5-point Bratu CSR at G = 4096 (n = 4095^2 = 16.8 M rows, 84 M non-zeros) and a random CSR of the
//     same row count with skewed row lengths (most rows 1..4 entries, one in 64 rows up to 256);
//   * widths k = 1, 8, 30, 50, 255 where memory allows (input and output panels are n x k doubles each);
//   * every k: the two outputs are compared bit for bit on the device, and each kernel's time (CUDA events, median of
//     5 after a warm-up) is reported with GB/s over its own algorithmic bytes
//       old: 12 nnz k + 8 n_cols k + 8 n_rows k          new: 12 nnz ceil(k/8) + 8 n_cols k + 8 n_rows k
//     (matrix values + column indices per read of the matrix, the input panel read once, the output written once; the
//     row pointer and repeated gathers of in[] that hit the cache are not counted);
//   * gnk_csr_pattern (validation + transpose pattern, synchronous) and gnk_csr_gather at the same size.
// Inputs are far larger than the 126 MB L2.  Stand-alone, linked against the library built by __graft_entry__.build():
//
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -Iinclude -o tools/microbench_spmm_csr \
//        tools/microbench_spmm_csr.cu -Lgauss_newton_via_generalized_krylov_subspaces_b200 -lgnk_b200 \
//        -Xlinker -rpath -Xlinker "$PWD/gauss_newton_via_generalized_krylov_subspaces_b200"
//   tools/microbench_spmm_csr [G=4096]
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <vector>

#include <thrust/device_ptr.h>
#include <thrust/scan.h>

#include "gnk_b200.h"

#define CK(x)                                                                                   \
  do {                                                                                          \
    cudaError_t e_ = (x);                                                                       \
    if (e_ != cudaSuccess) {                                                                    \
      fprintf(stderr, "%s:%d %s: %s\n", __FILE__, __LINE__, #x, cudaGetErrorString(e_));        \
      exit(1);                                                                                  \
    }                                                                                           \
  } while (0)
#define GK(x)                                                                                   \
  do {                                                                                          \
    int r_ = (x);                                                                               \
    if (r_ != 0) {                                                                              \
      fprintf(stderr, "%s:%d %s: rc %d: %s\n", __FILE__, __LINE__, #x, r_, gnk_last_error());   \
      exit(1);                                                                                  \
    }                                                                                           \
  } while (0)

// the kernel gnk_spmm_csr launched before the column blocking (csr.cu of the parent commit), unchanged
__global__ void __launch_bounds__(128) old_spmm_kernel(int64_t n_rows, const int32_t* __restrict__ rowptr,
                                                       const int32_t* __restrict__ col, const double* __restrict__ val,
                                                       const double* __restrict__ in, int64_t in_ld, int64_t in_off,
                                                       double sign, double* __restrict__ out, int64_t out_ld,
                                                       int64_t out_off) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n_rows) return;
  const double* x = in + (int64_t)blockIdx.y * in_ld + in_off;
  double acc = 0.0;
  const int e1 = rowptr[row + 1];
  for (int e = rowptr[row]; e < e1; ++e) acc = fma(val[e], x[col[e]], acc);
  out[(int64_t)blockIdx.y * out_ld + out_off + row] = sign * acc;
}

__device__ __forceinline__ uint64_t mix(uint64_t z) {
  z += 0x9e3779b97f4a7c15ull;
  z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
  z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
  return z ^ (z >> 31);
}
__device__ __forceinline__ double unit(uint64_t h) { return (double)(h >> 11) * (1.0 / 9007199254740992.0) - 0.5; }

__global__ void fill_kernel(double* p, int64_t n, uint64_t seed) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    p[i] = unit(mix(seed * 0x100000001b3ull + (uint64_t)i));
}

// 5-point stencil rows on an m x m grid, columns in ascending order
__global__ void bratu_len_kernel(int64_t m, int32_t* len) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= m * m) return;
  const int64_t i = r / m, j = r % m;
  len[r] = 1 + (i > 0) + (j > 0) + (j < m - 1) + (i < m - 1);
}
__global__ void bratu_fill_kernel(int64_t m, const int32_t* rowptr, int32_t* col, double* val) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= m * m) return;
  const int64_t i = r / m, j = r % m;
  int e = rowptr[r];
  const double c = 4095.0 * 4095.0;
  if (i > 0) col[e] = (int32_t)(r - m), val[e++] = -c;
  if (j > 0) col[e] = (int32_t)(r - 1), val[e++] = -c - 5.0 * 4095.0;
  col[e] = (int32_t)r, val[e++] = 4.0 * c + 10.0 * unit(mix(r));
  if (j < m - 1) col[e] = (int32_t)(r + 1), val[e++] = -c + 5.0 * 4095.0;
  if (i < m - 1) col[e] = (int32_t)(r + m), val[e++] = -c;
}

// skewed rows: 1..4 entries, one row in 64 has 16..256; distinct ascending columns by random strides
__global__ void skew_len_kernel(int64_t n, int32_t* len) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const uint64_t h = mix(r ^ 0x5eedull);
  len[r] = (h & 63) == 0 ? 16 + (int32_t)((h >> 8) % 241) : 1 + (int32_t)((h >> 8) & 3);
}
__global__ void skew_fill_kernel(int64_t n, int64_t n_cols, const int32_t* rowptr, int32_t* col, double* val) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const int e0 = rowptr[r], e1 = rowptr[r + 1];
  const int64_t len = e1 - e0, span = n_cols / 2;
  int64_t c = (int64_t)(mix(r * 7 + 1) % (uint64_t)(n_cols - span));
  const int64_t step = len > 0 && span / len > 1 ? span / len : 1;
  for (int e = e0; e < e1; ++e) {
    col[e] = (int32_t)c;
    val[e] = unit(mix((uint64_t)e * 3 + 11));
    c += 1 + (int64_t)(mix((uint64_t)e) % (uint64_t)step);
  }
}

__global__ void diff_kernel(const double* a, const double* b, int64_t n, unsigned long long* count) {
  unsigned long long d = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    d += __double_as_longlong(a[i]) != __double_as_longlong(b[i]);
  if (d) atomicAdd(count, d);
}

struct Csr {
  const char* name;
  int64_t n_rows, n_cols, nnz;
  int32_t* rowptr;
  int32_t* col;
  double* val;
};

static Csr make_csr(const char* name, int64_t n, bool bratu, int64_t m) {
  Csr A{name, n, n, 0, nullptr, nullptr, nullptr};
  CK(cudaMalloc(&A.rowptr, 4 * (n + 1)));
  const unsigned grid = (unsigned)((n + 255) / 256);
  if (bratu)
    bratu_len_kernel<<<grid, 256>>>(m, A.rowptr);
  else
    skew_len_kernel<<<grid, 256>>>(n, A.rowptr);
  CK(cudaMemset(A.rowptr + n, 0, 4));
  thrust::exclusive_scan(thrust::device_ptr<int32_t>(A.rowptr), thrust::device_ptr<int32_t>(A.rowptr + n + 1),
                         thrust::device_ptr<int32_t>(A.rowptr));
  int32_t nnz = 0;
  CK(cudaMemcpy(&nnz, A.rowptr + n, 4, cudaMemcpyDeviceToHost));
  A.nnz = nnz;
  CK(cudaMalloc(&A.col, 4 * (size_t)nnz));
  CK(cudaMalloc(&A.val, 8 * (size_t)nnz));
  if (bratu)
    bratu_fill_kernel<<<grid, 256>>>(m, A.rowptr, A.col, A.val);
  else
    skew_fill_kernel<<<grid, 256>>>(n, n, A.rowptr, A.col, A.val);
  CK(cudaDeviceSynchronize());
  return A;
}

template <class F>
static float median_ms(F&& launch, int reps = 5) {
  cudaEvent_t a, b;
  CK(cudaEventCreate(&a));
  CK(cudaEventCreate(&b));
  launch();  // warm-up
  CK(cudaDeviceSynchronize());
  std::vector<float> t;
  for (int i = 0; i < reps; ++i) {
    CK(cudaEventRecord(a));
    launch();
    CK(cudaEventRecord(b));
    CK(cudaEventSynchronize(b));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, a, b));
    t.push_back(ms);
  }
  std::sort(t.begin(), t.end());
  CK(cudaEventDestroy(a));
  CK(cudaEventDestroy(b));
  return t[t.size() / 2];
}

int main(int argc, char** argv) {
  const int64_t G = argc > 1 ? atoll(argv[1]) : 4096;
  const int64_t m = G - 1, n = m * m;
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, 0));
  gnk_ctx* ctx = nullptr;
  GK(gnk_create(&ctx, 0));
  printf("device %s, grid %lld^2 (n = %lld)\n", prop.name, (long long)m, (long long)n);
  Csr mats[2] = {make_csr("bratu5", n, true, m), make_csr("skewed", n, false, m)};
  const int ks[] = {1, 8, 30, 50, 255};
  int bad = 0;
  for (const Csr& A : mats) {
    printf("\n%s: %lld x %lld, nnz %lld (%.2f per row)\n", A.name, (long long)A.n_rows, (long long)A.n_cols,
           (long long)A.nnz, (double)A.nnz / A.n_rows);
    printf("%4s %12s %10s %12s %10s %8s %s\n", "k", "old ms", "old GB/s", "blocked ms", "blk GB/s", "speedup", "bitwise");
    for (int k : ks) {
      const size_t panel = 8ull * (size_t)n * k;
      size_t free_b = 0, total_b = 0;
      CK(cudaMemGetInfo(&free_b, &total_b));
      if (3 * panel + (1ull << 30) > free_b) {
        printf("%4d  skipped: 3 panels of %.1f GB do not fit the %.1f GB free\n", k, panel / 1e9, free_b / 1e9);
        continue;
      }
      double *in, *o_old, *o_new;
      CK(cudaMalloc(&in, panel));
      CK(cudaMalloc(&o_old, panel));
      CK(cudaMalloc(&o_new, panel));
      fill_kernel<<<4 * prop.multiProcessorCount, 256>>>(in, (int64_t)n * k, 1234 + k);
      const dim3 grid_old((unsigned)((n + 127) / 128), k);
      const float t_old = median_ms([&] {
        old_spmm_kernel<<<grid_old, 128>>>(n, A.rowptr, A.col, A.val, in, n, 0, -1.0, o_old, n, 0);
      });
      CK(cudaGetLastError());
      const float t_new = median_ms([&] {
        GK(gnk_spmm_csr(ctx, n, A.rowptr, A.col, A.val, in, n, 0, k, -1.0, o_new, n, 0, nullptr));
      });
      unsigned long long* d_count;
      CK(cudaMalloc(&d_count, 8));
      CK(cudaMemset(d_count, 0, 8));
      diff_kernel<<<4 * prop.multiProcessorCount, 256>>>(o_old, o_new, (int64_t)n * k, d_count);
      unsigned long long diffs = 0;
      CK(cudaMemcpy(&diffs, d_count, 8, cudaMemcpyDeviceToHost));
      CK(cudaFree(d_count));
      const double io = 8.0 * (double)A.n_cols * k + 8.0 * (double)A.n_rows * k;
      const double b_old = 12.0 * A.nnz * k + io, b_new = 12.0 * A.nnz * ((k + 7) / 8) + io;
      printf("%4d %12.3f %10.1f %12.3f %10.1f %8.2f %s\n", k, t_old, b_old / t_old / 1e6, t_new, b_new / t_new / 1e6,
             t_old / t_new, diffs ? "DIFFER" : "equal");
      if (diffs) {
        printf("     %llu of %lld entries differ\n", diffs, (long long)n * k);
        bad = 1;
      }
      CK(cudaFree(in));
      CK(cudaFree(o_old));
      CK(cudaFree(o_new));
    }
    // pattern (validation + transpose) and the J^T value gather at this size
    int32_t *rp32, *c32, *rpt, *ct, *perm;
    double* vt;
    CK(cudaMalloc(&rp32, 4 * (A.n_rows + 1)));
    CK(cudaMalloc(&c32, 4 * A.nnz));
    CK(cudaMalloc(&rpt, 4 * (A.n_cols + 1)));
    CK(cudaMalloc(&ct, 4 * A.nnz));
    CK(cudaMalloc(&perm, 4 * A.nnz));
    CK(cudaMalloc(&vt, 8 * A.nnz));
    const float t_pat = median_ms([&] {
      GK(gnk_csr_pattern(ctx, A.n_rows, A.n_cols, A.nnz, A.rowptr, A.col, 4, rp32, c32, rpt, ct, perm, nullptr));
    });
    const float t_gat = median_ms([&] { GK(gnk_csr_gather(ctx, A.nnz, perm, A.val, vt, nullptr)); });
    int32_t* d_diff;
    CK(cudaMalloc(&d_diff, 4));
    const float t_eq = median_ms([&] {
      GK(gnk_csr_pattern_equal(ctx, A.n_rows, A.nnz, A.rowptr, A.col, 4, rp32, c32, d_diff, nullptr));
    });
    int32_t differ = -1;
    CK(cudaMemcpy(&differ, d_diff, 4, cudaMemcpyDeviceToHost));
    printf("gnk_csr_pattern %.3f ms (synchronous: validation, radix sort, scan) | gnk_csr_pattern_equal %.3f ms "
           "(%.1f GB/s over 8 (n + nnz), same pattern -> %d) | gnk_csr_gather %.3f ms (%.1f GB/s over 20 nnz)\n",
           t_pat, t_eq, 8.0 * (A.n_rows + A.nnz) / t_eq / 1e6, differ, t_gat, 20.0 * A.nnz / t_gat / 1e6);
    if (differ != 0) bad = 1;
    for (void* p : {(void*)rp32, (void*)c32, (void*)rpt, (void*)ct, (void*)perm, (void*)vt, (void*)d_diff})
      CK(cudaFree(p));
  }
  for (Csr& A : mats) {
    CK(cudaFree(A.rowptr));
    CK(cudaFree(A.col));
    CK(cudaFree(A.val));
  }
  GK(gnk_destroy(ctx));
  printf("%s\n", bad ? "FAILED: outputs differ" : "all outputs bitwise equal");
  return bad;
}
