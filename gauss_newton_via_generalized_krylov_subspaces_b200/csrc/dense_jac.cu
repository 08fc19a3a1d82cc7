// dense_jac.cu -- dense Jacobians that device callables return as strided CUDA tensors, used as they arrive: no CSR
// form, no index pattern, no copy of J^T.
//   gnk_dense_matmat   out[:, j] = sign * J @ in[:, j], j < k      (J @ V_k, gauss_newton_krylow.py:86; J d of the
//                                                                  Armijo rule, gauss_newton.py)
//   gnk_dense_rmatvec  out = sign * J^T @ r                        (-J^T r, krylow.py:62)
//   gnk_dense_col_sumsq out[c] = sum_i J[i, c]^2                    (diag(A^T A), the Jacobi preconditioner of
//                                                                  cg_least_squares, gauss_newton.py:50-52)
// Bits: every output is sign * acc, acc an fma chain from 0.0 over the NON-ZERO entries of its row of J (matmat) or
// column of J (rmatvec) in ascending index order -- exactly what gnk_spmm_csr computes on the CSR of J resp. on the
// sorted CSR of J^T, because CSR drops exact zeros (+0.0 and -0.0) and keeps NaN.  So an entry a takes part iff
// a != 0.0.  gnk_dense_col_sumsq is the fma(a, a, acc) chain of gnk_csr_row_sumsq on the sorted CSR of J^T (skipping
// +-0.0 cannot change that sum; NaN is kept).  No FP64 tensor-core MMA: its partial sums round differently.
#include "common.cuh"

namespace {

__device__ __forceinline__ void cp_async8(void* smem, const double* gmem, bool valid) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(d), "l"(gmem), "r"(valid ? 8 : 0) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ---- J @ V ------------------------------------------------------------------------------------------------------
// One CTA of 256 threads owns BM = NY * TM rows and BN = NX * TN basis columns; a thread owns TM rows x TN columns
// (rows ty + NY i, columns tx + NX j; ty varies fastest over the lanes, so the stores of a column are coalesced) and
// keeps their TM x TN chains in registers.  The chain dimension (the columns of J) is walked in chunks of BK: a
// BM x BK tile of J and a BK x BN tile of V are staged into shared memory with cp.async (double buffered), J's tile
// transposed so that the TM values a thread needs at one chain step are a conflict-free read.  The loads are
// coalesced for either layout of J: along a row for row-major J, along a column for column-major J.  Entries outside
// J are zero-filled, which the chains skip, and columns of V beyond k are never stored.
// k > BN runs ceil(k / BN) passes; the passes of one row tile are adjacent in the (1-D) grid, so they run at the same
// time and the tile is read from HBM once and from L2 by the other passes.
constexpr int MM_THREADS = 256;

template <int TM, int TN, int NX, int BK, bool ROW_MAJOR>
__global__ void __launch_bounds__(MM_THREADS) dense_matmat_kernel(int64_t n_rows, int64_t n_cols,
                                                                   const double* __restrict__ J, int64_t rs, int64_t cs,
                                                                   const double* __restrict__ in, int64_t in_ld,
                                                                   int64_t in_off, int k, int passes, double sign,
                                                                   double* __restrict__ out, int64_t out_ld,
                                                                   int64_t out_off) {
  constexpr int NY = MM_THREADS / NX, BM = NY * TM, BN = NX * TN;
  __shared__ double Js[2][BK][BM + 1];
  __shared__ double Vs[2][BK][BN + 1];
  const int tid = threadIdx.x, ty = tid % NY, tx = tid / NY;
  const int64_t pass = blockIdx.x % passes, row0 = (int64_t)(blockIdx.x / passes) * BM;
  const int64_t j0 = pass * BN;

  auto load = [&](int buf, int64_t c0) {
    for (int e = tid; e < BM * BK; e += MM_THREADS) {
      const int i = ROW_MAJOR ? e / BK : e % BM, c = ROW_MAJOR ? e % BK : e / BM;
      const int64_t r = row0 + i, cc = c0 + c;
      const bool ok = r < n_rows && cc < n_cols;
      cp_async8(&Js[buf][c][i], ok ? J + r * rs + cc * cs : J, ok);
    }
    for (int e = tid; e < BK * BN; e += MM_THREADS) {
      const int c = e % BK, j = e / BK;
      const int64_t cc = c0 + c, jj = j0 + j;
      const bool ok = cc < n_cols && jj < k;
      cp_async8(&Vs[buf][c][j], ok ? in + jj * in_ld + in_off + cc : in, ok);
    }
  };

  double acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.0;

  const int64_t chunks = (n_cols + BK - 1) / BK;
  if (chunks > 0) load(0, 0);
  cp_async_commit();
  for (int64_t t = 0; t < chunks; ++t) {
    const int buf = (int)(t & 1);
    if (t + 1 < chunks) load(buf ^ 1, (t + 1) * BK);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
#pragma unroll 4
    for (int c = 0; c < BK; ++c) {
      double a[TM], v[TN];
#pragma unroll
      for (int i = 0; i < TM; ++i) a[i] = Js[buf][c][ty + NY * i];
#pragma unroll
      for (int j = 0; j < TN; ++j) v[j] = Vs[buf][c][tx + NX * j];
#pragma unroll
      for (int i = 0; i < TM; ++i)
        if (a[i] != 0.0) {
#pragma unroll
          for (int j = 0; j < TN; ++j) acc[i][j] = fma(a[i], v[j], acc[i][j]);
        }
    }
    __syncthreads();
  }
#pragma unroll
  for (int j = 0; j < TN; ++j) {
    const int64_t col = j0 + tx + NX * j;
    if (col >= k) continue;
#pragma unroll
    for (int i = 0; i < TM; ++i) {
      const int64_t r = row0 + ty + NY * i;
      if (r < n_rows) out[col * out_ld + out_off + r] = sign * acc[i][j];
    }
  }
}

template <int TM, int TN, int NX, int BK>
cudaError_t launch_matmat(bool row_major, int64_t n_rows, int64_t n_cols, const double* J, int64_t rs, int64_t cs,
                          const double* in, int64_t in_ld, int64_t in_off, int k, double sign, double* out,
                          int64_t out_ld, int64_t out_off, cudaStream_t st) {
  constexpr int BM = (MM_THREADS / NX) * TM, BN = NX * TN;
  const int passes = (k + BN - 1) / BN;
  const int64_t blocks = ceil_div(n_rows, BM) * passes;
  if (blocks > INT32_MAX) return cudaErrorInvalidConfiguration;
  if (row_major)
    dense_matmat_kernel<TM, TN, NX, BK, true><<<(unsigned)blocks, MM_THREADS, 0, st>>>(
        n_rows, n_cols, J, rs, cs, in, in_ld, in_off, k, passes, sign, out, out_ld, out_off);
  else
    dense_matmat_kernel<TM, TN, NX, BK, false><<<(unsigned)blocks, MM_THREADS, 0, st>>>(
        n_rows, n_cols, J, rs, cs, in, in_ld, in_off, k, passes, sign, out, out_ld, out_off);
  return cudaGetLastError();
}

// ---- J @ v, one column (k = 1: the A p of every CG iteration, the J d of the Armijo rule) -----------------------
// The smallest dense_matmat_kernel configuration carries two basis columns, one stage of look-ahead and 256 rows per
// CTA; with few rows (8192 x 8192) that leaves most SMs idle: 0.07 of the HBM bound on a B200, against 0.33 here.  On
// tall matrices both reach 0.50 (DESIGN.md section 6).  Here a CTA owns BM rows, one chain per row run by threads 0..BM-1, and all 256 threads
// keep MV_STAGES - 1 tiles of BM rows x BK = MV_TILE / BM columns (and the matching entries of v) in flight with
// cp.async, coalesced along rows for row-major J and along columns for column-major J.  Each thread issues its loads
// at the same place of every tile, so its addresses advance by a constant.  Few rows (fewer CTAs than the SMs can
// hold) take BM = 32: more CTAs, and 512-byte row segments.
constexpr int MV_THREADS = 256, MV_TILE = 2048, MV_STAGES = 4;

constexpr size_t matvec_smem(int bm) { return sizeof(double) * MV_STAGES * (MV_TILE / bm) * (bm + 2); }

template <int BM, bool ROW_MAJOR>
__global__ void __launch_bounds__(MV_THREADS) dense_matvec_kernel(int64_t n_rows, int64_t n_cols,
                                                                   const double* __restrict__ J, int64_t rs,
                                                                   int64_t cs, const double* __restrict__ v,
                                                                   double sign, double* __restrict__ out) {
  constexpr int BK = MV_TILE / BM, PER = MV_TILE / MV_THREADS;
  static_assert(MV_THREADS % BM == 0 && MV_THREADS % BK == 0, "tile mapping");
  extern __shared__ double mv_smem[];
  auto Js = reinterpret_cast<double(*)[BK][BM + 1]>(mv_smem);              // [MV_STAGES][BK][BM + 1], J transposed
  auto Xs = reinterpret_cast<double(*)[BK]>(mv_smem + MV_STAGES * BK * (BM + 1));  // [MV_STAGES][BK]
  const int tid = threadIdx.x;
  const int64_t row0 = (int64_t)blockIdx.x * BM;
  const int64_t tiles = (n_cols + BK - 1) / BK;
  // load m of this thread in every tile: row i0 + m * DI, column c0 + m * DC of the tile
  const int i0 = ROW_MAJOR ? tid / BK : tid % BM, c0 = ROW_MAJOR ? tid % BK : tid / BM;
  constexpr int DI = ROW_MAJOR ? MV_THREADS / BK : 0, DC = ROW_MAJOR ? 0 : MV_THREADS / BM;

  auto load = [&](int64_t t) {
    if (t >= tiles) return;
    const int buf = (int)(t % MV_STAGES);
    const int64_t cb = t * BK;
#pragma unroll
    for (int m = 0; m < PER; ++m) {
      const int i = i0 + m * DI, c = c0 + m * DC;
      const int64_t rr = row0 + i, cc = cb + c;
      const bool ok = rr < n_rows && cc < n_cols;
      cp_async8(&Js[buf][c][i], ok ? J + rr * rs + cc * cs : J, ok);
    }
    if (tid < BK) {
      const bool ok = cb + tid < n_cols;
      cp_async8(&Xs[buf][tid], ok ? v + cb + tid : v, ok);
    }
  };

#pragma unroll
  for (int s = 0; s < MV_STAGES - 1; ++s) {
    load(s);
    cp_async_commit();
  }
  double acc = 0.0;
  for (int64_t t = 0; t < tiles; ++t) {
    cp_async_wait<MV_STAGES - 2>();
    __syncthreads();  // tile t has landed, and the chains of tile t - 1 are done with their buffer
    load(t + MV_STAGES - 1);
    cp_async_commit();
    if (tid < BM) {
      const int buf = (int)(t % MV_STAGES);
#pragma unroll
      for (int c = 0; c < BK; ++c) {
        const double a = Js[buf][c][tid];
        if (a != 0.0) acc = fma(a, Xs[buf][c], acc);
      }
    }
  }
  if (tid < BM && row0 + tid < n_rows) out[row0 + tid] = sign * acc;
}

template <int BM>
int launch_matvec(gnk_ctx* ctx, bool row_major, int64_t n_rows, int64_t n_cols, const double* J, int64_t rs,
                  int64_t cs, const double* v, double sign, double* out, cudaStream_t st) {
  auto kern = row_major ? dense_matvec_kernel<BM, true> : dense_matvec_kernel<BM, false>;
  static bool attr_set[2][64] = {};  // per layout and device
  bool& set = attr_set[row_major ? 1 : 0][ctx->device & 63];
  if (!set) {
    GNK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)matvec_smem(BM)));
    set = true;
  }
  const int64_t blocks = ceil_div(n_rows, BM);
  if (blocks > INT32_MAX) return gnk_fail("kernel launch", cudaErrorInvalidConfiguration, __FILE__, __LINE__);
  kern<<<(unsigned)blocks, MV_THREADS, matvec_smem(BM), st>>>(n_rows, n_cols, J, rs, cs, v, sign, out);
  GNK_LAUNCH_CHECK(ctx);
  return 0;
}

int launch_matvec_sized(gnk_ctx* ctx, bool row_major, int64_t n_rows, int64_t n_cols, const double* J, int64_t rs,
                        int64_t cs, const double* v, double sign, double* out, cudaStream_t st) {
  if (ceil_div(n_rows, 256) >= 3 * (int64_t)ctx->sm_count)
    return launch_matvec<256>(ctx, row_major, n_rows, n_cols, J, rs, cs, v, sign, out, st);
  return launch_matvec<32>(ctx, row_major, n_rows, n_cols, J, rs, cs, v, sign, out, st);
}

// ---- J^T @ r and the squared column norms --------------------------------------------------------------------------
// The bit contract fixes one sequential chain of n_rows steps per column of J, so the parallelism is n_cols threads.
// A CTA owns RV_CW = 16 columns: all 256 threads keep RV_STAGES - 1 tiles of RV_R rows x 16 columns (and the matching
// entries of r) in flight with cp.async -- 128-byte row segments for row-major J, 512-byte column segments for
// column-major J -- while 16 threads run the chains out of shared memory.  The time is about n_rows dependent FMA
// latencies unless n_cols is large enough for the loads to saturate HBM.  SQUARE: the chain is fma(a, a, acc) and r is
// neither read nor loaded (gnk_dense_col_sumsq).
constexpr int RV_THREADS = 256, RV_CW = 16, RV_R = 64, RV_STAGES = 5;

template <bool ROW_MAJOR, bool SQUARE>
__device__ __forceinline__ void column_chains(int64_t n_rows, int64_t n_cols, const double* __restrict__ J, int64_t rs,
                                              int64_t cs, const double* __restrict__ r, double sign,
                                              double* __restrict__ out) {
  __shared__ double Js[RV_STAGES][RV_R][RV_CW + 1];
  __shared__ double Rs[SQUARE ? 1 : RV_STAGES][RV_R];
  const int tid = threadIdx.x;
  const int64_t c0 = (int64_t)blockIdx.x * RV_CW;
  const int64_t tiles = (n_rows + RV_R - 1) / RV_R;

  auto load = [&](int64_t t) {
    if (t >= tiles) return;
    const int buf = (int)(t % RV_STAGES);
    const int64_t row0 = t * RV_R;
    for (int e = tid; e < RV_R * RV_CW; e += RV_THREADS) {
      const int i = ROW_MAJOR ? e / RV_CW : e % RV_R, c = ROW_MAJOR ? e % RV_CW : e / RV_R;
      const int64_t rr = row0 + i, cc = c0 + c;
      const bool ok = rr < n_rows && cc < n_cols;
      cp_async8(&Js[buf][i][c], ok ? J + rr * rs + cc * cs : J, ok);
    }
    if (!SQUARE && tid < RV_R) {
      const bool ok = row0 + tid < n_rows;
      cp_async8(&Rs[buf][tid], ok ? r + row0 + tid : r, ok);
    }
  };

#pragma unroll
  for (int s = 0; s < RV_STAGES - 1; ++s) {
    load(s);
    cp_async_commit();
  }
  double acc = 0.0;
  for (int64_t t = 0; t < tiles; ++t) {
    cp_async_wait<RV_STAGES - 2>();
    __syncthreads();  // tile t has landed, and the chains of tile t - 1 are done with their buffer
    load(t + RV_STAGES - 1);
    cp_async_commit();
    if (tid < RV_CW) {
      const int buf = (int)(t % RV_STAGES);
#pragma unroll 8
      for (int i = 0; i < RV_R; ++i) {
        const double a = Js[buf][i][tid];
        if (a != 0.0) acc = fma(a, SQUARE ? a : Rs[buf][i], acc);
      }
    }
  }
  if (tid < RV_CW && c0 + tid < n_cols) out[c0 + tid] = SQUARE ? acc : sign * acc;
}

template <bool ROW_MAJOR>
__global__ void __launch_bounds__(RV_THREADS) dense_rmatvec_kernel(int64_t n_rows, int64_t n_cols,
                                                                    const double* __restrict__ J, int64_t rs,
                                                                    int64_t cs, const double* __restrict__ r,
                                                                    double sign, double* __restrict__ out) {
  column_chains<ROW_MAJOR, false>(n_rows, n_cols, J, rs, cs, r, sign, out);
}

template <bool ROW_MAJOR>
__global__ void __launch_bounds__(RV_THREADS) dense_col_sumsq_kernel(int64_t n_rows, int64_t n_cols,
                                                                      const double* __restrict__ J, int64_t rs,
                                                                      int64_t cs, double* __restrict__ out) {
  column_chains<ROW_MAJOR, true>(n_rows, n_cols, J, rs, cs, nullptr, 1.0, out);
}

bool dense_layout_ok(int64_t n_rows, int64_t n_cols, int64_t rs, int64_t cs) {
  return n_rows >= 0 && n_cols >= 0 && n_rows < INT32_MAX && n_cols < INT32_MAX && rs >= 0 && cs >= 0 &&
         (rs == 1 || cs == 1);
}

// which load mapping is coalesced: along rows when the column stride is 1 (a single column with row stride 1 is read
// as the column it is)
bool row_major(int64_t n_cols, int64_t rs, int64_t cs) { return cs == 1 && !(rs == 1 && n_cols == 1); }

}  // namespace

extern "C" {

int gnk_dense_matmat(gnk_ctx* ctx, int64_t n_rows, int64_t n_cols, const double* d_J, int64_t row_stride,
                     int64_t col_stride, const double* d_in, int64_t in_ld, int64_t in_off, int k, double sign,
                     double* d_out, int64_t out_ld, int64_t out_off, void* stream) {
  GNK_REQUIRE(ctx && d_J && d_in && d_out, "gnk_dense_matmat: null argument");
  GNK_REQUIRE(k >= 1 && dense_layout_ok(n_rows, n_cols, row_stride, col_stride),
              "gnk_dense_matmat: bad sizes or strides (n_rows, n_cols < 2^31 - 1; one stride must be 1)");
  if (n_rows == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const bool rm = row_major(n_cols, row_stride, col_stride);
  if (k == 1)
    return launch_matvec_sized(ctx, rm, n_rows, n_cols, d_J, row_stride, col_stride, d_in + in_off, sign,
                               d_out + out_off, st);
  cudaError_t e;
  // basis columns one pass carries: 1 (dense_matvec_kernel) / 2 / 4 / 16 / 32 while k fits, then passes of 64 columns
  // (k <= 255: at most 4)
  if (k <= 2)
    e = launch_matmat<1, 2, 1, 8>(rm, n_rows, n_cols, d_J, row_stride, col_stride, d_in, in_ld, in_off, k, sign, d_out,
                                  out_ld, out_off, st);
  else if (k <= 4)
    e = launch_matmat<2, 2, 2, 8>(rm, n_rows, n_cols, d_J, row_stride, col_stride, d_in, in_ld, in_off, k, sign, d_out,
                                  out_ld, out_off, st);
  else if (k <= 16)
    e = launch_matmat<2, 4, 4, 16>(rm, n_rows, n_cols, d_J, row_stride, col_stride, d_in, in_ld, in_off, k, sign,
                                   d_out, out_ld, out_off, st);
  else if (k <= 32)
    e = launch_matmat<4, 4, 8, 16>(rm, n_rows, n_cols, d_J, row_stride, col_stride, d_in, in_ld, in_off, k, sign,
                                   d_out, out_ld, out_off, st);
  else
    e = launch_matmat<4, 4, 16, 16>(rm, n_rows, n_cols, d_J, row_stride, col_stride, d_in, in_ld, in_off, k, sign,
                                    d_out, out_ld, out_off, st);
  ctx->launches++;
  if (e != cudaSuccess) return gnk_fail("kernel launch", e, __FILE__, __LINE__);
  return 0;
}

int gnk_dense_rmatvec(gnk_ctx* ctx, int64_t n_rows, int64_t n_cols, const double* d_J, int64_t row_stride,
                      int64_t col_stride, const double* d_r, double sign, double* d_out, void* stream) {
  GNK_REQUIRE(ctx && d_J && d_r && d_out, "gnk_dense_rmatvec: null argument");
  GNK_REQUIRE(dense_layout_ok(n_rows, n_cols, row_stride, col_stride),
              "gnk_dense_rmatvec: bad sizes or strides (n_rows, n_cols < 2^31 - 1; one stride must be 1)");
  if (n_cols == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const bool rm = row_major(n_cols, row_stride, col_stride);
  const unsigned grid = (unsigned)ceil_div(n_cols, RV_CW);
  if (rm)
    dense_rmatvec_kernel<true><<<grid, RV_THREADS, 0, st>>>(n_rows, n_cols, d_J, row_stride, col_stride, d_r, sign,
                                                            d_out);
  else
    dense_rmatvec_kernel<false><<<grid, RV_THREADS, 0, st>>>(n_rows, n_cols, d_J, row_stride, col_stride, d_r, sign,
                                                             d_out);
  GNK_LAUNCH_CHECK(ctx);
  return 0;
}

int gnk_dense_col_sumsq(gnk_ctx* ctx, int64_t n_rows, int64_t n_cols, const double* d_J, int64_t row_stride,
                        int64_t col_stride, double* d_out, void* stream) {
  GNK_REQUIRE(ctx && d_J && d_out, "gnk_dense_col_sumsq: null argument");
  GNK_REQUIRE(dense_layout_ok(n_rows, n_cols, row_stride, col_stride),
              "gnk_dense_col_sumsq: bad sizes or strides (n_rows, n_cols < 2^31 - 1; one stride must be 1)");
  if (n_cols == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned grid = (unsigned)ceil_div(n_cols, RV_CW);
  if (row_major(n_cols, row_stride, col_stride))
    dense_col_sumsq_kernel<true><<<grid, RV_THREADS, 0, st>>>(n_rows, n_cols, d_J, row_stride, col_stride, d_out);
  else
    dense_col_sumsq_kernel<false><<<grid, RV_THREADS, 0, st>>>(n_rows, n_cols, d_J, row_stride, col_stride, d_out);
  GNK_LAUNCH_CHECK(ctx);
  return 0;
}

}  // extern "C"
