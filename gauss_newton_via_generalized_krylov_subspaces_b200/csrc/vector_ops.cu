// vector_ops.cu -- basis-sized streaming kernels of the GNK hot path (all HBM-bound, fp64):
//   combine     x = V_k (c + s d)                 krylow.py:41-42, armijo_goldstein.py:56
//   norm_stats  sum x^2, max|x|                   krylow.py:31,36,66,71
//   normalize   x / ||x||                         krylow.py:37,71
//   cgs_dots    h = V_k^T w                       krylow.py:64 (inner product half)
//   cgs_update  w -= V_k h  (+ stats of new w)    krylow.py:64 (update half) + :66,:71
//   axpby, dot                                    gauss_newton.py:123-129
// combine, cgs_dots and cgs_update have wide twins for bases of 256..4095 columns (*_wide_kernel).
// Every thread moves 128-bit (double2) words, columns are walked with independent loads in flight,
// grids are sized in multiples of the SM count, cross-CTA reductions use a fixed-order
// "last CTA finishes" tree so results are run-to-run deterministic.
#include "common.cuh"

namespace {

constexpr int TPB = 256;

__device__ __forceinline__ double2 ld2(const double* p) { return *reinterpret_cast<const double2*>(p); }
__device__ __forceinline__ double2 ld2_stream(const double* p) {
  return __ldcs(reinterpret_cast<const double2*>(p));
}
__device__ __forceinline__ void st2(double* p, double2 v) { *reinterpret_cast<double2*>(p) = v; }

// ---------------------------------------------------------------------------------------------
// c_out / cprev2 (optional): the coordinate bookkeeping of combine_coefficients (common.cuh).  Saves three tiny
// launches per outer iteration.
__global__ void __launch_bounds__(TPB) combine_kernel(const double* __restrict__ V, int64_t ld, int64_t len,
                                                       int k, const double* __restrict__ c,
                                                       const double* __restrict__ d, double s,
                                                       double* __restrict__ x, double* __restrict__ c_out,
                                                       double* __restrict__ cprev2) {
  __shared__ double coef[GNK_MAX_BASIS];
  pdl_begin();
  combine_coefficients(k, c, d, s, coef, c_out, cprev2);
  const int64_t nv = len >> 1;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += stride) {
    const double* p = V + 2 * i;
    double2 acc = make_double2(0.0, 0.0);
    int j = 0;
    for (; j + 8 <= k; j += 8) {
      double2 v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = ld2_stream(p + (int64_t)(j + u) * ld);
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        acc.x = fma(v[u].x, coef[j + u], acc.x);
        acc.y = fma(v[u].y, coef[j + u], acc.y);
      }
    }
    for (; j < k; ++j) {
      double2 v = ld2_stream(p + (int64_t)j * ld);
      acc.x = fma(v.x, coef[j], acc.x);
      acc.y = fma(v.y, coef[j], acc.y);
    }
    st2(x + 2 * i, acc);
  }
}

// ---------------------------------------------------------------------------------------------
// sum of squares + max abs over x[0..n); partials[b*2 + {0,1}]
__global__ void __launch_bounds__(TPB) stats_kernel(const double* __restrict__ x, int64_t n,
                                                     double* __restrict__ partials, unsigned int* ticket,
                                                     double* __restrict__ out) {
  __shared__ double sh[32];
  const int64_t nv = n >> 1;
  const int64_t gt = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  double ss = 0.0, mx = 0.0;
  for (int64_t i = gt; i < nv; i += stride) {
    double2 v = ld2(x + 2 * i);
    ss = fma(v.x, v.x, ss);
    ss = fma(v.y, v.y, ss);
    mx = fmax(mx, fmax(fabs(v.x), fabs(v.y)));
  }
  if ((n & 1) && gt == 0) {
    double v = x[n - 1];
    ss = fma(v, v, ss);
    mx = fmax(mx, fabs(v));
  }
  ss = block_sum(ss, sh);
  mx = block_max(mx, sh);
  if (threadIdx.x == 0) {
    partials[2 * blockIdx.x] = ss;
    partials[2 * blockIdx.x + 1] = mx;
  }
  if (grid_arrive_last(ticket)) {
    double a = 0.0, b = 0.0;
    for (int i = threadIdx.x; i < (int)gridDim.x; i += blockDim.x) {
      a += __ldcg(partials + 2 * i);
      b = fmax(b, __ldcg(partials + 2 * i + 1));
    }
    a = block_sum(a, sh);
    b = block_max(b, sh);
    if (threadIdx.x == 0) {
      out[0] = a;
      out[1] = b;
    }
  }
}

__global__ void __launch_bounds__(TPB) normalize_kernel(const double* __restrict__ x, int64_t len,
                                                         const double* __restrict__ stats, double atol,
                                                         double* __restrict__ out, int32_t* flag) {
  pdl_begin();
  const double ss = stats[0], mx = stats[1];
  const bool bad = (mx <= atol);
  if (blockIdx.x == 0 && threadIdx.x == 0) *flag = bad ? 1 : 0;
  if (bad) return;
  const double nrm = sqrt(ss);
  const int64_t nv = len >> 1;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  // four independent 128-bit loads in flight per thread (one per iteration kept the kernel at 0.67 of the roofline:
  // 4.8 MB in flight on the whole GPU), true divisions as in the reference (w /= norm, krylow.py:71)
  for (; i + 3 * stride < nv; i += 4 * stride) {
    double2 a = ld2(x + 2 * i), b = ld2(x + 2 * (i + stride)), c = ld2(x + 2 * (i + 2 * stride)),
            d = ld2(x + 2 * (i + 3 * stride));
    a.x /= nrm; a.y /= nrm; b.x /= nrm; b.y /= nrm; c.x /= nrm; c.y /= nrm; d.x /= nrm; d.y /= nrm;
    st2(out + 2 * i, a);
    st2(out + 2 * (i + stride), b);
    st2(out + 2 * (i + 2 * stride), c);
    st2(out + 2 * (i + 3 * stride), d);
  }
  for (; i < nv; i += stride) {
    double2 v = ld2(x + 2 * i);
    v.x = v.x / nrm;
    v.y = v.y / nrm;
    st2(out + 2 * i, v);
  }
}

// normalize fused with the halo exchange of the column it writes (multi-GPU, peer mailboxes attached): the threads that
// write the first / last `cnt` owned doubles also push them into the lower / upper neighbour's mailbox over NVLink, as
// 16-byte flag-in-data lines {lo, tag, hi, tag} (st_ll, common.cuh); the first HALO_RECV CTAs then poll the lines the
// neighbours push into THIS rank's mailbox and write them into the halo rows of `out`.  No system-scope fence, no flag
// hop, no grid-wide ticket and no single-CTA copy (round-2 history: data + fence + flag + one CTA copying 2 x 64 KB
// cost 15-17 us per outer iteration at 8 GPUs on top of the 5 us of streaming): a line is complete when both tags
// carry this exchange's number.  Lines are double-buffered on the parity of the exchange number; a rank can be at most
// one exchange ahead of its neighbour because it cannot finish exchange s without the neighbour's lines of s.
// A breakdown (max|w| <= atol) is decided from the all-reduced statistics, identically on every rank: nobody pushes
// and nobody waits.  A receiving CTA may spin until the neighbour's kernel has started; the neighbour's progress never
// depends on this rank's normalize kernel, so this cannot deadlock, and ld_ll traps after P2P_TIMEOUT_NS.
struct HaloPush {
  void* const* peers;
  int rank, nranks, has_lo, has_hi;
  int64_t off, rows_m, cnt;  // first owned double, owned doubles, doubles per message (depth * m)
  unsigned long long seq;
};
constexpr int HALO_RECV = 32;
__global__ void __launch_bounds__(TPB) normalize_halo_kernel(const double* __restrict__ x, int64_t len,
                                                              const double* __restrict__ stats, double atol,
                                                              double* __restrict__ out, int32_t* flag, HaloPush hp) {
  pdl_begin();
  const double ss = stats[0], mx = stats[1];
  const bool bad = (mx <= atol);
  if (blockIdx.x == 0 && threadIdx.x == 0) *flag = bad ? 1 : 0;
  if (bad) return;
  const int parity = (int)(hp.seq & 1ull);
  const unsigned tag = (unsigned)(hp.seq % 0xFFFFFFFFull) + 1u;
  const double nrm = sqrt(ss);
  // my first rows become the lower neighbour's upper halo (its side 1), my last rows the upper neighbour's side 0
  char* lo_dst = hp.has_lo ? static_cast<char*>(hp.peers[hp.rank - 1]) + p2p_hll_off(hp.nranks, parity, 1) : nullptr;
  char* hi_dst = hp.has_hi ? static_cast<char*>(hp.peers[hp.rank + 1]) + p2p_hll_off(hp.nranks, parity, 0) : nullptr;
  const int64_t lo_end = hp.off + hp.cnt, hi_beg = hp.off + hp.rows_m - hp.cnt, hi_end = hp.off + hp.rows_m;
  const int64_t nv = len >> 1;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += stride) {
    const int64_t e = 2 * i;  // off, cnt and rows_m are even: a pair never straddles a piece
    // the halo rows that a neighbour fills are written by the receiving CTAs below and by nobody else
    if ((lo_dst && e >= hp.off - hp.cnt && e < hp.off) || (hi_dst && e >= hi_end && e < hi_end + hp.cnt)) continue;
    double2 v = ld2(x + 2 * i);
    v.x = v.x / nrm;
    v.y = v.y / nrm;
    st2(out + 2 * i, v);
    if (lo_dst && e >= hp.off && e < lo_end) {
      st_ll(lo_dst + 16 * (e - hp.off), v.x, tag);
      st_ll(lo_dst + 16 * (e - hp.off + 1), v.y, tag);
    }
    if (hi_dst && e >= hi_beg && e < hi_end) {
      st_ll(hi_dst + 16 * (e - hi_beg), v.x, tag);
      st_ll(hi_dst + 16 * (e - hi_beg + 1), v.y, tag);
    }
  }
  if (blockIdx.x >= HALO_RECV) return;
  const char* mine = static_cast<const char*>(hp.peers[hp.rank]);
  const int64_t pairs = hp.cnt >> 1;
  const int64_t rstride = (int64_t)(gridDim.x < HALO_RECV ? gridDim.x : HALO_RECV) * blockDim.x;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < 2 * pairs; p += rstride) {
    const int side = p >= pairs ? 1 : 0;
    if (!(side == 0 ? hp.has_lo : hp.has_hi)) continue;
    const int64_t j = p - side * pairs;
    const char* line = mine + p2p_hll_off(hp.nranks, parity, side) + 32 * j;
    double2 v;
    v.x = ld_ll(line, tag);
    v.y = ld_ll(line + 16, tag);
    st2(out + (side == 0 ? hp.off - hp.cnt : hp.off + hp.rows_m) + 2 * j, v);
  }
}

// ---------------------------------------------------------------------------------------------
// h[j] = sum_i V[j*ld + i] * w[i], i in [0, n) (pointers already offset to the owned part)
constexpr int JB = 8;  // columns per pass: 8 accumulators keep the kernel at ~64 registers -> 32+ warps per SM

// one pass over NJ (compile-time) columns starting at Vb: every thread keeps NJ running sums
template <int NJ>
__device__ __forceinline__ void dots_pass(const double* __restrict__ Vb, int64_t ld, int64_t n,
                                          const double* __restrict__ w, double (&acc)[JB]) {
  const int64_t nv = n >> 1;
  const int64_t gt = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
#pragma unroll 1
  for (int64_t i = gt; i < nv; i += stride) {
    const double2 wv = ld2(w + 2 * i);
    double2 v[NJ];
#pragma unroll
    for (int u = 0; u < NJ; ++u) v[u] = ld2_stream(Vb + (int64_t)u * ld + 2 * i);
#pragma unroll
    for (int u = 0; u < NJ; ++u) acc[u] = fma(v[u].y, wv.y, fma(v[u].x, wv.x, acc[u]));
  }
  if ((n & 1) && gt == 0) {
    const double wv = w[n - 1];
#pragma unroll
    for (int u = 0; u < NJ; ++u) acc[u] = fma(Vb[(int64_t)u * ld + n - 1], wv, acc[u]);
  }
}

__global__ void __launch_bounds__(TPB, 4) dots_kernel(const double* __restrict__ V, int64_t ld, int64_t n, int k,
                                                    const double* __restrict__ w, double* __restrict__ partials,
                                                    unsigned int* ticket, double* __restrict__ h, gnk_p2p_dev pd) {
  // per-warp sums of every column; ONE barrier per launch instead of two per column (at n ~ 1e6 -- the 8-GPU slabs and
  // the 1024^2 grid -- the 2 k barriers of the per-column block reductions were most of the kernel: 51 us for 20 us
  // of traffic)
  __shared__ double wpart[TPB / 32][GNK_MAX_BASIS];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  pdl_begin();
  for (int jb = 0; jb < k; jb += JB) {
    double acc[JB];
#pragma unroll
    for (int u = 0; u < JB; ++u) acc[u] = 0.0;
    const int nj = min(JB, k - jb);
    const double* Vb = V + (int64_t)jb * ld;
    switch (nj) {  // block-uniform; the remainder pass runs unmasked code too
      case 8: dots_pass<8>(Vb, ld, n, w, acc); break;
      case 7: dots_pass<7>(Vb, ld, n, w, acc); break;
      case 6: dots_pass<6>(Vb, ld, n, w, acc); break;
      case 5: dots_pass<5>(Vb, ld, n, w, acc); break;
      case 4: dots_pass<4>(Vb, ld, n, w, acc); break;
      case 3: dots_pass<3>(Vb, ld, n, w, acc); break;
      case 2: dots_pass<2>(Vb, ld, n, w, acc); break;
      default: dots_pass<1>(Vb, ld, n, w, acc); break;
    }
#pragma unroll
    for (int u = 0; u < JB; ++u) {
      if (u < nj) {
        const double r = warp_sum(acc[u]);
        if (lane == 0) wpart[wid][jb + u] = r;
      }
    }
  }
  dots_finish(wpart, k, partials, ticket, h, pd);
}

// w[i] -= sum_j V[j*ld+i] h[j]; stats of the new w
__global__ void __launch_bounds__(TPB) update_kernel(const double* __restrict__ V, int64_t ld, int64_t n, int k,
                                                      const double* __restrict__ h, double* __restrict__ w,
                                                      double* __restrict__ partials, unsigned int* ticket,
                                                      double* __restrict__ stats, gnk_p2p_dev pd) {
  __shared__ double coef[GNK_MAX_BASIS];
  __shared__ double sh[32];
  pdl_begin();
  for (int j = threadIdx.x; j < k; j += blockDim.x) coef[j] = h[j];
  __syncthreads();
  const int64_t nv = n >> 1;
  const int64_t gt = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  double ss = 0.0, mx = 0.0;
  for (int64_t i = gt; i < nv; i += stride) {
    const double* p = V + 2 * i;
    double2 acc = make_double2(0.0, 0.0);
    int j = 0;
    for (; j + 8 <= k; j += 8) {
      double2 v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = ld2_stream(p + (int64_t)(j + u) * ld);
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        acc.x = fma(v[u].x, coef[j + u], acc.x);
        acc.y = fma(v[u].y, coef[j + u], acc.y);
      }
    }
    for (; j < k; ++j) {
      double2 v = ld2_stream(p + (int64_t)j * ld);
      acc.x = fma(v.x, coef[j], acc.x);
      acc.y = fma(v.y, coef[j], acc.y);
    }
    double2 wv = ld2(w + 2 * i);
    wv.x -= acc.x;
    wv.y -= acc.y;
    st2(w + 2 * i, wv);
    ss = fma(wv.x, wv.x, ss);
    ss = fma(wv.y, wv.y, ss);
    mx = fmax(mx, fmax(fabs(wv.x), fabs(wv.y)));
  }
  if ((n & 1) && gt == 0) {
    double acc = 0.0;
    for (int j = 0; j < k; ++j) acc = fma(V[(int64_t)j * ld + n - 1], coef[j], acc);
    double wv = w[n - 1] - acc;
    w[n - 1] = wv;
    ss = fma(wv, wv, ss);
    mx = fmax(mx, fabs(wv));
  }
  if (stats == nullptr) return;
  ss = block_sum(ss, sh);
  mx = block_max(mx, sh);
  if (threadIdx.x == 0) {
    partials[2 * blockIdx.x] = ss;
    partials[2 * blockIdx.x + 1] = mx;
  }
  if (grid_arrive_last(ticket)) {
    double a = 0.0, b = 0.0;
    for (int i = threadIdx.x; i < (int)gridDim.x; i += blockDim.x) {
      a += __ldcg(partials + 2 * i);
      b = fmax(b, __ldcg(partials + 2 * i + 1));
    }
    a = block_sum(a, sh);
    b = block_max(b, sh);
    if (threadIdx.x == 0) {
      stats[0] = a;
      stats[1] = b;
    }
    if (pd.peers) {  // (sum, max) over the ranks, in this CTA, over the peers' mailboxes
      __syncthreads();
      p2p_tail_allreduce(pd, stats, 2, 2);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Bases of GNK_MAX_BASIS <= k < GNK_MAX_BASIS_WIDE columns (runs without a restart).  Same per-element arithmetic as the
// kernels above, with the k coefficients in 8k bytes of dynamic shared memory (at most 32 KB: 7 CTAs of 256 threads
// per SM) and the per-warp sums of the dots staged in chunks of WCH columns.  Still one pass over V_k per launch.
constexpr int WCH = 256;  // columns per chunk of the per-warp sums of dots_wide_kernel (a multiple of JB)

// combine_coefficients (common.cuh) for any k: c_out receives k + 1 doubles
__device__ __forceinline__ void combine_coefficients_wide(int k, const double* __restrict__ c,
                                                          const double* __restrict__ d, double s, double* coef,
                                                          double* __restrict__ c_out, double* __restrict__ cprev2) {
  for (int j = threadIdx.x; j < k; j += blockDim.x) coef[j] = d ? __fma_rn(s, d[j], c[j]) : c[j];
  __syncthreads();
  if (blockIdx.x == 0) {
    if (c_out) {
      for (int j = threadIdx.x; j <= k; j += blockDim.x) c_out[j] = (j < k) ? coef[j] : 0.0;
    }
    if (cprev2 && threadIdx.x < 32) {
      double a = 0.0;
      for (int j = threadIdx.x; j < k; j += 32) a = fma(c[j], c[j], a);
      a = warp_sum(a);
      if (threadIdx.x == 0) cprev2[0] = a;
    }
  }
}

// sum_j V[j*ld + 2i .. 2i+1] coef[j], eight 128-bit loads in flight
__device__ __forceinline__ double2 combine_row(const double* __restrict__ p, int64_t ld, int k,
                                               const double* __restrict__ coef) {
  double2 acc = make_double2(0.0, 0.0);
  int j = 0;
  for (; j + 8 <= k; j += 8) {
    double2 v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) v[u] = ld2_stream(p + (int64_t)(j + u) * ld);
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      acc.x = fma(v[u].x, coef[j + u], acc.x);
      acc.y = fma(v[u].y, coef[j + u], acc.y);
    }
  }
  for (; j < k; ++j) {
    double2 v = ld2_stream(p + (int64_t)j * ld);
    acc.x = fma(v.x, coef[j], acc.x);
    acc.y = fma(v.y, coef[j], acc.y);
  }
  return acc;
}

__global__ void __launch_bounds__(TPB) combine_wide_kernel(const double* __restrict__ V, int64_t ld, int64_t len,
                                                            int k, const double* __restrict__ c,
                                                            const double* __restrict__ d, double s,
                                                            double* __restrict__ x, double* __restrict__ c_out,
                                                            double* __restrict__ cprev2) {
  extern __shared__ double coef[];
  pdl_begin();
  combine_coefficients_wide(k, c, d, s, coef, c_out, cprev2);
  const int64_t nv = len >> 1;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += stride)
    st2(x + 2 * i, combine_row(V + 2 * i, ld, k, coef));
}

// h = V_k^T w.  partials: column-major per CTA (partials[j * gridDim.x + b]), so that the last CTA reads them coalesced
// while summing in dots_finish's order (lanes strided over the CTAs, then the warp tree): per entry the bits of
// dots_kernel at the same n.
__global__ void __launch_bounds__(TPB, 4) dots_wide_kernel(const double* __restrict__ V, int64_t ld, int64_t n, int k,
                                                         const double* __restrict__ w, double* __restrict__ partials,
                                                         unsigned int* ticket, double* __restrict__ h,
                                                         gnk_p2p_dev pd) {
  __shared__ double wpart[TPB / 32][WCH];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int G = gridDim.x;
  pdl_begin();
  for (int c0 = 0; c0 < k; c0 += WCH) {
    const int kc = min(WCH, k - c0);
    for (int jb = 0; jb < kc; jb += JB) {
      double acc[JB];
#pragma unroll
      for (int u = 0; u < JB; ++u) acc[u] = 0.0;
      const int nj = min(JB, kc - jb);
      const double* Vb = V + (int64_t)(c0 + jb) * ld;
      switch (nj) {
        case 8: dots_pass<8>(Vb, ld, n, w, acc); break;
        case 7: dots_pass<7>(Vb, ld, n, w, acc); break;
        case 6: dots_pass<6>(Vb, ld, n, w, acc); break;
        case 5: dots_pass<5>(Vb, ld, n, w, acc); break;
        case 4: dots_pass<4>(Vb, ld, n, w, acc); break;
        case 3: dots_pass<3>(Vb, ld, n, w, acc); break;
        case 2: dots_pass<2>(Vb, ld, n, w, acc); break;
        default: dots_pass<1>(Vb, ld, n, w, acc); break;
      }
#pragma unroll
      for (int u = 0; u < JB; ++u) {
        if (u < nj) {
          const double r = warp_sum(acc[u]);
          if (lane == 0) wpart[wid][jb + u] = r;
        }
      }
    }
    __syncthreads();
    for (int j = threadIdx.x; j < kc; j += blockDim.x) {
      double r = wpart[0][j];
#pragma unroll
      for (int q = 1; q < TPB / 32; ++q) r += wpart[q][j];
      partials[(int64_t)(c0 + j) * G + blockIdx.x] = r;
    }
    __syncthreads();  // wpart is refilled by the next chunk
  }
  if (grid_arrive_last(ticket)) {
    for (int j = wid; j < k; j += TPB / 32) {
      const double* pj = partials + (int64_t)j * G;
      double a = 0.0;
      for (int b = lane; b < G; b += 32) a += __ldcg(pj + b);
      a = warp_sum(a);
      if (lane == 0) h[j] = a;
    }
    if (pd.peers) {  // sum over the ranks, in this CTA, over the peers' mailboxes
      __syncthreads();
      p2p_tail_allreduce_wide(pd, h, k);
    }
  }
}

// w[i] -= sum_j V[j*ld+i] h[j]; stats of the new w (update_kernel for any k)
__global__ void __launch_bounds__(TPB) update_wide_kernel(const double* __restrict__ V, int64_t ld, int64_t n, int k,
                                                           const double* __restrict__ h, double* __restrict__ w,
                                                           double* __restrict__ partials, unsigned int* ticket,
                                                           double* __restrict__ stats, gnk_p2p_dev pd) {
  extern __shared__ double coef[];
  __shared__ double sh[32];
  pdl_begin();
  for (int j = threadIdx.x; j < k; j += blockDim.x) coef[j] = h[j];
  __syncthreads();
  const int64_t nv = n >> 1;
  const int64_t gt = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  double ss = 0.0, mx = 0.0;
  for (int64_t i = gt; i < nv; i += stride) {
    const double2 acc = combine_row(V + 2 * i, ld, k, coef);
    double2 wv = ld2(w + 2 * i);
    wv.x -= acc.x;
    wv.y -= acc.y;
    st2(w + 2 * i, wv);
    ss = fma(wv.x, wv.x, ss);
    ss = fma(wv.y, wv.y, ss);
    mx = fmax(mx, fmax(fabs(wv.x), fabs(wv.y)));
  }
  if ((n & 1) && gt == 0) {
    double acc = 0.0;
    for (int j = 0; j < k; ++j) acc = fma(V[(int64_t)j * ld + n - 1], coef[j], acc);
    double wv = w[n - 1] - acc;
    w[n - 1] = wv;
    ss = fma(wv, wv, ss);
    mx = fmax(mx, fabs(wv));
  }
  if (stats == nullptr) return;
  ss = block_sum(ss, sh);
  mx = block_max(mx, sh);
  if (threadIdx.x == 0) {
    partials[2 * blockIdx.x] = ss;
    partials[2 * blockIdx.x + 1] = mx;
  }
  if (grid_arrive_last(ticket)) {
    double a = 0.0, b = 0.0;
    for (int i = threadIdx.x; i < (int)gridDim.x; i += blockDim.x) {
      a += __ldcg(partials + 2 * i);
      b = fmax(b, __ldcg(partials + 2 * i + 1));
    }
    a = block_sum(a, sh);
    b = block_max(b, sh);
    if (threadIdx.x == 0) {
      stats[0] = a;
      stats[1] = b;
    }
    if (pd.peers) {
      __syncthreads();
      p2p_tail_allreduce(pd, stats, 2, 2);
    }
  }
}

// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(TPB) axpby_kernel(int64_t n, double a, const double* x, double b,
                                                     const double* y, double* out) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    double r = 0.0;
    if (a != 0.0) r = a * x[i];
    if (b != 0.0) r = fma(b, y[i], r);
    out[i] = r;
  }
}

__global__ void __launch_bounds__(TPB) dot_kernel(int64_t n, const double* __restrict__ x,
                                                   const double* __restrict__ y, double* __restrict__ partials,
                                                   unsigned int* ticket, double* __restrict__ out) {
  __shared__ double sh[32];
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  double s = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) s = fma(x[i], y[i], s);
  s = block_sum(s, sh);
  if (threadIdx.x == 0) partials[blockIdx.x] = s;
  if (grid_arrive_last(ticket)) {
    double a = 0.0;
    for (int i = threadIdx.x; i < (int)gridDim.x; i += blockDim.x) a += __ldcg(partials + i);
    a = block_sum(a, sh);
    if (threadIdx.x == 0) out[0] = a;
  }
}

inline int stream_grid(const gnk_ctx* ctx, int64_t items, int per_sm) {
  int64_t g = ceil_div(items, TPB);
  int64_t cap = (int64_t)ctx->sm_count * per_sm;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

}  // namespace

extern "C" {

int gnk_combine_step(gnk_ctx* ctx, const gnk_layout* lay, const double* d_V, int k, const double* d_c,
                     const double* d_d, double s, double* d_x, double* d_c_out, double* d_cprev2, void* stream) {
  GNK_REQUIRE(ctx && lay && d_V && d_c && d_x, "gnk_combine: null argument");
  GNK_REQUIRE(k >= 1 && k < GNK_MAX_BASIS_WIDE, "gnk_combine: k out of range");
  GNK_REQUIRE((lay->ld & 1) == 0, "gnk_combine: ld must be even");
  GNK_REQUIRE(d_c_out != d_c, "gnk_combine_step: c_out must not alias c (rejected trials re-read c)");
  int grid = stream_grid(ctx, lay->ld / 2, 8);
  if (k >= GNK_MAX_BASIS) {
    GNK_CUDA(gnk_launch(gnk_pdl_for(lay->n_own), combine_wide_kernel, dim3(grid), dim3(TPB), sizeof(double) * k,
                        (cudaStream_t)stream, d_V, lay->ld, lay->ld, k, d_c, d_d, s, d_x, d_c_out, d_cprev2));
    GNK_LAUNCH_CHECK(ctx);
    return 0;
  }
  GNK_CUDA(gnk_launch(gnk_pdl_for(lay->n_own), combine_kernel, dim3(grid), dim3(TPB), 0, (cudaStream_t)stream, d_V, lay->ld, lay->ld, k, d_c, d_d, s,
                      d_x, d_c_out, d_cprev2));
  GNK_LAUNCH_CHECK(ctx);
  return 0;
}

int gnk_combine(gnk_ctx* ctx, const gnk_layout* lay, const double* d_V, int k, const double* d_c,
                const double* d_d, double s, double* d_x, void* stream) {
  return gnk_combine_step(ctx, lay, d_V, k, d_c, d_d, s, d_x, nullptr, nullptr, stream);
}

int gnk_norm_stats(gnk_ctx* ctx, const gnk_layout* lay, const double* d_x, double* d_stats, void* stream) {
  GNK_REQUIRE(ctx && lay && d_x && d_stats, "gnk_norm_stats: null argument");
  GNK_REQUIRE((lay->off & 1) == 0, "gnk_norm_stats: off must be even");
  int grid = stream_grid(ctx, lay->n_own / 2, 4);
  stats_kernel<<<grid, TPB, 0, (cudaStream_t)stream>>>(d_x + lay->off, lay->n_own, ctx->d_partials + PART_STATS,
                                                       ctx->d_tickets + TK_STATS, d_stats);
  GNK_LAUNCH_CHECK(ctx);
  return 0;
}

int gnk_normalize(gnk_ctx* ctx, const gnk_layout* lay, const double* d_x, const double* d_stats, double atol,
                  double* d_out, int32_t* d_flag, void* stream) {
  GNK_REQUIRE(ctx && lay && d_x && d_stats && d_out && d_flag, "gnk_normalize: null argument");
  GNK_REQUIRE((lay->ld & 1) == 0, "gnk_normalize: ld must be even");
  int grid = stream_grid(ctx, lay->ld / 2, 8);
  GNK_CUDA(gnk_launch(gnk_pdl_for(lay->n_own), normalize_kernel, dim3(grid), dim3(TPB), 0, (cudaStream_t)stream, d_x, lay->ld, d_stats, atol, d_out,
                      d_flag));
  GNK_LAUNCH_CHECK(ctx);
  return 0;
}

int gnk_comm_halo_exchange(gnk_ctx* ctx, const gnk_layout* lay, double* d_col, int depth, void* stream);

int gnk_normalize_halo(gnk_ctx* ctx, const gnk_layout* lay, const double* d_x, const double* d_stats, double atol,
                       double* d_out, int32_t* d_flag, void* stream) {
  GNK_REQUIRE(ctx && lay && d_x && d_stats && d_out && d_flag, "gnk_normalize_halo: null argument");
  const int depth = lay->halo;
  const int64_t cnt = (int64_t)depth * lay->m;
  // The fused kernel and the stand-alone exchange (comm.cu) use different wire formats, so the choice must come out
  // the same on every rank: it depends on the row length and the halo depth only, never on this rank's slab.
  const bool fused = ctx->nranks > 1 && ctx->p2p_ready && ctx->p2p_fused && lay->m > 0 && (lay->m & 1) == 0 &&
                     depth >= 1 && cnt <= P2P_HMAX;
  if (fused)
    GNK_REQUIRE(depth <= lay->rows && (lay->ld & 1) == 0 && (lay->off & 1) == 0 && (lay->n_own & 1) == 0,
                "gnk_normalize_halo: slab layout (an even row length implies even off / n_own / ld; depth <= rows)");
  if (!fused) {
    if (int rc = gnk_normalize(ctx, lay, d_x, d_stats, atol, d_out, d_flag, stream)) return rc;
    if (ctx->nranks > 1 && lay->m > 0) return gnk_comm_halo_exchange(ctx, lay, d_out, depth, stream);
    return 0;
  }
  HaloPush hp{ctx->d_p2p_peer, ctx->rank, ctx->nranks, lay->has_lo, lay->has_hi, lay->off, lay->n_own, cnt,
              ++ctx->p2p_hseq};
  int grid = stream_grid(ctx, lay->ld / 2, 8);
  GNK_CUDA(gnk_launch(gnk_pdl_for(lay->n_own), normalize_halo_kernel, dim3(grid), dim3(TPB), 0, (cudaStream_t)stream, d_x, lay->ld, d_stats, atol,
                      d_out, d_flag, hp));
  GNK_LAUNCH_CHECK(ctx);
  return 0;
}

int gnk_cgs_dots(gnk_ctx* ctx, const gnk_layout* lay, const double* d_V, int k, const double* d_w, double* d_h,
                 void* stream) {
  GNK_REQUIRE(ctx && lay && d_V && d_w && d_h, "gnk_cgs_dots: null argument");
  GNK_REQUIRE(k >= 1 && k < GNK_MAX_BASIS_WIDE, "gnk_cgs_dots: k out of range");
  GNK_REQUIRE((lay->off & 1) == 0 && (lay->ld & 1) == 0, "gnk_cgs_dots: off/ld must be even");
  static_assert(TPB == DOTS_TPB, "dots_kernel runs dots_finish's block size");
  const int grid = dots_grid(ctx, lay->n_own);
  if (k >= GNK_MAX_BASIS) {
    static_assert(P2P_LLMAX >= GNK_MAX_BASIS_WIDE - 1, "the mailbox lines must hold the widest h");
    if (!ctx->d_wdots)  // dots_grid is at most 4 CTAs per SM
      GNK_CUDA(cudaMalloc(&ctx->d_wdots, sizeof(double) * 4 * (size_t)ctx->sm_count * GNK_MAX_BASIS_WIDE));
    GNK_CUDA(gnk_launch(gnk_pdl_for(lay->n_own), dots_wide_kernel, dim3(grid), dim3(TPB), 0, (cudaStream_t)stream,
                        d_V + lay->off, lay->ld, lay->n_own, k, d_w + lay->off, ctx->d_wdots,
                        ctx->d_tickets + TK_DOTS, d_h, p2p_next(ctx)));
    GNK_LAUNCH_CHECK(ctx);
    return 0;
  }
  GNK_CUDA(gnk_launch(gnk_pdl_for(lay->n_own), dots_kernel, dim3(grid), dim3(TPB), 0, (cudaStream_t)stream, d_V + lay->off, lay->ld, lay->n_own, k,
                      d_w + lay->off, ctx->d_partials + PART_DOTS, ctx->d_tickets + TK_DOTS, d_h, p2p_next(ctx)));
  GNK_LAUNCH_CHECK(ctx);
  return 0;
}

int gnk_cgs_update(gnk_ctx* ctx, const gnk_layout* lay, const double* d_V, int k, const double* d_h, double* d_w,
                   double* d_stats, void* stream) {
  GNK_REQUIRE(ctx && lay && d_V && d_w && d_h, "gnk_cgs_update: null argument");
  GNK_REQUIRE(k >= 1 && k < GNK_MAX_BASIS_WIDE, "gnk_cgs_update: k out of range");
  GNK_REQUIRE((lay->off & 1) == 0 && (lay->ld & 1) == 0, "gnk_cgs_update: off/ld must be even");
  int grid = stream_grid(ctx, lay->n_own / 2, 8);
  if (k >= GNK_MAX_BASIS) {
    GNK_CUDA(gnk_launch(gnk_pdl_for(lay->n_own), update_wide_kernel, dim3(grid), dim3(TPB), sizeof(double) * k,
                        (cudaStream_t)stream, d_V + lay->off, lay->ld, lay->n_own, k, d_h, d_w + lay->off,
                        ctx->d_partials + PART_UPDATE, ctx->d_tickets + TK_UPDATE, d_stats,
                        d_stats ? p2p_next(ctx) : gnk_p2p_dev{nullptr, 0, 1, 0ull}));
    GNK_LAUNCH_CHECK(ctx);
    return 0;
  }
  GNK_CUDA(gnk_launch(gnk_pdl_for(lay->n_own), update_kernel, dim3(grid), dim3(TPB), 0, (cudaStream_t)stream, d_V + lay->off, lay->ld, lay->n_own, k,
                      d_h, d_w + lay->off, ctx->d_partials + PART_UPDATE, ctx->d_tickets + TK_UPDATE, d_stats,
                      d_stats ? p2p_next(ctx) : gnk_p2p_dev{nullptr, 0, 1, 0ull}));
  GNK_LAUNCH_CHECK(ctx);
  return 0;
}

int gnk_axpby(gnk_ctx* ctx, int64_t n, double a, const double* d_x, double b, const double* d_y, double* d_out,
              void* stream) {
  GNK_REQUIRE(ctx && d_out && n >= 0, "gnk_axpby: bad argument");
  GNK_REQUIRE((a == 0.0 || d_x) && (b == 0.0 || d_y), "gnk_axpby: null operand with non-zero weight");
  if (n == 0) return 0;
  int grid = stream_grid(ctx, n, 8);
  axpby_kernel<<<grid, TPB, 0, (cudaStream_t)stream>>>(n, a, d_x, b, d_y, d_out);
  GNK_LAUNCH_CHECK(ctx);
  return 0;
}

int gnk_dot(gnk_ctx* ctx, int64_t n, const double* d_x, const double* d_y, double* d_out, void* stream) {
  GNK_REQUIRE(ctx && d_x && d_y && d_out && n >= 0, "gnk_dot: bad argument");
  int grid = stream_grid(ctx, n, 4);
  dot_kernel<<<grid, TPB, 0, (cudaStream_t)stream>>>(n, d_x, d_y, ctx->d_partials + PART_DOT1,
                                                     ctx->d_tickets + TK_DOT1, d_out);
  GNK_LAUNCH_CHECK(ctx);
  return 0;
}

}  // extern "C"
