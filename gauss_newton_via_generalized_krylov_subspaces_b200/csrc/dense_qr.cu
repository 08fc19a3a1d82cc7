// dense_qr.cu -- least squares on a dense panel of 256 <= p <= 4095 columns (gnk_dense_qr_ls): right-looking blocked
// Householder QR (LAPACK dgeqrf form) of the augmented panel [sign_a * A | y], in place, for the dense-Jacobian branch
// of gauss_newton (scipy.linalg.lstsq(-J, r), gauss_newton.py:116).
//
// Per panel of NB = 32 columns (j0 .. j0 + nbp - 1, rows j0 .. n - 1):
//   panel:   one cooperative kernel over the SMs factors the panel column by column in global memory.  Rows are dealt
//            round-robin to the threads of the grid; a thread keeps its rows for the whole panel.  Column j needs
//            |x_j|^2 below the diagonal and x_j^T a_c for the panel columns c > j: both come from ONE pass (the dots of
//            v_j = x_j / (alpha - beta) are scale * x_j^T a_c), summed per CTA in a fixed tree and over the CTAs in CTA
//            order by every CTA after a grid barrier, so every CTA derives the same IEEE dlarfg scalars (as wide_fold_tile
//            in tsqr.cu).  The pass that applies reflector j also forms the sums of column j + 1: one barrier per column.
//   T:       G = V^T V comes out of the V^T C product below (V's own columns are the first columns of that product);
//            dlarft builds T of Q = I - V T V^T from G and the taus.
//   update:  W = V^T C split over row blocks (partials summed in split order), W <- -T^T W, C <- C + V W, all three
//            products with mma.m8n8k4.f64 on the FP64 tensor pipe.  Column p (y) is a trailing column like the others,
//            so Q^T y comes out of the same updates.
// Then a single-CTA back substitution R d = (Q^T y)[0..p) and the scalar block of gnk_tsqr_ls.
// Every cross-CTA sum has a fixed order that depends on n, p and the SM count only: two calls give the same bits, and
// power-of-two scaling of A and y changes no rounding.
#include <cooperative_groups.h>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace {

constexpr int NB = 32;          // panel width
constexpr int PT = 256;         // threads of the panel kernel
constexpr int UT = 256;         // threads of the product kernels (8 warps)
constexpr int TM = 64;          // rows per tile of the product kernels
constexpr int TN = 64;          // columns per tile of the product kernels
constexpr int SLD = TM + 4;     // column stride of the shared tiles (DMMA fragment loads without bank conflicts)
constexpr int WLDS = TN + 4;    // row stride of W in shared memory
constexpr int TLD = NB + 4;     // row stride of T and G
constexpr int VK = 32;          // rows per chunk of the V^T C product
constexpr int VLD = VK + 4;     // column stride of its shared tiles
constexpr int ST = 1024;        // threads of the solve kernel

__device__ __forceinline__ void dmma(double (&d)[2], double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(d[0]), "+d"(d[1])
               : "d"(a), "d"(b));
}

// entry (row i, panel column l) of the unit lower trapezoidal V of the panel starting at column j0 (nbp reflectors)
__device__ __forceinline__ double v_entry(const double* __restrict__ P, int64_t lda, int64_t n, int j0, int nbp,
                                          int64_t i, int l) {
  if (l >= nbp || i >= n) return 0.0;
  const int64_t rel = i - j0;
  return rel > l ? P[(int64_t)(j0 + l) * lda + i] : (rel == l ? 1.0 : 0.0);
}

// per-CTA sums of the panel pass: slot `first` = nrm (|x|^2 below the next pivot), slots first+1 .. nbp-1 = acc[c];
// fixed warp tree, then warps in order
__device__ __forceinline__ void panel_publish(const double (&acc)[NB], double nrm, int first, int nbp,
                                              double (*red)[NB], double* __restrict__ dst) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int c = 0; c < NB; ++c) {
    if (c >= first && c < nbp) {
      const double v = warp_sum(c == first ? nrm : acc[c]);
      if (lane == 0) red[warp][c] = v;
    }
  }
  __syncthreads();
  const int t = threadIdx.x;
  if (t >= first && t < nbp) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < PT / 32; ++w) s += red[w][t];
    dst[t] = s;
  }
  __syncthreads();
}

// Factor panel columns j0 .. j0 + nbp - 1 over rows j0 .. n - 1 (cooperative launch).  part: 2 x gridDim.x x NB
// doubles (double-buffered per column), rowv: 2 x NB (the next pivot row, published by its owner), taus: NB.
__global__ void __launch_bounds__(PT) dqr_panel_kernel(double* __restrict__ P, int64_t lda, int64_t n, int j0, int nbp,
                                                       double* __restrict__ part, double* __restrict__ rowv,
                                                       double* __restrict__ taus) {
  cg::grid_group grid = cg::this_grid();
  __shared__ double red[PT / 32][NB];
  __shared__ double S[NB], rj[NB], w[NB];
  __shared__ double sc[3];
  const int G = gridDim.x;
  const int64_t stride = (int64_t)G * PT;
  const int64_t i0 = j0 + (int64_t)blockIdx.x * PT + threadIdx.x;
  double* const col = P + (int64_t)j0 * lda;  // panel column l of row i: col[l * lda + i]

  {  // sums of column 0 and the pivot row j0
    double acc[NB], nrm = 0.0;
#pragma unroll
    for (int c = 0; c < NB; ++c) acc[c] = 0.0;
    for (int64_t i = i0; i < n; i += stride) {
      const double* pi = col + i;
      if (i == j0) {
        for (int c = 0; c < nbp; ++c) rowv[c] = pi[(int64_t)c * lda];
        continue;
      }
      const double x = pi[0];
      nrm = fma(x, x, nrm);
#pragma unroll
      for (int c = 1; c < NB; ++c)
        if (c < nbp) acc[c] = fma(x, pi[(int64_t)c * lda], acc[c]);
    }
    panel_publish(acc, nrm, 0, nbp, red, part + (int64_t)blockIdx.x * NB);
  }

  for (int jl = 0; jl < nbp; ++jl) {
    grid.sync();
    const int par = jl & 1;
    const int64_t j = j0 + jl;
    const int t = threadIdx.x;
    if (t >= jl && t < nbp) {
      const double* src = part + (int64_t)par * G * NB + t;
      double s = 0.0;
      for (int b = 0; b < G; ++b) s += __ldcg(src + (int64_t)b * NB);
      S[t] = s;
      rj[t] = __ldcg(rowv + par * NB + t);
    }
    __syncthreads();
    if (t == 0) {  // dlarfg: H = I when the column is already zero below the diagonal
      const double alpha = rj[jl], sigma = S[jl];
      double beta = alpha, tau = 0.0, scale = 0.0;
      if (sigma != 0.0) {
        beta = -copysign(sqrt(fma(alpha, alpha, sigma)), alpha);
        tau = (beta - alpha) / beta;
        scale = 1.0 / (alpha - beta);
      }
      sc[0] = beta;
      sc[1] = tau;
      sc[2] = scale;
      if (blockIdx.x == 0) taus[jl] = tau;
    }
    __syncthreads();
    const double beta = sc[0], tau = sc[1], scale = sc[2];
    if (t > jl && t < nbp) w[t] = (rj[t] + scale * S[t]) * tau;  // tau * v^T a_t
    __syncthreads();

    const bool more = jl + 1 < nbp;
    const int64_t jn = j + 1;
    double* const rnext = rowv + (par ^ 1) * NB;
    double acc[NB], nrm = 0.0;
#pragma unroll
    for (int c = 0; c < NB; ++c) acc[c] = 0.0;
    for (int64_t i = i0; i < n; i += stride) {
      if (i < j) continue;
      double* pi = col + i;
      double vi;
      if (i == j) {
        vi = 1.0;
        pi[(int64_t)jl * lda] = beta;
      } else {
        vi = pi[(int64_t)jl * lda] * scale;
        pi[(int64_t)jl * lda] = vi;
      }
      if (!more) continue;
      const double xn = fma(-w[jl + 1], vi, pi[(int64_t)(jl + 1) * lda]);
      pi[(int64_t)(jl + 1) * lda] = xn;
      const bool below = i > jn;
      if (i == jn) rnext[jl + 1] = xn;
      const double xm = below ? xn : 0.0;
      nrm = fma(xm, xm, nrm);
#pragma unroll
      for (int c = 0; c < NB; ++c) {
        if (c > jl + 1 && c < nbp) {
          const double a = fma(-w[c], vi, pi[(int64_t)c * lda]);
          pi[(int64_t)c * lda] = a;
          if (i == jn) rnext[c] = a;
          acc[c] = fma(xm, a, acc[c]);
        }
      }
    }
    if (more) panel_publish(acc, nrm, jl + 1, nbp, red, part + ((int64_t)(par ^ 1) * G + blockIdx.x) * NB);
  }
}

// Wpart[s] (NB x ldw, row-major) = V^T [panel V | C] over row block s (rows j0 + s * rps ..), column tile blockIdx.x
// (columns j0 + TN * blockIdx.x ..): relative columns < nbp give G = V^T V, the others V^T C.
__global__ void __launch_bounds__(UT) dqr_vtc_kernel(const double* __restrict__ P, int64_t lda, int64_t n, int c,
                                                     int j0, int nbp, int64_t rps, double* __restrict__ Wpart,
                                                     int64_t ldw) {
  __shared__ double Vs[NB * VLD];
  __shared__ double Cs[TN * VLD];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int l4 = lane >> 2, m4 = lane & 3;
  const int row = threadIdx.x & (VK - 1), cgp = threadIdx.x / VK;
  const int ct0 = TN * blockIdx.x;
  const int64_t rb = j0 + (int64_t)blockIdx.y * rps;
  const int64_t re = min(rb + rps, n);
  double acc[4][2] = {{0.0, 0.0}, {0.0, 0.0}, {0.0, 0.0}, {0.0, 0.0}};
  for (int64_t r0 = rb; r0 < re; r0 += VK) {
    const int64_t i = r0 + row;
    const bool ok = i < re;
    __syncthreads();
#pragma unroll 4
    for (int l = cgp; l < NB; l += UT / VK) Vs[l * VLD + row] = ok ? v_entry(P, lda, n, j0, nbp, i, l) : 0.0;
#pragma unroll 8
    for (int q = cgp; q < TN; q += UT / VK) {
      const int rel = ct0 + q;
      const int cc = j0 + rel;
      double v = 0.0;
      if (ok) v = rel < nbp ? v_entry(P, lda, n, j0, nbp, i, rel) : (cc < c ? P[(int64_t)cc * lda + i] : 0.0);
      Cs[q * VLD + row] = v;
    }
    __syncthreads();
#pragma unroll
    for (int k0 = 0; k0 < VK; k0 += 4) {
      const double b = Cs[(8 * warp + l4) * VLD + k0 + m4];
#pragma unroll
      for (int mt = 0; mt < 4; ++mt) dmma(acc[mt], Vs[(8 * mt + l4) * VLD + k0 + m4], b);
    }
  }
  double* dst = Wpart + (int64_t)blockIdx.y * NB * ldw;
#pragma unroll
  for (int mt = 0; mt < 4; ++mt)
#pragma unroll
    for (int e = 0; e < 2; ++e) dst[(int64_t)(8 * mt + l4) * ldw + ct0 + 8 * warp + 2 * m4 + e] = acc[mt][e];
}

// W2 (NB x ldw, row-major) = -T^T (sum over the nsplit partials of W), column tile blockIdx.x, for relative columns
// >= nbp; every CTA sums G and builds T itself (dlarft, forward columnwise).
__global__ void __launch_bounds__(UT) dqr_tw_kernel(const double* __restrict__ Wpart, int64_t ldw, int nsplit, int nbp,
                                                    const double* __restrict__ taus, double* __restrict__ W2) {
  __shared__ double G[NB * TLD];
  __shared__ double T[NB * TLD];
  __shared__ double Ws[NB * WLDS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int l4 = lane >> 2, m4 = lane & 3;
  const int ct0 = TN * blockIdx.x;
  const int64_t sstride = (int64_t)NB * ldw;
  for (int e = threadIdx.x; e < NB * NB; e += UT) {
    const int a = e / NB, b = e - a * NB;
    double s = 0.0;
    for (int q = 0; q < nsplit; ++q) s += __ldcg(Wpart + q * sstride + (int64_t)a * ldw + b);
    G[a * TLD + b] = s;
  }
  for (int e = threadIdx.x; e < NB * TN; e += UT) {
    const int a = e / TN, b = e - a * TN;
    double s = 0.0;
    for (int q = 0; q < nsplit; ++q) s += __ldcg(Wpart + q * sstride + (int64_t)a * ldw + ct0 + b);
    Ws[a * WLDS + b] = s;
  }
  __syncthreads();
  if (warp == 0) {  // lane t forms row t of T from its own earlier entries
    const int t = lane;
    for (int i = 0; i < NB; ++i) {
      const double ti = i < nbp ? taus[i] : 0.0;
      double v = 0.0;
      if (i == t) {
        v = ti;
      } else if (i > t) {
        double s = 0.0;
        for (int l = t; l < i; ++l) s = fma(T[t * TLD + l], G[l * TLD + i], s);
        v = -ti * s;
      }
      T[t * TLD + i] = v;
    }
  }
  __syncthreads();
  double acc[4][2] = {{0.0, 0.0}, {0.0, 0.0}, {0.0, 0.0}, {0.0, 0.0}};
#pragma unroll
  for (int k0 = 0; k0 < NB; k0 += 4) {
    const double b = Ws[(k0 + m4) * WLDS + 8 * warp + l4];
#pragma unroll
    for (int mt = 0; mt < 4; ++mt) dmma(acc[mt], T[(k0 + m4) * TLD + 8 * mt + l4], b);
  }
#pragma unroll
  for (int mt = 0; mt < 4; ++mt)
#pragma unroll
    for (int e = 0; e < 2; ++e) W2[(int64_t)(8 * mt + l4) * ldw + ct0 + 8 * warp + 2 * m4 + e] = -acc[mt][e];
}

// C += V W2 on rows j0 + TM * blockIdx.x .. and the trailing columns (relative column >= nbp) of column tile blockIdx.y
// (columns j0 + TN * blockIdx.y .., the tiles of W2)
__global__ void __launch_bounds__(UT) dqr_update_kernel(double* __restrict__ P, int64_t lda, int64_t n, int c, int j0,
                                                        int nbp, const double* __restrict__ W2, int64_t ldw) {
  __shared__ double Vs[NB * SLD];
  __shared__ double Ws[NB * WLDS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int l4 = lane >> 2, m4 = lane & 3;
  const int64_t r0 = j0 + (int64_t)TM * blockIdx.x;
  const int rel0 = TN * blockIdx.y;
  const int cs = j0 + rel0;
  {
    const int row = threadIdx.x & (TM - 1), cgp = threadIdx.x / TM;
#pragma unroll 4
    for (int l = cgp; l < NB; l += UT / TM) Vs[l * SLD + row] = v_entry(P, lda, n, j0, nbp, r0 + row, l);
  }
  for (int e = threadIdx.x; e < NB * TN; e += UT) {
    const int a = e / TN, b = e - a * TN;
    Ws[a * WLDS + b] = W2[(int64_t)a * ldw + rel0 + b];
  }
  __syncthreads();
  const int64_t i = r0 + 8 * warp + l4;
  const bool rok = i < n;
  double cacc[TN / 8][2];
#pragma unroll
  for (int nt = 0; nt < TN / 8; ++nt)
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int cc = cs + 8 * nt + 2 * m4 + e;
      cacc[nt][e] = (rok && cc >= j0 + nbp && cc < c) ? P[(int64_t)cc * lda + i] : 0.0;
    }
#pragma unroll
  for (int k0 = 0; k0 < NB; k0 += 4) {
    const double av = Vs[(k0 + m4) * SLD + 8 * warp + l4];
#pragma unroll
    for (int nt = 0; nt < TN / 8; ++nt) dmma(cacc[nt], av, Ws[(k0 + m4) * WLDS + 8 * nt + l4]);
  }
#pragma unroll
  for (int nt = 0; nt < TN / 8; ++nt)
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int cc = cs + 8 * nt + 2 * m4 + e;
      if (rok && cc >= j0 + nbp && cc < c) P[(int64_t)cc * lda + i] = cacc[nt][e];
    }
}

__global__ void dqr_scale_kernel(double* __restrict__ P, int64_t lda, int64_t n, int p, double s) {
  const int64_t total = n * (int64_t)p;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t j = e / n, i = e - j * n;
    P[j * lda + i] *= s;
  }
}

__device__ __forceinline__ double solve_block_sum(double v, double* sh) {  // result in every thread, fixed order
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  double r = 0.0;
#pragma unroll
  for (int w = 0; w < ST / 32; ++w) r += sh[w];
  return r;
}

// back substitution R d = z = (Q^T y)[0..p) (column-oriented: once d_j is known every row above subtracts R_ij d_j) and
// the scalar block of gnk_tsqr_ls
__global__ void __launch_bounds__(ST) dqr_solve_kernel(const double* __restrict__ P, int64_t lda, int64_t n, int p,
                                                       double* __restrict__ out) {
  __shared__ double zs[GNK_DENSE_QR_MAX];
  __shared__ double sh[ST / 32];
  const int tid = threadIdx.x;
  const double* qy = P + (int64_t)p * lda;
  for (int i = tid; i < p; i += ST) zs[i] = qy[i];
  __syncthreads();
  for (int j = p - 1; j >= 0; --j) {
    const double* rc = P + (int64_t)j * lda;
    const double dj = zs[j] / rc[j];
    if (tid == 0) out[j] = dj;
    for (int i = tid; i < j; i += ST) zs[i] = fma(-rc[i], dj, zs[i]);
    __syncthreads();
  }
  double z2 = 0.0, d2 = 0.0, nd = 0.0, r2 = 0.0;
  for (int i = tid; i < p; i += ST) {
    const double rii = P[(int64_t)i * lda + i], z = qy[i], d = out[i];
    z2 = fma(z, z, z2);
    d2 = fma(d, d, d2);
    if (fabs(rii) <= 1e-8) nd += 1.0;
    out[p + 4 + i] = rii;
  }
  for (int64_t i = p + tid; i < n; i += ST) r2 = fma(qy[i], qy[i], r2);
  z2 = solve_block_sum(z2, sh);
  d2 = solve_block_sum(d2, sh);
  nd = solve_block_sum(nd, sh);
  r2 = solve_block_sum(r2, sh);
  if (tid == 0) {
    out[p] = z2;
    out[p + 1] = r2;
    out[p + 2] = nd;
    out[p + 3] = d2;
  }
}

// row splits of the V^T C product for the panel at j0: about two CTAs per SM over the column tiles
void vtc_split(int64_t n, int c, int j0, int sm, int* nsplit, int64_t* rps) {
  const int64_t m = n - j0;
  const int64_t ntile = ceil_div(c - j0, TN);
  const int64_t rtiles = ceil_div(m, VK);
  int64_t s = ceil_div(2 * (int64_t)sm, ntile);
  if (s > rtiles) s = rtiles;
  if (s < 1) s = 1;
  *rps = ceil_div(rtiles, s) * VK;
  *nsplit = (int)ceil_div(m, *rps);
}

int panel_grid_max(gnk_ctx* ctx) {
  static int occ_dev[64] = {0};
  int& occ = occ_dev[ctx->device & 63];
  if (occ == 0) {
    int o = 0;
    GNK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, dqr_panel_kernel, PT, 0));
    GNK_REQUIRE(o >= 1, "gnk_dense_qr_ls: the panel kernel does not fit an SM");
    occ = o < 2 ? o : 2;
  }
  return occ * ctx->sm_count;
}

// Blocked Householder factorisation of [sign_a * A | y] in place (everything of gnk_dense_qr_ls but the solve).
int dqr_factor(gnk_ctx* ctx, double* d_A, int64_t lda, int64_t n_rows, int p, double sign_a, cudaStream_t st) {
  const int c = p + 1;
  const int gmax = panel_grid_max(ctx);
  if (gmax <= 0) return -1;

  // workspace: panel partials 2 x gmax x NB, pivot rows 2 x NB, taus NB, W partials, W2 (NB x ldw)
  const int64_t ldw = ceil_div(c, TN) * TN;
  int64_t wpart = 0;
  for (int j0 = 0; j0 < p; j0 += NB) {
    int ns;
    int64_t rps;
    vtc_split(n_rows, c, j0, ctx->sm_count, &ns, &rps);
    const int64_t need = (int64_t)ns * NB * ldw;
    if (need > wpart) wpart = need;
  }
  const int64_t off_rowv = 2LL * gmax * NB, off_taus = off_rowv + 2 * NB, off_wpart = off_taus + NB;
  const int64_t off_w2 = off_wpart + wpart, total = off_w2 + NB * ldw;
  const size_t bytes = sizeof(double) * (size_t)total;
  if (bytes > ctx->dqr_bytes) {
    GNK_CUDA(cudaStreamSynchronize(st));
    if (ctx->d_dqr) GNK_CUDA(cudaFree(ctx->d_dqr));
    ctx->d_dqr = nullptr;
    ctx->dqr_bytes = 0;
    GNK_CUDA(cudaMalloc(&ctx->d_dqr, bytes));
    ctx->dqr_bytes = bytes;
  }
  double* part = ctx->d_dqr;
  double* rowv = part + off_rowv;
  double* taus = part + off_taus;
  double* wp = part + off_wpart;
  double* w2 = part + off_w2;

  if (sign_a != 1.0) {
    dqr_scale_kernel<<<4 * ctx->sm_count, 256, 0, st>>>(d_A, lda, n_rows, p, sign_a);
    GNK_LAUNCH_CHECK(ctx);
  }
  for (int j0 = 0; j0 < p; j0 += NB) {
    const int nbp = p - j0 < NB ? p - j0 : NB;
    const int64_t m = n_rows - j0;
    int64_t g = ceil_div(m, PT);
    if (g > gmax) g = gmax;
    int j0a = j0, nbpa = nbp;
    int64_t na = n_rows, ldaa = lda;
    void* args[] = {&d_A, &ldaa, &na, &j0a, &nbpa, &part, &rowv, &taus};
    GNK_CUDA(cudaLaunchCooperativeKernel((void*)dqr_panel_kernel, dim3((unsigned)g), dim3(PT), args, 0, st));
    GNK_LAUNCH_CHECK(ctx);

    int ns;
    int64_t rps;
    vtc_split(n_rows, c, j0, ctx->sm_count, &ns, &rps);
    const unsigned ntile = (unsigned)ceil_div(c - j0, TN);
    dqr_vtc_kernel<<<dim3(ntile, (unsigned)ns), UT, 0, st>>>(d_A, lda, n_rows, c, j0, nbp, rps, wp, ldw);
    GNK_LAUNCH_CHECK(ctx);
    // the column tiles of V^T C, T^T W and the update coincide; relative columns < nbp (the panel) are not updated
    dqr_tw_kernel<<<ntile, UT, 0, st>>>(wp, ldw, ns, nbp, taus, w2);
    GNK_LAUNCH_CHECK(ctx);
    dqr_update_kernel<<<dim3((unsigned)ceil_div(m, TM), ntile), UT, 0, st>>>(d_A, lda, n_rows, c, j0, nbp, w2, ldw);
    GNK_LAUNCH_CHECK(ctx);
  }
  return 0;
}

// ---- gnk_basis_ls_wide on several ranks -------------------------------------------------------------------------
// src: n x (p+1) panel (stride ld, n rows valid), dst: the same with rows_to >= n rows (stride ldd), zero-padded
__global__ void wls_pad_kernel(const double* __restrict__ src, int64_t ld, int64_t n, int p, double* __restrict__ dst,
                               int64_t ldd, int64_t rows_to) {
  const int64_t total = rows_to * (int64_t)(p + 1);
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t j = e / rows_to, i = e - j * rows_to;
    dst[j * ldd + i] = i < n ? src[j * ld + i] : 0.0;
  }
}

// T ((p+1) x (p+1), column-major, stride p+1) = [[R, z], [0, rho]] of a factored panel: R the upper triangle of
// columns 0..p-1, z = (Q^T y)[0..p); T[p][p] (rho) is written by wls_rho_kernel
__global__ void wls_pack_kernel(const double* __restrict__ P, int64_t lda, int p, double* __restrict__ T) {
  const int64_t c = p + 1, total = c * c;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t j = e / c, i = e - j * c;
    if (i == p && j == p) continue;
    T[e] = (i <= j && i < p) ? P[j * lda + i] : 0.0;
  }
}

// rho = sqrt(sum_{i >= p} (Q^T y)_i^2) in one CTA, fixed order
__global__ void __launch_bounds__(ST) wls_rho_kernel(const double* __restrict__ P, int64_t lda, int64_t n, int p,
                                                     double* __restrict__ T) {
  __shared__ double sh[ST / 32];
  const double* qy = P + (int64_t)p * lda;
  double s = 0.0;
  for (int64_t i = p + threadIdx.x; i < n; i += ST) s = fma(qy[i], qy[i], s);
  s = solve_block_sum(s, sh);
  if (threadIdx.x == 0) T[(int64_t)p * (p + 1) + p] = sqrt(s);
}

// stack (column-major, stride lds): rank r's triangle in rows r (p+1) .. (r+1) (p+1) - 1
__global__ void wls_stack_kernel(const double* __restrict__ G, int nranks, int p, double* __restrict__ S,
                                 int64_t lds) {
  const int64_t c = p + 1, tri = c * c, total = tri * nranks;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = e / tri, q = e - r * tri, j = q / c, i = q - j * c;
    S[j * lds + r * c + i] = G[e];
  }
}

int ensure_wls(gnk_ctx* ctx, size_t bytes, cudaStream_t st) {
  if (bytes <= ctx->wls_bytes) return 0;
  GNK_CUDA(cudaStreamSynchronize(st));
  if (ctx->d_wls) GNK_CUDA(cudaFree(ctx->d_wls));
  ctx->d_wls = nullptr;
  ctx->wls_bytes = 0;
  GNK_CUDA(cudaMalloc(&ctx->d_wls, bytes));
  ctx->wls_bytes = bytes;
  return 0;
}

}  // namespace

int gnk_comm_allgather_doubles(gnk_ctx* ctx, const double* d_send, double* d_recv, int64_t count, void* stream);

extern "C" int gnk_dense_qr_ls(gnk_ctx* ctx, double* d_A, int64_t lda, int64_t n_rows, int p, double sign_a,
                               double* d_out, void* stream) {
  GNK_REQUIRE(ctx && d_A && d_out, "gnk_dense_qr_ls: null argument");
  GNK_REQUIRE(p >= GNK_DENSE_QR_MIN && p <= GNK_DENSE_QR_MAX, "gnk_dense_qr_ls: p out of range");
  GNK_REQUIRE(n_rows >= p && lda >= n_rows, "gnk_dense_qr_ls: bad panel (needs n_rows >= p and lda >= n_rows)");
  GNK_REQUIRE(((uintptr_t)d_A & 7) == 0, "gnk_dense_qr_ls: the panel must be 8-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = dqr_factor(ctx, d_A, lda, n_rows, p, sign_a, st)) return rc;
  dqr_solve_kernel<<<1, ST, 0, st>>>(d_A, lda, n_rows, p, d_out);
  GNK_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" int gnk_basis_ls_wide(gnk_ctx* ctx, double* d_P, int64_t ldp, int64_t n_rows, int k, double sign_a,
                                 double* d_out, void* stream) {
  GNK_REQUIRE(ctx && d_P && d_out, "gnk_basis_ls_wide: null argument");
  GNK_REQUIRE(k >= GNK_DENSE_QR_MIN && k < GNK_MAX_BASIS_WIDE, "gnk_basis_ls_wide: k out of range (256..4095)");
  GNK_REQUIRE(n_rows >= 0 && ldp >= n_rows, "gnk_basis_ls_wide: bad panel (needs ldp >= n_rows)");
  GNK_REQUIRE(((uintptr_t)d_P & 7) == 0, "gnk_basis_ls_wide: the panel must be 8-byte aligned");
  if (ctx->nranks == 1) {
    GNK_REQUIRE(n_rows >= (int64_t)k + 1,
                "gnk_basis_ls_wide: fewer residuals than basis columns + 1 (the projected problem is underdetermined)");
    return gnk_dense_qr_ls(ctx, d_P, ldp, n_rows, k, sign_a, d_out, stream);
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t c = (int64_t)k + 1, tri = c * c, N = ctx->nranks;
  const int64_t ldpad = (c + 1) & ~(int64_t)1, lds = (N * c + 1) & ~(int64_t)1;
  const bool pad = n_rows < c;
  // scratch: [padded slab | own triangle | gathered triangles | stacked panel]
  const int64_t off_tri = pad ? ldpad * c : 0, off_all = off_tri + tri, off_stack = off_all + N * tri;
  if (int rc = ensure_wls(ctx, sizeof(double) * (size_t)(off_stack + lds * c), st)) return rc;
  double* base = ctx->d_wls;
  double* slab = d_P;
  int64_t ld = ldp, rows = n_rows;
  if (pad) {
    wls_pad_kernel<<<ctx->sm_count, 256, 0, st>>>(d_P, ldp, n_rows, k, base, ldpad, c);
    GNK_LAUNCH_CHECK(ctx);
    slab = base;
    ld = ldpad;
    rows = c;
  }
  if (int rc = dqr_factor(ctx, slab, ld, rows, k, sign_a, st)) return rc;
  wls_pack_kernel<<<ctx->sm_count, 256, 0, st>>>(slab, ld, k, base + off_tri);
  GNK_LAUNCH_CHECK(ctx);
  wls_rho_kernel<<<1, ST, 0, st>>>(slab, ld, rows, k, base + off_tri);
  GNK_LAUNCH_CHECK(ctx);
  if (int rc = gnk_comm_allgather_doubles(ctx, base + off_tri, base + off_all, tri, st)) return rc;
  wls_stack_kernel<<<4 * ctx->sm_count, 256, 0, st>>>(base + off_all, (int)N, k, base + off_stack, lds);
  GNK_LAUNCH_CHECK(ctx);
  if (int rc = dqr_factor(ctx, base + off_stack, lds, N * c, k, 1.0, st)) return rc;
  dqr_solve_kernel<<<1, ST, 0, st>>>(base + off_stack, lds, N * c, k, d_out);
  GNK_LAUNCH_CHECK(ctx);
  return 0;
}
