// cholqr.cu -- projected least squares  min || sign*A d - y ||  on the FP64 tensor pipe: Gram matrix by DMMA,
// Cholesky, then one refinement pass (or the second pass of CholeskyQR2 for ill-conditioned panels).
// Second implementation of scipy.linalg.qr + solve_triangular (gauss_newton_krylow.py:30-35) for the large panels of
// the Bratu runs; the Householder TSQR of tsqr.cu stays the reference implementation and the fallback.
//
// Why: Householder QR of a 64 x c tile is a chain of c dependent reflector steps; measured on B200 the warp-autonomous
// leaf keeps the FP64 pipe 48 % busy (4.2 ms at n = 4096^2, c = 31; DESIGN.md section 3).  The Gram matrix
// G = P^T P of the panel P = [sign*A | y] has no dependency chain at all: it is a stream of independent
// mma.sync.m8n8k4.f64 (DMMA) instructions whose A and B fragments are the SAME registers -- lane (g, t) of a warp holds
// P[row t][column 8 I + g], which is both the A fragment of block row I and the B fragment of block column I, so
// every panel element is loaded from HBM exactly once (128-bit loads) and used in NB + 1 DMMAs.
//
// Numerics: a single Cholesky factor of G loses cond(P)^2 eps.  Two second passes repair that; the first factor kernel
// picks one ON THE DEVICE from the Cholesky pivot ratios (status word; the kernel of the other form returns at once):
//   refinement form (cond <~ 1e5, every Bratu run): d0 from the normal equations, one HBM-bound pass
//     rho = y - A d0, g = A^T rho, and d = d0 + (R1^T R1)^{-1} g; the iteration contracts by cond^2 eps per step;
//   CholeskyQR2 (Yamamoto, Nakatsukasa, Yanagisawa, Fukaya 2015): B = P R1^{-1}, R2 = chol(B^T B), R = R2 R1.  B is never
//     stored: pass 2 re-reads the panel, multiplies each 8-row group by T = R1^{-1} with DMMAs whose OUTPUT fragments
//     (lane (g, t): B^T[8 J + g][rows 2t, 2t+1]) are again directly the A/B fragments of the Gram DMMAs.
// The factor kernels refuse (sentinel in the result block, see gnk_b200.h) when a Cholesky pivot falls below 1e-12 of
// its diagonal entry -- near-consistent or rank-deficient systems -- or when the refinement step is not small, and the
// host re-issues the solve with the Householder path.
//
// Cost per 8 panel rows at c <= 32: 20 DMMAs (pass 1) + 4 k FMAs per row pair (refinement) or 40 DMMAs (CholeskyQR2)
// against ~c^2 dependent DFMAs per row; two reads of the panel (16 n c bytes).  Multi-GPU: the Gram matrices are summed
// over the ranks in rank order inside the single-CTA factor kernels (peer-mailbox all-reduce, bit-identical decisions
// on every rank), replacing the TSQR triangle gather and the tree levels.
#include <cuda.h>
#include <stdint.h>
#include <stdlib.h>

#include "common.cuh"

int gnk_comm_allgather_doubles(gnk_ctx* ctx, const double* d_send, double* d_recv, int64_t count, void* stream);

namespace {

constexpr int GW = 12;          // warps per CTA: one CTA per SM with up to 168 registers per thread
constexpr int GT = 32 * GW;
constexpr int CH = 16;          // panel rows per warp and load group (RU groups per step)
constexpr int TLD = 36;         // leading dimension of T in shared memory (conflict-free fragment reads)
constexpr int MAXC = 32;        // widest panel (k + 1)

__host__ __device__ constexpr int nblocks(int NB) { return NB * (NB + 1) / 2; }
__host__ __device__ constexpr int blk_index(int NB, int I, int J) { return I * NB - I * (I - 1) / 2 + (J - I); }

__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
      : "+d"(c0), "+d"(c1)
      : "d"(a), "d"(b));
}

struct PanelSource {
  const double* A;
  int64_t lda;
  const double* y;
  int k;
  int64_t n_rows;
};

__device__ __forceinline__ const double* column_ptr(const PanelSource& s, int col) {
  return col < s.k ? s.A + (int64_t)col * s.lda : (col == s.k ? s.y : nullptr);
}
__device__ __forceinline__ double2 load_pair(const double* p, int64_t r, int64_t limit) {
  if (p != nullptr && r < limit) return __ldcs(reinterpret_cast<const double2*>(p + r));
  return make_double2(0.0, 0.0);
}

// Sum the per-warp fragment accumulators of a CTA in warp order, publish the CTA's partial, and let the CTA that
// arrives last add the partials of all CTAs in CTA order (deterministic).  NE = doubles per Gram matrix in fragment
// order: block (I <= J) * 64 + lane * 2 + {0, 1}  <->  G[8 I + g][8 J + 2 t + {0, 1}].
// NW = warps of the CTA that hold accumulators (the first NW warps), NT = threads of the CTA (all take part in the
// barriers and the copies).
template <int NBLK, int NW = GW, int NT = GT>
__device__ __forceinline__ void reduce_gram(double (&acc)[NBLK][2], double* red, double* __restrict__ partials,
                                            unsigned int* ticket, double* __restrict__ Gout) {
  constexpr int NE = NBLK * 64;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int w = 0; w < NW; ++w) {
    if (warp == w) {
#pragma unroll
      for (int b = 0; b < NBLK; ++b) {
        double2* p = reinterpret_cast<double2*>(red + b * 64 + lane * 2);
        double2 v = make_double2(acc[b][0], acc[b][1]);
        if (w > 0) {
          const double2 o = *p;
          v.x += o.x;
          v.y += o.y;
        }
        *p = v;
      }
    }
    __syncthreads();
  }
  double* mine = partials + (int64_t)blockIdx.x * NE;
  for (int e = threadIdx.x; e < NE; e += NT) mine[e] = red[e];
  __threadfence();  // every thread publishes its own stores before the CTA takes its ticket
  if (!grid_arrive_last(ticket)) return;
  const int nb = gridDim.x;
  for (int e = threadIdx.x; e < NE; e += NT) {
    double s = 0.0;
    int b = 0;
    for (; b + 4 <= nb; b += 4) {
      const double v0 = __ldcg(partials + (int64_t)(b + 0) * NE + e);
      const double v1 = __ldcg(partials + (int64_t)(b + 1) * NE + e);
      const double v2 = __ldcg(partials + (int64_t)(b + 2) * NE + e);
      const double v3 = __ldcg(partials + (int64_t)(b + 3) * NE + e);
      s = (((s + v0) + v1) + v2) + v3;
    }
    for (; b < nb; ++b) s += __ldcg(partials + (int64_t)b * NE + e);
    Gout[e] = s;
  }
}

// ---- pass 1: G = P^T P --------------------------------------------------------------------------------------------
template <int NB, int RU>
struct GramTile {
  double2 v[NB][2 * RU];  // [column block][8-row group]: rows r0 + 8 h + 2 t + {0, 1} of column 8 I + g
};

template <int NB, int RU>
__device__ __forceinline__ void gram_load(GramTile<NB, RU>& T, const double* const (&cp)[NB], int64_t r0,
                                          int64_t limit, int t) {
#pragma unroll
  for (int I = 0; I < NB; ++I)
#pragma unroll
    for (int h = 0; h < 2 * RU; ++h) T.v[I][h] = load_pair(cp[I], r0 + 8 * h + 2 * t, limit);
}
template <int NB, int RU>
__device__ __forceinline__ void gram_accumulate(const GramTile<NB, RU>& T, double (&acc)[nblocks(NB)][2]) {
#pragma unroll
  for (int h = 0; h < 2 * RU; ++h)
#pragma unroll
    for (int I = 0; I < NB; ++I)
#pragma unroll
      for (int J = I; J < NB; ++J) {
        const int b = blk_index(NB, I, J);
        dmma(acc[b][0], acc[b][1], T.v[I][h].x, T.v[J][h].x);
        dmma(acc[b][0], acc[b][1], T.v[I][h].y, T.v[J][h].y);
      }
}

template <int NB, int RU>
__global__ void __launch_bounds__(GT, 1)
    cholqr_gram_kernel(PanelSource src, int64_t rows_per_cta, double* __restrict__ partials, unsigned int* ticket,
                       double* __restrict__ Gout) {
  constexpr int NBLK = nblocks(NB);
  __shared__ __align__(16) double red[NBLK * 64];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  pdl_begin();
  const double* cp[NB];
#pragma unroll
  for (int I = 0; I < NB; ++I) cp[I] = column_ptr(src, 8 * I + g);
  double acc[NBLK][2];
#pragma unroll
  for (int b = 0; b < NBLK; ++b) acc[b][0] = acc[b][1] = 0.0;

  const int64_t row0 = (int64_t)blockIdx.x * rows_per_cta;
  int64_t limit = row0 + rows_per_cta;
  if (limit > src.n_rows) limit = src.n_rows;
  constexpr int64_t STRIDE = (int64_t)CH * RU * GW;
  int64_t r = row0 + (int64_t)warp * (CH * RU);
  if constexpr (NB <= 3) {
    // three rotating register tiles: two steps are in flight while the third is multiplied -- with one step in flight
    // the narrow panels waited on HBM (ncu: long_scoreboard; 4.8 TB/s at NB = 3).  Measured: NB = 3 -5 %, NB = 2 equal
    GramTile<NB, RU> ta, tb, tc;
    gram_load(ta, cp, r, limit, t);
    gram_load(tb, cp, r + STRIDE, limit, t);
    while (r < limit) {
      gram_load(tc, cp, r + 2 * STRIDE, limit, t);
      gram_accumulate(ta, acc);
      r += STRIDE;
      if (r >= limit) break;
      gram_load(ta, cp, r + 2 * STRIDE, limit, t);
      gram_accumulate(tb, acc);
      r += STRIDE;
      if (r >= limit) break;
      gram_load(tb, cp, r + 2 * STRIDE, limit, t);
      gram_accumulate(tc, acc);
      r += STRIDE;
    }
  } else {
    // NB = 4 is bound by the tensor pipe and HBM at the same time; a third tile (168 registers) measured 10 % slower
    GramTile<NB, RU> ta, tb;
    gram_load(ta, cp, r, limit, t);
    while (r < limit) {
      gram_load(tb, cp, r + STRIDE, limit, t);
      gram_accumulate(ta, acc);
      r += STRIDE;
      if (r >= limit) break;
      gram_load(ta, cp, r + STRIDE, limit, t);
      gram_accumulate(tb, acc);
      r += STRIDE;
    }
  }
  reduce_gram<NBLK>(acc, red, partials, ticket, Gout);
}

// ---- pass 2: G2 = B^T B with B = P T formed on the fly ---------------------------------------------------------------
template <int NB, int RU>
struct RowTile {
  double2 v[RU][2 * NB];  // [16-row group u][4-column chunk I']: rows r0 + 16 u + 2 g + {0, 1} of column 4 I' + t
};
template <int NB, int RU>
__device__ __forceinline__ void row_load(RowTile<NB, RU>& T, const PanelSource& s, int64_t r0, int64_t limit, int g,
                                         int t) {
#pragma unroll
  for (int Ip = 0; Ip < 2 * NB; ++Ip) {
    const double* p = column_ptr(s, 4 * Ip + t);
#pragma unroll
    for (int u = 0; u < RU; ++u) T.v[u][Ip] = load_pair(p, r0 + 16 * u + 2 * g, limit);
  }
}
// one group of 8 panel rows (the .x or the .y halves of a RowTile): B^T = T^T P^T block by block, then B^T B
template <int NB>
__device__ __forceinline__ void row_group(const double (&p)[2 * NB], const double* __restrict__ Ts, int g, int t,
                                          double (&acc)[nblocks(NB)][2]) {
  double bt[NB][2];
#pragma unroll
  for (int J = 0; J < NB; ++J) {
    bt[J][0] = bt[J][1] = 0.0;
#pragma unroll
    for (int Ip = 0; Ip < 2 * NB; ++Ip) {
      if (Ip <= 2 * J + 1) {  // T is upper triangular: rows 4 I' .. 4 I' + 3 reach block column J only if 4 I' <= 8 J + 7
        const double a = Ts[(4 * Ip + t) * TLD + 8 * J + g];
        dmma(bt[J][0], bt[J][1], a, p[Ip]);
      }
    }
  }
#pragma unroll
  for (int I = 0; I < NB; ++I)
#pragma unroll
    for (int J = I; J < NB; ++J) {
      const int b = blk_index(NB, I, J);
      dmma(acc[b][0], acc[b][1], bt[I][0], bt[J][0]);
      dmma(acc[b][0], acc[b][1], bt[I][1], bt[J][1]);
    }
}
template <int NB, int RU>
__device__ __forceinline__ void row_accumulate(const RowTile<NB, RU>& T, const double* __restrict__ Ts, int g, int t,
                                               double (&acc)[nblocks(NB)][2]) {
  double p[2 * NB];
#pragma unroll
  for (int u = 0; u < RU; ++u) {
#pragma unroll
    for (int Ip = 0; Ip < 2 * NB; ++Ip) p[Ip] = T.v[u][Ip].x;
    row_group<NB>(p, Ts, g, t, acc);
#pragma unroll
    for (int Ip = 0; Ip < 2 * NB; ++Ip) p[Ip] = T.v[u][Ip].y;
    row_group<NB>(p, Ts, g, t, acc);
  }
}

template <int NB, int RU>
__global__ void __launch_bounds__(GT, 1)
    cholqr_gram2_kernel(PanelSource src, int64_t rows_per_cta, const double* __restrict__ Tg,
                        const int* __restrict__ status, double* __restrict__ partials, unsigned int* ticket,
                        double* __restrict__ Gout) {
  constexpr int NBLK = nblocks(NB);
  __shared__ __align__(16) double red[NBLK * 64];
  __shared__ __align__(16) double Ts[MAXC * TLD];
  if (*status != 2) return;  // refused, or the refinement form was chosen (uniform across the grid)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  for (int e = threadIdx.x; e < MAXC * TLD; e += GT) Ts[e] = Tg[e];
  __syncthreads();
  double acc[NBLK][2];
#pragma unroll
  for (int b = 0; b < NBLK; ++b) acc[b][0] = acc[b][1] = 0.0;

  const int64_t row0 = (int64_t)blockIdx.x * rows_per_cta;
  int64_t limit = row0 + rows_per_cta;
  if (limit > src.n_rows) limit = src.n_rows;
  constexpr int64_t STRIDE = (int64_t)CH * RU * GW;
  int64_t r = row0 + (int64_t)warp * (CH * RU);
  RowTile<NB, RU> ta, tb;
  row_load(ta, src, r, limit, g, t);
  while (r < limit) {
    row_load(tb, src, r + STRIDE, limit, g, t);
    row_accumulate(ta, Ts, g, t, acc);
    r += STRIDE;
    if (r >= limit) break;
    row_load(ta, src, r + STRIDE, limit, g, t);
    row_accumulate(tb, Ts, g, t, acc);
    r += STRIDE;
  }
  reduce_gram<NBLK>(acc, red, partials, ticket, Gout);
}

// ---- pass 2, refinement form: rho = y - (sign A) d0,  g = (sign A)^T rho,  sum rho^2 ---------------------------------
// One HBM-bound pass: a thread owns two adjacent rows (128-bit loads, a warp reads 512 contiguous bytes per column),
// holds their k entries in registers between the two loops (rho needs the whole row before g can start), and keeps
// its k partial sums of g in registers until the end.  FP64 work is 4 k FMAs per row pair -- the pipe idles.
constexpr int RT = 256;  // threads per CTA
template <int KC>
__global__ void __launch_bounds__(RT, 1)
    cholqr_refine_kernel(PanelSource src, double sign, const double* __restrict__ d0g, const int* __restrict__ status,
                         int64_t rows_per_cta, double* __restrict__ partials, unsigned int* ticket,
                         double* __restrict__ gout) {
  __shared__ double ds[KC];
  __shared__ double wsum[RT / 32][KC + 1];
  pdl_begin();
  if (*status != 0) return;  // the CholeskyQR2 form was chosen, or pass 1 refused (uniform across the grid)
  const int k = src.k;
  for (int j = threadIdx.x; j < KC; j += RT) ds[j] = (j < k) ? sign * d0g[j] : 0.0;
  __syncthreads();
  double g[KC];
#pragma unroll
  for (int j = 0; j < KC; ++j) g[j] = 0.0;
  double rr = 0.0;
  const int64_t row0 = (int64_t)blockIdx.x * rows_per_cta;
  int64_t limit = row0 + rows_per_cta;
  if (limit > src.n_rows) limit = src.n_rows;
  for (int64_t r = row0 + 2 * threadIdx.x; r < limit; r += 2 * RT) {
    double2 a[KC];
#pragma unroll
    for (int j = 0; j < KC; ++j)
      a[j] = (j < k) ? __ldcs(reinterpret_cast<const double2*>(src.A + (int64_t)j * src.lda + r)) : make_double2(0.0, 0.0);
    double2 rho = __ldcs(reinterpret_cast<const double2*>(src.y + r));
#pragma unroll
    for (int j = 0; j < KC; ++j) {
      rho.x = fma(-ds[j], a[j].x, rho.x);
      rho.y = fma(-ds[j], a[j].y, rho.y);
    }
#pragma unroll
    for (int j = 0; j < KC; ++j) g[j] = fma(a[j].x, rho.x, fma(a[j].y, rho.y, g[j]));
    rr = fma(rho.x, rho.x, fma(rho.y, rho.y, rr));
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int j = 0; j < KC; ++j) {
    const double v = warp_sum(g[j]);
    if (lane == 0) wsum[warp][j] = v;
  }
  rr = warp_sum(rr);
  if (lane == 0) wsum[warp][KC] = rr;
  __syncthreads();
  double* mine = partials + (int64_t)blockIdx.x * (KC + 1);
  if (threadIdx.x <= KC) {
    double v = wsum[0][threadIdx.x];
#pragma unroll
    for (int w = 1; w < RT / 32; ++w) v += wsum[w][threadIdx.x];
    mine[threadIdx.x] = v;
    __threadfence();
  }
  if (!grid_arrive_last(ticket)) return;
  if (threadIdx.x <= KC) {
    double v = 0.0;
    const int nb = gridDim.x;
    for (int b = 0; b < nb; ++b) v += __ldcg(partials + (int64_t)b * (KC + 1) + threadIdx.x);
    if (threadIdx.x < k) gout[threadIdx.x] = sign * v;   // (sign A)^T rho
    if (threadIdx.x == KC) gout[k] = v;                  // sum rho^2
  }
}

// ---- the small factorisations (one warp) -------------------------------------------------------------------------------
constexpr int GLD = MAXC + 1;
constexpr double PIVOT_FLOOR_1 = 1e-12;  // pass 1: reduced pivot / diagonal entry ~ 1 / cond^2 of the leading columns
constexpr double PIVOT_FLOOR_2 = 0.25;   // pass 2: G2 = I + O(cond^2 eps)
// The second pass has two forms (status word written by the first factor kernel selects one, the other kernel exits):
//   status 0  REFINE   one step of iterative refinement of the normal-equation solution: rho = y - A d0,
//                      g = A^T rho in one HBM-bound pass (2 k FMAs per row), d = d0 + (R1^T R1)^{-1} g.  The iteration
//                      contracts by cond^2 eps per step, so it is taken when every pivot ratio of the A columns is
//                      >= REFINE_FLOOR (cond <~ 1e5: the correction is then <~ 1e-6 |d| and what is left after it
//                      is below eps cond); the finishing kernel re-checks |delta| <= REFINE_ACCEPT |d| and refuses
//                      otherwise (-> Householder).
//   status 2  CHOLQR2  the Gram matrix of P R1^{-1} (above); any conditioning the pivot floor admits.
//   status 1  refused by the pivot floor.
constexpr double REFINE_FLOOR = 1e-10;
constexpr double REFINE_ACCEPT = 1e-5;
constexpr int GPAD = 40;  // g (k values) + sum rho^2, padded; the Gram matrix of pass 2 follows in the gather buffer
constexpr int64_t NE_MAX = nblocks(4) * 64;  // doubles of the widest Gram matrix in fragment order (640)

// The small factorisations run in ONE CTA of 32 x 32 threads: thread (i = warp, l = lane) owns matrix entry [i][l].
// (History: one warp with the matrix in shared memory took 40 us for c = 31 -- a chain of shared-memory round trips;
// one warp with the matrix in registers and everything unrolled took the same, waiting for 100 KB of straight-line
// code to arrive from the instruction cache.  Compact loops over a 1024-thread CTA: a few us.)
constexpr int FT = MAXC * MAXC;
constexpr int RB = MAXC + 2;  // published row + the reciprocal of its pivot

// Upper Cholesky factor G = R^T R, right-looking.  a: my entry of G (upper part; anything finite elsewhere).  Step j:
// warp j publishes row j and 1 / a_jj, one barrier, every thread below row j subtracts a_ji * a_jl / a_jj.  The
// square roots and the divisions R_jl = a_jl / sqrt(a_jj) are all taken after the loop (one latency, not c).
// Returns R[i][l] in r (zero outside the upper triangle of the leading c x c block); false (uniformly) if a pivot is
// not safely positive.
__device__ __forceinline__ bool block_cholesky(double a, int c, double floor_rel, double* rowbuf, double* diag,
                                               double& r, double& min_ratio) {
  const int i = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (i == l) diag[l] = a;  // read after the first barrier
  double a_pub = 0.0, piv_pub = 1.0;
  bool ok = true;
  min_ratio = 1.0;  // min over the first c - 1 columns of reduced pivot / diagonal entry ~ 1 / cond^2 of [A] alone
  for (int j = 0; j < c; ++j) {
    double* rb = rowbuf + (j & 1) * RB;
    if (i == j) {
      const double ajj = __shfl_sync(0xffffffffu, a, j);
      rb[l] = a;
      if (l == 0) rb[MAXC] = __drcp_rn(ajj);
      a_pub = a;
      piv_pub = ajj;
    }
    __syncthreads();
    const double ajj = rb[j], dj = diag[j];
    if (!(ajj > floor_rel * dj) || !(dj > 0.0)) {  // every thread reads the same two numbers
      ok = false;
      break;
    }
    if (j < c - 1) min_ratio = fmin(min_ratio, ajj / dj);
    if (i > j && l >= i) a = fma(-rb[i], rb[l] * rb[MAXC], a);  // the lower triangle stays zero
  }
  r = 0.0;
  if (ok && i < c && l < c && l >= i) {
    const double piv = sqrt(piv_pub);
    r = (l == i) ? piv : a_pub / piv;
  }
  return ok;
}

// T = R^{-1} for the upper triangular R in Rs (row * GLD + column): back substitution with the 32 unit vectors as
// right-hand sides, thread (i, l) carries entry [i][l] of the running right-hand side.  Returns T[i][l].
__device__ __forceinline__ double block_tri_inverse(const double* Rs, int c, double* rowbuf) {
  const int i = threadIdx.x >> 5, l = threadIdx.x & 31;
  const bool in = (i < c && l < c);
  const double rinv = in ? 1.0 / Rs[i * GLD + i] : 0.0;
  double x = (in && i == l) ? 1.0 : 0.0, t = 0.0;
  for (int m = c - 1; m >= 0; --m) {
    double* rb = rowbuf + (m & 1) * RB;
    if (i == m) {
      t = x * rinv;
      rb[l] = t;
    }
    __syncthreads();
    if (i < m) x = fma(-Rs[i * GLD + m], rb[l], x);
  }
  return (in && l >= i) ? t : 0.0;
}

// the Gram matrix in fragment order (ranks added in rank order) -> my entry [i][l] (upper part; zero elsewhere)
__device__ __forceinline__ double gather_gram(const double* __restrict__ parts, int nparts, int NB, int c,
                                              int stride) {
  const int i = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (!(i <= l && l < c)) return 0.0;
  const int I = i >> 3, J = l >> 3;
  const int b = I * NB - I * (I - 1) / 2 + (J - I);
  const int e = b * 64 + ((i & 7) * 4 + ((l & 7) >> 1)) * 2 + (l & 1);
  double s = parts[e];
  for (int r = 1; r < nparts; ++r) s += parts[(int64_t)r * stride + e];
  return s;
}

// Result block of a refused solve: d = 0 (the trial the host has already queued evaluates the unchanged iterate),
// rank-deficiency count -1 = "re-issue with the Householder path" (gnk_b200.h).
__device__ void write_refusal(int k, double* out) {
  for (int i = threadIdx.x; i < k; i += blockDim.x) {
    out[i] = 0.0;
    out[k + 4 + i] = 1.0;
  }
  if (threadIdx.x == 0) {
    out[k] = 0.0;
    out[k + 1] = 0.0;
    out[k + 2] = -1.0;
    out[k + 3] = 0.0;
  }
}

// phase 1: R1 = chol(G), T = R1^{-1} with the sign of the A columns folded in (rows i < k of T scaled by sign), the
// normal-equation solution d0 = R1[:k,:k]^{-1} R1[:k,k] and ||A d0||^2 = |R1[:k,k]|^2 for the refinement form, and
// the choice of the second pass (status).
__global__ void __launch_bounds__(FT) cholqr_factor1_kernel(const double* __restrict__ parts, int nparts, int NB, int k,
                                                            double sign, int method, double* __restrict__ Tg,
                                                            double* __restrict__ R1g, double* __restrict__ d0g,
                                                            double* __restrict__ aux, int* __restrict__ status,
                                                            gnk_p2p_dev pd) {
  __shared__ double Rs[MAXC * GLD];
  __shared__ double rowbuf[2 * RB];
  __shared__ double diag[MAXC];
  __shared__ double gsh[NE_MAX];
  const int c = k + 1;
  const int i = threadIdx.x >> 5, l = threadIdx.x & 31;
  pdl_begin();
  if (pd.peers) {
    // compute step + collective in one kernel: this single CTA runs the mailbox all-reduce of the rank's Gram matrix
    // itself (p2p_tail_allreduce, common.cuh: stores into the peers' HBM over NVLink, flags, rank-ordered sum)
    const int NE = nblocks(NB) * 64;
    if (threadIdx.x < NE) gsh[threadIdx.x] = parts[threadIdx.x];
    __syncthreads();
    p2p_tail_allreduce(pd, gsh, NE, 0);
    __syncthreads();
    parts = gsh;
    nparts = 1;
  }
  double a = gather_gram(parts, nparts, NB, c, nblocks(NB) * 64);
  if (l == k && i < k) a *= sign;  // (sign A)^T y
  if (l == k && i < k) aux[1 + i] = a;  // b = (sign A)^T y for the finishing kernel: ||A d||^2 = b^T d at the solution
  double r, min_ratio;
  const bool ok = block_cholesky(a, c, PIVOT_FLOOR_1, rowbuf, diag, r, min_ratio);
  if (threadIdx.x == 0) *status = ok ? ((method != 2 && min_ratio >= REFINE_FLOOR) ? 0 : 2) : 1;
  R1g[i * MAXC + l] = ok ? r : 0.0;
  double t = 0.0;
  if (ok) {
    Rs[i * GLD + l] = r;
    __syncthreads();  // also separates the row buffers of the two loops
    if (threadIdx.x < 32) {
      // normal-equation solution by back substitution R1[:k,:k] d0 = z, z = R1[:k,k] (lane = row; once d0_j is known
      // every row above subtracts R_ij d0_j) -- the explicit inverse T = R1^{-1} (c more block-wide steps with a
      // barrier each) is formed only for the second CholeskyQR2 pass, which the default chain no longer runs
      const bool row = l < k;
      double z = row ? Rs[l * GLD + k] : 0.0;
      const double rinv = row ? 1.0 / Rs[l * GLD + l] : 1.0;
      const double z2 = warp_sum(z * z);
      double d = 0.0;
      for (int j = k - 1; j >= 0; --j) {
        const double dj = __shfl_sync(0xffffffffu, z, j) * __shfl_sync(0xffffffffu, rinv, j);
        if (l == j) d = dj;
        if (l < j) z = fma(-Rs[l * GLD + j], dj, z);
      }
      if (row) d0g[l] = d;
      if (l == 0) aux[0] = z2;
    }
    if (method == 2) {
      t = block_tri_inverse(Rs, c, rowbuf);
      if (i < k) t *= sign;
    }
  }
  Tg[i * TLD + l] = t;
  if (l < TLD - MAXC) Tg[i * TLD + MAXC + l] = 0.0;
}

// phase 2: R2 = chol(G2), R = R2 R1, back substitution and the scalar block of gnk_tsqr_ls.
__global__ void __launch_bounds__(FT) cholqr_factor2_kernel(const double* __restrict__ parts, int nparts, int NB, int k,
                                                            const double* __restrict__ R1g,
                                                            const double* __restrict__ Tg,
                                                            const double* __restrict__ d0g,
                                                            const double* __restrict__ aux,
                                                            const int* __restrict__ status, int have_g2,
                                                            double* __restrict__ out, gnk_p2p_dev pd) {
  __shared__ double R2s[MAXC * GLD];
  __shared__ double R1s[MAXC * GLD];
  __shared__ double Rs[MAXC * GLD];
  __shared__ double rowbuf[2 * RB];
  __shared__ double diag[MAXC];
  const int c = k + 1;
  const int i = threadIdx.x >> 5, l = threadIdx.x & 31;
  pdl_begin();
  if (pd.peers) {
    // the mailbox all-reduce of [g, sum rho^2 | G2] comes first and unconditionally: every collective of the channel
    // must be executed by every rank (the double-buffered slots rely on it), whatever the status word says
    double* gsh = R2s;  // NE2_MAX <= MAXC * GLD; R2s is not written before the Cholesky below
    const int NE2 = GPAD + nblocks(NB) * 64;
    if (threadIdx.x < NE2) gsh[threadIdx.x] = parts[threadIdx.x];
    __syncthreads();
    p2p_tail_allreduce(pd, gsh, NE2, 0);
    __syncthreads();
    // keep the sums where the two forms expect them: a private copy, R2s is reused below
    double* keep = Rs;  // Rs is written only after the last read of `parts`
    if (threadIdx.x < NE2) keep[threadIdx.x] = gsh[threadIdx.x];
    __syncthreads();
    parts = keep;
    nparts = 1;
  }
  const int mode = *status;
  if (mode == 1 || (mode == 2 && !have_g2)) {
    // refused by the pivot floor -- or too ill-conditioned for the refinement form while the second CholeskyQR2 pass
    // was not run (it is no longer part of the default chain: no Bratu run needs it, and its no-op launch cost 2.5 us
    // per outer iteration); the host re-issues the solve with the Householder path either way
    write_refusal(k, out);
    return;
  }
  if (mode == 0) {
    // refinement form: delta = (R1^T R1)^{-1} g, d = d0 + delta
    double* gs = rowbuf;   // k + 1 values (2 * RB >= MAXC + 1)
    double* us = diag;
    __shared__ double dsum[2];
    const int pstride = GPAD + nblocks(NB) * 64;
    if (threadIdx.x <= k) {
      double g = parts[threadIdx.x];
      for (int r = 1; r < nparts; ++r) g += parts[(int64_t)r * pstride + threadIdx.x];
      gs[threadIdx.x] = g;
    }
    R1s[i * GLD + l] = R1g[i * MAXC + l];  // R1 (upper triangular)
    __syncthreads();
    if (threadIdx.x < 32) {
      // delta = (R1^T R1)^{-1} g by two triangular solves (lane = row): forward R1^T u = g, backward R1 delta = u.
      // (sign^2 = 1: g = (sign A)^T rho already carries the sign, the Gram block of the A columns does not.)
      const bool row = l < k;
      const double rinv = row ? 1.0 / R1s[l * GLD + l] : 1.0;
      double z = row ? gs[l] : 0.0, u = 0.0;
      for (int j = 0; j < k; ++j) {
        const double uj = __shfl_sync(0xffffffffu, z, j) * __shfl_sync(0xffffffffu, rinv, j);
        if (l == j) u = uj;
        if (l > j && row) z = fma(-R1s[j * GLD + l], uj, z);
      }
      z = u;
      double dl_ = 0.0;
      for (int j = k - 1; j >= 0; --j) {
        const double dj = __shfl_sync(0xffffffffu, z, j) * __shfl_sync(0xffffffffu, rinv, j);
        if (l == j) dl_ = dj;
        if (l < j) z = fma(-R1s[l * GLD + j], dj, z);
      }
      if (row) us[l] = dl_;
    }
    __syncthreads();
    if (threadIdx.x < 32) {
      const bool row = l < k;
      const double dl = row ? us[l] : 0.0;
      const double d = row ? d0g[l] + dl : 0.0;
      const double rii = row ? R1g[l * MAXC + l] : 1.0;
      const double d2 = warp_sum(d * d), dl2 = warp_sum(dl * dl);
      const double ndef = warp_sum((row && fabs(rii) <= 1e-8) ? 1.0 : 0.0);
      // ||A d||^2 for the Armijo rule (armijo_goldstein.py:50).  At the least-squares solution A^T A d = A^T y, so
      // ||A d||^2 = b^T d with b = (sign A)^T y straight from the Gram pass: no conditioning enters (the error is
      // second order in the remaining gradient), unlike ||A d0||^2 = |R1^{-T} b|^2 of the unrefined solution, which is
      // only good to cond^2 eps ~ 1e-7.
      const double bd = warp_sum(row ? aux[1 + l] * d : 0.0);
      if (l == 0) {
        dsum[0] = d2;
        dsum[1] = dl2;
      }
      __syncwarp();
      if (dl2 <= REFINE_ACCEPT * REFINE_ACCEPT * d2) {  // uniform
        if (row) {
          out[l] = d;
          out[k + 4 + l] = rii;
        }
        if (l == 0) {
          out[k] = bd;
          out[k + 1] = gs[k];
          out[k + 2] = ndef;
          out[k + 3] = d2;
        }
      }
    }
    __syncthreads();
    if (!(dsum[1] <= REFINE_ACCEPT * REFINE_ACCEPT * dsum[0])) write_refusal(k, out);
    return;
  }
  parts += GPAD;  // the Gram matrix of pass 2 follows g in every rank's slot
  R1s[i * GLD + l] = R1g[i * MAXC + l];
  const double a = gather_gram(parts, nparts, NB, c, GPAD + nblocks(NB) * 64);
  double r2, min_ratio;
  if (!block_cholesky(a, c, PIVOT_FLOOR_2, rowbuf, diag, r2, min_ratio)) {
    write_refusal(k, out);
    return;
  }
  R2s[i * GLD + l] = r2;
  __syncthreads();
  {  // R = R2 R1 (upper x upper), ascending inner index
    double s = 0.0;
    if (i <= l && l < c)
      for (int m = i; m <= l; ++m) s = fma(R2s[i * GLD + m], R1s[m * GLD + l], s);
    Rs[i * GLD + l] = s;
  }
  __syncthreads();
  if (threadIdx.x < 32) {
    // back substitution R[:k,:k] d = R[:k,k], lane = row: once d_j is known every row above subtracts R_ij d_j.  The
    // reciprocals of the diagonal are formed up front, so a step costs two shuffles and two FMAs, no division.
    const int lane = threadIdx.x;
    const bool row = lane < k;
    double z = row ? Rs[lane * GLD + k] : 0.0;
    const double rii = row ? Rs[lane * GLD + lane] : 1.0;
    const double rinv = 1.0 / rii;
    const double zk = z;
    double d = 0.0;
    for (int j = k - 1; j >= 0; --j) {
      const double dj = __shfl_sync(0xffffffffu, z, j) * __shfl_sync(0xffffffffu, rinv, j);
      if (lane == j) d = dj;
      if (lane < j) z = fma(-Rs[lane * GLD + j], dj, z);
    }
    double z2 = row ? zk * zk : 0.0, d2 = row ? d * d : 0.0, ndef = (row && fabs(rii) <= 1e-8) ? 1.0 : 0.0;
    if (row) {
      out[lane] = d;
      out[k + 4 + lane] = rii;
    }
    z2 = warp_sum(z2);
    d2 = warp_sum(d2);
    ndef = warp_sum(ndef);
    if (lane == 0) {
      out[k] = z2;
      out[k + 1] = Rs[k * GLD + k] * Rs[k * GLD + k];
      out[k + 2] = ndef;
      out[k + 3] = d2;
    }
  }
}

// scratch layout inside gnk_ctx::d_cholqr (doubles)
constexpr int64_t CQ_PART = 0;                                     // per-CTA partials: MAX_CTAS * NE_MAX
constexpr int64_t CQ_MAX_CTAS = 512;
constexpr int64_t CQ_LOCAL = CQ_PART + CQ_MAX_CTAS * NE_MAX;       // this rank's Gram matrix (pass 1)
constexpr int64_t CQ_ALL = CQ_LOCAL + NE_MAX;                      // all ranks' Gram matrices (pass 1)
constexpr int64_t NE2_MAX = GPAD + NE_MAX;                         // pass 2: [g, sum rho^2 | Gram matrix]
constexpr int64_t CQ_LOCAL2 = CQ_ALL + P2P_MAXR * NE_MAX;
constexpr int64_t CQ_ALL2 = CQ_LOCAL2 + NE2_MAX;
constexpr int64_t CQ_T = CQ_ALL2 + P2P_MAXR * NE2_MAX;             // T (MAXC x TLD)
constexpr int64_t CQ_R1 = CQ_T + MAXC * TLD;                       // R1 (MAXC x MAXC)
constexpr int64_t CQ_D0 = CQ_R1 + MAXC * MAXC;                     // normal-equation solution d0
constexpr int64_t CQ_AUX = CQ_D0 + MAXC;                           // ||A d0||^2, then b = (sign A)^T y (k doubles)
constexpr int64_t CQ_STATUS = CQ_AUX + 8 + MAXC;                   // int status word
constexpr int64_t CQ_TOTAL = CQ_STATUS + 8;

template <int KC>
int launch_refine(gnk_ctx* ctx, const PanelSource& src, double sign, double* base, int* status, cudaStream_t st) {
  auto kern = cholqr_refine_kernel<KC>;
  static int occ_dev[64] = {0};
  int& occ = occ_dev[ctx->device & 63];
  if (occ == 0) {
    int o = 1;
    GNK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, kern, RT, 0));
    occ = o < 1 ? 1 : o;
  }
  constexpr int64_t GRAN = 2 * RT;
  int64_t ctas = (int64_t)ctx->sm_count * occ;
  if (ctas > CQ_MAX_CTAS) ctas = CQ_MAX_CTAS;
  if (ctas * GRAN > src.n_rows) ctas = ceil_div(src.n_rows, GRAN);
  const int64_t rows_per_cta = ceil_div(ceil_div(src.n_rows, ctas), GRAN) * GRAN;
  ctas = ceil_div(src.n_rows, rows_per_cta);
  GNK_CUDA(gnk_launch(gnk_pdl_for(src.n_rows), kern, dim3((unsigned)ctas), dim3(RT), 0, st, src, sign, base + CQ_D0, status, rows_per_cta,
                      base + CQ_PART, ctx->d_tickets + TK_CHOLQR, base + CQ_LOCAL2));
  GNK_LAUNCH_CHECK(ctx);
  return 0;
}

int launch_refine_any(gnk_ctx* ctx, const PanelSource& src, double sign, double* base, int* status, cudaStream_t st) {
  if (src.k <= 8) return launch_refine<8>(ctx, src, sign, base, status, st);
  if (src.k <= 16) return launch_refine<16>(ctx, src, sign, base, status, st);
  if (src.k <= 24) return launch_refine<24>(ctx, src, sign, base, status, st);
  return launch_refine<32>(ctx, src, sign, base, status, st);
}

// second pass: 0 the refinement form (chosen on the device, see cholqr_factor1_kernel), 2 always CholeskyQR2
int second_pass_method(const gnk_ctx* ctx) {
  static const int refine_on = getenv("GNK_LS_REFINE") ? atoi(getenv("GNK_LS_REFINE")) : 1;
  return (ctx->ls_method == 2 || !refine_on) ? 2 : 0;
}

int ensure_scratch(gnk_ctx* ctx, cudaStream_t st) {
  if (!ctx->d_cholqr) {
    GNK_CUDA(cudaMalloc(&ctx->d_cholqr, sizeof(double) * CQ_TOTAL));
    GNK_CUDA(cudaMemsetAsync(ctx->d_cholqr, 0, sizeof(double) * CQ_TOTAL, st));
  }
  return 0;
}

// Everything after pass 1: this rank's Gram matrix of [A | y] (fragment order) is at base + CQ_LOCAL.  refine(status)
// launches the refinement form of pass 2 (d_A may be null if it does not read A; the CholeskyQR2 pass does).
template <int NB, int RU, class Refine>
int cholqr_tail(gnk_ctx* ctx, const double* d_A, int64_t lda, int64_t n_rows, int k, const double* d_y, double sign,
                double* d_out, cudaStream_t st, Refine&& refine) {
  double* base = ctx->d_cholqr;
  int* status = reinterpret_cast<int*>(base + CQ_STATUS);
  PanelSource src{d_A, lda, d_y, k, n_rows};
  constexpr int64_t GRAN = (int64_t)CH * RU * GW;
  int64_t ctas = ctx->sm_count < CQ_MAX_CTAS ? ctx->sm_count : CQ_MAX_CTAS;
  if (ctas * GRAN > n_rows) ctas = ceil_div(n_rows, GRAN);
  const int64_t rows_per_cta = ceil_div(ceil_div(n_rows, ctas), GRAN) * GRAN;
  ctas = ceil_div(n_rows, rows_per_cta);
  const int NE = nblocks(NB) * 64;
  const bool multi = ctx->nranks > 1;
  GNK_REQUIRE(ctx->nranks <= P2P_MAXR, "cholqr: more ranks than the Gram gather buffer holds");
  const int method = second_pass_method(ctx);
  // with the peer mailboxes attached the factor kernels (single CTAs) run the cross-rank sum themselves
  const gnk_p2p_dev none{nullptr, 0, 1, 0ull};
  const gnk_p2p_dev pd1 = multi ? p2p_next(ctx) : none;
  const bool gather1 = multi && !pd1.peers;
  if (gather1)
    if (int rc = gnk_comm_allgather_doubles(ctx, base + CQ_LOCAL, base + CQ_ALL, NE, st)) return rc;
  GNK_CUDA(gnk_launch(gnk_pdl_for(n_rows), cholqr_factor1_kernel, dim3(1), dim3(FT), 0, st, gather1 ? base + CQ_ALL : base + CQ_LOCAL,
                      gather1 ? ctx->nranks : 1, NB, k, sign, method, base + CQ_T, base + CQ_R1, base + CQ_D0,
                      base + CQ_AUX, status, pd1));
  GNK_LAUNCH_CHECK(ctx);
  // pass 2: the refinement form by default (it returns at once unless the status word says 0); the second CholeskyQR2
  // pass only when the caller asked for it (gnk_tsqr_ls_method 2)
  if (method == 0)
    if (int rc = refine(status)) return rc;
  if (method == 2) {
    cholqr_gram2_kernel<NB, RU><<<(unsigned)ctas, GT, 0, st>>>(src, rows_per_cta, base + CQ_T, status, base + CQ_PART,
                                                           ctx->d_tickets + TK_CHOLQR, base + CQ_LOCAL2 + GPAD);
    GNK_LAUNCH_CHECK(ctx);
  }
  const gnk_p2p_dev pd2 = multi ? p2p_next(ctx) : none;
  const bool gather2 = multi && !pd2.peers;
  if (gather2)
    if (int rc = gnk_comm_allgather_doubles(ctx, base + CQ_LOCAL2, base + CQ_ALL2, GPAD + NE, st)) return rc;
  GNK_CUDA(gnk_launch(gnk_pdl_for(n_rows), cholqr_factor2_kernel, dim3(1), dim3(FT), 0, st, gather2 ? base + CQ_ALL2 : base + CQ_LOCAL2,
                      gather2 ? ctx->nranks : 1, NB, k, base + CQ_R1, base + CQ_T, base + CQ_D0, base + CQ_AUX, status,
                      method == 2 ? 1 : 0, d_out, pd2));
  GNK_LAUNCH_CHECK(ctx);
  return 0;
}

template <int NB, int RU>
int run_cholqr(gnk_ctx* ctx, const double* d_A, int64_t lda, int64_t n_rows, int k, const double* d_y, double sign,
               double* d_out, cudaStream_t st) {
  if (int rc = ensure_scratch(ctx, st)) return rc;
  double* base = ctx->d_cholqr;
  PanelSource src{d_A, lda, d_y, k, n_rows};
  constexpr int64_t GRAN = (int64_t)CH * RU * GW;
  int64_t ctas = ctx->sm_count < CQ_MAX_CTAS ? ctx->sm_count : CQ_MAX_CTAS;
  if (ctas * GRAN > n_rows) ctas = ceil_div(n_rows, GRAN);
  const int64_t rows_per_cta = ceil_div(ceil_div(n_rows, ctas), GRAN) * GRAN;
  ctas = ceil_div(n_rows, rows_per_cta);
  // pass 1 and its factorisation
  GNK_CUDA(gnk_launch(gnk_pdl_for(n_rows), cholqr_gram_kernel<NB, RU>, dim3((unsigned)ctas), dim3(GT), 0, st, src, rows_per_cta,
                      base + CQ_PART, ctx->d_tickets + TK_CHOLQR, base + CQ_LOCAL));
  GNK_LAUNCH_CHECK(ctx);
  return cholqr_tail<NB, RU>(ctx, d_A, lda, n_rows, k, d_y, sign, d_out, st, [&](int* status) {
    return launch_refine_any(ctx, src, sign, base, status, st);
  });
}

// ======================================================================================================================
// Pass 1 fused with the projected operator: J V_k (gauss_newton_krylow.py:86) is formed from the basis, WRITTEN for the
// second pass, and its Gram matrix with the residual accumulated in the same sweep -- the least-squares panel is read
// once instead of being written by the SpMM, read by pass 1 and read again by pass 2 (24 n k -> 16 n k + 8 n k).
//
// Warp-specialised, TMA-staged (measured stand-alone in tools/microbench_stencil_gram.cu, version 3):
//  * a task is TI grid rows x TJ = 8 CW grid points; one producer warp (lane 0) streams its rows through a ring of
//    shared-memory slots with cp.async.bulk.tensor: a 3-D box {TJ + 8 points, 1 row, 8 NB columns} of the basis and a
//    2-D box each of the residual and of e^u, all completing on the slot's `full` mbarrier.  Out-of-range j (j0 - 4 < 0,
//    j0 + TJ + 4 > m) is zero-filled by the TMA unit, which IS the Dirichlet condition; halo rows are stored;
//  * CW consumer warps own one 8-point segment each.  Lane (g, t) holds grid points 2t, 2t+1 of basis column 8 I + g
//    -- the DMMA fragment of cholqr_gram_kernel -- keeps the (up, mid, dn) rows of that fragment in registers, reads
//    the left / right neighbours and e^u from the mid row's slot, applies the stencil with apply_refbits (scipy's
//    rounding order: J V is bit-identical to gnk_stencil_apply), stores J V and feeds the Gram DMMAs;
//  * a slot goes back to the producer (`empty`, one arrival per consumer warp) once its row has been the mid row;
//  * plane stride (TJ + 8) * 8 bytes = 64 mod 128 for CW = 8, 10, 12: the two 64-byte pieces a quarter-warp reads with
//    one LDS.128 fall into disjoint banks.
// ======================================================================================================================
struct StencilPanel {
  int m, rows, k;       // row length, owned grid rows, basis columns
  int has_e;            // 0: lam == 0, no e^u plane
  int64_t ldjv;
  double c_lap, c_adv, lam, sign;
};

template <int CW> __host__ __device__ constexpr int sg_plane_bytes() { return (8 * CW + 8) * 8; }
template <int CW> __host__ __device__ constexpr int sg_ye_bytes() { return (sg_plane_bytes<CW>() + 127) / 128 * 128; }
template <int NB, int CW> __host__ __device__ constexpr int sg_slot_bytes() {
  return 8 * NB * sg_plane_bytes<CW>() + 2 * sg_ye_bytes<CW>();
}
template <int NB, int CW> __host__ __device__ constexpr int sg_nslot() {
  return (200 * 1024 / sg_slot_bytes<NB, CW>()) < 16 ? (200 * 1024 / sg_slot_bytes<NB, CW>()) : 16;
}
template <int NB, int CW> __host__ __device__ constexpr int sg_dyn_bytes() {
  return sg_slot_bytes<NB, CW>() * sg_nslot<NB, CW>();
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}\n" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* tm, int c0, int c1, int c2, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(dst),
      "l"(tm), "r"(c0), "r"(c1), "r"(c2), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* tm, int c0, int c1, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
               "l"(tm), "r"(c0), "r"(c1), "r"(bar)
               : "memory");
}
__device__ __forceinline__ double2 lds2(uint32_t a) {
  double2 v;
  asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(a));
  return v;
}
__device__ __forceinline__ double lds1(uint32_t a) {
  double v;
  asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a));
  return v;
}

// The sweep shared by the Gram pass and the store-free refinement: ring set-up, producer warp and the 3-row register
// window.  Every consumer lane calls on_row(tile, e) once per grid row of its segment, e = flat offset of its point pair
// (grid row * m + j) among the owned unknowns, tile[I] = (sign J V)[e, e + 1] of column 8 I + g -- bit-identical to
// gnk_stencil_apply -- where the column after the basis holds the residual exactly and the columns beyond it zeros.
// Returns false at once (nothing issued) if `status` is given and is not 0 (the refinement form was not chosen);
// otherwise every consumer lane calls on_start() before its first row (after the wait on the predecessor kernel).
template <int NB, int CW, class OnStart, class OnRow>
__device__ __forceinline__ bool stencil_sweep(const CUtensorMap& tmV, const CUtensorMap& tmY, const CUtensorMap& tmE,
                                              const StencilPanel& p, int TI, const int* status, OnStart&& on_start,
                                              OnRow&& on_row) {
  constexpr int SB = sg_slot_bytes<NB, CW>();
  constexpr int NS = sg_nslot<NB, CW>();
  constexpr int TJ = 8 * CW, PB = sg_plane_bytes<CW>(), YE = sg_ye_bytes<CW>();
  extern __shared__ __align__(128) unsigned char ring[];
  __shared__ __align__(8) unsigned long long bars[2 * NS];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int m = p.m;
  const int ntj = (m + TJ - 1) / TJ;
  const int nstrip = (p.rows + TI - 1) / TI;
  const int64_t ntask = (int64_t)ntj * nstrip;
  const uint32_t ring0 = smem_u32(ring), full0 = smem_u32(bars), empty0 = full0 + 8 * NS;
  if (threadIdx.x == 0) {
    for (int s = 0; s < NS; ++s) {
      mbar_init(full0 + 8 * s, 1);
      mbar_init(empty0 + 8 * s, CW);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  pdl_begin();  // the ring is set up while the predecessor drains; nothing global has been touched yet
  if (status != nullptr && *status != 0) return false;  // uniform across the grid

  if (warp == CW) {
    if (lane == 0) {
      uint32_t s = 0, ph = 0;
      const uint32_t tx = (uint32_t)((8 * NB + 1 + (p.has_e ? 1 : 0)) * PB);
      for (int64_t task = blockIdx.x; task < ntask; task += gridDim.x) {
        const int strip = (int)(task / ntj), tj = (int)(task - (int64_t)strip * ntj);
        const int i0 = strip * TI, i1 = min(i0 + TI, p.rows), j0 = tj * TJ;
        for (int r = i0 - 1; r <= i1; ++r) {
          mbar_wait(empty0 + 8 * s, ph ^ 1u);
          const uint32_t dst = ring0 + s * SB, fb = full0 + 8 * s;
          mbar_expect_tx(fb, tx);
          tma_load_3d(dst, &tmV, j0 - 4, r + 2, 0, fb);  // stored row index = grid row + halo (2)
          tma_load_2d(dst + 8 * NB * PB, &tmY, j0 - 4, r + 2, fb);
          if (p.has_e) tma_load_2d(dst + 8 * NB * PB + YE, &tmE, j0 - 4, r + 2, fb);
          if (++s == NS) {
            s = 0;
            ph ^= 1u;
          }
        }
      }
    }
    return true;
  }
  // the sign is folded into the weights (exact: every product and every sum is negated symmetrically)
  const double sg = p.sign;
  const double d0 = __dadd_rn(4.0 * p.c_lap, -p.c_adv);
  const double cd = sg * __dadd_rn(-p.c_lap, p.c_adv), cu = sg * -p.c_lap, cl = sg * -p.c_lap;
  // per column block: byte offset of this lane's pair inside a slot, and what the column is.  Only the LAST block can
  // hold anything but basis columns (k >= 8 (NB - 1) by the choice of NB).
  uint32_t poff[NB];
#pragma unroll
  for (int I = 0; I < NB; ++I) poff[I] = (uint32_t)((8 * I + g) * PB + 8 * (4 + 8 * warp + 2 * t));
  const int lastcol = 8 * (NB - 1) + g;
  const int lastkind = lastcol < p.k ? 0 : (lastcol == p.k ? 1 : 2);  // 0 basis column, 1 the residual, 2 padding
  if (lastkind == 1) poff[NB - 1] = (uint32_t)(8 * NB * PB + 8 * (4 + 8 * warp + 2 * t));
  if (lastkind == 2) poff[NB - 1] = poff[0];                          // any valid (finite) data; multiplied by 0
  // No selects in the loop: the last block runs the same stencil code with per-lane weights -- a basis column keeps
  // (cu, cl, dg, cd); the residual column uses (0, 0, 1, 0), which returns `mid` exactly (0 * finite = 0, 0 + x = x);
  // a padding column uses all zeros.  dg = wsel * (d0 + lam e) + wone is exact for wsel, wone in {0, 1}.
  const double wsel = lastkind == 0 ? 1.0 : 0.0, wone = lastkind == 1 ? 1.0 : 0.0;
  const double cuL = wsel * cu, clL = wsel * cl, cdL = wsel * cd;
  const uint32_t eoff = (uint32_t)(8 * NB * PB + YE + 8 * (4 + 8 * warp + 2 * t));
  on_start();
  // ring position: slot index and phase advance together (no modulo in the loop)
  uint32_t slot = 0, phase = 0;
  auto advance = [&]() {
    if (++slot == NS) {
      slot = 0;
      phase ^= 1u;
    }
  };
  // One grid row: `dn` receives row i + 1 from the ring, then row i (held in `mid`, its slot still resident at
  // mid_base) is processed with `up` = row i - 1.  Called with the three register rows in rotating roles, so the
  // window never has to be copied.
  // a warp whose segment lies beyond the row end (last tile of a row, m not a multiple of TJ) only keeps the ring moving
  auto row_skip = [&](uint32_t& mid_slot) {
    mbar_wait(full0 + 8 * slot, phase);
    __syncwarp();
    if (lane == 0) mbar_arrive(empty0 + 8 * mid_slot);
    mid_slot = slot;
    advance();
  };
  auto row_step = [&](double2 (&up)[NB], double2 (&mid)[NB], double2 (&dn)[NB], uint32_t& mid_base,
                      uint32_t& mid_slot, int64_t e_off) {
    mbar_wait(full0 + 8 * slot, phase);
    const uint32_t base = ring0 + slot * SB;
#pragma unroll
    for (int I = 0; I < NB; ++I) dn[I] = lds2(base + poff[I]);
    double lf[NB], rt[NB];
#pragma unroll
    for (int I = 0; I < NB; ++I) {
      lf[I] = lds1(mid_base + poff[I] - 8);
      rt[I] = lds1(mid_base + poff[I] + 16);
    }
    double2 e = make_double2(0.0, 0.0);
    if (p.has_e) e = lds2(mid_base + eoff);
    __syncwarp();
    if (lane == 0) mbar_arrive(empty0 + 8 * mid_slot);  // the mid row's slot goes back to the producer
    mid_base = base;
    mid_slot = slot;
    advance();
    const double dga = sg * __dadd_rn(d0, __dmul_rn(p.lam, e.x)), dgb = sg * __dadd_rn(d0, __dmul_rn(p.lam, e.y));
    const double dgaL = fma(wsel, dga, wone), dgbL = fma(wsel, dgb, wone);
    double2 tile[NB];
#pragma unroll
    for (int I = 0; I < NB; ++I) {
      const bool last = I == NB - 1;
      const double oa = apply_refbits(last ? cuL : cu, last ? clL : cl, last ? dgaL : dga, last ? cdL : cd, up[I].x,
                                      lf[I], mid[I].x, mid[I].y, dn[I].x);
      const double ob = apply_refbits(last ? cuL : cu, last ? clL : cl, last ? dgbL : dgb, last ? cdL : cd, up[I].y,
                                      mid[I].x, mid[I].y, rt[I], dn[I].y);
      tile[I] = make_double2(oa, ob);
    }
    on_row(tile, e_off);
  };
  for (int64_t task = blockIdx.x; task < ntask; task += gridDim.x) {
    const int strip = (int)(task / ntj), tj = (int)(task - (int64_t)strip * ntj);
    const int i0 = strip * TI, i1 = min(i0 + TI, p.rows);
    const bool active = tj * TJ + 8 * warp < m;  // the last tile of a row may be narrower than TJ (whole segments)
    double2 ra[NB], rb[NB], rc[NB];
    {  // row i0 - 1
      mbar_wait(full0 + 8 * slot, phase);
      const uint32_t base = ring0 + slot * SB;
#pragma unroll
      for (int I = 0; I < NB; ++I) ra[I] = lds2(base + poff[I]);
      __syncwarp();
      if (lane == 0) mbar_arrive(empty0 + 8 * slot);
      advance();
    }
    uint32_t mid_base, mid_slot;
    {  // row i0
      mbar_wait(full0 + 8 * slot, phase);
      mid_base = ring0 + slot * SB;
      mid_slot = slot;
#pragma unroll
      for (int I = 0; I < NB; ++I) rb[I] = lds2(mid_base + poff[I]);
      advance();
    }
    int64_t e_off = (int64_t)i0 * m + tj * TJ + 8 * warp + 2 * t;
    int i = i0;
    if (active) {
      while (true) {  // three rows per trip, the window rotating through (ra, rb, rc)
        row_step(ra, rb, rc, mid_base, mid_slot, e_off);
        e_off += m;
        if (++i == i1) break;
        row_step(rb, rc, ra, mid_base, mid_slot, e_off);
        e_off += m;
        if (++i == i1) break;
        row_step(rc, ra, rb, mid_base, mid_slot, e_off);
        e_off += m;
        if (++i == i1) break;
      }
    } else {
      for (; i < i1; ++i) row_skip(mid_slot);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(empty0 + 8 * mid_slot);  // row i1 was only ever a dn row
  }
  return true;
}

// Pass 1: the Gram matrix of the panel [sign J V | r], and J V itself when STORE (the CholeskyQR2 pass and the
// Householder fallback read it back; the refinement form recomputes it in stencil_refine_kernel).
template <int NB, int CW, bool STORE>
__global__ void __launch_bounds__(32 * (CW + 1), 1)
    stencil_gram_kernel(const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmY,
                        const __grid_constant__ CUtensorMap tmE, StencilPanel p, int TI, double* __restrict__ JV,
                        double* __restrict__ partials, unsigned int* ticket, double* __restrict__ Gout) {
  constexpr int NBLK = nblocks(NB);
  __shared__ __align__(16) double red[NBLK * 64];
  const int g = (threadIdx.x & 31) >> 2;
  double acc[NBLK][2];
#pragma unroll
  for (int b = 0; b < NBLK; ++b) acc[b][0] = acc[b][1] = 0.0;
  double* jp[NB];  // this lane's J V columns
#pragma unroll
  for (int I = 0; I < NB; ++I) jp[I] = JV + (int64_t)(8 * I + g) * p.ldjv;
  const bool last_is_basis = 8 * (NB - 1) + g < p.k;
  stencil_sweep<NB, CW>(tmV, tmY, tmE, p, TI, nullptr, [] {}, [&](const double2 (&tile)[NB], int64_t e) {
    if constexpr (STORE) {
      // J V goes out with plain 128-bit streaming stores (a quad writes 64 contiguous bytes of a column); staging it in
      // shared memory for cp.async.bulk.tensor stores was built and measured SLOWER in situ (46.2 vs 41.0 ms per solve)
#pragma unroll
      for (int I = 0; I < NB; ++I)
        if (I < NB - 1 || last_is_basis) __stcs(reinterpret_cast<double2*>(jp[I] + e), tile[I]);
    }
#pragma unroll
    for (int I = 0; I < NB; ++I)
#pragma unroll
      for (int J = I; J < NB; ++J) {
        const int b = blk_index(NB, I, J);
        dmma(acc[b][0], acc[b][1], tile[I].x, tile[J].x);
        dmma(acc[b][0], acc[b][1], tile[I].y, tile[J].y);
      }
  });
  reduce_gram<NBLK, CW, 32 * (CW + 1)>(acc, red, partials, ticket, Gout);
}

// Pass 2, refinement form, with J V recomputed instead of read back: rho = y - (sign A) d0, g = (sign A)^T rho and
// sum rho^2 for A = J V_k, the same quantities as cholqr_refine_kernel, without the 8 n k bytes of the J V store in
// pass 1.  The sweep's lanes hold 8 columns of a point pair each: rho is their weighted sum, completed over the 8 g-lanes
// by a butterfly (all eight end with the same bits), then every lane accumulates g for its own columns.
// Output as cholqr_refine_kernel: the last CTA writes (sign A)^T rho, then sum rho^2, to gout.
template <int NB, int CW>
__global__ void __launch_bounds__(32 * (CW + 1), 1)
    stencil_refine_kernel(const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmY,
                          const __grid_constant__ CUtensorMap tmE, StencilPanel p, int TI, double sign,
                          const double* __restrict__ d0g, const int* __restrict__ status,
                          double* __restrict__ partials, unsigned int* ticket, double* __restrict__ gout) {
  constexpr int NC = 8 * NB;  // panel columns held by a warp (basis, residual, padding)
  __shared__ double wsum[CW][NC + 1];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2;
  double gacc[NB], rr = 0.0;
#pragma unroll
  for (int I = 0; I < NB; ++I) gacc[I] = 0.0;
  double w[NB];  // rho = sum over the panel columns of w * column: -sign d0 on the basis, 1 on the residual, 0 beyond
  auto weights = [&] {
#pragma unroll
    for (int I = 0; I < NB; ++I) {
      const int col = 8 * I + g;
      w[I] = col < p.k ? -sign * d0g[col] : (col == p.k ? 1.0 : 0.0);
    }
  };
  const bool run = stencil_sweep<NB, CW>(tmV, tmY, tmE, p, TI, status, weights, [&](const double2 (&tile)[NB], int64_t) {
    double2 q = make_double2(0.0, 0.0);
#pragma unroll
    for (int I = 0; I < NB; ++I) {
      q.x = fma(w[I], tile[I].x, q.x);
      q.y = fma(w[I], tile[I].y, q.y);
    }
#pragma unroll
    for (int o = 4; o < 32; o <<= 1) {
      q.x += __shfl_xor_sync(0xffffffffu, q.x, o);
      q.y += __shfl_xor_sync(0xffffffffu, q.y, o);
    }
#pragma unroll
    for (int I = 0; I < NB; ++I) gacc[I] = fma(tile[I].x, q.x, fma(tile[I].y, q.y, gacc[I]));
    rr = fma(q.x, q.x, fma(q.y, q.y, rr));
  });
  if (!run) return;
  // CTA partial: over the 4 t-lanes of a column, then over the consumer warps in warp order
#pragma unroll
  for (int I = 0; I < NB; ++I) {
    gacc[I] += __shfl_xor_sync(0xffffffffu, gacc[I], 1);
    gacc[I] += __shfl_xor_sync(0xffffffffu, gacc[I], 2);
  }
  rr += __shfl_xor_sync(0xffffffffu, rr, 1);
  rr += __shfl_xor_sync(0xffffffffu, rr, 2);
  if (warp < CW && (lane & 3) == 0) {
#pragma unroll
    for (int I = 0; I < NB; ++I) wsum[warp][8 * I + g] = gacc[I];
    if (lane == 0) wsum[warp][NC] = rr;  // rho is the same on every g-lane: one lane counts each point
  }
  __syncthreads();
  constexpr int PS = MAXC + 1;  // partial stride: 32 columns, then sum rho^2
  double* mine = partials + (int64_t)blockIdx.x * PS;
  if (threadIdx.x <= NC) {
    double v = wsum[0][threadIdx.x];
    for (int q = 1; q < CW; ++q) v += wsum[q][threadIdx.x];
    mine[threadIdx.x == NC ? MAXC : threadIdx.x] = v;
    __threadfence();
  }
  if (!grid_arrive_last(ticket)) return;
  if (threadIdx.x < PS) {
    double v = 0.0;
    const int nb = gridDim.x;
    const int e = threadIdx.x;
    if (e < p.k || e == MAXC) {
      for (int b = 0; b < nb; ++b) v += __ldcg(partials + (int64_t)b * PS + e);
      if (e < p.k) gout[e] = sign * v;  // (sign A)^T rho
      else gout[p.k] = v;               // sum rho^2
    }
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)f;
    else
      (void)cudaGetLastError();
  }
  return fn;
}
// tensor map over stored columns: [ncols][rows + 2 halo][m] doubles, column stride ld; box {pw, 1, ncol_box}
int make_column_map(CUtensorMap* tm, const double* base, int m, int stored_rows, int64_t ld, int ncols, int ncol_box,
                    int pw, bool force_3d = false) {
  EncodeTiledFn enc = encode_tiled_fn();
  GNK_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled is not available from this driver");
  CUresult r;
  if (ncol_box > 1 || ncols > 1 || force_3d) {
    cuuint64_t dims[3] = {(cuuint64_t)m, (cuuint64_t)stored_rows, (cuuint64_t)ncols};
    cuuint64_t strides[2] = {(cuuint64_t)m * 8, (cuuint64_t)ld * 8};
    cuuint32_t box[3] = {(cuuint32_t)pw, 1, (cuuint32_t)ncol_box};
    cuuint32_t es[3] = {1, 1, 1};
    r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, (void*)base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  } else {
    cuuint64_t dims[2] = {(cuuint64_t)m, (cuuint64_t)stored_rows};
    cuuint64_t strides[1] = {(cuuint64_t)m * 8};
    cuuint32_t box[2] = {(cuuint32_t)pw, 1};
    cuuint32_t es[2] = {1, 1};
    r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, (void*)base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  }
  if (r != CUDA_SUCCESS) {
    gnk_set_error("cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)r));
    return -3;
  }
  return 0;
}

// dynamic shared memory of a ring kernel, set once per device (done: one flag per device of that kernel)
template <class Kern>
int ring_smem_attr(gnk_ctx* ctx, Kern kern, int dyn, bool (&done)[64]) {
  if (!done[ctx->device & 63]) {
    GNK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn));
    done[ctx->device & 63] = true;
  }
  return 0;
}

template <int NB, int RU, int CW>
int run_stencil_gram_cw(gnk_ctx* ctx, const gnk_layout* lay, const gnk_bratu* prm, const double* d_expu, const double* d_V,
                     int64_t ldv, int k, const double* d_r, double sign, double* d_JV, int64_t ldjv,
                     double sign_a, double* d_out, cudaStream_t st) {
  if (int rc = ensure_scratch(ctx, st)) return rc;
  double* base = ctx->d_cholqr;
  constexpr int PW = 8 * CW + 8, TJ = 8 * CW;
  const int stored_rows = lay->rows + 2 * lay->halo;
  CUtensorMap tmV, tmY, tmE;
  // the map ends at column k although a box spans 8 NB columns: no lane consumes a basis column >= k (column k's lanes
  // read the residual plane, padding lanes column g), so the TMA unit zero-fills them instead of reading them from HBM
  if (int rc = make_column_map(&tmV, d_V, lay->m, stored_rows, ldv, k, 8 * NB, PW)) return rc;
  if (int rc = make_column_map(&tmY, d_r, lay->m, stored_rows, lay->ld, 1, 1, PW)) return rc;
  const bool has_e = prm->lam != 0.0;
  if (int rc = make_column_map(&tmE, has_e ? d_expu : d_r, lay->m, stored_rows, lay->ld, 1, 1, PW)) return rc;
  const int ntj = (lay->m + TJ - 1) / TJ;
  int TI = 64;
  while (TI > 8 && (int64_t)ntj * ceil_div(lay->rows, TI) < 6LL * ctx->sm_count) TI >>= 1;
  const int64_t ntask = (int64_t)ntj * ceil_div(lay->rows, TI);
  const int ctas = (int)(ntask < ctx->sm_count ? ntask : ctx->sm_count);
  StencilPanel p{lay->m, lay->rows, k, has_e ? 1 : 0, ldjv, prm->c_lap, prm->c_adv, prm->lam, sign};
  constexpr int dyn = sg_dyn_bytes<NB, CW>();
  static bool attr_store[64] = {false}, attr_free[64] = {false}, attr_refine[64] = {false};  // per template instance
  const bool store = d_JV != nullptr;
  auto gram = store ? stencil_gram_kernel<NB, CW, true> : stencil_gram_kernel<NB, CW, false>;
  if (int rc = ring_smem_attr(ctx, gram, dyn, store ? attr_store : attr_free)) return rc;
  GNK_CUDA(gnk_launch(gnk_pdl_for(lay->n_own), gram, dim3(ctas), dim3(32 * (CW + 1)), (size_t)dyn, st, tmV, tmY, tmE, p, TI, d_JV, base + CQ_PART,
                      ctx->d_tickets + TK_CHOLQR, base + CQ_LOCAL));
  GNK_LAUNCH_CHECK(ctx);
  const double* d_y = d_r + lay->off;
  if (store)
    return cholqr_tail<NB, RU>(ctx, d_JV, ldjv, lay->n_own, k, d_y, sign_a, d_out, st, [&](int* status) {
      return launch_refine_any(ctx, PanelSource{d_JV, ldjv, d_y, k, lay->n_own}, sign_a, base, status, st);
    });
  // J V was not stored: the refinement pass streams V_k through the same ring and applies the stencil again
  return cholqr_tail<NB, RU>(ctx, nullptr, ldjv, lay->n_own, k, d_y, sign_a, d_out, st, [&](int* status) {
    auto refine = stencil_refine_kernel<NB, CW>;
    if (int rc = ring_smem_attr(ctx, refine, dyn, attr_refine)) return rc;
    GNK_CUDA(gnk_launch(gnk_pdl_for(lay->n_own), refine, dim3(ctas), dim3(32 * (CW + 1)), (size_t)dyn, st, tmV, tmY, tmE, p, TI,
                        sign_a, (const double*)(base + CQ_D0), (const int*)status, base + CQ_PART,
                        ctx->d_tickets + TK_CHOLQR, base + CQ_LOCAL2));
    GNK_LAUNCH_CHECK(ctx);
    return 0;
  });
}

}  // namespace

// Called by gnk_tsqr_ls (tsqr.cu) for the panels it found eligible (3 <= k+1 <= 32 columns, >= 16384 rows, even row
// count, 16-byte aligned, sign = +-1); returns 1 for a panel wider than 32 columns.
int gnk_cholqr_try(gnk_ctx* ctx, const double* d_A, int64_t lda, int64_t n_rows, int k, const double* d_y,
                   double sign_a, double* d_out, void* stream) {
  const int c = k + 1;
  cudaStream_t st = (cudaStream_t)stream;
  if (c <= 8) return run_cholqr<1, 4>(ctx, d_A, lda, n_rows, k, d_y, sign_a, d_out, st);
  if (c <= 16) return run_cholqr<2, 2>(ctx, d_A, lda, n_rows, k, d_y, sign_a, d_out, st);
  if (c <= 24) return run_cholqr<3, 1>(ctx, d_A, lda, n_rows, k, d_y, sign_a, d_out, st);
  if (c <= 32) return run_cholqr<4, 1>(ctx, d_A, lda, n_rows, k, d_y, sign_a, d_out, st);
  return 1;
}

// 8 consumer warps (64-point tiles).  Measured and not kept (profiles/r02_pair_kernel_experiment.txt, DESIGN.md 3.1):
// 10 consumer warps with 80-point tiles (no gain), two warps per segment that split the column blocks (slower: the
// kernel is power-/FP64-bound, more FP64 work in flight lowers the SM clock under the power cap).
template <int NB, int RU>
int run_stencil_gram(gnk_ctx* ctx, const gnk_layout* lay, const gnk_bratu* prm, const double* d_expu, const double* d_V,
                     int64_t ldv, int k, const double* d_r, double sign, double* d_JV, int64_t ldjv,
                     double sign_a, double* d_out, cudaStream_t st) {
  return run_stencil_gram_cw<NB, RU, 8>(ctx, lay, prm, d_expu, d_V, ldv, k, d_r, sign, d_JV, ldjv, sign_a, d_out,
                                        st);
}

// gnk_stencil_gram_ls (gnk_b200.h): J V_k written (unless d_JV is null) AND the projected least squares solved with the
// panel read once.  Returns 1 when the panel is not eligible for the fused tensor-pipe path (the caller then runs
// gnk_stencil_apply + gnk_tsqr_ls): the same conditions as gnk_tsqr_ls's tensor-pipe path, plus whole 8-point segments
// per grid row, plus -- without J V -- the refinement form of the second pass (CholeskyQR2 reads J V back).
extern "C" int gnk_stencil_gram_ls(gnk_ctx* ctx, const gnk_layout* lay, const gnk_bratu* prm, const double* d_expu,
                                   const double* d_V, int64_t ldv, int v_cols, int k, const double* d_r, double sign,
                                   double* d_JV, int64_t ldjv, double sign_a, double* d_out, void* stream) {
  GNK_REQUIRE(ctx && lay && prm && d_V && d_r && d_out, "gnk_stencil_gram_ls: null argument");
  GNK_REQUIRE(lay->m > 0 && lay->rows > 0 && lay->halo == 2 && lay->off == 2LL * lay->m &&
                  lay->n_own == (int64_t)lay->rows * lay->m && lay->ld >= (int64_t)(lay->rows + 4) * lay->m,
              "gnk_stencil_gram_ls: inconsistent stencil layout");
  GNK_REQUIRE(k >= 1 && k + 1 <= GNK_MAX_BASIS && v_cols >= k, "gnk_stencil_gram_ls: k out of range");
  GNK_REQUIRE(prm->lam == 0.0 || d_expu, "gnk_stencil_gram_ls: e^u diagonal required when lam != 0");
  cudaStream_t st = (cudaStream_t)stream;
  static const int cholqr_on = getenv("GNK_LS_CHOLQR") ? atoi(getenv("GNK_LS_CHOLQR")) : 1;
  static const int cholqr_min = getenv("GNK_LS_CHOLQR_MIN") ? atoi(getenv("GNK_LS_CHOLQR_MIN")) : 3;
  static const int fused_on = getenv("GNK_LS_FUSED") ? atoi(getenv("GNK_LS_FUSED")) : 1;
  // narrowest panel that takes the fused kernel: with one column block the per-row ring hand-over outweighs the saved
  // pass (k = 2: 0.54 ms fused against 0.33 ms for the two kernels; break-even at k = 6..7, measured at 4096^2)
  static const int fused_min = getenv("GNK_LS_FUSED_MIN") ? atoi(getenv("GNK_LS_FUSED_MIN")) : 8;
  const int c = k + 1;
  const bool aligned = (lay->m % 8 == 0) && (ldv % 2 == 0) && (ldjv % 2 == 0) && (lay->ld % 2 == 0) &&
                       ((uintptr_t)d_V % 16 == 0) && ((uintptr_t)d_r % 16 == 0) && ((uintptr_t)d_JV % 16 == 0) &&
                       (d_expu == nullptr || (uintptr_t)d_expu % 16 == 0);
  if (!(fused_on && cholqr_on && ctx->ls_method != 1 && (sign == 1.0 || sign == -1.0) &&
        (sign_a == 1.0 || sign_a == -1.0) && aligned && lay->n_own >= 16384 && c <= 32 && c >= cholqr_min &&
        c >= fused_min && (d_JV != nullptr || second_pass_method(ctx) == 0) && encode_tiled_fn() != nullptr))
    return 1;
  if (c <= 8) return run_stencil_gram<1, 4>(ctx, lay, prm, d_expu, d_V, ldv, k, d_r, sign, d_JV, ldjv, sign_a, d_out, st);
  if (c <= 16) return run_stencil_gram<2, 2>(ctx, lay, prm, d_expu, d_V, ldv, k, d_r, sign, d_JV, ldjv, sign_a, d_out, st);
  if (c <= 24) return run_stencil_gram<3, 1>(ctx, lay, prm, d_expu, d_V, ldv, k, d_r, sign, d_JV, ldjv, sign_a, d_out, st);
  return run_stencil_gram<4, 1>(ctx, lay, prm, d_expu, d_V, ldv, k, d_r, sign, d_JV, ldjv, sign_a, d_out, st);
}
