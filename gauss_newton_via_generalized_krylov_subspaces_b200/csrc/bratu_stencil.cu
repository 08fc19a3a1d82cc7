// bratu_stencil.cu -- matrix-free 5-point-stencil kernels for the Bratu problem
// (bratu_pde_problem.py:43-96).  Index (i, j) -> i*m + j, i = x1 (slow), j = x2 (fast).
//   P(u)_ij = c_lap (4 u_ij - u_i-1j - u_i+1j - u_ij-1 - u_ij+1) + c_adv (u_i+1j - u_ij) + lam e^{u_ij}
//   J(u)    = -(L + alpha D + lam diag(e^u)): only the diagonal depends on u, so the Jacobian is
//             represented by the n-vector e^u plus three constants -- nothing is assembled.
// Each thread owns two adjacent j (one 128-bit word) and marches down a strip of grid rows keeping
// the three-row window in registers, so every input word is fetched once per CTA; the j-1 / j+2
// neighbours are 64-bit loads that hit L1.  HBM traffic is the algorithmic minimum plus one halo
// row per row tile.  All kernels are HBM-bound (SURVEY 8d: residual 32n B, J V_k 16nk+8n B,
// J^T r 24n B).
#include "common.cuh"

namespace {

constexpr int TPBX = 128;  // threads per CTA; each covers 2 columns (VEC) or 1 (scalar, odd m)

template <bool VEC>
struct Pair {
  double a, b;
};

template <bool VEC>
__device__ __forceinline__ Pair<VEC> load_pair(const double* p) {
  Pair<VEC> r;
  if (VEC) {
    double2 v = *reinterpret_cast<const double2*>(p);
    r.a = v.x;
    r.b = v.y;
  } else {
    r.a = *p;
    r.b = 0.0;
  }
  return r;
}
template <bool VEC>
__device__ __forceinline__ void store_pair(double* p, double a, double b) {
  if (VEC)
    *reinterpret_cast<double2*>(p) = make_double2(a, b);
  else
    *p = a;
}

// The linear part of P(u) in the reference's floating-point order (bratu_pde_problem.py:78-82 on scipy 1.18):
// laplace2d is sorted CSR with data {4 h^-2, -h^-2} -> csr_matvec adds data*x entry by entry in column order
// (i-1,j), (i,j-1), (i,j), (i,j+1), (i+1,j); ALPHA*partial_diff_x is COO -> -c u_ij then +c u_i+1,j; the two
// products are then added.  Every product and sum is rounded separately (no FMA contraction): h^-2 (4u - sum nb)
// cancels 4-6 digits on the fine grids, so any other order changes F by ~1e-16 h^-2 |u|, which the GNK trajectory
// amplifies by 1e3 .. 1e5 (DESIGN.md, parity).  Missing neighbours are exact zeros (x + 0 = x).
__device__ __forceinline__ double pde_refbits(const gnk_bratu& prm, double c4, double up, double lf, double mid,
                                              double rt, double dn) {
  const double mc = -prm.c_lap;
  double lap = __dadd_rn(__dmul_rn(mc, up), __dmul_rn(mc, lf));
  lap = __dadd_rn(lap, __dmul_rn(c4, mid));
  lap = __dadd_rn(lap, __dmul_rn(mc, rt));
  lap = __dadd_rn(lap, __dmul_rn(mc, dn));
  const double adv = __dadd_rn(__dmul_rn(-prm.c_adv, mid), __dmul_rn(prm.c_adv, dn));
  return __dadd_rn(lap, adv);
}

// F = y - P(u), expu = e^u, loss = sum_owned F^2
template <bool VEC>
__global__ void __launch_bounds__(TPBX) residual_kernel(gnk_layout lay, gnk_bratu prm, const double* __restrict__ u,
                                                         const double* __restrict__ y, double* __restrict__ F,
                                                         double* __restrict__ expu, int depth, int TR,
                                                         double* __restrict__ partials, unsigned int* ticket,
                                                         double* __restrict__ loss, gnk_p2p_dev pd) {
  __shared__ double sh[32];
  constexpr int W = VEC ? 2 : 1;
  pdl_begin();
  const int m = lay.m;
  const int j0 = W * (blockIdx.x * TPBX + threadIdx.x);
  const int rbeg = -depth + (int)blockIdx.y * TR;
  const int rend = min(rbeg + TR, lay.rows + depth);
  double acc = 0.0;
  if (j0 < m) {
    const double* ub = u + lay.off + j0;
    const bool has_l = j0 > 0, has_r = (j0 + W) < m;
    const double c4 = 4.0 * prm.c_lap;
    Pair<VEC> up = load_pair<VEC>(ub + (int64_t)(rbeg - 1) * m);
    Pair<VEC> mid = load_pair<VEC>(ub + (int64_t)rbeg * m);
#pragma unroll 2
    for (int r = rbeg; r < rend; ++r) {
      const int64_t ro = (int64_t)r * m;
      Pair<VEC> dn = load_pair<VEC>(ub + ro + m);
      const double lf = has_l ? ub[ro - 1] : 0.0;
      const double rt = has_r ? ub[ro + W] : 0.0;
      Pair<VEC> yy = load_pair<VEC>(y + lay.off + j0 + ro);
      // neighbours in j for the two lanes of the pair
      const double la = lf, ra = VEC ? mid.b : rt;
      const double lb = mid.a, rb = rt;
      double ea = 1.0, eb = 1.0;
      double pa = pde_refbits(prm, c4, up.a, la, mid.a, ra, dn.a);
      double pb = VEC ? pde_refbits(prm, c4, up.b, lb, mid.b, rb, dn.b) : 0.0;
      if (prm.lam != 0.0) {
        ea = exp(mid.a);
        pa = __dadd_rn(pa, __dmul_rn(prm.lam, ea));
        if (VEC) {
          eb = exp(mid.b);
          pb = __dadd_rn(pb, __dmul_rn(prm.lam, eb));
        }
      }
      double fa = __dsub_rn(yy.a, pa), fb = __dsub_rn(yy.b, pb);
      const bool owned = (r >= 0 && r < lay.rows);
      const bool in_domain = owned || (r < 0 ? lay.has_lo : lay.has_hi);
      if (!in_domain) {
        fa = 0.0;
        fb = 0.0;
      }
      store_pair<VEC>(F + lay.off + j0 + ro, fa, fb);
      if (expu) store_pair<VEC>(expu + lay.off + j0 + ro, ea, eb);
      if (owned) {
        acc = fma(fa, fa, acc);
        if (VEC) acc = fma(fb, fb, acc);
      }
      up = mid;
      mid = dn;
    }
  }
  acc = block_sum(acc, sh);
  const unsigned int bid = linear_block_id();
  if (threadIdx.x == 0) partials[bid] = acc;
  if (grid_arrive_last(ticket)) {
    double a = 0.0;
    const unsigned int nb = total_blocks();
    for (unsigned int i = threadIdx.x; i < nb; i += blockDim.x) a += __ldcg(partials + i);
    a = block_sum(a, sh);
    if (threadIdx.x == 0) loss[0] = a;
    if (pd.peers) {  // sum over the ranks, in this CTA, over the peers' mailboxes
      __syncthreads();
      p2p_tail_allreduce(pd, loss, 1, 0);
    }
  }
}

// out[:, col] = sign * Op * in[:, col];  grid = (k, j-tiles, row-tiles): the column index is the
// fastest block coordinate so that the CTAs sharing one e^u tile are co-resident and the tile is
// served from L2 after its first HBM read.
template <bool VEC>
__global__ void __launch_bounds__(TPBX) apply_kernel(gnk_layout lay, gnk_bratu prm, const double* __restrict__ expu,
                                                      const double* __restrict__ in, int64_t in_ld, double sign,
                                                      int transpose, int TR, double* __restrict__ out,
                                                      int64_t out_ld, int64_t out_off) {
  constexpr int W = VEC ? 2 : 1;
  pdl_begin();
  const int m = lay.m;
  const int col = blockIdx.x;
  const int j0 = W * (blockIdx.y * TPBX + threadIdx.x);
  if (j0 >= m) return;
  const int rbeg = (int)blockIdx.z * TR;
  const int rend = min(rbeg + TR, lay.rows);
  const double* vb = in + (int64_t)col * in_ld + lay.off + j0;
  const double* eb_ = expu ? expu + lay.off + j0 : nullptr;
  double* ob = out + (int64_t)col * out_ld + out_off + j0;
  const bool has_l = j0 > 0, has_r = (j0 + W) < m;
  const double d0 = __dadd_rn(4.0 * prm.c_lap, -prm.c_adv);          // (L + alpha D) diagonal, as scipy adds it
  const double c_sup = __dadd_rn(-prm.c_lap, prm.c_adv);             // entry (i, i+1): -h^-2 + alpha h^-1
  const double cu = transpose ? c_sup : -prm.c_lap;                  // weight of row i-1
  const double cd = transpose ? -prm.c_lap : c_sup;                  // weight of row i+1
  const double cl = -prm.c_lap;
  Pair<VEC> up = load_pair<VEC>(vb + (int64_t)(rbeg - 1) * m);
  Pair<VEC> mid = load_pair<VEC>(vb + (int64_t)rbeg * m);
#pragma unroll 2
  for (int r = rbeg; r < rend; ++r) {
    const int64_t ro = (int64_t)r * m;
    Pair<VEC> dn = load_pair<VEC>(vb + ro + m);
    const double lf = has_l ? vb[ro - 1] : 0.0;
    const double rt = has_r ? vb[ro + W] : 0.0;
    double dga = d0, dgb = d0;
    if (eb_) {
      Pair<VEC> e = load_pair<VEC>(eb_ + ro);
      dga = __dadd_rn(d0, __dmul_rn(prm.lam, e.a));
      dgb = __dadd_rn(d0, __dmul_rn(prm.lam, e.b));
    }
    const double ra = VEC ? mid.b : rt;
    const double oa = apply_refbits(cu, cl, dga, cd, up.a, lf, mid.a, ra, dn.a);
    const double ob2 = VEC ? apply_refbits(cu, cl, dgb, cd, up.b, mid.a, mid.b, rt, dn.b) : 0.0;
    store_pair<VEC>(ob + ro, sign * oa, sign * ob2);
    up = mid;
    mid = dn;
  }
}

// The speculative trial of a res_old outer iteration in one pass over V_k (gauss_newton_krylow.py:91 + krylow.py:62,64):
//   x = V_k (c + s d)                 over the whole stored column            == combine_kernel
//   w = -J(x)^T F = M(x)^T F          owned points; M(x) = L + alpha D + lam diag(e^x)  == apply_kernel, transpose 1
//   h = V_k^T w                                                               == dots_kernel
// F is the residual at the CURRENT point (depth-1 halo rows valid), and x enters w only through the diagonal e^{x_i} at
// the same point, so every owned point is self-contained: no neighbouring x, no halo of x.  Every value has the bits
// of the kernels it replaces: x is the same fma chain over the columns; e^x the residual kernel's exp; w apply_refbits
// with the same operands; h walks the points exactly as dots_kernel does (same grid, same points per thread in the
// same order, same fma form, same warp -> CTA -> last-CTA tree) -- holding all k <= 8 NB columns of a point at once
// instead of sweeping 8-column blocks leaves each column's accumulation sequence unchanged.  V is read from HBM once
// (the k double2 of a point stay in registers between the x and h phases), F with default caching: its +-m rows are
// L2 hits.  NB = 4 needs 254 registers; ptxas spills 24 bytes there, only inside exp's out-of-range branch.
template <int NB>
__global__ void __launch_bounds__(DOTS_TPB) trial_project_kernel(
    gnk_layout lay, gnk_bratu prm, const double* __restrict__ V, int k, const double* __restrict__ c,
    const double* __restrict__ d, double s, double* __restrict__ x, double* __restrict__ c_out,
    double* __restrict__ cprev2, const double* __restrict__ F, double* __restrict__ w,
    double* __restrict__ partials, unsigned int* ticket, double* __restrict__ h, gnk_p2p_dev pd) {
  constexpr int NJ = 8 * NB;
  constexpr int NFULL = 8 * (NB - 1);  // columns every launch of this instance has (k > 8 (NB - 1))
  __shared__ double coef[GNK_MAX_BASIS];
  __shared__ double wpart[DOTS_TPB / 32][GNK_MAX_BASIS];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  pdl_begin();
  combine_coefficients(k, c, d, s, coef, c_out, cprev2);
  const int m = lay.m;
  const int64_t ld = lay.ld;
  const double d0 = __dadd_rn(4.0 * prm.c_lap, -prm.c_adv);  // as apply_kernel forms the transposed operator
  const double cu = __dadd_rn(-prm.c_lap, prm.c_adv);        // weight of row i-1 (c_sup)
  const double cl = -prm.c_lap;                              // row i+1 and the j neighbours
  const double* Vo = V + lay.off;
  const double* Fo = F + lay.off;
  const int64_t nv = lay.n_own >> 1;
  const int64_t gt = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  double acc[NJ];
#pragma unroll
  for (int u = 0; u < NJ; ++u) acc[u] = 0.0;
#pragma unroll 1
  for (int64_t i = gt; i < nv; i += stride) {
    // a column step the compiler cannot hoist: otherwise it keeps k 64-bit column offsets live across the loop
    int64_t step = ld;
    asm volatile("" : "+l"(step));
    double2 v[NJ];
    const double* pv = Vo + 2 * i;
#pragma unroll
    for (int u = 0; u < NJ; ++u) {
      if (u < NFULL || u < k) v[u] = __ldcs(reinterpret_cast<const double2*>(pv));
      pv += step;
    }
    double2 xv = make_double2(0.0, 0.0);
#pragma unroll
    for (int u = 0; u < NJ; ++u) {
      if (u < NFULL || u < k) {
        xv.x = fma(v[u].x, coef[u], xv.x);
        xv.y = fma(v[u].y, coef[u], xv.y);
      }
    }
    *reinterpret_cast<double2*>(x + lay.off + 2 * i) = xv;
    const int64_t p = 2 * i;
    const int j0 = (int)((unsigned)p % (unsigned)m);  // the entry takes slabs of < 2^31 owned unknowns
    const double2 mid = *reinterpret_cast<const double2*>(Fo + p);
    const double2 up = *reinterpret_cast<const double2*>(Fo + p - m);
    const double2 dn = *reinterpret_cast<const double2*>(Fo + p + m);
    const double lf = j0 > 0 ? Fo[p - 1] : 0.0;
    const double rt = (j0 + 2) < m ? Fo[p + 2] : 0.0;
    double dga = d0, dgb = d0;
    if (prm.lam != 0.0) {
      dga = __dadd_rn(d0, __dmul_rn(prm.lam, exp(xv.x)));
      dgb = __dadd_rn(d0, __dmul_rn(prm.lam, exp(xv.y)));
    }
    double2 wv;
    wv.x = apply_refbits(cu, cl, dga, cl, up.x, lf, mid.x, mid.y, dn.x);
    wv.y = apply_refbits(cu, cl, dgb, cl, up.y, mid.x, mid.y, rt, dn.y);
    *reinterpret_cast<double2*>(w + lay.off + p) = wv;
#pragma unroll
    for (int u = 0; u < NJ; ++u) {
      if (u < NFULL || u < k) acc[u] = fma(v[u].y, wv.y, fma(v[u].x, wv.x, acc[u]));
    }
  }
  // x on the rest of the stored column, [0, off) and [off + n_own, ld): combine_kernel covers the whole column, and the
  // residual at depth 1 reads x on the halo rows
  const int64_t nlo = lay.off >> 1, nrest = nlo + ((ld - lay.off - lay.n_own) >> 1);
  for (int64_t q = gt; q < nrest; q += stride) {
    const int64_t e = q < nlo ? 2 * q : lay.off + lay.n_own + 2 * (q - nlo);
    double2 xv = make_double2(0.0, 0.0);
    for (int u = 0; u < k; ++u) {
      const double2 vv = __ldcs(reinterpret_cast<const double2*>(V + (int64_t)u * ld + e));
      xv.x = fma(vv.x, coef[u], xv.x);
      xv.y = fma(vv.y, coef[u], xv.y);
    }
    *reinterpret_cast<double2*>(x + e) = xv;
  }
#pragma unroll
  for (int u = 0; u < NJ; ++u) {
    if (u < k) {
      const double r = warp_sum(acc[u]);
      if (lane == 0) wpart[wid][u] = r;
    }
  }
  dots_finish(wpart, k, partials, ticket, h, pd);
}

// diag(J^T J): squared column norms of P
template <bool VEC>
__global__ void __launch_bounds__(TPBX) normal_diag_kernel(gnk_layout lay, gnk_bratu prm,
                                                            const double* __restrict__ expu, int TR,
                                                            double* __restrict__ out) {
  constexpr int W = VEC ? 2 : 1;
  const int m = lay.m;
  const int j0 = W * (blockIdx.x * TPBX + threadIdx.x);
  if (j0 >= m) return;
  const int rbeg = (int)blockIdx.y * TR;
  const int rend = min(rbeg + TR, lay.rows);
  const double d0 = 4.0 * prm.c_lap - prm.c_adv;
  const double cl2 = prm.c_lap * prm.c_lap;
  const double cd2 = (prm.c_adv - prm.c_lap) * (prm.c_adv - prm.c_lap);
  for (int r = rbeg; r < rend; ++r) {
    const int64_t ro = lay.off + (int64_t)r * m + j0;
    double dga = d0, dgb = d0;
    if (expu) {
      Pair<VEC> e = load_pair<VEC>(expu + ro);
      dga = fma(prm.lam, e.a, d0);
      dgb = fma(prm.lam, e.b, d0);
    }
    const bool above = (r > 0) || lay.has_lo;               // a grid row i-1 exists
    const bool below = (r < lay.rows - 1) || lay.has_hi;    // a grid row i+1 exists
    double base = (above ? cd2 : 0.0) + (below ? cl2 : 0.0);
    double a = dga * dga + base + ((j0 > 0) ? cl2 : 0.0) + ((j0 + 1 < m) ? cl2 : 0.0);
    double b = 0.0;
    if (VEC) b = dgb * dgb + base + cl2 + ((j0 + 2 < m) ? cl2 : 0.0);
    store_pair<VEC>(out + ro, a, b);
  }
}


// Rows per CTA strip.  A strip re-reads one halo row above and below (from L2), so taller is cheaper per row, but
// the grid should fill whole waves of resident CTAs (8 x 128 threads per SM at <= 64 registers): a 1.7-wave grid
// leaves a quarter of the machine idle in its second wave.  Pick the height with the best wave efficiency, charging
// the halo re-reads lightly.
inline int pick_tr(const gnk_ctx* ctx, int gx, int rows, int mult) {
  const double cap = 8.0 * ctx->sm_count;
  int best = 1;
  double best_score = -1.0;
  for (int tr = 32; tr >= 1; tr >>= 1) {
    const double ctas = (double)gx * mult * (double)ceil_div(rows, tr);
    const double waves = ctas / cap;
    const double eff = (waves <= 1.0) ? waves : waves / (double)(int64_t)(waves + 0.999999);
    const double score = eff - 0.05 * (2.0 / tr);
    if (score > best_score + 1e-9) {
      best_score = score;
      best = tr;
    }
  }
  return best;
}

// the fused residual kernel carries exp() and a block reduction per strip: measured best with the tallest strip that
// still gives every SM six 128-thread CTAs (two were enough to fill the machine at 4096^2 but left the 512-row slabs
// of an 8-GPU run at 14 warps per SM: 34 us for 10 us of traffic)
inline int pick_tr_tall(const gnk_ctx* ctx, int gx, int rows) {
  int tr = 32;
  while (tr > 2 && (int64_t)gx * ceil_div(rows, tr) < 6LL * ctx->sm_count) tr >>= 1;
  return tr;
}

inline int check_layout(const gnk_layout* lay) {
  if (!lay || lay->m <= 0 || lay->rows <= 0 || lay->halo < 2) return -1;
  if (lay->off != (int64_t)lay->halo * lay->m) return -1;
  if (lay->n_own != (int64_t)lay->rows * lay->m) return -1;
  if (lay->ld < (int64_t)(lay->rows + 2 * lay->halo) * lay->m) return -1;
  return 0;
}

}  // namespace

extern "C" {

int gnk_bratu_residual(gnk_ctx* ctx, const gnk_layout* lay, const gnk_bratu* prm, const double* d_u,
                       const double* d_y, double* d_F, double* d_expu, int depth, double* d_loss, void* stream) {
  GNK_REQUIRE(ctx && prm && d_u && d_y && d_F && d_loss, "gnk_bratu_residual: null argument");
  GNK_REQUIRE(check_layout(lay) == 0, "gnk_bratu_residual: inconsistent stencil layout");
  GNK_REQUIRE(depth == 0 || depth == 1, "gnk_bratu_residual: depth must be 0 or 1");
  const bool vec = (lay->m % 2) == 0;
  const int gx = (int)ceil_div(lay->m, (vec ? 2 : 1) * TPBX);
  const int R = lay->rows + 2 * depth;
  const int tr = pick_tr_tall(ctx, gx, R);
  dim3 grid(gx, (unsigned)ceil_div(R, tr));
  GNK_REQUIRE((int64_t)grid.x * grid.y <= 65536, "gnk_bratu_residual: grid exceeds the partials scratch");
  double* part = ctx->d_partials + PART_RESID;
  const gnk_p2p_dev pd = p2p_next(ctx);
  if (vec)
    GNK_CUDA(gnk_launch(gnk_pdl_for(lay->n_own), residual_kernel<true>, grid, dim3(TPBX), 0, (cudaStream_t)stream, *lay, *prm, d_u, d_y, d_F, d_expu,
                        depth, tr, part, ctx->d_tickets + TK_RESID, d_loss, pd));
  else
    GNK_CUDA(gnk_launch(gnk_pdl_for(lay->n_own), residual_kernel<false>, grid, dim3(TPBX), 0, (cudaStream_t)stream, *lay, *prm, d_u, d_y, d_F,
                        d_expu, depth, tr, part, ctx->d_tickets + TK_RESID, d_loss, pd));
  GNK_LAUNCH_CHECK(ctx);
  return 0;
}

int gnk_stencil_apply(gnk_ctx* ctx, const gnk_layout* lay, const gnk_bratu* prm, const double* d_expu,
                      const double* d_in, int64_t in_ld, int k, double sign, int transpose, double* d_out,
                      int64_t out_ld, int64_t out_off, void* stream) {
  GNK_REQUIRE(ctx && prm && d_in && d_out, "gnk_stencil_apply: null argument");
  GNK_REQUIRE(check_layout(lay) == 0, "gnk_stencil_apply: inconsistent stencil layout");
  GNK_REQUIRE(k >= 1 && k <= 65535, "gnk_stencil_apply: k out of range");
  GNK_REQUIRE(prm->lam == 0.0 || d_expu, "gnk_stencil_apply: e^u diagonal required when lam != 0");
  const bool vec = (lay->m % 2) == 0 && (in_ld % 2) == 0 && (out_ld % 2) == 0 && (out_off % 2) == 0;
  const int gx = (int)ceil_div(lay->m, (vec ? 2 : 1) * TPBX);
  const int tr = pick_tr(ctx, gx, lay->rows, k);
  dim3 grid(k, gx, (unsigned)ceil_div(lay->rows, tr));
  GNK_REQUIRE(grid.z <= 65535, "gnk_stencil_apply: too many row tiles");
  const double* e = (prm->lam == 0.0) ? nullptr : d_expu;
  if (vec)
    GNK_CUDA(gnk_launch(gnk_pdl_for(lay->n_own), apply_kernel<true>, grid, dim3(TPBX), 0, (cudaStream_t)stream, *lay, *prm, e, d_in, in_ld, sign,
                        transpose, tr, d_out, out_ld, out_off));
  else
    GNK_CUDA(gnk_launch(gnk_pdl_for(lay->n_own), apply_kernel<false>, grid, dim3(TPBX), 0, (cudaStream_t)stream, *lay, *prm, e, d_in, in_ld, sign,
                        transpose, tr, d_out, out_ld, out_off));
  GNK_LAUNCH_CHECK(ctx);
  return 0;
}

int gnk_bratu_trial_project(gnk_ctx* ctx, const gnk_layout* lay, const gnk_bratu* prm, const double* d_V, int k,
                            const double* d_c, const double* d_d, double s, double* d_x, double* d_c_out,
                            double* d_cprev2, const double* d_F, double* d_w, double* d_h, void* stream) {
  GNK_REQUIRE(ctx && prm && d_V && d_c && d_x && d_F && d_w && d_h, "gnk_bratu_trial_project: null argument");
  GNK_REQUIRE(check_layout(lay) == 0, "gnk_bratu_trial_project: inconsistent stencil layout");
  GNK_REQUIRE(k >= 1, "gnk_bratu_trial_project: k out of range");
  GNK_REQUIRE(d_c_out != d_c, "gnk_bratu_trial_project: c_out must not alias c (rejected trials re-read c)");
  // double2 points never straddle a grid row and stay 16-byte aligned; k columns of a point fit the registers
  if ((lay->m & 1) || (lay->off & 1) || (lay->ld & 1) || k > 32 || lay->n_own >= (int64_t(1) << 31)) return 1;
  const int grid = dots_grid(ctx, lay->n_own);  // gnk_cgs_dots' grid: it fixes the summation order of h
  auto kern = trial_project_kernel<4>;
  if (k <= 8)
    kern = trial_project_kernel<1>;
  else if (k <= 16)
    kern = trial_project_kernel<2>;
  else if (k <= 24)
    kern = trial_project_kernel<3>;
  GNK_CUDA(gnk_launch(gnk_pdl_for(lay->n_own), kern, dim3(grid), dim3(DOTS_TPB), 0, (cudaStream_t)stream, *lay, *prm,
                      d_V, k, d_c, d_d, s, d_x, d_c_out, d_cprev2, d_F, d_w, ctx->d_partials + PART_DOTS,
                      ctx->d_tickets + TK_DOTS, d_h, p2p_next(ctx)));
  GNK_LAUNCH_CHECK(ctx);
  return 0;
}

int gnk_stencil_normal_diag(gnk_ctx* ctx, const gnk_layout* lay, const gnk_bratu* prm, const double* d_expu,
                            double* d_out, void* stream) {
  GNK_REQUIRE(ctx && prm && d_out, "gnk_stencil_normal_diag: null argument");
  GNK_REQUIRE(check_layout(lay) == 0, "gnk_stencil_normal_diag: inconsistent stencil layout");
  GNK_REQUIRE(prm->lam == 0.0 || d_expu, "gnk_stencil_normal_diag: e^u diagonal required when lam != 0");
  const bool vec = (lay->m % 2) == 0;
  const int gx = (int)ceil_div(lay->m, (vec ? 2 : 1) * TPBX);
  const int tr = pick_tr(ctx, gx, lay->rows, 1);
  dim3 grid(gx, (unsigned)ceil_div(lay->rows, tr));
  const double* e = (prm->lam == 0.0) ? nullptr : d_expu;
  if (vec)
    normal_diag_kernel<true><<<grid, TPBX, 0, (cudaStream_t)stream>>>(*lay, *prm, e, tr, d_out);
  else
    normal_diag_kernel<false><<<grid, TPBX, 0, (cudaStream_t)stream>>>(*lay, *prm, e, tr, d_out);
  GNK_LAUNCH_CHECK(ctx);
  return 0;
}

}  // extern "C"
