// common.cuh -- shared device helpers and the context object of the gnk_b200 library (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>

#include "gnk_b200.h"

// ------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------
struct gnk_ctx {
  int device = 0;
  int sm_count = 148;
  int64_t launches = 0;
  // cross-CTA reduction scratch: partial sums and self-resetting tickets (one per call site)
  double* d_partials = nullptr;   // GNK_PARTIALS doubles
  unsigned int* d_tickets = nullptr;  // GNK_TICKETS uints, zero-initialised
  // TSQR R-factor ping/pong buffers
  double* d_rbuf[2] = {nullptr, nullptr};
  size_t rbuf_bytes = 0;
  // communicator (comm.cu)
  void* nccl_comm = nullptr;
  int rank = 0, nranks = 1;
  double* d_gather = nullptr;     // all-gather staging
  size_t gather_bytes = 0;
  // pinned host scalars for the C-side loops (cgls)
  double* h_pinned = nullptr;
  // peer-memory mailboxes (comm.cu): one device block per rank, mapped into every peer of the node with CUDA IPC;
  // the small all-gathers and the halo rows are written straight into the peers' mailboxes over NVLink
  void* p2p_local = nullptr;          // this rank's mailbox
  void* p2p_peer[16] = {nullptr};     // every rank's mailbox as seen from this process (own entry = p2p_local)
  void** d_p2p_peer = nullptr;        // the same table in device memory
  unsigned long long p2p_seq = 0;     // gathers issued so far (identical on all ranks: same call sequence)
  unsigned long long p2p_hseq = 0;    // halo exchanges issued so far
  int p2p_ready = 0;
  int p2p_fused = 0;                  // the reducing kernels finish their cross-rank reduction themselves
  // per-CTA partial dot products of gnk_stencil_apply_dots (k * CTAs-per-column doubles, grown on demand)
  double* d_apart = nullptr;
  size_t apart_bytes = 0;
  // CholeskyQR2 scratch (cholqr.cu): per-CTA Gram partials, the gathered Gram matrices, T, R1, status word
  double* d_cholqr = nullptr;
  double* d_gramw = nullptr;          // wide Gram matrix scratch of gnk_gram_cgls (gram_cgls.cu)
  int ls_method = 0;                  // gnk_tsqr_ls_method: 0 automatic, 1 Householder TSQR only
  // gnk_scalars_fetch / gnk_scalars_wait (api.cu): the copy stream and event of the scalar read-back
  cudaStream_t fetch_stream = nullptr;
  cudaEvent_t fetch_event = nullptr;
  // gnk_cgls (cgls.cu): the stopping test of CG iteration i is read while iteration i + 1 is already queued; two reads in
  // flight, each with an event on the caller's stream ([0..1]) and one on the copy stream ([2..3])
  cudaEvent_t cg_event[4] = {nullptr, nullptr, nullptr, nullptr};
  // gnk_csr_pattern (csr.cu): row of every non-zero, sort keys and values, column histogram, cub temp (grown on demand)
  void* d_pattern = nullptr;
  size_t pattern_bytes = 0;
  // gnk_dense_qr_ls (dense_qr.cu): panel partials, pivot rows, taus, split partials of V^T C and T^T W (grown on demand)
  double* d_dqr = nullptr;
  size_t dqr_bytes = 0;
};
int gnk_ensure_fetch_stream(gnk_ctx* ctx);  // api.cu: creates fetch_stream / fetch_event on first use

constexpr int GNK_PARTIALS = 1 << 19;  // doubles (4 MiB)
constexpr int GNK_TICKETS = 64;

// regions inside gnk_ctx::d_partials (doubles); one per call site so that no two kernels share scratch
constexpr int64_t PART_STATS = 0;                                   // 2 * grid
constexpr int64_t PART_DOTS = 8192;                                 // grid(<=1184) * GNK_MAX_BASIS
constexpr int64_t PART_UPDATE = PART_DOTS + 1184 * GNK_MAX_BASIS;   // 2 * grid
constexpr int64_t PART_DOT1 = PART_UPDATE + 8192;                   // grid
constexpr int64_t PART_CG = PART_DOT1 + 8192;                       // 2 * grid
constexpr int64_t PART_SCAL = PART_CG + 8192;                       // 64 device scalars of the C-side loops
constexpr int64_t PART_RESID = GNK_PARTIALS - 65536;                // residual kernel: one per CTA
static_assert(PART_SCAL + 64 <= PART_RESID, "partials scratch overflow");

enum TicketSlot { TK_RESID = 0, TK_STATS = 1, TK_DOTS = 2, TK_UPDATE = 3, TK_DOT1 = 4, TK_CG = 5, TK_APPLY_DOTS = 6,
                  TK_CHOLQR = 7, TK_NORMALIZE = 8, TK_GRAMW = 9 };

void gnk_set_error(const std::string& s);
int gnk_fail(const char* what, cudaError_t e, const char* file, int line);

#define GNK_CUDA(expr)                                                    \
  do {                                                                    \
    cudaError_t e__ = (expr);                                             \
    if (e__ != cudaSuccess) return gnk_fail(#expr, e__, __FILE__, __LINE__); \
  } while (0)

#define GNK_LAUNCH_CHECK(ctx)                                             \
  do {                                                                    \
    (ctx)->launches++;                                                    \
    cudaError_t e__ = cudaGetLastError();                                 \
    if (e__ != cudaSuccess) return gnk_fail("kernel launch", e__, __FILE__, __LINE__); \
  } while (0)

#define GNK_REQUIRE(cond, msg)                                            \
  do {                                                                    \
    if (!(cond)) {                                                        \
      gnk_set_error(std::string(msg) + " (" #cond ")");                   \
      return -2;                                                          \
    }                                                                     \
  } while (0)

// ------------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Block-wide sum with a fixed reduction tree (deterministic).  `sh` needs 32 doubles.  The result is
// valid in every thread of warp 0.  Ends with the shared buffer free for reuse after a __syncthreads.
__device__ __forceinline__ double block_sum(double v, double* sh) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) sh[w] = v;
  __syncthreads();
  const int nw = (blockDim.x + 31) >> 5;
  double r = (w == 0 && lane < nw) ? sh[lane] : 0.0;
  if (w == 0) r = warp_sum(r);
  return r;
}
__device__ __forceinline__ double block_max(double v, double* sh) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  v = warp_max(v);
  __syncthreads();
  if (lane == 0) sh[w] = v;
  __syncthreads();
  const int nw = (blockDim.x + 31) >> 5;
  double r = (w == 0 && lane < nw) ? sh[lane] : 0.0;  // inputs are |.| >= 0
  if (w == 0) r = warp_max(r);
  return r;
}

// "last CTA finishes" pattern.  Thread 0 of every CTA has published its partial(s) to global memory
// before calling; returns true in ALL threads of the CTA that arrives last.  The ticket wraps back
// to 0, so the same slot serves the next launch without a memset.
__device__ __forceinline__ bool grid_arrive_last(unsigned int* ticket) {
  __shared__ int s_last;
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    unsigned int t = atomicInc(ticket, gridDim.x * gridDim.y * gridDim.z - 1);
    s_last = (t == gridDim.x * gridDim.y * gridDim.z - 1);
    __threadfence();
  }
  __syncthreads();
  return s_last != 0;
}

__device__ __forceinline__ unsigned int linear_block_id() {
  return blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z);
}
__device__ __forceinline__ unsigned int total_blocks() { return gridDim.x * gridDim.y * gridDim.z; }

// ------------------------------------------------------------------------------------------------
// peer-memory mailboxes (comm.cu): layout and the device side of a gather, shared with the kernels that finish their
// cross-rank reduction in their own last CTA (residual, Gram-Schmidt dots, update statistics)
// Mailbox layout (bytes): [0, 4096) flags: u64 gather[16], u64 halo[2] at +1024;
//                         gather data 2 x nranks x P2P_GMAX doubles; halo data 2 parities x 2 sides x P2P_HMAX doubles;
//                         2 x nranks x P2P_LLMAX 16-byte lines {lo, tag, hi, tag} of the in-kernel all-reduces;
//                         2 parities x 2 sides x P2P_HMAX such lines for the halo rows pushed by normalize_halo_kernel.
// ------------------------------------------------------------------------------------------------
constexpr int P2P_MAXR = 16;
constexpr int64_t P2P_GMAX = (int64_t)GNK_TSQR_MAX * GNK_TSQR_MAX;    // largest gather: one R triangle
constexpr int64_t P2P_HMAX = 2 * 16384;                              // largest halo message: 2 grid rows of 16384
constexpr size_t P2P_FLAG_BYTES = 4096;
constexpr unsigned long long P2P_TIMEOUT_NS = 20ull * 1000 * 1000 * 1000;

__host__ __device__ inline size_t p2p_gather_off(int nranks, int parity, int r) {
  return P2P_FLAG_BYTES + sizeof(double) * (size_t)((parity * nranks + r) * P2P_GMAX);
}
__host__ __device__ inline size_t p2p_halo_off(int nranks, int parity, int side) {
  return P2P_FLAG_BYTES + sizeof(double) * (size_t)(2 * nranks * P2P_GMAX) +
         sizeof(double) * (size_t)((parity * 2 + side) * P2P_HMAX);
}
// flag-in-data lines of the in-kernel all-reduces (p2p_tail_allreduce): 16 bytes per double, after the halo slots
constexpr int P2P_LLMAX = 1024;
__host__ __device__ inline size_t p2p_ll_off(int nranks, int parity, int r) {
  return p2p_halo_off(nranks, 2, 0) + 16 * (size_t)((parity * nranks + r) * P2P_LLMAX);
}
// the same lines for the halo rows pushed by normalize_halo_kernel (vector_ops.cu): 2 parities x 2 sides x P2P_HMAX
__host__ __device__ inline size_t p2p_hll_off(int nranks, int parity, int side) {
  return p2p_ll_off(nranks, 2, 0) + 16 * (size_t)((parity * 2 + side) * P2P_HMAX);
}

struct gnk_p2p_dev {        // kernel argument; peers == nullptr: single rank or NCCL path, nothing to do
  void* const* peers;
  int rank, nranks;
  unsigned long long seq;
};
// the next collective of the gather channel, if the library finishes reductions inside the producing kernels
static inline gnk_p2p_dev p2p_next(gnk_ctx* ctx) {
  gnk_p2p_dev pd{nullptr, 0, 1, 0ull};
  if (ctx->p2p_ready && ctx->p2p_fused) {
    pd.peers = ctx->d_p2p_peer;
    pd.rank = ctx->rank;
    pd.nranks = ctx->nranks;
    pd.seq = ++ctx->p2p_seq;
  }
  return pd;
}

__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
// spin until *flag >= seq; a peer that never arrives (diverged control flow, dead process) must not hang the GPU
__device__ __forceinline__ void wait_flag(const unsigned long long* flag, unsigned long long seq) {
  const unsigned long long t0 = global_ns();
  while (ld_acquire_sys(flag) < seq) {
    if (global_ns() - t0 > P2P_TIMEOUT_NS) __trap();
  }
}
__device__ __forceinline__ double ld_volatile(const double* p) {
  double v;
  asm volatile("ld.volatile.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
  return v;
}

// Cross-rank reduction of vals[0..count) (count <= blockDim.x, count <= P2P_LLMAX), executed by ALL threads of ONE
// CTA -- the CTA that has just written this rank's values (make them visible with a __syncthreads first).  Same
// rank-ordered arithmetic as p2p_gather_kernel (comm.cu), but a flag-in-data protocol instead of data + fence + flag:
// every double travels as ONE 16-byte store {lo, seq32, hi, seq32} into the peer's mailbox, and the receiver polls the
// line itself until both tags carry this collective's number (each 8-byte half of the line is written atomically, so a
// line whose two tags match holds both halves of the value).  No __threadfence_system (a full NVLink round trip), no
// separate flag hop, no block barrier: the cost is one one-way store latency plus the ranks' skew.  Lines are
// double-buffered on the parity of the sequence number like the other slots (a rank is never more than one collective
// ahead of a peer), and a tag can only match a stale line after 2^32 - 1 collectives.  op: 0 sum, 1 max, 2 (sum, max).
__device__ __forceinline__ void st_ll(void* p, double v, unsigned tag) {
  const unsigned lo = (unsigned)__double2loint(v), hi = (unsigned)__double2hiint(v);
  asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(lo), "r"(tag), "r"(hi), "r"(tag)
               : "memory");
}
__device__ __forceinline__ double ld_ll(const void* p, unsigned tag) {
  unsigned lo, t1, hi, t2;
  asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(lo), "=r"(t1), "=r"(hi), "=r"(t2) : "l"(p) : "memory");
  if (t1 != tag || t2 != tag) {
    const unsigned long long t0 = global_ns();
    do {
      asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(lo), "=r"(t1), "=r"(hi), "=r"(t2) : "l"(p) : "memory");
      if (global_ns() - t0 > P2P_TIMEOUT_NS) __trap();  // a peer that never arrives must not hang the GPU
    } while (t1 != tag || t2 != tag);
  }
  return __hiloint2double((int)hi, (int)lo);
}
__device__ __forceinline__ void p2p_tail_allreduce(const gnk_p2p_dev& pd, double* vals, int count, int op) {
  const int t = threadIdx.x;
  if (t >= count) return;
  const int parity = (int)(pd.seq & 1ull);
  const unsigned tag = (unsigned)(pd.seq % 0xFFFFFFFFull) + 1u;  // never 0: the mailbox starts zeroed
  const double v = vals[t];
  for (int r = 0; r < pd.nranks; ++r)
    st_ll(static_cast<char*>(pd.peers[r]) + p2p_ll_off(pd.nranks, parity, pd.rank) + 16 * (size_t)t, v, tag);
  const char* mine = static_cast<const char*>(pd.peers[pd.rank]);
  const bool is_max = (op == 1) || (op == 2 && t == 1);
  double a = ld_ll(mine + p2p_ll_off(pd.nranks, parity, 0) + 16 * (size_t)t, tag);
  for (int r = 1; r < pd.nranks; ++r) {
    const double b = ld_ll(mine + p2p_ll_off(pd.nranks, parity, r) + 16 * (size_t)t, tag);
    a = is_max ? fmax(a, b) : a + b;
  }
  vals[t] = a;
}

// One row of sign * (M v) or sign * (M^T v), M = L + alpha D + lam diag(e^u), in the order scipy uses for
// J @ V (csr_matvecs, gauss_newton_krylow.py:86) and -J.T @ r (csc_matvec, krylow.py:62): five rounded products
// added one at a time, neighbours in ascending index order.  cu / cd are the weights of rows i-1 / i+1.
__device__ __forceinline__ double apply_refbits(double cu, double cl, double dg, double cd, double up, double lf,
                                                double mid, double rt, double dn) {
  double s = __dadd_rn(__dmul_rn(cu, up), __dmul_rn(cl, lf));
  s = __dadd_rn(s, __dmul_rn(dg, mid));
  s = __dadd_rn(s, __dmul_rn(cl, rt));
  s = __dadd_rn(s, __dmul_rn(cd, dn));
  return s;
}

static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// ------------------------------------------------------------------------------------------------
// Programmatic dependent launch between the ~11 kernels of an outer iteration.  A kernel launched with gnk_launch may
// be scheduled as soon as every CTA of its predecessor has passed pdl_begin(): its CTAs become resident while the
// predecessor drains and start the instant it has completed, which hides the launch latency and the block-scheduling
// ramp between dependent kernels (2-3 us each; ~30 us per outer iteration in the latency regime: the 8-GPU slabs, the
// 1024^2 grid).  pdl_begin() is the first statement of every such kernel: it waits until the predecessor has completed
// and its memory operations are visible (so neither read-after-write nor write-after-read hazards can arise: nothing
// global is touched before it), then lets the successor be scheduled.  Launched without the attribute, both
// instructions are no-ops.  The attribute is set only for slabs of at most GNK_PDL_MAX_N unknowns (measured on one GPU:
// 1024^2 restart 30 4236 -> 4498 it/s with it, 4096^2 371 -> 365 it/s: on big slabs the early-resident CTAs of the
// successor take warp slots from a predecessor that is still streaming).  GNK_PDL=0 switches it off, GNK_PDL=2 forces it.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void pdl_begin() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
int gnk_pdl_mode();  // 0 off, 1 by size, 2 always
constexpr int64_t GNK_PDL_MAX_N = 6 * 1024 * 1024;
inline bool gnk_pdl_for(int64_t n_unknowns) {
  const int mode = gnk_pdl_mode();
  return mode == 2 || (mode == 1 && n_unknowns <= GNK_PDL_MAX_N);
}
template <typename... P, typename... A>
inline cudaError_t gnk_launch(bool pdl, void (*kern)(P...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                              A&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = pdl ? 1 : 0;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<P>(args)...);
}
