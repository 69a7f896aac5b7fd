// gp64_kernel: the hot kernel for batches of small objects (N <= 64), one WARP per object,
// the block count NB = ceil(N_max/8) a compile-time constant so that every tile loop is
// straight-line code the scheduler can overlap (ncu, round 1: the generic kernel spent
// 40 % of its issue slots waiting on dependent FP64 results and 12 % on loop/index code).
//
// Same algorithm as cgp_small.cu (8x8 tiles, left-looking block Cholesky on DMMA, T_J = L_JJ^-1 on the
// diagonal slots), restructured in phases that are each dense in independent FP64 work.
//
// Tile layout (round 2; ncu r02c: the factor kernel ran at 80 % of the SM's shared-memory wavefront rate,
// 27 % of the wavefronts bank conflicts): element (r, c) of a tile lives in 16-byte unit
// rho(r)*4 + ((c>>1) ^ sigma(r)), half c&1, with rho(r) = r ^ ((r>>1)&1) and sigma(r) = (r>>1)&2.  Then
//   * lane (g,t)'s DMMA accumulator pair (row g, columns 2t, 2t+1) is ONE 16-byte unit, and the same unit is the
//     lane's operand of both k-halves of a product X*Y^T (the two DMMAs of a tile product sum over the even and the
//     odd k): accumulators are stored with one conflict-free STS.128, fragments loaded with one LDS.128, and a
//     tile that was just accumulated can be fed to the next DMMA straight from its registers (the panel
//     solve and the triangular inverse need no shared-memory round trip);
//   * the transposed fragment (elements (2t,g), (2t+1,g)) is two conflict-free 8-byte loads.
// Phases:
//   K   covariance tiles: generated up front, 8 independent exp chains per lane in flight (gp64_kernel), or column by
//       column right where they are consumed (gp64_ll_kernel, whose rows retire and free their slots)
//   C   column J: every tile of the column accumulates its rank-8J update at once (2 (NB-J) independent DMMA
//       chains), in-register diagonal factorisation (T_J = L_JJ^-1), panel solve by DMMA from registers,
//       z_J = T_J (r_J - sum L[J][P] z_P) behind the next column
//   I   pulls only: L^-1 by rows (held transposed while it is built), column norms, alpha
//   P   prediction: TWO blocks of 8 grid points per pass; the 4 NB cross-covariance fragments are generated into the
//       accumulators, then L v = h is solved by block forward substitution on the tensor cores (4 NB(NB+1)/2 DMMAs),
//       mean = v . z, var = amp* - |v|^2 -- no L^-1, no alpha
// Objects with fewer than NB blocks are padded with identity rows (exact, just wasteful);
// per-object n masks the covariance entries.  Reference: see cgp_small.cu header.
#include <atomic>
#include "cgp_internal.h"
#include "cgp_math.cuh"

#include <math.h>
#include <stdlib.h>
#include <type_traits>

#ifndef CGP64_GRID_U
#define CGP64_GRID_U 2            // blocks of 8 grid points per pass of the prediction kernels
#endif

namespace cgp {
namespace {

constexpr int TILE = 64;
constexpr unsigned FULL = 0xffffffffu;
constexpr double LOG_2PI = 1.8378770664093454835606594728112;
constexpr double LN2 = 0.693147180559945309417232;

// (I << 4 | J) of the q-th tile of the lower block triangle, row by row (slot order)
__constant__ unsigned char kTri[36] = {
    0x00, 0x10, 0x11, 0x20, 0x21, 0x22, 0x30, 0x31, 0x32, 0x33, 0x40, 0x41, 0x42, 0x43, 0x44,
    0x50, 0x51, 0x52, 0x53, 0x54, 0x55, 0x60, 0x61, 0x62, 0x63, 0x64, 0x65, 0x66,
    0x70, 0x71, 0x72, 0x73, 0x74, 0x75, 0x76, 0x77};

__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
      : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
__host__ __device__ constexpr int slot(int i, int j) { return ((i * (i + 1)) >> 1) + j; }
__device__ __forceinline__ int tile_off(int r, int c) {
  const int rho = r ^ ((r >> 1) & 1), sig = (r >> 1) & 2;
  return ((rho * 4 + ((c >> 1) ^ sig)) << 1) + (c & 1);
}

struct Lane {
  int g, t, nat, tr0, tr1;
  __device__ explicit Lane(int lane) {
    g = lane >> 2; t = lane & 3;
    nat = tile_off(g, 2 * t);                            // (g, 2t), (g, 2t+1): accumulator pair == operand fragment
    tr0 = tile_off(2 * t, g); tr1 = tile_off(2 * t + 1, g);
  }
};
__device__ __forceinline__ double2 ld_frag(const double* tiles, int s, const Lane& L) {
  return *reinterpret_cast<const double2*>(tiles + s * TILE + L.nat);
}
__device__ __forceinline__ void st_frag(double* tiles, int s, const Lane& L, double v0, double v1) {
  *reinterpret_cast<double2*>(tiles + s * TILE + L.nat) = make_double2(v0, v1);
}
__device__ __forceinline__ double2 ld_frag_t(const double* tiles, int s, const Lane& L) {   // fragment of the transpose
  const double* p = tiles + s * TILE;
  return make_double2(p[L.tr0], p[L.tr1]);
}
__device__ __forceinline__ double2 ld_vec2(const double* v, int i) { return *reinterpret_cast<const double2*>(v + i); }
__device__ __forceinline__ double red_t(double v) {
  v += __shfl_xor_sync(FULL, v, 1); v += __shfl_xor_sync(FULL, v, 2); return v;
}
__device__ __forceinline__ double red_g(double v) {
  v += __shfl_xor_sync(FULL, v, 4); v += __shfl_xor_sync(FULL, v, 8); v += __shfl_xor_sync(FULL, v, 16); return v;
}

template <int DIM>
__device__ __forceinline__ double rbf_arg(const Cov& c, double ax, double ay, double bx, double by) {
  const double dx = ax - bx;
  if (DIM == 1) return dx * dx * c.h00;
  const double dy = ay - by;
  return fma(dy * c.h11, dy, fma(dx, c.h00, dy * c.h01) * dx);
}

// 8x8 Cholesky of a diagonal tile in accumulator layout + T = L^-1 by the same row operations on an identity
// (see cgp_small.cu).  ONE out-of-line copy per kernel with the eight pivot steps unrolled (static k: shuffle
// sources, the a0/a1 choice and the row predicates become immediates -- about half the instructions of the
// rolled loop), arguments and results in registers.  Inlined at its 8 call sites the unrolled form is 46 KB of
// code and the kernels stall on instruction fetch (the L1.5 instruction cache holds 32 KB).
struct DiagOut { double t0, t1, piv; int badk; };
template <int K>
__device__ __forceinline__ void diag_step(double& a0, double& a1, double& t0, double& t1, double& pivprod, int& badk,
                                          const int g, const int t) {
  constexpr int kc = K >> 1;
  const double ak = (K & 1) ? a1 : a0;
  const double d = __shfl_sync(FULL, ak, K * 4 + kc);
  if (!(d > 0.0) && badk == 0) badk = K + 1;
  const double rinv = cgp_rsqrt(d);
  pivprod *= d;
  const double lg = __shfl_sync(FULL, ak, g * 4 + kc) * rinv;
  // column K again, for the columns this lane owns (only the lower triangle of the tile is meaningful: the
  // covariance tiles are generated with a zero upper triangle, so row K cannot stand in for column K)
  const double lc0 = __shfl_sync(FULL, ak, (2 * t) * 4 + kc) * rinv;
  const double lc1 = __shfl_sync(FULL, ak, (2 * t + 1) * 4 + kc) * rinv;
  a0 = fma(-lg, lc0, a0); a1 = fma(-lg, lc1, a1);
  const double tk0 = __shfl_sync(FULL, t0, K * 4 + t) * rinv;
  const double tk1 = __shfl_sync(FULL, t1, K * 4 + t) * rinv;
  const double f = (g > K) ? lg : 0.0;
  const double n0 = fma(-f, tk0, t0), n1 = fma(-f, tk1, t1);
  t0 = (g == K) ? tk0 : n0; t1 = (g == K) ? tk1 : n1;
}
__device__ __noinline__ DiagOut diag_factor_impl(double a0, double a1, int g, int t) {
  double t0 = (g == 2 * t) ? 1.0 : 0.0;
  double t1 = (g == 2 * t + 1) ? 1.0 : 0.0;
  double pivprod = 1.0; int badk = 0;
  diag_step<0>(a0, a1, t0, t1, pivprod, badk, g, t); diag_step<1>(a0, a1, t0, t1, pivprod, badk, g, t);
  diag_step<2>(a0, a1, t0, t1, pivprod, badk, g, t); diag_step<3>(a0, a1, t0, t1, pivprod, badk, g, t);
  diag_step<4>(a0, a1, t0, t1, pivprod, badk, g, t); diag_step<5>(a0, a1, t0, t1, pivprod, badk, g, t);
  diag_step<6>(a0, a1, t0, t1, pivprod, badk, g, t); diag_step<7>(a0, a1, t0, t1, pivprod, badk, g, t);
  DiagOut o; o.t0 = t0; o.t1 = t1; o.piv = pivprod; o.badk = badk;
  return o;
}
__device__ __forceinline__ void diag_factor(double a0, double a1, const Lane& L,
                                            double& t0, double& t1, double& pivprod, int& badk) {
  const DiagOut o = diag_factor_impl(a0, a1, L.g, L.t);
  t0 = o.t0; t1 = o.t1; pivprod = o.piv; badk = o.badk;
}

// Ring of work counters (one per launch in flight), zeroed in stream order before each launch.
static unsigned long long* next_ticket(cudaStream_t stream) {
  constexpr unsigned RING = 4096;                         // launches that may be in flight on different streams
  constexpr int MAX_DEV = 16;
  static unsigned long long* ring[MAX_DEV] = {nullptr};   // one ring per device of this process
  static std::atomic<unsigned> idx[MAX_DEV];             // host threads may launch concurrently
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= MAX_DEV) return nullptr;
  if (!ring[dev] && cudaMalloc((void**)&ring[dev], RING * sizeof(unsigned long long)) != cudaSuccess) return nullptr;
  unsigned long long* t = ring[dev] + (idx[dev].fetch_add(1) % RING);
  if (cudaMemsetAsync(t, 0, sizeof(unsigned long long), stream) != cudaSuccess) return nullptr;
  return t;
}

__host__ __device__ constexpr int n_vec64(int task) { return task == TASK_LOO ? 6 : 1; }
// covariance phase of gp64_kernel with the table-driven exp (512 more bytes of shared memory per CTA) where that does not
// cost an object per SM: the pulls kernel (9 objects per SM at NB = 8 either way, register-capped at 16 below) and the
// one-pass kernels below NB = 8; at NB = 8 the 36-tile one-pass kernels have 139 bytes to spare before 11 objects become 10
__host__ __device__ constexpr bool ktab64(int task, int nb) {
  return task == TASK_LOO || ((task == TASK_PREDICT || task == TASK_PREDICT_U || task == TASK_LL) && nb < 8);
}
__host__ __device__ constexpr bool uni64(int task) { return task == TASK_PREDICT_FU || task == TASK_PREDICT_U; }
// uniform-grid kernels: per object point, the powers of the pass anchors E_a R^g (g < 8) and R^8 (see UNI in gp64_kernel)
constexpr int UNI_ROWS = 9;
// doubles per object point staged per warp: the coordinates and the noise, or the anchor powers of the uniform grid
__host__ __device__ constexpr int px_rows64(int task, int dim) { return uni64(task) ? UNI_ROWS : dim + 1; }
// the 2^(j/64) table of cgp_exp_tab: covariance tiles (ktab64) or the anchors of the uniform grid
__host__ __device__ constexpr bool etab64(int task, int nb) { return ktab64(task, nb) || uni64(task); }
// Warps per CTA that share one staged factor in the grid kernels (see WPC in gp64_kernel).  Measured at C2 with 2: 16 warps
// per SM on 8 factors, but 7 passes split 4 + 3 between the two warps, two CTA barriers per object and 128-register
// spills: grid kernel 2.13 -> 2.42 ms.  Kept at 1 (CGP64_GRID_WPC=2 at compile time selects the shared form; tested).
#ifndef CGP64_GRID_WPC
#define CGP64_GRID_WPC 1
#endif
__host__ __device__ constexpr int warps_per_cta(int task) { return (task == TASK_PREDICT_F || task == TASK_PREDICT_FU) ? CGP64_GRID_WPC : 1; }

// Registers are allocated per SM sub-partition (16 K each): 3 warps per partition need <= 168
// registers per thread (grid phase: 64 accumulators + 32 fragments), 4 warps <= 128 (factorisation,
// pulls: shared memory allows 16+ objects per SM below 56 points); hence the minimum-blocks bounds.
template <int DIM, int TASK, int NB>
__global__ void __launch_bounds__(32 * warps_per_cta(TASK), warps_per_cta(TASK) > 1 ? 16 / warps_per_cta(TASK) :
                                  (TASK == TASK_PREDICT || TASK == TASK_PREDICT_F || TASK == TASK_PREDICT_FU || TASK == TASK_PREDICT_U) ? 12 : 16)
gp64_kernel(const SmallArgs a, unsigned long long* __restrict__ ticket) {
  extern __shared__ __align__(16) double smem[];
  // WPC warps per CTA share ONE object: the grid kernels (factor staged from the workspace) run two warps on the
  // same shared-memory tiles, alternating over the passes of the grid -- 16 warps per SM on 8 staged factors where one
  // warp per object was limited to 11 by shared memory (the grid phase needs < 128 registers since the forward
  // substitution keeps no separate cross-covariance fragments).  Every other task: one warp, one object.
  constexpr int WPC = warps_per_cta(TASK);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const Lane L(lane);
  Cov cov = a.cov;
  constexpr int LD = 8 * NB;
  constexpr int NT = NB * (NB + 1) / 2;
  double* tiles = smem;
  constexpr int PXR = px_rows64(TASK, DIM);
  double* px = tiles + NT * TILE + warp * PXR * LD;           // DIM * LD, one set per warp (the uniform-grid anchors live here)
  double* noise = px + DIM * LD;
  double* vr = tiles + NT * TILE + WPC * PXR * LD;            // r (becomes z); shared by the warps of the CTA
  constexpr bool PF = TASK == TASK_PREDICT_F || TASK == TASK_PREDICT_FU;      // predict from a stored factor
  constexpr bool UNI = uni64(TASK);                                            // ... on a uniformly spaced shared grid
  constexpr bool FUSED = TASK == TASK_PREDICT || TASK == TASK_PREDICT_U;       // factorise and predict in one pass (no workspace)
  constexpr bool PRED_LIKE = FUSED || TASK == TASK_FACTOR || PF;
  // Prediction needs no L^-1 (round 2): with the accumulator == operand layout the grid phase solves L v = h by block
  // FORWARD SUBSTITUTION on the tensor cores -- V_J = (H_J - sum_{P<J} V_P L[J][P]^T) T_J^T, every V_P fed to the next
  // DMMA straight from its accumulator registers -- at the same DMMA count as a product with L^-1, and the mean is
  // v . z with z = L^-1 r from the likelihood's forward solve (alpha is never formed).  The factorisation of these
  // tasks therefore stops after the Cholesky factor; its off-diagonal tiles are stored NEGATED (the products of the
  // later columns do not notice: (-a)(-b) = ab) so that the grid phase accumulates h + sum V_P (-L)^T directly.
  constexpr bool NEGL = PRED_LIKE;
  double* vz = PRED_LIKE ? vr : vr + LD;                // prediction tasks: z = L^-1 r overwrites r in place (block by block)
  double* va = PRED_LIKE ? vr : vz + LD;
  double* vd = va + LD;
  double* v1 = vd + LD;
  double* vu = v1 + LD;

  // the general-grid prediction from a stored factor never stages the noise vector: at NB = 8 its 64 doubles hold the
  // table of the table-driven exp (cgp_math.cuh) for the cross-covariance entries (one exp per grid point and data point)
  constexpr bool TAB = PF && !UNI && NB == 8 && WPC == 1;
  if (TAB) { exp_table_to_shared(noise, lane); __syncwarp(); }
  constexpr bool KTAB = ktab64(TASK, NB);
  double* const ktab = tiles + NT * TILE + (WPC * PXR + n_vec64(TASK)) * LD;      // behind the last vector
  if (etab64(TASK, NB)) { exp_table_to_shared(ktab, lane); __syncwarp(); }
  const int split = (FUSED || PF) ? a.split : 1;
  const int64_t* const part_off = (FUSED || PF) ? a.part_off : nullptr;
  const int64_t n_work = part_off ? a.n_parts : (a.n_obj_dev ? (int64_t)*a.n_obj_dev : a.n_obj) * split;
  // factor workspace of one object: NT tiles (T_J on the diagonal, -L[I][J] below) followed by z (LD doubles)
  __shared__ __align__(8) unsigned long long s_mbar;       // TMA completion barrier (TASK_PREDICT_F)
  __shared__ long long s_tk[2];                            // WPC > 1: the ticket drawn by thread 0, double buffered
  unsigned mbar_parity = 0;
  if (PF) {
    if (threadIdx.x == 0) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"((unsigned)__cvta_generic_to_shared(&s_mbar)));
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (WPC > 1) __syncthreads(); else __syncwarp();
  }

  // Dynamic work distribution: 11 one-warp CTAs per SM land 3/3/3/2 on the four sub-partitions,
  // so equal static shares would leave the 2-warp partition idle a quarter of the time.
  // Software pipeline over objects: while object i is processed, the inputs of object i+1 are
  // already in flight into registers (HBM latency ~700 cycles would otherwise be exposed per
  // object) and the ticket for object i+2 is being drawn.
  constexpr int NR = (LD + 31) / 32;                     // staged values per lane
  // prediction: the factor kernel's status and the object's offset of the shared mean template come with the inputs
  struct Next { int64_t o0; int n, bad; double ydiff, x[NR], y2[NR], r[NR], ye[NR]; };
  auto fetch = [&](int64_t w, Next& nx) {
    nx.n = -1;
    if (w >= n_work) return;
    int part, parts;
    const int64_t oi = work_item(part_off, a.n_obj, split, w, part, parts);
    const int64_t b = a.order ? a.order[oi] : oi;
    nx.o0 = a.off[b];
    nx.n = (int)(a.off[b + 1] - nx.o0);
    nx.bad = PF ? a.info[b] : 0;
    nx.ydiff = ((FUSED || PF) && a.new_y0 && a.new_y0_diff) ? a.new_y0_diff[b] : 0.0;
#pragma unroll
    for (int k = 0; k < NR; ++k) {
      const int i = k * 32 + lane;
      const bool in = i < nx.n;
      if (DIM == 1) { nx.x[k] = in ? a.x[nx.o0 + i] : 0.0; nx.y2[k] = 0.0; }
      else { nx.x[k] = in ? a.x[2 * (nx.o0 + i)] : 0.0; nx.y2[k] = in ? a.x[2 * (nx.o0 + i) + 1] : 0.0; }
      if (PF) { nx.ye[k] = 0.0; nx.r[k] = 0.0; continue; }
      nx.ye[k] = (in && a.yerr) ? a.yerr[nx.o0 + i] : 0.0;
      nx.r[k] = in ? (a.y[nx.o0 + i] - (a.y0 ? a.y0[nx.o0 + i] : 0.0)) : 0.0;
    }
  };
  // Uniform shared grid (UNI): g_j = g_first + j*delta.  Within a pass of 16 grid rows anchored at row j0,
  //   exp(h00 (g_j0 + k delta - x)^2) = E_a(x) * R(x)^k * C_k,  E_a = exp(h00 u^2), R = exp(2 h00 delta u), u = g_j0 - x,
  // C_k = exp(h00 k^2 delta^2): two exps per object point and pass instead of one per (grid row, object point).
  // The caller guarantees l >= |delta|: whenever E_a underflows every product it scales is < 1e-110.  The substitution
  // runs on H' = E_a R^k and C_k scales its results (k < 24: E_a R^k <= 1 / C_k <= e^264.5, C_k^2 >= e^-529).
  double uni_g0 = 0.0, uni_delta = 0.0, uni_2hd = 0.0;
  double* const uni_c = ktab + 64;                       // C_k, k < 24, behind the exp table (read at the stores only)
  if (UNI) {
    uni_g0 = a.xnew[0];
    uni_delta = (a.xnew[a.m_shared - 1] - uni_g0) / (double)(a.m_shared - 1);
    const double kd = (double)lane * uni_delta;
    if (lane < 24) uni_c[lane] = cgp_exp(cov.h00 * kd * kd);
    uni_2hd = 2.0 * cov.h00 * uni_delta;
    __syncwarp();
  }
  int64_t w = blockIdx.x, w_nxt = (int64_t)blockIdx.x + gridDim.x, t_next = 0;
  int it = 0;
  // next work item: one warp per CTA shuffles it from lane 0; several warps meet at a barrier (which also says that
  // every warp is done with the staged factor of the current object) and read it from shared memory
  auto advance = [&]() -> int64_t {
    if (WPC > 1) { __syncthreads(); return s_tk[(it++) & 1]; }
    return __shfl_sync(FULL, t_next, 0);
  };
  Next nx;
  fetch(w, nx);
  for (;; w = w_nxt, w_nxt = advance()) {
    if (w >= n_work) break;
    if (threadIdx.x == 0) {
      t_next = (int64_t)atomicAdd(ticket, 1ULL) + 2 * (int64_t)gridDim.x;
      if (WPC > 1) s_tk[it & 1] = t_next;
    }
    int part, parts;
    const int64_t oi = work_item(part_off, a.n_obj, split, w, part, parts);
    const int64_t b = a.order ? a.order[oi] : oi;
    const int64_t o0 = nx.o0;
    const int n = nx.n;
    const int64_t io = a.compact_io ? oi : b;
    if (a.hyp_obj) cov = cov_from_hyp(DIM, a.hyp_obj + io * a.n_hyp, a.nugget_obj ? a.nugget_obj[io] : a.nugget_shared,
                                      a.floor_shared, a.flags);

    // ---------------- stage (from the prefetched registers), then start the next object's loads
    __syncwarp();
    double rsum = 0.0;
#pragma unroll
    for (int k = 0; k < NR; ++k) {
      const int i = k * 32 + lane;
      if (i < LD) {
        px[i] = nx.x[k];
        if (DIM == 2) px[LD + i] = nx.y2[k];
        if (!PF) {                                         // PF: z arrives by TMA into vr, nothing else is staged
          noise[i] = nx.ye[k] * nx.ye[k] + cov.noise_const;
          vr[i] = nx.r[k]; rsum += nx.r[k];
        }
      }
    }
    double xo[NR];                                       // UNI: this lane owns columns lane, lane+32
#pragma unroll
    for (int k = 0; k < NR; ++k) xo[k] = UNI ? nx.x[k] : 0.0;
    const double ydiff = nx.ydiff;
    int bad = nx.bad;
    fetch(w_nxt, nx);
    __syncwarp();
    if (TASK == TASK_LOO) rsum = red_g(red_t(rsum));
    double lp_m = 1.0; int lp_e = 0;
    const bool want_u = (TASK == TASK_LOO) && (a.loo_mode == 1);
    if (PF) {
      // factor tiles + z of this object: one TMA bulk copy each, global -> shared, completion on an mbarrier
      const unsigned mb = (unsigned)__cvta_generic_to_shared(&s_mbar);
      if (threadIdx.x == 0) {
        const unsigned bytes = NT * TILE * 8;
        const double* src = a.fws + b * a.fws_stride;
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // earlier generic reads of the buffer are done
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(mb), "r"(bytes + LD * 8) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     :: "r"((unsigned)__cvta_generic_to_shared(tiles)), "l"(src), "r"(bytes), "r"(mb) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     :: "r"((unsigned)__cvta_generic_to_shared(va)), "l"(src + NT * TILE), "r"((unsigned)(LD * 8)), "r"(mb) : "memory");
      }
      unsigned done = 0;
      while (!done) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(mb), "r"(mbar_parity) : "memory");
      }
      mbar_parity ^= 1;
    }
    if (!PF) {

    // ---------------- phase K: covariance tiles, parked in their slots (accumulator values at
    // fragment-order positions).  Two tiles per pass, unrolled twice: 8 exp chains per lane.
    constexpr int TPP = 4;                               // tiles per pass: 16 exp chains per lane in flight
#pragma unroll 1
    for (int q = 0; q < NT; q += TPP) {
      double kv[TPP][2];
#pragma unroll
      for (int u = 0; u < TPP; ++u) {
        const int qq = (q + u < NT) ? q + u : q;
        const int ij = kTri[qq];
        const int I = ij >> 4, J = ij & 15;
        const int gi = 8 * I + L.g, cj = 8 * J + 2 * L.t;
        const double xi = px[gi], yi = DIM == 2 ? px[LD + gi] : 0.0;
        // branch-free: a conditional exp would serialise the chains (ncu r01c: 34 % of the time)
        const double q0 = rbf_arg<DIM>(cov, xi, yi, px[cj], DIM == 2 ? px[LD + cj] : 0.0);
        const double q1 = rbf_arg<DIM>(cov, xi, yi, px[cj + 1], DIM == 2 ? px[LD + cj + 1] : 0.0);
        double e0 = KTAB ? cgp_exp_tab(q0, ktab) : cgp_exp(q0);
        double e1 = KTAB ? cgp_exp_tab(q1, ktab) : cgp_exp(q1);
        e0 = (gi < n && cj < gi) ? e0 : 0.0;
        e1 = (gi < n && cj + 1 < gi) ? e1 : 0.0;
        const double dg = (gi < n) ? cov.amp_auto + noise[gi] : 1.0;
        kv[u][0] = (cj == gi) ? dg : cov.amp_auto * e0;
        kv[u][1] = (cj + 1 == gi) ? dg : cov.amp_auto * e1;
      }
#pragma unroll
      for (int u = 0; u < TPP; ++u) {
        if (q + u < NT) st_frag(tiles, q + u, L, kv[u][0], kv[u][1]);
      }
    }
    __syncwarp();

    // ---------------- phase C: left-looking block Cholesky, column by column (static)
#pragma unroll
    for (int J = 0; J < NB; ++J) {
      double s0[NB], s1[NB], u0[NB], u1[NB];
#pragma unroll
      for (int i = 0; i < NB; ++i) { s0[i] = 0.0; s1[i] = 0.0; u0[i] = 0.0; u1[i] = 0.0; }
#pragma unroll
      for (int P = 0; P < J; ++P) {
        const double2 fb = ld_frag(tiles, slot(J, P), L);
        dmma(s0[0], s1[0], fb.x, fb.x); dmma(u0[0], u1[0], fb.y, fb.y);
#pragma unroll
        for (int i = 1; i < NB - J; ++i) {
          const double2 fa = ld_frag(tiles, slot(J + i, P), L);
          dmma(s0[i], s1[i], fa.x, fb.x); dmma(u0[i], u1[i], fa.y, fb.y);
        }
      }
      // C = K (parked: every lane reads back the unit it wrote) - update
#pragma unroll
      for (int i = 0; i < NB - J; ++i) {
        const double2 kk = ld_frag(tiles, slot(J + i, J), L);
        s0[i] = kk.x - (s0[i] + u0[i]);
        s1[i] = kk.y - (s1[i] + u1[i]);
      }
      double t0, t1;
      {
        double piv; int badk;
        diag_factor(s0[0], s1[0], L, t0, t1, piv, badk);
        st_frag(tiles, slot(J, J), L, t0, t1);
        if (TASK == TASK_LL || TASK == TASK_FACTOR || FUSED) {
          lp_m *= piv;
          const int hi = __double2hiint(lp_m);
          const int e = ((hi >> 20) & 0x7ff) - 1023;
          lp_e += e;
          lp_m = __hiloint2double(hi - (e << 20), __double2loint(lp_m));
        }
        if (badk && bad == 0) bad = 8 * J + badk;
      }
      // L[I][J] = C[I][J] T_J^T: both operands are accumulators of this lane (see the layout note)
#pragma unroll
      for (int i = 1; i < NB - J; ++i) {
        const double c0 = s0[i], c1 = s1[i];
        s0[i] = 0.0; s1[i] = 0.0; u0[i] = 0.0; u1[i] = 0.0;
        dmma(s0[i], s1[i], c0, t0); dmma(u0[i], u1[i], c1, t1);
      }
#pragma unroll
      for (int i = 1; i < NB - J; ++i) {
        if (NEGL) st_frag(tiles, slot(J + i, J), L, -s0[i] - u0[i], -s1[i] - u1[i]);
        else st_frag(tiles, slot(J + i, J), L, s0[i] + u0[i], s1[i] + u1[i]);
      }
      if (NEGL) {
        // z_J = T_J (r_J - sum_{P<J} L[J][P] z_P), in place over r (the tiles hold -L): behind the next column's DMMAs
        double pz = 0.0, pz2 = 0.0;
#pragma unroll
        for (int P = 0; P < J; ++P) {
          const double2 f = ld_frag(tiles, slot(J, P), L);
          const double2 rv = ld_vec2(vr, 8 * P + 2 * L.t);
          pz = fma(f.x, rv.x, pz); pz2 = fma(f.y, rv.y, pz2);
        }
        const double wv = vr[8 * J + L.g] + red_t(pz + pz2);
        double q = t0 * __shfl_sync(FULL, wv, L.t * 8) + t1 * __shfl_sync(FULL, wv, L.t * 8 + 4);
        q = red_t(q);
        if (L.t == 0) vr[8 * J + L.g] = q;
      }
      __syncwarp();
    }

    if (TASK == TASK_LL) {
      // ---------------- z = L^-1 r by block forward substitution, quad = |z|^2
      double quad = 0.0;
#pragma unroll
      for (int J = 0; J < NB; ++J) {
        double p = 0.0, p2 = 0.0;
#pragma unroll
        for (int P = 0; P < J; ++P) {
          const double2 f = ld_frag(tiles, slot(J, P), L);
          const double2 rv = ld_vec2(vr, 8 * P + 2 * L.t);
          p = fma(f.x, rv.x, p); p2 = fma(f.y, rv.y, p2);
        }
        const double wv = vr[8 * J + L.g] - red_t(p + p2);
        const double2 f = ld_frag(tiles, slot(J, J), L);
        double q = f.x * __shfl_sync(FULL, wv, L.t * 8) + f.y * __shfl_sync(FULL, wv, L.t * 8 + 4);
        q = red_t(q);
        if (L.t == 0) { vr[8 * J + L.g] = q; quad = fma(q, q, quad); }
        __syncwarp();
      }
      quad = red_g(red_t(quad));
      if (lane == 0) {
        a.info[io] = bad;
        const double logdet = log(lp_m) + (double)lp_e * LN2;
        a.ll[io] = bad ? nan("") : -0.5 * (quad + logdet + n * LOG_2PI);
      }
      continue;
    }

    if constexpr (TASK == TASK_LOO) {
    // ---------------- L^-1 in place, row by row, held TRANSPOSED while it is built: with Xt[J][I] = (L^-1[I][J])^T
    //   Xt[J][I] = -(sum_{P=J..I-1} Xt[J][P] L[I][P]^T) T_I^T,   Xt[J][J] = T_J^T,
    // every product is of the form X*Y^T on natural fragments and the bracket feeds the second product from its
    // accumulator registers.  Slot (I,J) holds Xt[J][I] until the conversion pass below transposes it in place.
#pragma unroll
    for (int I = 1; I < NB; ++I) {
      double s0[NB], s1[NB];
#pragma unroll
      for (int j = 0; j < NB; ++j) { s0[j] = 0.0; s1[j] = 0.0; }
#pragma unroll
      for (int P = 0; P < I; ++P) {
        const double2 fb = ld_frag(tiles, slot(I, P), L);
#pragma unroll
        for (int J = 0; J <= P; ++J) {
          const double2 fa = (J == P) ? ld_frag_t(tiles, slot(P, P), L) : ld_frag(tiles, slot(P, J), L);
          dmma(s0[J], s1[J], fa.x, fb.x); dmma(s0[J], s1[J], fa.y, fb.y);
        }
      }
      const double2 ft = ld_frag(tiles, slot(I, I), L);
#pragma unroll
      for (int J = 0; J < I; ++J) {
        double r0 = 0.0, r1 = 0.0, e0 = 0.0, e1 = 0.0;
        dmma(r0, r1, s0[J], ft.x); dmma(e0, e1, s1[J], ft.y);
        s0[J] = -(r0 + e0); s1[J] = -(r1 + e1);
      }
#pragma unroll
      for (int J = 0; J < I; ++J) st_frag(tiles, slot(I, J), L, s0[J], s1[J]);
      __syncwarp();
    }
    // conversion: slot (I,J) <- its transpose = L^-1[I][J], row by row (reads cross lanes, writes stay in the lane's unit)
#pragma unroll
    for (int I = 1; I < NB; ++I) {
      double2 v[NB];
#pragma unroll
      for (int J = 0; J < I; ++J) v[J] = ld_frag_t(tiles, slot(I, J), L);
      __syncwarp();
#pragma unroll
      for (int J = 0; J < I; ++J) st_frag(tiles, slot(I, J), L, v[J].x, v[J].y);
    }
    __syncwarp();

    // ---------------- z = L^-1 r (and L^-1 1), alpha = L^-T z, d = colnorm^2(L^-1), u = L^-T L^-1 1
#pragma unroll
    for (int I = 0; I < NB; ++I) {
      double p = 0.0, p2 = 0.0, p1 = 0.0;
#pragma unroll
      for (int J = 0; J <= I; ++J) {
        const double2 f = ld_frag(tiles, slot(I, J), L);
        const double2 rv = ld_vec2(vr, 8 * J + 2 * L.t);
        p = fma(f.x, rv.x, p); p2 = fma(f.y, rv.y, p2);
        if (TASK == TASK_LOO) { p1 += f.x; p1 += f.y; }
      }
      p = red_t(p + p2);
      if (L.t == 0) vz[8 * I + L.g] = p;
      if (TASK == TASK_LOO) { p1 = red_t(p1); if (L.t == 0) v1[8 * I + L.g] = (8 * I + L.g < n) ? p1 : 0.0; }
    }
    __syncwarp();
#pragma unroll
    for (int J = 0; J < NB; ++J) {
      double pa0 = 0.0, pa1 = 0.0, pd0 = 0.0, pd1 = 0.0, pu0 = 0.0, pu1 = 0.0;
#pragma unroll
      for (int I = J; I < NB; ++I) {
        const double2 f = ld_frag(tiles, slot(I, J), L);
        const double zi = vz[8 * I + L.g];
        pa0 = fma(f.x, zi, pa0); pa1 = fma(f.y, zi, pa1);
        if (TASK == TASK_LOO) {
          const bool in = 8 * I + L.g < n;               // identity rows of the padding stay out
          pd0 = in ? fma(f.x, f.x, pd0) : pd0; pd1 = in ? fma(f.y, f.y, pd1) : pd1;
          const double ui = v1[8 * I + L.g];
          pu0 = fma(f.x, ui, pu0); pu1 = fma(f.y, ui, pu1);
        }
      }
      pa0 = red_g(pa0); pa1 = red_g(pa1);
      if (L.g == 0) { va[8 * J + 2 * L.t] = pa0; va[8 * J + 2 * L.t + 1] = pa1; }
      if (TASK == TASK_LOO) {
        pd0 = red_g(pd0); pd1 = red_g(pd1); pu0 = red_g(pu0); pu1 = red_g(pu1);
        if (L.g == 0) {
          vd[8 * J + 2 * L.t] = pd0; vd[8 * J + 2 * L.t + 1] = pd1;
          vu[8 * J + 2 * L.t] = pu0; vu[8 * J + 2 * L.t + 1] = pu1;
        }
      }
    }
    __syncwarp();
    }   // TASK_LOO
    if (lane == 0 && part == 0) a.info[b] = bad;
    }   // !PF

    if (FUSED && a.ll && part == 0) {                    // the likelihood from the same factorisation (z, pivots)
      double quad = 0.0;
#pragma unroll
      for (int i0 = 0; i0 < LD; i0 += 32) { const int i = i0 + lane; if (i < LD) quad = fma(vz[i], vz[i], quad); }
      quad = red_g(red_t(quad));
      if (lane == 0) {
        const double logdet = log(lp_m) + (double)lp_e * LN2;
        a.ll[b] = bad ? nan("") : -0.5 * (quad + logdet + n * LOG_2PI);
      }
      __syncwarp();                                      // z is read before the anchors of the grid phase overwrite it
    }
    if (TASK == TASK_FACTOR) {
      if (a.ll) {                                        // the likelihood comes for free: z and the pivots are here
        double quad = 0.0;
#pragma unroll
        for (int i0 = 0; i0 < LD; i0 += 32) { const int i = i0 + lane; if (i < LD) quad = fma(vz[i], vz[i], quad); }
        quad = red_g(red_t(quad));
        if (lane == 0) {
          const double logdet = log(lp_m) + (double)lp_e * LN2;
          a.ll[b] = bad ? nan("") : -0.5 * (quad + logdet + n * LOG_2PI);
        }
      }
      // ---------------- spill the factor (T_J on the diagonal, -L[I][J] below, then z) for the prediction kernel: 512-byte rows
      double* dst = a.fws + b * a.fws_stride;
#pragma unroll 4
      for (int q = 0; q < NT; ++q)
        reinterpret_cast<double2*>(dst + q * TILE)[lane] = reinterpret_cast<const double2*>(tiles + q * TILE)[lane];
#pragma unroll
      for (int i0 = 0; i0 < LD; i0 += 32) { const int i = i0 + lane; if (i < LD) dst[NT * TILE + i] = va[i]; }
      continue;
    }

    if (TASK == TASK_LOO) {
      const double rho = cov.amp_cross / cov.amp_auto;
      const double amp_star = cov.amp_auto + cov.nugget2;
#pragma unroll
      for (int i0 = 0; i0 < LD; i0 += 32) {
        const int i = i0 + lane;
        if (i < n) {
          const double d = vd[i], r = vr[i];
          const double yv = a.y[o0 + i];
          const double m = a.y0 ? a.y0[o0 + i] : 0.0;
          const double ye = a.yerr ? a.yerr[o0 + i] : 0.0;
          double pr = m + rho * (r - va[i] / d);
          if (want_u) {
            const double delta = (rsum - r) / (double)(n - 1);
            pr += delta - delta * rho * (1.0 - vu[i] / d);
          }
          double pv = fabs(amp_star - rho * rho * (cov.amp_auto + noise[i] - 1.0 / d));
          double res = pr - yv;
          double pl = res / sqrt(ye * ye + pv + cov.nugget2);
          if (bad) { pr = nan(""); pv = pr; res = pr; pl = pr; }
          if (a.pred) a.pred[o0 + i] = pr;
          if (a.pvar) a.pvar[o0 + i] = pv;
          if (a.resid) a.resid[o0 + i] = res;
          if (a.pull) a.pull[o0 + i] = pl;
        }
      }
      continue;
    }

    if (FUSED || PF) {
      // ---------------- U blocks of 8 grid points per pass (CGP64_GRID_U, 1 or 2)
      constexpr int UB = CGP64_GRID_U;                     // blocks per regular pass
      // uniform shared grid, one CTA per object: passes of THREE blocks (and at most two of two) cover the grid exactly, instead
      // of passes of two whose last one runs past the end of the grid (M = 100: 13 blocks = 3 + 3 + 3 + 2 + 2 instead of 7 x 2)
      constexpr bool TAIL3 = UNI && PF && UB == 2 && WPC == 1;
      constexpr int UMAX = TAIL3 ? 3 : UB;
      const int64_t g0 = a.goff ? a.goff[b] : 0;
      const int64_t m_pts = a.goff ? (a.goff[b + 1] - g0) : a.m_shared;
      const int64_t out0 = a.goff ? g0 : b * a.m_shared;
      const int64_t n_rb = (m_pts + 7) >> 3;
      const double amp_star = cov.amp_auto + cov.nugget2;
      double pgx[UMAX], pgy[UMAX], pny0[UMAX];
      auto grid_fetch = [&](int64_t rb) {
#pragma unroll
        for (int u = 0; u < UMAX; ++u) {
          const int64_t m = 8 * (rb + u) + L.g;
          const bool lv = m < m_pts;
          pgx[u] = 0.0; pgy[u] = 0.0;
          if (lv && !UNI) {
            if (DIM == 1) pgx[u] = a.xnew[g0 + m];
            else { pgx[u] = a.xnew[2 * (g0 + m)]; pgy[u] = a.xnew[2 * (g0 + m) + 1]; }
          }
          pny0[u] = (lv && a.new_y0) ? a.new_y0[a.new_y0_diff ? m : out0 + m] : 0.0;     // + ydiff at the store
        }
      };
      const int64_t rb0 = (int64_t)(part * WPC + warp) * UB, rbs = (int64_t)parts * WPC * UB;   // the warps of a CTA alternate over the passes
      grid_fetch(rb0);
      auto pass = [&](auto Uc, const int64_t rb, const int64_t rb_next) {
        constexpr int U = decltype(Uc)::value;
        int64_t mi[U]; bool live[U]; double gx[U], gy[U], ny0[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          mi[u] = 8 * (rb + u) + L.g;
          live[u] = mi[u] < m_pts;
          gx[u] = pgx[u]; gy[u] = pgy[u]; ny0[u] = pny0[u];
        }
        grid_fetch(rb_next);                               // next pass's coordinates, behind this pass's math
        // cross-covariance fragments (no amplitude), generated straight into the accumulators of the forward
        // substitution: lane (g,t) holds H[grid row g][columns 8P+2t, 8P+2t+1] = the start value of W_P
        double acc0[U][NB], acc1[U][NB];
        // the anchors serve 16 grid rows: with one block per pass they are computed for every even block and the odd
        // block that follows reuses them (rows g + 8); blocks that do not follow each other (split > 1) get their own
        const bool second = UNI && (U == 1) && (rbs == 1) && (rb & 1);
        if constexpr (UNI) {
          // the powers of the anchors, computed once per object point by the lane that owns it (the 8 lanes that share
          // a column would otherwise each repeat them): E_a R^g in row g, g < 8, and R^8 in row 8.  With an even NB the
          // odd rows are swizzled by 8 columns so that the 16-byte loads of a quarter warp (rows g, g + 1) hit distinct banks
          double* pw = px;                                     // UNI_ROWS * LD doubles
          constexpr int SWZ = (NB & 1) ? 0 : 8;
          if (!second) {
          __syncwarp();                                        // the previous pass has read its anchors
          const double gj0 = fma((double)(8 * rb), uni_delta, uni_g0);
#pragma unroll
          for (int k = 0; k < NR; ++k) {
            const int c = k * 32 + lane;
            const double uu = gj0 - xo[k];
            double ea = cgp_exp_tab(cov.h00 * uu * uu, ktab), rr = cgp_exp_tab(uni_2hd * uu, ktab);
            // padding columns and underflowed anchors contribute exactly 0 (R = 0 keeps 0 * R^k away from 0 * inf);
            // the consumers below then need no masks: rows past the end of the grid are never stored
            ea = (c < n && ea > 0.0) ? ea : 0.0;
            rr = (ea > 0.0) ? rr : 0.0;
            if (c < LD) {
              const double r2 = rr * rr, r4 = r2 * r2;
              // E_a first: every partial product E_a R^j = exp(h00 (u + j delta)^2) / C_j stays below e^24.5
              const double e1 = ea * rr, e2 = ea * r2, e3 = e1 * r2;
              const double e[8] = {ea, e1, e2, e3, ea * r4, e1 * r4, e2 * r4, e3 * r4};
#pragma unroll
              for (int g = 0; g < 8; ++g) pw[g * LD + (c ^ ((g & 1) * SWZ))] = e[g];
              pw[(UNI_ROWS - 1) * LD + c] = r4 * r4;
            }
          }
          __syncwarp();
          }
#pragma unroll
          for (int P = 0; P < NB; ++P) {
            const int c0 = 8 * P + 2 * L.t;                // this lane's two k-values of block P (see the layout note)
            const double2 r8 = ld_vec2(pw + (UNI_ROWS - 1) * LD, c0);
            const double2 er = ld_vec2(pw + L.g * LD, c0 ^ ((L.g & 1) * SWZ));
            const double t0 = er.x, t1 = er.y;
            // H' = E_a R^k (C_k is applied to the results, see the store): multiplied up in this order nothing overflows
            if constexpr (U >= 2) {
              const double s0 = t0 * r8.x, s1 = t1 * r8.y;
              acc0[0][P] = t0; acc0[1][P] = s0; acc1[0][P] = t1; acc1[1][P] = s1;
              if constexpr (U == 3) { acc0[2][P] = s0 * r8.x; acc1[2][P] = s1 * r8.y; }
            } else {
              acc0[0][P] = second ? t0 * r8.x : t0; acc1[0][P] = second ? t1 * r8.y : t1;
            }
          }
        } else {
#pragma unroll
        for (int P = 0; P < NB; ++P) {
          const int c0 = 8 * P + 2 * L.t, c1 = c0 + 1;
          const double2 xx = ld_vec2(px, c0);
          const double x0 = xx.x, x1 = xx.y;
          double y0c = 0.0, y1c = 0.0;
          if (DIM == 2) { const double2 yy = ld_vec2(px + LD, c0); y0c = yy.x; y1c = yy.y; }
#pragma unroll
          for (int u = 0; u < U; ++u) {
            double e0 = TAB ? cgp_exp_tab(rbf_arg<DIM>(cov, gx[u], gy[u], x0, y0c), noise) : cgp_exp(rbf_arg<DIM>(cov, gx[u], gy[u], x0, y0c));
            double e1 = TAB ? cgp_exp_tab(rbf_arg<DIM>(cov, gx[u], gy[u], x1, y1c), noise) : cgp_exp(rbf_arg<DIM>(cov, gx[u], gy[u], x1, y1c));
            e0 = (live[u] && c0 < n) ? e0 : 0.0;
            e1 = (live[u] && c1 < n) ? e1 : 0.0;
            acc0[u][P] = e0; acc1[u][P] = e1;
          }
        }
        }
        // block forward substitution L v = h on the tensor cores (see the NEGL note): block P is finished by
        // V_P = W_P T_P^T, then added into every later block through the stored -L[J][P]; mean = v . z, var = amp* - |v|^2
        double pm[U], pm2[U], vs[U], vs2[U];
#pragma unroll
        for (int u = 0; u < U; ++u) { pm[u] = 0.0; pm2[u] = 0.0; vs[u] = 0.0; vs2[u] = 0.0; }
#pragma unroll
        for (int P = 0; P < NB; ++P) {
          const double2 ft = ld_frag(tiles, slot(P, P), L);
          const double2 zz = ld_vec2(va, 8 * P + 2 * L.t);
#pragma unroll
          for (int u = 0; u < U; ++u) {
            double v0 = 0.0, v1 = 0.0;
            dmma(v0, v1, acc0[u][P], ft.x); dmma(v0, v1, acc1[u][P], ft.y);
            acc0[u][P] = v0; acc1[u][P] = v1;
            if (TASK == TASK_PREDICT && a.vout && live[u])      // bulk covariance writer: keep v (16 bytes per lane, 64-byte rows per quad)
              *reinterpret_cast<double2*>(a.vout + (out0 + mi[u]) * LD + 8 * P + 2 * L.t) = make_double2(v0, v1);
            pm[u] = fma(v0, zz.x, pm[u]); pm2[u] = fma(v1, zz.y, pm2[u]);
            vs[u] = fma(v0, v0, vs[u]); vs2[u] = fma(v1, v1, vs2[u]);
          }
#pragma unroll
          for (int J = P + 1; J < NB; ++J) {
            const double2 fb = ld_frag(tiles, slot(J, P), L);
#pragma unroll
            for (int u = 0; u < U; ++u) dmma(acc0[u][J], acc1[u][J], acc0[u][P], fb.x);
#pragma unroll
            for (int u = 0; u < U; ++u) dmma(acc0[u][J], acc1[u][J], acc1[u][P], fb.y);
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          double vv = vs[u], vv2 = vs2[u];
          const double pmt = red_t(pm[u] + pm2[u]);
          vv = red_t(vv + vv2);
          if (live[u] && L.t == 0) {
            // UNI: v = C_k v' (k = g + 8u, or g + 8 for the second block of a pair): mean = amp C_k v'.z, var = amp* - (amp C_k)^2 |v'|^2
            const double ac = UNI ? cov.amp_cross * uni_c[L.g + 8 * (second ? 1 : u)] : cov.amp_cross;
            double mean = fma(ac, pmt, a.new_y0_diff ? ny0[u] + ydiff : ny0[u]);
            double var = fma(-ac * ac, vv, amp_star);
            if (bad) { mean = nan(""); var = mean; }
            a.mean[out0 + mi[u]] = mean;
            if (a.var) a.var[out0 + mi[u]] = var;
          }
        }
      };
      if (TAIL3 && rbs == UB) {
        // the whole grid belongs to this warp: cover its n_rb blocks exactly with passes of three (three interleaved
        // substitutions hide each other's dependent DMMA chains better than two, and the anchors and the 36 tile loads
        // of a pass serve 24 rows) and at most two passes of two
        for (int64_t rb = rb0; rb < n_rb;) {
          const int64_t left = n_rb - rb;
          if (left == 1 || left == 2 || left == 4) { pass(std::integral_constant<int, UB>{}, rb, rb + UB); rb += UB; }
          else { pass(std::integral_constant<int, UMAX>{}, rb, rb + UMAX); rb += UMAX; }
        }
      } else {
        for (int64_t rb = rb0; rb < n_rb; rb += rbs) pass(std::integral_constant<int, UB>{}, rb, rb + rbs);
      }
    }
  }
}


// ---------------------------------------------------------------------------------------
// Compact log-likelihood kernel.  The likelihood needs row J of L only until z_J is solved,
// so rows are RETIRED as the factorisation advances and their shared-memory slots are reused
// by later columns: at most (NB-J)(J+1) tiles are live (20 instead of 36 at NB = 8), the
// covariance column is generated in registers right when it is consumed (no parking), and
// 16 warps (4 per sub-partition, balanced) fit on an SM instead of 11.
template <int B, int E, class F>
__device__ __forceinline__ void static_for(F&& f) {
  if constexpr (B < E) { f(std::integral_constant<int, B>{}); static_for<B + 1, E>(f); }
}

// kPhys[NB-1][I][P]: shared-memory slot of tile (I,P) when rows are retired after their solve
// (first-free allocation, generated by the simulation in the comment of gp64_ll_kernel)
constexpr int kPhys[8][8][8] = {
    {{0, 0, 0, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0}},
    {{0, 0, 0, 0, 0, 0, 0, 0}, {1, 0, 0, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0}},
    {{0, 0, 0, 0, 0, 0, 0, 0}, {1, 0, 0, 0, 0, 0, 0, 0}, {2, 3, 0, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0}},
    {{0, 0, 0, 0, 0, 0, 0, 0}, {1, 0, 0, 0, 0, 0, 0, 0}, {2, 4, 0, 0, 0, 0, 0, 0}, {3, 5, 1, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0}},
    {{0, 0, 0, 0, 0, 0, 0, 0}, {1, 0, 0, 0, 0, 0, 0, 0}, {2, 5, 0, 0, 0, 0, 0, 0}, {3, 6, 1, 0, 0, 0, 0, 0}, {4, 7, 8, 2, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0}},
    {{0, 0, 0, 0, 0, 0, 0, 0}, {1, 0, 0, 0, 0, 0, 0, 0}, {2, 6, 0, 0, 0, 0, 0, 0}, {3, 7, 1, 0, 0, 0, 0, 0}, {4, 8, 10, 2, 0, 0, 0, 0}, {5, 9, 11, 6, 1, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0}},
    {{0, 0, 0, 0, 0, 0, 0, 0}, {1, 0, 0, 0, 0, 0, 0, 0}, {2, 7, 0, 0, 0, 0, 0, 0}, {3, 8, 1, 0, 0, 0, 0, 0}, {4, 9, 12, 2, 0, 0, 0, 0}, {5, 10, 13, 7, 1, 0, 0, 0}, {6, 11, 14, 15, 3, 2, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0}},
    {{0, 0, 0, 0, 0, 0, 0, 0}, {1, 0, 0, 0, 0, 0, 0, 0}, {2, 8, 0, 0, 0, 0, 0, 0}, {3, 9, 1, 0, 0, 0, 0, 0}, {4, 10, 14, 2, 0, 0, 0, 0}, {5, 11, 15, 8, 1, 0, 0, 0}, {6, 12, 16, 18, 3, 2, 0, 0}, {7, 13, 17, 19, 9, 4, 1, 0}}};
constexpr int kPhysSlots[8] = {1, 2, 4, 6, 9, 12, 16, 20};

template <int DIM, int NB>
__global__ void __launch_bounds__(32, 16)
gp64_ll_kernel(const SmallArgs a, unsigned long long* __restrict__ ticket) {
  extern __shared__ __align__(16) double smem[];
  const int lane = threadIdx.x;
  const Lane L(lane);
  Cov cov = a.cov;
  constexpr int LD = 8 * NB;
  constexpr int NSLOT = kPhysSlots[NB - 1];
  double* tiles = smem;
  double* px = tiles + NSLOT * TILE;
  double* noise = px + DIM * LD;
  double* vr = noise + LD;
  double* etab = vr + LD;                                 // 2^(j/64) for the table-driven exp (cgp_math.cuh)
  exp_table_to_shared(etab, lane);
  __syncwarp();
  const int64_t n_work = a.n_obj_dev ? (int64_t)*a.n_obj_dev : a.n_obj;

  constexpr int NR = (LD + 31) / 32;
  struct Next { int64_t b, io; int n; double x[NR], y2[NR], r[NR], ye[NR]; };
  auto fetch = [&](int64_t w, Next& nx) {
    nx.n = -1; nx.b = 0; nx.io = 0;
    if (w >= n_work) return;
    nx.b = a.order ? a.order[w] : w;
    nx.io = a.compact_io ? w : nx.b;
    const int64_t o0 = a.off[nx.b];
    nx.n = (int)(a.off[nx.b + 1] - o0);
#pragma unroll
    for (int k = 0; k < NR; ++k) {
      const int i = k * 32 + lane;
      const bool in = i < nx.n;
      if (DIM == 1) { nx.x[k] = in ? a.x[o0 + i] : 0.0; nx.y2[k] = 0.0; }
      else { nx.x[k] = in ? a.x[2 * (o0 + i)] : 0.0; nx.y2[k] = in ? a.x[2 * (o0 + i) + 1] : 0.0; }
      nx.ye[k] = (in && a.yerr) ? a.yerr[o0 + i] : 0.0;
      nx.r[k] = in ? (a.y[o0 + i] - (a.y0 ? a.y0[o0 + i] : 0.0)) : 0.0;
    }
  };
  int64_t w = blockIdx.x, w_nxt = (int64_t)blockIdx.x + gridDim.x, t_next = 0;
  Next nx;
  fetch(w, nx);
  for (;; w = w_nxt, w_nxt = __shfl_sync(FULL, t_next, 0)) {
    if (w >= n_work) break;
    if (lane == 0) t_next = (int64_t)atomicAdd(ticket, 1ULL) + 2 * (int64_t)gridDim.x;
    const int64_t io = nx.io, nx_b = nx.b;
    const int n = nx.n;
    if (a.hyp_obj) cov = cov_from_hyp(DIM, a.hyp_obj + io * a.n_hyp, a.nugget_obj ? a.nugget_obj[io] : a.nugget_shared,
                                      a.floor_shared, a.flags);
    __syncwarp();
#pragma unroll
    for (int k = 0; k < NR; ++k) {
      const int i = k * 32 + lane;
      if (i < LD) {
        px[i] = nx.x[k];
        if (DIM == 2) px[LD + i] = nx.y2[k];
        noise[i] = nx.ye[k] * nx.ye[k] + cov.noise_const;
        vr[i] = nx.r[k];
      }
    }
    fetch(w_nxt, nx);
    __syncwarp();

    double lp_m = 1.0, quad = 0.0; int lp_e = 0; int bad = 0;
    constexpr int NTF = NB * (NB + 1) / 2;
    double* const fdst = a.fws ? a.fws + nx_b * a.fws_stride : nullptr;    // TASK_FACTOR served by this kernel
    static_for<0, NB>([&](auto Jc) {
      constexpr int J = decltype(Jc)::value;
      constexpr int NTJ = NB - J;
      // covariance column J, straight into accumulator layout (2 NTJ independent exp chains)
      double k0[NTJ], k1[NTJ];
      static_for<0, NTJ>([&](auto ic) {
        constexpr int i = decltype(ic)::value;
        const int gi = 8 * (J + i) + L.g, cj = 8 * J + 2 * L.t;
        const double xi = px[gi], yi = DIM == 2 ? px[LD + gi] : 0.0;
        double e0 = cgp_exp_tab(rbf_arg<DIM>(cov, xi, yi, px[cj], DIM == 2 ? px[LD + cj] : 0.0), etab);
        double e1 = cgp_exp_tab(rbf_arg<DIM>(cov, xi, yi, px[cj + 1], DIM == 2 ? px[LD + cj + 1] : 0.0), etab);
        e0 = (gi < n && cj < gi) ? e0 : 0.0;
        e1 = (gi < n && cj + 1 < gi) ? e1 : 0.0;
        const double dg = (gi < n) ? cov.amp_auto + noise[gi] : 1.0;
        k0[i] = (i == 0 && cj == gi) ? dg : cov.amp_auto * e0;
        k1[i] = (i == 0 && cj + 1 == gi) ? dg : cov.amp_auto * e1;
      });
      // rank-8J update of the whole column: 2 NTJ independent DMMA chains
      double s0[NTJ], s1[NTJ], u0[NTJ], u1[NTJ];
      static_for<0, NTJ>([&](auto ic) { constexpr int i = decltype(ic)::value; s0[i] = 0.0; s1[i] = 0.0; u0[i] = 0.0; u1[i] = 0.0; });
      static_for<0, J>([&](auto Pc) {
        constexpr int P = decltype(Pc)::value;
        const double2 fb = ld_frag(tiles, kPhys[NB - 1][J][P], L);
        dmma(s0[0], s1[0], fb.x, fb.x); dmma(u0[0], u1[0], fb.y, fb.y);
        static_for<1, NTJ>([&](auto ic) {
          constexpr int i = decltype(ic)::value;
          const double2 fa = ld_frag(tiles, kPhys[NB - 1][J + i][P], L);
          dmma(s0[i], s1[i], fa.x, fb.x); dmma(u0[i], u1[i], fa.y, fb.y);
        });
      });
      static_for<0, NTJ>([&](auto ic) {
        constexpr int i = decltype(ic)::value;
        s0[i] = k0[i] - (s0[i] + u0[i]); s1[i] = k1[i] - (s1[i] + u1[i]);
      });
      double t0, t1;                                    // T_J = L_JJ^-1 stays in registers: both its uses take it from there
      {
        double piv; int badk;
        diag_factor(s0[0], s1[0], L, t0, t1, piv, badk);
        lp_m *= piv;
        const int hi = __double2hiint(lp_m);
        const int e = ((hi >> 20) & 0x7ff) - 1023;
        lp_e += e;
        lp_m = __hiloint2double(hi - (e << 20), __double2loint(lp_m));
        if (badk && bad == 0) bad = 8 * J + badk;
      }
      if constexpr (NTJ > 1) {
        static_for<1, NTJ>([&](auto ic) {               // L[I][J] = C[I][J] T_J^T, operands = accumulators (layout note)
          constexpr int i = decltype(ic)::value;
          const double c0 = s0[i], c1 = s1[i];
          s0[i] = 0.0; s1[i] = 0.0; u0[i] = 0.0; u1[i] = 0.0;
          dmma(s0[i], s1[i], c0, t0); dmma(u0[i], u1[i], c1, t1);
        });
        static_for<1, NTJ>([&](auto ic) {
          constexpr int i = decltype(ic)::value;
          constexpr int ps = kPhys[NB - 1][J + i][J];
          st_frag(tiles, ps, L, s0[i] + u0[i], s1[i] + u1[i]);
        });
      }
      // z_J = T_J (r_J - sum_{P<J} L[J][P] z_P); afterwards row J is dead and its slots are reused
      double pz = 0.0, pz2 = 0.0;
      static_for<0, J>([&](auto Pc) {
        constexpr int P = decltype(Pc)::value;
        const double2 f = ld_frag(tiles, kPhys[NB - 1][J][P], L);
        const double2 rv = ld_vec2(vr, 8 * P + 2 * L.t);
        pz = fma(f.x, rv.x, pz); pz2 = fma(f.y, rv.y, pz2);
        // factor-once / predict-many: the retiring row leaves for the workspace of the grid kernel (-L[J][P]: see
        // the NEGL note of gp64_kernel); every lane moves the 16-byte unit it owns, 512 contiguous bytes per tile
        if (fdst) *reinterpret_cast<double2*>(fdst + slot(J, P) * TILE + L.nat) = make_double2(-f.x, -f.y);
      });
      if (fdst) *reinterpret_cast<double2*>(fdst + slot(J, J) * TILE + L.nat) = make_double2(t0, t1);
      const double wv = vr[8 * J + L.g] - red_t(pz + pz2);
      double q = t0 * __shfl_sync(FULL, wv, L.t * 8) + t1 * __shfl_sync(FULL, wv, L.t * 8 + 4);
      q = red_t(q);
      if (L.t == 0) { vr[8 * J + L.g] = q; quad = fma(q, q, quad); }
      __syncwarp();
    });
    quad = red_g(red_t(quad));
    if (fdst) {                                           // z = L^-1 r behind the tiles
#pragma unroll
      for (int i0 = 0; i0 < LD; i0 += 32) { const int i = i0 + lane; if (i < LD) fdst[NTF * TILE + i] = vr[i]; }
    }
    if (lane == 0) {
      a.info[io] = bad;
      const double logdet = log(lp_m) + (double)lp_e * LN2;
      if (a.ll) a.ll[io] = bad ? nan("") : -0.5 * (quad + logdet + n * LOG_2PI);
    }
  }
}


template <int DIM, int NB>
int launch64_ll(const SmallArgs& a, cudaStream_t stream) {
  auto kern = gp64_ll_kernel<DIM, NB>;
  const size_t smem = ((size_t)kPhysSlots[NB - 1] * TILE + (size_t)(DIM + 2) * 8 * NB + 64) * sizeof(double);   // + the exp table
  static int sm_counts[16] = {0}, per_sms[16] = {0};   // per device of this process (function attributes are per device)
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 16) return (int)cudaErrorInvalidDevice;
  int& sm_count = sm_counts[dev]; int& per_sm = per_sms[dev];
  if (!sm_count) cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev);
  if (!per_sm) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    int occ = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, 32, smem);
    if (e != cudaSuccess) return (int)e;
    if (occ < 1) return (int)cudaErrorInvalidConfiguration;
    per_sm = occ > 16 ? 16 : occ;                        // 4 warps per sub-partition
  }
  static int cap = -1;
  if (cap < 0) { const char* e = getenv("CGP_GP64_PER_SM"); cap = e ? atoi(e) : 0; }
  int64_t grid = (int64_t)sm_count * ((cap > 0 && cap < per_sm) ? cap : per_sm);
  if (grid > a.n_obj) grid = a.n_obj;
  if (grid < 1) return 0;
  unsigned long long* ticket = next_ticket(stream);
  if (!ticket) return (int)cudaErrorMemoryAllocation;
  kern<<<(unsigned)grid, 32, smem, stream>>>(a, ticket);
  count_launch();
  return (int)cudaGetLastError();
}

template <int DIM, int TASK, int NB>
int launch64(const SmallArgs& a, cudaStream_t stream) {
  static int compact = -1;                                // CGP_LL_COMPACT=0 falls back to the 36-slot kernel
  if (compact < 0) { const char* e = getenv("CGP_LL_COMPACT"); compact = (e && !atoi(e)) ? 0 : 1; }
  // TASK_FACTOR = the compact likelihood kernel with a workspace: rows are written out as they retire, so the factor
  // kernel keeps the 16 warps per SM of the likelihood kernel instead of 11 (CGP_FACTOR_COMPACT=0: the 36-slot kernel)
  static int fcompact = -1;
  if (fcompact < 0) { const char* e = getenv("CGP_FACTOR_COMPACT"); fcompact = (e && !atoi(e)) ? 0 : 1; }
  if ((TASK == TASK_LL && compact) || (TASK == TASK_FACTOR && fcompact)) return launch64_ll<DIM, NB>(a, stream);
  auto kern = gp64_kernel<DIM, TASK, NB>;
  constexpr int WPC = warps_per_cta(TASK);
  const size_t smem = ((size_t)(NB * (NB + 1) / 2) * TILE + (size_t)(WPC * px_rows64(TASK, DIM) + n_vec64(TASK)) * 8 * NB
                       + (etab64(TASK, NB) ? 64 : 0) + (uni64(TASK) ? 24 : 0)) * sizeof(double);
  static int sm_counts[16] = {0}, per_sms[16] = {0};   // per device of this process
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 16) return (int)cudaErrorInvalidDevice;
  int& sm_count = sm_counts[dev]; int& per_sm = per_sms[dev];
  if (!sm_count) cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev);
  if (!per_sm) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    int occ = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, 32 * WPC, smem);
    if (e != cudaSuccess) return (int)e;
    if (occ < 1) return (int)cudaErrorInvalidConfiguration;
    per_sm = occ;
  }
  constexpr bool GRID_TASK = TASK == TASK_PREDICT || TASK == TASK_PREDICT_F || TASK == TASK_PREDICT_FU || TASK == TASK_PREDICT_U;
  const int64_t n_work = !GRID_TASK ? a.n_obj : a.part_off ? a.n_parts : a.n_obj * a.split;
  static int cap = -1;                                    // experiment knob: CGP_GP64_PER_SM=<blocks per SM>
  if (cap < 0) { const char* e = getenv("CGP_GP64_PER_SM"); cap = e ? atoi(e) : 0; }
  int64_t grid = (int64_t)sm_count * ((cap > 0 && cap < per_sm) ? cap : per_sm);
  if (grid > n_work) grid = n_work;
  if (grid < 1) return 0;
  unsigned long long* ticket = next_ticket(stream);
  if (!ticket) return (int)cudaErrorMemoryAllocation;
  kern<<<(unsigned)grid, 32 * WPC, smem, stream>>>(a, ticket);
  count_launch();
  return (int)cudaGetLastError();
}

template <int DIM, int TASK>
int launch64_nb(int nb, const SmallArgs& a, cudaStream_t stream) {
  switch (nb) {
    case 1: return launch64<DIM, TASK, 1>(a, stream);
    case 2: return launch64<DIM, TASK, 2>(a, stream);
    case 3: return launch64<DIM, TASK, 3>(a, stream);
    case 4: return launch64<DIM, TASK, 4>(a, stream);
    case 5: return launch64<DIM, TASK, 5>(a, stream);
    case 6: return launch64<DIM, TASK, 6>(a, stream);
    case 7: return launch64<DIM, TASK, 7>(a, stream);
    case 8: return launch64<DIM, TASK, 8>(a, stream);
  }
  return (int)cudaErrorInvalidValue;
}

}  // namespace

// One (DIM, TASK) pair per translation unit (build.py compiles this file eleven times with
// -DCGP64_DIM / -DCGP64_TASK) so the 88 static instantiations build in parallel.
#ifndef CGP64_DIM
#error "compile with -DCGP64_DIM=1|2 -DCGP64_TASK=0|1|2|4|5|6|7"
#endif
#define CGP64_CAT2(a, b, c, d) a##b##c##d
#define CGP64_CAT(a, b, c, d) CGP64_CAT2(a, b, c, d)
int CGP64_CAT(launch_small64_d, CGP64_DIM, _t, CGP64_TASK)(int nb, const SmallArgs& a, cudaStream_t stream) {
  return launch64_nb<CGP64_DIM, CGP64_TASK>(nb, a, stream);
}

}  // namespace cgp
