// Small-object Gaussian-process kernels for B200 (sm_100a): objects of N <= 224 points,
// one warp (N <= 64) or one 4-warp CTA per object, everything resident in shared memory.
//
// What one object costs the reference (citations into PFLeget/cosmogp):
//   K = kernel(x, hyp, nugget, y_err)          cosmogp/kernel.py:25-77 / 80-155
//   inv, logdet = cholesky_inverse(K)          cosmogp/inv_matrix.py:21-31
//   LL (Gaussian_process.py:68-73), mean / covariance (:332-335, :356-361),
//   leave-one-out pulls (pull.py:66-94)
// Here K is never written to HBM.  It is generated tile by tile (8x8) straight into
// DMMA accumulator registers, factorised by a left-looking block Cholesky whose
// rank-8 updates, triangular solves, L^-1 and L^-1-applications all run on the FP64
// tensor pipe (mma.sync.m8n8k4.f64 -> SASS DMMA.8x8x4), and consumed in place.
//
// Tile storage (the layout of cgp_small64.cu, see its header): element (r, c) of an 8x8 tile lives in 16-byte unit
//   rho(r)*4 + ((c>>1) ^ sigma(r)), half c&1,   rho(r) = r ^ ((r>>1)&1), sigma(r) = (r>>1)&2
// so that lane (g = lane/4, t = lane%4) finds its DMMA accumulator pair {tile[g][2t], tile[g][2t+1]} -- which is also its
// operand of both k-halves of a product X*Y^T (the two DMMAs sum over the even and the odd k) -- in ONE conflict-free
// 16-byte unit, and the transposed fragment {tile[2t][g], tile[2t+1][g]} with two conflict-free 8-byte loads.  With the
// m8n8k4 layouts (A[g][k], B[k][g], C[g][2t..2t+1]) this gives all three products the algorithm needs,
//   X*Y^T (frag, frag)   X*Y (frag, fragT)   X^T*Y (fragT, fragT),
// and lets a tile that was just accumulated feed the next DMMA straight from its registers.
#include <type_traits>
#include "cgp_internal.h"
#include "cgp_math.cuh"

#pragma nv_diag_suppress 128      // TASK_PREDICT leaves the object loop before the L^-1 phase: "loop is not reachable" there

#include <math.h>
#include <stdio.h>
#include <stdlib.h>

namespace cgp {
namespace {

constexpr int TILE = 64;                      // doubles per 8x8 tile
constexpr unsigned FULL = 0xffffffffu;
constexpr double LOG_2PI = 1.8378770664093454835606594728112;

__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
      : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

__device__ __forceinline__ int slot(int i, int j) { return ((i * (i + 1)) >> 1) + j; }   // i >= j
__host__ __device__ __forceinline__ int frag_off(int r, int c) {
  const int rho = r ^ ((r >> 1) & 1), sig = (r >> 1) & 2;
  return ((rho * 4 + ((c >> 1) ^ sig)) << 1) + (c & 1);
}

struct Lane {
  int g, t;
  int fr;          // this lane's 16-byte unit: elements (g,2t), (g,2t+1) = accumulator pair = operand fragment
  int tr0, tr1;    // transposed fragment: (2t,g), (2t+1,g)
  __device__ explicit Lane(int lane) {
    g = lane >> 2; t = lane & 3; fr = frag_off(g, 2 * t);
    tr0 = frag_off(2 * t, g); tr1 = frag_off(2 * t + 1, g);
  }
};

__device__ __forceinline__ double2 ld_frag(const double* tiles, int s, const Lane& L) {
  return *reinterpret_cast<const double2*>(tiles + s * TILE + L.fr);
}
__device__ __forceinline__ double2 ld_fragT(const double* tiles, int s, const Lane& L) {
  const double* p = tiles + s * TILE;
  return make_double2(p[L.tr0], p[L.tr1]);
}
__device__ __forceinline__ void st_acc(double* tiles, int s, const Lane& L, double c0, double c1) {
  *reinterpret_cast<double2*>(tiles + s * TILE + L.fr) = make_double2(c0, c1);
}
__device__ __forceinline__ double red_t(double v) {     // sum over the 4 lanes of a row group
  v += __shfl_xor_sync(FULL, v, 1); v += __shfl_xor_sync(FULL, v, 2); return v;
}
__device__ __forceinline__ double red_g(double v) {     // sum over the 8 row groups
  v += __shfl_xor_sync(FULL, v, 4); v += __shfl_xor_sync(FULL, v, 8); v += __shfl_xor_sync(FULL, v, 16);
  return v;
}
__device__ __forceinline__ double red_warp(double v) { return red_g(red_t(v)); }

// f(integral_constant<int, I>) for I = BEGIN .. END-1, unrolled by the template machinery
template <int BEGIN, int END, class F>
__device__ __forceinline__ void static_for(F&& f) {
  if constexpr (BEGIN < END) {
    f(std::integral_constant<int, BEGIN>{});
    static_for<BEGIN + 1, END>(f);
  }
}

template <int WARPS> __device__ __forceinline__ void cta_sync() {
  if (WARPS == 1) __syncwarp(); else __syncthreads();
}

// RBF exponent -q/2 (<= 0): 1D -(a-b)^2/(2 l^2); 2D Mahalanobis form under the inverse
// metric.  Cov carries the metric pre-multiplied by -1/2, so this is 3 (1D) / 7 (2D) FP64 ops.
template <int DIM>
__device__ __forceinline__ double rbf_arg(const Cov& c, double ax, double ay, double bx, double by) {
  const double dx = ax - bx;
  if (DIM == 1) return dx * dx * c.h00;
  const double dy = ay - by;
  const double u = fma(dx, c.h00, dy * c.h01);
  return fma(dy * c.h11, dy, u * dx);
}

// In-register Cholesky of one 8x8 diagonal tile held in accumulator layout (lower
// triangle valid), returning T = L^-1 in the same layout, the product of the pivots
// (= prod L_kk^2) and the first non-positive pivot (1-based, 0 = none).
// Right-looking: the row operations that reduce A to I are applied to an identity.
__device__ __forceinline__ void diag_factor(double a0, double a1, const Lane& L,
                                            double& t0, double& t1, double& pivprod, int& badk) {
  t0 = (L.g == 2 * L.t) ? 1.0 : 0.0;
  t1 = (L.g == 2 * L.t + 1) ? 1.0 : 0.0;
  pivprod = 1.0; badk = 0;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int kc = k >> 1;
    const double ak = (k & 1) ? a1 : a0;                            // A[g][k] on lanes with t == kc
    const double d = __shfl_sync(FULL, ak, k * 4 + kc);             // pivot
    if (!(d > 0.0) && badk == 0) badk = k + 1;
    const double rinv = cgp_rsqrt(d);
    pivprod *= d;
    const double lg = __shfl_sync(FULL, ak, L.g * 4 + kc) * rinv;            // L[g][k]
    const double lc0 = __shfl_sync(FULL, ak, (2 * L.t) * 4 + kc) * rinv;     // L[2t][k]
    const double lc1 = __shfl_sync(FULL, ak, (2 * L.t + 1) * 4 + kc) * rinv; // L[2t+1][k]
    a0 = fma(-lg, lc0, a0); a1 = fma(-lg, lc1, a1);
    const double tk0 = __shfl_sync(FULL, t0, k * 4 + L.t) * rinv;   // row k of T, scaled
    const double tk1 = __shfl_sync(FULL, t1, k * 4 + L.t) * rinv;
    // branch-free row operation on T: rows above k keep their value (coefficient 0), row k takes the
    // scaled pivot row (ncu r01f: the branchy form cost 544 register moves per object)
    const double f = (L.g > k) ? lg : 0.0;
    const double n0 = fma(-f, tk0, t0), n1 = fma(-f, tk1, t1);
    t0 = (L.g == k) ? tk0 : n0; t1 = (L.g == k) ? tk1 : n1;
  }
}

template <int TASK> __host__ __device__ constexpr int n_vec() {
  return TASK == TASK_LL ? 1 : (TASK == TASK_PREDICT ? 3 : (TASK == TASK_LOO ? 6 : 0));
}

// ---------------------------------------------------------------------------------------
// Covariance entry e = exp(-q/2) between staged points i and j (amplitude applied by the caller).
template <int DIM>
__device__ __forceinline__ double cov_e(const Cov& c, const double* px, int ld, int i, int j) {
  return cgp_exp(rbf_arg<DIM>(c, px[i], DIM == 2 ? px[ld + i] : 0.0, px[j], DIM == 2 ? px[ld + j] : 0.0));
}

// K tile (I,J) minus the accumulated update s, in accumulator layout.  Rows/cols >= n pad
// with the identity; the strict upper triangle of a diagonal tile is never read.
template <int DIM>
__device__ __forceinline__ void k_tile_minus(const Cov& cov, const double* px, const double* noise, int ld, int n,
                                             int I, int J, const Lane& L, double s0, double s1,
                                             double& k0, double& k1, const double* amat = nullptr, int64_t lda = 0) {
  const int gi = 8 * I + L.g, cj = 8 * J + 2 * L.t;
  if (amat) {                                             // covariance supplied in HBM (lower triangle)
    k0 = -s0; k1 = -s1;
    if (gi < n && cj <= gi) k0 += amat[(int64_t)gi * lda + cj];
    if (gi < n && cj + 1 <= gi) k1 += amat[(int64_t)gi * lda + cj + 1];
    if (gi >= n && cj == gi) k0 = 1.0 - s0;
    if (gi >= n && cj + 1 == gi) k1 = 1.0 - s1;
    return;
  }
  // branch-free (a conditional exp serialises the two chains); indices are always inside the staged arrays
  double e0 = cov_e<DIM>(cov, px, ld, gi, cj);
  double e1 = cov_e<DIM>(cov, px, ld, gi, cj + 1);
  e0 = (gi < n && cj < gi) ? e0 : 0.0;
  e1 = (gi < n && cj + 1 < gi) ? e1 : 0.0;
  k0 = fma(cov.amp_auto, e0, -s0);
  k1 = fma(cov.amp_auto, e1, -s1);
  const double dg = (gi < n) ? cov.amp_auto + noise[gi] : 1.0;
  if (cj == gi) k0 = dg - s0;
  if (cj + 1 == gi) k1 = dg - s1;
}

// The tiles (I,J) and (I2,J), I2 > I >= J, of one block column at once: the four exp chains of a lane sit in one
// straight line and interleave (two calls of k_tile_minus are separated by its branch on `amat`).  (I2,J) is never diagonal.
template <int DIM>
__device__ __forceinline__ void k_tile2_minus(const Cov& cov, const double* px, const double* noise, int ld, int n,
                                              int I, int I2, int J, const Lane& L, double s0, double s1, double u0, double u1,
                                              double& k0, double& k1, double& m0, double& m1,
                                              const double* amat = nullptr, int64_t lda = 0) {
  if (amat) {
    k_tile_minus<DIM>(cov, px, noise, ld, n, I, J, L, s0, s1, k0, k1, amat, lda);
    k_tile_minus<DIM>(cov, px, noise, ld, n, I2, J, L, u0, u1, m0, m1, amat, lda);
    return;
  }
  const int gi = 8 * I + L.g, gi2 = 8 * I2 + L.g, cj = 8 * J + 2 * L.t;
  double e0 = cov_e<DIM>(cov, px, ld, gi, cj);
  double e1 = cov_e<DIM>(cov, px, ld, gi, cj + 1);
  double f0 = cov_e<DIM>(cov, px, ld, gi2, cj);
  double f1 = cov_e<DIM>(cov, px, ld, gi2, cj + 1);
  e0 = (gi < n && cj < gi) ? e0 : 0.0;
  e1 = (gi < n && cj + 1 < gi) ? e1 : 0.0;
  f0 = (gi2 < n) ? f0 : 0.0;                              // cj + 1 < 8 (J + 1) <= 8 I2 <= gi2
  f1 = (gi2 < n) ? f1 : 0.0;
  k0 = fma(cov.amp_auto, e0, -s0);
  k1 = fma(cov.amp_auto, e1, -s1);
  m0 = fma(cov.amp_auto, f0, -u0);
  m1 = fma(cov.amp_auto, f1, -u1);
  const double dg = (gi < n) ? cov.amp_auto + noise[gi] : 1.0;
  if (cj == gi) k0 = dg - s0;
  if (cj + 1 == gi) k1 = dg - s1;
}

template <int DIM, int TASK, int NB_MAX, int WARPS, bool FWD_BIG = false>
__global__ void __launch_bounds__(WARPS * 32)
small_gp_kernel(const SmallArgs a, const int nbm, const int mode) {
  extern __shared__ __align__(16) double smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const Lane L(lane);
  Cov cov = a.cov;
  constexpr int NT = WARPS * 32;
  constexpr int KMAX = (NB_MAX - 1 + WARPS - 1) / WARPS;   // L^-1 row: tiles per warp
  // Prediction by block forward substitution (no L^-1, see below).  FWD_BIG selects it above 128 points as well (eight
  // warps, one object per SM; N = 224: 6.4 ms against 8.6 ms through an explicit L^-1 -- once the 406-tile triangle is
  // unrolled by template recursion; left to the loop unroller its accumulators went to local memory: 21 ms).  The
  // L^-1 product of the grid phase further down remains for CGP_BIG_FWD=0 and CGP_BIG_WARPS=4.
  constexpr bool FWD = (TASK == TASK_PREDICT) && (NB_MAX <= 16 || FWD_BIG);

  const int ld = 8 * nbm;
  double* tiles = smem;                                   // nbm(nbm+1)/2 tiles
  double* px = tiles + ((nbm * (nbm + 1)) >> 1) * TILE;   // coordinates, DIM * ld
  double* noise = px + DIM * ld;                          // y_err^2 + floor^2 + nugget^2
  double* vr = noise + ld;                                // r = y - y0  (LL: overwritten by z)
  double* vz = vr + ld;                                   // z = L^-1 r
  double* va = vz + ld;                                   // alpha = K^-1 r
  double* vd = va + ld;                                   // diag(K^-1)
  double* v1 = vd + ld;                                   // L^-1 1
  double* vu = v1 + ld;                                   // K^-1 1
  __shared__ double s_rsum, s_quad;
  __shared__ int s_bad;

  const int split = (TASK == TASK_PREDICT) ? a.split : 1;
  const int64_t* const part_off = (TASK == TASK_PREDICT) ? a.part_off : nullptr;
  const int64_t n_work = part_off ? a.n_parts : (a.n_obj_dev ? (int64_t)*a.n_obj_dev : a.n_obj) * split;

  for (int64_t w = blockIdx.x; w < n_work; w += gridDim.x) {
    int part, parts;
    const int64_t oi = work_item(part_off, a.n_obj, split, w, part, parts);
    const int64_t b = a.order ? a.order[oi] : oi;
    const int64_t o0 = a.off[b];
    const int n = (int)(a.off[b + 1] - o0);
    const int nb = (n + 7) >> 3;
    const double* amat = a.amat ? a.amat + a.aoff[b] : nullptr;
    const int64_t lda = (TASK == TASK_MATRICES && a.ld_obj) ? a.ld_obj[b] : a.lda;
    const int64_t io = a.compact_io ? oi : b;
    if (a.hyp_obj) cov = cov_from_hyp(DIM, a.hyp_obj + io * a.n_hyp, a.nugget_obj ? a.nugget_obj[io] : a.nugget_shared,
                                      a.floor_shared, a.flags);

    // ---------------- stage the object
    cta_sync<WARPS>();                                    // previous object fully consumed
    double rsum = 0.0;
    for (int i = tid; i < 8 * nb; i += NT) {
      const bool in = i < n;
      if (!amat) {
        if (DIM == 1) {
          px[i] = in ? a.x[o0 + i] : 0.0;
        } else {
          px[i] = in ? a.x[2 * (o0 + i)] : 0.0;
          px[ld + i] = in ? a.x[2 * (o0 + i) + 1] : 0.0;
        }
      }
      const double ye = (in && a.yerr) ? a.yerr[o0 + i] : 0.0;
      noise[i] = ye * ye + cov.noise_const;
      if (TASK != TASK_MATRICES) {
        const double r = in ? (a.y[o0 + i] - (a.y0 ? a.y0[o0 + i] : 0.0)) : 0.0;
        vr[i] = r; rsum += r;
      }
    }
    if (tid == 0) { s_rsum = 0.0; s_bad = 0; }
    cta_sync<WARPS>();
    if (TASK == TASK_LOO && a.loo_mode == 1) {
      rsum = red_warp(rsum);
      if (lane == 0) atomicAdd(&s_rsum, rsum);
    }

    // ---------------- left-looking block Cholesky; slot(J,J) receives T_J = L_JJ^-1.
    // log det accumulates as mantissa * 2^exponent of the pivot product (one log per object).
    double lp_m = 1.0; int lp_e = 0;
    // mode bit 0 (diagonal warp): warp 0 owns the diagonal tile alone -- its eight serial pivots are the critical path of
    // a column -- while the other warps share the off-diagonal tiles, instead of taking an equal share of the column first.
    // mode bit 1 (look-ahead): the rank-8(J-1) part of C[J][J] is accumulated one column early by the last warp and parked
    // in slot(J,J); warp 0 solves L[J][J-1] itself right after T_{J-1}, subtracts its square and carries C[J][J] in
    // registers into the next column: it only ARRIVES at the barrier that ends the solve phase, so that the chain
    // pivots -> one panel tile -> one rank-8 update -> pivots is all that is left on the critical path.
    const bool dwarp = WARPS > 1 && (mode & 1);
    const bool la = dwarp && (mode & 2);
    // sum_{P<cnt} X[row][P] X[row][P]^T: both operands are the same fragment; four chains (k-halves x parity of P)
    auto self_syrk = [&](int row, int cnt, double& r0, double& r1) {
      double a0 = 0.0, a1 = 0.0, b0 = 0.0, b1 = 0.0, c0 = 0.0, c1 = 0.0, d0 = 0.0, d1 = 0.0;
      const double* tj = tiles + slot(row, 0) * TILE + L.fr;
      int P = 0;
      for (; P + 1 < cnt; P += 2) {
        const double2 f = *reinterpret_cast<const double2*>(tj + P * TILE);
        const double2 g = *reinterpret_cast<const double2*>(tj + (P + 1) * TILE);
        dmma(a0, a1, f.x, f.x); dmma(b0, b1, f.y, f.y);
        dmma(c0, c1, g.x, g.x); dmma(d0, d1, g.y, g.y);
      }
      if (P < cnt) {
        const double2 f = *reinterpret_cast<const double2*>(tj + P * TILE);
        dmma(a0, a1, f.x, f.x); dmma(b0, b1, f.y, f.y);
      }
      r0 = (a0 + b0) + (c0 + d0); r1 = (a1 + b1) + (c1 + d1);
    };
    // mode bit 2 (z in the loop): z = L^-1 r rides along as one more row -- the last warp forms r_J - sum L[J][P] z_P
    // beside the tiles of column J and multiplies by T_J in the solve phase -- instead of a serial substitution by
    // warp 0 after the factorisation, which the other warps spend at the barrier of the next object.
    // (prediction with several CTAs per SM: measured slower, 4.16 -> 4.55 ms at N = 128; with one object per SM it pays)
    constexpr bool ZTASK = (TASK == TASK_LL && WARPS > 1) || (FWD && WARPS >= 8 && NB_MAX > 16);
    const bool zin = ZTASK && (mode & 4);
    double zquad = 0.0;
    double ck0 = 0.0, ck1 = 0.0;                           // look-ahead: C[J][J], carried by warp 0 out of column J-1
    for (int J = 0; J < nb; ++J) {
      auto finish_diag = [&](double k0, double k1) {
        double t0, t1, piv; int badk;
        diag_factor(k0, k1, L, t0, t1, piv, badk);
        st_acc(tiles, slot(J, J), L, t0, t1);
        if (TASK == TASK_LL || TASK == TASK_MATRICES) {
          lp_m *= piv;
          const int hi = __double2hiint(lp_m);
          const int e = ((hi >> 20) & 0x7ff) - 1023;
          lp_e += e;
          lp_m = __hiloint2double(hi - (e << 20), __double2loint(lp_m));
        }
        if (badk && lane == 0 && s_bad == 0) s_bad = 8 * J + badk;
      };
      double dk0 = 0.0, dk1 = 0.0;                         // C[J][J] in warp 0, factorised once its other tiles are parked
      if (dwarp && warp == 0) {
        if (la && J > 0) { dk0 = ck0; dk1 = ck1; }
        else {
          double r0, r1;
          self_syrk(J, J, r0, r1);
          k_tile_minus<DIM>(cov, px, noise, ld, n, J, J, L, r0, r1, dk0, dk1, amat, lda);
        }
      }
      // tiles of block column J owned by this warp, two at a time; each tile accumulates its
      // rank-8J update on two independent DMMA chains (k-halves) -> 4 chains in flight
      const int nw = dwarp ? WARPS - 1 : WARPS;
      const int i_first = dwarp ? (warp == 0 ? nb : J + warp) : J + warp;
      for (int I = i_first; I < nb; I += 2 * nw) {
        const int I2 = I + nw;
        const bool two = I2 < nb;
        double a0 = 0.0, a1 = 0.0, b0 = 0.0, b1 = 0.0, c0 = 0.0, c1 = 0.0, d0 = 0.0, d1 = 0.0;
        const double* tj = tiles + slot(J, 0) * TILE + L.fr;
        const double* ti = tiles + slot(I, 0) * TILE + L.fr;
        const double* ti2 = tiles + slot(two ? I2 : I, 0) * TILE + L.fr;
        if (two) {
#pragma unroll 2
          for (int P = 0; P < J; ++P) {
            const double2 fb = *reinterpret_cast<const double2*>(tj + P * TILE);
            const double2 fa = *reinterpret_cast<const double2*>(ti + P * TILE);
            const double2 fc = *reinterpret_cast<const double2*>(ti2 + P * TILE);
            dmma(a0, a1, fa.x, fb.x); dmma(b0, b1, fa.y, fb.y);
            dmma(c0, c1, fc.x, fb.x); dmma(d0, d1, fc.y, fb.y);
          }
        } else {                                          // a single tile: the four chains split P by parity instead
          int P = 0;
          for (; P + 1 < J; P += 2) {
            const double2 fb = *reinterpret_cast<const double2*>(tj + P * TILE);
            const double2 fa = *reinterpret_cast<const double2*>(ti + P * TILE);
            const double2 gb = *reinterpret_cast<const double2*>(tj + (P + 1) * TILE);
            const double2 ga = *reinterpret_cast<const double2*>(ti + (P + 1) * TILE);
            dmma(a0, a1, fa.x, fb.x); dmma(b0, b1, fa.y, fb.y);
            dmma(c0, c1, ga.x, gb.x); dmma(d0, d1, ga.y, gb.y);
          }
          if (P < J) {
            const double2 fb = *reinterpret_cast<const double2*>(tj + P * TILE);
            const double2 fa = *reinterpret_cast<const double2*>(ti + P * TILE);
            dmma(a0, a1, fa.x, fb.x); dmma(b0, b1, fa.y, fb.y);
          }
          a0 += c0; a1 += c1; b0 += d0; b1 += d1;
        }
        // both covariance tiles of a pair before either store: their four exp chains interleave in one straight line
        double k0, k1, m0 = 0.0, m1 = 0.0;
        if (two) k_tile2_minus<DIM>(cov, px, noise, ld, n, I, I2, J, L, a0 + b0, a1 + b1, c0 + d0, c1 + d1, k0, k1, m0, m1, amat, lda);
        else k_tile_minus<DIM>(cov, px, noise, ld, n, I, J, L, a0 + b0, a1 + b1, k0, k1, amat, lda);
        if (I == J) {                                     // warp 0 (only without a dedicated diagonal warp)
          dk0 = k0; dk1 = k1;
        } else {
          st_acc(tiles, slot(I, J), L, k0, k1);           // park C[I][J] in its own slot
        }
        if (two) st_acc(tiles, slot(I2, J), L, m0, m1);
      }
      if (la && warp == WARPS - 1 && J + 1 < nb) {        // next diagonal tile, all but its last rank-8 term
        double r0, r1, k0, k1;
        self_syrk(J + 1, J, r0, r1);
        k_tile_minus<DIM>(cov, px, noise, ld, n, J + 1, J + 1, L, r0, r1, k0, k1, amat, lda);
        st_acc(tiles, slot(J + 1, J + 1), L, k0, k1);
      }
      double zw = 0.0;
      if (ZTASK && zin && warp == WARPS - 1) {
        double p = 0.0, p2 = 0.0;
        const double* tj = tiles + slot(J, 0) * TILE + L.fr;
        for (int P = 0; P < J; ++P) {
          const double2 f = *reinterpret_cast<const double2*>(tj + P * TILE);
          p = fma(f.x, vr[8 * P + 2 * L.t], p); p2 = fma(f.y, vr[8 * P + 2 * L.t + 1], p2);
        }
        zw = FWD ? vr[8 * J + L.g] + red_t(p + p2) : vr[8 * J + L.g] - red_t(p + p2);      // FWD: the tiles hold -L
      }
      if (warp == 0) finish_diag(dk0, dk1);
      cta_sync<WARPS>();
      const double2 ft = ld_frag(tiles, slot(J, J), L);
      if (ZTASK && zin && warp == WARPS - 1) {
        double q = ft.x * __shfl_sync(FULL, zw, L.t * 8) + ft.y * __shfl_sync(FULL, zw, L.t * 8 + 4);
        q = red_t(q);
        if (L.t == 0) { vr[8 * J + L.g] = q; zquad = fma(q, q, zquad); }
      }
      // prediction keeps -L below the diagonal: the forward substitution of the grid phase then accumulates
      // h + sum V_P (-L[J][P])^T directly (the rank updates of later columns do not notice the sign)
      constexpr double sgn = FWD ? -1.0 : 1.0;
      if (la && warp == 0) {
        if (J + 1 < nb) {
          const double2 fc = ld_frag(tiles, slot(J + 1, J), L);
          double d0 = 0.0, d1 = 0.0, e0 = 0.0, e1 = 0.0, m0 = 0.0, m1 = 0.0, q0 = 0.0, q1 = 0.0;
          dmma(d0, d1, fc.x, ft.x); dmma(e0, e1, fc.y, ft.y);
          const double2 dp = ld_frag(tiles, slot(J + 1, J + 1), L);
          const double l0 = d0 + e0, l1 = d1 + e1;          // the accumulator pair is the operand fragment of the tile
          __syncwarp();
          st_acc(tiles, slot(J + 1, J), L, sgn * l0, sgn * l1);
          dmma(m0, m1, l0, l0); dmma(q0, q1, l1, l1);
          ck0 = dp.x - (m0 + q0); ck1 = dp.y - (m1 + q1);
        }
        asm volatile("bar.arrive 1, %0;" :: "r"(NT) : "memory");
      } else {
        const int s_first = J + 1 + warp;                   // with look-ahead warp 0 is not here: rows J+2.. over warps 1..
        const int s_nw = la ? WARPS - 1 : WARPS;
        for (int I = s_first; I < nb; I += 2 * s_nw) {      // L[I][J] = C[I][J] T_J^T
          const int I2 = I + s_nw;
          const bool two = I2 < nb;
          const double2 fc = ld_frag(tiles, slot(I, J), L);
          const double2 fe = ld_frag(tiles, slot(two ? I2 : I, J), L);
          double d0 = 0.0, d1 = 0.0, e0 = 0.0, e1 = 0.0, f0 = 0.0, f1 = 0.0, g0 = 0.0, g1 = 0.0;
          dmma(d0, d1, fc.x, ft.x); dmma(e0, e1, fc.y, ft.y);
          if (two) { dmma(f0, f1, fe.x, ft.x); dmma(g0, g1, fe.y, ft.y); }
          __syncwarp();
          st_acc(tiles, slot(I, J), L, sgn * (d0 + e0), sgn * (d1 + e1));
          if (two) st_acc(tiles, slot(I2, J), L, sgn * (f0 + g0), sgn * (f1 + g1));
        }
        if (la) asm volatile("bar.sync 1, %0;" :: "r"(NT) : "memory");
        else cta_sync<WARPS>();
      }
    }
    if (la) cta_sync<WARPS>();                              // warp 0 ran ahead of the last solve phases

    if (TASK == TASK_LL && ZTASK && zin) {
      if (warp == WARPS - 1) {
        zquad = red_warp(zquad);
        if (lane == 0) s_quad = zquad;
      }
      cta_sync<WARPS>();
      if (tid == 0) {                                     // log det lives in warp 0
        const int bad = s_bad;
        a.info[io] = bad;
        const double logdet = log(lp_m) + (double)lp_e * 0.693147180559945309417232;
        a.ll[io] = bad ? nan("") : -0.5 * (s_quad + logdet + n * LOG_2PI);
      }
      continue;
    }
    if (TASK == TASK_LL) {
      // ---------------- z = L^-1 r by block forward substitution (warp 0), quad = |z|^2
      if (warp == 0) {
        double quad = 0.0;
        for (int J = 0; J < nb; ++J) {
          double p = 0.0, p2 = 0.0;
          const double* tj = tiles + slot(J, 0) * TILE + L.fr;
          for (int P = 0; P < J; ++P) {
            const double2 f = *reinterpret_cast<const double2*>(tj + P * TILE);
            p = fma(f.x, vr[8 * P + 2 * L.t], p); p2 = fma(f.y, vr[8 * P + 2 * L.t + 1], p2);
          }
          const double wv = vr[8 * J + L.g] - red_t(p + p2);
          const double2 f = *reinterpret_cast<const double2*>(tj + J * TILE);
          double q = f.x * __shfl_sync(FULL, wv, L.t * 8) + f.y * __shfl_sync(FULL, wv, L.t * 8 + 4);
          q = red_t(q);
          if (L.t == 0) { vr[8 * J + L.g] = q; quad = fma(q, q, quad); }
          __syncwarp();
        }
        quad = red_warp(quad);
        if (lane == 0) {
          const int bad = s_bad;
          a.info[io] = bad;
          const double logdet = log(lp_m) + (double)lp_e * 0.693147180559945309417232;
          a.ll[io] = bad ? nan("") : -0.5 * (quad + logdet + n * LOG_2PI);
        }
      }
      continue;
    }

    if (FWD) {
      // ---------------- prediction without L^-1 (see cgp_small64.cu): z = L^-1 r by block forward substitution (warp 0),
      // then per block of 8 grid points the same substitution for the cross-covariance rows ON THE TENSOR CORES:
      // V_P = W_P T_P^T (operands: the accumulator registers and the T_P tile), W_J += V_P (-L[J][P])^T for J > P;
      // mean = v . z + y0*, var = amp* - |v|^2.  h is kept WITHOUT its amplitude (applied once per grid point).
      if (warp == 0 && !(ZTASK && zin)) {
        for (int J = 0; J < nb; ++J) {
          double p = 0.0, p2 = 0.0;
          const double* tj = tiles + slot(J, 0) * TILE + L.fr;
          for (int P = 0; P < J; ++P) {
            const double2 f = *reinterpret_cast<const double2*>(tj + P * TILE);
            p = fma(f.x, vr[8 * P + 2 * L.t], p); p2 = fma(f.y, vr[8 * P + 2 * L.t + 1], p2);
          }
          const double wv = vr[8 * J + L.g] + red_t(p + p2);                 // the tiles hold -L
          const double2 f = *reinterpret_cast<const double2*>(tj + J * TILE);
          double q = f.x * __shfl_sync(FULL, wv, L.t * 8) + f.y * __shfl_sync(FULL, wv, L.t * 8 + 4);
          q = red_t(q);
          if (L.t == 0) vr[8 * J + L.g] = q;
          __syncwarp();
        }
      }
      cta_sync<WARPS>();
      const int bad = s_bad;
      if (tid == 0 && part == 0) a.info[b] = bad;
      const int64_t g0 = a.goff ? a.goff[b] : 0;
      const int64_t m_pts = a.goff ? (a.goff[b + 1] - g0) : a.m_shared;
      const int64_t out0 = a.goff ? g0 : b * a.m_shared;
      const int64_t n_rb = (m_pts + 7) >> 3;
      const double amp_star = cov.amp_auto + cov.nugget2;
      for (int64_t rb = (int64_t)part * WARPS + warp; rb < n_rb; rb += (int64_t)parts * WARPS) {
        const int64_t mi = 8 * rb + L.g;
        const bool live = mi < m_pts;
        double gx = 0.0, gy = 0.0;
        if (live) {
          if (DIM == 1) gx = a.xnew[g0 + mi];
          else { gx = a.xnew[2 * (g0 + mi)]; gy = a.xnew[2 * (g0 + mi) + 1]; }
        }
        double acc0[NB_MAX], acc1[NB_MAX];
#pragma unroll
        for (int P = 0; P < NB_MAX; ++P) {                // cross-covariance fragments = start values of W_P
          acc0[P] = 0.0; acc1[P] = 0.0;
          if (P < nb) {
            const int c0 = 8 * P + 2 * L.t, c1 = c0 + 1;
            if (live && c0 < n) acc0[P] = cgp_exp(rbf_arg<DIM>(cov, gx, gy, px[c0], DIM == 2 ? px[ld + c0] : 0.0));
            if (live && c1 < n) acc1[P] = cgp_exp(rbf_arg<DIM>(cov, gx, gy, px[c1], DIM == 2 ? px[ld + c1] : 0.0));
          }
        }
        double pm = 0.0, pm2 = 0.0, vv = 0.0, vv2 = 0.0;
        // unrolled by template recursion: the accumulators must stay in registers, and at NB_MAX = 28 the loop unroller
        // gives up on the 406-tile triangle (the arrays then live in local memory: 544 bytes of stack, 21 ms instead of 14)
        static_for<0, NB_MAX>([&](auto Pc) {
          constexpr int P = decltype(Pc)::value;
          if (P < nb) {
            const double2 ft = ld_frag(tiles, slot(P, P), L);
            double r0 = 0.0, r1 = 0.0, e0 = 0.0, e1 = 0.0;
            dmma(r0, r1, acc0[P], ft.x); dmma(e0, e1, acc1[P], ft.y);
            const double v0 = r0 + e0, v1 = r1 + e1;
            acc0[P] = v0; acc1[P] = v1;
            pm = fma(v0, vr[8 * P + 2 * L.t], pm); pm2 = fma(v1, vr[8 * P + 2 * L.t + 1], pm2);
            vv = fma(v0, v0, vv); vv2 = fma(v1, v1, vv2);
            if (a.vout && live)                           // bulk covariance writer (cgp_covariance_batched_dev)
              *reinterpret_cast<double2*>(a.vout + (out0 + mi) * ld + 8 * P + 2 * L.t) = make_double2(v0, v1);
            static_for<P + 1, NB_MAX>([&](auto Jc) {      // compile-time triangle: no wasted DMMA
              constexpr int J = decltype(Jc)::value;
              if (J < nb) {
                const double2 fb = ld_frag(tiles, slot(J, P), L);
                dmma(acc0[J], acc1[J], v0, fb.x); dmma(acc0[J], acc1[J], v1, fb.y);
              }
            });
          }
        });
        pm = red_t(pm + pm2); vv = red_t(vv + vv2);
        if (live && L.t == 0) {
          const double m0 = !a.new_y0 ? 0.0 : (a.new_y0_diff ? a.new_y0[mi] + a.new_y0_diff[b] : a.new_y0[out0 + mi]);
          double mean = fma(cov.amp_cross, pm, m0);
          double var = fma(-cov.amp_cross * cov.amp_cross, vv, amp_star);
          if (bad) { mean = nan(""); var = mean; }
          a.mean[out0 + mi] = mean;
          if (a.var) a.var[out0 + mi] = var;
        }
      }
      continue;
    }

    // ---------------- L^-1, row by row, in place (slot(I,J) <- L^-1[I][J]);
    // L^-1[I][J] = -T_I * sum_{P=J..I-1} L[I][P] L^-1[P][J]; one A fragment per P feeds all J <= P
    for (int I = 1; I < nb; ++I) {
      double s0[KMAX], s1[KMAX];
#pragma unroll
      for (int k = 0; k < KMAX; ++k) { s0[k] = 0.0; s1[k] = 0.0; }
      const double* ti = tiles + slot(I, 0) * TILE + L.fr;
      for (int P = 0; P < I; ++P) {
        const double2 fa = *reinterpret_cast<const double2*>(ti + P * TILE);
        const double* tp = tiles + slot(P, 0) * TILE;
#pragma unroll
        for (int k = 0; k < KMAX; ++k) {
          const int J = warp + k * WARPS;
          if (J <= P) {
            const double* q = tp + J * TILE;
            dmma(s0[k], s1[k], fa.x, q[L.tr0]); dmma(s0[k], s1[k], fa.y, q[L.tr1]);
          }
        }
      }
      cta_sync<WARPS>();                                  // every read of row I of L is done
      const double2 ft = ld_frag(tiles, slot(I, I), L);
#pragma unroll
      for (int k = 0; k < KMAX; ++k) {
        const int J = warp + k * WARPS;
        if (J < I) {
          st_acc(tiles, slot(I, J), L, s0[k], s1[k]);
          __syncwarp();
          const double2 fs = ld_fragT(tiles, slot(I, J), L);
          double d0 = 0.0, d1 = 0.0, e0 = 0.0, e1 = 0.0;
          dmma(d0, d1, ft.x, fs.x); dmma(e0, e1, ft.y, fs.y);
          __syncwarp();
          st_acc(tiles, slot(I, J), L, -(d0 + e0), -(d1 + e1));
        }
      }
      cta_sync<WARPS>();
    }

    if (TASK == TASK_MATRICES) {
      const int bad = s_bad;
      if (tid == 0) {
        a.info[b] = bad;
        if (a.logdet) a.logdet[b] = bad ? nan("") : log(lp_m) + (double)lp_e * 0.693147180559945309417232;
      }
      const int64_t mo = a.moff[b];
      const int64_t mld = a.ld_obj ? lda : (a.mld ? a.mld : n);
      if (a.kmat && !amat) {
        for (int e = tid; e < n * n; e += NT) {
          const int i = e / n, j = e - i * n;
          a.kmat[mo + (int64_t)i * mld + j] = (i == j) ? cov.amp_auto + noise[i] : cov.amp_auto * cov_e<DIM>(cov, px, ld, i, j);
        }
      }
      if (a.linv) {       // L^-1 tiles (lower) and explicit zeros above the diagonal
        int q = 0;
        for (int I = 0; I < nb; ++I)
          for (int J = 0; J < nb; ++J, ++q) {
            if (q % WARPS != warp) continue;
            const double* tp = tiles + slot(I, J <= I ? J : 0) * TILE;
            const int gi = 8 * I + L.g, cj = 8 * J + 2 * L.t;
            double c0 = (J <= I) ? tp[L.fr] : 0.0, c1 = (J <= I) ? tp[L.fr + 1] : 0.0;
            if (bad) { c0 = nan(""); c1 = c0; }
            if (gi < n && cj < n) a.linv[mo + (int64_t)gi * mld + cj] = c0;
            if (gi < n && cj + 1 < n) a.linv[mo + (int64_t)gi * mld + cj + 1] = c1;
          }
      }
      if (a.kinv) {       // K^-1 = L^-T L^-1: tile (I,J) = sum_{P>=I} Linv[P][I]^T Linv[P][J]
        int q = 0;
        for (int I = 0; I < nb; ++I)
          for (int J = 0; J <= I; ++J, ++q) {
            if (q % WARPS != warp) continue;
            double c0 = 0.0, c1 = 0.0;
            for (int P = I; P < nb; ++P) {
              const double2 fa = ld_fragT(tiles, slot(P, I), L);
              const double2 fb = ld_fragT(tiles, slot(P, J), L);
              dmma(c0, c1, fa.x, fb.x); dmma(c0, c1, fa.y, fb.y);
            }
            if (bad) { c0 = nan(""); c1 = c0; }
            const int gi = 8 * I + L.g, cj = 8 * J + 2 * L.t;
            if (gi < n) {
              if (cj < n) { a.kinv[mo + (int64_t)gi * mld + cj] = c0; a.kinv[mo + (int64_t)cj * mld + gi] = c0; }
              if (cj + 1 < n) { a.kinv[mo + (int64_t)gi * mld + cj + 1] = c1; a.kinv[mo + (int64_t)(cj + 1) * mld + gi] = c1; }
            }
          }
      }
      continue;
    }

    // ---------------- z = L^-1 r  (and L^-1 1), then alpha = L^-T z, d = colnorm^2(L^-1), u = L^-T(L^-1 1)
    const bool want_u = (TASK == TASK_LOO) && (a.loo_mode == 1);
    for (int I = warp; I < nb; I += WARPS) {
      double p = 0.0, p2 = 0.0, p1 = 0.0;
      const double* ti = tiles + slot(I, 0) * TILE + L.fr;
      for (int J = 0; J <= I; ++J) {
        const double2 f = *reinterpret_cast<const double2*>(ti + J * TILE);
        p = fma(f.x, vr[8 * J + 2 * L.t], p); p2 = fma(f.y, vr[8 * J + 2 * L.t + 1], p2);
        if (want_u) {                                     // padded columns multiply exact zeros of L^-1
          p1 += f.x; p1 += f.y;
        }
      }
      p = red_t(p + p2);
      if (L.t == 0) vz[8 * I + L.g] = p;
      if (want_u) { p1 = red_t(p1); if (L.t == 0) v1[8 * I + L.g] = (8 * I + L.g < n) ? p1 : 0.0; }
    }
    cta_sync<WARPS>();
    for (int J = warp; J < nb; J += WARPS) {
      double pa0 = 0.0, pa1 = 0.0, pd0 = 0.0, pd1 = 0.0, pu0 = 0.0, pu1 = 0.0;
      for (int I = J; I < nb; ++I) {
        const double2 f = ld_frag(tiles, slot(I, J), L);
        const double zi = vz[8 * I + L.g];
        pa0 = fma(f.x, zi, pa0); pa1 = fma(f.y, zi, pa1);
        if (TASK == TASK_LOO) {
          // rows >= n of L^-1 are identity rows: keep them out of the column norms
          const bool in = 8 * I + L.g < n;
          pd0 = in ? fma(f.x, f.x, pd0) : pd0; pd1 = in ? fma(f.y, f.y, pd1) : pd1;
          if (want_u) { const double ui = v1[8 * I + L.g]; pu0 = fma(f.x, ui, pu0); pu1 = fma(f.y, ui, pu1); }
        }
      }
      pa0 = red_g(pa0); pa1 = red_g(pa1);
      if (L.g == 0) { va[8 * J + 2 * L.t] = pa0; va[8 * J + 2 * L.t + 1] = pa1; }
      if (TASK == TASK_LOO) {
        pd0 = red_g(pd0); pd1 = red_g(pd1);
        if (L.g == 0) { vd[8 * J + 2 * L.t] = pd0; vd[8 * J + 2 * L.t + 1] = pd1; }
        if (want_u) {
          pu0 = red_g(pu0); pu1 = red_g(pu1);
          if (L.g == 0) { vu[8 * J + 2 * L.t] = pu0; vu[8 * J + 2 * L.t + 1] = pu1; }
        }
      }
    }
    cta_sync<WARPS>();
    const int bad = s_bad;
    if (tid == 0 && part == 0) a.info[b] = bad;

    if (TASK == TASK_LOO) {
      // ---------------- closed-form leave-one-out (pull.py:66-94; SURVEY.md row a8)
      const double rho = cov.amp_cross / cov.amp_auto;
      const double amp_star = cov.amp_auto + cov.nugget2;
      const double rs = s_rsum;
      for (int i = tid; i < n; i += NT) {
        const double d = vd[i], r = vr[i];
        const double yv = a.y[o0 + i];
        const double m = a.y0 ? a.y0[o0 + i] : 0.0;
        const double ye = a.yerr ? a.yerr[o0 + i] : 0.0;
        double pr = m + rho * (r - va[i] / d);
        if (want_u) {
          const double delta = (rs - r) / (double)(n - 1);
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
      continue;
    }

    if (TASK == TASK_PREDICT) {
      // ---------------- N > 128: grid points in blocks of 8 against the explicit L^-1: v = L^-1 h, mean = h.alpha + y0*,
      // var = amp* - |v|^2.  h is kept WITHOUT its amplitude (applied once per grid point at the end).
      const int64_t g0 = a.goff ? a.goff[b] : 0;
      const int64_t m_pts = a.goff ? (a.goff[b + 1] - g0) : a.m_shared;
      const int64_t out0 = a.goff ? g0 : b * a.m_shared;
      const int64_t n_rb = (m_pts + 7) >> 3;
      const double amp_star = cov.amp_auto + cov.nugget2;
      for (int64_t rb = (int64_t)part * WARPS + warp; rb < n_rb; rb += (int64_t)parts * WARPS) {
        const int64_t mi = 8 * rb + L.g;
        const bool live = mi < m_pts;
        double gx = 0.0, gy = 0.0;
        if (live) {
          if (DIM == 1) gx = a.xnew[g0 + mi];
          else { gx = a.xnew[2 * (g0 + mi)]; gy = a.xnew[2 * (g0 + mi) + 1]; }
        }
        double acc0[NB_MAX], acc1[NB_MAX];
#pragma unroll
        for (int J = 0; J < NB_MAX; ++J) { acc0[J] = 0.0; acc1[J] = 0.0; }
        double pm = 0.0, pm2 = 0.0;
#pragma unroll
        for (int P = 0; P < NB_MAX; ++P) {
          if (P < nb) {
            const int c0 = 8 * P + 2 * L.t, c1 = c0 + 1;
            double h0 = 0.0, h1 = 0.0;                    // A fragment of the cross-covariance block
            if (live && c0 < n) h0 = cgp_exp(rbf_arg<DIM>(cov, gx, gy, px[c0], DIM == 2 ? px[ld + c0] : 0.0));
            if (live && c1 < n) h1 = cgp_exp(rbf_arg<DIM>(cov, gx, gy, px[c1], DIM == 2 ? px[ld + c1] : 0.0));
            pm = fma(h0, va[c0], pm); pm2 = fma(h1, va[c1], pm2);
#pragma unroll
            for (int J = P; J < NB_MAX; ++J) {            // compile-time triangle: no wasted DMMA
              if (J < nb) {
                const double2 fb = ld_frag(tiles, slot(J, P), L);
                dmma(acc0[J], acc1[J], h0, fb.x); dmma(acc0[J], acc1[J], h1, fb.y);
              }
            }
          }
        }
        double vv = 0.0, vv2 = 0.0;
#pragma unroll
        for (int J = 0; J < NB_MAX; ++J) {
          vv = fma(acc0[J], acc0[J], vv); vv2 = fma(acc1[J], acc1[J], vv2);
          if (a.vout && live && J < nb)
            *reinterpret_cast<double2*>(a.vout + (out0 + mi) * ld + 8 * J + 2 * L.t) = make_double2(acc0[J], acc1[J]);
        }
        pm = red_t(pm + pm2); vv = red_t(vv + vv2);
        if (live && L.t == 0) {
          const double m0 = !a.new_y0 ? 0.0 : (a.new_y0_diff ? a.new_y0[mi] + a.new_y0_diff[b] : a.new_y0[out0 + mi]);
          double mean = fma(cov.amp_cross, pm, m0);
          double var = fma(-cov.amp_cross * cov.amp_cross, vv, amp_star);
          if (bad) { mean = nan(""); var = mean; }
          a.mean[out0 + mi] = mean;
          if (a.var) a.var[out0 + mi] = var;
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------
template <int DIM, int TASK, int NB_MAX, int WARPS, bool FWD_BIG = false>
int launch_one(int nbm, const SmallArgs& a, cudaStream_t stream) {
  auto kern = small_gp_kernel<DIM, TASK, NB_MAX, WARPS, FWD_BIG>;
  const size_t smem = small_smem_bytes((Task)TASK, DIM, nbm);
  static int sm_count = 0;
  if (!sm_count) {
    int dev; cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev);
  }
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  int per_sm = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, WARPS * 32, smem);
  if (e != cudaSuccess) return (int)e;
  if (per_sm < 1) return (int)cudaErrorInvalidConfiguration;
  const int64_t n_work = TASK != TASK_PREDICT ? a.n_obj : a.part_off ? a.n_parts : a.n_obj * a.split;
  int64_t grid = (int64_t)sm_count * per_sm;
  if (grid > n_work) grid = n_work;
  if (grid < 1) return 0;
  // the Cholesky schedule of the kernel (see its column loop): CGP_DIAG_WARP=0|1, CGP_LOOKAHEAD=0|1, CGP_Z_IN_LOOP=0|1
  static int mode = -1;
  if (mode < 0) {
    const char* e = getenv("CGP_DIAG_WARP"); const char* f = getenv("CGP_LOOKAHEAD"); const char* g = getenv("CGP_Z_IN_LOOP");
    mode = ((e ? atoi(e) : 1) ? 1 : 0) | ((f ? atoi(f) : 0) ? 2 : 0) | ((g ? atoi(g) : 1) ? 4 : 0);
  }
  const int dw = mode;
  kern<<<(unsigned)grid, WARPS * 32, smem, stream>>>(a, nbm, dw);
  count_launch();
  return (int)cudaGetLastError();
}

// warps per object for nb <= 8: tuned per task on B200 (override: CGP_SMALL_WARPS=1|2|4)
static int small_warps(int task) {
  static int forced = -1;
  if (forced < 0) { const char* e = getenv("CGP_SMALL_WARPS"); forced = e ? atoi(e) : 0; }
  if (forced == 1 || forced == 2 || forced == 4) return forced;
  return task == TASK_PREDICT ? 4 : 1;     // B200, C2 shape: predict 9.2 / 8.3 / 7.7 ms at 1 / 2 / 4 warps; LL 2.1 / 2.6 / 3.2
}

template <int DIM, int TASK>
int launch_cfg(int nbm, const SmallArgs& a, cudaStream_t stream) {
  if (nbm <= 8) {
    const int w = small_warps(TASK);
    if (w == 2) return launch_one<DIM, TASK, 8, 2>(nbm, a, stream);
    if (w == 4) return launch_one<DIM, TASK, 8, 4>(nbm, a, stream);
    return launch_one<DIM, TASK, 8, 1>(nbm, a, stream);
  }
  static int mid = -1;
  if (mid < 0) { const char* e = getenv("CGP_MID_WARPS"); mid = (e && atoi(e) == 8) ? 8 : 4; }
  if (nbm <= 16) {
    if (mid == 8 && TASK != TASK_MATRICES) return launch_one<DIM, TASK, 16, 8>(nbm, a, stream);
    return launch_one<DIM, TASK, 16, 4>(nbm, a, stream);
  }
  // above 128 points one object fills the shared memory of an SM: eight warps (two per sub-partition) instead of four
  // hide more of each other's dependent chains (CGP_BIG_WARPS=4 for the round-1 shape)
  static int big = -1;
  if (big < 0) { const char* e = getenv("CGP_BIG_WARPS"); big = (e && atoi(e) == 4) ? 4 : 8; }
  if (big == 4 || TASK == TASK_MATRICES) return launch_one<DIM, TASK, 28, 4>(nbm, a, stream);
  static int bigfwd = -1;
  if (bigfwd < 0) { const char* e = getenv("CGP_BIG_FWD"); bigfwd = e ? atoi(e) : 1; }
  if (TASK == TASK_PREDICT && bigfwd) return launch_one<DIM, TASK, 28, 8, true>(nbm, a, stream);
  return launch_one<DIM, TASK, 28, 8>(nbm, a, stream);
}

template <int DIM>
int launch_task(Task task, int nbm, const SmallArgs& a, cudaStream_t stream) {
  switch (task) {
    case TASK_LL: return launch_cfg<DIM, TASK_LL>(nbm, a, stream);
    case TASK_PREDICT: return launch_cfg<DIM, TASK_PREDICT>(nbm, a, stream);
    case TASK_LOO: return launch_cfg<DIM, TASK_LOO>(nbm, a, stream);
    case TASK_MATRICES: return launch_cfg<DIM, TASK_MATRICES>(nbm, a, stream);
  }
  return (int)cudaErrorInvalidValue;
}

// ---------------------------------------------------------------------------------------
// FP64 ceiling probes (the roofline denominator is measured on the box, not assumed).
__global__ void peak_dfma(double* out, int iters, double a, double b) {
  double acc[8];
#pragma unroll
  for (int i = 0; i < 8; i++) acc[i] = threadIdx.x + i;
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int i = 0; i < 8; i++) acc[i] = fma(acc[i], a, b);
  }
  double s = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) s += acc[i];
  if (s == 123.456) out[0] = s;
}
__global__ void peak_dmma(double* out, int iters, double a, double b) {
  double c0[8], c1[8];
#pragma unroll
  for (int i = 0; i < 8; i++) { c0[i] = threadIdx.x; c1[i] = i; }
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int i = 0; i < 8; i++) {
      asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                   : "+d"(c0[i]), "+d"(c1[i]) : "d"(a), "d"(b));
    }
  }
  double s = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) s += c0[i] + c1[i];
  if (s == 123.456) out[0] = s;
}

}  // namespace

size_t small_smem_bytes(Task task, int dim, int nb) {
  const int nv = task == TASK_LL ? 1 : (task == TASK_PREDICT ? 3 : (task == TASK_LOO ? 6 : 0));
  size_t doubles = (size_t)((nb * (nb + 1)) / 2) * TILE + (size_t)(dim + 1 + nv) * 8 * nb;
  return doubles * sizeof(double);
}

int launch_small(Task task, int dim, int max_n, const SmallArgs& a, cudaStream_t stream) {
  const int nbm = max_n < 1 ? 1 : (max_n + 7) / 8;
  if (nbm > 28) return (int)cudaErrorInvalidValue;
  // N <= 64: the static one-warp-per-object kernel (CGP_SMALL_GENERIC=1 forces the generic one)
  static int generic = -1;
  if (generic < 0) { const char* e = getenv("CGP_SMALL_GENERIC"); generic = (e && atoi(e)) ? 1 : 0; }
  if (task == TASK_PREDICT_FU) {
    if (nbm > 8 || dim != 1 || a.goff || a.hyp_obj || a.m_shared < 2) return (int)cudaErrorInvalidValue;
    return launch_small64_d1_t6(nbm, a, stream);
  }
  if (task == TASK_PREDICT_U) {
    if (nbm > 8 || dim != 1 || a.goff || a.hyp_obj || a.m_shared < 2) return (int)cudaErrorInvalidValue;
    return launch_small64_d1_t7(nbm, a, stream);
  }
  if (task == TASK_FACTOR || task == TASK_PREDICT_F) {
    if (nbm > 8) return (int)cudaErrorInvalidValue;
    if (dim == 1) return task == TASK_FACTOR ? launch_small64_d1_t4(nbm, a, stream) : launch_small64_d1_t5(nbm, a, stream);
    return task == TASK_FACTOR ? launch_small64_d2_t4(nbm, a, stream) : launch_small64_d2_t5(nbm, a, stream);
  }
  if (!generic && nbm <= 8 && !a.amat && task != TASK_MATRICES) {
    if (dim == 1) {
      if (task == TASK_LL) return launch_small64_d1_t0(nbm, a, stream);
      if (task == TASK_PREDICT) return launch_small64_d1_t1(nbm, a, stream);
      return launch_small64_d1_t2(nbm, a, stream);
    }
    if (task == TASK_LL) return launch_small64_d2_t0(nbm, a, stream);
    if (task == TASK_PREDICT) return launch_small64_d2_t1(nbm, a, stream);
    return launch_small64_d2_t2(nbm, a, stream);
  }
  return dim == 1 ? launch_task<1>(task, nbm, a, stream) : launch_task<2>(task, nbm, a, stream);
}

int measure_fp64_peak(int kind, double* tflops) {
  int dev, sms;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  double* d;
  cudaError_t e = cudaMalloc(&d, 64);
  if (e != cudaSuccess) return (int)e;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  const int iters = 8192, grid = sms * 4, threads = 256;
  float best = 1e30f;
  for (int rep = 0; rep < 6; ++rep) {
    cudaEventRecord(e0);
    if (kind == 0) peak_dfma<<<grid, threads>>>(d, iters, 1.0000001, 1e-9);
    else peak_dmma<<<grid, threads>>>(d, iters, 1e-3, 1e-3);
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    float ms; cudaEventElapsedTime(&ms, e0, e1);
    if (rep && ms < best) best = ms;
  }
  count_launch(6);
  const double fl = kind == 0 ? 2.0 * 8 * iters * (double)grid * threads
                              : 2.0 * 256 * 8 * iters * (double)grid * (threads / 32);
  *tflops = fl / best * 1e-9;
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaFree(d);
  return (int)cudaGetLastError();
}

}  // namespace cgp
