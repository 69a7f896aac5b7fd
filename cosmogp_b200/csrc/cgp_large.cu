// Large single objects (N > 224, e.g. 2D PSF fits with 2,000..20,000 stars): the covariance
// lives in HBM and is factorised by a right-looking BLOCKED Cholesky with 128-wide panels.
//   diagonal block  : one CTA, the shared-memory DMMA kernel of cgp_small.cu in matrix-source
//                     mode -> T_kk = L_kk^-1 (stored in place of the block) + log det
//   panel           : L_ik = A_ik T_kk^T            (gemm_nt, in place)
//   trailing update : A_ij -= L_ik L_jk^T, i >= j   (gemm_nt, lower tiles only)  <- N^3/3 of the work
// gemm_nt is a 64x128x16 double-buffered (cp.async) FP64 tensor-core GEMM: 4 warps, each
// 32x64 of C as 32 m8n8k4 DMMA accumulators, 3 CTAs per SM; operands staged in shared memory
// with a 20-double row pitch so the per-lane fragment loads are bank-conflict free.
// Reference path replaced: scipy.linalg.cholesky / inv / dot in cosmogp/inv_matrix.py:21-31 and
// the H K^-1 products of cosmogp/Gaussian_process.py:332-361.
#include "cgp_internal.h"
#include "cgp_math.cuh"

#include <math.h>
#include <string.h>

#include <algorithm>
#include <vector>

namespace cgp {
namespace {

// 64 x 128 tiles, 4 warps, 3 CTAs per SM: while one CTA is in its prologue (first cp.async latency) or
// epilogue (C read-modify-write) the other two keep the DMMA pipe busy -- matters at K = 128, the
// panel width of the blocked Cholesky (r01: 128x128 tiles with 1 CTA/SM gave 23 TFLOP/s there).
constexpr int BM = 64, BN = 128, BK = 16, PITCH = BK + 4;   // PITCH % 16 == 4 -> conflict-free LDS.64
constexpr int GEMM_THREADS = 128;
constexpr size_t GEMM_SMEM = (size_t)2 * (BM + BN) * PITCH * sizeof(double);

__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
      : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" :: "n"(N)); }

// One 64 x 128 tile (or one 64-row half of a lower-triangle 128 x 128 block) of C, `tile` in the launch order of
// launch_gemm_nt.  Shared by the single-problem and the grouped kernels, so that a tile's arithmetic does not
// depend on which launch computes it.
__device__ __forceinline__ void gemm_nt_tile(double* sm, const GemmArgs& g, const int tile) {
  double* As = sm;                                 // [2][BM][PITCH]
  double* Bs = sm + 2 * BM * PITCH;                // [2][BN][PITCH]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int gq = lane >> 2, tq = lane & 3;
  const int wm = warp >> 1, wn = warp & 1;         // 2 x 2 warps: 32 x 64 of C each

  int bi, bj;                                      // bi: 64-row block, bj: 128-column block
  if (g.lower_only) {                              // linear index -> (I, bj) with I >= bj, two 64-row halves each
    const int t = tile >> 1;
    int I = (int)((sqrt(8.0 * t + 1.0) - 1.0) * 0.5);
    while ((I + 1) * (I + 2) / 2 <= t) ++I;
    while (I * (I + 1) / 2 > t) --I;
    bj = t - I * (I + 1) / 2;
    bi = 2 * I + (tile & 1);
  } else {
    const int nbn = g.n / BN;
    bi = tile / nbn; bj = tile - bi * nbn;
  }
  const double* ga = g.a + (int64_t)bi * BM * g.lda;
  const double* gb = g.b + (int64_t)bj * BN * g.ldb;

  auto load_stage = [&](int st, int kc) {
    double* as = As + st * BM * PITCH;
    double* bs = Bs + st * BN * PITCH;
#pragma unroll
    for (int i = 0; i < BM * 8 / GEMM_THREADS; ++i) {          // 16-byte pieces: 8 per row
      const int p = tid + i * GEMM_THREADS;
      const int row = p >> 3, c2 = (p & 7) << 1;
      cp_async16(as + row * PITCH + c2, ga + (int64_t)row * g.lda + kc * BK + c2);
    }
#pragma unroll
    for (int i = 0; i < BN * 8 / GEMM_THREADS; ++i) {
      const int p = tid + i * GEMM_THREADS;
      const int row = p >> 3, c2 = (p & 7) << 1;
      cp_async16(bs + row * PITCH + c2, gb + (int64_t)row * g.ldb + kc * BK + c2);
    }
    cp_async_commit();
  };

  double acc0[4][8], acc1[4][8];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) { acc0[i][j] = 0.0; acc1[i][j] = 0.0; }

  const int nk = g.k / BK;
  load_stage(0, 0);
  for (int kc = 0; kc < nk; ++kc) {
    const int st = kc & 1;
    if (kc + 1 < nk) { load_stage(st ^ 1, kc + 1); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
    __syncthreads();
    const double* as = As + st * BM * PITCH + (wm * 32 + gq) * PITCH + tq;
    const double* bs = Bs + st * BN * PITCH + (wn * 64 + gq) * PITCH + tq;
#pragma unroll
    for (int ks = 0; ks < BK / 4; ++ks) {
      double af[4], bf[8];
#pragma unroll
      for (int i = 0; i < 4; ++i) af[i] = as[i * 8 * PITCH + ks * 4];
#pragma unroll
      for (int j = 0; j < 8; ++j) bf[j] = bs[j * 8 * PITCH + ks * 4];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) dmma(acc0[i][j], acc1[i][j], af[i], bf[j]);
    }
    __syncthreads();
  }

  double* gc = g.c + ((int64_t)bi * BM + wm * 32 + gq) * g.ldc + (int64_t)bj * BN + wn * 64 + 2 * tq;
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      double2* p = reinterpret_cast<double2*>(gc + (int64_t)i * 8 * g.ldc + j * 8);
      double2 v = make_double2(g.alpha * acc0[i][j], g.alpha * acc1[i][j]);
      if (g.beta != 0.0) { const double2 o = *p; v.x = fma(g.beta, o.x, v.x); v.y = fma(g.beta, o.y, v.y); }
      *p = v;
    }
}

__global__ void __launch_bounds__(GEMM_THREADS, 3)
gemm_nt_kernel(const GemmArgs g) {
  extern __shared__ __align__(16) double sm[];
  gemm_nt_tile(sm, g, blockIdx.x);
}

// Many independent GEMMs in one launch: problem q owns tiles [tile_start[q], tile_start[q+1]) of the grid and
// computes them exactly as gemm_nt_kernel would for that problem alone.
__global__ void __launch_bounds__(GEMM_THREADS, 3)
gemm_nt_grouped_kernel(const GemmArgs* __restrict__ probs, const int* __restrict__ tile_start, const int nprob) {
  extern __shared__ __align__(16) double sm[];
  __shared__ GemmArgs g;                           // read from shared memory where used: kernel-parameter-like register use
  __shared__ int tile;
  if (threadIdx.x == 0) {
    const int t = blockIdx.x;
    int lo = 0, hi = nprob - 1;                    // last problem with tile_start <= t
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (tile_start[mid] <= t) lo = mid; else hi = mid - 1;
    }
    g = probs[lo];
    tile = t - tile_start[lo];
  }
  __syncthreads();
  gemm_nt_tile(sm, g, tile);
}

// ---------------------------------------------------------------------------------------
// Covariance builder: out[r][c] = amp * exp(-q(row point r, col point c)/2) (+ noise on the
// diagonal of an auto-covariance; identity padding beyond n / m).  One thread per 2 columns,
// coalesced 16-byte stores; the write (8 B/entry) and the exp (15 FP64 ops) bound it.
struct CovArgs {
  int dim; Cov cov; int autocov;
  const double* xc; int64_t n;          // column points (the object's epochs / stars)
  const double* xr; int64_t m;          // row points (== xc for auto-covariance)
  const double* yerr;
  double* out; int64_t ld; int64_t rows_pad, cols_pad;
};

template <int DIM>
__device__ __forceinline__ void cov_build_at(const CovArgs& a, const int64_t r, const int64_t c) {
  if (c >= a.cols_pad) return;
  double rx = 0.0, ry = 0.0;
  const bool rin = r < a.m;
  if (rin) { if (DIM == 1) rx = a.xr[r]; else { rx = a.xr[2 * r]; ry = a.xr[2 * r + 1]; } }
  double v[2];
#pragma unroll
  for (int e = 0; e < 2; ++e) {
    const int64_t cc = c + e;
    double val = 0.0;
    if (rin && cc < a.n) {
      double cx, cy = 0.0;
      if (DIM == 1) cx = a.xc[cc]; else { cx = a.xc[2 * cc]; cy = a.xc[2 * cc + 1]; }
      const double dx = cx - rx;                  // kernel.py:71: A = x - x2[:,None]
      double arg;
      if (DIM == 1) arg = dx * dx * a.cov.h00;
      else { const double dy = cy - ry; arg = fma(dy * a.cov.h11, dy, fma(dx, a.cov.h00, dy * a.cov.h01) * dx); }
      val = (a.autocov ? a.cov.amp_auto : a.cov.amp_cross) * cgp_exp(arg);
    }
    if (a.autocov && cc == r) {
      if (rin) { const double ye = a.yerr ? a.yerr[r] : 0.0; val = a.cov.amp_auto + ye * ye + a.cov.noise_const; }
      else val = 1.0;                              // identity padding keeps the factorisation valid
    }
    v[e] = val;
  }
  double* p = a.out + r * a.ld + c;
  if (c + 1 < a.cols_pad) *reinterpret_cast<double2*>(p) = make_double2(v[0], v[1]);
  else p[0] = v[0];
}
template <int DIM>
__global__ void cov_build_kernel(const CovArgs a) {
  cov_build_at<DIM>(a, blockIdx.y, ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 2);
}

// ---------------------------------------------------------------------------------------
// Triangular solves against the blocked factor (diagonal blocks hold T = L_kk^-1).
// Fused sweep steps (one launch per 128-block instead of two): every CTA recomputes the small
// triangular product of the step in shared memory (128 KB of T_kk from L2), CTA 0 publishes it, the
// others apply it to their slice.  Input and output vectors are distinct, so there is no race on
// the block being read.
// forward step k: z_k = T_kk u_k -> zout;  u[row] -= L[row, k-block] z_k for rows below (in place).
__device__ __forceinline__ void fwd_step_at(const double* a, int64_t ld, int64_t k0, int64_t n_pad, double* u, double* zout,
                                            const int cta) {
  __shared__ double sw[128], sz[128];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid < 128) sw[tid] = u[k0 + tid];
  __syncthreads();
  const double* t = a + k0 * ld + k0;
  for (int r = warp * 16; r < warp * 16 + 16; ++r) {              // 8 warps x 16 rows, 4 columns per lane
    const double* p = t + (int64_t)r * ld + lane * 4;
    const double2 q0 = *reinterpret_cast<const double2*>(p), q1 = *reinterpret_cast<const double2*>(p + 2);
    double acc = q0.x * sw[lane * 4] + q0.y * sw[lane * 4 + 1] + q1.x * sw[lane * 4 + 2] + q1.y * sw[lane * 4 + 3];
#pragma unroll
    for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) sz[r] = acc;
  }
  __syncthreads();
  if (cta == 0) { if (tid < 128) zout[k0 + tid] = sz[tid]; return; }
  const int64_t row0 = k0 + 128 + (int64_t)(cta - 1) * 64;
  for (int rr = warp * 8; rr < warp * 8 + 8; ++rr) {               // 64 rows per CTA
    const int64_t row = row0 + rr;
    if (row >= n_pad) break;
    const double* p = a + row * ld + k0 + lane * 4;
    const double2 q0 = *reinterpret_cast<const double2*>(p), q1 = *reinterpret_cast<const double2*>(p + 2);
    double acc = q0.x * sz[lane * 4] + q0.y * sz[lane * 4 + 1] + q1.x * sz[lane * 4 + 2] + q1.y * sz[lane * 4 + 3];
#pragma unroll
    for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) u[row] -= acc;
  }
}
__global__ void __launch_bounds__(256) fwd_step_kernel(const double* a, int64_t ld, int64_t k0, int64_t n_pad,
                                                       double* u, double* zout) {
  fwd_step_at(a, ld, k0, n_pad, u, zout, blockIdx.x);
}
// backward step k: alpha_k = T_kk^T z_k -> aout;  z[col] -= L[k-block, col]^T alpha_k for cols left of k (in place).
__global__ void __launch_bounds__(256) bwd_step_kernel(const double* a, int64_t ld, int64_t k0, double* z, double* aout) {
  __shared__ double sw[128], sa[128], part[256];
  const int tid = threadIdx.x;
  if (tid < 128) sw[tid] = z[k0 + tid];
  __syncthreads();
  const double* t = a + k0 * ld + k0;
  {                                                                 // column c = tid % 128, rows split in two halves
    const int c = tid & 127, h = tid >> 7;
    double acc = 0.0;
#pragma unroll 8
    for (int r = h * 64; r < h * 64 + 64; ++r) acc = fma(t[(int64_t)r * ld + c], sw[r], acc);
    part[tid] = acc;
  }
  __syncthreads();
  if (tid < 128) sa[tid] = part[tid] + part[tid + 128];
  __syncthreads();
  if (blockIdx.x == 0) { if (tid < 128) aout[k0 + tid] = sa[tid]; return; }
  const int64_t col = (int64_t)(blockIdx.x - 1) * 128 + (tid & 127);
  const int h = tid >> 7;
  const double* p = a + (k0 + h * 64) * ld + col;
  double acc = 0.0;
#pragma unroll 8
  for (int r = 0; r < 64; ++r) acc = fma(p[(int64_t)r * ld], sa[h * 64 + r], acc);
  part[tid] = acc;
  __syncthreads();
  if (tid < 128) z[col] -= part[tid] + part[tid + 128];
}

// ---------------------------------------------------------------------------------------
// Prediction epilogues.
// mean[m] = amp_cross * sum_n exp(-q(m,n)/2) alpha_n + y0*[m]  -- cross-covariance never stored.
template <int DIM>
__global__ void __launch_bounds__(256) stream_mean_kernel(const Cov cov, const double* x, const double* alpha, int64_t n,
                                                          const double* xnew, const double* new_y0, int64_t m, double* mean) {
  extern __shared__ double sh[];
  double* sx = sh; double* sy = sh + 1024; double* sa = sh + (DIM == 2 ? 2048 : 1024);
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  double gx = 0.0, gy = 0.0;
  if (i < m) { if (DIM == 1) gx = xnew[i]; else { gx = xnew[2 * i]; gy = xnew[2 * i + 1]; } }
  double acc = 0.0, acc2 = 0.0;
  for (int64_t c0 = 0; c0 < n; c0 += 1024) {
    __syncthreads();
    for (int j = threadIdx.x; j < 1024; j += blockDim.x) {
      const int64_t c = c0 + j;
      const bool in = c < n;
      if (DIM == 1) sx[j] = in ? x[c] : 0.0; else { sx[j] = in ? x[2 * c] : 0.0; sy[j] = in ? x[2 * c + 1] : 0.0; }
      sa[j] = in ? alpha[c] : 0.0;                  // zero weight beyond n
    }
    __syncthreads();
#pragma unroll 4
    for (int j = 0; j < 1024; j += 2) {
      double a0, a1;
      {
        const double dx = sx[j] - gx;
        if (DIM == 1) a0 = dx * dx * cov.h00;
        else { const double dy = sy[j] - gy; a0 = fma(dy * cov.h11, dy, fma(dx, cov.h00, dy * cov.h01) * dx); }
      }
      {
        const double dx = sx[j + 1] - gx;
        if (DIM == 1) a1 = dx * dx * cov.h00;
        else { const double dy = sy[j + 1] - gy; a1 = fma(dy * cov.h11, dy, fma(dx, cov.h00, dy * cov.h01) * dx); }
      }
      acc = fma(cgp_exp(a0), sa[j], acc); acc2 = fma(cgp_exp(a1), sa[j + 1], acc2);
    }
  }
  if (i < m) mean[i] = fma(cov.amp_cross, acc + acc2, new_y0 ? new_y0[i] : 0.0);
}
// var[m] = amp* - |v_m|^2 with v_m = row m of V (mc x n_pad): one warp per row.
__global__ void __launch_bounds__(256) row_norm_var_kernel(const double* v, int64_t ld, int64_t n_pad, int64_t rows,
                                                           double amp_star, double* var) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (r >= rows) return;
  const double* p = v + r * ld;
  double acc = 0.0, acc2 = 0.0;
  for (int64_t c = lane * 2; c < n_pad; c += 64) {
    const double2 u = *reinterpret_cast<const double2*>(p + c);
    acc = fma(u.x, u.x, acc); acc2 = fma(u.y, u.y, acc2);
  }
  acc += acc2;
#pragma unroll
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) var[r] = amp_star - acc;
}
__device__ __forceinline__ double block_dot_sq(const double* v, int64_t n) {   // |v|^2, valid in thread 0
  __shared__ double s[32];
  double acc = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) acc = fma(v[i], v[i], acc);
#pragma unroll
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    acc = threadIdx.x < (blockDim.x >> 5) ? s[threadIdx.x] : 0.0;
#pragma unroll
    for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  }
  return acc;
}
__global__ void dot_sq_kernel(const double* v, int64_t n, double* out) {      // out[0] = |v|^2 (one CTA)
  const double acc = block_dot_sq(v, n);
  if (threadIdx.x == 0) out[0] = acc;
}
__global__ void sum_kernel(const double* v, int64_t n, double* out) {         // out[0] = sum v (one CTA, fixed order)
  __shared__ double s[32];
  double acc = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) acc += v[i];
#pragma unroll
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    acc = threadIdx.x < (blockDim.x >> 5) ? s[threadIdx.x] : 0.0;
#pragma unroll
    for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (threadIdx.x == 0) out[0] = acc;
  }
}
// Mean function at the epochs on the device: the cubic B-spline scipy's InterpolatedUnivariateSpline holds
// (knots t[0..nt), coefficients c) evaluated as FITPACK does (splev.f: knot interval by search, clamped to the end
// intervals = polynomial extrapolation; fpbspl.f: de Boor recurrence; same operation order, no FMA contraction),
// plus the object's offset diff[b] (cosmogp/mean.py:28-31,84-90).  One thread per point; the object of a point
// comes from a binary search in the CSR offsets.
__global__ void __launch_bounds__(256) spline_mean_kernel(const double* __restrict__ t, const double* __restrict__ c, int nt,
                                                          const double* __restrict__ x, int64_t n_pts,
                                                          const int64_t* __restrict__ off, int64_t n_obj,
                                                          const double* __restrict__ diff, double* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_pts) return;
  const double arg = x[i];
  constexpr int K = 3, K1 = K + 1;
  const int nk1 = nt - K1;                       // 1-based: l in [K1, nk1] with t(l) <= arg < t(l+1) where possible
  int lo = K1, hi = nk1;                         // largest l in [lo, hi] with t(l) <= arg (lo when none)
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (t[mid - 1] <= arg) lo = mid; else hi = mid - 1;
  }
  const int l = lo;
  double h[K1 + 1], hh[K1];
  h[0] = 1.0;
#pragma unroll
  for (int j = 1; j <= K; ++j) {
#pragma unroll
    for (int q = 0; q < j; ++q) hh[q] = h[q];
    h[0] = 0.0;
#pragma unroll
    for (int q = 1; q <= j; ++q) {
      const double tli = t[l + q - 1], tlj = t[l + q - j - 1];
      if (tli == tlj) { h[q] = 0.0; continue; }
      const double f = __ddiv_rn(hh[q - 1], __dsub_rn(tli, tlj));
      h[q - 1] = __dadd_rn(h[q - 1], __dmul_rn(f, __dsub_rn(tli, arg)));
      h[q] = __dmul_rn(f, __dsub_rn(arg, tlj));
    }
  }
  double sp = 0.0;
#pragma unroll
  for (int j = 0; j < K1; ++j) sp = __dadd_rn(sp, __dmul_rn(c[l - K1 + j], h[j]));
  if (diff) {
    int64_t a = 0, b = n_obj - 1;                // object of point i: last b with off[b] <= i
    while (a < b) {
      const int64_t mid = (a + b + 1) >> 1;
      if (off[mid] <= i) a = mid; else b = mid - 1;
    }
    sp = __dadd_rn(sp, diff[a]);
  }
  out[i] = sp;
}

// Centred moments of a long vector, for scipy.stats.norm.fit of the pulls (cosmogp/pull.py:102) without a
// download: partial[2*blk] = sum (v - c), partial[2*blk+1] = sum (v - c)^2 over the block's contiguous
// segment (16-byte loads, HBM bound); a second one-CTA pass adds the partials in a fixed order.
__global__ void __launch_bounds__(256) moments_partial_kernel(const double* __restrict__ v, int64_t n, double c,
                                                              double* __restrict__ partial) {
  __shared__ double s1[8], s2[8];
  const int64_t per = ((n + gridDim.x - 1) / gridDim.x + 1) & ~(int64_t)1;      // even: segments stay 16-byte aligned
  const int64_t lo = (int64_t)blockIdx.x * per, hi = lo + per < n ? lo + per : n;
  double a1 = 0.0, a2 = 0.0, b1 = 0.0, b2 = 0.0;
  const bool aligned = (reinterpret_cast<uintptr_t>(v) & 15) == 0;
  int64_t i = lo + 2 * (int64_t)threadIdx.x;
  if (aligned) {
    for (; i + 1 < hi; i += 2 * blockDim.x) {
      const double2 w = *reinterpret_cast<const double2*>(v + i);
      const double d0 = w.x - c, d1 = w.y - c;
      a1 += d0; a2 = fma(d0, d0, a2); b1 += d1; b2 = fma(d1, d1, b2);
    }
    if (i < hi) { const double d0 = v[i] - c; a1 += d0; a2 = fma(d0, d0, a2); }
  } else {
    for (; i < hi; i += 2 * blockDim.x) {
      const double d0 = v[i] - c; a1 += d0; a2 = fma(d0, d0, a2);
      if (i + 1 < hi) { const double d1 = v[i + 1] - c; b1 += d1; b2 = fma(d1, d1, b2); }
    }
  }
  a1 += b1; a2 += b2;
#pragma unroll
  for (int o = 16; o; o >>= 1) { a1 += __shfl_xor_sync(0xffffffffu, a1, o); a2 += __shfl_xor_sync(0xffffffffu, a2, o); }
  if ((threadIdx.x & 31) == 0) { s1[threadIdx.x >> 5] = a1; s2[threadIdx.x >> 5] = a2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double t1 = 0.0, t2 = 0.0;
    for (int w = 0; w < 8; ++w) { t1 += s1[w]; t2 += s2[w]; }
    partial[2 * blockIdx.x] = t1; partial[2 * blockIdx.x + 1] = t2;
  }
}
__global__ void moments_final_kernel(const double* __restrict__ partial, int nblk, double* __restrict__ out) {
  __shared__ double s1[32], s2[32];
  double a1 = 0.0, a2 = 0.0;
  for (int i = threadIdx.x; i < nblk; i += blockDim.x) { a1 += partial[2 * i]; a2 += partial[2 * i + 1]; }
#pragma unroll
  for (int o = 16; o; o >>= 1) { a1 += __shfl_xor_sync(0xffffffffu, a1, o); a2 += __shfl_xor_sync(0xffffffffu, a2, o); }
  if ((threadIdx.x & 31) == 0) { s1[threadIdx.x >> 5] = a1; s2[threadIdx.x >> 5] = a2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double t1 = 0.0, t2 = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { t1 += s1[w]; t2 += s2[w]; }
    out[0] = t1; out[1] = t2;
  }
}
__global__ void potrf_setup_kernel(int64_t* blk_off, int64_t* blk_aoff, int nblk, int64_t ld) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k == 0) { blk_off[0] = 0; blk_off[1] = 128; }
  if (k < nblk) blk_aoff[k] = (int64_t)k * 128 * ld + (int64_t)k * 128;
}
__global__ void potrf_finish_kernel(const double* ld_blocks, const int* info_blocks, int nblk, double* logdet, int* info) {
  if (threadIdx.x == 0) {
    double s = 0.0; int bad = 0;
    for (int k = 0; k < nblk; ++k) { s += ld_blocks[k]; if (!bad && info_blocks[k]) bad = k * 128 + info_blocks[k]; }
    if (logdet) *logdet = bad ? nan("") : s;
    if (info) *info = bad;
  }
}
__global__ void residual_kernel(const double* y, const double* y0, int64_t n, int64_t n_pad, double* r) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_pad) r[i] = i < n ? y[i] - (y0 ? y0[i] : 0.0) : 0.0;
}
__global__ void ones_kernel(int64_t n, int64_t n_pad, double* v) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_pad) v[i] = i < n ? 1.0 : 0.0;
}
// v[r][c] = (r == c) for r < rows, c < cols (cols even): the identity rows the diag(K^-1) solve starts from.
__global__ void __launch_bounds__(256) identity_rows_kernel(double* v, int64_t ldv, int64_t rows, int64_t cols) {
  const int64_t half = cols / 2, total = rows * half;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = t / half, c = (t - r * half) * 2;
    *reinterpret_cast<double2*>(v + r * ldv + c) = make_double2(c == r ? 1.0 : 0.0, c + 1 == r ? 1.0 : 0.0);
  }
}
// Closed-form leave-one-out of one object, the formulas of the shared-memory path (cgp_small.cu TASK_LOO):
// d = diag(K^-1) arrives negated (row_norm_var_kernel with amp* = 0), alpha = K^-1 r; u = K^-1 1 and rsum = sum r
// for the recentred mode only (u == nullptr otherwise).  NaN everywhere when the factorisation failed.
__global__ void __launch_bounds__(256) loo_epilogue_kernel(const Cov cov, int64_t n, const double* __restrict__ y,
                                                           const double* __restrict__ m, const double* __restrict__ yerr,
                                                           const double* __restrict__ alpha, const double* __restrict__ negd,
                                                           const double* __restrict__ u, const double* __restrict__ rsum,
                                                           const int* __restrict__ info, double* pred, double* pvar,
                                                           double* pull, double* resid) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double rho = cov.amp_cross / cov.amp_auto;
  const double amp_star = cov.amp_auto + cov.nugget2;
  const double d = -negd[i];
  const double yv = y[i], mi = m ? m[i] : 0.0, r = yv - mi;
  const double ye = yerr ? yerr[i] : 0.0;
  double pr = mi + rho * (r - alpha[i] / d);
  if (u) {
    const double delta = (rsum[0] - r) / (double)(n - 1);
    pr += delta - delta * rho * (1.0 - u[i] / d);
  }
  double pv = fabs(amp_star - rho * rho * (cov.amp_auto + (ye * ye + cov.noise_const) - 1.0 / d));
  double res = pr - yv;
  double pl = res / sqrt(ye * ye + pv + cov.nugget2);
  if (*info) { pr = nan(""); pv = pr; res = pr; pl = pr; }
  if (pred) pred[i] = pr;
  if (pvar) pvar[i] = pv;
  if (resid) resid[i] = res;
  if (pull) pull[i] = pl;
}

// ---------------------------------------------------------------------------------------
// Grouped likelihood of many large objects, each with its own hyperparameters (large_ll_grouped).  Every kernel
// below runs the body of its single-object counterpart on one object at a time, so an object's arithmetic does not
// depend on the other objects of its launch.
struct GroupObj {
  const double* x; const double* y; const double* y0; const double* yerr;
  double* a;                 // n_pad x n_pad covariance -> blocked factor (leading dimension n_pad)
  double* u;                 // residual y - y0 (n_pad, zero padded), consumed by the forward sweep
  double* z;                 // z = L^-1 (y - y0)
  int64_t n, n_pad;
  int64_t io;                // position in `order`: compact hyperparameters, nugget, ll and info
  int64_t cta0;              // first CTA of the object in the covariance launch
};
struct GroupHyp {
  const double* hyp_obj; const double* nugget_obj; double nugget, floor; unsigned flags;
};

template <int DIM>
__device__ __forceinline__ Cov group_cov(const GroupHyp& h, int64_t io) {
  return cov_from_hyp(DIM, h.hyp_obj + io * (DIM == 1 ? 2 : 4), h.nugget_obj ? h.nugget_obj[io] : h.nugget, h.floor, h.flags);
}

// Covariance of every object of a wave (the layout of cov_build_kernel) and its residual.  Object i owns
// n_pad * ceil(n_pad / 256) CTAs from objs[i].cta0 on: one row, 256 columns each.
template <int DIM>
__global__ void __launch_bounds__(128) cov_build_grouped_kernel(const GroupObj* __restrict__ objs, const int n_obj,
                                                                const GroupHyp h) {
  const int64_t t = blockIdx.x;
  int lo = 0, hi = n_obj - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (objs[mid].cta0 <= t) lo = mid; else hi = mid - 1;
  }
  const GroupObj& o = objs[lo];
  const int64_t per_row = (o.n_pad + 255) / 256;
  const int64_t local = t - o.cta0, r = local / per_row, chunk = local - r * per_row;
  CovArgs a;
  a.dim = DIM; a.cov = group_cov<DIM>(h, o.io); a.autocov = 1;
  a.xc = o.x; a.n = o.n; a.xr = o.x; a.m = o.n; a.yerr = o.yerr;
  a.out = o.a; a.ld = o.n_pad; a.rows_pad = o.n_pad; a.cols_pad = o.n_pad;
  cov_build_at<DIM>(a, r, (chunk * 128 + threadIdx.x) * 2);
  if (chunk == 0 && threadIdx.x == 0) o.u[r] = r < o.n ? o.y[r] - (o.y0 ? o.y0[r] : 0.0) : 0.0;   // residual_kernel
}

// Forward sweep step k of the objects objs[0 .. gridDim.y): CTA x of object y runs fwd_step_kernel's CTA x.
__global__ void __launch_bounds__(256) fwd_step_grouped_kernel(const GroupObj* __restrict__ objs, const int64_t k0) {
  const GroupObj& o = objs[blockIdx.y];
  if ((int64_t)blockIdx.x >= 1 + (o.n_pad - k0 - 128 + 63) / 64) return;
  fwd_step_at(o.a, o.n_pad, k0, o.n_pad, o.u, o.z, blockIdx.x);
}

// One CTA per object: quad = |z|^2 (dot_sq_kernel), log det and info summed over the blocks in the order of
// potrf_finish_kernel (block k of object i at ld_blocks[koff[k] + i]), and ll with the operation order of
// dense.LargeObject.factor: -0.5 * ((quad + logdet) + n log 2 pi).  NaN where the factorisation failed.
__global__ void __launch_bounds__(1024) ll_finish_grouped_kernel(const GroupObj* __restrict__ objs,
                                                                 const double* __restrict__ ld_blocks,
                                                                 const int* __restrict__ info_blocks,
                                                                 const int64_t* __restrict__ koff,
                                                                 double* __restrict__ ll, int* __restrict__ info) {
  const int i = blockIdx.x;
  const GroupObj& o = objs[i];
  const double quad = block_dot_sq(o.z, o.n_pad);
  if (threadIdx.x == 0) {
    const int nblk = (int)(o.n_pad / 128);
    double s = 0.0; int bad = 0;
    for (int k = 0; k < nblk; ++k) {
      s += ld_blocks[koff[k] + i];
      const int ik = info_blocks[koff[k] + i];
      if (!bad && ik) bad = k * 128 + ik;
    }
    const double log_2pi = 1.8378770664093453;                 // math.log(2 * math.pi)
    ll[o.io] = bad ? nan("") : __dmul_rn(-0.5, __dadd_rn(__dadd_rn(quad, s), __dmul_rn((double)o.n, log_2pi)));
    info[o.io] = bad;
  }
}

}  // namespace

// =========================================================================================
int launch_gemm_nt(const GemmArgs& g, cudaStream_t stream) {
  if (g.m % 128 || g.n % BN || g.k % BK || g.m <= 0 || g.n <= 0 || g.k <= 0) return (int)cudaErrorInvalidValue;
  static bool init[16] = {false};                         // function attributes are per device
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 16) return (int)cudaErrorInvalidDevice;
  if (!init[dev]) {
    cudaError_t e = cudaFuncSetAttribute(gemm_nt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GEMM_SMEM);
    if (e != cudaSuccess) return (int)e;
    init[dev] = true;
  }
  const int64_t tm = g.m / BM, tn = g.n / BN;
  const int64_t t128 = g.m / 128;
  const int64_t tiles = g.lower_only ? t128 * (t128 + 1) : tm * tn;       // two 64-row halves per 128x128 block
  gemm_nt_kernel<<<(unsigned)tiles, GEMM_THREADS, GEMM_SMEM, stream>>>(g);
  count_launch();
  return (int)cudaGetLastError();
}

int large_cov_build(int dim, const Cov& cov, int autocov, const double* xc, int64_t n, const double* xr, int64_t m,
                    const double* yerr, double* out, int64_t ld, int64_t rows_pad, int64_t cols_pad, cudaStream_t st) {
  CovArgs a;
  a.dim = dim; a.cov = cov; a.autocov = autocov; a.xc = xc; a.n = n; a.xr = xr; a.m = m; a.yerr = yerr;
  a.out = out; a.ld = ld; a.rows_pad = rows_pad; a.cols_pad = cols_pad;
  if (rows_pad <= 0 || cols_pad <= 0) return 0;
  if (rows_pad > 2147483647) return (int)cudaErrorInvalidValue;
  dim3 grid((unsigned)((cols_pad / 2 + 1 + 127) / 128), 1);
  // grid.y is limited to 65535: sweep the rows in slabs
  for (int64_t r0 = 0; r0 < rows_pad; r0 += 65535) {
    CovArgs s = a;
    const int64_t rows = rows_pad - r0 < 65535 ? rows_pad - r0 : 65535;
    s.out = out + r0 * ld;
    s.xr = xr + r0 * dim;
    s.m = m - r0 > 0 ? m - r0 : 0;
    s.rows_pad = rows;
    if (autocov) {                                  // diagonal test uses absolute indices: shift the columns instead
      // (auto-covariances larger than 65535 rows are built slab by slab with a column origin)
      if (r0) return (int)cudaErrorInvalidValue;
    }
    grid.y = (unsigned)rows;
    if (dim == 1) cov_build_kernel<1><<<grid, 128, 0, st>>>(s); else cov_build_kernel<2><<<grid, 128, 0, st>>>(s);
    count_launch();
  }
  return (int)cudaGetLastError();
}

// In-place blocked Cholesky of the lower triangle of a (n_pad x n_pad, n_pad % 128 == 0).
// On exit: strictly-lower 128-blocks = L, diagonal blocks = (L_kk)^-1 with zeros above the
// diagonal, logdet_blocks[k] = sum log pivots of block k, info_blocks[k] = failing pivot (0 = ok).
int large_potrf(double* a, int64_t n_pad, int64_t ld, double* logdet_out, int* info_out, cudaStream_t st) {
  const int nblk = (int)(n_pad / 128);
  // stream-ordered scratch: per-block log det / info and the two tiny CSR arrays the block kernel reads
  char* scratch = nullptr;
  const size_t bytes = (size_t)nblk * (sizeof(double) + sizeof(int) + sizeof(int64_t)) + 4 * sizeof(int64_t) + 64;
  cudaError_t ce = cudaMallocAsync((void**)&scratch, bytes, st);
  if (ce != cudaSuccess) return (int)ce;
  double* logdet_blocks = (double*)scratch;
  int64_t* blk_aoff = (int64_t*)(scratch + (size_t)nblk * sizeof(double));
  int64_t* blk_off = blk_aoff + nblk;
  int* info_blocks = (int*)(blk_off + 2);
  potrf_setup_kernel<<<(nblk + 127) / 128, 128, 0, st>>>(blk_off, blk_aoff, nblk, ld);
  count_launch();
  int rc = 0;
  // Look-ahead: the diagonal blocks and panels of the NEXT pair of block columns (two CTAs + skinny
  // GEMMs, latency bound) run on a high-priority side stream while the main stream applies the
  // current pair to the rest of the trailing matrix; only the next pair's columns are updated first.
  constexpr int MAX_DEV = 16;
  static cudaStream_t sides[MAX_DEV] = {nullptr};          // per device of this process
  static cudaEvent_t evs[MAX_DEV][2] = {{nullptr, nullptr}};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= MAX_DEV) { cudaFreeAsync(scratch, st); return (int)cudaErrorInvalidDevice; }
  if (!sides[dev]) {
    int lo = 0, hi = 0;
    cudaDeviceGetStreamPriorityRange(&lo, &hi);
    if (cudaStreamCreateWithPriority(&sides[dev], cudaStreamNonBlocking, hi) != cudaSuccess) {
      cudaFreeAsync(scratch, st);
      return (int)cudaGetLastError();
    }
    cudaEventCreateWithFlags(&evs[dev][0], cudaEventDisableTiming);
    cudaEventCreateWithFlags(&evs[dev][1], cudaEventDisableTiming);
  }
  cudaStream_t side = sides[dev];
  cudaEvent_t ev_col = evs[dev][0], ev_panel = evs[dev][1];
  auto factor_panel = [&](int k, cudaStream_t s_) -> int {      // diag block k -> T_kk, then L_ik = A_ik T_kk^T
    const int64_t k0 = (int64_t)k * 128;
    SmallArgs s; memset(&s, 0, sizeof s);
    s.n_obj = 1; s.off = blk_off;                  // {0, 128}
    s.amat = a; s.aoff = blk_aoff + k; s.lda = ld;
    s.moff = blk_aoff + k; s.mld = ld; s.linv = a;
    s.logdet = logdet_blocks + k; s.info = info_blocks + k;
    s.cov.amp_auto = 1.0; s.cov.amp_cross = 1.0;
    int e = launch_small(TASK_MATRICES, 1, 128, s, s_);
    if (e) return e;
    const int64_t rest = n_pad - k0 - 128;
    if (rest <= 0) return 0;
    GemmArgs p;                                      // in place, one tile column
    p.a = a + (k0 + 128) * ld + k0; p.lda = ld;
    p.b = a + k0 * ld + k0; p.ldb = ld;
    p.c = a + (k0 + 128) * ld + k0; p.ldc = ld;
    p.m = (int)rest; p.n = 128; p.k = 128; p.alpha = 1.0; p.beta = 0.0; p.lower_only = 0;
    return launch_gemm_nt(p, s_);
  };
  // Two block columns form one 256-wide pair: the trailing update then runs with K = 256 (one pass
  // over C for two panels, and a deeper K loop per tile).
  auto factor_pair = [&](int p, cudaStream_t s_) -> int {
    const int k = 2 * p;
    int e = factor_panel(k, s_);
    if (e || k + 1 >= nblk) return e;
    const int64_t k0 = (int64_t)k * 128;
    const double* panel = a + (k0 + 128) * ld + k0;            // L[k+1:, k]
    GemmArgs c;                                                // block column k+1 (with its diagonal block)
    c.a = panel; c.lda = ld; c.b = panel; c.ldb = ld;
    c.c = a + (k0 + 128) * ld + (k0 + 128); c.ldc = ld;
    c.m = (int)(n_pad - k0 - 128); c.n = 128; c.k = 128; c.alpha = -1.0; c.beta = 1.0; c.lower_only = 0;
    if ((e = launch_gemm_nt(c, s_))) return e;
    return factor_panel(k + 1, s_);
  };
  const int npair = (nblk + 1) / 2;
  rc = factor_pair(0, st);
  for (int p = 0; p + 1 < npair && !rc; ++p) {
    const int64_t k0 = (int64_t)p * 256;
    const int64_t rest = n_pad - k0 - 256;             // rows below the pair
    const double* w = a + (k0 + 256) * ld + k0;        // L[2p+2:, 2p..2p+1], K = 256 contiguous
    GemmArgs c;                                        // the next pair's block columns first
    c.a = w; c.lda = ld; c.b = w; c.ldb = ld;
    c.c = a + (k0 + 256) * ld + (k0 + 256); c.ldc = ld;
    c.m = (int)rest; c.n = 128; c.k = 256; c.alpha = -1.0; c.beta = 1.0; c.lower_only = 0;
    if ((rc = launch_gemm_nt(c, st))) break;
    if (rest > 128) {
      c.a = w + 128 * ld; c.b = w + 128 * ld;
      c.c = a + (k0 + 384) * ld + (k0 + 384);
      c.m = (int)(rest - 128);
      if ((rc = launch_gemm_nt(c, st))) break;
    }
    cudaEventRecord(ev_col, st);
    cudaStreamWaitEvent(side, ev_col, 0);
    if ((rc = factor_pair(p + 1, side))) break;
    cudaEventRecord(ev_panel, side);
    if (rest > 256) {                                  // the rest of the trailing matrix, lower triangle
      GemmArgs u;
      u.a = w + 256 * ld; u.lda = ld; u.b = u.a; u.ldb = ld;
      u.c = a + (k0 + 512) * ld + (k0 + 512); u.ldc = ld;
      u.m = (int)(rest - 256); u.n = (int)(rest - 256); u.k = 256; u.alpha = -1.0; u.beta = 1.0; u.lower_only = 1;
      if ((rc = launch_gemm_nt(u, st))) break;
    }
    cudaStreamWaitEvent(st, ev_panel, 0);
  }
  if (rc) {                                            // error exit: the side stream may still be using the scratch
    cudaEventRecord(ev_panel, side);
    cudaStreamWaitEvent(st, ev_panel, 0);
  }
  potrf_finish_kernel<<<1, 32, 0, st>>>(logdet_blocks, info_blocks, nblk, logdet_out, info_out);
  count_launch();
  cudaFreeAsync(scratch, st);
  return rc ? rc : (int)cudaGetLastError();
}

// v <- L^-1 v (forward) then, if backward, v <- L^-T v.  z_out (optional) receives L^-1 v.
// One fused launch per 128-block and direction; a stream-ordered scratch vector holds z.
int large_potrs(const double* a, int64_t n_pad, int64_t ld, double* v, double* z_out, int backward, cudaStream_t st) {
  const int nblk = (int)(n_pad / 128);
  double* z = nullptr;
  cudaError_t ce = cudaMallocAsync((void**)&z, n_pad * sizeof(double), st);
  if (ce != cudaSuccess) return (int)ce;
  for (int k = 0; k < nblk; ++k) {
    const int64_t k0 = (int64_t)k * 128;
    const int64_t rest = n_pad - k0 - 128;
    fwd_step_kernel<<<(unsigned)(1 + (rest + 63) / 64), 256, 0, st>>>(a, ld, k0, n_pad, v, z);
  }
  count_launch(nblk);
  if (z_out) cudaMemcpyAsync(z_out, z, n_pad * sizeof(double), cudaMemcpyDeviceToDevice, st);
  if (backward) {
    for (int k = nblk - 1; k >= 0; --k) bwd_step_kernel<<<(unsigned)(1 + k), 256, 0, st>>>(a, ld, (int64_t)k * 128, z, v);
    count_launch(nblk);
  } else {
    cudaMemcpyAsync(v, z, n_pad * sizeof(double), cudaMemcpyDeviceToDevice, st);
  }
  cudaFreeAsync(z, st);
  return (int)cudaGetLastError();
}

// alpha = L^-T z for a vector z that already holds L^-1 r (in place).
int large_potrs_backward(const double* a, int64_t n_pad, int64_t ld, double* v, cudaStream_t st) {
  const int nblk = (int)(n_pad / 128);
  double* z = nullptr;
  cudaError_t ce = cudaMallocAsync((void**)&z, n_pad * sizeof(double), st);
  if (ce != cudaSuccess) return (int)ce;
  cudaMemcpyAsync(z, v, n_pad * sizeof(double), cudaMemcpyDeviceToDevice, st);
  for (int k = nblk - 1; k >= 0; --k) bwd_step_kernel<<<(unsigned)(1 + k), 256, 0, st>>>(a, ld, (int64_t)k * 128, z, v);
  count_launch(nblk);
  cudaFreeAsync(z, st);
  return (int)cudaGetLastError();
}

// V (rows x n_pad, row-major, leading dimension ldv) holds cross-covariance rows h_m on entry
// and v_m = L^-1 h_m on exit: blocked left-looking solve, all FLOPs in gemm_nt.  rows % 128 == 0.
int large_trsm_rows(const double* a, int64_t n_pad, int64_t ld, double* v, int64_t ldv, int64_t rows, cudaStream_t st) {
  const int nblk = (int)(n_pad / 128);
  for (int k = 0; k < nblk; ++k) {
    const int64_t k0 = (int64_t)k * 128;
    int e;
    if (k > 0) {                                     // V[:,k] -= V[:,0:k] L[k,0:k]^T
      GemmArgs u;
      u.a = v; u.lda = ldv; u.b = a + k0 * ld; u.ldb = ld; u.c = v + k0; u.ldc = ldv;
      u.m = (int)rows; u.n = 128; u.k = (int)k0; u.alpha = -1.0; u.beta = 1.0; u.lower_only = 0;
      if ((e = launch_gemm_nt(u, st))) return e;
    }
    GemmArgs p;                                      // V[:,k] = V[:,k] T_kk^T
    p.a = v + k0; p.lda = ldv; p.b = a + k0 * ld + k0; p.ldb = ld; p.c = v + k0; p.ldc = ldv;
    p.m = (int)rows; p.n = 128; p.k = 128; p.alpha = 1.0; p.beta = 0.0; p.lower_only = 0;
    if ((e = launch_gemm_nt(p, st))) return e;
  }
  return 0;
}

int large_stream_mean(int dim, const Cov& cov, const double* x, const double* alpha, int64_t n,
                      const double* xnew, const double* new_y0, int64_t m, double* mean, cudaStream_t st) {
  if (m <= 0) return 0;
  const unsigned grid = (unsigned)((m + 255) / 256);
  if (dim == 1) stream_mean_kernel<1><<<grid, 256, 2 * 1024 * sizeof(double), st>>>(cov, x, alpha, n, xnew, new_y0, m, mean);
  else stream_mean_kernel<2><<<grid, 256, 3 * 1024 * sizeof(double), st>>>(cov, x, alpha, n, xnew, new_y0, m, mean);
  count_launch();
  return (int)cudaGetLastError();
}
int large_row_var(const double* v, int64_t ldv, int64_t n_pad, int64_t rows, double amp_star, double* var, cudaStream_t st) {
  if (rows <= 0) return 0;
  row_norm_var_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, st>>>(v, ldv, n_pad, rows, amp_star, var);
  count_launch();
  return (int)cudaGetLastError();
}
int large_dot_sq(const double* v, int64_t n, double* out, cudaStream_t st) {
  dot_sq_kernel<<<1, 1024, 0, st>>>(v, n, out); count_launch(); return (int)cudaGetLastError();
}
int large_spline_mean(const double* t, const double* c, int nt, const double* x, int64_t n_pts, const int64_t* off,
                      int64_t n_obj, const double* diff, double* out, cudaStream_t st) {
  if (n_pts <= 0) return 0;
  spline_mean_kernel<<<(unsigned)((n_pts + 255) / 256), 256, 0, st>>>(t, c, nt, x, n_pts, off, n_obj, diff, out);
  count_launch();
  return (int)cudaGetLastError();
}
int large_moments(const double* v, int64_t n, double center, double* out2, cudaStream_t st) {
  const int nblk = n < (int64_t)1 << 16 ? 1 : 148 * 8;
  double* partial = nullptr;
  cudaError_t ce = cudaMallocAsync((void**)&partial, sizeof(double) * 2 * nblk, st);
  if (ce != cudaSuccess) return (int)ce;
  moments_partial_kernel<<<nblk, 256, 0, st>>>(v, n, center, partial);
  moments_final_kernel<<<1, 256, 0, st>>>(partial, nblk, out2);
  count_launch(2);
  cudaFreeAsync(partial, st);
  return (int)cudaGetLastError();
}
// sum of the per-object log-likelihoods in a FIXED order (block b sums its contiguous segment with 256 strided
// lanes + a tree, one thread adds the block partials in index order) and the number of objects with info != 0.
__global__ void __launch_bounds__(256) ll_total_partial_kernel(const double* __restrict__ ll, const int* __restrict__ info,
                                                               int64_t n, double* __restrict__ partial) {
  __shared__ double s1[8], s2[8];
  const int64_t per = (n + gridDim.x - 1) / gridDim.x;
  const int64_t lo = (int64_t)blockIdx.x * per, hi = lo + per < n ? lo + per : n;
  double a = 0.0, b = 0.0;
  for (int64_t i = lo + threadIdx.x; i < hi; i += blockDim.x) { a += ll[i]; b += info[i] != 0 ? 1.0 : 0.0; }
#pragma unroll
  for (int o = 16; o; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); }
  if ((threadIdx.x & 31) == 0) { s1[threadIdx.x >> 5] = a; s2[threadIdx.x >> 5] = b; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double t1 = 0.0, t2 = 0.0;
    for (int w = 0; w < 8; ++w) { t1 += s1[w]; t2 += s2[w]; }
    if (gridDim.x == 1) { partial[0] = t1; partial[1] = t2; }           // `partial` is the output itself
    else { partial[2 * blockIdx.x] = t1; partial[2 * blockIdx.x + 1] = t2; }
  }
}
__global__ void ll_total_final_kernel(const double* __restrict__ partial, int nblk, double* __restrict__ out) {
  if (threadIdx.x == 0) {
    double t1 = 0.0, t2 = 0.0;
    for (int i = 0; i < nblk; ++i) { t1 += partial[2 * i]; t2 += partial[2 * i + 1]; }
    out[0] = t1; out[1] = t2;
  }
}
int large_ll_total(const double* ll, const int* info, int64_t n, double* out2, cudaStream_t st) {
  if (n <= 16384) {                                      // one block: one launch
    ll_total_partial_kernel<<<1, 256, 0, st>>>(ll, info, n, out2); count_launch();
    return (int)cudaGetLastError();
  }
  int nblk = (int)((n + 8191) / 8192); if (nblk > 256) nblk = 256;
  double* partial = nullptr;
  cudaError_t e = cudaMallocAsync((void**)&partial, sizeof(double) * 2 * nblk, st);
  if (e != cudaSuccess) return (int)e;
  ll_total_partial_kernel<<<nblk, 256, 0, st>>>(ll, info, n, partial);
  ll_total_final_kernel<<<1, 32, 0, st>>>(partial, nblk, out2);
  count_launch(2);
  cudaFreeAsync(partial, st);
  return (int)cudaGetLastError();
}
// Predictive covariance of one object from V = rows L^-1 e(x*_m, .):  C = amp_auto K(g,g) + nugget^2 I - amp_cross^2 V V^T
// (cosmogp/Gaussian_process.py:356-361).  One CTA per 64 x 64 block: V_i^T and V_j^T staged in shared memory
// (k-major, so that a thread's four rows are 32 contiguous bytes), 4 x 4 outputs per thread, K(g_i, g_j) generated
// on the fly.  8 bytes written per ~64 FMAs + one exp: bound by the HBM write of the M x M matrices.
template <int DIM>
__global__ void __launch_bounds__(256) cov_gram_kernel(Cov cov, const double* __restrict__ grid, const int64_t* __restrict__ goff,
                                                       int64_t m_shared, const double* __restrict__ v, int ldv,
                                                       const int* __restrict__ info, double* __restrict__ out,
                                                       const int64_t* __restrict__ coff) {
  extern __shared__ __align__(16) double sm[];
  const int64_t b = blockIdx.z;
  const int64_t g0 = goff ? goff[b] : 0;
  const int64_t m = goff ? goff[b + 1] - g0 : m_shared;
  const int64_t i0 = (int64_t)blockIdx.y * 64, j0 = (int64_t)blockIdx.x * 64;
  if (i0 >= m || j0 >= m) return;
  const int64_t row0 = goff ? g0 : b * m_shared;            // first row of this object's V / grid block
  constexpr int LDS_ = 66;                                  // k-major rows of 64 + 2: 16-byte aligned, transposing stores spread over banks
  double* vi = sm; double* vj = sm + (size_t)ldv * LDS_;    // [k][64]
  for (int e = threadIdx.x; e < 64 * ldv; e += 256) {
    const int r = e / ldv, k = e - r * ldv;                 // coalesced reads of V rows
    vi[k * LDS_ + r] = (i0 + r < m) ? v[(row0 + i0 + r) * ldv + k] : 0.0;
    vj[k * LDS_ + r] = (j0 + r < m) ? v[(row0 + j0 + r) * ldv + k] : 0.0;
  }
  __syncthreads();
  const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
  double acc[4][4];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[r][c] = 0.0;
  for (int k = 0; k < ldv; ++k) {
    const double2 a0 = *reinterpret_cast<const double2*>(vi + k * LDS_ + ty * 4), a1 = *reinterpret_cast<const double2*>(vi + k * LDS_ + ty * 4 + 2);
    const double2 b0 = *reinterpret_cast<const double2*>(vj + k * LDS_ + tx * 4), b1 = *reinterpret_cast<const double2*>(vj + k * LDS_ + tx * 4 + 2);
    const double av[4] = {a0.x, a0.y, a1.x, a1.y}, bv[4] = {b0.x, b0.y, b1.x, b1.y};
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[r][c] = fma(av[r], bv[c], acc[r][c]);
  }
  const bool bad = info && info[b] != 0;
  const double a2 = cov.amp_cross * cov.amp_cross;
  double* ob = out + (coff ? coff[b] : b * m_shared * m_shared);
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int64_t i = i0 + ty * 4 + r;
    if (i >= m) continue;
    const double xi = grid[(g0 + i) * DIM], yi = DIM == 2 ? grid[(g0 + i) * DIM + 1] : 0.0;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int64_t j = j0 + tx * 4 + c;
      if (j >= m) continue;
      const double dx = xi - grid[(g0 + j) * DIM];
      double q = dx * dx * cov.h00;
      if (DIM == 2) { const double dy = yi - grid[(g0 + j) * DIM + 1]; q = fma(dy * cov.h11, dy, fma(dx, cov.h00, dy * cov.h01) * dx); }
      double kk = (i == j) ? cov.amp_auto + cov.nugget2 : cov.amp_auto * cgp_exp(q);
      ob[i * m + j] = bad ? nan("") : fma(-a2, acc[r][c], kk);
    }
  }
}
int large_cov_gram(int dim, const Cov& cov, const double* grid, const int64_t* goff, int64_t m_shared, int64_t n_obj,
                   const double* v, int ldv, const int* info, double* out, const int64_t* coff, cudaStream_t st) {
  if (n_obj <= 0 || m_shared <= 0) return 0;               // m_shared: the largest grid of the chunk (the grid's x / y extent)
  const size_t smem = (size_t)2 * 66 * ldv * sizeof(double);
  const unsigned nb = (unsigned)((m_shared + 63) / 64);
  if (n_obj > 65535) return (int)cudaErrorInvalidValue;
  const dim3 g(nb, nb, (unsigned)n_obj);
  cudaError_t e;
  if (dim == 1) {
    e = cudaFuncSetAttribute(cov_gram_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    cov_gram_kernel<1><<<g, 256, smem, st>>>(cov, grid, goff, goff ? 0 : m_shared, v, ldv, info, out, coff);
  } else {
    e = cudaFuncSetAttribute(cov_gram_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    cov_gram_kernel<2><<<g, 256, smem, st>>>(cov, grid, goff, goff ? 0 : m_shared, v, ldv, info, out, coff);
  }
  count_launch();
  return (int)cudaGetLastError();
}
int large_sum(const double* v, int64_t n, double* out, cudaStream_t st) {
  sum_kernel<<<1, 1024, 0, st>>>(v, n, out); count_launch(); return (int)cudaGetLastError();
}
int large_residual(const double* y, const double* y0, int64_t n, int64_t n_pad, double* r, cudaStream_t st) {
  residual_kernel<<<(unsigned)((n_pad + 255) / 256), 256, 0, st>>>(y, y0, n, n_pad, r); count_launch();
  return (int)cudaGetLastError();
}

// negd[m] = -(K^-1)_mm = -|L^-1 e_m|^2 for m < n_pad, without forming K^-1.  Identity rows e_m, m in [r0, r0 + c),
// are solved in chunks of c = chunk_rows rows staged in v (c x n_pad, leading dimension n_pad): row i of the chunk
// becomes (L^-1 e_{r0+i})^T, which is zero left of column r0 + i, so the chunk only spans columns [r0, n_pad) and
// block column k only involves the chunk's row blocks <= k.  Right-looking over pairs of block columns, as in
// large_potrf: finish block columns k, k+1 (T_kk^T, one 128-wide update, T_{k+1}^T), then
// V[:, k+2:] -= V[:, k:k+2] L[k+2:, k:k+2]^T with K = 256.  N^3/3 FLOPs in all, every one in gemm_nt.
int large_diag_inv(const double* a, int64_t n_pad, int64_t ld, double* v, int64_t chunk_rows, double* negd, cudaStream_t st) {
  const int nblk = (int)(n_pad / 128);
  int e = 0;
  auto gemm = [&](const double* A, const double* B, int64_t ldb, double* C, int64_t m, int64_t n, int k, double alpha,
                  double beta) {
    GemmArgs g;
    g.a = A; g.lda = n_pad; g.b = B; g.ldb = ldb; g.c = C; g.ldc = n_pad;
    g.m = (int)m; g.n = (int)n; g.k = k; g.alpha = alpha; g.beta = beta; g.lower_only = 0;
    return launch_gemm_nt(g, st);
  };
  for (int64_t r0 = 0; r0 < n_pad && !e; r0 += chunk_rows) {
    const int64_t c = n_pad - r0 < chunk_rows ? n_pad - r0 : chunk_rows;
    const int kb0 = (int)(r0 / 128);
    const int64_t w = n_pad - r0;
    double* vc = v + r0;                               // column r0 of the chunk's rows
    auto rows = [&](int k) { const int64_t r = (int64_t)(k - kb0 + 1) * 128; return r < c ? r : c; };
    int64_t blocks = (c * (w / 2) + 255) / 256;
    identity_rows_kernel<<<(unsigned)(blocks < 148 * 16 ? blocks : 148 * 16), 256, 0, st>>>(vc, n_pad, c, w);
    count_launch();
    for (int k = kb0; k < nblk && !e; k += 2) {
      const int64_t j0 = (int64_t)(k - kb0) * 128;     // block column k inside the chunk
      const double* lk = a + (int64_t)k * 128 * ld + (int64_t)k * 128;
      if ((e = gemm(vc + j0, lk, ld, vc + j0, rows(k), 128, 128, 1.0, 0.0))) break;                 // V_k T_kk^T
      if (k + 1 == nblk) break;
      if ((e = gemm(vc + j0, lk + 128 * ld, ld, vc + j0 + 128, rows(k), 128, 128, -1.0, 1.0))) break;  // -= V_k L_{k+1,k}^T
      if ((e = gemm(vc + j0 + 128, lk + 128 * ld + 128, ld, vc + j0 + 128, rows(k + 1), 128, 128, 1.0, 0.0))) break;
      if (k + 2 < nblk)
        e = gemm(vc + j0, lk + 256 * ld, ld, vc + j0 + 256, rows(k + 1), n_pad - (int64_t)(k + 2) * 128, 256, -1.0, 1.0);
    }
    if (!e) e = large_row_var(vc, n_pad, w, c, 0.0, negd + r0, st);
  }
  return e ? e : (int)cudaGetLastError();
}

// Leave-one-out pulls of one factored object (see cgp_large_loo_dev).  Stream-ordered scratch: alpha, -diag(K^-1),
// K^-1 1 (n_pad each) and sum r.
int large_loo(const double* a, int64_t n, int64_t n_pad, int64_t ld, const Cov& cov, const double* y, const double* m,
              const double* yerr, int recenter, const int* info, double* vwork, int64_t chunk_rows,
              double* pred, double* pvar, double* pull, double* resid, cudaStream_t st) {
  double* ws = nullptr;
  cudaError_t ce = cudaMallocAsync((void**)&ws, (3 * n_pad + 2) * sizeof(double), st);
  if (ce != cudaSuccess) return (int)ce;
  double* alpha = ws;
  double* negd = ws + n_pad;
  double* u = recenter ? ws + 2 * n_pad : nullptr;
  double* rsum = ws + 3 * n_pad;
  int e = large_residual(y, m, n, n_pad, alpha, st);
  if (!e && recenter) e = large_sum(alpha, n, rsum, st);
  if (!e) e = large_potrs(a, n_pad, ld, alpha, nullptr, 1, st);
  if (!e && recenter) {
    ones_kernel<<<(unsigned)((n_pad + 255) / 256), 256, 0, st>>>(n, n_pad, u); count_launch();
    e = large_potrs(a, n_pad, ld, u, nullptr, 1, st);
  }
  if (!e) e = large_diag_inv(a, n_pad, ld, vwork, chunk_rows, negd, st);
  if (!e) {
    loo_epilogue_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(cov, n, y, m, yerr, alpha, negd, u, rsum, info,
                                                                     pred, pvar, pull, resid);
    count_launch();
    e = (int)cudaGetLastError();
  }
  cudaFreeAsync(ws, st);
  return e;
}

int64_t large_ll_ws_doubles(int64_t n) {
  const int64_t np = n <= 0 ? 128 : (n + 127) / 128 * 128;
  return np * np + 2 * np + 2 * (np / 128);          // covariance, residual, z, per-block log det and info
}

// Log-likelihoods of the objects order[0 .. n_active) (object ids; NULL: 0 .. n_active), object order[j] with the
// hyperparameters of row j, by the blocked factorisation of large_potrf run for all objects of a wave at once.
// Consecutive objects are packed into waves of at most work_doubles (each object's part: large_ll_ws_doubles); inside
// a wave they are sorted by block count, so that the objects taking part in any step are a prefix of the wave.  Per
// wave: one covariance launch; per pair of block columns two diagonal-block launches (launch_small in matrix-source
// mode) and four grouped GEMM launches, with the shapes, tile split and alpha / beta large_potrf uses for each object
// alone (the next pair's columns and the lower trailing update touch disjoint tiles, so they share one launch); one
// forward-sweep launch per block; one epilogue.  The schedule (object descriptors, GEMM problems, block offsets)
// crosses to the device in one copy into stream-ordered scratch.  The caller checks that every object fits.
int large_ll_grouped(int dim, const int64_t* off, const double* x, const double* y, const double* y0, const double* yerr,
                     const double* hyp_obj, const double* nugget_obj, double nugget, double floor, unsigned flags,
                     const int* order, int64_t n_active, double* ll, int* info, double* work, int64_t work_doubles,
                     cudaStream_t st) {
  struct Item { int64_t j, b, n, n_pad; int nblk; };
  std::vector<std::vector<Item>> waves;
  {
    std::vector<Item> cur; int64_t used = 0;
    for (int64_t j = 0; j < n_active; ++j) {
      Item it; it.j = j; it.b = order ? order[j] : j; it.n = off[it.b + 1] - off[it.b];
      it.n_pad = it.n <= 0 ? 128 : (it.n + 127) / 128 * 128; it.nblk = (int)(it.n_pad / 128);
      const int64_t need = large_ll_ws_doubles(it.n);
      if (!cur.empty() && (used + need > work_doubles || cur.size() >= 65535)) { waves.push_back(cur); cur.clear(); used = 0; }
      cur.push_back(it); used += need;
    }
    if (!cur.empty()) waves.push_back(cur);
  }
  std::vector<char> tab;
  auto put = [&](const void* p, size_t bytes) {
    const size_t o = (tab.size() + 15) & ~(size_t)15;
    tab.resize(o + bytes);
    memcpy(tab.data() + o, p, bytes);
    return o;
  };
  struct Launch { int kind; int64_t grid, count, k0; size_t t0, t1, t2; double* ldb; int* infob; };
  enum { L_COV, L_DIAG, L_GEMM, L_FWD, L_FIN };
  std::vector<Launch> launches;
  size_t w_max = 0;
  for (auto& w : waves) w_max = std::max(w_max, w.size());
  std::vector<int64_t> csr(w_max + 1);
  for (size_t i = 0; i <= w_max; ++i) csr[i] = (int64_t)i * 128;
  const size_t t_csr = put(csr.data(), csr.size() * sizeof(int64_t));

  for (auto& w : waves) {
    std::stable_sort(w.begin(), w.end(), [](const Item& p, const Item& q) { return p.nblk > q.nblk; });
    const int W = (int)w.size(), nb_max = w[0].nblk;
    std::vector<GroupObj> objs(W);
    std::vector<int64_t> ld(W), koff(nb_max + 1, 0);
    int64_t cur = 0, cta = 0;
    for (int i = 0; i < W; ++i) {
      const Item& it = w[i];
      const int64_t o0 = off[it.b], np = it.n_pad;
      GroupObj& g = objs[i];
      g.x = x + dim * o0; g.y = y + o0; g.y0 = y0 ? y0 + o0 : nullptr; g.yerr = yerr ? yerr + o0 : nullptr;
      g.a = work + cur; g.u = g.a + np * np; g.z = g.u + np;
      g.n = it.n; g.n_pad = np; g.io = it.j; g.cta0 = cta;
      cur += np * np + 2 * np; cta += np * ((np + 255) / 256);
      ld[i] = np;
    }
    if (cta > 2147483647LL) return (int)cudaErrorInvalidValue;
    auto count = [&](int k) { int c = 0; while (c < W && w[c].nblk > k) ++c; return c; };   // objects with block k
    for (int k = 0; k < nb_max; ++k) koff[k + 1] = koff[k] + count(k);
    double* ldb = work + cur;
    int* infob = reinterpret_cast<int*>(work + cur + koff[nb_max]);
    const size_t t_objs = put(objs.data(), W * sizeof(GroupObj));
    const size_t t_ld = put(ld.data(), W * sizeof(int64_t));
    const size_t t_koff = put(koff.data(), koff.size() * sizeof(int64_t));
    launches.push_back({L_COV, cta, W, 0, t_objs, 0, 0, nullptr, nullptr});

    auto diag = [&](int k) {
      const int c = count(k);
      std::vector<int64_t> aoff(c);
      for (int i = 0; i < c; ++i) aoff[i] = (objs[i].a - work) + (int64_t)k * 128 * ld[i] + (int64_t)k * 128;
      launches.push_back({L_DIAG, c, c, 0, put(aoff.data(), c * sizeof(int64_t)), t_ld, 0, ldb + koff[k], infob + koff[k]});
    };
    std::vector<GemmArgs> probs;
    auto gemm = [&](double* A, double* B, double* C, int64_t ldx, int64_t m, int64_t n, int k, double alpha, double beta,
                    int lower) {
      GemmArgs g;
      g.a = A; g.b = B; g.c = C; g.lda = ldx; g.ldb = ldx; g.ldc = ldx;
      g.m = (int)m; g.n = (int)n; g.k = k; g.alpha = alpha; g.beta = beta; g.lower_only = lower;
      probs.push_back(g);
    };
    auto flush = [&]() -> int {
      if (probs.empty()) return 0;
      std::vector<int> start(probs.size() + 1, 0);
      for (size_t q = 0; q < probs.size(); ++q) {
        const GemmArgs& g = probs[q];
        const int64_t t128 = g.m / 128;
        const int64_t tiles = g.lower_only ? t128 * (t128 + 1) : (int64_t)(g.m / BM) * (g.n / BN);
        if (start[q] + tiles > 2147483647LL) return (int)cudaErrorInvalidValue;
        start[q + 1] = start[q] + (int)tiles;
      }
      const size_t tp = put(probs.data(), probs.size() * sizeof(GemmArgs));
      const size_t ts = put(start.data(), start.size() * sizeof(int));
      launches.push_back({L_GEMM, start.back(), (int64_t)probs.size(), 0, tp, ts, 0, nullptr, nullptr});
      probs.clear();
      return 0;
    };
    int e = 0;
    for (int p = 0; 2 * p < nb_max && !e; ++p) {
      const int k = 2 * p;
      const int64_t k0 = (int64_t)p * 256;
      diag(k);
      for (int i = 0; i < W && w[i].nblk > k + 1; ++i) {            // panel of block column k: L_ik = A_ik T_kk^T
        const int64_t np = ld[i];
        double* a = objs[i].a;
        gemm(a + (k0 + 128) * np + k0, a + k0 * np + k0, a + (k0 + 128) * np + k0, np, np - k0 - 128, 128, 128, 1.0, 0.0, 0);
      }
      if ((e = flush())) break;
      for (int i = 0; i < W && w[i].nblk > k + 1; ++i) {            // block column k+1 -= L[k+1:, k] L[k+1, k]^T
        const int64_t np = ld[i];
        double* a = objs[i].a;
        double* panel = a + (k0 + 128) * np + k0;
        gemm(panel, panel, a + (k0 + 128) * np + (k0 + 128), np, np - k0 - 128, 128, 128, -1.0, 1.0, 0);
      }
      if ((e = flush())) break;
      if (nb_max <= k + 1) break;
      diag(k + 1);
      const int64_t k1 = k0 + 128;
      for (int i = 0; i < W && w[i].nblk > k + 2; ++i) {            // panel of block column k+1
        const int64_t np = ld[i];
        double* a = objs[i].a;
        gemm(a + (k1 + 128) * np + k1, a + k1 * np + k1, a + (k1 + 128) * np + k1, np, np - k1 - 128, 128, 128, 1.0, 0.0, 0);
      }
      if ((e = flush())) break;
      for (int i = 0; i < W && w[i].nblk > k + 2; ++i) {            // the pair applied to what lies right of it, K = 256
        const int64_t np = ld[i], rest = np - k0 - 256;
        double* a = objs[i].a;
        double* wp = a + (k0 + 256) * np + k0;
        gemm(wp, wp, a + (k0 + 256) * np + (k0 + 256), np, rest, 128, 256, -1.0, 1.0, 0);
        if (rest > 128) gemm(wp + 128 * np, wp + 128 * np, a + (k0 + 384) * np + (k0 + 384), np, rest - 128, 128, 256, -1.0, 1.0, 0);
        if (rest > 256) gemm(wp + 256 * np, wp + 256 * np, a + (k0 + 512) * np + (k0 + 512), np, rest - 256, rest - 256, 256, -1.0, 1.0, 1);
      }
      e = flush();
    }
    if (e) return e;
    for (int k = 0; k < nb_max; ++k)
      launches.push_back({L_FWD, 1 + (ld[0] - (int64_t)k * 128 - 128 + 63) / 64, count(k), (int64_t)k * 128, t_objs, 0, 0,
                          nullptr, nullptr});
    launches.push_back({L_FIN, W, W, 0, t_objs, t_koff, 0, ldb, infob});
  }

  static bool init[16] = {false};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 16) return (int)cudaErrorInvalidDevice;
  if (!init[dev]) {
    cudaError_t ce = cudaFuncSetAttribute(gemm_nt_grouped_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GEMM_SMEM);
    if (ce != cudaSuccess) return (int)ce;
    init[dev] = true;
  }
  char* td = nullptr;
  cudaError_t ce = cudaMallocAsync((void**)&td, tab.size(), st);
  if (ce == cudaSuccess) ce = cudaMemcpyAsync(td, tab.data(), tab.size(), cudaMemcpyHostToDevice, st);
  if (ce != cudaSuccess) { if (td) cudaFreeAsync(td, st); return (int)ce; }
  GroupHyp h; h.hyp_obj = hyp_obj; h.nugget_obj = nugget_obj; h.nugget = nugget; h.floor = floor; h.flags = flags;
  int e = 0;
  for (const Launch& l : launches) {
    const GroupObj* objs = reinterpret_cast<const GroupObj*>(td + l.t0);
    switch (l.kind) {
      case L_COV:
        if (dim == 1) cov_build_grouped_kernel<1><<<(unsigned)l.grid, 128, 0, st>>>(objs, (int)l.count, h);
        else cov_build_grouped_kernel<2><<<(unsigned)l.grid, 128, 0, st>>>(objs, (int)l.count, h);
        break;
      case L_DIAG: {
        SmallArgs s; memset(&s, 0, sizeof s);
        s.n_obj = l.count; s.off = reinterpret_cast<const int64_t*>(td + t_csr);
        s.amat = work; s.aoff = reinterpret_cast<const int64_t*>(td + l.t0); s.ld_obj = reinterpret_cast<const int64_t*>(td + l.t1);
        s.moff = s.aoff; s.linv = work;
        s.logdet = l.ldb; s.info = l.infob;
        s.cov.amp_auto = 1.0; s.cov.amp_cross = 1.0;
        e = launch_small(TASK_MATRICES, 1, 128, s, st);  // counts its own launch
        break;
      }
      case L_GEMM:
        gemm_nt_grouped_kernel<<<(unsigned)l.grid, GEMM_THREADS, GEMM_SMEM, st>>>(
            reinterpret_cast<const GemmArgs*>(td + l.t0), reinterpret_cast<const int*>(td + l.t1), (int)l.count);
        break;
      case L_FWD:
        fwd_step_grouped_kernel<<<dim3((unsigned)l.grid, (unsigned)l.count), 256, 0, st>>>(objs, l.k0);
        break;
      case L_FIN:
        ll_finish_grouped_kernel<<<(unsigned)l.grid, 1024, 0, st>>>(objs, l.ldb, l.infob,
                                                                    reinterpret_cast<const int64_t*>(td + l.t1), ll, info);
        break;
    }
    if (l.kind != L_DIAG) count_launch();
    if (e) break;
  }
  cudaFreeAsync(td, st);
  return e ? e : (int)cudaGetLastError();
}

}  // namespace cgp
