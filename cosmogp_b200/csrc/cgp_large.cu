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
__device__ __forceinline__ void bwd_step_at(const double* a, int64_t ld, int64_t k0, double* z, double* aout, const int cta) {
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
  if (cta == 0) { if (tid < 128) aout[k0 + tid] = sa[tid]; return; }
  const int64_t col = (int64_t)(cta - 1) * 128 + (tid & 127);
  const int h = tid >> 7;
  const double* p = a + (k0 + h * 64) * ld + col;
  double acc = 0.0;
#pragma unroll 8
  for (int r = 0; r < 64; ++r) acc = fma(p[(int64_t)r * ld], sa[h * 64 + r], acc);
  part[tid] = acc;
  __syncthreads();
  if (tid < 128) z[col] -= part[tid] + part[tid + 128];
}
__global__ void __launch_bounds__(256) bwd_step_kernel(const double* a, int64_t ld, int64_t k0, double* z, double* aout) {
  bwd_step_at(a, ld, k0, z, aout, blockIdx.x);
}

// ---------------------------------------------------------------------------------------
// Prediction epilogues.
// mean[m] = amp_cross * sum_n exp(-q(m,n)/2) alpha_n + y0*[m]  -- cross-covariance never stored.  CTA `cta` takes grid
// rows [256 cta, 256 cta + 256); sh: 1024 staged columns of x (two rows of them in 2D) and alpha.
template <int DIM>
__device__ __forceinline__ void stream_mean_at(double* sh, const Cov& cov, const double* x, const double* alpha, int64_t n,
                                               const double* xnew, const double* new_y0, int64_t m, double* mean,
                                               const int64_t cta) {
  double* sx = sh; double* sy = sh + 1024; double* sa = sh + (DIM == 2 ? 2048 : 1024);
  const int64_t i = cta * blockDim.x + threadIdx.x;
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
template <int DIM>
__global__ void __launch_bounds__(256) stream_mean_kernel(const Cov cov, const double* x, const double* alpha, int64_t n,
                                                          const double* xnew, const double* new_y0, int64_t m, double* mean) {
  extern __shared__ double sh[];
  stream_mean_at<DIM>(sh, cov, x, alpha, n, xnew, new_y0, m, mean, blockIdx.x);
}
// var[m] = amp* - |v_m|^2 with v_m = row m of V (mc x n_pad): one warp per row, rows [8 cta, 8 cta + 8).
__device__ __forceinline__ void row_norm_var_at(const double* v, int64_t ld, int64_t n_pad, int64_t rows, double amp_star,
                                                double* var, const int64_t cta) {
  const int lane = threadIdx.x & 31;
  const int64_t r = cta * 8 + (threadIdx.x >> 5);
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
__global__ void __launch_bounds__(256) row_norm_var_kernel(const double* v, int64_t ld, int64_t n_pad, int64_t rows,
                                                           double amp_star, double* var) {
  row_norm_var_at(v, ld, n_pad, rows, amp_star, var, blockIdx.x);
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
__device__ __forceinline__ double block_sum(const double* v, int64_t n) {     // sum v in a fixed order, valid in thread 0
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
  }
  return acc;
}
__global__ void sum_kernel(const double* v, int64_t n, double* out) {         // out[0] = sum v (one CTA)
  const double acc = block_sum(v, n);
  if (threadIdx.x == 0) out[0] = acc;
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
// Pairs t0, t0 + step, .. of the rows * cols / 2 pairs of entries.
__device__ __forceinline__ void identity_rows_at(double* v, int64_t ldv, int64_t rows, int64_t cols, int64_t t0, int64_t step) {
  const int64_t half = cols / 2, total = rows * half;
  for (int64_t t = t0; t < total; t += step) {
    const int64_t r = t / half, c = (t - r * half) * 2;
    *reinterpret_cast<double2*>(v + r * ldv + c) = make_double2(c == r ? 1.0 : 0.0, c + 1 == r ? 1.0 : 0.0);
  }
}
__global__ void __launch_bounds__(256) identity_rows_kernel(double* v, int64_t ldv, int64_t rows, int64_t cols) {
  identity_rows_at(v, ldv, rows, cols, (int64_t)blockIdx.x * blockDim.x + threadIdx.x, (int64_t)gridDim.x * blockDim.x);
}
// Closed-form leave-one-out at point i of one object, the formulas of the shared-memory path (cgp_small.cu TASK_LOO):
// d = diag(K^-1) arrives negated (row_norm_var_at with amp* = 0), alpha = K^-1 r; u = K^-1 1 and rsum = sum r for the
// recentred mode only (u == nullptr otherwise).  NaN everywhere when the factorisation failed (bad != 0).
__device__ __forceinline__ void loo_epilogue_at(const Cov& cov, int64_t n, const double* __restrict__ y,
                                                const double* __restrict__ m, const double* __restrict__ yerr,
                                                const double* __restrict__ alpha, const double* __restrict__ negd,
                                                const double* __restrict__ u, const double* __restrict__ rsum, const int bad,
                                                double* pred, double* pvar, double* pull, double* resid, const int64_t i) {
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
  if (bad) { pr = nan(""); pv = pr; res = pr; pl = pr; }
  if (pred) pred[i] = pr;
  if (pvar) pvar[i] = pv;
  if (resid) resid[i] = res;
  if (pull) pull[i] = pl;
}
__global__ void __launch_bounds__(256) loo_epilogue_kernel(const Cov cov, int64_t n, const double* __restrict__ y,
                                                           const double* __restrict__ m, const double* __restrict__ yerr,
                                                           const double* __restrict__ alpha, const double* __restrict__ negd,
                                                           const double* __restrict__ u, const double* __restrict__ rsum,
                                                           const int* __restrict__ info, double* pred, double* pvar,
                                                           double* pull, double* resid) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  loo_epilogue_at(cov, n, y, m, yerr, alpha, negd, u, rsum, *info, pred, pvar, pull, resid, i);
}

// ---------------------------------------------------------------------------------------
// Grouped pipelines of large objects (large_ll_grouped, large_predict_grouped, large_loo_grouped, large_cov_grouped).
// Every kernel below runs the body of its single-object counterpart on one object at a time, so an object's arithmetic
// does not depend on the other objects of its launch.

// What build_grouped_kernel reads of an object of a grouped likelihood, prediction or leave-one-out: its covariance
// function, built on the host with the floor (as cgp_cov_matrix_dev's make_cov builds it), its data (y0: the mean
// subtracted from y, may be null; yerr may be null) and where A, the residual and the ones vector go.
struct BuildObj {
  Cov cov;
  const double* x; const double* y; const double* y0; const double* yerr;
  double* a;                 // n_pad x n_pad covariance -> blocked factor (leading dimension n_pad)
  double* r;                 // residual y - y0 (n_pad, zero padded), consumed by the forward sweep
  double* ones;              // ones vector, consumed by the forward sweep (leave-one-out recentred mode; null otherwise)
  int64_t n, n_pad;
  int64_t cta;               // first CTA of the object in the build launch
};
// One object of a grouped likelihood (large_ll_grouped).
struct GroupObj : BuildObj {
  double* z;                 // z = L^-1 (y - y0)
  int64_t io;                // position in `order`: ll and info
};
// Per-object hyperparameter rows in device memory, from which cov_gram_kernel<OBJHYP> builds each object's Cov.
struct GroupHyp {
  const double* hyp_obj; const double* nugget_obj; double nugget, floor; unsigned flags;
};

// The last object of objs[0 .. n_obj) whose first CTA (field f) is <= t: the object that owns CTA t of a grouped launch
// (objects without CTAs share their successor's first CTA and are skipped).
template <class O>
__device__ __forceinline__ const O& owner(const O* __restrict__ objs, const int n_obj, const int64_t t, int64_t O::*f) {
  int lo = 0, hi = n_obj - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (objs[mid].*f <= t) lo = mid; else hi = mid - 1;
  }
  return objs[lo];
}

// The first failing pivot of object i of a wave, as potrf_finish_kernel reports it: k * 128 + info of its first block k
// with info != 0 (block k at infob[koff[k] + i]), 0 when every block is positive definite.
__device__ __forceinline__ int first_bad_pivot(const int* __restrict__ infob, const int64_t* __restrict__ koff, int i, int nblk) {
  for (int k = 0; k < nblk; ++k) {
    const int ik = infob[koff[k] + i];
    if (ik) return k * 128 + ik;
  }
  return 0;
}

template <int DIM>
__device__ __forceinline__ Cov group_cov(const GroupHyp& h, int64_t io) {
  return cov_from_hyp(DIM, h.hyp_obj + io * (DIM == 1 ? 2 : 4), h.nugget_obj ? h.nugget_obj[io] : h.nugget, h.floor, h.flags);
}

// A = K(x, x) + noise (the layout of cov_build_kernel), the residual (residual_kernel) and, where `ones` is set, the
// ones vector (ones_kernel) of every object of a wave.  Object i owns n_pad * ceil(n_pad / 256) CTAs from objs[i].cta
// on: one row, 256 columns each.  O: the pipeline's descriptor, which sets the stride of objs.
template <int DIM, class O>
__global__ void __launch_bounds__(128) build_grouped_kernel(const O* __restrict__ objs, const int n_obj) {
  const int64_t t = blockIdx.x;
  const BuildObj& o = owner<O>(objs, n_obj, t, &O::cta);
  const int64_t per_row = (o.n_pad + 255) / 256;
  const int64_t local = t - o.cta, r = local / per_row, chunk = local - r * per_row;
  if (chunk == 0 && threadIdx.x == 0) {
    o.r[r] = r < o.n ? o.y[r] - (o.y0 ? o.y0[r] : 0.0) : 0.0;      // residual_kernel
    if (o.ones) o.ones[r] = r < o.n ? 1.0 : 0.0;                   // ones_kernel
  }
  CovArgs a;
  a.dim = DIM; a.cov = o.cov; a.autocov = 1;
  a.xc = o.x; a.n = o.n; a.xr = o.x; a.m = o.n; a.yerr = o.yerr;
  a.out = o.a; a.ld = o.n_pad; a.rows_pad = o.n_pad; a.cols_pad = o.n_pad;
  cov_build_at<DIM>(a, r, (chunk * 128 + threadIdx.x) * 2);
}

// Forward sweep step k of the objects 0 .. gridDim.y, gridDim.z right-hand sides each (the descriptors of one object
// consecutive): CTA x of right-hand side z of object y runs fwd_step_kernel's CTA x.
template <class Obj>
__global__ void __launch_bounds__(256) fwd_step_grouped_kernel(const Obj* __restrict__ objs, const int64_t k0) {
  const Obj& o = objs[blockIdx.y * gridDim.z + blockIdx.z];
  if ((int64_t)blockIdx.x >= 1 + (o.n_pad - k0 - 128 + 63) / 64) return;
  fwd_step_at(o.a, o.n_pad, k0, o.n_pad, o.r, o.z, blockIdx.x);
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
    double s = 0.0;
    for (int k = 0; k < nblk; ++k) s += ld_blocks[koff[k] + i];
    const int bad = first_bad_pivot(info_blocks, koff, i, nblk);
    const double log_2pi = 1.8378770664093453;                 // math.log(2 * math.pi)
    ll[o.io] = bad ? nan("") : __dmul_rn(-0.5, __dadd_rn(__dadd_rn(quad, s), __dmul_rn((double)o.n, log_2pi)));
    info[o.io] = bad;
  }
}

// One object of a grouped predictive covariance (large_cov_grouped).  `cov` (with the floor, for A) and `cov_g` (without
// it, for H and K**) come from the host, as cgp_cov_matrix_dev's do: the device's cov_from_hyp may contract the 2D
// metric differently.
struct CovObj {
  Cov cov, cov_g;
  const double* x; const double* yerr; const double* g;   // epochs, their errors (may be null), grid
  double* a;                 // n_pad x n_pad covariance -> blocked factor
  double* v;                 // m_pad x n_pad: H = K(g, x) -> V = rows of L^-1 H^T
  double* c;                 // m_pad x m_pad: K(g, g) + nugget^2 I -> C
  double* out;               // the object's m x m block of the packed output
  int64_t n, n_pad, m, m_pad;
  int64_t io;                // position in `order`: info
  int64_t cta0;              // first CTA of the object in the build launch
};

// The three builds of dense.predictive_covariance (cgp_cov_matrix_dev's arguments) for every object of a wave:
// A = K(x, x) + noise, H = K(g, x) and K** = K(g, g) + nugget^2 I.  Object i owns (n_pad + m_pad) * ceil(n_pad / 256)
// + m_pad * ceil(m_pad / 256) CTAs from objs[i].cta0 on: one row of one matrix, 256 columns each.
template <int DIM>
__global__ void __launch_bounds__(128) cov3_build_grouped_kernel(const CovObj* __restrict__ objs, const int n_obj) {
  const int64_t t = blockIdx.x;
  const CovObj& o = owner(objs, n_obj, t, &CovObj::cta0);
  const int64_t pn = (o.n_pad + 255) / 256, pm = (o.m_pad + 255) / 256;
  int64_t local = t - o.cta0, per_row;
  CovArgs a;
  a.dim = DIM; a.cov = o.cov_g;
  if (local < o.n_pad * pn) {                                     // A: auto-covariance of the epochs with y_err
    per_row = pn;
    a.cov = o.cov;
    a.autocov = 1; a.xc = o.x; a.n = o.n; a.xr = o.x; a.m = o.n; a.yerr = o.yerr;
    a.out = o.a; a.ld = o.n_pad; a.rows_pad = o.n_pad; a.cols_pad = o.n_pad;
  } else if ((local -= o.n_pad * pn) < o.m_pad * pn) {           // H: grid rows against the epochs, zero padding
    per_row = pn;
    a.autocov = 0; a.xc = o.x; a.n = o.n; a.xr = o.g; a.m = o.m; a.yerr = nullptr;
    a.out = o.v; a.ld = o.n_pad; a.rows_pad = o.m_pad; a.cols_pad = o.n_pad;
  } else {                                                        // K**: auto-covariance of the grid, no y_err
    local -= o.m_pad * pn;
    per_row = pm;
    a.autocov = 1; a.xc = o.g; a.n = o.m; a.xr = o.g; a.m = o.m; a.yerr = nullptr;
    a.out = o.c; a.ld = o.m_pad; a.rows_pad = o.m_pad; a.cols_pad = o.m_pad;
  }
  const int64_t r = local / per_row, chunk = local - r * per_row;
  cov_build_at<DIM>(a, r, (chunk * 128 + threadIdx.x) * 2);
}

// Object blockIdx.y of a wave: its info (first_bad_pivot) and its leading m x m block of C packed to `out`, all NaN
// where info != 0.
__global__ void __launch_bounds__(256) cov_pack_grouped_kernel(const CovObj* __restrict__ objs, const int* __restrict__ infob,
                                                               const int64_t* __restrict__ koff, int* __restrict__ info) {
  const int i = blockIdx.y;
  const CovObj& o = objs[i];
  __shared__ int bad_s;
  if (threadIdx.x == 0) {
    const int bad = first_bad_pivot(infob, koff, i, (int)(o.n_pad / 128));
    bad_s = bad;
    if (blockIdx.x == 0) info[o.io] = bad;
  }
  __syncthreads();
  const bool bad = bad_s != 0;
  const int64_t m = o.m, mm = m * m;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < mm; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = e / m;
    o.out[e] = bad ? nan("") : o.c[r * o.m_pad + (e - r * m)];
  }
}

// One object of a grouped prediction (large_predict_grouped).  `cov_g` (without the floor, for the mean, H and the
// variance) comes from the host, as the make_cov calls of LargeObject.factor / cgp_large_predict_dev build it.
struct PredObj : BuildObj {
  Cov cov_g;
  const double* g; const double* new_y0;   // grid (m points) and the mean function on it (may be null)
  double* z;                 // L^-1 (y - y0), consumed by the backward sweep
  double* alpha;             // K^-1 (y - y0)
  double* mean; double* var; // the object's m outputs
  int64_t m;
  int64_t io;                // position in `order`: info
  int64_t cta_mean;          // first CTA of the object in the mean launch
};
// One object's rows [r0, r0 + rows) of one variance pass.
struct PassObj {
  Cov cov_g;
  const double* x; const double* g;       // epochs; grid row r0
  double* v;                 // rows_pad x n_pad: H -> V
  double* var;               // output row r0
  int64_t n, n_pad, rows, rows_pad;
  int64_t cta_h, cta_var;    // first CTA of the object in the H build and in the variance launch
};

// Backward sweep launch s of the objects 0 .. gridDim.y, gridDim.z right-hand sides each (as fwd_step_grouped_kernel):
// right-hand side z of object y runs bwd_step_kernel's CTA x of its block n_pad / 128 - 1 - s.
template <class Obj>
__global__ void __launch_bounds__(256) bwd_step_grouped_kernel(const Obj* __restrict__ objs, const int64_t s) {
  const Obj& o = objs[blockIdx.y * gridDim.z + blockIdx.z];
  const int64_t k = o.n_pad / 128 - 1 - s;
  if ((int64_t)blockIdx.x > k) return;
  bwd_step_at(o.a, o.n_pad, k * 128, o.z, o.alpha, blockIdx.x);
}

// stream_mean_kernel for every object of a wave: object i owns ceil(m / 256) CTAs from cta_mean on.
template <int DIM>
__global__ void __launch_bounds__(256) stream_mean_grouped_kernel(const PredObj* __restrict__ objs, const int n_obj) {
  extern __shared__ double sh[];
  const int64_t t = blockIdx.x;
  const PredObj& o = owner(objs, n_obj, t, &PredObj::cta_mean);
  stream_mean_at<DIM>(sh, o.cov_g, o.x, o.alpha, o.n, o.g, o.new_y0, o.m, o.mean, t - o.cta_mean);
}

// H = K(grid rows of the pass, x) of every object of a pass, zero padded as large_cov_build pads it: rows_pad *
// ceil(n_pad / 256) CTAs per object.
template <int DIM>
__global__ void __launch_bounds__(128) pass_build_grouped_kernel(const PassObj* __restrict__ objs, const int n_obj) {
  const int64_t t = blockIdx.x;
  const PassObj& o = owner(objs, n_obj, t, &PassObj::cta_h);
  const int64_t per_row = (o.n_pad + 255) / 256;
  const int64_t local = t - o.cta_h, r = local / per_row, chunk = local - r * per_row;
  CovArgs a;
  a.dim = DIM; a.cov = o.cov_g; a.autocov = 0;
  a.xc = o.x; a.n = o.n; a.xr = o.g; a.m = o.rows; a.yerr = nullptr;
  a.out = o.v; a.ld = o.n_pad; a.rows_pad = o.rows_pad; a.cols_pad = o.n_pad;
  cov_build_at<DIM>(a, r, (chunk * 128 + threadIdx.x) * 2);
}

// var = (amp_auto + nugget^2) - |v|^2 for the rows of a pass (row_norm_var_kernel): ceil(rows / 8) CTAs per object.
__global__ void __launch_bounds__(256) row_var_grouped_kernel(const PassObj* __restrict__ objs, const int n_obj) {
  const int64_t t = blockIdx.x;
  const PassObj& o = owner(objs, n_obj, t, &PassObj::cta_var);
  row_norm_var_at(o.v, o.n_pad, o.n_pad, o.rows, o.cov_g.amp_auto + o.cov_g.nugget2, o.var, t - o.cta_var);
}

// Object blockIdx.y of a wave: its info (first_bad_pivot) and NaN over its mean and variance rows where info != 0.
__global__ void __launch_bounds__(256) pred_finish_grouped_kernel(const PredObj* __restrict__ objs, const int* __restrict__ infob,
                                                                  const int64_t* __restrict__ koff, int* __restrict__ info) {
  const int i = blockIdx.y;
  const PredObj& o = objs[i];
  __shared__ int bad_s;
  if (threadIdx.x == 0) {
    const int bad = first_bad_pivot(infob, koff, i, (int)(o.n_pad / 128));
    bad_s = bad;
    if (blockIdx.x == 0) info[o.io] = bad;
  }
  __syncthreads();
  if (!bad_s) return;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < o.m; e += (int64_t)gridDim.x * blockDim.x) {
    o.mean[e] = nan("");
    if (o.var) o.var[e] = nan("");
  }
}

// One object of a grouped leave-one-out (large_loo_grouped); y0 is the mean m, as cgp_large_loo_dev takes it.
struct LooObj : BuildObj {
  double* alpha;             // K^-1 r
  double* kinv1;             // K^-1 1 (recentred mode; null otherwise)
  double* negd;              // -diag(K^-1)
  double* rsum;              // sum r
  double* pred; double* pvar; double* pull; double* resid;   // the object's n outputs (each may be null)
  int64_t io;                // position in `order`: info
  int64_t cta_epi;           // first CTA of the object in the epilogue launch
};
// One right-hand side of the sweeps: r -> z = L^-1 r (forward), z -> alpha = L^-T z (backward).
struct SolveObj { double* a; double* r; double* z; double* alpha; int64_t n_pad; };
// One object's pass of the diag(K^-1) solve: `rows` identity rows of width w staged at v (leading dimension ld), their
// negated squared norms to negd.
struct DiagObj { double* v; int64_t ld, w, rows; double* negd; int64_t cta; };

// sum r of object blockIdx.x (sum_kernel, 1024 threads).
__global__ void __launch_bounds__(1024) sum_grouped_kernel(const LooObj* __restrict__ objs) {
  const LooObj& o = objs[blockIdx.x];
  const double s = block_sum(o.r, o.n);
  if (threadIdx.x == 0) *o.rsum = s;
}

// The identity rows of object blockIdx.y of a diag(K^-1) pass (identity_rows_kernel).
__global__ void __launch_bounds__(256) identity_rows_grouped_kernel(const DiagObj* __restrict__ objs) {
  const DiagObj& o = objs[blockIdx.y];
  identity_rows_at(o.v, o.ld, o.rows, o.w, (int64_t)blockIdx.x * blockDim.x + threadIdx.x, (int64_t)gridDim.x * blockDim.x);
}

// -|row|^2 of the rows of a diag(K^-1) pass (row_norm_var_kernel with amp* = 0): ceil(rows / 8) CTAs per object.
__global__ void __launch_bounds__(256) diag_norm_grouped_kernel(const DiagObj* __restrict__ objs, const int n_obj) {
  const int64_t t = blockIdx.x;
  const DiagObj& o = owner(objs, n_obj, t, &DiagObj::cta);
  row_norm_var_at(o.v, o.ld, o.w, o.rows, 0.0, o.negd, t - o.cta);
}

// loo_epilogue_kernel for every object of a wave: object i owns max(1, ceil(n / 256)) CTAs from cta_epi on; its first
// CTA writes info (first_bad_pivot).
__global__ void __launch_bounds__(256) loo_finish_grouped_kernel(const LooObj* __restrict__ objs, const int n_obj,
                                                                 const int* __restrict__ infob, const int64_t* __restrict__ koff,
                                                                 int* __restrict__ info) {
  const int64_t t = blockIdx.x;
  const LooObj& o = owner(objs, n_obj, t, &LooObj::cta_epi);
  __shared__ int bad_s;
  if (threadIdx.x == 0) {
    const int bad = first_bad_pivot(infob, koff, (int)(&o - objs), (int)(o.n_pad / 128));
    bad_s = bad;
    if (t == o.cta_epi) info[o.io] = bad;
  }
  __syncthreads();
  const int64_t i = (t - o.cta_epi) * blockDim.x + threadIdx.x;
  if (i < o.n)
    loo_epilogue_at(o.cov, o.n, o.y, o.y0, o.yerr, o.alpha, o.negd, o.kinv1, o.rsum, bad_s, o.pred, o.pvar, o.pull, o.resid, i);
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
// OBJHYP: object b's CTAs build their own Cov from h (group_cov of row b) instead of reading `cov`.
template <int DIM, bool OBJHYP>
__global__ void __launch_bounds__(256) cov_gram_kernel(Cov cov, const double* __restrict__ grid, const int64_t* __restrict__ goff,
                                                       int64_t m_shared, const double* __restrict__ v, int ldv,
                                                       const int* __restrict__ info, double* __restrict__ out,
                                                       const int64_t* __restrict__ coff, const GroupHyp h) {
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
  if constexpr (OBJHYP) cov = group_cov<DIM>(h, b);
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
template <int DIM, bool OBJHYP>
static cudaError_t launch_cov_gram(dim3 g, size_t smem, cudaStream_t st, const Cov& cov, const double* grid, const int64_t* goff,
                                   int64_t m_shared, const double* v, int ldv, const int* info, double* out, const int64_t* coff,
                                   const GroupHyp& h) {
  cudaError_t e = cudaFuncSetAttribute(cov_gram_kernel<DIM, OBJHYP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  cov_gram_kernel<DIM, OBJHYP><<<g, 256, smem, st>>>(cov, grid, goff, goff ? 0 : m_shared, v, ldv, info, out, coff, h);
  return cudaSuccess;
}
int large_cov_gram(int dim, const Cov& cov, const double* hyp_obj, const double* nugget_obj, double nugget, unsigned flags,
                   const double* grid, const int64_t* goff, int64_t m_shared, int64_t n_obj,
                   const double* v, int ldv, const int* info, double* out, const int64_t* coff, cudaStream_t st) {
  if (n_obj <= 0 || m_shared <= 0) return 0;               // m_shared: the largest grid of the chunk (the grid's x / y extent)
  const size_t smem = (size_t)2 * 66 * ldv * sizeof(double);
  const unsigned nb = (unsigned)((m_shared + 63) / 64);
  if (n_obj > 65535) return (int)cudaErrorInvalidValue;
  const dim3 g(nb, nb, (unsigned)n_obj);
  GroupHyp h; h.hyp_obj = hyp_obj; h.nugget_obj = nugget_obj; h.nugget = nugget; h.floor = 0.0; h.flags = flags;
  cudaError_t e;
  if (dim == 1) e = hyp_obj ? launch_cov_gram<1, true>(g, smem, st, cov, grid, goff, m_shared, v, ldv, info, out, coff, h)
                            : launch_cov_gram<1, false>(g, smem, st, cov, grid, goff, m_shared, v, ldv, info, out, coff, h);
  else e = hyp_obj ? launch_cov_gram<2, true>(g, smem, st, cov, grid, goff, m_shared, v, ldv, info, out, coff, h)
                   : launch_cov_gram<2, false>(g, smem, st, cov, grid, goff, m_shared, v, ldv, info, out, coff, h);
  if (e != cudaSuccess) return (int)e;
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

// ---------------------------------------------------------------------------------------
// Schedules of the grouped large-object pipelines (large_ll_grouped, large_cov_grouped, large_predict_grouped).  Every
// launch of every wave is recorded on the host first; the arguments (object descriptors, GEMM problems, block offsets)
// are packed into one byte table that crosses to the device in one copy into stream-ordered scratch.
namespace {
enum { L_DIAG, L_GEMM, L_COV, L_FWD, L_FIN, L_PACK, L_BWD, L_MEAN, L_HB, L_VAR, L_ID, L_NORM, L_SUM };
struct Launch { int kind; int64_t grid, count, k0; size_t t0, t1, t2; double* ldb; int* infob; };

// One object of a wave: position j in `order`, object id b, n points, n_pad = 128 nblk (at least one block).
struct WaveItem { int64_t j, b, n, n_pad; int nblk; };
using Waves = std::vector<std::vector<WaveItem>>;

// The objects order[0 .. n_active) (object ids; NULL: 0 .. n_active) packed into consecutive waves: a wave closes
// before the object whose part of the workspace, need(item), would take it above work_doubles, and at 65535 objects
// (the y extent of the per-object launches).  Inside a wave the objects are sorted by decreasing block count (stable),
// so that the objects taking part in any step of the factorisation are a prefix of the wave.
template <class F>
Waves plan_waves(const int* order, int64_t n_active, const int64_t* off, int64_t work_doubles, F&& need) {
  Waves waves;
  std::vector<WaveItem> cur; int64_t used = 0;
  for (int64_t j = 0; j < n_active; ++j) {
    WaveItem it; it.j = j; it.b = order ? order[j] : j; it.n = off[it.b + 1] - off[it.b];
    it.n_pad = it.n <= 0 ? 128 : (it.n + 127) / 128 * 128; it.nblk = (int)(it.n_pad / 128);
    const int64_t w = need(it);
    if (!cur.empty() && (used + w > work_doubles || cur.size() >= 65535)) { waves.push_back(cur); cur.clear(); used = 0; }
    cur.push_back(it); used += w;
  }
  if (!cur.empty()) waves.push_back(cur);
  for (auto& w : waves)
    std::stable_sort(w.begin(), w.end(), [](const WaveItem& p, const WaveItem& q) { return p.nblk > q.nblk; });
  return waves;
}

// One sorted wave as the factorisation sees it: object i's n_pad x n_pad matrix at a[i], leading dimension ld[i] =
// n_pad, nblk[i] = n_pad / 128 blocks.  Block k of object i leaves its log det and info at [koff[k] + i] of the wave's
// block arrays.  t_ld, t_koff: ld and koff in the schedule's table.
struct WaveTables {
  std::vector<double*> a;
  std::vector<int64_t> ld, koff;
  std::vector<int> nblk;
  size_t t_ld = 0, t_koff = 0;
  int count(int k) const { int c = 0; while (c < (int)nblk.size() && nblk[c] > k) ++c; return c; }   // objects with block k
};

// Per-block log dets and infos of the wave being factored (large_cov_grouped, large_predict_grouped), in stream-ordered
// scratch sized for the wave with the most blocks and freed when it goes out of scope.
struct BlockScratch {
  double* p = nullptr;
  cudaStream_t st;
  explicit BlockScratch(cudaStream_t s) : st(s) {}
  ~BlockScratch() { if (p) cudaFreeAsync(p, st); }
  int alloc(const Waves& waves) {
    int64_t blocks = 0;
    for (const auto& w : waves) {
      int64_t b = 0;
      for (const WaveItem& it : w) b += it.nblk;
      blocks = std::max(blocks, b);
    }
    return (int)cudaMallocAsync((void**)&p, (size_t)blocks * (sizeof(double) + sizeof(int)) + 16, st);
  }
  double* ldb() const { return p; }
  int* infob(const WaveTables& t) const { return reinterpret_cast<int*>(p + t.koff.back()); }
};

struct GroupSchedule {
  std::vector<char> tab;
  std::vector<Launch> launches;
  std::vector<GemmArgs> probs;
  size_t t_csr = 0;

  size_t put(const void* p, size_t bytes) {
    const size_t o = (tab.size() + 15) & ~(size_t)15;
    tab.resize(o + bytes);
    memcpy(tab.data() + o, p, bytes);
    return o;
  }
  // the CSR {0, 128, 256, ..} the diagonal-block launches read, for the largest wave
  void block_csr(const Waves& waves) {
    size_t w_max = 0;
    for (const auto& w : waves) w_max = std::max(w_max, w.size());
    std::vector<int64_t> csr(w_max + 1);
    for (size_t i = 0; i <= w_max; ++i) csr[i] = (int64_t)i * 128;
    t_csr = put(csr.data(), csr.size() * sizeof(int64_t));
  }
  // the tables of the sorted wave w whose matrices are at a[i]; ld and koff go into the table
  WaveTables tables(const std::vector<WaveItem>& w, std::vector<double*> a) {
    WaveTables t;
    const int W = (int)w.size(), nb_max = w[0].nblk;
    t.a = std::move(a); t.ld.resize(W); t.nblk.resize(W); t.koff.assign(nb_max + 1, 0);
    for (int i = 0; i < W; ++i) { t.ld[i] = w[i].n_pad; t.nblk[i] = w[i].nblk; }
    for (int k = 0; k < nb_max; ++k) t.koff[k + 1] = t.koff[k] + t.count(k);
    t.t_ld = put(t.ld.data(), W * sizeof(int64_t));
    t.t_koff = put(t.koff.data(), t.koff.size() * sizeof(int64_t));
    return t;
  }
  void gemm(const double* A, int64_t lda, const double* B, int64_t ldb, double* C, int64_t ldc, int64_t m, int64_t n,
            int64_t k, double alpha, double beta, int lower) {
    GemmArgs g;
    g.a = A; g.b = B; g.c = C; g.lda = lda; g.ldb = ldb; g.ldc = ldc;
    g.m = (int)m; g.n = (int)n; g.k = (int)k; g.alpha = alpha; g.beta = beta; g.lower_only = lower;
    probs.push_back(g);
  }
  // the GEMM problems recorded since the last flush as one grouped launch, tiles split as launch_gemm_nt splits them
  int flush() {
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
  }
  // The blocked Cholesky of large_potrf for the matrices of one wave (the objects taking part in any step are a prefix).
  // Per pair of block columns two diagonal-block launches (launch_small in matrix-source mode, ld table at t.t_ld) and
  // four grouped GEMM launches, with the shapes, tile split and alpha / beta large_potrf uses for each object alone (the
  // next pair's columns and the lower trailing update touch disjoint tiles, so they share one launch).  Block k of
  // object i leaves its log det and info at ldb / infob[t.koff[k] + i].
  int factor(double* work, const WaveTables& t, double* ldb, int* infob) {
    const std::vector<double*>& a = t.a;
    const std::vector<int64_t>& ld = t.ld;
    const std::vector<int>& nblk = t.nblk;
    const int W = (int)a.size(), nb_max = nblk[0];
    auto diag = [&](int k) {
      const int c = t.count(k);
      std::vector<int64_t> aoff(c);
      for (int i = 0; i < c; ++i) aoff[i] = (a[i] - work) + (int64_t)k * 128 * ld[i] + (int64_t)k * 128;
      launches.push_back({L_DIAG, c, c, 0, put(aoff.data(), c * sizeof(int64_t)), t.t_ld, 0, ldb + t.koff[k], infob + t.koff[k]});
    };
    int e = 0;
    for (int p = 0; 2 * p < nb_max && !e; ++p) {
      const int k = 2 * p;
      const int64_t k0 = (int64_t)p * 256;
      diag(k);
      for (int i = 0; i < W && nblk[i] > k + 1; ++i) {            // panel of block column k: L_ik = A_ik T_kk^T
        const int64_t np = ld[i];
        double* ai = a[i];
        gemm(ai + (k0 + 128) * np + k0, np, ai + k0 * np + k0, np, ai + (k0 + 128) * np + k0, np, np - k0 - 128, 128, 128,
             1.0, 0.0, 0);
      }
      if ((e = flush())) break;
      for (int i = 0; i < W && nblk[i] > k + 1; ++i) {            // block column k+1 -= L[k+1:, k] L[k+1, k]^T
        const int64_t np = ld[i];
        double* ai = a[i];
        double* panel = ai + (k0 + 128) * np + k0;
        gemm(panel, np, panel, np, ai + (k0 + 128) * np + (k0 + 128), np, np - k0 - 128, 128, 128, -1.0, 1.0, 0);
      }
      if ((e = flush())) break;
      if (nb_max <= k + 1) break;
      diag(k + 1);
      const int64_t k1 = k0 + 128;
      for (int i = 0; i < W && nblk[i] > k + 2; ++i) {            // panel of block column k+1
        const int64_t np = ld[i];
        double* ai = a[i];
        gemm(ai + (k1 + 128) * np + k1, np, ai + k1 * np + k1, np, ai + (k1 + 128) * np + k1, np, np - k1 - 128, 128, 128,
             1.0, 0.0, 0);
      }
      if ((e = flush())) break;
      for (int i = 0; i < W && nblk[i] > k + 2; ++i) {            // the pair applied to what lies right of it, K = 256
        const int64_t np = ld[i], rest = np - k0 - 256;
        double* ai = a[i];
        double* wp = ai + (k0 + 256) * np + k0;
        gemm(wp, np, wp, np, ai + (k0 + 256) * np + (k0 + 256), np, rest, 128, 256, -1.0, 1.0, 0);
        if (rest > 128)
          gemm(wp + 128 * np, np, wp + 128 * np, np, ai + (k0 + 384) * np + (k0 + 384), np, rest - 128, 128, 256, -1.0, 1.0, 0);
        if (rest > 256)
          gemm(wp + 256 * np, np, wp + 256 * np, np, ai + (k0 + 512) * np + (k0 + 512), np, rest - 256, rest - 256, 256, -1.0,
               1.0, 1);
      }
      e = flush();
    }
    return e;
  }
  // V = rows of L^-1 H^T for objects of a factored wave, as large_trsm_rows computes it: per block column k,
  // V[:, k] -= V[:, 0:k] L[k, 0:k]^T (from k = 1 on), then V[:, k] T_kk^T, each one grouped launch over the entries
  // whose object has block k.  Entry: the rows_pad x n_pad matrix V at v of wave object i.
  struct RowSolve { double* v; int64_t rows_pad; int i; };
  int trsm_rows(const WaveTables& t, const std::vector<RowSolve>& vs) {
    int e = 0;
    for (int k = 0; k < t.nblk[0] && !e; ++k) {
      const int64_t k0 = (int64_t)k * 128;
      if (k > 0) {
        for (const RowSolve& r : vs) {
          const int64_t ld = t.ld[r.i];
          if (t.nblk[r.i] > k) gemm(r.v, ld, t.a[r.i] + k0 * ld, ld, r.v + k0, ld, r.rows_pad, 128, k0, -1.0, 1.0, 0);
        }
        if ((e = flush())) break;
      }
      for (const RowSolve& r : vs) {
        const int64_t ld = t.ld[r.i];
        if (t.nblk[r.i] > k) gemm(r.v + k0, ld, t.a[r.i] + k0 * ld + k0, ld, r.v + k0, ld, r.rows_pad, 128, 128, 1.0, 0.0, 0);
      }
      e = flush();
    }
    return e;
  }
  // negd[i] = -diag(K^-1) for the objects of a factored wave, as large_diag_inv computes it: passes of chunk_rows identity
  // rows staged at v[i] (chunk_rows x n_pad); in pass r0 every object with n_pad > r0 (a prefix) takes part with
  // min(chunk_rows, n_pad - r0) rows.  Per pass one identity-rows launch, per pair of block columns from r0 / 128 on the
  // four GEMMs of large_diag_inv (shapes, row clipping, alpha / beta) as grouped launches over the objects with those
  // blocks, then one row-norm launch.
  int diag_inv(const WaveTables& t, const std::vector<double*>& v, const std::vector<double*>& negd, int64_t chunk_rows) {
    int e = 0;
    for (int64_t r0 = 0; r0 < t.ld[0] && !e; r0 += chunk_rows) {
      const int kb0 = (int)(r0 / 128);
      std::vector<DiagObj> d;
      int64_t cta = 0, blocks = 0;
      for (int i = 0; i < (int)t.ld.size() && t.ld[i] > r0; ++i) {
        const int64_t np = t.ld[i], c = std::min(chunk_rows, np - r0), w = np - r0;
        d.push_back({v[i] + r0, np, w, c, negd[i] + r0, cta});
        cta += (c + 7) / 8;
        blocks = std::max(blocks, (c * (w / 2) + 255) / 256);
      }
      const int P = (int)d.size();
      const size_t td = put(d.data(), P * sizeof(DiagObj));
      launches.push_back({L_ID, std::min<int64_t>(blocks, 148 * 16), P, 0, td, 0, 0, nullptr, nullptr});
      auto rows = [&](int i, int k) { return std::min<int64_t>((int64_t)(k - kb0 + 1) * 128, d[i].rows); };
      auto lk = [&](int i, int k) { return t.a[i] + (int64_t)k * 128 * t.ld[i] + (int64_t)k * 128; };
      for (int k = kb0; k < t.nblk[0] && !e; k += 2) {
        const int64_t j0 = (int64_t)(k - kb0) * 128;    // block column k inside the pass
        for (int i = 0; i < P && t.nblk[i] > k; ++i)   // V_k T_kk^T
          gemm(d[i].v + j0, d[i].ld, lk(i, k), t.ld[i], d[i].v + j0, d[i].ld, rows(i, k), 128, 128, 1.0, 0.0, 0);
        if ((e = flush())) break;
        for (int i = 0; i < P && t.nblk[i] > k + 1; ++i)   // V_{k+1} -= V_k L_{k+1,k}^T
          gemm(d[i].v + j0, d[i].ld, lk(i, k) + 128 * t.ld[i], t.ld[i], d[i].v + j0 + 128, d[i].ld, rows(i, k), 128, 128, -1.0, 1.0, 0);
        if ((e = flush())) break;
        for (int i = 0; i < P && t.nblk[i] > k + 1; ++i)   // V_{k+1} T_{k+1,k+1}^T
          gemm(d[i].v + j0 + 128, d[i].ld, lk(i, k) + 128 * t.ld[i] + 128, t.ld[i], d[i].v + j0 + 128, d[i].ld, rows(i, k + 1), 128,
               128, 1.0, 0.0, 0);
        if ((e = flush())) break;
        for (int i = 0; i < P && t.nblk[i] > k + 2; ++i)   // V[:, k+2:] -= V[:, k:k+2] L[k+2:, k:k+2]^T, K = 256
          gemm(d[i].v + j0, d[i].ld, lk(i, k) + 256 * t.ld[i], t.ld[i], d[i].v + j0 + 256, d[i].ld, rows(i, k + 1),
               t.ld[i] - (int64_t)(k + 2) * 128, 256, -1.0, 1.0, 0);
        e = flush();
      }
      if (cta > 2147483647LL) return (int)cudaErrorInvalidValue;
      launches.push_back({L_NORM, cta, P, 0, td, 0, 0, nullptr, nullptr});
    }
    return e;
  }
  // Copies the table to the device and runs the recorded launches in order: the diagonal blocks and the GEMMs here,
  // every other kind through other(launch, device table).
  template <class F>
  int run(double* work, cudaStream_t st, F&& other) {
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
    int e = 0;
    for (const Launch& l : launches) {
      switch (l.kind) {
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
        case L_ID:
          identity_rows_grouped_kernel<<<dim3((unsigned)l.grid, (unsigned)l.count), 256, 0, st>>>(
              reinterpret_cast<const DiagObj*>(td + l.t0));
          break;
        case L_NORM:
          diag_norm_grouped_kernel<<<(unsigned)l.grid, 256, 0, st>>>(reinterpret_cast<const DiagObj*>(td + l.t0), (int)l.count);
          break;
        default:
          other(l, td);
      }
      if (l.kind != L_DIAG) count_launch();
      if (e) break;
    }
    cudaFreeAsync(td, st);
    return e ? e : (int)cudaGetLastError();
  }
};
}  // namespace

// Log-likelihoods of the objects order[0 .. n_active) (object ids; NULL: 0 .. n_active), object order[j] with the
// covariance function covs[j] (built on the host, with the floor), by every step of cgp_cov_matrix_dev + cgp_potrf_dev +
// cgp_large_solve_dev run for all objects of a wave at once: one covariance launch; the factorisation
// (GroupSchedule::factor); one forward-sweep launch per block; one epilogue.  Waves: plan_waves, each object's part of
// the workspace large_ll_ws_doubles.  The caller checks that every object fits.
int large_ll_grouped(int dim, const int64_t* off, const double* x, const double* y, const double* y0, const double* yerr,
                     const Cov* covs, const int* order, int64_t n_active, double* ll, int* info, double* work,
                     int64_t work_doubles, cudaStream_t st) {
  const Waves waves = plan_waves(order, n_active, off, work_doubles, [](const WaveItem& it) { return large_ll_ws_doubles(it.n); });
  GroupSchedule s;
  s.block_csr(waves);

  for (const auto& w : waves) {
    const int W = (int)w.size();
    std::vector<GroupObj> objs(W);
    std::vector<double*> a(W);
    int64_t cur = 0, cta = 0;
    for (int i = 0; i < W; ++i) {
      const WaveItem& it = w[i];
      const int64_t o0 = off[it.b], np = it.n_pad;
      GroupObj& g = objs[i];
      g.cov = covs[it.j];
      g.x = x + dim * o0; g.y = y + o0; g.y0 = y0 ? y0 + o0 : nullptr; g.yerr = yerr ? yerr + o0 : nullptr;
      g.a = work + cur; g.r = g.a + np * np; g.ones = nullptr; g.z = g.r + np;
      g.n = it.n; g.n_pad = np; g.io = it.j; g.cta = cta;
      cur += np * np + 2 * np; cta += np * ((np + 255) / 256);
      a[i] = g.a;
    }
    if (cta > 2147483647LL) return (int)cudaErrorInvalidValue;
    const size_t t_objs = s.put(objs.data(), W * sizeof(GroupObj));
    const WaveTables t = s.tables(w, std::move(a));
    double* ldb = work + cur;                        // the block log dets and infos follow the objects
    int* infob = reinterpret_cast<int*>(ldb + t.koff.back());
    s.launches.push_back({L_COV, cta, W, 0, t_objs, 0, 0, nullptr, nullptr});
    if (int e = s.factor(work, t, ldb, infob)) return e;
    for (int k = 0; k < w[0].nblk; ++k)
      s.launches.push_back({L_FWD, 1 + (t.ld[0] - (int64_t)k * 128 - 128 + 63) / 64, t.count(k), (int64_t)k * 128, t_objs, 0, 0,
                            nullptr, nullptr});
    s.launches.push_back({L_FIN, W, W, 0, t_objs, t.t_koff, 0, ldb, infob});
  }
  return s.run(work, st, [&](const Launch& l, const char* td) {
    const GroupObj* objs = reinterpret_cast<const GroupObj*>(td + l.t0);
    switch (l.kind) {
      case L_COV:
        if (dim == 1) build_grouped_kernel<1><<<(unsigned)l.grid, 128, 0, st>>>(objs, (int)l.count);
        else build_grouped_kernel<2><<<(unsigned)l.grid, 128, 0, st>>>(objs, (int)l.count);
        break;
      case L_FWD:
        fwd_step_grouped_kernel<GroupObj><<<dim3((unsigned)l.grid, (unsigned)l.count), 256, 0, st>>>(objs, l.k0);
        break;
      case L_FIN:
        ll_finish_grouped_kernel<<<(unsigned)l.grid, 1024, 0, st>>>(objs, l.ldb, l.infob,
                                                                    reinterpret_cast<const int64_t*>(td + l.t1), ll, info);
        break;
    }
  });
}

int64_t large_cov_ws_doubles(int64_t n, int64_t m) {
  const int64_t np = n <= 0 ? 128 : (n + 127) / 128 * 128, mp = m <= 0 ? 128 : (m + 127) / 128 * 128;
  return np * np + mp * np + mp * mp;                // covariance / factor, H -> V, K** -> C
}

// Predictive covariance matrices of the objects order[0 .. n_active) (object ids; NULL: 0 .. n_active), object
// order[j] with covs[j] for its own covariance and covs_g[j] for H and K**, on its grid (goff: xnew + dim * goff[b], m_b = goff[b+1] - goff[b]; NULL: the shared grid
// xnew of m_shared points), by every step of dense.predictive_covariance run for all objects of a wave at once:
// A = K(x, x) + noise, H and K** in one launch; the factorisation (GroupSchedule::factor); V = rows of L^-1 H^T
// (GroupSchedule::trsm_rows); C = K** - V V^T (one grouped GEMM launch); the packing of each leading m_b x m_b block to
// out + coff[j], NaN where info[j] != 0.  Waves: plan_waves, each object's part of the workspace
// large_cov_ws_doubles(n_b, m_b).  The caller checks that every object fits.
int large_cov_grouped(int dim, const int64_t* off, const double* x, const double* yerr, const Cov* covs, const Cov* covs_g,
                      const double* xnew, const int64_t* goff, int64_t m_shared, const int* order, int64_t n_active, double* out,
                      const int64_t* coff, int* info, double* work, int64_t work_doubles, cudaStream_t st) {
  auto grid_size = [&](int64_t b) { return goff ? goff[b + 1] - goff[b] : m_shared; };
  const Waves waves = plan_waves(order, n_active, off, work_doubles,
                                 [&](const WaveItem& it) { return large_cov_ws_doubles(it.n, grid_size(it.b)); });
  GroupSchedule s;
  s.block_csr(waves);
  BlockScratch blk(st);
  if (int ce = blk.alloc(waves)) return ce;

  for (const auto& w : waves) {
    const int W = (int)w.size();
    std::vector<CovObj> objs(W);
    std::vector<double*> a(W);
    std::vector<GroupSchedule::RowSolve> vs(W);
    int64_t cur = 0, cta = 0, mm_max = 0;
    for (int i = 0; i < W; ++i) {
      const WaveItem& it = w[i];
      const int64_t m = grid_size(it.b), np = it.n_pad, mp = m <= 0 ? 128 : (m + 127) / 128 * 128;
      CovObj& o = objs[i];
      o.cov = covs[it.j]; o.cov_g = covs_g[it.j];
      o.x = x + dim * off[it.b]; o.yerr = yerr ? yerr + off[it.b] : nullptr; o.g = goff ? xnew + dim * goff[it.b] : xnew;
      o.a = work + cur; o.v = o.a + np * np; o.c = o.v + mp * np; o.out = out + coff[it.j];
      o.n = it.n; o.n_pad = np; o.m = m; o.m_pad = mp; o.io = it.j; o.cta0 = cta;
      cur += large_cov_ws_doubles(it.n, m);
      cta += (np + mp) * ((np + 255) / 256) + mp * ((mp + 255) / 256);
      mm_max = std::max(mm_max, m * m);
      a[i] = o.a; vs[i] = {o.v, mp, i};
    }
    if (cta > 2147483647LL) return (int)cudaErrorInvalidValue;
    const size_t t_objs = s.put(objs.data(), W * sizeof(CovObj));
    const WaveTables t = s.tables(w, std::move(a));
    s.launches.push_back({L_COV, cta, W, 0, t_objs, 0, 0, nullptr, nullptr});
    if (int e = s.factor(work, t, blk.ldb(), blk.infob(t))) return e;
    if (int e = s.trsm_rows(t, vs)) return e;
    for (const CovObj& o : objs)                     // C = K** - V V^T, the whole m_pad x m_pad block
      s.gemm(o.v, o.n_pad, o.v, o.n_pad, o.c, o.m_pad, o.m_pad, o.m_pad, o.n_pad, -1.0, 1.0, 0);
    if (int e = s.flush()) return e;
    const int64_t gx = std::min<int64_t>(std::max<int64_t>((mm_max + 1023) / 1024, 1), 1024);
    s.launches.push_back({L_PACK, gx, W, 0, t_objs, t.t_koff, 0, blk.ldb(), blk.infob(t)});
  }
  return s.run(work, st, [&](const Launch& l, const char* td) {
    const CovObj* objs = reinterpret_cast<const CovObj*>(td + l.t0);
    switch (l.kind) {
      case L_COV:
        if (dim == 1) cov3_build_grouped_kernel<1><<<(unsigned)l.grid, 128, 0, st>>>(objs, (int)l.count);
        else cov3_build_grouped_kernel<2><<<(unsigned)l.grid, 128, 0, st>>>(objs, (int)l.count);
        break;
      case L_PACK:
        cov_pack_grouped_kernel<<<dim3((unsigned)l.grid, (unsigned)l.count), 256, 0, st>>>(
            objs, l.infob, reinterpret_cast<const int64_t*>(td + l.t1), info);
        break;
    }
  });
}

int64_t large_pred_ws_doubles(int64_t n, int64_t rows) {
  const int64_t np = n <= 0 ? 128 : (n + 127) / 128 * 128, rp = rows <= 0 ? 0 : (rows + 127) / 128 * 128;
  return np * np + 3 * np + rp * np;                 // covariance / factor, u, z, alpha, H -> V of one pass
}

// Means (and variance diagonals when var != null) of the objects order[0 .. n_active) on their grids (goff: xnew + dim *
// goff[b], m_b = goff[b+1] - goff[b]; NULL: the shared grid xnew of m_shared points), object order[j] with covs[j] for A
// and covs_g[j] for the rest, outputs at mean / var / new_y0 + moff[j], by every step of LargeObject.factor followed by
// cgp_large_predict_dev run for all objects of a wave at once: A and u in one launch; the factorisation
// (GroupSchedule::factor); one forward- and one backward-sweep launch per block; the streamed mean in one launch; then per
// pass of at most chunk_rows grid rows (% 128 == 0) per object: H in one launch, V = rows of L^-1 H^T
// (GroupSchedule::trsm_rows), and the variance in one launch; last, info and NaN rows where info != 0.  A row's
// arithmetic does not depend on the pass it falls in.  Waves: plan_waves, each object's part of the workspace
// large_pred_ws_doubles(n_b, var ? min(m_b, chunk_rows) : 0).  The caller checks that every object fits.
int large_predict_grouped(int dim, const int64_t* off, const double* x, const double* y, const double* y0, const double* yerr,
                          const Cov* covs, const Cov* covs_g, const double* xnew, const int64_t* goff, int64_t m_shared,
                          const double* new_y0, const int* order, int64_t n_active, const int64_t* moff, double* mean,
                          double* var, int* info, int64_t chunk_rows, double* work, int64_t work_doubles, cudaStream_t st) {
  auto grid_size = [&](int64_t b) { return goff ? goff[b + 1] - goff[b] : m_shared; };
  auto pass_rows = [&](int64_t b) { return var ? std::min(grid_size(b), chunk_rows) : (int64_t)0; };
  const Waves waves = plan_waves(order, n_active, off, work_doubles,
                                 [&](const WaveItem& it) { return large_pred_ws_doubles(it.n, pass_rows(it.b)); });
  GroupSchedule s;
  s.block_csr(waves);
  BlockScratch blk(st);
  if (int ce = blk.alloc(waves)) return ce;

  for (const auto& w : waves) {
    const int W = (int)w.size(), nb_max = w[0].nblk;
    std::vector<PredObj> objs(W);
    std::vector<double*> a(W), v(W);
    int64_t cur = 0, cta = 0, cta_mean = 0, m_max = 0;
    for (int i = 0; i < W; ++i) {
      const WaveItem& it = w[i];
      const int64_t np = it.n_pad, o0 = off[it.b];
      PredObj& o = objs[i];
      o.cov = covs[it.j]; o.cov_g = covs_g[it.j];
      o.x = x + dim * o0; o.y = y + o0; o.y0 = y0 ? y0 + o0 : nullptr; o.yerr = yerr ? yerr + o0 : nullptr;
      o.g = goff ? xnew + dim * goff[it.b] : xnew; o.new_y0 = new_y0 ? new_y0 + moff[it.j] : nullptr;
      o.a = work + cur; o.r = o.a + np * np; o.ones = nullptr; o.z = o.r + np; o.alpha = o.z + np; v[i] = o.alpha + np;
      o.mean = mean + moff[it.j]; o.var = var ? var + moff[it.j] : nullptr;
      o.n = it.n; o.n_pad = np; o.m = grid_size(it.b); o.io = it.j; o.cta = cta; o.cta_mean = cta_mean;
      cur += large_pred_ws_doubles(it.n, pass_rows(it.b));
      cta += np * ((np + 255) / 256); cta_mean += (o.m + 255) / 256;
      m_max = std::max(m_max, o.m);
      a[i] = o.a;
    }
    if (cta > 2147483647LL || cta_mean > 2147483647LL) return (int)cudaErrorInvalidValue;
    const size_t t_objs = s.put(objs.data(), W * sizeof(PredObj));
    const WaveTables t = s.tables(w, std::move(a));
    s.launches.push_back({L_COV, cta, W, 0, t_objs, 0, 0, nullptr, nullptr});
    if (int e = s.factor(work, t, blk.ldb(), blk.infob(t))) return e;
    for (int k = 0; k < nb_max; ++k)                 // large_potrs: z = L^-1 u
      s.launches.push_back({L_FWD, 1 + (t.ld[0] - (int64_t)k * 128 - 128 + 63) / 64, t.count(k), (int64_t)k * 128, t_objs, 0, 0,
                            nullptr, nullptr});
    for (int q = 0; q < nb_max; ++q)                 // large_potrs_backward: alpha = L^-T z, block nblk - 1 - q of each
      s.launches.push_back({L_BWD, nb_max - q, t.count(q), q, t_objs, 0, 0, nullptr, nullptr});
    if (cta_mean) s.launches.push_back({L_MEAN, cta_mean, W, 0, t_objs, 0, 0, nullptr, nullptr});
    for (int64_t r0 = 0; var && r0 < m_max; r0 += chunk_rows) {   // variance passes
      std::vector<PassObj> pass;
      std::vector<GroupSchedule::RowSolve> vs;
      int64_t cta_h = 0, cta_var = 0;
      for (int i = 0; i < W; ++i) {
        const PredObj& o = objs[i];
        if (o.m <= r0) continue;
        PassObj p;
        p.cov_g = o.cov_g; p.x = o.x; p.g = o.g + dim * r0; p.v = v[i]; p.var = o.var + r0;
        p.n = o.n; p.n_pad = o.n_pad; p.rows = std::min(chunk_rows, o.m - r0); p.rows_pad = (p.rows + 127) / 128 * 128;
        p.cta_h = cta_h; p.cta_var = cta_var;
        cta_h += p.rows_pad * ((p.n_pad + 255) / 256); cta_var += (p.rows + 7) / 8;
        pass.push_back(p); vs.push_back({v[i], p.rows_pad, i});
      }
      if (cta_h > 2147483647LL) return (int)cudaErrorInvalidValue;
      const int P = (int)pass.size();
      const size_t t_pass = s.put(pass.data(), P * sizeof(PassObj));
      s.launches.push_back({L_HB, cta_h, P, 0, t_pass, 0, 0, nullptr, nullptr});
      if (int e = s.trsm_rows(t, vs)) return e;
      s.launches.push_back({L_VAR, cta_var, P, 0, t_pass, 0, 0, nullptr, nullptr});
    }
    const int64_t gx = std::min<int64_t>(std::max<int64_t>((m_max + 1023) / 1024, 1), 1024);
    s.launches.push_back({L_FIN, gx, W, 0, t_objs, t.t_koff, 0, blk.ldb(), blk.infob(t)});
  }
  return s.run(work, st, [&](const Launch& l, const char* td) {
    const PredObj* objs = reinterpret_cast<const PredObj*>(td + l.t0);
    const PassObj* pass = reinterpret_cast<const PassObj*>(td + l.t0);
    switch (l.kind) {
      case L_COV:
        if (dim == 1) build_grouped_kernel<1><<<(unsigned)l.grid, 128, 0, st>>>(objs, (int)l.count);
        else build_grouped_kernel<2><<<(unsigned)l.grid, 128, 0, st>>>(objs, (int)l.count);
        break;
      case L_FWD:
        fwd_step_grouped_kernel<PredObj><<<dim3((unsigned)l.grid, (unsigned)l.count), 256, 0, st>>>(objs, l.k0);
        break;
      case L_BWD:
        bwd_step_grouped_kernel<PredObj><<<dim3((unsigned)l.grid, (unsigned)l.count), 256, 0, st>>>(objs, l.k0);
        break;
      case L_MEAN:
        if (dim == 1) stream_mean_grouped_kernel<1><<<(unsigned)l.grid, 256, 2 * 1024 * sizeof(double), st>>>(objs, (int)l.count);
        else stream_mean_grouped_kernel<2><<<(unsigned)l.grid, 256, 3 * 1024 * sizeof(double), st>>>(objs, (int)l.count);
        break;
      case L_HB:
        if (dim == 1) pass_build_grouped_kernel<1><<<(unsigned)l.grid, 128, 0, st>>>(pass, (int)l.count);
        else pass_build_grouped_kernel<2><<<(unsigned)l.grid, 128, 0, st>>>(pass, (int)l.count);
        break;
      case L_VAR:
        row_var_grouped_kernel<<<(unsigned)l.grid, 256, 0, st>>>(pass, (int)l.count);
        break;
      case L_FIN:
        pred_finish_grouped_kernel<<<dim3((unsigned)l.grid, (unsigned)l.count), 256, 0, st>>>(
            objs, l.infob, reinterpret_cast<const int64_t*>(td + l.t1), info);
        break;
    }
  });
}

int64_t large_loo_ws_doubles(int64_t n, int64_t chunk_rows) {
  const int64_t np = n <= 0 ? 128 : (n + 127) / 128 * 128;
  // factor, the first diag(K^-1) pass, r / z / alpha, 1 / z_1 / K^-1 1, -d, sum r and one double that keeps the next
  // object 16-byte aligned
  return np * np + std::min(np, chunk_rows) * np + 7 * np + 2;
}

// Leave-one-out pulls of the objects order[0 .. n_active) (object ids; NULL: 0 .. n_active), object order[j] with covs[j],
// outputs at pred / pvar / pull / resid + off[b] (each may be null), by every step of cgp_cov_matrix_dev + cgp_potrf_dev +
// cgp_large_loo_dev run for all objects of a wave at once: A, r (and the ones vector) in one launch; sum r in one launch
// (recentred mode); the factorisation (GroupSchedule::factor); one forward- and one backward-sweep launch per block for
// both right-hand sides; -diag(K^-1) (GroupSchedule::diag_inv); one epilogue launch that writes info[j] and NaN outputs
// where info != 0.  Waves: plan_waves, each object's part of the workspace large_loo_ws_doubles(n_b, chunk_rows).  The
// caller checks that every object fits.
int large_loo_grouped(int dim, const int64_t* off, const double* x, const double* y, const double* m, const double* yerr,
                      const Cov* covs, int recenter, const int* order, int64_t n_active, int* info, double* pred, double* pvar,
                      double* pull, double* resid, int64_t chunk_rows, double* work, int64_t work_doubles, cudaStream_t st) {
  const Waves waves = plan_waves(order, n_active, off, work_doubles,
                                 [&](const WaveItem& it) { return large_loo_ws_doubles(it.n, chunk_rows); });
  GroupSchedule s;
  s.block_csr(waves);
  BlockScratch blk(st);
  if (int ce = blk.alloc(waves)) return ce;
  const int nrhs = recenter ? 2 : 1;

  for (const auto& w : waves) {
    const int W = (int)w.size(), nb_max = w[0].nblk;
    std::vector<LooObj> objs(W);
    std::vector<SolveObj> rhs;
    std::vector<double*> a(W), v(W), negd(W);
    int64_t cur = 0, cta = 0, cta_epi = 0;
    for (int i = 0; i < W; ++i) {
      const WaveItem& it = w[i];
      const int64_t np = it.n_pad, o0 = off[it.b];
      LooObj& o = objs[i];
      o.cov = covs[it.j];
      o.x = x + dim * o0; o.y = y + o0; o.y0 = m ? m + o0 : nullptr; o.yerr = yerr ? yerr + o0 : nullptr;
      o.a = work + cur; v[i] = o.a + np * np;
      double* vec = v[i] + std::min(np, chunk_rows) * np;
      o.r = vec; o.alpha = vec + 2 * np;
      o.ones = recenter ? vec + 3 * np : nullptr; o.kinv1 = recenter ? vec + 5 * np : nullptr;
      o.negd = negd[i] = vec + 6 * np; o.rsum = vec + 7 * np;
      o.pred = pred ? pred + o0 : nullptr; o.pvar = pvar ? pvar + o0 : nullptr;
      o.pull = pull ? pull + o0 : nullptr; o.resid = resid ? resid + o0 : nullptr;
      o.n = it.n; o.n_pad = np; o.io = it.j; o.cta = cta; o.cta_epi = cta_epi;
      rhs.push_back({o.a, o.r, vec + np, o.alpha, np});
      if (recenter) rhs.push_back({o.a, o.ones, vec + 4 * np, o.kinv1, np});
      cur += large_loo_ws_doubles(it.n, chunk_rows);
      cta += np * ((np + 255) / 256); cta_epi += std::max<int64_t>((it.n + 255) / 256, 1);
      a[i] = o.a;
    }
    if (cta > 2147483647LL || cta_epi > 2147483647LL) return (int)cudaErrorInvalidValue;
    const size_t t_objs = s.put(objs.data(), W * sizeof(LooObj));
    const size_t t_rhs = s.put(rhs.data(), rhs.size() * sizeof(SolveObj));
    const WaveTables t = s.tables(w, std::move(a));
    s.launches.push_back({L_COV, cta, W, 0, t_objs, 0, 0, nullptr, nullptr});
    if (recenter) s.launches.push_back({L_SUM, W, W, 0, t_objs, 0, 0, nullptr, nullptr});   // before the sweep consumes r
    if (int e = s.factor(work, t, blk.ldb(), blk.infob(t))) return e;
    for (int k = 0; k < nb_max; ++k)                 // large_potrs forward, both right-hand sides
      s.launches.push_back({L_FWD, 1 + (t.ld[0] - (int64_t)k * 128 - 128 + 63) / 64, t.count(k), (int64_t)k * 128, t_rhs, 0, 0,
                            nullptr, nullptr});
    for (int q = 0; q < nb_max; ++q)                 // large_potrs backward: block nblk - 1 - q of each
      s.launches.push_back({L_BWD, nb_max - q, t.count(q), q, t_rhs, 0, 0, nullptr, nullptr});
    if (int e = s.diag_inv(t, v, negd, chunk_rows)) return e;
    s.launches.push_back({L_FIN, cta_epi, W, 0, t_objs, t.t_koff, 0, blk.ldb(), blk.infob(t)});
  }
  return s.run(work, st, [&](const Launch& l, const char* td) {
    const LooObj* objs = reinterpret_cast<const LooObj*>(td + l.t0);
    const SolveObj* rhs = reinterpret_cast<const SolveObj*>(td + l.t0);
    switch (l.kind) {
      case L_COV:
        if (dim == 1) build_grouped_kernel<1><<<(unsigned)l.grid, 128, 0, st>>>(objs, (int)l.count);
        else build_grouped_kernel<2><<<(unsigned)l.grid, 128, 0, st>>>(objs, (int)l.count);
        break;
      case L_SUM:
        sum_grouped_kernel<<<(unsigned)l.grid, 1024, 0, st>>>(objs);
        break;
      case L_FWD:
        fwd_step_grouped_kernel<SolveObj><<<dim3((unsigned)l.grid, (unsigned)l.count, nrhs), 256, 0, st>>>(rhs, l.k0);
        break;
      case L_BWD:
        bwd_step_grouped_kernel<SolveObj><<<dim3((unsigned)l.grid, (unsigned)l.count, nrhs), 256, 0, st>>>(rhs, l.k0);
        break;
      case L_FIN:
        loo_finish_grouped_kernel<<<(unsigned)l.grid, 256, 0, st>>>(objs, (int)l.count, l.infob,
                                                                    reinterpret_cast<const int64_t*>(td + l.t1), info);
        break;
    }
  });
}

}  // namespace cgp
