// Internal declarations shared by the kernel translation units and the C ABI.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace cgp {

// Covariance function, prepared on the host from hyp / nugget / floor / flags.
//   K(a,b) = amp * exp(-q/2);  1D: q = (a-b)^2 / l^2 (cosmogp/kernel.py:71-72)
//   2D: q = d^T M d with M the inverse metric (cosmogp/kernel.py:127-130).
//   h00, h01, h11 hold -M00/2, -M01, -M11/2, so that -q/2 = dx^2 h00 + dx dy h01 + dy^2 h11.
struct Cov {
  double amp_auto;     // auto-covariance amplitude: sigma^2 (1D) or 1 (2D at HEAD, kernel.py:146-148)
  double amp_cross;    // cross-covariance amplitude: sigma^2 (kernel.py:72,141)
  double h00, h01, h11;
  double noise_const;  // floor^2 + nugget^2, added to y_err^2 on the diagonal (kernel.py:75,151)
  double nugget2;      // nugget^2: K(x*,x*) carries it but not y_err^2 (Gaussian_process.py:357)
};

#define CGP_FLAG_AMP_ON_AUTOCOV 1u
#define CGP_FLAG_MEAN_TEMPLATE 2u
#define CGP_FLAG_GRID_UNIFORM 4u

// hyp -> Cov (cosmogp/kernel.py:71-75 for 1D, :127-151 for 2D); shared by the host API and by the
// kernels when every object carries its own hyperparameters.  A singular / NaN metric propagates.
__host__ __device__ inline Cov cov_from_hyp(int dim, const double* hyp, double nugget, double floor, unsigned flags) {
  Cov c;
  const double s2 = hyp[0] * hyp[0];
  c.amp_cross = s2;
  if (dim == 1) {
    c.amp_auto = s2;
    c.h00 = -0.5 / (hyp[1] * hyp[1]); c.h01 = 0.0; c.h11 = 0.0;
  } else {
    const double lx2 = hyp[1] * hyp[1], ly2 = hyp[2] * hyp[2], lxy = hyp[3];
    const double sc = 1.0 / (lx2 * ly2 - lxy * lxy);
    c.h00 = -0.5 * (ly2 * sc); c.h01 = lxy * sc; c.h11 = -0.5 * (lx2 * sc);
    c.amp_auto = (flags & CGP_FLAG_AMP_ON_AUTOCOV) ? s2 : 1.0;   // HEAD drops sigma^2 (kernel.py:146-148)
  }
  c.noise_const = floor * floor + nugget * nugget;
  c.nugget2 = nugget * nugget;
  return c;
}

// TASK_FACTOR writes the Cholesky factor (T_J = L_JJ^-1 on the diagonal, -L[I][J] below, in the tile layout of
// cgp_small64.cu) + z = L^-1 r per object to a workspace; TASK_PREDICT_F
// predicts from that workspace (staged into shared memory by one TMA bulk copy per object).
// TASK_PREDICT_FU: TASK_PREDICT_F for dim 1 on a uniformly spaced shared grid with l >= spacing (exps by recurrence).
// TASK_PREDICT_U: TASK_PREDICT (factorise + predict in ONE pass, nothing spilled) on a uniform shared 1D grid; like
// TASK_PREDICT it also writes the log-likelihood of the same factorisation when SmallArgs::ll is set.
enum Task { TASK_LL = 0, TASK_PREDICT = 1, TASK_LOO = 2, TASK_MATRICES = 3, TASK_FACTOR = 4, TASK_PREDICT_F = 5, TASK_PREDICT_FU = 6,
            TASK_PREDICT_U = 7 };

struct SmallArgs {
  int64_t n_obj;
  const int* n_obj_dev;    // optional: the number of work items is read from device memory (<= n_obj, which
                           // then only sizes the grid) -- device-side optimiser loops, no host round trip
  const int64_t* off;      // CSR [n_obj+1]
  const int* order;        // optional processing order (object ids), may be null
  const double* x;         // dim doubles per point
  const double* y;
  const double* y0;        // may be null
  const double* yerr;      // may be null
  Cov cov;
  // per-object hyperparameters (lock-step per-object fits): when hyp_obj != null object b uses
  // hyp_obj[b*n_hyp ..] and nugget_obj[b] (or nugget_shared) instead of `cov`
  const double* hyp_obj; int n_hyp; const double* nugget_obj; double nugget_shared; double floor_shared; unsigned flags;
  int compact_io;          // with `order`: hyp_obj / nugget_obj / ll / info are indexed by position in `order`, not by object id
  int* info;               // [n_obj]
  // TASK_LL
  double* ll;              // [n_obj]
  // TASK_PREDICT
  const double* xnew;
  const int64_t* goff;     // null -> shared grid of m_shared points
  int64_t m_shared;
  const double* new_y0;    // may be null
  const double* new_y0_diff; // non-null: new_y0 is ONE shared row (m_shared values) and object b adds new_y0_diff[b]
  double* mean;
  double* var;             // may be null
  int split;               // CTAs per object (each takes every split-th block of 8 grid points)
  // optional, TASK_PREDICT on per-object grids: object oi has the work items [part_off[oi], part_off[oi+1]) (device,
  // n_obj+1 entries, every object at least one item), which replace `split`; n_parts = part_off[n_obj] sizes the launch
  const int64_t* part_off; int64_t n_parts;
  double* fws;             // TASK_FACTOR / TASK_PREDICT_F: factor workspace, fws_stride doubles per object
  int64_t fws_stride;
  // TASK_LOO
  int loo_mode;
  double* pred; double* pvar; double* pull; double* resid;
  // TASK_MATRICES
  const int64_t* moff;
  double* kmat; double* kinv;
  double* linv;            // L^-1 (lower, zeros above), row-major, same offsets as kmat / kinv
  int64_t mld;             // leading dimension of the matrix outputs (0 -> N of the object)
  // matrix source: when non-null the covariance of object b is READ from amat + aoff[b] (row-major,
  // leading dimension lda, lower triangle) instead of being generated from x (blocked large-object path)
  const double* amat; const int64_t* aoff; int64_t lda;
  const int64_t* ld_obj;   // TASK_MATRICES, optional: object b's leading dimension of amat and of the matrix outputs
                           // (replaces lda and mld), for groups of matrices of different sizes
  double* logdet;          // TASK_MATRICES: sum of log pivots per object (may be null)
  // TASK_PREDICT (N <= 64 kernel): when non-null, row (out0 + m) of vout (8 NB doubles per row) receives
  // v = L^-1 e(x*_m, .) of grid point m (unit amplitude) -- the factor of the bulk predictive-covariance writer
  double* vout;
};

// Work item w of a grid-spreading task -> the position oi of its object; part / parts: which of the object's items it
// is and how many the object has.  `split` items per object, or the table part_off (SmallArgs; binary search, as the
// grouped GEMM finds its problem).  Each item takes every parts-th block of 8 grid points of its object.
__device__ __forceinline__ int64_t work_item(const int64_t* part_off, int64_t n_obj, int split, int64_t w, int& part, int& parts) {
  if (!part_off) {
    const int64_t oi = w / split;
    part = (int)(w - oi * split); parts = split;
    return oi;
  }
  int64_t lo = 0, hi = n_obj - 1;
  while (lo < hi) {
    const int64_t mid = (lo + hi + 1) >> 1;
    if (part_off[mid] <= w) lo = mid; else hi = mid - 1;
  }
  part = (int)(w - part_off[lo]); parts = (int)(part_off[lo + 1] - part_off[lo]);
  return lo;
}

struct GemmArgs {          // C[m x n] = beta*C + alpha * A[m x k] * B[n x k]^T, all row-major
  const double* a; const double* b; double* c;
  int64_t lda, ldb, ldc;
  int m, n, k;             // multiples of 128 / 128 / 16
  double alpha, beta;
  int lower_only;          // 1: only tiles with row-block >= col-block (SYRK on the lower triangle)
};
int launch_gemm_nt(const GemmArgs& g, cudaStream_t stream);

// large-object building blocks (cgp_large.cu); all return cudaError_t as int
int large_cov_build(int dim, const Cov& cov, int autocov, const double* xc, int64_t n, const double* xr, int64_t m,
                    const double* yerr, double* out, int64_t ld, int64_t rows_pad, int64_t cols_pad, cudaStream_t st);
int large_potrf(double* a, int64_t n_pad, int64_t ld, double* logdet_out, int* info_out, cudaStream_t st);
int large_potrs(const double* a, int64_t n_pad, int64_t ld, double* v, double* z_out, int backward, cudaStream_t st);
int large_potrs_backward(const double* a, int64_t n_pad, int64_t ld, double* v, cudaStream_t st);
int large_trsm_rows(const double* a, int64_t n_pad, int64_t ld, double* v, int64_t ldv, int64_t rows, cudaStream_t st);
int large_stream_mean(int dim, const Cov& cov, const double* x, const double* alpha, int64_t n,
                      const double* xnew, const double* new_y0, int64_t m, double* mean, cudaStream_t st);
int large_row_var(const double* v, int64_t ldv, int64_t n_pad, int64_t rows, double amp_star, double* var, cudaStream_t st);
int large_spline_mean(const double* t, const double* c, int nt, const double* x, int64_t n_pts, const int64_t* off,
                      int64_t n_obj, const double* diff, double* out, cudaStream_t st);
int large_moments(const double* v, int64_t n, double center, double* out2, cudaStream_t st);
int large_ll_total(const double* ll, const int* info, int64_t n, double* out2, cudaStream_t st);
// cov[b] = amp_auto K(g,g) + nugget^2 I - amp_cross^2 V_b V_b^T for objects b of a chunk (V rows from SmallArgs::vout, ldv doubles).
// hyp_obj null: every object uses `cov`; otherwise object b uses hyp_obj[b * nh ..] and nugget_obj[b] (null -> nugget)
int large_cov_gram(int dim, const Cov& cov, const double* hyp_obj, const double* nugget_obj, double nugget, unsigned flags,
                   const double* grid, const int64_t* goff, int64_t m_shared, int64_t n_obj,
                   const double* v, int ldv, const int* info, double* out, const int64_t* coff, cudaStream_t st);
int large_dot_sq(const double* v, int64_t n, double* out, cudaStream_t st);
int large_residual(const double* y, const double* y0, int64_t n, int64_t n_pad, double* r, cudaStream_t st);
int large_sum(const double* v, int64_t n, double* out, cudaStream_t st);
// negd[m] = -diag(K^-1)_m from the blocked factor, chunk_rows (% 128 == 0) rows at a time in v (chunk_rows x n_pad)
int large_diag_inv(const double* a, int64_t n_pad, int64_t ld, double* v, int64_t chunk_rows, double* negd, cudaStream_t st);
int large_loo(const double* a, int64_t n, int64_t n_pad, int64_t ld, const Cov& cov, const double* y, const double* m,
              const double* yerr, int recenter, const int* info, double* vwork, int64_t chunk_rows,
              double* pred, double* pvar, double* pull, double* resid, cudaStream_t st);
// grouped likelihood of large objects with per-object hyperparameters (see cgp_large_ll_objhyp_dev)
int64_t large_ll_ws_doubles(int64_t n);
int large_ll_grouped(int dim, const int64_t* off, const double* x, const double* y, const double* y0, const double* yerr,
                     const double* hyp_obj, const double* nugget_obj, double nugget, double floor, unsigned flags,
                     const int* order, int64_t n_active, double* ll, int* info, double* work, int64_t work_doubles,
                     cudaStream_t st);
// grouped predictive covariance matrices of large objects, covs[j] (data covariance, with the floor) and covs_g[j] (H and
// K**, without it) built on the host (see cgp_large_covariance_dev)
int64_t large_cov_ws_doubles(int64_t n, int64_t m);
int large_cov_grouped(int dim, const int64_t* off, const double* x, const double* yerr, const Cov* covs, const Cov* covs_g,
                      const double* xnew, const int64_t* goff, int64_t m_shared, const int* order, int64_t n_active, double* out,
                      const int64_t* coff, int* info, double* work, int64_t work_doubles, cudaStream_t st);

// Launchers (cgp_small.cu).  max_n = largest object in the batch.  Return cudaError_t as int.
int launch_small(Task task, int dim, int max_n, const SmallArgs& a, cudaStream_t stream);
size_t small_smem_bytes(Task task, int dim, int nb);

// N <= 64 fast path (cgp_small64.cu, one TU per dim/task)
int launch_small64_d1_t0(int nb, const SmallArgs& a, cudaStream_t stream);
int launch_small64_d1_t1(int nb, const SmallArgs& a, cudaStream_t stream);
int launch_small64_d1_t2(int nb, const SmallArgs& a, cudaStream_t stream);
int launch_small64_d2_t0(int nb, const SmallArgs& a, cudaStream_t stream);
int launch_small64_d2_t1(int nb, const SmallArgs& a, cudaStream_t stream);
int launch_small64_d2_t2(int nb, const SmallArgs& a, cudaStream_t stream);
int launch_small64_d1_t4(int nb, const SmallArgs& a, cudaStream_t stream);
int launch_small64_d1_t5(int nb, const SmallArgs& a, cudaStream_t stream);
int launch_small64_d2_t4(int nb, const SmallArgs& a, cudaStream_t stream);
int launch_small64_d2_t5(int nb, const SmallArgs& a, cudaStream_t stream);
int launch_small64_d1_t6(int nb, const SmallArgs& a, cudaStream_t stream);
int launch_small64_d1_t7(int nb, const SmallArgs& a, cudaStream_t stream);
// doubles per object in the factor workspace for nb blocks of 8 points
inline int64_t factor_ws_doubles(int nb) { return (int64_t)(nb * (nb + 1) / 2) * 64 + 8 * nb; }

// device-side Nelder-Mead over all objects (cgp_fit.cu); returns cudaError_t as int
int fit_nelder_mead(int64_t n_obj, const int64_t* off, int max_n, int dim,
                    const double* x, const double* y, const double* y0, const double* y_err,
                    const double* x0, int n_par, double nugget, double floor, unsigned flags,
                    double xatol, double fatol, int maxiter, int maxfun,
                    double* x_out, double* f_out, int* it_out, int* fc_out, cudaStream_t st);

// FP64 ceiling probes (cgp_small.cu)
int measure_fp64_peak(int kind, double* tflops);

void count_launch(int n = 1);

// uniform-grid fast path of the factored prediction (cgp_api.cu): the check on a host copy of the grid, and the
// entry point that trusts it (cgp_predict_factored_dev verifies by reading the grid back from the device)
int uniform_grid_ok(const double* grid_host, int64_t m, const double* hyp);
int predict_factored(int64_t n_obj, const int64_t* off, int max_n, int dim, const double* x,
                     const double* hyp, double nugget, unsigned flags, const double* ws, const int* info,
                     const double* xnew, const int64_t* goff, int64_t m_shared,
                     const double* new_y0, double* mean, double* var, int uniform, void* stream,
                     const double* template_offsets = nullptr);   // CGP_MEAN_TEMPLATE: offsets from here instead of new_y0 + m_shared

// records the message cgp_last_error() returns (thread-local) and hands back `code` (cgp_api.cu)
int fail(int code, const char* fmt, ...);

}  // namespace cgp
