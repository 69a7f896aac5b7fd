/* cosmogp_b200 -- C ABI of the B200 (sm_100a) Gaussian-process hot path.
 *
 * Drop-in boundary for PFLeget/cosmogp (reference citations are file:line into
 * that repository).  The reference has no FFI; its only plugin seams are
 *   (1) the inverse operators `svd` / `chol` bound at cosmogp/Gaussian_process.py:6-9
 *       (svd_tmv.computeSVDInverse / computeLDLInverse if importable),
 *   (2) the kernel callable chosen at cosmogp/Gaussian_process.py:136-154,
 *   (3) the object API (Gaussian_process / build_pull) whose per-object Python
 *       loops (Gaussian_process.py:207,264,304,349; pull.py:51,66) are the hot path.
 * Each entry point below replaces one of those loops or operators for a whole
 * batch of objects.  INTEGRATION.md shows the ctypes stubs a cosmogp maintainer
 * would add.
 *
 * Conventions
 *   - every function returns int: 0 ok; <0 error (text via cgp_last_error());
 *     >0 = number of objects whose covariance was not positive definite
 *     (the LinAlgError of scipy.linalg.cholesky at cosmogp/inv_matrix.py:23);
 *     their info[] holds the 1-based failing pivot and their outputs are NaN.
 *   - "_dev" functions take DEVICE pointers and a cudaStream_t (as void*); they
 *     enqueue work and return without synchronising unless stated.
 *     "_host" functions take HOST pointers, do H2D + compute + D2H and return
 *     when the outputs are valid.
 *   - ragged batches are CSR: off[n_obj+1] (int64) into x / y / y0 / y_err.
 *     "_dev" functions also take max_n, the largest object size in the batch (the
 *     host picks the kernel configuration from it); pass 0 to have the library read
 *     off[] back from the device (this synchronises the stream).
 *     x holds dim doubles per point (dim = 1: RBF1D, dim = 2: RBF2D, xy interleaved).
 *     y0 and y_err may be NULL (zeros), like the reference defaults
 *     (Gaussian_process.py:161-169,187).
 *   - hyp = [sigma, l] (dim 1, cosmogp/kernel.py:25-77) or
 *           [sigma, l_x, l_y, l_xy] (dim 2, cosmogp/kernel.py:80-155).
 *   - flags: CGP_AMP_ON_AUTOCOV applies sigma^2 to the 2D auto-covariance; the
 *     default (0) reproduces HEAD, which omits it (kernel.py:146-148).
 *     CGP_MEAN_TEMPLATE (prediction entry points, shared grid only): new_y0 is
 *     not one row per object but the SHARED mean template on the grid (m_shared
 *     values) followed by one offset per object (n_obj values, the reference's
 *     `diff`): mean function of object b at grid point j = new_y0[j] +
 *     new_y0[m_shared + b] -- what mean.py:92-101 evaluates per object, without
 *     materialising (or uploading) n_obj x m_shared doubles.
 *     CGP_GRID_UNIFORM (prediction entry points, dim 1, shared grid, shared hyp): a hint that
 *     xnew[j] = xnew[0] + j*delta.  The library verifies it (to 4 ulp) and that l >= |delta|; the
 *     cross-covariance of 16 grid rows is then built from two exps per data point
 *     (exp(-(g_0 + k delta - x)^2 / 2 l^2) = E(x) R(x)^k C_k) instead of one per (grid point, data point).
 *     Results agree with the general path to ~1e-14 relative; without the flag nothing changes.
 *   - all arithmetic is IEEE float64.
 */
#ifndef COSMOGP_B200_H
#define COSMOGP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CGP_AMP_ON_AUTOCOV 1u      /* opt-in fix of the 2D sigma^2 omission */
#define CGP_MEAN_TEMPLATE  2u      /* new_y0 = [template on the shared grid | per-object offsets] */
#define CGP_GRID_UNIFORM   4u      /* hint: the shared 1D grid is uniformly spaced (verified by the library) */

#define CGP_SMALL_MAX_N 224        /* largest object the shared-memory path takes */

/* leave-one-out mean handling (cosmogp/pull.py:43-102, SURVEY.md row a8) */
#define CGP_LOO_PLAIN    0         /* pred = m + loo(y - m); m may be NULL (modes A, C) */
#define CGP_LOO_RECENTER 1         /* diff re-estimated on the N-1 kept points (modes B, D) */

/* ---- library ------------------------------------------------------------ */
int         cgp_version(void);
const char* cgp_last_error(void);
/* number of visible CUDA devices, <0 on error */
int         cgp_device_count(void);
/* measured FP64 ceiling of the current device in TFLOP/s: kind 0 = DFMA, 1 = DMMA (m8n8k4). */
int         cgp_fp64_peak(int kind, double* tflops);
/* kernels launched by this library since load (all streams); bench.py reports the delta. */
int64_t     cgp_launch_count(void);

/* ---- log-likelihood: replaces the loop of Gaussian_process.compute_log_likelihood
 *      (cosmogp/Gaussian_process.py:191-213) over log_likelihood_gp (:13-75) with
 *      svd_method=False (Cholesky, inv_matrix.py:21-31).
 *      ll_obj[n_obj]: per-object log-likelihood; info[n_obj]. */
int cgp_ll_batched_dev(int64_t n_obj, const int64_t* off, int max_n, int dim,
                       const double* x, const double* y, const double* y0, const double* y_err,
                       const double* hyp, double nugget, double floor, unsigned flags,
                       double* ll_obj, int* info, void* stream);
/* host buffers; *ll_sum = sum over objects in index order (Gaussian_process.py:205-213). */
/* The likelihood evaluation as the optimiser sees it (cosmogp/Gaussian_process.py:205-213: the sum over objects):
 * cgp_ll_batched_dev followed by a reduction on the device.  total_dev[2] (device) receives
 * { sum of ll_obj in a fixed order, number of objects with info != 0 }; when total_host (pinned host memory, 2 doubles)
 * is given the 16 bytes are copied there, the stream is synchronised and the return value is the number of
 * non-positive-definite objects -- one call, 16 bytes over PCIe per simplex point.  ll_obj / info stay on the device. */
int cgp_ll_total_dev(int64_t n_obj, const int64_t* off, int max_n, int dim,
                     const double* x, const double* y, const double* y0, const double* y_err,
                     const double* hyp, double nugget, double floor, unsigned flags,
                     double* ll_obj, int* info, double* total_dev, double* total_host, void* stream);
int cgp_ll_batched_host(int64_t n_obj, const int64_t* off, int dim,
                        const double* x, const double* y, const double* y0, const double* y_err,
                        const double* hyp, double nugget, double floor, unsigned flags,
                        double* ll_obj, int* info, double* ll_sum);

/* ---- host-resident batches, pipelined.  A streamer owns n_streams CUDA streams and one set of device
 *      buffers per stream for chunks of up to chunk_objects objects of EXACTLY n_pts points each and a
 *      shared grid of m_grid points.  cgp_streamer_run cuts the batch into chunks and, per chunk and
 *      stream: uploads the inputs, evaluates the log-likelihood (Gaussian_process.py:205-213) and the
 *      prediction on the grid (:270-361) at the same hyperparameters, downloads ll / mean / var / info --
 *      chunk k uploads while chunk k-1 computes and chunk k-2 downloads (PCIe is full duplex).  All
 *      pointers are HOST pointers (page-locked memory is needed for the copies to overlap); y0, y_err,
 *      new_y0 and var may be NULL; new_y0 is (n_obj, m_grid) or, with CGP_MEAN_TEMPLATE, [template | offsets].
 *      ll_sum = ll[0] + ll[1] + ... in that order.  Returns the number of objects whose covariance was not
 *      positive definite (their info[] != 0), or < 0.  h2d_bytes / d2h_bytes (may be NULL) count the copies. */
typedef struct cgp_streamer cgp_streamer;
/* host only: the chunk sizes cgp_streamer_run uses for n_obj objects (a ramp 2048, x1.6 ... up to chunk_objects,
 * equal chunks in the middle, a x2 ramp down; plain equal chunks when chunk_objects < 2048 or n_pts > 64).
 * Writes up to max_sizes entries, returns the number of chunks (sizes may be NULL), or -1. */
int64_t cgp_streamer_schedule(int64_t n_obj, int64_t chunk_objects, int n_pts, int64_t* sizes, int64_t max_sizes);
int cgp_streamer_create(int64_t chunk_objects, int n_pts, int64_t m_grid, int dim, int n_streams, cgp_streamer** out);
void cgp_streamer_destroy(cgp_streamer* s);
/* Optional: the mean template as scipy's cubic spline (host arrays t, c of n_knots entries, see cgp_spline_mean_dev).
 * A run with y0 == NULL and CGP_MEAN_TEMPLATE then evaluates y0 = S(x) + offset of the object on the device instead
 * of uploading it.  t == NULL clears it. */
int cgp_streamer_set_mean_spline(cgp_streamer* s, const double* t, const double* c, int n_knots);
int cgp_streamer_run(cgp_streamer* s, int64_t n_obj,
                     const double* x, const double* y, const double* y0, const double* y_err,
                     const double* hyp, double nugget, double floor, unsigned flags,
                     const double* xnew, const double* new_y0,
                     double* ll, double* mean, double* var, int* info, double* ll_sum,
                     int64_t* h2d_bytes, int64_t* d2h_bytes);

/* ---- per-object fits: one likelihood evaluation where object b uses its OWN hyperparameters
 *      hyp_obj[b*nh .. b*nh+nh) (nh = 2 or 4) and nugget_obj[b] (NULL -> the shared `nugget`).
 *      order (device, may be NULL) restricts the evaluation to n_active object ids; hyp_obj,
 *      nugget_obj, ll_obj and info are then COMPACT (entry k belongs to object order[k]); without
 *      order they are indexed by object id.  This is the batched form of the reference's per-object loop
 *      `gaussian_process(y[i], x[i]).find_hyperparameters()` (docs/notebook/1D_kernel_example_with_noise.ipynb
 *      cell 13): scipy's Nelder-Mead runs in lock step over all objects on the host. */
int cgp_ll_objhyp_dev(int64_t n_obj, const int64_t* off, int max_n, int dim,
                      const double* x, const double* y, const double* y0, const double* y_err,
                      const double* hyp_obj, const double* nugget_obj, double nugget, double floor, unsigned flags,
                      const int* order, int64_t n_active, double* ll_obj, int* info, void* stream);

/* Log-likelihoods of objects of ANY size (up to 65535 points) through the blocked HBM factorisation of cgp_potrf_dev,
 * all active objects of a wave sharing each launch, each object with its own hyperparameter row: per-object fits of
 * objects above 224 points, and joint fits of batches that hold one.
 * off_host: the CSR offsets (HOST copy); x, y, y0 (may be NULL), y_err (may be NULL): device arrays of the batch.
 * order_host (HOST, may be NULL = objects 0 .. n_obj-1) lists the n_active object ids to evaluate; hyp_rows_host
 * (k x nh, nh = 2 or 4) and nugget_rows_host (k, may be NULL -> `nugget`) are HOST rows, row j for order_host[j]
 * (shared hyperparameters: one row repeated); ll_obj and info (k each) are device arrays indexed by position in the
 * list.  The covariance function of each object is built on the host, as cgp_cov_matrix_dev builds it, so that
 * ll_obj[j] and info[j] are bit for bit those of cgp_cov_matrix_dev + cgp_potrf_dev + cgp_large_solve_dev on that
 * object alone (dense.LargeObject.factor), whatever the other objects of the call, their order or the wave it lands
 * in: ll_obj = -0.5 ((|z|^2 + log det K) + n log 2 pi), NaN where info != 0 (the first failing pivot, as cgp_potrf_dev
 * reports it); an object without points gives -0.0.
 * work: caller-owned device workspace of work_doubles doubles (16-byte aligned); an object of n points needs
 * cgp_large_ll_ws_doubles(n) of it.  Consecutive objects are packed into waves that fit; a workspace of at least
 * the sum over the active objects runs them as one wave.  Does not synchronise.  Returns 0, or < 0 with nothing
 * launched (-2 for a workspace below the largest active object's need). */
int64_t cgp_large_ll_ws_doubles(int64_t n);
int cgp_large_ll_rows_dev(int64_t n_obj, const int64_t* off_host, int dim,
                          const double* x, const double* y, const double* y0, const double* y_err,
                          const double* hyp_rows_host, const double* nugget_rows_host, double nugget, double floor,
                          unsigned flags, const int* order_host, int64_t n_active, double* ll_obj, int* info,
                          double* work, int64_t work_doubles, void* stream);

/* The whole per-object fit on the device: scipy.optimize.fmin's Nelder-Mead (what
 * Gaussian_process.py:246-247 calls) as one state machine per object, the objective of all pending
 * trial points evaluated by one batched likelihood launch per step; the host only enqueues launches.
 * start, par_out: (n_obj, n_par) device arrays, n_par = nh (nugget fixed to `nugget`) or nh+1 (the last
 * parameter is the object's nugget, Gaussian_process.py:241-245).  nll_out = -log-likelihood at par_out
 * (+inf where the covariance never was positive definite), iterations / evaluations as scipy reports
 * them.  xatol, fatol, maxiter, maxfun as in scipy (fmin defaults: 1e-4, 1e-4, 200*n_par, 200*n_par).
 * Synchronises the stream before returning. */
int cgp_fit_objects_dev(int64_t n_obj, const int64_t* off, int max_n, int dim,
                        const double* x, const double* y, const double* y0, const double* y_err,
                        const double* start, int n_par, double nugget, double floor, unsigned flags,
                        double xatol, double fatol, int maxiter, int maxfun,
                        double* par_out, double* nll_out, int* iterations, int* evaluations, void* stream);

/* prediction and pulls with per-object hyperparameters (hyp_obj / nugget_obj indexed by object id):
 * the rest of the reference's per-object loop (fit, predict, build_pull with each object's own fit). */
int cgp_predict_objhyp_dev(int64_t n_obj, const int64_t* off, int max_n, int dim,
                           const double* x, const double* y, const double* y0, const double* y_err,
                           const double* hyp_obj, const double* nugget_obj, double nugget, double floor, unsigned flags,
                           const double* xnew, const int64_t* goff, int64_t m_shared,
                           const double* new_y0, double* mean, double* var, int* info, void* stream);
int cgp_loo_objhyp_dev(int64_t n_obj, const int64_t* off, int max_n, int dim,
                       const double* x, const double* y, const double* m, const double* y_err,
                       const double* hyp_obj, const double* nugget_obj, double nugget, double floor, unsigned flags,
                       int mode, double* pred, double* pred_var, double* pull, double* resid,
                       int* info, void* stream);

/* ---- prediction: replaces Gaussian_process.get_prediction + get_covariance_matrix
 *      (cosmogp/Gaussian_process.py:270-361).
 *      Grid: if goff == NULL the m_shared points of xnew are shared by all objects
 *      (new_binning given) and outputs are (n_obj, m_shared) row-major; otherwise
 *      goff[n_obj+1] is a CSR into xnew / new_y0 / mean / var (per-object grids:
 *      new_binning=None or one grid per object).  Below 296 objects the entry then reads
 *      goff back (one synchronisation) to spread long grids over several CTAs.
 *      new_y0 (mean function on the grid, may be NULL) has the output layout.
 *      mean = H K^-1 (y - y0) + new_y0                      (:332-335)
 *      var  = diag(K(x*,x*) + nugget^2 - H K^-1 H^T)         (:356-361), may be NULL. */
int cgp_predict_batched_dev(int64_t n_obj, const int64_t* off, int max_n, int dim,
                            const double* x, const double* y, const double* y0, const double* y_err,
                            const double* hyp, double nugget, double floor, unsigned flags,
                            const double* xnew, const int64_t* goff, int64_t m_shared,
                            const double* new_y0, double* mean, double* var, int* info, void* stream);
int cgp_predict_batched_host(int64_t n_obj, const int64_t* off, int dim,
                             const double* x, const double* y, const double* y0, const double* y_err,
                             const double* hyp, double nugget, double floor, unsigned flags,
                             const double* xnew, const int64_t* goff, int64_t m_shared,
                             const double* new_y0, double* mean, double* var, int* info);

/* ---- one pass of the hot path: compute_log_likelihood (cosmogp/Gaussian_process.py:191-213) AND get_prediction
 *      (:270-361) at the same hyperparameters from ONE factorisation per object -- what a fit's final evaluation
 *      followed by the interpolation amounts to.  Arguments as cgp_predict_batched_dev plus ll_obj[n_obj]
 *      (per-object log-likelihood, NaN where info != 0).  Objects of <= 64 points: a single kernel, the covariance
 *      and its factor never leave shared memory. */
int cgp_step_batched_dev(int64_t n_obj, const int64_t* off, int max_n, int dim,
                         const double* x, const double* y, const double* y0, const double* y_err,
                         const double* hyp, double nugget, double floor, unsigned flags,
                         const double* xnew, const int64_t* goff, int64_t m_shared,
                         const double* new_y0, double* ll_obj, double* mean, double* var, int* info, void* stream);

/* ---- factor once, predict on any number of grids (objects of <= 64 points): the two halves of
 *      cgp_predict_batched_dev as separate calls.  ws holds, per object, the Cholesky factor as 8x8 tiles in the
 *      kernels' tile layout (inv(L_JJ) on the diagonal, -L[I][J] below) followed by z = L^-1 (y - y0): an opaque
 *      block of cgp_factor_ws_doubles(max_n) doubles each, to be consumed by cgp_predict_factored_dev only.
 *      cgp_predict_factored_dev stages each object's factor into shared memory with one TMA bulk
 *      copy; var may be NULL.  hyp / nugget / flags must be those used for the factorisation.
 *      ll_obj (may be NULL) receives each object's log-likelihood (Gaussian_process.py:13-75) from the
 *      same factorisation: an evaluation of LL and prediction at the same hyperparameters factorises once. */
int64_t cgp_factor_ws_doubles(int max_n);
int cgp_factor_batched_dev(int64_t n_obj, const int64_t* off, int max_n, int dim,
                           const double* x, const double* y, const double* y0, const double* y_err,
                           const double* hyp, double nugget, double floor, unsigned flags,
                           double* ws, double* ll_obj, int* info, void* stream);
int cgp_predict_factored_dev(int64_t n_obj, const int64_t* off, int max_n, int dim, const double* x,
                             const double* hyp, double nugget, unsigned flags, const double* ws, const int* info,
                             const double* xnew, const int64_t* goff, int64_t m_shared,
                             const double* new_y0, double* mean, double* var, void* stream);

/* ---- leave-one-out pulls: replaces build_pull.compute_pull (cosmogp/pull.py:43-102)
 *      by the closed form on diag(K^-1).  m (template mean incl. any fixed diff) may be
 *      NULL.  Outputs (each sum-of-N doubles, any may be NULL): pred, pred_var, pull, resid. */
int cgp_loo_batched_dev(int64_t n_obj, const int64_t* off, int max_n, int dim,
                        const double* x, const double* y, const double* m, const double* y_err,
                        const double* hyp, double nugget, double floor, unsigned flags, int mode,
                        double* pred, double* pred_var, double* pull, double* resid,
                        int* info, void* stream);
int cgp_loo_batched_host(int64_t n_obj, const int64_t* off, int dim,
                         const double* x, const double* y, const double* m, const double* y_err,
                         const double* hyp, double nugget, double floor, unsigned flags, int mode,
                         double* pred, double* pred_var, double* pull, double* resid, int* info);

/* ---- covariance_matrix of every object at once: replaces the loop of get_covariance_matrix
 *      (cosmogp/Gaussian_process.py:340-361).  cov[b] = K(grid,grid) + nugget^2 I - H K^-1 H^T, row-major M x M
 *      blocks: at b * m_shared^2 for a shared grid, at coff[b] for per-object grids (then goff (device), goff_host
 *      (the same offsets on the host) and coff (device, CSR of M_b^2) are all required).  Objects of <= 64 points.
 *      NaN blocks where info != 0. */
int cgp_covariance_batched_dev(int64_t n_obj, const int64_t* off, int max_n, int dim,
                               const double* x, const double* y_err,
                               const double* hyp, double nugget, double floor, unsigned flags,
                               const double* xnew, const int64_t* goff, const int64_t* goff_host, int64_t m_shared,
                               double* cov, const int64_t* coff, int* info, void* stream);
/* cgp_covariance_batched_dev where object b uses its OWN hyperparameters hyp_obj[b*nh .. b*nh+nh) (nh = 2 or 4) and
 * nugget_obj[b] (NULL -> the shared `nugget`), both device arrays indexed by position in this call: the
 * covariance_matrix of each object of a per-object fit (get_prediction(per_object=True, COV=True)).  Same limits,
 * layouts and NaN blocks. */
int cgp_covariance_objhyp_dev(int64_t n_obj, const int64_t* off, int max_n, int dim, const double* x, const double* y_err,
                              const double* hyp_obj, const double* nugget_obj, double nugget, double floor, unsigned flags,
                              const double* xnew, const int64_t* goff, const int64_t* goff_host, int64_t m_shared,
                              double* cov, const int64_t* coff, int* info, void* stream);
/* The covariance matrices of objects of any size (0..65408 points, grids of 0..65408: padded to 128, at most 65535
 * rows), computed for all active objects of a wave at once by the blocked HBM path, each bit for bit as
 * dense.predictive_covariance computes it alone: cov_j = K(g, g) + nugget_j^2 I - V V^T, V = rows of L^-1 H^T, where
 * L L^T = K(x, x) + diag(y_err^2) + (floor^2 + nugget_j^2) I (floor = 0 is dense.predictive_covariance; the floor
 * never enters K(g, g)).  off_host: the CSR offsets (HOST copy); x, y_err (may be NULL): device
 * arrays of the batch.  The grid: one shared grid xnew of m_shared points (goff_host NULL), or object b's grid at
 * xnew + dim * goff_host[b] with goff_host[b+1] - goff_host[b] points (HOST CSR; xnew = x, goff_host = off_host for the
 * objects' own epochs).  order_host (HOST, may be NULL = objects 0 .. n_obj-1) lists the n_active object ids;
 * hyp_rows_host (k x nh) and nugget_rows_host (k, may be NULL -> `nugget`) are HOST arrays indexed by position in the
 * list (shared hyperparameters: one row repeated), as is coff_host (k+1, CSR of m_j^2: cov_j is the m_j x m_j
 * row-major block at cov + coff_host[j]) and info (k, device).  A block is all NaN where info != 0 (the first failing
 * pivot, as cgp_potrf_dev reports it).  work: caller-owned device workspace of work_doubles doubles (16-byte aligned);
 * an object of n points on a grid of m needs cgp_large_cov_ws_doubles(n, m) of it; consecutive objects are packed into
 * waves that fit.  An object's result does not depend on the other objects of the call, their order or the wave it
 * lands in.  Does not synchronise.  Returns 0, or < 0 with nothing launched (-2 for a workspace below the largest
 * active object's need). */
int64_t cgp_large_cov_ws_doubles(int64_t n, int64_t m);
int cgp_large_covariance_dev(int64_t n_obj, const int64_t* off_host, int dim, const double* x, const double* y_err,
                             const double* hyp_rows_host, const double* nugget_rows_host, double nugget, double floor,
                             unsigned flags, const double* xnew, const int64_t* goff_host, int64_t m_shared,
                             const int* order_host, int64_t n_active, double* cov, const int64_t* coff_host, int* info,
                             double* work, int64_t work_doubles, void* stream);
/* The means (and variance diagonals) of objects of any size (0..65408 points) on grids of any length, computed for all
 * active objects of a wave at once by the blocked HBM path, each bit for bit what cgp_cov_matrix_dev + cgp_potrf_dev +
 * cgp_large_solve_dev (dense.LargeObject.factor) followed by cgp_large_predict_dev compute for it alone:
 * mean_j = amp_cross H K^-1 (y - y0) + new_y0 and var_j = (amp_auto + nugget_j^2) - |rows of L^-1 H^T|^2, where
 * L L^T = K(x, x) + diag(y_err^2) + (floor^2 + nugget_j^2) I.  Objects, grids, order_host, hyp_rows_host and
 * nugget_rows_host as in cgp_large_covariance_dev; y, y0 (may be NULL) and y_err (may be NULL): device arrays of the
 * batch.  moff_host (HOST, k+1): CSR of m_j over the list; object order_host[j]'s outputs are mean / var + moff_host[j]
 * (device; var NULL: means only) and it reads new_y0 + moff_host[j] (device, may be NULL: zero mean function).
 * info (k, device): the first failing pivot; NaN rows where info != 0.  Variances are computed chunk_rows (a positive
 * multiple of 128) grid rows per object at a time; a row's bits do not depend on chunk_rows.  work: caller-owned device
 * workspace of work_doubles doubles (16-byte aligned); an object of n points on a grid of m needs
 * cgp_large_pred_ws_doubles(n, var ? min(m, chunk_rows) : 0) of it; consecutive objects are packed into waves that fit.
 * Does not synchronise.  Returns 0, or < 0 with nothing launched (-2 for a workspace below the largest active object's
 * need). */
int64_t cgp_large_pred_ws_doubles(int64_t n, int64_t rows);
int cgp_large_predict_objhyp_dev(int64_t n_obj, const int64_t* off_host, int dim, const double* x, const double* y,
                                 const double* y0, const double* y_err, const double* hyp_rows_host,
                                 const double* nugget_rows_host, double nugget, double floor, unsigned flags,
                                 const double* xnew, const int64_t* goff_host, int64_t m_shared, const double* new_y0,
                                 const int* order_host, int64_t n_active, const int64_t* moff_host, double* mean,
                                 double* var, int* info, int64_t chunk_rows, double* work, int64_t work_doubles,
                                 void* stream);
/* Leave-one-out pulls of objects of any size (0..65408 points), computed for all active objects of a wave at once by the
 * blocked HBM path, each output bit for bit what cgp_cov_matrix_dev + cgp_potrf_dev + cgp_large_loo_dev (with the same
 * hyperparameters, floor, flags, mode and chunk_rows) compute for it alone (dense.LargeLoo.run).  Objects, order_host,
 * hyp_rows_host and nugget_rows_host as in cgp_large_covariance_dev; y, m (may be NULL) and y_err (may be NULL): device
 * arrays of the batch; mode: CGP_LOO_PLAIN or CGP_LOO_RECENTER.  Object order_host[j]'s outputs go to pred / pred_var /
 * pull / resid + off_host[b] (device, the batch's own layout; each may be NULL); points of objects not listed are not
 * touched.  info (k, device): the first failing pivot; the object's outputs are NaN where info != 0.  diag(K^-1) is
 * solved chunk_rows (a positive multiple of 128) identity rows at a time; the bits depend on chunk_rows as those of
 * cgp_large_loo_dev do.  work: caller-owned device workspace of work_doubles doubles (16-byte aligned); an object of
 * n points needs cgp_large_loo_ws_doubles(n, chunk_rows) of it, whatever the mode; consecutive objects are packed into
 * waves that fit.  Does not synchronise.  Returns 0, or < 0 with nothing launched (-2 for a workspace below the largest
 * active object's need). */
int64_t cgp_large_loo_ws_doubles(int64_t n, int64_t chunk_rows);
int cgp_large_loo_objhyp_dev(int64_t n_obj, const int64_t* off_host, int dim, const double* x, const double* y,
                             const double* m, const double* y_err, const double* hyp_rows_host,
                             const double* nugget_rows_host, double nugget, double floor, unsigned flags, int mode,
                             const int* order_host, int64_t n_active, int* info, double* pred, double* pred_var,
                             double* pull, double* resid, int64_t chunk_rows, double* work, int64_t work_doubles,
                             void* stream);

/* ---- matrices for the attribute surface (kernel_matrix, inv_kernel_matrix:
 *      Gaussian_process.py:256-267, 319-325).  moff[n_obj+1]: CSR into the outputs in
 *      doubles (object b is an N_b x N_b row-major block).  kmat / kinv may be NULL. */
int cgp_matrices_batched_dev(int64_t n_obj, const int64_t* off, int max_n, int dim,
                             const double* x, const double* y_err,
                             const double* hyp, double nugget, double floor, unsigned flags,
                             const int64_t* moff, double* kmat, double* kinv, int* info, void* stream);

/* ======================================================================================
 * Large single objects (N > CGP_SMALL_MAX_N; BASELINE configs 3 and 4) and the per-matrix
 * operator seams.  The covariance lives in HBM in a caller-provided (n_pad x n_pad) row-major
 * buffer, n_pad = cgp_pad128(n); rows/columns beyond n are identity padding.
 * ==================================================================================== */
int64_t cgp_pad128(int64_t n);

/* kernel(x, hyp, new_x, nugget, floor, y_err) -- the kernel-callable seam of
 * cosmogp/Gaussian_process.py:136-154 (cosmogp/kernel.py:25-77, 80-155).
 * xnew == NULL: auto-covariance, out is (rows_pad x cols_pad) >= (n x n) with the noise diagonal
 * (and identity padding); else cross-covariance K(xnew, x) of shape (m x n), zero padding. */
int cgp_cov_matrix_dev(int dim, const double* x, int64_t n, const double* xnew, int64_t m,
                       const double* y_err, const double* hyp, double nugget, double floor, unsigned flags,
                       double* out, int64_t ld, int64_t rows_pad, int64_t cols_pad, void* stream);

/* Blocked Cholesky, in place on the lower triangle (scipy.linalg.cholesky at
 * cosmogp/inv_matrix.py:23).  On exit the strictly-lower 128-blocks hold L and each diagonal
 * 128-block holds inv(L_kk) (zeros above its diagonal).  logdet (device double) = sum 2 log L_ii
 * (inv_matrix.py:28); info (device int) = 1-based failing pivot or 0. */
int cgp_potrf_dev(double* a, int64_t n_pad, int64_t ld, double* logdet, int* info, void* stream);

/* v <- L^-1 v, optionally copied to z_out, then (backward != 0) v <- L^-T v. v has n_pad entries. */
int cgp_potrs_dev(const double* a, int64_t n_pad, int64_t ld, double* v, double* z_out, int backward, void* stream);

/* r = y - y0 (zero padded), z = L^-1 r, *quad = |z|^2 (device double), alpha = K^-1 r.
 * With cgp_potrf_dev's logdet this is log_likelihood_gp (cosmogp/Gaussian_process.py:68-73):
 * LL = -(quad + logdet + n log 2 pi)/2. */
int cgp_large_solve_dev(const double* a, int64_t n, int64_t n_pad, int64_t ld,
                        const double* y, const double* y0, double* alpha, double* quad, void* stream);

/* Prediction against a factored large object (cosmogp/Gaussian_process.py:332-361, diagonal of
 * the covariance): mean by a streaming kernel that never stores K(x*,x); var (may be NULL) by a
 * blocked triangular solve on chunks of `chunk_rows` grid points (multiple of 128) staged in
 * vwork (chunk_rows x n_pad doubles). */
int cgp_large_predict_dev(const double* a, int64_t n, int64_t n_pad, int64_t ld, int dim, const double* x,
                          const double* alpha, const double* hyp, double nugget, unsigned flags,
                          const double* xnew, int64_t m, const double* new_y0, double* mean, double* var,
                          double* vwork, int64_t chunk_rows, void* stream);

/* Leave-one-out pulls of one object factored by cgp_potrf_dev (build_pull.compute_pull, cosmogp/pull.py:43-102,
 * for objects of any size), with the closed form and the mean modes of cgp_loo_batched_dev.  hyp / nugget / floor /
 * flags must be those the factored covariance was built with; y, m (may be NULL), y_err (may be NULL) hold n values.
 * diag(K^-1) comes from a blocked triangular solve on identity rows, N^3/3 FLOPs on the FP64 tensor pipe, in chunks
 * of `chunk_rows` rows (multiple of 128) staged in vwork (chunk_rows x n_pad doubles).  info (device int) is the
 * factorisation's: where it is nonzero the outputs are NaN (read on the device, no synchronisation).  Outputs
 * (n doubles each, any may be NULL): pred, pred_var, pull, resid. */
int cgp_large_loo_dev(const double* a, int64_t n, int64_t n_pad, int64_t ld, int dim,
                      const double* y, const double* m, const double* y_err,
                      const double* hyp, double nugget, double floor, unsigned flags, int mode,
                      const int* info, double* vwork, int64_t chunk_rows,
                      double* pred, double* pred_var, double* pull, double* resid, void* stream);

/* v_m = L^-1 h_m for `rows` rows of V (rows x n_pad, rows % 128 == 0), in place. */
int cgp_trsm_rows_dev(const double* a, int64_t n_pad, int64_t ld, double* v, int64_t ldv, int64_t rows, void* stream);

/* The mean function at the epochs, on the device: out[i] = S(x[i]) + diff[object of i], S the cubic spline through
 * the template (cosmogp/mean.py:28-31: InterpolatedUnivariateSpline(Time_mean, Mean_Y)) given by its FITPACK knots t
 * (n_knots) and B-spline coefficients c (n_knots; what scipy keeps in spl._eval_args), evaluated like FITPACK's splev
 * (extrapolating with the end polynomials).  dim 1 only.  off / n_obj / diff may be NULL / 0 / NULL (no offsets).
 * All pointers are device pointers.  Saves the upload of one double per data point (mean.py:84-90's y0). */
int cgp_spline_mean_dev(const double* t, const double* c, int n_knots, const double* x, int64_t n_pts,
                        const int64_t* off, int64_t n_obj, const double* diff, double* out, void* stream);

/* host only: 1 when a shared 1D grid (host array of m points) qualifies for the CGP_GRID_UNIFORM kernel with
 * hyperparameters hyp = [sigma, l]: grid[j] = grid[0] + j*delta to within 4 ulp and |l| >= |delta| > 0.
 * This is the check the prediction entry points apply to the hint. */
int cgp_grid_is_uniform(const double* grid_host, int64_t m, const double* hyp);

/* Centred moments of a device vector: out2[0] = sum (v[i] - center), out2[1] = sum (v[i] - center)^2
 * (out2: 2 doubles on the device; fixed summation order, reproducible).  Two calls give what
 * scipy.stats.norm.fit(pull) returns at cosmogp/pull.py:102 (mean, then the population standard
 * deviation about it) without bringing 10^6 x N pulls to the host. */
int cgp_moments_dev(const double* v, int64_t n, double center, double* out2, void* stream);

/* C[m x n] = beta C + alpha A[m x k] B[n x k]^T on the FP64 tensor pipe; m, n % 128 == 0, k % 16 == 0;
 * lower_only != 0 computes only the tiles on or below the block diagonal. */
int cgp_gemm_nt_dev(const double* a, int64_t lda, const double* b, int64_t ldb, double* c, int64_t ldc,
                    int64_t m, int64_t n, int64_t k, double alpha, double beta, int lower_only, void* stream);

/* ---- single-process multi-GPU context (SURVEY section 8(b)): the objects of a batch are sharded over the GPUs of
 *      one box in contiguous ranges balanced by sum N^3; every GPU keeps its shard resident and runs the kernels of
 *      the one-GPU entry points; nothing is exchanged on the data path.  What the reference does in ONE Python loop
 *      over objects (cosmogp/Gaussian_process.py:205-213, :304-335; cosmogp/pull.py:66-94) stays one call with one
 *      set of host arrays in and out.  NCCL (ncclCommInitAll over the context's devices) is loaded at run time from
 *      the libnccl.so.2 of the process (PyTorch ships one) or from cgp_set_nccl_library(path); it carries the final
 *      gather of per-object outputs on device 0 over NVLink (gather = 1) and the scalar all-reduce.
 *      gather = 0: every device writes its slice of the host outputs over its own PCIe link (no exchange at all).
 *      Calls on one context are serialised by the caller; each call returns with the host outputs valid. */
int cgp_set_nccl_library(const char* path);
int cgp_shard_ranges(int64_t n_obj, const int64_t* off, int n_parts, int64_t* starts /* n_parts + 1 */);   /* host only */
int cgp_ctx_create(int n_dev /* <= 0: all */, const int* dev_ids /* NULL: 0..n_dev-1 */, void** ctx);
void cgp_ctx_destroy(void* ctx);
int cgp_ctx_info(void* ctx, int* n_dev, int* have_nccl);
/* thin NCCL wrappers on per-device buffers: send_dev[d] (counts[d] doubles on device d) -> recv_root_dev (on device
 * `root`, sum of counts) by ncclSend / ncclRecv in one group; buf_dev[d] (count doubles each) summed in place. */
int cgp_ctx_gather_f64(void* ctx, double* const* send_dev, const int64_t* counts, double* recv_root_dev, int root);
int cgp_ctx_allreduce_sum_f64(void* ctx, double* const* buf_dev, int64_t count);
/* a batch (HOST arrays, CSR like the *_host entry points) uploaded once and kept resident, shard by shard */
int cgp_ctx_batch_create(void* ctx, int64_t n_obj, const int64_t* off, int dim,
                         const double* x, const double* y, const double* y0, const double* y_err, void** batch);
void cgp_ctx_batch_destroy(void* batch);
int cgp_ctx_batch_ranges(void* batch, int64_t* starts /* n_dev + 1 */);
/* compute_log_likelihood (Gaussian_process.py:191-213): one launch + one reduction per device, 16 bytes back from
 * each, added in device order; ll_obj / info (host, n_obj) may be NULL.  Returns the number of non-PD objects. */
int cgp_ctx_batch_ll(void* batch, const double* hyp, double nugget, double floor, unsigned flags,
                     double* ll_sum, double* ll_obj, int* info);
/* get_prediction on a shared grid (:270-361); with ll_obj != NULL also the likelihood from the same factorisation
 * (cgp_step_batched_dev).  new_y0: NULL, (n_obj, m), or with CGP_MEAN_TEMPLATE the packed [template (m) | offsets (n_obj)]. */
int cgp_ctx_batch_predict(void* batch, const double* hyp, double nugget, double floor, unsigned flags,
                          const double* xnew, int64_t m, const double* new_y0,
                          double* ll_obj, double* mean, double* var, int* info, int gather);
/* build_pull.compute_pull (pull.py:43-102) in closed form; the batch's y0 is the template mean.  moments (2 doubles,
 * may be NULL): sum of the pulls and of their squares (norm.fit, pull.py:102), all-reduced over NVLink when gather = 1. */
int cgp_ctx_batch_loo(void* batch, const double* hyp, double nugget, double floor, unsigned flags, int mode,
                      double* pred, double* pred_var, double* pull, double* resid, int* info, double* moments, int gather);

#ifdef __cplusplus
}
#endif
#endif /* COSMOGP_B200_H */
