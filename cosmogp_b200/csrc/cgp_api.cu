// C ABI of cosmogp_b200 (see include/cosmogp_b200.h for the contract and the
// reference interfaces each entry point replaces).  No C++ exception crosses it.
#include "../../include/cosmogp_b200.h"
#include "cgp_internal.h"

#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdint>
#include <cstdlib>
#include <vector>

namespace cgp {

static thread_local char g_err[512] = "";
static std::atomic<int64_t> g_launches{0};

void count_launch(int n) { g_launches += n; }

int fail(int code, const char* fmt, ...) {
  va_list ap; va_start(ap, fmt);
  vsnprintf(g_err, sizeof g_err, fmt, ap);
  va_end(ap);
  return code;
}
static int cuda_fail(int e, const char* where) {
  return fail(-100 - e, "%s: CUDA error %d (%s)", where, e, cudaGetErrorString((cudaError_t)e));
}

#define CGP_ERR_ARG   (-1)
#define CGP_ERR_SIZE  (-2)

// hyp -> Cov  (cosmogp/kernel.py:71-75 for 1D, :127-151 for 2D)
static int make_cov(int dim, const double* hyp, double nugget, double floor, unsigned flags, Cov* c) {
  if (!hyp) return fail(CGP_ERR_ARG, "hyp is NULL");
  if (dim != 1 && dim != 2) return fail(CGP_ERR_ARG, "dim must be 1 or 2, got %d", dim);
  *c = cov_from_hyp(dim, hyp, nugget, floor, flags);
  return 0;
}

static int max_n_from_device(int64_t n_obj, const int64_t* off_dev, cudaStream_t st, int* max_n) {
  std::vector<int64_t> h((size_t)n_obj + 1);
  cudaError_t e = cudaMemcpyAsync(h.data(), off_dev, sizeof(int64_t) * (n_obj + 1), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return cuda_fail((int)e, "read off[]");
  int64_t m = 0;
  for (int64_t i = 0; i < n_obj; ++i) { int64_t n = h[i + 1] - h[i]; if (n > m) m = n; }
  *max_n = (int)m;
  return 0;
}
static int max_n_host(int64_t n_obj, const int64_t* off) {
  int64_t m = 0;
  for (int64_t i = 0; i < n_obj; ++i) { int64_t n = off[i + 1] - off[i]; if (n > m) m = n; }
  return (int)m;
}

static int run_small(Task task, int dim, int max_n, SmallArgs& a, cudaStream_t st, const char* who) {
  if (a.n_obj == 0) return 0;
  if (max_n > CGP_SMALL_MAX_N)
    return fail(CGP_ERR_SIZE, "%s: object with %d points exceeds the shared-memory path (max %d); "
                "use the large-object entry points", who, max_n, CGP_SMALL_MAX_N);
  int e = launch_small(task, dim, max_n, a, st);
  if (e) return cuda_fail(e, who);
  return 0;
}

// CGP_GRID_UNIFORM is a hint: the recurrence kernel (TASK_PREDICT_FU) runs only if the shared 1D grid really is
// g0 + j*delta to within a few ulp and the length scale is at least one spacing (see cgp_small64.cu).
// `grid` is a host copy.  Returns 1 when the fast path applies.
int uniform_grid_ok(const double* grid, int64_t m, const double* hyp) {
  if (!grid || !hyp || m < 2) return 0;
  const double g0 = grid[0], delta = (grid[m - 1] - g0) / (double)(m - 1);
  const double l = std::fabs(hyp[1]);
  if (!(delta != 0.0) || !std::isfinite(delta) || !std::isfinite(g0) || !(l >= std::fabs(delta))) return 0;
  double gmax = std::fabs(g0) > std::fabs(grid[m - 1]) ? std::fabs(g0) : std::fabs(grid[m - 1]);
  const double tol = 4.0 * 2.220446049250313e-16 * (gmax > 0.0 ? gmax : 1.0);
  for (int64_t j = 0; j < m; ++j)
    if (!(std::fabs(grid[j] - std::fma((double)j, delta, g0)) <= tol)) return 0;
  return 1;
}
static int uniform_grid_ok_dev(const double* xnew_dev, int64_t m, const double* hyp, cudaStream_t st) {
  if (m < 2 || m > (int64_t)1 << 24) return 0;
  std::vector<double> g((size_t)m);
  cudaError_t e = cudaMemcpyAsync(g.data(), xnew_dev, sizeof(double) * (size_t)m, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) { cudaGetLastError(); return 0; }
  return uniform_grid_ok(g.data(), m, hyp);
}

// ---- tiny RAII helpers for the _host entry points ------------------------------------
struct DevBuf {
  void* p = nullptr; cudaStream_t st;
  explicit DevBuf(cudaStream_t s) : st(s) {}
  ~DevBuf() { if (p) cudaFreeAsync(p, st); }
  cudaError_t alloc(size_t bytes) { return cudaMallocAsync(&p, bytes ? bytes : 8, st); }
  template <class T> T* as() { return (T*)p; }
};
struct HostCall {
  cudaStream_t st = nullptr; cudaError_t err = cudaSuccess;
  HostCall() { err = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking); }
  ~HostCall() { if (st) cudaStreamDestroy(st); }
  // upload n elements (or leave null when the host pointer is null)
  template <class T> const T* up(DevBuf& b, const T* h, size_t n) {
    if (!h || err != cudaSuccess) return nullptr;
    err = b.alloc(n * sizeof(T));
    if (err == cudaSuccess) err = cudaMemcpyAsync(b.p, h, n * sizeof(T), cudaMemcpyHostToDevice, st);
    return b.as<T>();
  }
  template <class T> T* out(DevBuf& b, const T* h, size_t n) {
    if (!h || err != cudaSuccess) return nullptr;
    err = b.alloc(n * sizeof(T));
    return b.as<T>();
  }
  template <class T> void down(T* h, DevBuf& b, size_t n) {
    if (!h || err != cudaSuccess) return;
    err = cudaMemcpyAsync(h, b.p, n * sizeof(T), cudaMemcpyDeviceToHost, st);
  }
  bool sync() { if (err == cudaSuccess) err = cudaStreamSynchronize(st); return err == cudaSuccess; }
};

// Stream-ordered allocations are recycled instead of being returned to the driver at every
// synchronisation (the default release threshold is 0): workspaces of ~1 GB per call would
// otherwise cost milliseconds of cudaMalloc each time.
static void keep_pool_memory() {
  static thread_local int done_for = -1;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev == done_for) return;
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
    unsigned long long keep = ~0ULL;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
  }
  done_for = dev;
}

static int count_bad(const int* info, int64_t n) {
  int64_t c = 0;
  for (int64_t i = 0; i < n; ++i) c += info[i] != 0;
  return c > 2147483647 ? 2147483647 : (int)c;
}

// The active objects order[0 .. k) (object ids; NULL: 0 .. k) of a grouped large-object entry: each must be an object
// id with 0 .. max_pts points and pass check(j, b, n, w), the entry's own checks, which set w to its workspace; the
// workspace must hold the largest w.
template <class F>
static int check_active(const char* name, int64_t n_obj, const int64_t* off, const int* order, int64_t k, int64_t max_pts,
                        int64_t work_doubles, F&& check) {
  int64_t need = 0;
  for (int64_t j = 0; j < k; ++j) {
    const int64_t b = order ? order[j] : j;
    if (b < 0 || b >= n_obj) return fail(CGP_ERR_ARG, "%s: order[%lld] = %lld is not an object id", name, (long long)j, (long long)b);
    const int64_t n = off[b + 1] - off[b];
    if (n < 0 || n > max_pts)
      return fail(CGP_ERR_SIZE, "%s: object %lld has %lld points (0..%lld)", name, (long long)b, (long long)n, (long long)max_pts);
    int64_t w = 0;
    if (int rc = check(j, b, n, w)) return rc;
    if (w > need) need = w;
  }
  if (work_doubles < need)
    return fail(CGP_ERR_SIZE, "%s: workspace of %lld doubles is below the %lld the largest active object needs", name,
                (long long)work_doubles, (long long)need);
  return 0;
}

// Cov of the active objects on the host from their hyperparameter rows, as the per-object paths build them: covs[j]
// with the floor (the data covariance only), covs_g[j] without it.  Nugget j: nugget_rows[j], or `nugget` when NULL.
static void host_covs(int dim, const double* hyp_rows, const double* nugget_rows, double nugget, double floor, unsigned flags,
                      int64_t k, std::vector<Cov>& covs, std::vector<Cov>& covs_g) {
  const int nh = dim == 1 ? 2 : 4;
  covs.resize((size_t)k); covs_g.resize((size_t)k);
  for (int64_t j = 0; j < k; ++j) {
    const double nu = nugget_rows ? nugget_rows[j] : nugget;
    covs[j] = cov_from_hyp(dim, hyp_rows + j * nh, nu, floor, flags);
    covs_g[j] = cov_from_hyp(dim, hyp_rows + j * nh, nu, 0.0, flags);
  }
}

static int no_checks() { return 0; }

// The steps every grouped large-object entry shares, in this order: the object counts; pre(), the entry's checks that
// hold with no active object; the return for no active object; the NULL arguments (`args`: the entry's own pointers are
// set); dim; the alignment of work; post(), the entry's remaining argument checks; check_active with max_pts and the
// entry's per-object check; the host Covs of the active objects (host_covs); then launch(k, covs, covs_g), whose CUDA
// error is reported under `name`.
template <class Pre, class Post, class Check, class Launch>
static int grouped_entry(const char* name, int64_t n_obj, const int64_t* off, int dim, const int* order, int64_t n_active,
                         bool args, const double* hyp_rows, const double* nugget_rows, double nugget, double floor,
                         unsigned flags, const double* work, int64_t work_doubles, int64_t max_pts, Pre&& pre, Post&& post,
                         Check&& check, Launch&& launch) {
  if (n_obj < 0 || n_active < 0) return fail(CGP_ERR_ARG, "%s: negative object count", name);
  if (int rc = pre()) return rc;
  const int64_t k = order ? n_active : n_obj;
  if (k == 0) return 0;
  if (!args || !off || !hyp_rows || !work) return fail(CGP_ERR_ARG, "%s: NULL argument", name);
  if (dim != 1 && dim != 2) return fail(CGP_ERR_ARG, "dim must be 1 or 2, got %d", dim);
  if ((uintptr_t)work & 15) return fail(CGP_ERR_ARG, "%s: work must be 16-byte aligned", name);
  if (int rc = post()) return rc;
  if (int rc = check_active(name, n_obj, off, order, k, max_pts, work_doubles, check)) return rc;
  std::vector<Cov> covs, covs_g;
  host_covs(dim, hyp_rows, nugget_rows, nugget, floor, flags, k, covs, covs_g);
  keep_pool_memory();
  const int e = launch(k, covs.data(), covs_g.data());
  return e ? cuda_fail(e, name) : 0;
}
// padded sizes stay within the 65535 rows cgp_cov_matrix_dev builds an auto-covariance for
static const int64_t LARGE_MAX_PTS = 65535 / 128 * 128;

}  // namespace cgp

using namespace cgp;

extern "C" {

int cgp_version(void) { return 100; }
const char* cgp_last_error(void) { return g_err; }
int64_t cgp_launch_count(void) { return g_launches.load(); }

int cgp_device_count(void) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) return cuda_fail((int)e, "cgp_device_count");
  return n;
}

int cgp_fp64_peak(int kind, double* tflops) {
  if (!tflops || kind < 0 || kind > 1) return fail(CGP_ERR_ARG, "cgp_fp64_peak: bad arguments");
  int e = measure_fp64_peak(kind, tflops);
  return e ? cuda_fail(e, "cgp_fp64_peak") : 0;
}

// ------------------------------------------------------------------------------------ LL
int cgp_ll_batched_dev(int64_t n_obj, const int64_t* off, int max_n, int dim,
                       const double* x, const double* y, const double* y0, const double* y_err,
                       const double* hyp, double nugget, double floor, unsigned flags,
                       double* ll_obj, int* info, void* stream) {
  if (n_obj < 0 || (n_obj && (!off || !x || !y || !ll_obj || !info)))
    return fail(CGP_ERR_ARG, "cgp_ll_batched_dev: NULL argument");
  cudaStream_t st = (cudaStream_t)stream;
  SmallArgs a; memset(&a, 0, sizeof a);
  int rc = make_cov(dim, hyp, nugget, floor, flags, &a.cov);
  if (rc) return rc;
  if (n_obj && max_n <= 0 && (rc = max_n_from_device(n_obj, off, st, &max_n))) return rc;
  a.n_obj = n_obj; a.off = off; a.x = x; a.y = y; a.y0 = y0; a.yerr = y_err;
  a.ll = ll_obj; a.info = info;
  return run_small(TASK_LL, dim, max_n, a, st, "cgp_ll_batched_dev");
}

int cgp_ll_total_dev(int64_t n_obj, const int64_t* off, int max_n, int dim,
                     const double* x, const double* y, const double* y0, const double* y_err,
                     const double* hyp, double nugget, double floor, unsigned flags,
                     double* ll_obj, int* info, double* total_dev, double* total_host, void* stream) {
  if (n_obj < 0 || !total_dev) return fail(CGP_ERR_ARG, "cgp_ll_total_dev: NULL argument");
  cudaStream_t st = (cudaStream_t)stream;
  int rc = cgp_ll_batched_dev(n_obj, off, max_n, dim, x, y, y0, y_err, hyp, nugget, floor, flags, ll_obj, info, stream);
  if (rc) return rc;
  keep_pool_memory();
  int e = large_ll_total(ll_obj, info, n_obj, total_dev, st);
  if (e) return cuda_fail(e, "cgp_ll_total_dev (reduction)");
  if (!total_host) return 0;
  cudaError_t ce = cudaMemcpyAsync(total_host, total_dev, 2 * sizeof(double), cudaMemcpyDeviceToHost, st);
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(st);
  if (ce != cudaSuccess) return cuda_fail((int)ce, "cgp_ll_total_dev (read back)");
  return total_host[1] > 2147483647.0 ? 2147483647 : (int)total_host[1];
}

int cgp_ll_batched_host(int64_t n_obj, const int64_t* off, int dim,
                        const double* x, const double* y, const double* y0, const double* y_err,
                        const double* hyp, double nugget, double floor, unsigned flags,
                        double* ll_obj, int* info, double* ll_sum) {
  if (n_obj < 0 || (n_obj && (!off || !x || !y || !ll_obj || !info)))
    return fail(CGP_ERR_ARG, "cgp_ll_batched_host: NULL argument");
  if (ll_sum) *ll_sum = 0.0;
  if (n_obj == 0) return 0;
  const size_t np = (size_t)off[n_obj];
  HostCall hc;
  DevBuf b_off(hc.st), b_x(hc.st), b_y(hc.st), b_y0(hc.st), b_e(hc.st), b_ll(hc.st), b_info(hc.st);
  const int64_t* d_off = hc.up(b_off, off, (size_t)n_obj + 1);
  const double* d_x = hc.up(b_x, x, np * dim);
  const double* d_y = hc.up(b_y, y, np);
  const double* d_y0 = hc.up(b_y0, y0, np);
  const double* d_e = hc.up(b_e, y_err, np);
  double* d_ll = hc.out(b_ll, ll_obj, (size_t)n_obj);
  int* d_info = hc.out(b_info, info, (size_t)n_obj);
  if (hc.err != cudaSuccess) return cuda_fail((int)hc.err, "cgp_ll_batched_host (upload)");
  int rc = cgp_ll_batched_dev(n_obj, d_off, max_n_host(n_obj, off), dim, d_x, d_y, d_y0, d_e, hyp, nugget, floor,
                              flags, d_ll, d_info, hc.st);
  if (rc) return rc;
  hc.down(ll_obj, b_ll, (size_t)n_obj);
  hc.down(info, b_info, (size_t)n_obj);
  if (!hc.sync()) return cuda_fail((int)hc.err, "cgp_ll_batched_host");
  if (ll_sum) { double s = 0.0; for (int64_t i = 0; i < n_obj; ++i) s += ll_obj[i]; *ll_sum = s; }
  return count_bad(info, n_obj);
}

// One likelihood evaluation with PER-OBJECT hyperparameters (device arrays): the building block of
// lock-step per-object fits (the notebook loop `for i: gaussian_process(y[i], x[i]).find_hyperparameters()`).
int cgp_ll_objhyp_dev(int64_t n_obj, const int64_t* off, int max_n, int dim,
                      const double* x, const double* y, const double* y0, const double* y_err,
                      const double* hyp_obj, const double* nugget_obj, double nugget, double floor, unsigned flags,
                      const int* order, int64_t n_active, double* ll_obj, int* info, void* stream) {
  if (n_obj < 0 || (n_obj && (!off || !x || !y || !hyp_obj || !ll_obj || !info)))
    return fail(CGP_ERR_ARG, "cgp_ll_objhyp_dev: NULL argument");
  if (dim != 1 && dim != 2) return fail(CGP_ERR_ARG, "dim must be 1 or 2, got %d", dim);
  if (max_n <= 0) return fail(CGP_ERR_ARG, "cgp_ll_objhyp_dev: max_n is required");
  SmallArgs a; memset(&a, 0, sizeof a);
  a.n_obj = order ? n_active : n_obj; a.off = off; a.order = order;
  a.x = x; a.y = y; a.y0 = y0; a.yerr = y_err; a.ll = ll_obj; a.info = info;
  a.hyp_obj = hyp_obj; a.n_hyp = dim == 1 ? 2 : 4; a.nugget_obj = nugget_obj; a.nugget_shared = nugget;
  a.floor_shared = floor; a.flags = flags;
  a.compact_io = order ? 1 : 0;
  a.cov = Cov();
  return run_small(TASK_LL, dim, max_n, a, (cudaStream_t)stream, "cgp_ll_objhyp_dev");
}

int64_t cgp_large_ll_ws_doubles(int64_t n) { return n < 0 ? 0 : large_ll_ws_doubles(n); }

int cgp_large_ll_rows_dev(int64_t n_obj, const int64_t* off_host, int dim,
                          const double* x, const double* y, const double* y0, const double* y_err,
                          const double* hyp_rows_host, const double* nugget_rows_host, double nugget, double floor,
                          unsigned flags, const int* order_host, int64_t n_active, double* ll_obj, int* info,
                          double* work, int64_t work_doubles, void* stream) {
  return grouped_entry(
      "cgp_large_ll_rows_dev", n_obj, off_host, dim, order_host, n_active, x && y && ll_obj && info, hyp_rows_host,
      nugget_rows_host, nugget, floor, flags, work, work_doubles, 65535, no_checks, no_checks,
      [](int64_t, int64_t, int64_t n, int64_t& w) { w = large_ll_ws_doubles(n); return 0; },
      [&](int64_t k, const Cov* covs, const Cov*) {   // covs: as cgp_cov_matrix_dev builds them for LargeObject.factor
        return large_ll_grouped(dim, off_host, x, y, y0, y_err, covs, order_host, k, ll_obj, info, work, work_doubles,
                                (cudaStream_t)stream);
      });
}

int64_t cgp_large_cov_ws_doubles(int64_t n, int64_t m) { return n < 0 || m < 0 ? 0 : large_cov_ws_doubles(n, m); }

int cgp_large_covariance_dev(int64_t n_obj, const int64_t* off_host, int dim, const double* x, const double* y_err,
                             const double* hyp_rows_host, const double* nugget_rows_host, double nugget, double floor,
                             unsigned flags, const double* xnew, const int64_t* goff_host, int64_t m_shared,
                             const int* order_host, int64_t n_active, double* cov, const int64_t* coff_host, int* info,
                             double* work, int64_t work_doubles, void* stream) {
  const char* name = "cgp_large_covariance_dev";
  return grouped_entry(
      name, n_obj, off_host, dim, order_host, n_active, x && xnew && cov && coff_host && info, hyp_rows_host,
      nugget_rows_host, nugget, floor, flags, work, work_doubles, LARGE_MAX_PTS, no_checks,
      [&] {
        if (!goff_host && (m_shared < 0 || m_shared > LARGE_MAX_PTS))
          return fail(CGP_ERR_SIZE, "%s: shared grid of %lld points (0..%lld)", name, (long long)m_shared, (long long)LARGE_MAX_PTS);
        return 0;
      },
      [&](int64_t j, int64_t b, int64_t n, int64_t& w) {
        const int64_t m = goff_host ? goff_host[b + 1] - goff_host[b] : m_shared;
        if (m < 0 || m > LARGE_MAX_PTS)
          return fail(CGP_ERR_SIZE, "%s: grid of object %lld has %lld points (0..%lld)", name, (long long)b, (long long)m, (long long)LARGE_MAX_PTS);
        if (coff_host[j + 1] - coff_host[j] != m * m)
          return fail(CGP_ERR_ARG, "%s: coff[%lld + 1] - coff[%lld] is not the grid's %lld^2 entries", name, (long long)j, (long long)j, (long long)m);
        w = large_cov_ws_doubles(n, m);
        return 0;
      },
      [&](int64_t k, const Cov* covs, const Cov* covs_g) {   // as cgp_cov_matrix_dev builds them
        return large_cov_grouped(dim, off_host, x, y_err, covs, covs_g, xnew, goff_host, m_shared, order_host, k, cov,
                                 coff_host, info, work, work_doubles, (cudaStream_t)stream);
      });
}

int64_t cgp_large_pred_ws_doubles(int64_t n, int64_t rows) { return n < 0 || rows < 0 ? 0 : large_pred_ws_doubles(n, rows); }

int cgp_large_predict_objhyp_dev(int64_t n_obj, const int64_t* off_host, int dim, const double* x, const double* y,
                                 const double* y0, const double* y_err, const double* hyp_rows_host,
                                 const double* nugget_rows_host, double nugget, double floor, unsigned flags,
                                 const double* xnew, const int64_t* goff_host, int64_t m_shared, const double* new_y0,
                                 const int* order_host, int64_t n_active, const int64_t* moff_host, double* mean,
                                 double* var, int* info, int64_t chunk_rows, double* work, int64_t work_doubles,
                                 void* stream) {
  const char* name = "cgp_large_predict_objhyp_dev";
  return grouped_entry(
      name, n_obj, off_host, dim, order_host, n_active, x && y && xnew && moff_host && mean && info, hyp_rows_host,
      nugget_rows_host, nugget, floor, flags, work, work_doubles, LARGE_MAX_PTS, no_checks,
      [&] {
        if (var && (chunk_rows <= 0 || chunk_rows % 128)) return fail(CGP_ERR_ARG, "%s: chunk_rows must be a positive multiple of 128", name);
        if (!goff_host && m_shared < 0) return fail(CGP_ERR_ARG, "%s: negative grid size", name);
        return 0;
      },
      [&](int64_t j, int64_t b, int64_t n, int64_t& w) {
        const int64_t m = goff_host ? goff_host[b + 1] - goff_host[b] : m_shared;
        if (m < 0) return fail(CGP_ERR_ARG, "%s: grid of object %lld has %lld points", name, (long long)b, (long long)m);
        if (moff_host[j + 1] - moff_host[j] != m)
          return fail(CGP_ERR_ARG, "%s: moff[%lld + 1] - moff[%lld] is not the grid's %lld points", name, (long long)j, (long long)j, (long long)m);
        w = large_pred_ws_doubles(n, var ? std::min(m, chunk_rows) : 0);
        return 0;
      },
      [&](int64_t k, const Cov* covs, const Cov* covs_g) {   // as LargeObject's make_cov calls build them
        return large_predict_grouped(dim, off_host, x, y, y0, y_err, covs, covs_g, xnew, goff_host, m_shared, new_y0,
                                     order_host, k, moff_host, mean, var, info, chunk_rows, work, work_doubles,
                                     (cudaStream_t)stream);
      });
}

int64_t cgp_large_loo_ws_doubles(int64_t n, int64_t chunk_rows) {
  return n < 0 || chunk_rows <= 0 ? 0 : large_loo_ws_doubles(n, chunk_rows);
}

int cgp_large_loo_objhyp_dev(int64_t n_obj, const int64_t* off_host, int dim, const double* x, const double* y,
                             const double* m, const double* y_err, const double* hyp_rows_host,
                             const double* nugget_rows_host, double nugget, double floor, unsigned flags, int mode,
                             const int* order_host, int64_t n_active, int* info, double* pred, double* pred_var,
                             double* pull, double* resid, int64_t chunk_rows, double* work, int64_t work_doubles,
                             void* stream) {
  const char* name = "cgp_large_loo_objhyp_dev";
  return grouped_entry(
      name, n_obj, off_host, dim, order_host, n_active, x && y && info, hyp_rows_host, nugget_rows_host, nugget, floor,
      flags, work, work_doubles, LARGE_MAX_PTS,
      [&] {
        if (mode != CGP_LOO_PLAIN && mode != CGP_LOO_RECENTER) return fail(CGP_ERR_ARG, "%s: bad mode %d", name, mode);
        if (chunk_rows <= 0 || chunk_rows % 128) return fail(CGP_ERR_ARG, "%s: chunk_rows must be a positive multiple of 128", name);
        return 0;
      },
      no_checks,
      [&](int64_t, int64_t, int64_t n, int64_t& w) { w = large_loo_ws_doubles(n, chunk_rows); return 0; },
      [&](int64_t k, const Cov* covs, const Cov*) {   // covs: as cgp_cov_matrix_dev and cgp_large_loo_dev build them
        return large_loo_grouped(dim, off_host, x, y, m, y_err, covs, mode == CGP_LOO_RECENTER, order_host, k, info, pred,
                                 pred_var, pull, resid, chunk_rows, work, work_doubles, (cudaStream_t)stream);
      });
}

int cgp_fit_objects_dev(int64_t n_obj, const int64_t* off, int max_n, int dim,
                        const double* x, const double* y, const double* y0, const double* y_err,
                        const double* start, int n_par, double nugget, double floor, unsigned flags,
                        double xatol, double fatol, int maxiter, int maxfun,
                        double* par_out, double* nll_out, int* iterations, int* evaluations, void* stream) {
  if (n_obj < 0 || (n_obj && (!off || !x || !y || !start || !par_out || !nll_out || !iterations || !evaluations)))
    return fail(CGP_ERR_ARG, "cgp_fit_objects_dev: NULL argument");
  if (dim != 1 && dim != 2) return fail(CGP_ERR_ARG, "dim must be 1 or 2, got %d", dim);
  const int nh = dim == 1 ? 2 : 4;
  if (n_par != nh && n_par != nh + 1)
    return fail(CGP_ERR_ARG, "cgp_fit_objects_dev: n_par must be %d or %d, got %d", nh, nh + 1, n_par);
  if (n_obj > 2147483647LL) return fail(CGP_ERR_SIZE, "cgp_fit_objects_dev: more than 2^31-1 objects");
  if (max_n <= 0) return fail(CGP_ERR_ARG, "cgp_fit_objects_dev: max_n is required");
  if (max_n > CGP_SMALL_MAX_N)
    return fail(CGP_ERR_SIZE, "cgp_fit_objects_dev: object with %d points exceeds the shared-memory path (max %d)",
                max_n, CGP_SMALL_MAX_N);
  if (maxiter <= 0 || maxfun <= 0) return fail(CGP_ERR_ARG, "cgp_fit_objects_dev: maxiter and maxfun must be positive");
  keep_pool_memory();
  int e = fit_nelder_mead(n_obj, off, max_n, dim, x, y, y0, y_err, start, n_par, nugget, floor, flags,
                          xatol, fatol, maxiter, maxfun, par_out, nll_out, iterations, evaluations, (cudaStream_t)stream);
  if (e) return cuda_fail(e, "cgp_fit_objects_dev");
  return 0;
}

// ------------------------------------------------------------------------------------ predict
// hyp (shared) or hyp_obj / nugget_obj (per object, device arrays indexed by object id)
static void set_objhyp(SmallArgs& a, int dim, const double* hyp_obj, const double* nugget_obj, double nugget,
                       double floor, unsigned flags) {
  a.hyp_obj = hyp_obj; a.n_hyp = dim == 1 ? 2 : 4; a.nugget_obj = nugget_obj; a.nugget_shared = nugget;
  a.floor_shared = floor; a.flags = flags; a.compact_io = 0;
}

static int predict_impl(int64_t n_obj, const int64_t* off, int max_n, int dim,
                        const double* x, const double* y, const double* y0, const double* y_err,
                        const double* hyp, const double* hyp_obj, const double* nugget_obj,
                        double nugget, double floor, unsigned flags,
                        const double* xnew, const int64_t* goff, int64_t m_shared,
                        const double* new_y0, double* ll_obj, double* mean, double* var, int* info, void* stream) {
  if (n_obj < 0 || (n_obj && (!off || !x || !y || !xnew || !mean || !info)))
    return fail(CGP_ERR_ARG, "cgp_predict_batched_dev: NULL argument");
  if (!goff && m_shared < 0) return fail(CGP_ERR_ARG, "cgp_predict_batched_dev: m_shared < 0");
  if (dim != 1 && dim != 2) return fail(CGP_ERR_ARG, "dim must be 1 or 2, got %d", dim);
  cudaStream_t st = (cudaStream_t)stream;
  SmallArgs a; memset(&a, 0, sizeof a);
  int rc = 0;
  if (hyp_obj) set_objhyp(a, dim, hyp_obj, nugget_obj, nugget, floor, flags);
  else rc = make_cov(dim, hyp, nugget, floor, flags, &a.cov);
  if (rc) return rc;
  if (n_obj && max_n <= 0 && (rc = max_n_from_device(n_obj, off, st, &max_n))) return rc;
  a.n_obj = n_obj; a.off = off; a.x = x; a.y = y; a.y0 = y0; a.yerr = y_err; a.info = info;
  a.xnew = xnew; a.goff = goff; a.m_shared = m_shared; a.new_y0 = new_y0; a.mean = mean; a.var = var;
  const bool tmpl = (flags & CGP_MEAN_TEMPLATE) && new_y0;
  if (tmpl) {
    if (goff) return fail(CGP_ERR_ARG, "CGP_MEAN_TEMPLATE needs a shared grid (goff == NULL)");
    a.new_y0_diff = new_y0 + m_shared;
  }
  // few objects with long grids: several CTAs per object, each refactorising (cheap) and
  // taking every split-th block of 8 grid points
  int split = 1;
  if (!goff && n_obj < 296) {
    const int64_t rbs = (m_shared + 7) / 8;
    int64_t want = 592 / (n_obj > 0 ? n_obj : 1);
    int64_t cap = (rbs + 3) / 4;
    if (want > cap) want = cap;
    if (want > 1) split = (int)want;
  }
  a.split = split;
  // per-object grids, few objects: the same spreading with the number of work items set per object, by its share of
  // the grid rows (CGP_GRID_PARTS=0: one item per object).  Every item refactorises its object and the 8-row blocks of
  // the grid phase do not depend on which other blocks a warp takes, so the outputs equal those of one item per object.
  static int grid_parts = -1;
  if (grid_parts < 0) { const char* e = getenv("CGP_GRID_PARTS"); grid_parts = (e && !atoi(e)) ? 0 : 1; }
  int64_t* part_off = nullptr;
  if (goff && grid_parts && n_obj > 0 && n_obj < 296) {
    std::vector<int64_t> g((size_t)n_obj + 1), parts((size_t)n_obj + 1, 0);
    cudaError_t e = cudaMemcpyAsync(g.data(), goff, sizeof(int64_t) * (n_obj + 1), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return cuda_fail((int)e, "read goff[]");
    int64_t rbs_sum = 0;
    for (int64_t b = 0; b < n_obj; ++b) rbs_sum += (g[b + 1] - g[b] + 7) / 8;
    for (int64_t b = 0; b < n_obj; ++b) {
      const int64_t rbs = (g[b + 1] - g[b] + 7) / 8, cap = (rbs + 3) / 4;
      int64_t want = rbs_sum ? (int64_t)llround(592.0 * (double)rbs / (double)rbs_sum) : 1;
      if (want > cap) want = cap;
      parts[b + 1] = parts[b] + (want > 1 ? want : 1);   // an empty grid keeps one item: it writes the info
    }
    if (parts[n_obj] > n_obj) {
      keep_pool_memory();
      e = cudaMallocAsync((void**)&part_off, sizeof(int64_t) * (n_obj + 1), st);
      if (e == cudaSuccess) e = cudaMemcpyAsync(part_off, parts.data(), sizeof(int64_t) * (n_obj + 1), cudaMemcpyHostToDevice, st);
      if (e != cudaSuccess) {
        if (part_off) cudaFreeAsync(part_off, st);
        return cuda_fail((int)e, "cgp_predict_batched_dev (work table)");
      }
      a.part_off = part_off; a.n_parts = parts[n_obj];
    }
  }
  a.ll = ll_obj;                                          // the N <= 64 kernels emit it from the same factorisation
  if (ll_obj && max_n > 64) {                             // the generic kernel does not: one more launch
    SmallArgs l = a; l.split = 1; l.part_off = nullptr;
    if ((rc = run_small(TASK_LL, dim, max_n, l, st, "cgp_step_batched_dev (likelihood)"))) {
      if (part_off) cudaFreeAsync(part_off, st);
      return rc;
    }
    a.ll = nullptr;
  }
  // Many small objects with variances: two kernels by default.  FACTOR (latency-bound factorisation, L^-1 and alpha
  // spilled to a workspace) then PREDICT_F / PREDICT_FU (every warp in the DMMA-dense grid phase, factor staged by
  // TMA).  The one-pass kernel (TASK_PREDICT_U: factorise and predict from the same shared-memory tiles, nothing
  // spilled; CGP_PREDICT_FUSED=1) moves 11x less HBM traffic but is slower on B200 (4.4 vs 4.1 ms at C2, ncu r02c:
  // 20 % of its stalls are instruction fetch -- factorisation + grid code exceed the 32 KB L1.5 instruction cache --
  // and with 11 one-warp CTAs per SM a single warp in the grid phase cannot keep the FP64 pipe busy while its
  // neighbours factorise).  Small batches (< 2048 objects) always take the one-pass kernel.
  static int use_split = -1;
  if (use_split < 0) { const char* e = getenv("CGP_PREDICT_FUSED"); use_split = (e && atoi(e)) ? 0 : 1; }
  if (!use_split && var && max_n <= 64 && n_obj >= 2048 && split == 1 && (flags & CGP_GRID_UNIFORM) && dim == 1 && !goff &&
      !hyp_obj && m_shared >= 2 && uniform_grid_ok_dev(xnew, m_shared, hyp, st))
    return run_small(TASK_PREDICT_U, dim, max_n, a, st, "cgp_predict_batched_dev (one pass, uniform grid)");
  if (use_split && var && max_n <= 64 && n_obj >= 2048 && split == 1) {
    const int nb = max_n < 1 ? 1 : (max_n + 7) / 8;
    const int64_t stride = factor_ws_doubles(nb);
    const int64_t chunk = 65536;
    double* ws = nullptr;
    const bool uniform = (flags & CGP_GRID_UNIFORM) && dim == 1 && !goff && !hyp_obj && uniform_grid_ok_dev(xnew, m_shared, hyp, st);
    keep_pool_memory();
    cudaError_t ce = cudaMallocAsync((void**)&ws, (size_t)((n_obj < chunk ? n_obj : chunk) * stride) * sizeof(double), st);
    if (ce != cudaSuccess) return cuda_fail((int)ce, "cgp_predict_batched_dev (workspace)");
    int rc2 = 0;
    for (int64_t c0 = 0; c0 < n_obj && !rc2; c0 += chunk) {
      SmallArgs f = a;
      f.n_obj = n_obj - c0 < chunk ? n_obj - c0 : chunk;
      f.off = off + c0; f.info = info + c0;
      if (ll_obj) f.ll = ll_obj + c0;
      if (goff) f.goff = goff + c0;
      else {
        f.mean = mean + c0 * m_shared; f.var = var + c0 * m_shared;
        if (tmpl) f.new_y0_diff = a.new_y0_diff + c0;
        else if (new_y0) f.new_y0 = new_y0 + c0 * m_shared;
      }
      f.fws = ws; f.fws_stride = stride;
      if (hyp_obj) { f.hyp_obj = hyp_obj + c0 * f.n_hyp; if (nugget_obj) f.nugget_obj = nugget_obj + c0; }
      rc2 = run_small(TASK_FACTOR, dim, max_n, f, st, "cgp_predict_batched_dev (factor)");
      if (!rc2) rc2 = run_small(uniform ? TASK_PREDICT_FU : TASK_PREDICT_F, dim, max_n, f, st, "cgp_predict_batched_dev (predict)");
    }
    cudaFreeAsync(ws, st);
    return rc2;
  }
  rc = run_small(TASK_PREDICT, dim, max_n, a, st, "cgp_predict_batched_dev");
  if (part_off) cudaFreeAsync(part_off, st);
  return rc;
}

int cgp_predict_batched_dev(int64_t n_obj, const int64_t* off, int max_n, int dim,
                            const double* x, const double* y, const double* y0, const double* y_err,
                            const double* hyp, double nugget, double floor, unsigned flags,
                            const double* xnew, const int64_t* goff, int64_t m_shared,
                            const double* new_y0, double* mean, double* var, int* info, void* stream) {
  return predict_impl(n_obj, off, max_n, dim, x, y, y0, y_err, hyp, nullptr, nullptr, nugget, floor, flags,
                      xnew, goff, m_shared, new_y0, nullptr, mean, var, info, stream);
}

int cgp_step_batched_dev(int64_t n_obj, const int64_t* off, int max_n, int dim,
                         const double* x, const double* y, const double* y0, const double* y_err,
                         const double* hyp, double nugget, double floor, unsigned flags,
                         const double* xnew, const int64_t* goff, int64_t m_shared,
                         const double* new_y0, double* ll_obj, double* mean, double* var, int* info, void* stream) {
  if (n_obj && !ll_obj) return fail(CGP_ERR_ARG, "cgp_step_batched_dev: ll_obj is NULL");
  return predict_impl(n_obj, off, max_n, dim, x, y, y0, y_err, hyp, nullptr, nullptr, nugget, floor, flags,
                      xnew, goff, m_shared, new_y0, ll_obj, mean, var, info, stream);
}

int cgp_predict_objhyp_dev(int64_t n_obj, const int64_t* off, int max_n, int dim,
                           const double* x, const double* y, const double* y0, const double* y_err,
                           const double* hyp_obj, const double* nugget_obj, double nugget, double floor, unsigned flags,
                           const double* xnew, const int64_t* goff, int64_t m_shared,
                           const double* new_y0, double* mean, double* var, int* info, void* stream) {
  if (!hyp_obj) return fail(CGP_ERR_ARG, "cgp_predict_objhyp_dev: hyp_obj is NULL");
  return predict_impl(n_obj, off, max_n, dim, x, y, y0, y_err, nullptr, hyp_obj, nugget_obj, nugget, floor, flags,
                      xnew, goff, m_shared, new_y0, nullptr, mean, var, info, stream);
}

int cgp_predict_batched_host(int64_t n_obj, const int64_t* off, int dim,
                             const double* x, const double* y, const double* y0, const double* y_err,
                             const double* hyp, double nugget, double floor, unsigned flags,
                             const double* xnew, const int64_t* goff, int64_t m_shared,
                             const double* new_y0, double* mean, double* var, int* info) {
  if (n_obj < 0 || (n_obj && (!off || !x || !y || !xnew || !mean || !info)))
    return fail(CGP_ERR_ARG, "cgp_predict_batched_host: NULL argument");
  if (n_obj == 0) return 0;
  const size_t np = (size_t)off[n_obj];
  const size_t ng = goff ? (size_t)goff[n_obj] : (size_t)m_shared;        // grid points stored
  const size_t nout = goff ? (size_t)goff[n_obj] : (size_t)n_obj * (size_t)m_shared;
  HostCall hc;
  DevBuf b_off(hc.st), b_x(hc.st), b_y(hc.st), b_y0(hc.st), b_e(hc.st), b_g(hc.st), b_goff(hc.st),
      b_ny0(hc.st), b_mean(hc.st), b_var(hc.st), b_info(hc.st);
  const int64_t* d_off = hc.up(b_off, off, (size_t)n_obj + 1);
  const double* d_x = hc.up(b_x, x, np * dim);
  const double* d_y = hc.up(b_y, y, np);
  const double* d_y0 = hc.up(b_y0, y0, np);
  const double* d_e = hc.up(b_e, y_err, np);
  const double* d_g = hc.up(b_g, xnew, ng * dim);
  const int64_t* d_goff = hc.up(b_goff, goff, (size_t)n_obj + 1);
  const double* d_ny0 = hc.up(b_ny0, new_y0, (flags & CGP_MEAN_TEMPLATE) ? (size_t)m_shared + (size_t)n_obj : nout);
  double* d_mean = hc.out(b_mean, mean, nout);
  double* d_var = hc.out(b_var, var, nout);
  int* d_info = hc.out(b_info, info, (size_t)n_obj);
  if (hc.err != cudaSuccess) return cuda_fail((int)hc.err, "cgp_predict_batched_host (upload)");
  int rc = cgp_predict_batched_dev(n_obj, d_off, max_n_host(n_obj, off), dim, d_x, d_y, d_y0, d_e, hyp, nugget,
                                   floor, flags, d_g, d_goff, m_shared, d_ny0, d_mean, d_var, d_info, hc.st);
  if (rc) return rc;
  hc.down(mean, b_mean, nout);
  hc.down(var, b_var, nout);
  hc.down(info, b_info, (size_t)n_obj);
  if (!hc.sync()) return cuda_fail((int)hc.err, "cgp_predict_batched_host");
  return count_bad(info, n_obj);
}

// ------------------------------------------------------------------------------------ factor once, predict many
int64_t cgp_factor_ws_doubles(int max_n) {
  if (max_n > 64) return 0;
  return factor_ws_doubles(max_n < 1 ? 1 : (max_n + 7) / 8);
}

int cgp_factor_batched_dev(int64_t n_obj, const int64_t* off, int max_n, int dim,
                           const double* x, const double* y, const double* y0, const double* y_err,
                           const double* hyp, double nugget, double floor, unsigned flags,
                           double* ws, double* ll_obj, int* info, void* stream) {
  if (n_obj < 0 || (n_obj && (!off || !x || !y || !ws || !info))) return fail(CGP_ERR_ARG, "cgp_factor_batched_dev: NULL argument");
  if (max_n <= 0 || max_n > 64) return fail(CGP_ERR_SIZE, "cgp_factor_batched_dev: objects of 1..64 points only (max_n = %d)", max_n);
  SmallArgs a; memset(&a, 0, sizeof a);
  int rc = make_cov(dim, hyp, nugget, floor, flags, &a.cov);
  if (rc) return rc;
  a.n_obj = n_obj; a.off = off; a.x = x; a.y = y; a.y0 = y0; a.yerr = y_err; a.info = info;
  a.fws = ws; a.fws_stride = cgp_factor_ws_doubles(max_n); a.split = 1; a.ll = ll_obj;
  return run_small(TASK_FACTOR, dim, max_n, a, (cudaStream_t)stream, "cgp_factor_batched_dev");
}

int cgp_predict_factored_dev(int64_t n_obj, const int64_t* off, int max_n, int dim, const double* x,
                             const double* hyp, double nugget, unsigned flags, const double* ws, const int* info,
                             const double* xnew, const int64_t* goff, int64_t m_shared,
                             const double* new_y0, double* mean, double* var, void* stream) {
  int uniform = 0;
  if ((flags & CGP_GRID_UNIFORM) && dim == 1 && !goff && xnew && hyp && n_obj > 0)
    uniform = uniform_grid_ok_dev(xnew, m_shared, hyp, (cudaStream_t)stream);
  return cgp::predict_factored(n_obj, off, max_n, dim, x, hyp, nugget, flags, ws, info, xnew, goff, m_shared, new_y0, mean, var,
                               uniform, stream);
}

}  // extern "C"

// uniform: 1 = the caller has verified the grid on the host (uniform_grid_ok), 0 = general kernel
int cgp::predict_factored(int64_t n_obj, const int64_t* off, int max_n, int dim, const double* x,
                          const double* hyp, double nugget, unsigned flags, const double* ws, const int* info,
                          const double* xnew, const int64_t* goff, int64_t m_shared,
                          const double* new_y0, double* mean, double* var, int uniform, void* stream,
                          const double* template_offsets) {
  if (n_obj < 0 || (n_obj && (!off || !x || !ws || !info || !xnew || !mean)))
    return fail(CGP_ERR_ARG, "cgp_predict_factored_dev: NULL argument");
  if (max_n <= 0 || max_n > 64) return fail(CGP_ERR_SIZE, "cgp_predict_factored_dev: objects of 1..64 points only (max_n = %d)", max_n);
  SmallArgs a; memset(&a, 0, sizeof a);
  int rc = make_cov(dim, hyp, nugget, 0.0, flags, &a.cov);
  if (rc) return rc;
  a.n_obj = n_obj; a.off = off; a.x = x; a.info = const_cast<int*>(info);
  a.fws = const_cast<double*>(ws); a.fws_stride = cgp_factor_ws_doubles(max_n);
  a.xnew = xnew; a.goff = goff; a.m_shared = m_shared; a.new_y0 = new_y0; a.mean = mean; a.var = var;
  if ((flags & CGP_MEAN_TEMPLATE) && new_y0) {
    if (goff) return fail(CGP_ERR_ARG, "CGP_MEAN_TEMPLATE needs a shared grid (goff == NULL)");
    a.new_y0_diff = template_offsets ? template_offsets : new_y0 + m_shared;
  }
  int split = 1;
  if (!goff && n_obj < 296) {
    const int64_t rbs = (m_shared + 7) / 8;
    int64_t want = 1628 / (n_obj > 0 ? n_obj : 1), cap = (rbs + 1) / 2;
    if (want > cap) want = cap;
    if (want > 1) split = (int)want;
  }
  a.split = split;
  const bool fu = uniform && dim == 1 && !goff && m_shared >= 2;
  return run_small(fu ? TASK_PREDICT_FU : TASK_PREDICT_F, dim, max_n, a, (cudaStream_t)stream, "cgp_predict_factored_dev");
}

extern "C" {

// ------------------------------------------------------------------------------------ LOO
static int loo_impl(int64_t n_obj, const int64_t* off, int max_n, int dim,
                    const double* x, const double* y, const double* m, const double* y_err,
                    const double* hyp, const double* hyp_obj, const double* nugget_obj,
                    double nugget, double floor, unsigned flags, int mode,
                    double* pred, double* pred_var, double* pull, double* resid,
                    int* info, void* stream) {
  if (n_obj < 0 || (n_obj && (!off || !x || !y || !info)))
    return fail(CGP_ERR_ARG, "cgp_loo_batched_dev: NULL argument");
  if (mode != CGP_LOO_PLAIN && mode != CGP_LOO_RECENTER) return fail(CGP_ERR_ARG, "cgp_loo_batched_dev: bad mode %d", mode);
  if (dim != 1 && dim != 2) return fail(CGP_ERR_ARG, "dim must be 1 or 2, got %d", dim);
  cudaStream_t st = (cudaStream_t)stream;
  SmallArgs a; memset(&a, 0, sizeof a);
  int rc = 0;
  if (hyp_obj) set_objhyp(a, dim, hyp_obj, nugget_obj, nugget, floor, flags);
  else rc = make_cov(dim, hyp, nugget, floor, flags, &a.cov);
  if (rc) return rc;
  if (n_obj && max_n <= 0 && (rc = max_n_from_device(n_obj, off, st, &max_n))) return rc;
  a.n_obj = n_obj; a.off = off; a.x = x; a.y = y; a.y0 = m; a.yerr = y_err; a.info = info;
  a.loo_mode = mode; a.pred = pred; a.pvar = pred_var; a.pull = pull; a.resid = resid;
  return run_small(TASK_LOO, dim, max_n, a, st, "cgp_loo_batched_dev");
}

int cgp_loo_batched_dev(int64_t n_obj, const int64_t* off, int max_n, int dim,
                        const double* x, const double* y, const double* m, const double* y_err,
                        const double* hyp, double nugget, double floor, unsigned flags, int mode,
                        double* pred, double* pred_var, double* pull, double* resid,
                        int* info, void* stream) {
  return loo_impl(n_obj, off, max_n, dim, x, y, m, y_err, hyp, nullptr, nullptr, nugget, floor, flags, mode,
                  pred, pred_var, pull, resid, info, stream);
}

int cgp_loo_objhyp_dev(int64_t n_obj, const int64_t* off, int max_n, int dim,
                       const double* x, const double* y, const double* m, const double* y_err,
                       const double* hyp_obj, const double* nugget_obj, double nugget, double floor, unsigned flags,
                       int mode, double* pred, double* pred_var, double* pull, double* resid,
                       int* info, void* stream) {
  if (!hyp_obj) return fail(CGP_ERR_ARG, "cgp_loo_objhyp_dev: hyp_obj is NULL");
  return loo_impl(n_obj, off, max_n, dim, x, y, m, y_err, nullptr, hyp_obj, nugget_obj, nugget, floor, flags, mode,
                  pred, pred_var, pull, resid, info, stream);
}

int cgp_loo_batched_host(int64_t n_obj, const int64_t* off, int dim,
                         const double* x, const double* y, const double* m, const double* y_err,
                         const double* hyp, double nugget, double floor, unsigned flags, int mode,
                         double* pred, double* pred_var, double* pull, double* resid, int* info) {
  if (n_obj < 0 || (n_obj && (!off || !x || !y || !info)))
    return fail(CGP_ERR_ARG, "cgp_loo_batched_host: NULL argument");
  if (n_obj == 0) return 0;
  const size_t np = (size_t)off[n_obj];
  HostCall hc;
  DevBuf b_off(hc.st), b_x(hc.st), b_y(hc.st), b_m(hc.st), b_e(hc.st), b_p(hc.st), b_v(hc.st), b_pl(hc.st),
      b_r(hc.st), b_info(hc.st);
  const int64_t* d_off = hc.up(b_off, off, (size_t)n_obj + 1);
  const double* d_x = hc.up(b_x, x, np * dim);
  const double* d_y = hc.up(b_y, y, np);
  const double* d_m = hc.up(b_m, m, np);
  const double* d_e = hc.up(b_e, y_err, np);
  double* d_p = hc.out(b_p, pred, np);
  double* d_v = hc.out(b_v, pred_var, np);
  double* d_pl = hc.out(b_pl, pull, np);
  double* d_r = hc.out(b_r, resid, np);
  int* d_info = hc.out(b_info, info, (size_t)n_obj);
  if (hc.err != cudaSuccess) return cuda_fail((int)hc.err, "cgp_loo_batched_host (upload)");
  int rc = cgp_loo_batched_dev(n_obj, d_off, max_n_host(n_obj, off), dim, d_x, d_y, d_m, d_e, hyp, nugget, floor,
                               flags, mode, d_p, d_v, d_pl, d_r, d_info, hc.st);
  if (rc) return rc;
  hc.down(pred, b_p, np); hc.down(pred_var, b_v, np); hc.down(pull, b_pl, np); hc.down(resid, b_r, np);
  hc.down(info, b_info, (size_t)n_obj);
  if (!hc.sync()) return cuda_fail((int)hc.err, "cgp_loo_batched_host");
  return count_bad(info, n_obj);
}

// ------------------------------------------------------------------------------------ predictive covariance, in bulk
// hyp (shared) or hyp_obj / nugget_obj (per object, device arrays indexed by position in this call)
static int covariance_impl(int64_t n_obj, const int64_t* off, int max_n, int dim,
                           const double* x, const double* y_err, const double* hyp, const double* hyp_obj,
                           const double* nugget_obj, double nugget, double floor, unsigned flags,
                           const double* xnew, const int64_t* goff, const int64_t* goff_host, int64_t m_shared,
                           double* cov, const int64_t* coff, int* info, void* stream) {
  const char* name = hyp_obj ? "cgp_covariance_objhyp_dev" : "cgp_covariance_batched_dev";
  char where[64];
  if (n_obj < 0 || (n_obj && (!off || !x || !xnew || !cov || !info))) return fail(CGP_ERR_ARG, "%s: NULL argument", name);
  if (goff && (!goff_host || !coff)) return fail(CGP_ERR_ARG, "%s: per-object grids need goff_host and coff", name);
  if (max_n <= 0 || max_n > 64) return fail(CGP_ERR_SIZE, "%s: objects of 1..64 points (max_n = %d); larger ones go "
                                            "through cgp_cov_matrix_dev / cgp_trsm_rows_dev / cgp_gemm_nt_dev", name, max_n);
  if (n_obj == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  SmallArgs a; memset(&a, 0, sizeof a);
  int rc = 0;
  if (hyp_obj) {
    if (dim != 1 && dim != 2) return fail(CGP_ERR_ARG, "dim must be 1 or 2, got %d", dim);
    set_objhyp(a, dim, hyp_obj, nugget_obj, nugget, floor, flags);
  } else if ((rc = make_cov(dim, hyp, nugget, floor, flags, &a.cov))) {
    return rc;
  }
  const int nb = (max_n + 7) / 8, ldv = 8 * nb;
  keep_pool_memory();
  // chunks of objects bound the workspace of V rows (512 MB) and the z dimension of the gram launch
  const int64_t max_rows = ((int64_t)512 << 20) / (ldv * 8);
  int64_t c0 = 0;
  while (c0 < n_obj && !rc) {
    int64_t c1 = c0, rows = 0, m_max = 0;
    while (c1 < n_obj && c1 - c0 < 65535) {
      const int64_t m = goff ? goff_host[c1 + 1] - goff_host[c1] : m_shared;
      if (c1 > c0 && rows + m > max_rows) break;
      rows += m; if (m > m_max) m_max = m; ++c1;
    }
    double *vws = nullptr, *dummy = nullptr;
    cudaError_t ce = cudaMallocAsync((void**)&vws, (size_t)(rows ? rows : 1) * ldv * sizeof(double), st);
    if (ce == cudaSuccess) ce = cudaMallocAsync((void**)&dummy, (size_t)(rows ? rows : 1) * sizeof(double), st);
    if (ce != cudaSuccess) {
      if (vws) cudaFreeAsync(vws, st);
      snprintf(where, sizeof where, "%s (workspace)", name);
      return cuda_fail((int)ce, where);
    }
    const int64_t row0 = goff ? goff_host[c0] : 0;          // per-object grids index rows absolutely: shift the bases
    SmallArgs f = a;
    f.n_obj = c1 - c0; f.off = off + c0; f.x = x; f.y = x; f.yerr = y_err; f.info = info + c0;
    f.xnew = xnew; f.goff = goff ? goff + c0 : nullptr; f.m_shared = m_shared;
    f.mean = dummy - row0; f.vout = vws - row0 * ldv;
    if (hyp_obj) { f.hyp_obj = hyp_obj + c0 * f.n_hyp; if (nugget_obj) f.nugget_obj = nugget_obj + c0; }
    int split = 1;
    if (!goff && f.n_obj < 296) {
      const int64_t rbs = (m_shared + 7) / 8;
      int64_t want = 592 / f.n_obj, cap = (rbs + 3) / 4;
      if (want > cap) want = cap;
      if (want > 1) split = (int)want;
    }
    f.split = split;
    snprintf(where, sizeof where, "%s (factor)", name);
    rc = run_small(TASK_PREDICT, dim, max_n, f, st, where);
    if (!rc) {
      int e = large_cov_gram(dim, a.cov, f.hyp_obj, f.nugget_obj, nugget, flags, xnew, goff ? goff + c0 : nullptr,
                             goff ? m_max : m_shared, c1 - c0, vws - row0 * ldv, ldv, info + c0,
                             goff ? cov : cov + c0 * m_shared * m_shared, goff ? coff + c0 : nullptr, st);
      if (e) { snprintf(where, sizeof where, "%s (gram)", name); rc = cuda_fail(e, where); }
    }
    cudaFreeAsync(vws, st); cudaFreeAsync(dummy, st);
    c0 = c1;
  }
  return rc;
}

int cgp_covariance_batched_dev(int64_t n_obj, const int64_t* off, int max_n, int dim,
                               const double* x, const double* y_err,
                               const double* hyp, double nugget, double floor, unsigned flags,
                               const double* xnew, const int64_t* goff, const int64_t* goff_host, int64_t m_shared,
                               double* cov, const int64_t* coff, int* info, void* stream) {
  return covariance_impl(n_obj, off, max_n, dim, x, y_err, hyp, nullptr, nullptr, nugget, floor,
                         flags, xnew, goff, goff_host, m_shared, cov, coff, info, stream);
}

int cgp_covariance_objhyp_dev(int64_t n_obj, const int64_t* off, int max_n, int dim, const double* x, const double* y_err,
                              const double* hyp_obj, const double* nugget_obj, double nugget, double floor, unsigned flags,
                              const double* xnew, const int64_t* goff, const int64_t* goff_host, int64_t m_shared,
                              double* cov, const int64_t* coff, int* info, void* stream) {
  if (!hyp_obj) return fail(CGP_ERR_ARG, "cgp_covariance_objhyp_dev: hyp_obj is NULL");
  return covariance_impl(n_obj, off, max_n, dim, x, y_err, nullptr, hyp_obj, nugget_obj, nugget,
                         floor, flags, xnew, goff, goff_host, m_shared, cov, coff, info, stream);
}

// ------------------------------------------------------------------------------------ matrices
int cgp_matrices_batched_dev(int64_t n_obj, const int64_t* off, int max_n, int dim,
                             const double* x, const double* y_err,
                             const double* hyp, double nugget, double floor, unsigned flags,
                             const int64_t* moff, double* kmat, double* kinv, int* info, void* stream) {
  if (n_obj < 0 || (n_obj && (!off || !x || !moff || !info)))
    return fail(CGP_ERR_ARG, "cgp_matrices_batched_dev: NULL argument");
  cudaStream_t st = (cudaStream_t)stream;
  SmallArgs a; memset(&a, 0, sizeof a);
  int rc = make_cov(dim, hyp, nugget, floor, flags, &a.cov);
  if (rc) return rc;
  if (n_obj && max_n <= 0 && (rc = max_n_from_device(n_obj, off, st, &max_n))) return rc;
  a.n_obj = n_obj; a.off = off; a.x = x; a.yerr = y_err; a.info = info;
  a.moff = moff; a.kmat = kmat; a.kinv = kinv;
  return run_small(TASK_MATRICES, dim, max_n, a, st, "cgp_matrices_batched_dev");
}


// ==================================================================================== large objects
int64_t cgp_pad128(int64_t n) { return n <= 0 ? 128 : (n + 127) / 128 * 128; }

int cgp_cov_matrix_dev(int dim, const double* x, int64_t n, const double* xnew, int64_t m,
                       const double* y_err, const double* hyp, double nugget, double floor, unsigned flags,
                       double* out, int64_t ld, int64_t rows_pad, int64_t cols_pad, void* stream) {
  if (!x || !out || n < 0 || ld < cols_pad || cols_pad < n) return fail(CGP_ERR_ARG, "cgp_cov_matrix_dev: bad arguments");
  if (ld % 2 || ((uintptr_t)out & 15)) return fail(CGP_ERR_ARG, "cgp_cov_matrix_dev: out must be 16-byte aligned with even ld");
  Cov c; int rc = make_cov(dim, hyp, nugget, floor, flags, &c);
  if (rc) return rc;
  const int autocov = xnew == nullptr;
  if (autocov && rows_pad > 65535) {
    // slabs of rows: the builder's diagonal test is slab-relative, so build >65535-row
    // auto-covariances as cross blocks plus a diagonal pass is not needed below 65535 stars
    return fail(CGP_ERR_SIZE, "cgp_cov_matrix_dev: auto-covariance limited to 65535 rows");
  }
  int e = large_cov_build(dim, c, autocov, x, n, autocov ? x : xnew, autocov ? n : m, y_err, out, ld, rows_pad, cols_pad,
                          (cudaStream_t)stream);
  return e ? cuda_fail(e, "cgp_cov_matrix_dev") : 0;
}

int cgp_potrf_dev(double* a, int64_t n_pad, int64_t ld, double* logdet, int* info, void* stream) {
  if (!a || n_pad <= 0 || n_pad % 128 || ld < n_pad || ld % 2) return fail(CGP_ERR_ARG, "cgp_potrf_dev: n_pad must be a positive multiple of 128, ld even");
  int e = large_potrf(a, n_pad, ld, logdet, info, (cudaStream_t)stream);
  return e ? cuda_fail(e, "cgp_potrf_dev") : 0;
}

int cgp_potrs_dev(const double* a, int64_t n_pad, int64_t ld, double* v, double* z_out, int backward, void* stream) {
  if (!a || !v || n_pad <= 0 || n_pad % 128) return fail(CGP_ERR_ARG, "cgp_potrs_dev: bad arguments");
  int e = large_potrs(a, n_pad, ld, v, z_out, backward, (cudaStream_t)stream);
  return e ? cuda_fail(e, "cgp_potrs_dev") : 0;
}

int cgp_large_solve_dev(const double* a, int64_t n, int64_t n_pad, int64_t ld,
                        const double* y, const double* y0, double* alpha, double* quad, void* stream) {
  if (!a || !y || !alpha || n <= 0 || n_pad < n || n_pad % 128) return fail(CGP_ERR_ARG, "cgp_large_solve_dev: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  int e = large_residual(y, y0, n, n_pad, alpha, st);
  if (!e) e = large_potrs(a, n_pad, ld, alpha, nullptr, 0, st);
  if (!e && quad) e = large_dot_sq(alpha, n_pad, quad, st);
  if (!e) {
    // backward half only (forward already applied): reuse potrs with a zero-length forward by
    // running the backward sweep directly
    e = large_potrs_backward(a, n_pad, ld, alpha, st);
  }
  return e ? cuda_fail(e, "cgp_large_solve_dev") : 0;
}

int cgp_trsm_rows_dev(const double* a, int64_t n_pad, int64_t ld, double* v, int64_t ldv, int64_t rows, void* stream) {
  if (!a || !v || rows <= 0 || rows % 128 || n_pad % 128 || ldv < n_pad) return fail(CGP_ERR_ARG, "cgp_trsm_rows_dev: bad arguments");
  int e = large_trsm_rows(a, n_pad, ld, v, ldv, rows, (cudaStream_t)stream);
  return e ? cuda_fail(e, "cgp_trsm_rows_dev") : 0;
}

int cgp_spline_mean_dev(const double* t, const double* c, int n_knots, const double* x, int64_t n_pts,
                        const int64_t* off, int64_t n_obj, const double* diff, double* out, void* stream) {
  if (n_pts < 0 || (n_pts && (!t || !c || !x || !out))) return fail(CGP_ERR_ARG, "cgp_spline_mean_dev: NULL argument");
  if (n_knots < 8) return fail(CGP_ERR_ARG, "cgp_spline_mean_dev: a cubic spline has at least 8 knots, got %d", n_knots);
  if (diff && (!off || n_obj <= 0)) return fail(CGP_ERR_ARG, "cgp_spline_mean_dev: diff needs the CSR offsets");
  int e = large_spline_mean(t, c, n_knots, x, n_pts, off, n_obj, diff, out, (cudaStream_t)stream);
  return e ? cuda_fail(e, "cgp_spline_mean_dev") : 0;
}

int cgp_grid_is_uniform(const double* grid_host, int64_t m, const double* hyp) {
  return uniform_grid_ok(grid_host, m, hyp);
}

int cgp_moments_dev(const double* v, int64_t n, double center, double* out2, void* stream) {
  if (n < 0 || (n && !v) || !out2) return fail(CGP_ERR_ARG, "cgp_moments_dev: NULL argument");
  int e = large_moments(v, n, center, out2, (cudaStream_t)stream);
  return e ? cuda_fail(e, "cgp_moments_dev") : 0;
}

int cgp_gemm_nt_dev(const double* a, int64_t lda, const double* b, int64_t ldb, double* c, int64_t ldc,
                    int64_t m, int64_t n, int64_t k, double alpha, double beta, int lower_only, void* stream) {
  if (!a || !b || !c) return fail(CGP_ERR_ARG, "cgp_gemm_nt_dev: NULL argument");
  if (m % 128 || n % 128 || k % 16 || m <= 0 || n <= 0 || k <= 0 || lda % 2 || ldb % 2 || ldc % 2)
    return fail(CGP_ERR_ARG, "cgp_gemm_nt_dev: m, n must be multiples of 128, k of 16, leading dimensions even");
  GemmArgs g; g.a = a; g.b = b; g.c = c; g.lda = lda; g.ldb = ldb; g.ldc = ldc;
  g.m = (int)m; g.n = (int)n; g.k = (int)k; g.alpha = alpha; g.beta = beta; g.lower_only = lower_only;
  int e = launch_gemm_nt(g, (cudaStream_t)stream);
  return e ? cuda_fail(e, "cgp_gemm_nt_dev") : 0;
}

int cgp_large_predict_dev(const double* a, int64_t n, int64_t n_pad, int64_t ld, int dim, const double* x,
                          const double* alpha, const double* hyp, double nugget, unsigned flags,
                          const double* xnew, int64_t m, const double* new_y0, double* mean, double* var,
                          double* vwork, int64_t chunk_rows, void* stream) {
  if (!a || !x || !alpha || !xnew || !mean || m < 0) return fail(CGP_ERR_ARG, "cgp_large_predict_dev: NULL argument");
  if (var && (!vwork || chunk_rows <= 0 || chunk_rows % 128)) return fail(CGP_ERR_ARG, "cgp_large_predict_dev: vwork / chunk_rows (multiple of 128) required for var");
  cudaStream_t st = (cudaStream_t)stream;
  Cov c; int rc = make_cov(dim, hyp, nugget, 0.0, flags, &c);
  if (rc) return rc;
  int e = large_stream_mean(dim, c, x, alpha, n, xnew, new_y0, m, mean, st);
  if (e) return cuda_fail(e, "cgp_large_predict_dev (mean)");
  if (!var) return 0;
  const double amp_star = c.amp_auto + c.nugget2;
  for (int64_t r0 = 0; r0 < m; r0 += chunk_rows) {
    const int64_t rows = m - r0 < chunk_rows ? m - r0 : chunk_rows;
    const int64_t rows_pad = (rows + 127) / 128 * 128;
    e = large_cov_build(dim, c, 0, x, n, xnew + r0 * dim, rows, nullptr, vwork, n_pad, rows_pad, n_pad, st);
    if (!e) e = large_trsm_rows(a, n_pad, ld, vwork, n_pad, rows_pad, st);
    if (!e) e = large_row_var(vwork, n_pad, n_pad, rows, amp_star, var + r0, st);
    if (e) return cuda_fail(e, "cgp_large_predict_dev (var)");
  }
  return 0;
}

int cgp_large_loo_dev(const double* a, int64_t n, int64_t n_pad, int64_t ld, int dim,
                      const double* y, const double* m, const double* y_err,
                      const double* hyp, double nugget, double floor, unsigned flags, int mode,
                      const int* info, double* vwork, int64_t chunk_rows,
                      double* pred, double* pred_var, double* pull, double* resid, void* stream) {
  if (!a || !y || !info || !vwork) return fail(CGP_ERR_ARG, "cgp_large_loo_dev: NULL argument");
  if (n <= 0 || n_pad < n || n_pad % 128 || ld < n_pad || ld % 2)
    return fail(CGP_ERR_ARG, "cgp_large_loo_dev: need 0 < n <= n_pad, n_pad a multiple of 128, ld >= n_pad and even");
  if (chunk_rows <= 0 || chunk_rows % 128) return fail(CGP_ERR_ARG, "cgp_large_loo_dev: chunk_rows must be a positive multiple of 128");
  if (mode != CGP_LOO_PLAIN && mode != CGP_LOO_RECENTER) return fail(CGP_ERR_ARG, "cgp_large_loo_dev: bad mode %d", mode);
  Cov c; int rc = make_cov(dim, hyp, nugget, floor, flags, &c);
  if (rc) return rc;
  keep_pool_memory();
  int e = large_loo(a, n, n_pad, ld, c, y, m, y_err, mode == CGP_LOO_RECENTER, info, vwork, chunk_rows,
                    pred, pred_var, pull, resid, (cudaStream_t)stream);
  return e ? cuda_fail(e, "cgp_large_loo_dev") : 0;
}

}  // extern "C"
