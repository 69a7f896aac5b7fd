"""Large single objects and the per-matrix operator seams, on the device.

`LargeObject` is the N > 224 counterpart of DeviceBatch: the covariance is built in HBM
(never on the host), factorised by the blocked FP64 tensor-core Cholesky and reused for the
likelihood, alpha = K^-1 r, and predictions on arbitrarily long grids (BASELINE configs 3, 4).
`LargeLoo` gives the leave-one-out pulls of such objects for build_pull.
The free functions implement the reference's `kernel(...)` and `chol(matrix)` seams
(cosmogp/Gaussian_process.py:6-9, 136-154) for single matrices of any size.
"""
import math

import numpy as np
import torch

from . import _lib

LOG_2PI = math.log(2.0 * math.pi)


def _dev():
    _lib.require_device()
    return torch.device("cuda", torch.cuda.current_device())


def _stream(dev):
    return torch.cuda.current_stream(dev).cuda_stream


def _t(a, dev):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(dev)


def _p(t):
    return None if t is None else t.data_ptr()


def _hyp(hyp, dim):
    h = np.ascontiguousarray(np.asarray(hyp, dtype=np.float64).ravel())
    assert len(h) == (2 if dim == 1 else 4), "wrong number of hyperparameters for dim=%d" % dim
    return h


def pad128(n):
    return int(_lib.lib().cgp_pad128(int(n)))


def covariance(x, hyperparameter, dim, new_x=None, nugget=0., floor=0., y_err=None, flags=0):
    """K(x,x)+noise (N,N) or K(new_x,x) (M,N) as a host array, built by the streaming kernel."""
    dev = _dev()
    x = np.asarray(x, dtype=np.float64)
    n = len(x)
    h = _hyp(hyperparameter, dim)
    xd = _t(x, dev)
    if new_x is None:
        rows, gd = n, None
    else:
        g = np.asarray(new_x, dtype=np.float64)
        rows, gd = len(g), _t(g, dev)
    ld = n + (n & 1)
    out = torch.empty((max(rows, 1), max(ld, 2)), dtype=torch.float64, device=dev)
    if rows and n:
        rc = _lib.lib().cgp_cov_matrix_dev(dim, _p(xd), n, _p(gd), rows, _p(_t(y_err, dev)), _lib.hptr(h),
                                           float(nugget), float(floor), int(flags), _p(out), ld, rows, n, _stream(dev))
        _lib.check(rc, "cgp_cov_matrix_dev")
    return out[:rows, :n].cpu().numpy()


class LargeObject:
    """One object with its covariance resident in HBM.  x: (N,) or (N,2); y, y0, y_err: (N,)."""

    def __init__(self, x, y, y_err=None, y0=None, dim=1, flags=0):
        self.dev = _dev()
        self.dim, self.flags = int(dim), int(flags)
        self.n = int(len(y))
        self.n_pad = pad128(self.n)
        self.x, self.y = _t(x, self.dev), _t(y, self.dev)
        self.y_err, self.y0 = _t(y_err, self.dev), _t(y0, self.dev)
        self.a = None
        self.alpha = None

    def factor(self, hyp, nugget=0.0, floor=0.0):
        """Build K in HBM and factorise it.  Raises LinAlgError when K is not positive definite."""
        L = _lib.lib()
        h = _hyp(hyp, self.dim)
        self.hyp, self.nugget = h, float(nugget)
        if self.a is None:
            self.a = torch.empty((self.n_pad, self.n_pad), dtype=torch.float64, device=self.dev)
        st = _stream(self.dev)
        scal = torch.zeros(2, dtype=torch.float64, device=self.dev)
        info = torch.zeros(1, dtype=torch.int32, device=self.dev)
        _lib.check(L.cgp_cov_matrix_dev(self.dim, _p(self.x), self.n, None, 0, _p(self.y_err), _lib.hptr(h), float(nugget),
                                        float(floor), self.flags, _p(self.a), self.n_pad, self.n_pad, self.n_pad, st),
                   "cgp_cov_matrix_dev")
        _lib.check(L.cgp_potrf_dev(_p(self.a), self.n_pad, self.n_pad, _p(scal), _p(info), st), "cgp_potrf_dev")
        self.alpha = torch.empty(self.n_pad, dtype=torch.float64, device=self.dev)
        _lib.check(L.cgp_large_solve_dev(_p(self.a), self.n, self.n_pad, self.n_pad, _p(self.y), _p(self.y0),
                                         _p(self.alpha), scal[1:].data_ptr(), st), "cgp_large_solve_dev")
        bad = int(info.item())
        if bad:
            raise np.linalg.LinAlgError("%d-th leading minor of the covariance is not positive definite" % bad)
        logdet, quad = (float(v) for v in scal.cpu().numpy())
        self.logdet, self.quad = logdet, quad
        self.log_likelihood = -0.5 * (quad + logdet + self.n * LOG_2PI)      # Gaussian_process.py:68-73
        return self.log_likelihood

    def predict(self, grid, new_y0=None, want_var=True, chunk_rows=None):
        """mean (and variance diagonal) on a grid of any length; needs factor() first.
        chunk_rows: grid points per triangular-solve pass (default: as many as fit in ~2 GB of
        workspace, so that each 128-column GEMM of the solve has hundreds of row tiles)."""
        assert self.alpha is not None, "call factor() first"
        L = _lib.lib()
        g = _t(grid, self.dev)
        m = int(g.shape[0])
        mean = torch.empty(max(m, 1), dtype=torch.float64, device=self.dev)
        var = torch.empty(max(m, 1), dtype=torch.float64, device=self.dev) if want_var else None
        if chunk_rows is None:
            chunk_rows = max(128, (2 << 30) // (8 * self.n_pad))
        chunk = min(pad128(m), int(chunk_rows) // 128 * 128 or 128)
        vwork = torch.empty((chunk, self.n_pad), dtype=torch.float64, device=self.dev) if want_var else None
        _lib.check(L.cgp_large_predict_dev(_p(self.a), self.n, self.n_pad, self.n_pad, self.dim, _p(self.x), _p(self.alpha),
                                           _lib.hptr(self.hyp), self.nugget, self.flags, _p(g), m, _p(_t(new_y0, self.dev)),
                                           _p(mean), _p(var), _p(vwork), chunk, _stream(self.dev)), "cgp_large_predict_dev")
        return mean[:m].cpu().numpy(), (var[:m].cpu().numpy() if want_var else None)

    def inverse(self):
        """K^-1 (N,N) on the host from the factor: U = L^-T by the blocked solve on the identity,
        K^-1 = U U^T by the tensor-core GEMM."""
        assert self.a is not None
        L = _lib.lib()
        st = _stream(self.dev)
        u = torch.eye(self.n_pad, dtype=torch.float64, device=self.dev)
        _lib.check(L.cgp_trsm_rows_dev(_p(self.a), self.n_pad, self.n_pad, _p(u), self.n_pad, self.n_pad, st), "cgp_trsm_rows_dev")
        kinv = torch.empty((self.n_pad, self.n_pad), dtype=torch.float64, device=self.dev)
        _lib.check(L.cgp_gemm_nt_dev(_p(u), self.n_pad, _p(u), self.n_pad, _p(kinv), self.n_pad, self.n_pad, self.n_pad,
                                     self.n_pad, 1.0, 0.0, 0, st), "cgp_gemm_nt_dev")
        return kinv[:self.n, :self.n].cpu().numpy()


class LargeLoo:
    """Closed-form leave-one-out pulls of objects too large for the shared-memory path, one object per launch
    sequence: covariance build -> blocked Cholesky -> cgp_large_loo_dev, written straight into slices of device
    outputs.  The factor buffer and the diag(K^-1) workspace are allocated once, for the largest object (max_n
    points), and reused; nothing here synchronises.
    chunk_rows: identity rows per pass of the diag(K^-1) solve (default: all rows while the workspace stays under
    4 GB, i.e. up to about 23 000 points)."""

    def __init__(self, max_n, dim, flags=0, chunk_rows=None):
        self.dev = _dev()
        self.dim, self.flags = int(dim), int(flags)
        n_pad = pad128(max_n)
        if chunk_rows is None:
            chunk_rows = max(128, (4 << 30) // (8 * n_pad))
        self.chunk = min(n_pad, int(chunk_rows) // 128 * 128 or 128)
        self.a = torch.empty(n_pad * n_pad, dtype=torch.float64, device=self.dev)
        self.vwork = torch.empty(self.chunk * n_pad, dtype=torch.float64, device=self.dev)

    def run(self, x, y, m, y_err, hyp, nugget, mode, info, outs):
        """x, y (and m, y_err, either may be None): device tensors of one object; info: one-element int32 device
        tensor, receives the factorisation's status; outs: device tensors (pred, pred_var, pull, resid) of N doubles."""
        L = _lib.lib()
        n = int(y.numel())
        n_pad = pad128(n)
        h = _hyp(hyp, self.dim)
        st = _stream(self.dev)
        _lib.check(L.cgp_cov_matrix_dev(self.dim, _p(x), n, None, 0, _p(y_err), _lib.hptr(h), float(nugget), 0.0,
                                        self.flags, _p(self.a), n_pad, n_pad, n_pad, st), "cgp_cov_matrix_dev")
        _lib.check(L.cgp_potrf_dev(_p(self.a), n_pad, n_pad, None, _p(info), st), "cgp_potrf_dev")
        _lib.check(L.cgp_large_loo_dev(_p(self.a), n, n_pad, n_pad, self.dim, _p(y), _p(m), _p(y_err), _lib.hptr(h),
                                       float(nugget), 0.0, self.flags, int(mode), _p(info), _p(self.vwork), self.chunk,
                                       *[_p(o) for o in outs], st), "cgp_large_loo_dev")


def cholesky_inverse(matrix, return_logdet=False):
    """The `chol` seam (cosmogp/inv_matrix.py:21-31) for an arbitrary SPD matrix, on the device."""
    dev = _dev()
    L = _lib.lib()
    m = np.asarray(matrix, dtype=np.float64)
    n = m.shape[0]
    assert m.ndim == 2 and m.shape[1] == n, "expected a square matrix"
    n_pad = pad128(n)
    a = torch.eye(n_pad, dtype=torch.float64, device=dev)
    a[:n, :n] = torch.from_numpy(np.ascontiguousarray(m)).to(dev)
    st = _stream(dev)
    scal = torch.zeros(1, dtype=torch.float64, device=dev)
    info = torch.zeros(1, dtype=torch.int32, device=dev)
    _lib.check(L.cgp_potrf_dev(_p(a), n_pad, n_pad, _p(scal), _p(info), st), "cgp_potrf_dev")
    bad = int(info.item())
    if bad:
        raise np.linalg.LinAlgError("%d-th leading minor of the array is not positive definite" % bad)
    u = torch.eye(n_pad, dtype=torch.float64, device=dev)
    _lib.check(L.cgp_trsm_rows_dev(_p(a), n_pad, n_pad, _p(u), n_pad, n_pad, st), "cgp_trsm_rows_dev")
    kinv = torch.empty((n_pad, n_pad), dtype=torch.float64, device=dev)
    _lib.check(L.cgp_gemm_nt_dev(_p(u), n_pad, _p(u), n_pad, _p(kinv), n_pad, n_pad, n_pad, n_pad, 1.0, 0.0, 0, st),
               "cgp_gemm_nt_dev")
    inv = kinv[:n, :n].cpu().numpy()
    if return_logdet:
        return inv, float(scal.item())
    return inv


def object_matrices(x, y_err, hyp, nugget, dim, flags=0):
    """kernel_matrix / inv_kernel_matrix of one object too large for the shared-memory path (host arrays in and out)."""
    obj = LargeObject(x, np.zeros(len(x)), y_err, dim=dim, flags=flags)
    k = covariance(x, hyp, dim, nugget=nugget, y_err=y_err, flags=flags)
    obj.factor(hyp, nugget)
    return k, obj.inverse()


def predictive_covariance(x, y_err, grid, hyp, nugget, dim, flags=0):
    """Full covariance_matrix of one object (cosmogp/Gaussian_process.py:356-361):
    K(grid,grid) + nugget^2 I - V V^T with V = rows L^-1 h_m, all on the device."""
    dev = _dev()
    L = _lib.lib()
    obj = LargeObject(x, np.zeros(len(x)), y_err, dim=dim, flags=flags)
    obj.factor(hyp, nugget)
    h = _hyp(hyp, dim)
    st = _stream(dev)
    g = _t(grid, dev)
    m = int(g.shape[0])
    m_pad = pad128(m)
    v = torch.empty((m_pad, obj.n_pad), dtype=torch.float64, device=dev)
    _lib.check(L.cgp_cov_matrix_dev(dim, _p(obj.x), obj.n, _p(g), m, None, _lib.hptr(h), float(nugget), 0.0, int(flags),
                                    _p(v), obj.n_pad, m_pad, obj.n_pad, st), "cgp_cov_matrix_dev (H)")
    _lib.check(L.cgp_trsm_rows_dev(_p(obj.a), obj.n_pad, obj.n_pad, _p(v), obj.n_pad, m_pad, st), "cgp_trsm_rows_dev")
    c = torch.empty((m_pad, m_pad), dtype=torch.float64, device=dev)
    _lib.check(L.cgp_cov_matrix_dev(dim, _p(g), m, None, 0, None, _lib.hptr(h), float(nugget), 0.0, int(flags),
                                    _p(c), m_pad, m_pad, m_pad, st), "cgp_cov_matrix_dev (K**)")
    _lib.check(L.cgp_gemm_nt_dev(_p(v), obj.n_pad, _p(v), obj.n_pad, _p(c), m_pad, m_pad, m_pad, obj.n_pad,
                                 -1.0, 1.0, 0, st), "cgp_gemm_nt_dev")
    return c[:m, :m].cpu().numpy()


def cov_ws_doubles(n, m):
    """Device workspace (doubles) of objects of n points on grids of m in predictive_covariances, elementwise
    (cgp_large_cov_ws_doubles): n_pad^2 + m_pad n_pad + m_pad^2 with both padded to a multiple of 128 (at least 128)."""
    n_pad, m_pad = (np.maximum((np.asarray(v, dtype=np.int64) + 127) // 128, 1) * 128 for v in (n, m))
    return n_pad * n_pad + m_pad * n_pad + m_pad * m_pad


def plan_chunks(out_bytes, ws_bytes=None, out_budget=256 << 20, ws_budget=2 << 30):
    """Bounds [0, .., K] of consecutive chunks of K items: a chunk closes before the item that would take its output
    above out_budget or its workspace above ws_budget (a single item larger than either is a chunk of its own)."""
    bounds, acc_o, acc_w = [0], 0, 0
    ws = np.zeros(len(out_bytes), dtype=np.int64) if ws_bytes is None else ws_bytes
    for j in range(len(out_bytes)):
        if (acc_o or acc_w) and (acc_o + out_bytes[j] > out_budget or acc_w + ws[j] > ws_budget):
            bounds.append(j)
            acc_o = acc_w = 0
        acc_o += int(out_bytes[j])
        acc_w += int(ws[j])
    bounds.append(len(out_bytes))
    return bounds


def _gather(flat, off, ids):
    """The CSR segments `ids` of (flat, off) as a new CSR (flat rows, offsets)."""
    lens = off[ids + 1] - off[ids]
    new_off = np.zeros(len(ids) + 1, dtype=np.int64)
    np.cumsum(lens, out=new_off[1:])
    idx = np.repeat(off[ids] - new_off[:-1], lens) + np.arange(new_off[-1], dtype=np.int64)
    return flat[idx], new_off


def predictive_covariances(x, off, y_err, grid, goff, hyp, nugget, dim, flags=0, objects=None, work_doubles=None):
    """predictive_covariance of many objects in one grouped call (cgp_large_covariance_dev), each matrix bit for bit
    what predictive_covariance gives for that object alone.  x: the objects' points, flat ((P,) or (P, 2)) with CSR
    offsets off; y_err: flat (P,) or None.  grid: one shared grid ((M,) or (M, 2), goff None) or one grid per object,
    flat with CSR goff (grid = x, goff = off: the objects' own epochs).  objects: the object ids to compute (default
    all).  hyp: (n_hyp,) shared, or one row per object of `objects`; nugget: scalar or one per object.  work_doubles:
    device workspace (default: every object in one wave).  Returns (list of (m_b, m_b) host arrays, info per object);
    a matrix is NaN where info != 0."""
    dev = _dev()
    L = _lib.lib()
    off = np.asarray(off, dtype=np.int64)
    ids = np.arange(len(off) - 1, dtype=np.int64) if objects is None else np.asarray(objects, dtype=np.int64)
    k = len(ids)
    nh = 2 if dim == 1 else 4
    hyp = np.asarray(hyp, dtype=np.float64)
    rows = np.ascontiguousarray(np.broadcast_to(hyp.reshape(-1, nh), (k, nh)) if hyp.ndim == 1 else hyp.reshape(k, nh))
    nug_rows = None if np.ndim(nugget) == 0 else np.ascontiguousarray(nugget, dtype=np.float64).reshape(k)
    if not k:
        return [], np.zeros(0, dtype=np.int32)
    xs, loff = _gather(np.asarray(x, dtype=np.float64), off, ids)        # only the requested objects go to the device
    ye = None if y_err is None else _gather(np.asarray(y_err, dtype=np.float64), off, ids)[0]
    if goff is None:
        g, lgoff = np.asarray(grid, dtype=np.float64), None
        m = np.full(k, len(g), dtype=np.int64)
    else:
        g, lgoff = _gather(np.asarray(grid, dtype=np.float64), np.asarray(goff, dtype=np.int64), ids)
        m = np.diff(lgoff)
    coff = np.zeros(k + 1, dtype=np.int64)
    np.cumsum(m * m, out=coff[1:])
    if work_doubles is None:
        work_doubles = int(cov_ws_doubles(np.diff(loff), m).sum())
    xd, yd = _t(xs if xs.size else np.zeros(2), dev), _t(ye, dev)      # placeholders keep empty inputs non-NULL
    gd = _t(g.reshape(-1) if g.size else np.zeros(2), dev)
    work = torch.empty(max(int(work_doubles), 2), dtype=torch.float64, device=dev)
    out = torch.empty(max(int(coff[-1]), 1), dtype=torch.float64, device=dev)
    info = torch.zeros(k, dtype=torch.int32, device=dev)
    _lib.check(L.cgp_large_covariance_dev(k, _lib.hptr(loff), dim, _p(xd), _p(yd), _lib.hptr(rows), _lib.hptr(nug_rows),
                                          float(0.0 if nug_rows is not None else nugget), 0.0, int(flags), _p(gd),
                                          _lib.hptr(lgoff), int(m[0]) if lgoff is None else 0, None, k, _p(out),
                                          _lib.hptr(coff), _p(info), _p(work), int(work_doubles), _stream(dev)),
               "cgp_large_covariance_dev")
    host = out.cpu().numpy()
    mats = [host[coff[j]:coff[j + 1]].reshape(int(m[j]), int(m[j])) for j in range(k)]
    return mats, info.cpu().numpy()
