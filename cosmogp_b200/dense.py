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


def loo_chunk_rows(n_pad, chunk_rows=None):
    """Identity rows per pass of the diag(K^-1) solve for objects of at most n_pad (padded) points: chunk_rows rounded
    down to a multiple of 128 (default: all rows while a pass stays under 4 GB, i.e. up to about 23 000 points), at
    most n_pad."""
    if chunk_rows is None:
        chunk_rows = max(128, (4 << 30) // (8 * n_pad))
    return min(n_pad, int(chunk_rows) // 128 * 128 or 128)


class LargeLoo:
    """Closed-form leave-one-out pulls of objects too large for the shared-memory path, one object per launch
    sequence: covariance build -> blocked Cholesky -> cgp_large_loo_dev, written straight into slices of device
    outputs.  The factor buffer and the diag(K^-1) workspace are allocated once, for the largest object (max_n
    points), and reused; nothing here synchronises.  This is the per-object reference of loo_grouped; build_pull
    uses it for a call with exactly one large object, where large_potrf's look-ahead makes it the faster route, and
    loo_grouped for several.
    chunk_rows: identity rows per pass of the diag(K^-1) solve (loo_chunk_rows)."""

    def __init__(self, max_n, dim, flags=0, chunk_rows=None):
        self.dev = _dev()
        self.dim, self.flags = int(dim), int(flags)
        n_pad = pad128(max_n)
        self.chunk = loo_chunk_rows(n_pad, chunk_rows)
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


def _rows(hyp, nugget, k, dim):
    """The (k, n_hyp) hyperparameter rows and k nugget rows of a grouped call, C-contiguous host arrays: hyp (n_hyp,)
    shared or one row per object; nugget scalar or one per object."""
    nh = 2 if dim == 1 else 4
    rows = np.ascontiguousarray(np.broadcast_to(np.asarray(hyp, dtype=np.float64).reshape(-1, nh), (k, nh)))
    nug_rows = np.ascontiguousarray(np.broadcast_to(np.asarray(nugget, dtype=np.float64).reshape(-1), (k,)))
    return rows, nug_rows


def capped_ws_doubles(need, cap_bytes):
    """Workspace (doubles) of a grouped call whose objects need `need` doubles each: their needs summed up to cap_bytes,
    at least the largest need (objects beyond the cap run in further waves)."""
    need = np.asarray(need, dtype=np.int64).reshape(-1)
    return max(min(int(need.sum()), cap_bytes // 8), int(need.max()) if len(need) else 2)


def _request(off, objects, grid, goff, hyp, nugget, dim):
    """The objects of a grouped call: (off as int64, their ids (objects, default all), their hyperparameter and nugget
    rows (_rows), their grid sizes)."""
    off = np.asarray(off, dtype=np.int64)
    ids = np.arange(len(off) - 1, dtype=np.int64) if objects is None else np.asarray(objects, dtype=np.int64)
    k = len(ids)
    rows, nug_rows = _rows(hyp, nugget, k, dim)
    m = np.diff(np.asarray(goff, dtype=np.int64))[ids] if goff is not None else np.full(k, len(grid), dtype=np.int64)
    return off, ids, rows, nug_rows, m


def _upload(dev, sel, off, grid, goff, *points):
    """The objects `sel` on the device, and only those: each per-point array of `points` (x first; None stays None)
    gathered into one CSR, and the shared grid or their grids gathered into one CSR.  Returns (point CSR, grid CSR or
    None for a shared grid, grid size for a shared grid or 0, device grid, device point arrays); placeholders keep
    empty arrays non-NULL."""
    def up(a):
        return _t(a.reshape(-1) if a.size else np.zeros(2), dev)
    csr = [None if a is None else _gather(np.asarray(a, dtype=np.float64), off, sel) for a in points]
    if goff is None:
        g, lgoff = np.asarray(grid, dtype=np.float64), None
    else:
        g, lgoff = _gather(np.asarray(grid, dtype=np.float64), np.asarray(goff, dtype=np.int64), sel)
    return csr[0][1], lgoff, len(g) if lgoff is None else 0, up(g), [None if c is None else up(c[0]) for c in csr]


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
    off, ids, rows, nug_rows, m = _request(off, objects, grid, goff, hyp, nugget, dim)
    k = len(ids)
    if not k:
        return [], np.zeros(0, dtype=np.int32)
    loff, lgoff, m_shared, gd, (xd, yd) = _upload(dev, ids, off, grid, goff, x, y_err)
    coff = np.zeros(k + 1, dtype=np.int64)
    np.cumsum(m * m, out=coff[1:])
    if work_doubles is None:
        work_doubles = int(cov_ws_doubles(np.diff(loff), m).sum())
    work = torch.empty(max(int(work_doubles), 2), dtype=torch.float64, device=dev)
    out = torch.empty(max(int(coff[-1]), 1), dtype=torch.float64, device=dev)
    info = torch.zeros(k, dtype=torch.int32, device=dev)
    _lib.check(L.cgp_large_covariance_dev(k, _lib.hptr(loff), dim, _p(xd), _p(yd), _lib.hptr(rows), _lib.hptr(nug_rows),
                                          0.0, 0.0, int(flags), _p(gd), _lib.hptr(lgoff), m_shared, None, k, _p(out),
                                          _lib.hptr(coff), _p(info), _p(work), int(work_doubles), _stream(dev)),
               "cgp_large_covariance_dev")
    host = out.cpu().numpy()
    mats = [host[coff[j]:coff[j + 1]].reshape(int(m[j]), int(m[j])) for j in range(k)]
    return mats, info.cpu().numpy()


def pred_ws_doubles(n, rows):
    """Device workspace (doubles) of objects of n points in predictions, `rows` grid rows per variance pass (0: means
    only), elementwise (cgp_large_pred_ws_doubles): n_pad^2 + 3 n_pad + rows_pad n_pad."""
    n_pad = np.maximum((np.asarray(n, dtype=np.int64) + 127) // 128, 1) * 128
    rows_pad = (np.asarray(rows, dtype=np.int64) + 127) // 128 * 128
    return n_pad * n_pad + 3 * n_pad + rows_pad * n_pad


def predictions(x, off, y, y0, y_err, grid, goff, new_y0, hyp, nugget, dim, flags=0, objects=None, want_var=True,
                chunk_rows=None):
    """LargeObject(x_b, y_b, y_err_b, y0_b).factor(hyp, nugget) followed by .predict(grid_b, new_y0_b) for many objects,
    in grouped calls (cgp_large_predict_objhyp_dev), each mean and variance bit for bit that loop's.  x, y, y0, y_err:
    the objects' points, flat with CSR offsets off (y0, y_err may be None).  grid: one shared grid ((M,) or (M, 2), goff
    None) or one grid per object, flat with CSR goff (grid = x, goff = off: the objects' own epochs).  objects: the object
    ids to predict (default all).  new_y0: the mean function on the grids, flat in the output layout (the grids of
    `objects` one after the other), or None.  hyp: (n_hyp,) shared, or one row per object of `objects`; nugget: scalar or
    one per object.  chunk_rows: grid rows per variance pass and object (a multiple of 128; default: a pass of up to 2 GB
    per object, as LargeObject.predict).  The objects go in chunks of <= 256 MB of outputs and <= 2 GB of workspace
    (plan_chunks).  Returns (mean, variance or None, flat in the output layout; CSR of the output rows; info per
    object); an object's rows are NaN where info != 0."""
    dev = _dev()
    L = _lib.lib()
    off, ids, rows, nug_rows, m = _request(off, objects, grid, goff, hyp, nugget, dim)
    k = len(ids)
    n = off[ids + 1] - off[ids]
    moff = np.zeros(k + 1, dtype=np.int64)
    np.cumsum(m, out=moff[1:])
    mean = np.empty(int(moff[-1]))
    var = np.empty(int(moff[-1])) if want_var else None
    info = np.zeros(k, dtype=np.int32)
    if not k:
        return mean, var, moff, info
    if chunk_rows is None:
        chunk_rows = max(128, (2 << 30) // (8 * pad128(int(n.max()))))
    chunk_rows = int(chunk_rows) // 128 * 128 or 128
    ws = pred_ws_doubles(n, np.minimum(m, chunk_rows) if want_var else 0)
    bounds = plan_chunks(m * (16 if want_var else 8), ws * 8)
    work = torch.empty(max(max(int(ws[b0:b1].sum()) for b0, b1 in zip(bounds[:-1], bounds[1:])), 2),
                       dtype=torch.float64, device=dev)
    st = _stream(dev)
    new_y0 = None if new_y0 is None else np.asarray(new_y0, dtype=np.float64).reshape(-1)
    for b0, b1 in zip(bounds[:-1], bounds[1:]):
        # every device array bound to a name until the call has been enqueued
        loff, lgoff, m_shared, gd, (xd, yd, y0d, yed) = _upload(dev, ids[b0:b1], off, grid, goff, x, y, y0, y_err)
        c0, c1 = int(moff[b0]), int(moff[b1])
        lmoff = np.ascontiguousarray(moff[b0:b1 + 1] - c0)
        ny0 = None if new_y0 is None else _t(new_y0[c0:c1], dev)
        md = torch.empty(max(c1 - c0, 1), dtype=torch.float64, device=dev)
        vd = torch.empty(max(c1 - c0, 1), dtype=torch.float64, device=dev) if want_var else None
        infod = torch.zeros(b1 - b0, dtype=torch.int32, device=dev)
        hr, nr = np.ascontiguousarray(rows[b0:b1]), np.ascontiguousarray(nug_rows[b0:b1])
        _lib.check(L.cgp_large_predict_objhyp_dev(
            b1 - b0, _lib.hptr(loff), dim, _p(xd), _p(yd), _p(y0d), _p(yed), _lib.hptr(hr), _lib.hptr(nr), 0.0, 0.0,
            int(flags), _p(gd), _lib.hptr(lgoff), m_shared, _p(ny0), None, b1 - b0,
            _lib.hptr(lmoff), _p(md), _p(vd), _p(infod), chunk_rows, _p(work), int(work.numel()), st),
            "cgp_large_predict_objhyp_dev")
        mean[c0:c1] = md[:c1 - c0].cpu().numpy()
        if want_var:
            var[c0:c1] = vd[:c1 - c0].cpu().numpy()
        info[b0:b1] = infod.cpu().numpy()
    return mean, var, moff, info


LL_WS_BYTES = 2 << 30        # workspace of log_likelihoods (ll_workspace): objects beyond it run in further waves


def ll_ws_doubles(n):
    """Device workspace (doubles) of objects of n points in log_likelihoods, elementwise (cgp_large_ll_ws_doubles):
    n_pad^2 + 2 n_pad + 2 n_pad / 128 with n_pad a multiple of 128 (at least 128)."""
    n_pad = np.maximum((np.asarray(n, dtype=np.int64) + 127) // 128, 1) * 128
    return n_pad * n_pad + 2 * n_pad + 2 * (n_pad // 128)


def ll_workspace(n, device):
    """The device workspace of log_likelihoods for objects of n points: capped_ws_doubles of their needs with cap
    LL_WS_BYTES.  Allocate it once and pass it to every evaluation."""
    return torch.empty(capped_ws_doubles(ll_ws_doubles(n), LL_WS_BYTES), dtype=torch.float64, device=device)


def log_likelihoods_dev(batch, ids, hyp, nugget, ll, info, work, floor=0.0, flags=0):
    """Enqueue log_likelihoods' grouped call (cgp_large_ll_rows_dev) for the objects `ids` (k > 0) of a DeviceBatch:
    ll (k float64) and info (k int32), device tensors, receive the results.  hyp, nugget as in log_likelihoods; work: a
    device workspace from ll_workspace or larger.  Does not synchronise."""
    k = len(ids)
    rows, nug_rows = _rows(hyp, nugget, k, batch.dim)
    order = np.ascontiguousarray(ids, dtype=np.int32)
    with torch.cuda.device(batch.device):
        _lib.check(_lib.lib().cgp_large_ll_rows_dev(
            batch.n_obj, _lib.hptr(batch.off_host), batch.dim, _p(batch.x), _p(batch.y), _p(batch.y0), _p(batch.y_err),
            _lib.hptr(rows), _lib.hptr(nug_rows), 0.0, float(floor), int(flags), _lib.hptr(order), k, _p(ll), _p(info),
            _p(work), int(work.numel()), batch._stream()), "cgp_large_ll_rows_dev")


def log_likelihoods(batch, objects, hyp, nugget, flags=0, work=None):
    """LargeObject(x_b, y_b, y_err_b, y0_b, flags=flags).factor(hyp, nugget) of the objects `objects` (default all) of
    a DeviceBatch in one grouped call (log_likelihoods_dev), each ll and info bit for bit that loop's, whatever the
    objects around it.  hyp: (n_hyp,) shared, or one row per object of `objects`; nugget: scalar or one per object.
    work: a device workspace from ll_workspace, reused across calls (default: one allocated here).  One native call
    and one synchronisation.  Returns host (ll, info), info the first failing pivot and ll NaN where it is not 0."""
    ids = np.arange(batch.n_obj, dtype=np.int64) if objects is None else np.asarray(objects, dtype=np.int64)
    k = len(ids)
    if not k:
        return np.zeros(0), np.zeros(0, dtype=np.int32)
    if work is None:
        work = ll_workspace(batch.off_host[ids + 1] - batch.off_host[ids], batch.device)
    out = torch.empty(k + (k + 1) // 2, dtype=torch.float64, device=batch.device)   # ll, then info as int32
    log_likelihoods_dev(batch, ids, hyp, nugget, out[:k], out[k:].view(torch.int32), work, flags=flags)
    host = out.cpu().numpy()
    return host[:k].copy(), host[k:].view(np.int32)[:k].copy()


def loo_ws_doubles(n, chunk_rows):
    """Device workspace (doubles) of objects of n points in loo_grouped with chunk_rows identity rows per diag(K^-1)
    pass, elementwise (cgp_large_loo_ws_doubles): n_pad^2 + min(n_pad, chunk_rows) n_pad + 7 n_pad + 2."""
    n_pad = np.maximum((np.asarray(n, dtype=np.int64) + 127) // 128, 1) * 128
    return n_pad * n_pad + np.minimum(n_pad, np.int64(chunk_rows)) * n_pad + 7 * n_pad + 2


def loo_grouped(batch, objects, hyp, nugget, mode, outs, flags=0, chunk_rows=None, work_doubles=None):
    """LargeLoo.run of the objects `objects` of a DeviceBatch (its x, y, y0 as the mean, y_err) in one grouped call
    (cgp_large_loo_objhyp_dev), each output bit for bit LargeLoo's at the same chunk_rows.  hyp: (n_hyp,) shared, or
    one row per object of `objects`; nugget: scalar or one per object.  outs: (pred, pred_var, pull, resid, info)
    device tensors in the batch's layout, as DeviceBatch.loo_dev returns them; the objects' points and their info
    entries are written in place.  chunk_rows: as LargeLoo's for the largest object (loo_chunk_rows).  work_doubles:
    device workspace (default: capped_ws_doubles of the objects' needs with a cap of 2 GB).  Does not synchronise."""
    L = _lib.lib()
    ids = np.asarray(objects, dtype=np.int64)
    k = len(ids)
    if not k:
        return
    rows, nug_rows = _rows(hyp, nugget, k, batch.dim)
    n = batch.off_host[ids + 1] - batch.off_host[ids]
    chunk = loo_chunk_rows(pad128(int(n.max())), chunk_rows)
    if work_doubles is None:
        work_doubles = capped_ws_doubles(loo_ws_doubles(n, chunk), 2 << 30)
    work = torch.empty(int(work_doubles), dtype=torch.float64, device=batch.device)
    info = torch.empty(k, dtype=torch.int32, device=batch.device)
    order = np.ascontiguousarray(ids, dtype=np.int32)
    with torch.cuda.device(batch.device):
        _lib.check(L.cgp_large_loo_objhyp_dev(
            batch.n_obj, _lib.hptr(batch.off_host), batch.dim, _p(batch.x), _p(batch.y), _p(batch.y0), _p(batch.y_err),
            _lib.hptr(rows), _lib.hptr(nug_rows), 0.0, 0.0, int(flags), int(mode), _lib.hptr(order), k, _p(info),
            *[_p(o) for o in outs[:4]], chunk, _p(work), int(work_doubles), batch._stream()), "cgp_large_loo_objhyp_dev")
        outs[4][torch.from_numpy(ids).to(batch.device)] = info
