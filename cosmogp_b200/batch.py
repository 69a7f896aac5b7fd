"""Device-resident batch of GP objects: the numpy-in / numpy-out layer over the C ABI.

One `DeviceBatch` = the data a reference `Gaussian_process` holds (y, Time, y_err, y0:
cosmogp/Gaussian_process.py:156-186) packed as CSR arrays and uploaded ONCE to HBM;
every likelihood evaluation of the optimiser, the prediction and the pulls are then
single batched launches on it.  PyTorch only owns the buffers (pinned staging + device
tensors) and the stream; all arithmetic is in libcosmogp_b200.so.
"""
import functools

import numpy as np
import torch

from . import _lib, dense


def _as_list_of_arrays(seq, dim):
    out = []
    for a in seq:
        a = np.asarray(a, dtype=np.float64)
        out.append(a.reshape(-1, dim) if dim == 2 else a.reshape(-1))
    return out


def pack_csr(seq, dim=1):
    """list of per-object arrays (or a 2-D/3-D ndarray of equal-length objects) ->
    (flat C-contiguous float64 array, offsets int64[B+1])."""
    if isinstance(seq, np.ndarray) and seq.dtype != object and seq.ndim == (2 if dim == 1 else 3):
        b, n = seq.shape[0], seq.shape[1]
        flat = np.ascontiguousarray(seq, dtype=np.float64).reshape(b * n, *([2] if dim == 2 else []))
        return flat, np.arange(b + 1, dtype=np.int64) * n
    if not hasattr(seq, '__len__'):
        seq = list(seq)                                  # an iterator of per-object arrays
    want = 2 if dim == 2 else 1
    if all(type(a) is np.ndarray and a.ndim == want and (dim == 1 or a.shape[1] == 2) for a in seq):
        arrs = seq          # already per-object arrays of the right shape: no per-object conversion (0.6 s at 10^5 objects)
    else:
        arrs = _as_list_of_arrays(seq, dim)
    off = np.zeros(len(arrs) + 1, dtype=np.int64)
    if arrs:
        off[1:] = np.cumsum(np.fromiter(map(len, arrs), dtype=np.int64, count=len(arrs)))
        flat = np.ascontiguousarray(np.concatenate(arrs), dtype=np.float64)
    else:
        flat = np.zeros((0, 2) if dim == 2 else (0,), dtype=np.float64)
    return flat, off


class SizeSplit:
    """Which objects of a CSR batch (offsets `off`) the shared-memory kernels take: the "small" ones, of at most
    CGP_SMALL_MAX_N points.  The others ("large") go through the blocked HBM factorisation.  Small objects run with the
    largest small size as max_n, so that in a batch with large objects they get exactly the results of a batch without
    them.  Host only: this is the one place that rule is written down.

      sizes        points per object
      small        bool mask over the objects
      large        ids of the large objects, ascending
      small_max_n  max_n of the small objects (0 when there are none)
      runs         [(first, end)) ranges of consecutive small objects, maximal
      points       bool mask over the points: those of small objects
      small_off    CSR offsets of the small objects alone
      small_csr()  the same two for another CSR over the objects, e.g. one prediction grid per object"""

    def __init__(self, off):
        self.sizes = np.diff(np.asarray(off, dtype=np.int64))
        self.small = self.sizes <= _lib.CGP_SMALL_MAX_N
        self.large = np.nonzero(~self.small)[0]
        self.small_max_n = int(self.sizes[self.small].max(initial=0))
        edges = np.concatenate([[-1], self.large, [len(self.sizes)]])
        self.runs = [(int(a + 1), int(b)) for a, b in zip(edges[:-1], edges[1:]) if b > a + 1]

    # per point: only built when a batch of the small objects alone is needed
    @functools.cached_property
    def points(self):
        return np.repeat(self.small, self.sizes)

    @functools.cached_property
    def small_off(self):
        return self.small_csr(sizes=self.sizes)[1]

    def small_csr(self, off=None, sizes=None):
        """(bool mask over the entries of the small objects, offsets of the small objects alone) of a CSR over the
        objects, given by its offsets or its sizes"""
        sizes = np.diff(np.asarray(off, dtype=np.int64)) if sizes is None else sizes
        sub = np.zeros(int(self.small.sum()) + 1, dtype=np.int64)
        sub[1:] = np.cumsum(sizes[self.small])
        return np.repeat(self.small, sizes), sub


class RaggedView(object):
    """list-like view of per-object slices of a flat array (what the reference keeps as a Python
    list of arrays), built in O(1): at 10^6 objects a real list of slices costs seconds."""

    def __init__(self, flat, off):
        self.flat, self.off = flat, np.asarray(off, dtype=np.int64)

    def __len__(self):
        return len(self.off) - 1

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self[j] for j in range(*i.indices(len(self)))]
        if i < 0:
            i += len(self)
        if not 0 <= i < len(self):
            raise IndexError(i)
        return self.flat[self.off[i]:self.off[i + 1]]

    def __iter__(self):
        return (self[i] for i in range(len(self)))

    def __array__(self, dtype=None, copy=None):
        """equal-length objects -> the (B, n) array (a view of the flat data); ragged -> an object array of views"""
        sizes = np.diff(self.off)
        if len(sizes) and np.all(sizes == sizes[0]) and self.off[0] == 0:
            out = self.flat[:self.off[-1]].reshape(len(sizes), int(sizes[0]), *self.flat.shape[1:])
            return out if dtype is None else out.astype(dtype)
        out = np.empty(len(self), dtype=object)
        for i in range(len(self)):
            out[i] = self[i]
        return out

    def extended(self, flat, off):
        """view over this view's data followed by another batch (compute_pull appends across calls)."""
        off = np.asarray(off, dtype=np.int64)
        if len(self) == 0:
            return RaggedView(flat, off)
        return RaggedView(np.concatenate([self.flat, flat]), np.concatenate([self.off, off[1:] + self.off[-1]]))


def pinned_like(a):
    """Copy a numpy array into pinned host memory (returns the numpy view and its owner)."""
    t = torch.empty(a.shape, dtype=torch.float64 if a.dtype == np.float64 else torch.int64, pin_memory=True)
    v = t.numpy()
    v[...] = a
    return v, t


class DeviceBatch:
    """x: flat (sumN,) or (sumN,2); y, y0, y_err: flat (sumN,) (y0 / y_err may be None);
    off: int64 (B+1,).  Host arrays may live in pinned memory (fast path) or not."""

    def __init__(self, x, y, off, y0=None, y_err=None, dim=1, device=None, max_n=None):
        _lib.require_device()
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.dim = int(dim)
        self.n_obj = int(len(off) - 1)
        self.n_pts = int(off[-1]) if len(off) else 0
        self.off_host = np.ascontiguousarray(off, dtype=np.int64)
        sizes = np.diff(self.off_host)
        self.max_n = int(sizes.max()) if max_n is None and self.n_obj else int(max_n or 0)
        self.h2d_bytes = 0
        self.off = self._up(self.off_host)
        self.x = self._up(x)
        self.y = self._up(y)
        self.y0 = self._up(y0)
        self.y_err = self._up(y_err)
        self._info = torch.empty(max(self.n_obj, 1), dtype=torch.int32, device=self.device)
        self.d2h_bytes = 0

    # ---- plumbing
    def _up(self, a):
        if a is None:
            return None
        t = torch.from_numpy(np.ascontiguousarray(a))
        self.h2d_bytes += t.numel() * t.element_size()
        return t.to(self.device, non_blocking=True)

    def _up_grid(self, grid):
        """a flat per-object grid; when every grid is empty one unread point stands in, since the entries take no NULL grid"""
        g = np.asarray(grid, dtype=np.float64)
        return self._up(g if len(g) else np.zeros((1,) + g.shape[1:]))

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    @staticmethod
    def _p(t):
        return None if t is None else t.data_ptr()

    def _hyp(self, hyp):
        h = np.ascontiguousarray(np.asarray(hyp, dtype=np.float64).ravel())
        need = 2 if self.dim == 1 else 4
        assert len(h) == need, "expected %d hyperparameters, got %d" % (need, len(h))
        return h

    def _down(self, t, sync=True):
        """Device -> pinned host (torch's caching host allocator recycles the blocks).  sync=False only enqueues the
        copy: the caller batches several downloads and calls _sync() once before touching the arrays."""
        self.d2h_bytes += t.numel() * t.element_size()
        out = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
        out.copy_(t, non_blocking=True)
        if sync:
            torch.cuda.current_stream(self.device).synchronize()
        return out.numpy()

    def _sync(self):
        torch.cuda.current_stream(self.device).synchronize()

    # ---- the hot path
    def ll_dev(self, hyp, nugget=0.0, floor=0.0, flags=0):
        """Enqueue one batched log-likelihood evaluation; returns (ll_obj, info) device tensors."""
        h = self._hyp(hyp)
        ll = torch.empty(max(self.n_obj, 1), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            rc = _lib.lib().cgp_ll_batched_dev(self.n_obj, self._p(self.off), self.max_n, self.dim, self._p(self.x),
                                               self._p(self.y), self._p(self.y0), self._p(self.y_err), _lib.hptr(h),
                                               float(nugget), float(floor), int(flags), self._p(ll), self._p(self._info),
                                               self._stream())
        _lib.check(rc, "cgp_ll_batched_dev")
        return ll[:self.n_obj], self._info[:self.n_obj]

    def log_likelihood_total(self, hyp, nugget=0.0, floor=0.0, flags=0):
        """One likelihood evaluation as the optimiser needs it (cgp_ll_total_dev): the per-object values and the
        `info` flags stay on the device (`ll_host()` / `info_host()` fetch them), the sum over objects is reduced there
        in a fixed order and 16 bytes come back.  -> (sum, number of non-positive-definite objects).
        No allocation, one native call and one stream synchronisation per evaluation."""
        c = getattr(self, "_tot", None)
        if c is None:
            ll = torch.empty(max(self.n_obj, 1), dtype=torch.float64, device=self.device)
            tot_d = torch.zeros(2, dtype=torch.float64, device=self.device)
            tot_h = torch.zeros(2, dtype=torch.float64, pin_memory=True)
            nh = 2 if self.dim == 1 else 4
            c = self._tot = {"ll": ll, "tot_d": tot_d, "tot_h": tot_h, "tot_np": tot_h.numpy(), "hyp": np.zeros(nh),
                             "fn": _lib.lib().cgp_ll_total_dev, "dev_index": self.device.index,
                             "args": (self.n_obj, self._p(self.off), self.max_n, self.dim, self._p(self.x), self._p(self.y),
                                      self._p(self.y0), self._p(self.y_err)),
                             "out": (ll.data_ptr(), self._info.data_ptr(), tot_d.data_ptr(), tot_h.data_ptr())}
            c["hyp_ptr"] = c["hyp"].ctypes.data
        h = c["hyp"]
        h[:] = hyp                                           # raises on a wrong number of hyperparameters
        if torch.cuda.current_device() != c["dev_index"]:
            with torch.cuda.device(self.device):
                rc = c["fn"](*c["args"], c["hyp_ptr"], float(nugget), float(floor), int(flags), *c["out"], self._stream())
        else:
            rc = c["fn"](*c["args"], c["hyp_ptr"], float(nugget), float(floor), int(flags), *c["out"], self._stream())
        _lib.check(rc, "cgp_ll_total_dev")
        self.d2h_bytes += 16
        return float(c["tot_np"][0]), int(rc)

    def ll_host(self):
        """per-object log-likelihoods of the latest log_likelihood_total() call, brought to the host"""
        return self._down(self._tot["ll"][:self.n_obj])

    def info_host(self):
        return self._down(self._info[:self.n_obj])

    def log_likelihood(self, hyp, nugget=0.0, floor=0.0, flags=0):
        """-> (sum over objects in index order, per-object LL, info), all host numpy."""
        ll, info = self.ll_dev(hyp, nugget, floor, flags)
        ll_h = self._down(ll)
        info_h = self._down(info)
        total = float(np.add.accumulate(ll_h)[-1]) if self.n_obj else 0.0   # left-to-right, like :205-213
        return total, ll_h, info_h

    def ll_objhyp(self, hyp_rows, idx, nugget_rows=None, nugget=0.0, floor=0.0, flags=0):
        """Log-likelihood of the objects `idx` (int array), object idx[k] using its own
        hyperparameters hyp_rows[k] (and nugget_rows[k]).  -> (ll (k,), info (k,)) host arrays.
        Compact I/O: only the k active rows cross PCIe, through persistent pinned / device buffers.
        Objects of up to 224 points go through the shared-memory kernel (cgp_ll_objhyp_dev, with the largest small
        size as max_n: the kernel a batch of the small objects alone gets), larger ones through the grouped blocked
        factorisation (dense.log_likelihoods_dev, from the host rows: each bit for bit dense.LargeObject.factor) in a
        workspace allocated once per batch.  One synchronisation."""
        k, nh = len(idx), (2 if self.dim == 1 else 4)
        if k == 0:
            return np.zeros(0), np.zeros(0, dtype=np.int32)
        c = getattr(self, "_oh", None)
        if c is None:
            pin = lambda shape, dt: torch.empty(shape, dtype=dt, pin_memory=True)
            dev = lambda shape, dt: torch.empty(shape, dtype=dt, device=self.device)
            b = max(self.n_obj, 1)
            c = self._oh = {"hyp_h": pin((b, nh), torch.float64), "hyp_d": dev((b, nh), torch.float64),
                            "nug_h": pin((b,), torch.float64), "nug_d": dev((b,), torch.float64),
                            "ord_h": pin((b,), torch.int32), "ord_d": dev((b,), torch.int32),
                            "ll_h": pin((b,), torch.float64), "ll_d": dev((b,), torch.float64),
                            "info_h": pin((b,), torch.int32), "info_d": dev((b,), torch.int32)}
            split = SizeSplit(self.off_host)
            c["large"] = ~split.small
            c["small_max_n"] = split.small_max_n if len(split.large) else self.max_n
            if len(split.large):
                need = dense.ll_ws_doubles(split.sizes[split.large])
                c["work"] = torch.empty(dense.capped_ws_doubles(need, 4 << 30), dtype=torch.float64, device=self.device)
        idx = np.asarray(idx, dtype=np.int64)
        big = c["large"][idx]
        perm = np.concatenate([np.nonzero(~big)[0], np.nonzero(big)[0]]) if big.any() else None
        ks = k - int(big.sum())
        rows = np.asarray(hyp_rows, dtype=np.float64).reshape(k, nh)
        hyp_h, ord_h, nug_h = c["hyp_h"].numpy()[:k], c["ord_h"].numpy()[:k], c["nug_h"].numpy()[:k]
        hyp_h[:] = rows if perm is None else rows[perm]
        ord_h[:] = idx if perm is None else idx[perm]
        if nugget_rows is not None:
            nug = np.asarray(nugget_rows, dtype=np.float64)
            nug_h[:] = nug if perm is None else nug[perm]
        with torch.cuda.device(self.device):
            if ks:
                c["hyp_d"][:ks].copy_(c["hyp_h"][:ks], non_blocking=True)
                c["ord_d"][:ks].copy_(c["ord_h"][:ks], non_blocking=True)
                nd = None
                if nugget_rows is not None:
                    c["nug_d"][:ks].copy_(c["nug_h"][:ks], non_blocking=True)
                    nd = c["nug_d"]
                rc = _lib.lib().cgp_ll_objhyp_dev(self.n_obj, self._p(self.off), c["small_max_n"], self.dim, self._p(self.x),
                                                  self._p(self.y), self._p(self.y0), self._p(self.y_err), self._p(c["hyp_d"]),
                                                  self._p(nd), float(nugget), float(floor), int(flags), self._p(c["ord_d"]), ks,
                                                  self._p(c["ll_d"]), self._p(c["info_d"]), self._stream())
                _lib.check(rc, "cgp_ll_objhyp_dev")
            if ks < k:
                dense.log_likelihoods_dev(self, ord_h[ks:], hyp_h[ks:], nugget if nugget_rows is None else nug_h[ks:],
                                          c["ll_d"][ks:k], c["info_d"][ks:k], c["work"], floor, flags)
        c["ll_h"][:k].copy_(c["ll_d"][:k], non_blocking=True)
        c["info_h"][:k].copy_(c["info_d"][:k], non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        ll, info = c["ll_h"].numpy()[:k].copy(), c["info_h"].numpy()[:k].copy()
        if perm is not None:
            ll[perm], info[perm] = ll.copy(), info.copy()
        return ll, info

    def fit_objects(self, start, nugget=0.0, floor=0.0, flags=0, xatol=1e-4, fatol=1e-4, maxiter=None, maxfun=None):
        """One Nelder-Mead fit per object, entirely on the device (cgp_fit_objects_dev).
        start: (n_obj, nh) or (n_obj, nh+1) -- with nh+1 columns the last one is the object's nugget.
        -> (par (n_obj, n_par), nll (n_obj,), iterations, evaluations) host arrays; the decisions are
        scipy.optimize.fmin's, object by object (same results as fit.nelder_mead_lockstep)."""
        start = np.ascontiguousarray(start, dtype=np.float64)
        assert start.ndim == 2 and start.shape[0] == self.n_obj
        n_par = start.shape[1]
        maxiter = n_par * 200 if maxiter is None else int(maxiter)
        maxfun = n_par * 200 if maxfun is None else int(maxfun)
        b = max(self.n_obj, 1)
        x0 = self._up(start)
        par = torch.empty((b, n_par), dtype=torch.float64, device=self.device)
        nll = torch.empty(b, dtype=torch.float64, device=self.device)
        its = torch.empty(b, dtype=torch.int32, device=self.device)
        calls = torch.empty(b, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            rc = _lib.lib().cgp_fit_objects_dev(self.n_obj, self._p(self.off), self.max_n, self.dim, self._p(self.x),
                                                self._p(self.y), self._p(self.y0), self._p(self.y_err), self._p(x0), n_par,
                                                float(nugget), float(floor), int(flags), float(xatol), float(fatol),
                                                maxiter, maxfun, self._p(par), self._p(nll), self._p(its), self._p(calls),
                                                self._stream())
        _lib.check(rc, "cgp_fit_objects_dev")
        k = self.n_obj
        return (par[:k].cpu().numpy(), nll[:k].cpu().numpy(), its[:k].cpu().numpy().astype(np.int64),
                calls[:k].cpu().numpy().astype(np.int64))

    def _objhyp(self, hyp, nugget):
        """(B, nh) hyperparameters (+ optional (B,) nuggets) -> device tensors, or None for shared ones."""
        if np.ndim(hyp) != 2:
            return None
        nh = 2 if self.dim == 1 else 4
        h = np.ascontiguousarray(hyp, dtype=np.float64)
        assert h.shape == (self.n_obj, nh), "per-object hyperparameters must have shape (%d, %d)" % (self.n_obj, nh)
        nd = self._up(np.ascontiguousarray(nugget, dtype=np.float64)) if np.ndim(nugget) == 1 else None
        return self._up(h), nd, (0.0 if nd is not None else float(nugget))

    def predict_dev(self, hyp, nugget, grid, goff=None, new_y0=None, want_var=True, floor=0.0, flags=0):
        oh = self._objhyp(hyp, nugget)
        if oh is not None:
            m = 0 if goff is not None else int(grid.shape[0])
            nout = int(goff[-1].item()) if goff is not None else self.n_obj * m
            mean = torch.empty(max(nout, 1), dtype=torch.float64, device=self.device)
            var = torch.empty(max(nout, 1), dtype=torch.float64, device=self.device) if want_var else None
            with torch.cuda.device(self.device):
                rc = _lib.lib().cgp_predict_objhyp_dev(self.n_obj, self._p(self.off), self.max_n, self.dim,
                                                       self._p(self.x), self._p(self.y), self._p(self.y0), self._p(self.y_err),
                                                       self._p(oh[0]), self._p(oh[1]), oh[2], float(floor), int(flags),
                                                       self._p(grid), self._p(goff), m, self._p(new_y0),
                                                       self._p(mean), self._p(var), self._p(self._info), self._stream())
            _lib.check(rc, "cgp_predict_objhyp_dev")
            return mean[:nout], (var[:nout] if want_var else None), self._info[:self.n_obj]
        h = self._hyp(hyp)
        m = 0 if goff is not None else int(grid.shape[0])
        nout = int(goff[-1].item()) if goff is not None else self.n_obj * m
        mean = torch.empty(max(nout, 1), dtype=torch.float64, device=self.device)
        var = torch.empty(max(nout, 1), dtype=torch.float64, device=self.device) if want_var else None
        with torch.cuda.device(self.device):
            rc = _lib.lib().cgp_predict_batched_dev(self.n_obj, self._p(self.off), self.max_n, self.dim,
                                                    self._p(self.x), self._p(self.y), self._p(self.y0),
                                                    self._p(self.y_err), _lib.hptr(h), float(nugget), float(floor),
                                                    int(flags), self._p(grid), self._p(goff), m, self._p(new_y0),
                                                    self._p(mean), self._p(var), self._p(self._info), self._stream())
        _lib.check(rc, "cgp_predict_batched_dev")
        return mean[:nout], (var[:nout] if want_var else None), self._info[:self.n_obj]

    def step_dev(self, hyp, nugget, grid, goff=None, new_y0=None, want_var=True, floor=0.0, flags=0,
                 template_mean=False, uniform_grid=False, out=None):
        """One pass of the hot path (cgp_step_batched_dev): log-likelihood AND prediction at the same hyperparameters
        from ONE factorisation per object.  grid / goff / new_y0 are device tensors as in predict_dev; template_mean,
        uniform_grid as in predict_factored_dev.  out: optional dict of preallocated device tensors "ll", "mean", "var".
        -> (ll_obj, mean, var, info) device tensors."""
        h = self._hyp(hyp)
        m = 0 if goff is not None else int(grid.shape[0])
        nout = int(goff[-1].item()) if goff is not None else self.n_obj * m
        new = lambda n: torch.empty(max(n, 1), dtype=torch.float64, device=self.device)
        ll = out["ll"] if out else new(self.n_obj)
        mean = out["mean"] if out else new(nout)
        var = (out["var"] if out else new(nout)) if want_var else None
        fl = int(flags) | (_lib.CGP_MEAN_TEMPLATE if template_mean else 0) | (_lib.CGP_GRID_UNIFORM if uniform_grid else 0)
        with torch.cuda.device(self.device):
            rc = _lib.lib().cgp_step_batched_dev(self.n_obj, self._p(self.off), self.max_n, self.dim, self._p(self.x),
                                                 self._p(self.y), self._p(self.y0), self._p(self.y_err), _lib.hptr(h),
                                                 float(nugget), float(floor), fl, self._p(grid), self._p(goff), m,
                                                 self._p(new_y0), self._p(ll), self._p(mean), self._p(var),
                                                 self._p(self._info), self._stream())
        _lib.check(rc, "cgp_step_batched_dev")
        return ll[:self.n_obj], mean[:nout], (var[:nout] if want_var else None), self._info[:self.n_obj]

    def factor_dev(self, hyp, nugget=0.0, floor=0.0, flags=0, want_ll=False):
        """Factorise every object once (objects of <= 64 points): returns an opaque device workspace
        holding the Cholesky factor and z = L^-1 (y - y0), reusable by predict_factored_dev for any number of grids.
        want_ll: also return each object's log-likelihood (fac["ll"], device) from the same factorisation."""
        assert 0 < self.max_n <= 64, "factor_dev handles objects of 1..64 points"
        h = self._hyp(hyp)
        stride = int(_lib.lib().cgp_factor_ws_doubles(self.max_n))
        ws = torch.empty(max(self.n_obj, 1) * stride, dtype=torch.float64, device=self.device)
        ll = torch.empty(max(self.n_obj, 1), dtype=torch.float64, device=self.device) if want_ll else None
        with torch.cuda.device(self.device):
            rc = _lib.lib().cgp_factor_batched_dev(self.n_obj, self._p(self.off), self.max_n, self.dim, self._p(self.x),
                                                   self._p(self.y), self._p(self.y0), self._p(self.y_err), _lib.hptr(h),
                                                   float(nugget), float(floor), int(flags), self._p(ws), self._p(ll),
                                                   self._p(self._info), self._stream())
        _lib.check(rc, "cgp_factor_batched_dev")
        return {"ws": ws, "hyp": h, "nugget": float(nugget), "flags": int(flags), "ll": None if ll is None else ll[:self.n_obj]}

    def predict_factored_dev(self, fac, grid, goff=None, new_y0=None, want_var=True, template_mean=False, uniform_grid=False):
        """Prediction from a factor_dev() workspace; same outputs as predict_dev.  template_mean: new_y0 is
        the packed shared mean [template on the grid (M) | per-object offsets (B)] (CGP_MEAN_TEMPLATE).
        uniform_grid: hint that the shared 1D grid is uniformly spaced (CGP_GRID_UNIFORM; verified by the library)."""
        m = 0 if goff is not None else int(grid.shape[0])
        nout = int(goff[-1].item()) if goff is not None else self.n_obj * m
        mean = torch.empty(max(nout, 1), dtype=torch.float64, device=self.device)
        var = torch.empty(max(nout, 1), dtype=torch.float64, device=self.device) if want_var else None
        with torch.cuda.device(self.device):
            rc = _lib.lib().cgp_predict_factored_dev(self.n_obj, self._p(self.off), self.max_n, self.dim, self._p(self.x),
                                                     _lib.hptr(fac["hyp"]), fac["nugget"],
                                                     fac["flags"] | (_lib.CGP_MEAN_TEMPLATE if template_mean else 0)
                                                     | (_lib.CGP_GRID_UNIFORM if uniform_grid else 0), self._p(fac["ws"]),
                                                     self._p(self._info), self._p(grid), self._p(goff), m,
                                                     self._p(new_y0), self._p(mean), self._p(var), self._stream())
        _lib.check(rc, "cgp_predict_factored_dev")
        return mean[:nout], (var[:nout] if want_var else None), self._info[:self.n_obj]

    def predict(self, hyp, nugget, grid, goff=None, new_y0=None, want_var=True, floor=0.0, flags=0, mean_template=None):
        """grid: host array, shared (M,[2]) or per-object flat with goff (int64 B+1).
        new_y0: the mean function on the grid, one row per object; or mean_template=(template (M,),
        offsets (B,)) for a shared template plus one offset per object (shared grid only): only M + B
        doubles are uploaded instead of B x M.
        -> mean, var (host; shape (B,M) for a shared grid, flat otherwise), info."""
        g = self._up_grid(grid) if goff is not None else self._up(np.asarray(grid, dtype=np.float64))
        go = self._up(np.asarray(goff, dtype=np.int64)) if goff is not None else None
        if mean_template is not None:
            assert goff is None and new_y0 is None
            tmpl, diff = mean_template
            packed = np.concatenate([np.asarray(tmpl, dtype=np.float64).ravel(), np.asarray(diff, dtype=np.float64).ravel()])
            assert packed.size == int(g.shape[0]) + self.n_obj, "template must cover the grid, offsets the objects"
            new_y0, flags = packed, int(flags) | _lib.CGP_MEAN_TEMPLATE
        ny0 = self._up(np.asarray(new_y0, dtype=np.float64)) if new_y0 is not None else None
        if goff is None and self.dim == 1:
            flags = int(flags) | _lib.CGP_GRID_UNIFORM          # a hint; the library checks the grid and the length scale
        mean, var, info = self.predict_dev(hyp, nugget, g, go, ny0, want_var, floor, flags)
        mean_h = self._down(mean, sync=False)                # three copies in flight, one synchronisation
        var_h = self._down(var, sync=False) if want_var else None
        info_h = self._down(info, sync=False)
        self._sync()
        if goff is None:
            m = int(g.shape[0])
            mean_h = mean_h.reshape(self.n_obj, m)
            var_h = var_h.reshape(self.n_obj, m) if want_var else None
        return mean_h, var_h, info_h

    def covariance(self, hyp, nugget, grid=None, objects=None, floor=0.0, flags=0, goff=None):
        """covariance_matrix of the objects [i0, i1) (default: all) in ONE call (cgp_covariance_batched_dev):
        grid given (host array, shared by all objects) -> (k, M, M) host array; grid None -> every object on its own
        epochs (new_binning=None) -> list of (N_b, N_b) host arrays; grid flat with goff (host int64 (B+1,)) -> one grid
        per object, list of (M_b, M_b) host arrays.  Objects of <= 64 points.
        hyp (B, nh) with an optional (B,) nugget: object b with its own row, as in predict_dev (cgp_covariance_objhyp_dev)."""
        i0, i1 = (0, self.n_obj) if objects is None else (int(objects[0]), int(objects[1]))
        k = i1 - i0
        oh = self._objhyp(hyp, nugget)
        h = None if oh is not None else self._hyp(hyp)
        ragged = grid is None or goff is not None
        if ragged:
            if grid is None:
                g, d_goff, goff_h = self.x, self.off, self.off_host
            else:
                goff_h = np.ascontiguousarray(goff, dtype=np.int64)
                g, d_goff = self._up_grid(grid), self._up(goff_h)
            m = 0
            sizes = np.diff(goff_h[i0:i1 + 1])
            coff_h = np.zeros(self.n_obj + 1, dtype=np.int64)
            coff_h[i0 + 1:i1 + 1] = np.cumsum(sizes * sizes)
            coff, tot = self._up(coff_h), int(coff_h[i1])
            goff_ptr, goff_host_ptr, coff_ptr = d_goff.data_ptr() + 8 * i0, goff_h.ctypes.data + 8 * i0, coff.data_ptr() + 8 * i0
        else:
            g = self._up(np.asarray(grid, dtype=np.float64))
            m = int(g.shape[0]); tot = k * m * m
            goff_ptr = goff_host_ptr = coff_ptr = None
        out = torch.empty(max(tot, 1), dtype=torch.float64, device=self.device)
        batch_args = (k, self.off.data_ptr() + 8 * i0, self.max_n, self.dim, self._p(self.x), self._p(self.y_err))
        out_args = (self._p(g), goff_ptr, goff_host_ptr, m, self._p(out), coff_ptr, self._info.data_ptr() + 4 * i0,
                    self._stream())
        with torch.cuda.device(self.device):
            if oh is not None:
                nh = 2 if self.dim == 1 else 4
                rc = _lib.lib().cgp_covariance_objhyp_dev(*batch_args, self._p(oh[0]) + 8 * nh * i0,
                                                          None if oh[1] is None else self._p(oh[1]) + 8 * i0, oh[2],
                                                          float(floor), int(flags), *out_args)
            else:
                rc = _lib.lib().cgp_covariance_batched_dev(*batch_args, _lib.hptr(h), float(nugget), float(floor), int(flags),
                                                           *out_args)
        _lib.check(rc, "cgp_covariance_objhyp_dev" if oh is not None else "cgp_covariance_batched_dev")
        flat = self._down(out[:tot], sync=False)
        info = self._down(self._info[i0:i1], sync=False)
        self._sync()
        if ragged:
            return [flat[coff_h[i] :coff_h[i + 1]].reshape(sizes[i - i0], sizes[i - i0]) for i in range(i0, i1)], info
        return flat.reshape(k, m, m), info

    def loo_dev(self, hyp, nugget, mean=None, mode=_lib.CGP_LOO_PLAIN, floor=0.0, flags=0, ranges=None):
        """Closed-form leave-one-out; `mean` (flat, host) replaces the batch's y0 when given.
        ranges: (first, end) object ranges to compute, one launch each (default: every object in one launch); the
        outputs span every point either way, and those of objects outside the ranges are left unwritten.
        -> pred, pred_var, pull, resid (flat DEVICE tensors), info (device)."""
        m = self._up(np.asarray(mean, dtype=np.float64)) if mean is not None else self.y0
        outs = [torch.empty(max(self.n_pts, 1), dtype=torch.float64, device=self.device) for _ in range(4)]
        oh = self._objhyp(hyp, nugget)
        h = None if oh is not None else self._hyp(hyp)
        nh = 2 if self.dim == 1 else 4
        for a, b in ([(0, self.n_obj)] if ranges is None else ranges):
            # object range [a, b): the CSR offsets stay absolute, so the kernel reads and writes the full arrays
            off, info = self._p(self.off) + 8 * a, self._p(self._info) + 4 * a
            with torch.cuda.device(self.device):
                if oh is not None:
                    rc = _lib.lib().cgp_loo_objhyp_dev(b - a, off, self.max_n, self.dim, self._p(self.x),
                                                       self._p(self.y), self._p(m), self._p(self.y_err),
                                                       self._p(oh[0]) + 8 * nh * a,
                                                       None if oh[1] is None else self._p(oh[1]) + 8 * a, oh[2],
                                                       float(floor), int(flags), int(mode),
                                                       *[self._p(o) for o in outs], info, self._stream())
                else:
                    rc = _lib.lib().cgp_loo_batched_dev(b - a, off, self.max_n, self.dim, self._p(self.x),
                                                        self._p(self.y), self._p(m), self._p(self.y_err), _lib.hptr(h),
                                                        float(nugget), float(floor), int(flags), int(mode),
                                                        *[self._p(o) for o in outs], info, self._stream())
            _lib.check(rc, "cgp_loo_objhyp_dev" if oh is not None else "cgp_loo_batched_dev")
        return [o[:self.n_pts] for o in outs] + [self._info[:self.n_obj]]

    def loo(self, hyp, nugget, mean=None, mode=_lib.CGP_LOO_PLAIN, floor=0.0, flags=0):
        """loo_dev with the results brought to the host: pred, pred_var, pull, resid (flat), info."""
        return [self._down(t) for t in self.loo_dev(hyp, nugget, mean, mode, floor, flags)]

    def moments(self, v, center=0.0):
        """(sum (v - center), sum (v - center)^2) of a device tensor, reduced on the device (cgp_moments_dev)."""
        out = torch.empty(2, dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().cgp_moments_dev(self._p(v), int(v.numel()), float(center), self._p(out), self._stream()),
                       "cgp_moments_dev")
        s1, s2 = out.cpu().tolist()
        return s1, s2

    def matrices(self, hyp, nugget, want_k=True, want_kinv=True, floor=0.0, flags=0):
        """kernel_matrix / inv_kernel_matrix per object (lists of (N,N) host arrays)."""
        h = self._hyp(hyp)
        sizes = np.diff(self.off_host)
        moff_h = np.zeros(self.n_obj + 1, dtype=np.int64)
        moff_h[1:] = np.cumsum(sizes * sizes)
        moff = self._up(moff_h)
        tot = int(moff_h[-1])
        kmat = torch.empty(max(tot, 1), dtype=torch.float64, device=self.device) if want_k else None
        kinv = torch.empty(max(tot, 1), dtype=torch.float64, device=self.device) if want_kinv else None
        with torch.cuda.device(self.device):
            rc = _lib.lib().cgp_matrices_batched_dev(self.n_obj, self._p(self.off), self.max_n, self.dim,
                                                     self._p(self.x), self._p(self.y_err), _lib.hptr(h), float(nugget),
                                                     float(floor), int(flags), self._p(moff), self._p(kmat),
                                                     self._p(kinv), self._p(self._info), self._stream())
        _lib.check(rc, "cgp_matrices_batched_dev")
        out = []
        for t in (kmat, kinv):
            if t is None:
                out.append(None)
                continue
            flat = self._down(t[:tot])
            out.append([flat[moff_h[i]:moff_h[i + 1]].reshape(sizes[i], sizes[i]) for i in range(self.n_obj)])
        return out[0], out[1], self._down(self._info[:self.n_obj])


class StreamedEvaluator:
    """LL + prediction of a host-resident batch with copies and kernels overlapped (cgp_streamer_*).

    The batch is cut into chunks of objects; chunk k is uploaded on one of `n_streams` CUDA
    streams while chunk k-1 computes and chunk k-2 downloads (PCIe is full duplex), so the
    end-to-end time approaches max(copy, compute) instead of their sum.  The chunk loop (about a
    dozen copies and launches per chunk) runs inside the library: one native call per run().
    Inputs and outputs are pinned host arrays owned by this object; equal-length objects only
    (x, y, y0, y_err of shape (B, N)), shared prediction grid.  The mean function on the grid is
    either "new_y0" (B, M) or, with shared_mean=True, "template" (M,) + "diff" (B,) -- the
    reference's own inputs (Mean_Y interpolated on the grid, plus diff[sn]; mean.py:92-101) -- which
    saves 8 M bytes of upload per object."""

    def __init__(self, n_obj, n_pts, m_grid, dim=1, n_chunks=8, n_streams=3, device=None, shared_mean=False):
        _lib.require_device()
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.B, self.N, self.M, self.dim = int(n_obj), int(n_pts), int(m_grid), int(dim)
        self.chunk = max(1, -(-self.B // max(1, min(int(n_chunks), max(self.B, 1)))))
        xs = (self.B, self.N, 2) if dim == 2 else (self.B, self.N)
        pin = lambda *shape: torch.empty(shape, dtype=torch.float64, pin_memory=True)
        self.shared_mean = bool(shared_mean)
        # x | y | y_err | y0 as rows of ONE pinned block, mean | var of another: a chunk of all of them then travels as one
        # two-dimensional copy (with both directions of the link busy every extra copy costs ~20 us: cgp_stream.cu)
        self._in = pin(3 if dim == 2 else 4, self.B, self.N)
        self._out = pin(2, self.B, self.M)
        rows = (None, 0, 1, 2) if dim == 2 else (0, 1, 2, 3)
        self.h = {"x": pin(*xs) if dim == 2 else self._in[0], "y": self._in[rows[1]], "y_err": self._in[rows[2]],
                  "y0": self._in[rows[3]], "ll": pin(self.B), "mean": self._out[0], "var": self._out[1]}
        if self.shared_mean:
            self._packed_mean = pin(self.M + self.B)                # [template | offsets], what CGP_MEAN_TEMPLATE reads
            self.h["template"], self.h["diff"] = self._packed_mean[:self.M], self._packed_mean[self.M:]
        else:
            self.h["new_y0"] = pin(self.B, self.M)
        self.h_info = torch.empty(self.B, dtype=torch.int32, pin_memory=True)
        self._handle = _lib.C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().cgp_streamer_create(self.chunk, self.N, self.M, self.dim, int(n_streams),
                                                      _lib.C.byref(self._handle)), "cgp_streamer_create")
        self.h2d_bytes = self.d2h_bytes = 0

    def __del__(self):
        h = getattr(self, "_handle", None)
        if h is not None and h.value:
            try:
                _lib.lib().cgp_streamer_destroy(h)
            except Exception:
                pass
            h.value = None

    def host(self, name):
        """numpy view of a pinned staging array: fill inputs / read outputs in place."""
        return self.h[name].numpy()

    def set_mean_template(self, time_mean, mean_y):
        """The shared mean as the reference defines it (mean.py:28-31: cubic spline through (Time_mean, Mean_Y)):
        with shared_mean=True, y0 = spline(x) + diff[sn] is then evaluated on the device like FITPACK would
        (cgp_spline_mean_dev) instead of being uploaded ("y0" is ignored), and "template" is filled with the
        spline on `grid` at the next run()."""
        import scipy.interpolate as inter
        assert self.shared_mean and self.dim == 1, "a 1D template needs shared_mean=True"
        self._spline = inter.InterpolatedUnivariateSpline(time_mean, mean_y)
        t, c, k = self._spline._eval_args
        assert k == 3
        t = np.ascontiguousarray(t, dtype=np.float64); c = np.ascontiguousarray(c, dtype=np.float64)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().cgp_streamer_set_mean_spline(self._handle, _lib.hptr(t), _lib.hptr(c), len(t)),
                       "cgp_streamer_set_mean_spline")

    def run(self, hyp, nugget, grid, floor=0.0, flags=0):
        """-> (ll_sum, ll (B,), mean (B,M), var (B,M), info (B,)) as numpy views of the pinned outputs."""
        C = _lib.C
        h = np.ascontiguousarray(np.asarray(hyp, dtype=np.float64).ravel())
        g = np.ascontiguousarray(grid, dtype=np.float64)
        assert g.shape[0] == self.M, "grid must have the %d points the evaluator was built for" % self.M
        p = lambda t: t.data_ptr()
        mean_fn = self._packed_mean if self.shared_mean else self.h["new_y0"]
        spline = getattr(self, "_spline", None)
        if spline is not None:
            self.h["template"].numpy()[...] = spline(g)
        total, up, down = C.c_double(0.0), C.c_int64(0), C.c_int64(0)
        rc = _lib.lib().cgp_streamer_run(self._handle, self.B, p(self.h["x"]), p(self.h["y"]),
                                         None if spline is not None else p(self.h["y0"]), p(self.h["y_err"]),
                                         _lib.hptr(h), float(nugget), float(floor),
                                         int(flags) | (_lib.CGP_MEAN_TEMPLATE if self.shared_mean else 0) | _lib.CGP_GRID_UNIFORM,
                                         _lib.hptr(g), p(mean_fn), p(self.h["ll"]), p(self.h["mean"]), p(self.h["var"]),
                                         p(self.h_info), C.byref(total), C.byref(up), C.byref(down))
        _lib.check(rc, "cgp_streamer_run")
        self.h2d_bytes, self.d2h_bytes = int(up.value), int(down.value)
        return float(total.value), self.h["ll"].numpy(), self.h["mean"].numpy(), self.h["var"].numpy(), self.h_info.numpy()
