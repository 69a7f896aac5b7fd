"""Drop-in objects for cosmogp's Gaussian_process / gaussian_process /
gaussian_process_nobject (cosmogp/Gaussian_process.py:78-393): same constructor
arguments, methods, attributes and error behaviour; numpy in, numpy out.  The
per-object Python loops of the reference (:207, :264, :304, :349) are replaced by
single batched launches on a device-resident copy of the data.  Which objects are too large for those launches is
decided in one place, batch.SizeSplit; they go through the blocked HBM factorisation, all of them at once: for
likelihoods under shared hyperparameters (dense.log_likelihoods, every object of the batch then), for the likelihood
evaluations of per-object fits (dense.log_likelihoods_dev, from DeviceBatch.ll_objhyp) and for predictions
(dense.predictions: the large objects of a per-object prediction, or every object of a batch with a large one under
shared hyperparameters).  Each of these results is bit for bit that of the object alone on the blocked path.

Differences (SURVEY.md section 9.1):
  * `svd_method`: every object is factorised by the device Cholesky kernels whatever the flag says (for a
    positive-definite K the two reference paths agree to rounding).  They differ when an object's K is NOT
    numerically positive definite (noise-free data, duplicate epochs): with svd_method=False the call raises
    numpy.linalg.LinAlgError like the reference (inv_matrix.py:23); with svd_method=True (the reference's
    default) exactly those objects -- the ones whose device factorisation reported info != 0 -- are redone by
    the host reference check `inv_matrix.svd_inverse` (pseudo-inverse above s = 1e-15 and log det over the
    kept singular values, inv_matrix.py:4-18), so the call never raises, as in the reference.  A K that is
    positive definite in floating point but has singular values below 1e-15 keeps its Cholesky result where
    the reference would truncate (tests/test_gpu_facade.py::test_svd_method_* pin both behaviours).
  * `get_prediction(COV='diag')` computes only the variance diagonal
    (`prediction_variance`); COV=True keeps `covariance_matrix`, materialised per object
    on access.  `kernel_matrix` / `inv_kernel_matrix` are materialised on access too.
  * `fit_nugget` exists from construction (quirk Q4); `new_binning=None` predicts every
    object on its own epochs (the reference's stale loop index, quirk Q3, is not kept).
  * y, Time, y_err may also be 2-D ndarrays (equal-length objects), which avoids
    10^5 tiny numpy arrays.
"""
import numpy as np
from scipy.optimize import fmin

from . import _lib
from . import mean as _mean
from .batch import DeviceBatch, RaggedView, SizeSplit, pack_csr
from .kernel import init_rbf, rbf_kernel_1d, rbf_kernel_2d


_DEVICE = object()                       # marker: the per-object likelihoods of the latest evaluation are still on the device
_NO_BAD = np.zeros(0, dtype=np.int32)


class _LazyMatrices(object):
    """list-like of per-object matrices computed on the device on first access."""

    def __init__(self, n, make):
        self._n, self._make, self._cache = n, make, {}

    def __len__(self):
        return self._n

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self[j] for j in range(*i.indices(self._n))]
        if i < 0:
            i += self._n
        if not 0 <= i < self._n:
            raise IndexError(i)
        if i not in self._cache:
            self._cache[i] = self._make(i)
        return self._cache[i]

    def __iter__(self):
        return (self[i] for i in range(self._n))


class _LazyMeanOnGrid:
    """`warning_pf` of a shared-grid prediction: template + diff[sn], row sn built on access."""

    def __init__(self, template, diff):
        self.template, self.diff = np.asarray(template), np.asarray(diff)
        self.shape = (len(self.diff), len(self.template))

    def __len__(self):
        return len(self.diff)

    def __getitem__(self, i):
        return np.asarray(self)[i] if not isinstance(i, (int, np.integer)) else self.template + self.diff[i]

    def __array__(self, dtype=None, copy=None):
        out = self.template[None, :] + self.diff[:, None]
        return out if dtype is None else out.astype(dtype)


def is_per_object_grid(new_binning, dim):
    """True when `new_binning` of get_prediction is one grid per object rather than one grid shared by all: a sequence
    whose first element is itself a grid ((M_i,) in 1D, (M_i, 2) in 2D) -- a list, an object ndarray, or an equal-length
    (B, M) / (B, M, 2) ndarray, the forms y and Time take.  None, a 1-D array or list of floats and an (M, 2) array
    are shared grids."""
    return new_binning is not None and len(new_binning) > 0 and np.ndim(new_binning[0]) == dim


class Gaussian_process:
    "Gaussian process regressor (device-backed)."

    def __init__(self, y, Time, kernel='RBF1D',
                 y_err=None, diff=None, Mean_Y=None,
                 Time_mean=None, substract_mean=False, devices=None):
        """Arguments of cosmogp/Gaussian_process.py:82-88, plus `devices` (None: the current GPU; 'all', an int or a
        list of device ids: the objects are sharded over those GPUs of the box inside this process -- see
        cosmogp_b200.multi.ShardedBatch; likelihood, joint fit and shared-grid predictions are available there)."""
        kernel_choice = ['RBF1D', 'RBF2D']
        assert kernel in kernel_choice, '%s is not in implemented kernel' % (kernel)

        self._dim = 1 if kernel == 'RBF1D' else 2
        self.kernel = rbf_kernel_1d if kernel == 'RBF1D' else rbf_kernel_2d
        sigma, L = init_rbf(Time, y) if len(y) else (np.nan, np.nan)         # :145-146, :153-154 (empty: a rank's shard)
        self.hyperparameters = np.array([sigma, L]) if self._dim == 1 else np.array([sigma, L, L, 0.])

        self.y = y
        self.N_sn = len(y)
        self.Time = Time
        self.nugget = 0.
        self.fit_nugget = False
        self.flags = 0                      # _lib.CGP_AMP_ON_AUTOCOV to opt out of quirk Q2

        self._x_flat, self._off = pack_csr(Time, self._dim)
        self._y_flat, off_y = pack_csr(y, 1)
        assert np.array_equal(self._off, off_y), 'y and Time should have the same structure'
        self._split = SizeSplit(self._off)
        if y_err is not None:
            self.y_err = y_err
            self._ye_flat, off_e = pack_csr(y_err, 1)
            assert np.array_equal(self._off, off_e), 'y_err and y should have the same structure'
        else:
            self.y_err = [np.zeros(n) for n in np.diff(self._off)]         # :161-169
            self._ye_flat = None

        self.Mean_Y = Mean_Y
        self.Time_mean = Time_mean
        self.substract_mean = substract_mean
        self.diff = np.array([None] * self.N_sn) if diff is None else diff  # :175-178

        if self.substract_mean or self.Mean_Y is not None:                  # :180-186
            self._y0_flat, self._diff_used = _mean.batched_mean(
                self._x_flat, self._y_flat, self._off, self._dim, self.Mean_Y, self.Time_mean, self.diff)
            self.y0 = RaggedView(self._y0_flat, self._off)
        else:
            self._y0_flat, self._diff_used = None, np.zeros(self.N_sn)
            self.y0 = np.zeros(self.N_sn)

        self.as_the_same_time = True
        self._grid_csr = (self._x_flat, self._off)       # the prediction grid as a CSR when it is one grid per object
        self._ll_per_object = None
        self._devices = devices
        self.gather_over_nvlink = False     # multi-GPU outputs: False = every GPU's own PCIe link, True = NCCL gather on GPU 0 first
        self._batch = None
        self._dist = False              # True for objects made by `sharded()`: likelihoods are all-reduced

    @classmethod
    def sharded(cls, y, Time, kernel='RBF1D', y_err=None, diff=None, Mean_Y=None, Time_mean=None,
                substract_mean=False, rank=None, world=None):
        """One process per GPU (torch.distributed): every rank passes the FULL lists and keeps the
        contiguous range of objects `local_range`, balanced by sum N^3 (cosmogp_b200.sharding).  Objects
        are independent, so the only exchange is one all-reduced double per likelihood evaluation
        (summed in rank order: identical on every rank); `find_hyperparameters` therefore returns the
        same optimum everywhere and `get_prediction` fills the local objects (`gather` collects them)."""
        from . import sharding
        sizes = [len(v) for v in y]
        a, b = sharding.my_range(sizes, rank, world)
        cut = lambda v: None if v is None else v[a:b]
        obj = cls(y[a:b], Time[a:b], kernel=kernel, y_err=cut(y_err), diff=cut(diff), Mean_Y=Mean_Y,
                  Time_mean=Time_mean, substract_mean=substract_mean)
        sigma, L = init_rbf(Time, y)                     # the global initial guess (quirk Q6 uses the LAST object)
        obj.hyperparameters = np.array([sigma, L]) if obj._dim == 1 else np.array([sigma, L, L, 0.])
        obj._dist, obj.local_range, obj.N_total, obj._all_sizes = True, (a, b), len(y), sizes
        obj._all_split = SizeSplit(np.concatenate([[0], np.cumsum(sizes, dtype=np.int64)]))
        return obj

    def gather(self, per_object_arrays, root=None):
        """All ranks' per-object arrays (e.g. `Prediction`) concatenated in object order: on every rank (root=None,
        an all-gather) or on rank `root` only (the final gather: each rank sends its slice once; None elsewhere)."""
        from . import sharding
        flat = np.concatenate([np.asarray(v, dtype=np.float64).ravel() for v in per_object_arrays]) if len(per_object_arrays) else np.zeros(0)
        per = [len(np.asarray(v).ravel()) for v in per_object_arrays]
        import torch.distributed as dist
        if not (self._dist and dist.is_initialized() and dist.get_world_size() > 1):
            return list(per_object_arrays)
        # equal-length outputs (shared grid); the width comes from the grid, not from the local objects (a rank may own none)
        assert self.as_the_same_time or not is_per_object_grid(self.new_binning, self._dim), \
            "gather() needs a prediction on a shared grid, not one grid per object"
        width = 0 if self.as_the_same_time else len(self.new_binning)
        assert width and all(p == width for p in per), "gather() needs a prediction on a shared grid"
        ranges = sharding.balanced_ranges(self._all_sizes, dist.get_world_size())
        counts = [(r[1] - r[0]) * width for r in ranges]
        if root is not None:
            allflat = sharding.gather_to_root(flat, counts, root=root, device=self._device)
            return None if allflat is None else list(allflat.reshape(-1, width))
        allflat = sharding.gather_ragged(flat, counts, device=self._device)
        return list(allflat.reshape(-1, width)) if width else []

    # ------------------------------------------------------------------ device state
    @property
    def batch(self):
        if self._batch is None:
            if self._devices is not None:
                from .multi import ShardedBatch
                self._batch = ShardedBatch(self._x_flat, self._y_flat, self._off, y0=self._y0_flat,
                                           y_err=self._ye_flat, dim=self._dim, devices=self._devices)
            else:
                self._batch = DeviceBatch(self._x_flat, self._y_flat, self._off, y0=self._y0_flat,
                                          y_err=self._ye_flat, dim=self._dim)
        return self._batch

    @property
    def _any_large(self):
        """With shared hyperparameters, a batch with any large object (batch.SizeSplit) goes through the HBM-resident
        blocked factorisation, all objects in grouped calls: likelihoods (`_blocked_log_likelihoods`) and predictions
        (dense.predictions).  Sharded objects decide from the sizes of
        ALL objects, so that every rank takes the same branch (and the same collectives)."""
        return len((self._all_split if self._dist else self._split).large) > 0

    @property
    def _device(self):
        import torch
        return torch.device("cuda", torch.cuda.current_device())

    def _object_slices(self, i):
        """host views x, y, y_err, y0 of object i (y_err and y0 are None when the batch has none)"""
        o0, o1 = int(self._off[i]), int(self._off[i + 1])
        return tuple(None if a is None else a[o0:o1] for a in (self._x_flat, self._y_flat, self._ye_flat, self._y0_flat))

    def _blocked_log_likelihoods(self, hyperparameter, nugget):
        """(ll, info) of every object by the grouped blocked factorisation (dense.log_likelihoods), each ll bit for bit
        dense.LargeObject.factor's; info 1 where the covariance is not positive definite.  The batch (with devices=...,
        one of the facade's arrays on the current GPU) and a workspace bounded by dense.LL_WS_BYTES are made on the first
        call and kept: fits evaluate hundreds of times."""
        from . import dense
        if not self.N_sn:
            return np.zeros(0), np.zeros(0, dtype=np.int32)
        if getattr(self, "_blocked", None) is None:
            batch = self.batch if self._devices is None else DeviceBatch(
                self._x_flat, self._y_flat, self._off, y0=self._y0_flat, y_err=self._ye_flat, dim=self._dim)
            self._blocked = (batch, dense.ll_workspace(self._split.sizes, batch.device))
        batch, work = self._blocked
        ll, info = dense.log_likelihoods(batch, None, hyperparameter, nugget, self.flags, work)
        return ll, (info != 0).astype(np.int32)

    @staticmethod
    def _raise_if_bad(info):
        bad = np.nonzero(info)[0]
        if len(bad):
            raise np.linalg.LinAlgError(
                "%d-th leading minor of the covariance of object %d is not positive definite "
                "(%d object(s) affected)" % (int(info[bad[0]]), int(bad[0]), len(bad)))

    # ------------------------------------------------------------------ likelihood
    def compute_log_likelihood(self, Hyperparameter, svd_method=True):
        """Global log likelihood for a set of hyperparameters (:191-213): one launch."""
        if self.fit_nugget:
            Nugget = Hyperparameter[-1]
            hyperparameter = Hyperparameter[:-1]
        else:
            Nugget = self.nugget
            hyperparameter = Hyperparameter
        if self._any_large:
            per_object, info = self._blocked_log_likelihoods(hyperparameter, Nugget)
            total = None
        else:
            # the sum over objects is reduced on the device: 16 bytes come back per evaluation, the per-object
            # values stay there until `log_likelihood_per_object` is read
            total, n_bad = self.batch.log_likelihood_total(hyperparameter, Nugget, flags=self.flags)
            per_object, info = _DEVICE, _NO_BAD
            if n_bad:
                per_object, info = self.batch.ll_host(), self.batch.info_host()
        if info.any() and svd_method:                       # the reference's default never raises (inv_matrix.py:4-18)
            per_object = np.array(per_object, dtype=float)
            for i in np.nonzero(info)[0]:
                per_object[i] = self._svd_object(int(i), hyperparameter, Nugget)[0]
            info = np.zeros_like(info)
            total = None
        if total is None:                                   # left to right, like the loop at :205-213
            total = float(np.add.accumulate(per_object)[-1]) if len(per_object) else 0.0
        if self._dist:
            from . import sharding
            total, bad = sharding.allreduce_sums([total, float(np.count_nonzero(info))], device=self._device)
            if bad:
                raise np.linalg.LinAlgError("%d object(s) with a covariance that is not positive definite" % int(bad))
        self._raise_if_bad(info)
        self.log_likelihood_per_object = per_object
        self.log_likelihood = np.array([total])             # shape (1,), quirk Q5

    @property
    def log_likelihood_per_object(self):
        """per-object log-likelihoods of the latest evaluation (fetched from the device when first read)"""
        if self._ll_per_object is _DEVICE:
            self._ll_per_object = self.batch.ll_host().copy()
        return self._ll_per_object

    @log_likelihood_per_object.setter
    def log_likelihood_per_object(self, value):
        self._ll_per_object = value

    def _svd_object(self, i, hyperparameter, nugget, grid=None, new_y0=0.0, want_var=False):
        """ONE object through the host reference check (inv_matrix.svd_inverse): used only for objects whose
        device Cholesky reported a non-positive pivot, and only when the caller asked for svd_method=True.
        -> (log-likelihood, mean on `grid` or None, variance diagonal or None), formulas of
        Gaussian_process.py:59-73 and :332-361."""
        import warnings
        from .inv_matrix import svd_inverse
        x, y, ye, y0 = self._object_slices(i)
        r = y - (y0 if y0 is not None else 0.0)
        kw = {"flags": self.flags} if self._dim == 2 else {}
        hyp = np.asarray(hyperparameter, dtype=float)
        warnings.warn("covariance of object %d is not positive definite: pseudo-inverse by the host SVD reference "
                      "check (svd_method=True, cosmogp/inv_matrix.py:4-18)" % i, RuntimeWarning, stacklevel=3)
        inv, logdet = svd_inverse(self.kernel(x, hyp, nugget=nugget, y_err=ye, **kw), return_logdet=True)
        w = inv @ r
        ll = -0.5 * float(r @ w) - 0.5 * len(r) * np.log(2 * np.pi) - 0.5 * logdet
        if grid is None:
            return ll, None, None
        h = self.kernel(x, hyp, new_x=grid)
        mean = h @ w + new_y0
        var = None
        if want_var:
            amp = hyp[0] ** 2 if (self._dim == 1 or self.flags & _lib.CGP_AMP_ON_AUTOCOV) else 1.0
            var = amp + nugget ** 2 - ((h @ inv) * h).sum(axis=1)
        return ll, mean, var

    def find_hyperparameters(self, hyperparameter_guess=None, nugget=False, svd_method=True):
        """Maximum likelihood with scipy.optimize.fmin on the host (:216-253); every
        simplex evaluation is one batched device launch."""
        if hyperparameter_guess is not None:
            assert len(self.hyperparameters) == len(hyperparameter_guess), 'should be same len'
            self.hyperparameters = hyperparameter_guess

        def _compute_log_likelihood(Hyper, svd_method=svd_method):
            self.compute_log_likelihood(Hyper, svd_method=svd_method)
            return -self.log_likelihood[0]

        initial_guess = [self.hyperparameters[i] for i in range(len(self.hyperparameters))]
        if nugget:
            self.fit_nugget = True
            initial_guess.append(1.)
        else:
            self.fit_nugget = False

        hyperparameters = fmin(_compute_log_likelihood, initial_guess, disp=False)

        for i in range(len(self.hyperparameters)):
            self.hyperparameters[i] = np.sqrt(hyperparameters[i] ** 2)
        if self.fit_nugget:
            self.nugget = np.sqrt(hyperparameters[-1] ** 2)

    def find_hyperparameters_per_object(self, hyperparameter_guess=None, nugget=False, svd_method=True, optimizer='device'):
        """One maximum-likelihood fit PER OBJECT -- the batched form of the reference's loop
        `for i: gp = gaussian_process(y[i], Time[i], ...); gp.find_hyperparameters(guess)`
        (docs/notebook/1D_kernel_example_with_noise.ipynb cell 13).  scipy's Nelder-Mead is replayed
        for all objects at once; every evaluation is one device launch.  optimizer='device': the
        simplices live on the device too (cgp_fit_objects_dev, no host round trips); 'host': the numpy
        statement of the same rules (cosmogp_b200.fit), kept as the cross-check -- both give identical results.
        Objects above 224 points are fitted too: every evaluation factors all of them at once by the grouped blocked
        factorisation (dense.log_likelihoods_dev, each likelihood bit for bit dense.LargeObject.factor's), driven by the
        numpy statement in both modes; with optimizer='device' the objects of up to 224 points still run
        cgp_fit_objects_dev, on a batch of their own.
        Sets `hyperparameters_per_object` (N_sn, n_hyp), `nugget_per_object` (N_sn,) and
        `log_likelihood_per_object`; an object whose covariance is not positive definite at a trial
        point gets +inf there (the reference would abort with LinAlgError)."""
        from .fit import nelder_mead_lockstep
        guess = np.asarray(self.hyperparameters if hyperparameter_guess is None else hyperparameter_guess, dtype=float)
        assert len(self.hyperparameters) == len(guess), 'should be same len'
        nh = len(guess)
        start = list(guess) + ([1.] if nugget else [])
        x0 = np.tile(np.asarray(start, dtype=float), (self.N_sn, 1))
        base_nugget = float(self.nugget)

        def fun(X, idx):
            ll, info = self.batch.ll_objhyp(X[:, :nh], idx, nugget_rows=X[:, nh] if nugget else None,
                                            nugget=base_nugget, flags=self.flags)
            f = -ll
            f[(info != 0) | ~np.isfinite(f)] = np.inf
            return f

        assert optimizer in ('device', 'host')
        if optimizer == 'device':
            # small objects on the device optimiser, large ones in lock step over the grouped likelihood
            small, big = self._split.small, self._split.large
            x, fval = np.empty_like(x0), np.empty(self.N_sn)
            its, calls = np.empty(self.N_sn, dtype=np.int64), np.empty(self.N_sn, dtype=np.int64)
            sb = self._small_batch()
            if sb is not None:
                x[small], fval[small], its[small], calls[small] = sb.fit_objects(x0[small], nugget=base_nugget, flags=self.flags)
            if len(big):
                x[big], fval[big], its[big], calls[big] = nelder_mead_lockstep(lambda X, idx: fun(X, big[idx]), x0[big])
        else:
            x, fval, its, calls = nelder_mead_lockstep(fun, x0)
        self.hyperparameters_per_object = np.sqrt(x[:, :nh] ** 2)              # abs, like :249-250
        self.nugget_per_object = np.sqrt(x[:, nh] ** 2) if nugget else np.full(self.N_sn, base_nugget)
        self.log_likelihood_per_object = -fval
        self.fit_iterations, self.fit_evaluations = its, calls

    def _small_batch(self):
        """The batch per-object fits and predictions run their small objects (batch.SizeSplit) on: `self.batch` when no
        object is large, None when every object is, and otherwise a DeviceBatch of the small objects alone, uploaded
        once from host slices, so that they get exactly the results of a batch without the large objects."""
        split = self._split
        if not len(split.large):
            return self.batch
        if not split.small.any():
            return None
        if getattr(self, "_small", None) is None:
            cut = lambda a: None if a is None else np.ascontiguousarray(a[split.points])
            self._small = DeviceBatch(cut(self._x_flat), cut(self._y_flat), split.small_off, y0=cut(self._y0_flat),
                                      y_err=cut(self._ye_flat), dim=self._dim)
        return self._small

    # ------------------------------------------------------------------ matrices
    def compute_kernel_matrix(self):
        """kernel_matrix[sn] = K(Time[sn]) with nugget and y_err (:256-267), on access."""
        hyp, nug = np.array(self.hyperparameters, dtype=float), float(self.nugget)
        self.kernel_matrix = _LazyMatrices(self.N_sn, lambda i: self._object_matrices(i, hyp, nug, True)[0])

    def _object_matrices(self, i, hyp, nug, svd=False):
        x, y, ye, _ = self._object_slices(i)
        if not self._split.small[i]:
            from . import dense
            return dense.object_matrices(x, ye, hyp, nug, self._dim, self.flags)
        sub = DeviceBatch(x, y, np.array([0, len(y)], dtype=np.int64), y_err=ye, dim=self._dim)
        k, kinv, info = sub.matrices(hyp, nug, flags=self.flags)
        if info.any() and svd:                              # inv_kernel_matrix of the reference's default path (:319-320)
            from .inv_matrix import svd_inverse
            return k[0], svd_inverse(k[0])
        self._raise_if_bad(info)
        return k[0], kinv[0]

    # ------------------------------------------------------------------ prediction
    def get_prediction(self, new_binning=None, COV=True, svd_method=True, per_object=False):
        """Interpolation (and its covariance) on a new grid (:270-361).

        new_binning None -> each object's own epochs; one grid per object (is_per_object_grid: a list of (M_i,) arrays in
        1D, of (M_i, 2) arrays in 2D, or a (B, M) / (B, M, 2) ndarray) -> object i on its own grid, outputs as for
        None; otherwise one grid shared by all objects.  COV: True (full matrices on
        access + diagonal), 'diag' (diagonal only) or False.  per_object=True predicts every
        object with its own fit (`hyperparameters_per_object`, `nugget_per_object`); with COV=True
        `covariance_matrix[i]` is then object i's predictive covariance under its fit as it stood at this call.
        devices=... does not take per_object.  Objects go down one of three routes, by batch.SizeSplit: the batched
        kernels; the grouped blocked path, dense.predictions (the large objects of a per-object prediction, or every
        object of a batch with a large one under shared hyperparameters); and, under shared hyperparameters with svd_method=True,
        the host SVD redo of the objects whose covariance is not positive definite.  Otherwise such an object raises
        LinAlgError."""
        own = new_binning is None
        per_grid = own or is_per_object_grid(new_binning, self._dim)        # one grid per object: Time or the caller's
        assert not (per_grid and not own and (self._devices is not None or self._dist)), \
            "with devices=... or sharded(), predictions take a shared grid, not one grid per object"
        if self._devices is not None:
            assert new_binning is not None and not per_object and COV in ('diag', False) and not self._any_large, \
                "with devices=... predictions use the shared hyperparameters (not per_object) on a shared grid, " \
                "with COV='diag' or False"
        if per_object:
            assert COV in (True, 'diag', False), "per_object predictions take COV=True, 'diag' or False"
        has_mean = self.substract_mean or self.Mean_Y is not None
        want_var = bool(COV)

        # hyperparameters: shared, or one row per object
        hyp, nug = np.array(self.hyperparameters, dtype=float), float(self.nugget)
        if per_object:
            hyp_b, nug_b = np.asarray(self.hyperparameters_per_object, dtype=float), np.asarray(self.nugget_per_object, dtype=float)
        self.compute_kernel_matrix()
        self.inv_kernel_matrix = _LazyMatrices(self.N_sn, lambda i: self._object_matrices(i, hyp, nug, bool(svd_method))[1])

        # the grid and the mean function on it; the outputs of object i are mean[rows[i]:rows[i + 1]].  One grid per
        # object is the CSR (grid, rows), with the mean function flat on it; own epochs are the case grid = Time.
        if own:
            grid, rows = self._x_flat, self._off
            new_y0 = self._y0_flat if has_mean else None                   # :308-309
        elif per_grid:
            assert len(new_binning) == self.N_sn, "one grid per object: %d grids for %d objects" % (len(new_binning), self.N_sn)
            grid, rows = pack_csr(new_binning, self._dim)
            new_y0 = None
            if has_mean:                                                    # template(grid_i) + diff[i], mean.py:92-101
                tmpl = _mean.template_on_grid(grid, self._dim, self.Mean_Y, self.Time_mean) if len(grid) else None
                new_y0 = (np.zeros(len(grid)) if tmpl is None else tmpl) + np.repeat(self._diff_used, np.diff(rows))
        else:
            grid = np.ascontiguousarray(new_binning, dtype=np.float64)
            rows = np.arange(self.N_sn + 1, dtype=np.int64) * len(grid)
            new_y0 = None
            if has_mean:                                                    # :310-312 via mean.py:92-101
                # mean on the grid = template(grid) + diff[sn]; without a template return_mean hands back
                # y0 (= diff) for any new_x.  Only the M template values and the N_sn offsets are uploaded.
                tmpl = _mean.template_on_grid(grid, self._dim, self.Mean_Y, self.Time_mean)
                new_y0 = _LazyMeanOnGrid(np.zeros(len(grid)) if tmpl is None else tmpl, self._diff_used)

        def on_grid(i):
            """object i's grid and the mean function on it (None: zero)"""
            if per_grid:
                s = slice(int(rows[i]), int(rows[i + 1]))
                return grid[s], (None if new_y0 is None else new_y0[s])
            return grid, (None if new_y0 is None else new_y0[i])

        # routes: the batched kernels on `batched`, the grouped blocked path (dense.predictions) for `blocked`
        split = self._split
        if per_object:
            batched, blocked = self._small_batch(), split.large
        elif self._any_large:
            batched, blocked = None, np.arange(self.N_sn, dtype=np.int64)
        else:
            batched, blocked = self.batch, ()
        whole = batched is not None and not len(blocked)         # the batched outputs are the outputs
        if not whole:
            mean, info = np.empty(int(rows[-1])), np.zeros(self.N_sn, dtype=np.int32)
            var = np.empty(int(rows[-1])) if want_var else None
        if batched is not None:
            # the objects and points it holds: all of them, or the small ones of a mixed batch
            objs = slice(None) if whole else split.small
            if per_grid:                                     # the grid points of those objects, and their CSR
                pts, goff = (slice(None), rows) if whole else split.small_csr(rows)
                kw = {"goff": goff, "new_y0": None if new_y0 is None else new_y0[pts]}
            else:
                kw = {"mean_template": None if new_y0 is None else (new_y0.template, new_y0.diff[objs])}
            if self._devices is not None:
                kw["gather"] = self.gather_over_nvlink
            m, v, inf = batched.predict(hyp_b[objs] if per_object else hyp, nug_b[objs] if per_object else nug,
                                        grid[pts] if per_grid else grid, want_var=want_var, flags=self.flags, **kw)
            if whole:
                mean, var, info = m.reshape(-1), (v.reshape(-1) if want_var else None), inf
            else:
                at = pts if per_grid else np.repeat(objs, len(grid))
                mean[at] = m.reshape(-1)
                if want_var:
                    var[at] = v.reshape(-1)
                info[objs] = inf
        if len(blocked):
            from . import dense
            if new_y0 is None:                               # the mean function in the outputs' layout of `blocked`
                ny0 = None
            elif per_grid:
                ny0 = dense._gather(new_y0, rows, blocked)[0]
            else:                                            # template + diff[i], the add of _LazyMeanOnGrid
                ny0 = new_y0.template[None, :] + new_y0.diff[blocked][:, None]
            m, v, _, inf = dense.predictions(self._x_flat, self._off, self._y_flat, self._y0_flat, self._ye_flat, grid,
                                             rows if per_grid else None, ny0, hyp_b[blocked] if per_object else hyp,
                                             nug_b[blocked] if per_object else nug, self._dim, self.flags,
                                             objects=blocked, want_var=want_var)
            bad = np.nonzero(inf)[0]
            if len(bad) and not (per_object or svd_method):  # the error LargeObject.factor raises for the first one
                raise np.linalg.LinAlgError("%d-th leading minor of the covariance is not positive definite" % int(inf[bad[0]]))
            at = dense._gather(np.arange(int(rows[-1]), dtype=np.int64), rows, blocked)[0]
            mean[at] = m
            if want_var:
                var[at] = v
            info[blocked] = inf != 0
        if info.any() and svd_method and not per_object:
            for i in np.nonzero(info)[0]:
                s = slice(int(rows[i]), int(rows[i + 1]))
                g, ny0 = on_grid(i)
                _, mean[s], v = self._svd_object(int(i), hyp, nug, g, 0.0 if ny0 is None else ny0, want_var)
                if want_var:
                    var[s] = v
            info = np.zeros_like(info)
        self._raise_if_bad(info)

        self.as_the_same_time = own
        self.new_binning = self.Time if own else new_binning
        self._grid_csr = (grid, rows) if per_grid else None
        # list-like views built in O(1) (a real list of 10^5 row arrays costs ~15 ms)
        self.Prediction = RaggedView(mean, rows)
        self.prediction_variance = RaggedView(var, rows) if want_var else None
        self.warning_pf = RaggedView(new_y0, rows) if per_grid and not own and new_y0 is not None else new_y0
        if COV is True:
            if per_object:
                self.covariance_matrix = self._covariance_matrices(np.array(hyp_b), np.array(nug_b))
            else:
                self.get_covariance_matrix()

    def get_covariance_matrix(self):
        """covariance_matrix[sn] = K(grid,grid)+nugget^2 - H K^-1 H^T (:340-361) under the shared hyperparameters.
        Objects of <= 64 points: written in bulk by cgp_covariance_batched_dev, a chunk of objects (<= 256 MB of
        matrices) per launch pair, when first read; larger objects a chunk at a time through the grouped blocked
        large-object path (dense.predictive_covariances)."""
        self.covariance_matrix = self._covariance_matrices(np.array(self.hyperparameters, dtype=float), float(self.nugget))

    def _covariance_matrices(self, hyp, nug):
        """covariance_matrix on the latest prediction's grid, built on access.  hyp (n_hyp,) and nug: shared, on
        self.batch when every object has <= 64 points.  hyp (N_sn, n_hyp) and nug (N_sn,): object i with row i, the
        small objects (batch.SizeSplit) on _small_batch() when each has <= 64 points (cgp_covariance_objhyp_dev).
        Every other object with data and a non-empty grid goes through dense.predictive_covariances (the blocked
        large-object path, grouped): a chunk of such objects (<= 256 MB of matrices, <= 2 GB of workspace) per call,
        when one of them is first read; a non-positive-definite object raises LinAlgError when it is read.  Objects
        without data (the prior) and empty grids are built here; one chunk of each kind is alive at a time."""
        from . import dense
        rows = np.ndim(hyp) == 2
        own = self.as_the_same_time
        ragged = self._grid_csr is not None                  # one grid per object: own epochs or the caller's
        if ragged:
            grid, goff = self._grid_csr
        else:
            grid, goff = np.array(self.new_binning, dtype=np.float64), None

        def make(i):                                         # an empty grid, or no data: the prior on the grid
            g = grid[goff[i]:goff[i + 1]] if ragged else grid
            h, n = hyp[i] if rows else hyp, nug[i] if rows else nug
            if not len(g):
                return np.zeros((0, 0))
            return self.kernel(g, np.asarray(h, dtype=float), nugget=n, **({"flags": self.flags} if self._dim == 2 else {}))

        # the objects written in bulk (global ids, in the order of `batch`)
        split = self._split
        if rows:
            ids = np.nonzero(split.small)[0]
            if split.small_max_n > 64:
                ids = ids[:0]
        else:
            ids = np.arange(self.N_sn)
            if self._devices is not None or self.N_sn == 0 or int(split.sizes.max()) > 64:
                ids = ids[:0]
        # the objects of the grouped calls: every other object with data and a non-empty grid
        m_obj = np.diff(goff) if ragged else np.full(self.N_sn, len(grid), dtype=np.int64)
        grouped = np.ones(self.N_sn, dtype=bool)
        grouped[ids] = False
        grouped &= (split.sizes > 0) & (m_obj > 0)
        gids = np.nonzero(grouped)[0]
        if not len(ids) and not len(gids):
            return _LazyMatrices(self.N_sn, make)
        pos = np.full(self.N_sn, -1, dtype=np.int64)         # object i is the bulk batch's object pos[i] ...
        pos[ids] = np.arange(len(ids))
        gpos = np.full(self.N_sn, -1, dtype=np.int64)        # ... or the grouped call's object gpos[i]
        gpos[gids] = np.arange(len(gids))
        bulk_hyp, bulk_nug = (hyp[ids], nug[ids]) if rows else (hyp, nug)
        bounds = dense.plan_chunks(m_obj[ids] ** 2 * 8)      # chunks of objects with <= 256 MB of matrices
        gout = m_obj[gids] ** 2 * 8                          # ... and <= 2 GB of workspace for the grouped objects
        gbounds = dense.plan_chunks(gout, dense.cov_ws_doubles(split.sizes[gids], m_obj[gids]) * 8)
        # one bulk chunk and one grouped chunk of host matrices alive at a time: reading a batch that interleaves the
        # two kinds in index order builds each chunk once
        bulk_cache, grouped_cache = {}, {}

        def make_bulk(j):
            c = int(np.searchsorted(bounds, j, side="right")) - 1
            if c not in bulk_cache:
                bulk_cache.clear()
                batch = self._small_batch() if rows else self.batch
                if own:
                    g, kw = None, {}
                elif ragged:                                 # the grids of the batch's objects, as one CSR
                    pts, sub = (slice(None), goff) if len(ids) == self.N_sn else split.small_csr(goff)
                    g, kw = grid[pts], {"goff": sub}
                else:
                    g, kw = grid, {}
                mats, info = batch.covariance(bulk_hyp, bulk_nug, g, objects=(bounds[c], bounds[c + 1]), flags=self.flags, **kw)
                if info.any():
                    full = np.zeros(self.N_sn, dtype=info.dtype)
                    full[ids[bounds[c]:bounds[c + 1]]] = info
                    self._raise_if_bad(full)
                bulk_cache[c] = mats
            return bulk_cache[c][j - bounds[c]]

        def make_grouped(j):
            c = int(np.searchsorted(gbounds, j, side="right")) - 1
            if c not in grouped_cache:
                grouped_cache.clear()
                sel = gids[gbounds[c]:gbounds[c + 1]]
                grouped_cache[c] = dense.predictive_covariances(
                    self._x_flat, self._off, self._ye_flat, grid, goff if ragged else None, hyp[sel] if rows else hyp,
                    nug[sel] if rows else nug, self._dim, self.flags, objects=sel)
            mats, info = grouped_cache[c]
            bad = int(info[j - gbounds[c]])
            if bad:                                          # as LargeObject.factor: only this object raises
                raise np.linalg.LinAlgError("%d-th leading minor of the covariance is not positive definite" % bad)
            return mats[j - gbounds[c]]

        def make_any(i):
            if pos[i] >= 0:
                return make_bulk(int(pos[i]))
            if gpos[i] >= 0:
                return make_grouped(int(gpos[i]))
            return make(i)

        return _LazyMatrices(self.N_sn, make_any)


class gaussian_process(Gaussian_process):

    def __init__(self, y, Time, kernel='RBF1D',
                 y_err=None, diff=None, Mean_Y=None,
                 Time_mean=None, substract_mean=False):
        """Run gp for one object (:365-379): y, Time, y_err are wrapped in 1-lists, diff is not (Q14)."""
        if y_err is not None:
            y_err = [y_err]
        Gaussian_process.__init__(self, [y], [Time], kernel=kernel,
                                  y_err=y_err, Mean_Y=Mean_Y, Time_mean=Time_mean,
                                  diff=diff, substract_mean=substract_mean)


class gaussian_process_nobject(Gaussian_process):

    def __init__(self, y, Time, kernel='RBF1D',
                 y_err=None, diff=None, Mean_Y=None,
                 Time_mean=None, substract_mean=False, devices=None):
        """Run gp for n objects (:382-393)."""
        Gaussian_process.__init__(self, y, Time, kernel=kernel,
                                  y_err=y_err, diff=diff, Mean_Y=Mean_Y,
                                  Time_mean=Time_mean, substract_mean=substract_mean, devices=devices)
