"""Pull and residual of the GP interpolation: drop-in for cosmogp/pull.py build_pull.

The reference refits the GP N times per object on N-1 points (pull.py:66-90, O(N^4));
here one factorisation per object gives every leave-one-out prediction and variance in
closed form from K^-1 (SURVEY.md section 8 row a8), all objects in one launch.  The objects batch.SizeSplit calls
large are factorised in HBM in the same call, with no size limit: several of them in one grouped call
(dense.loo_grouped), a single one through dense.LargeLoo.
"""
import numpy as np

from . import _lib
from . import mean as _mean
from .batch import DeviceBatch, RaggedView, SizeSplit, pack_csr


class build_pull:

    def __init__(self, y, x, hyperparameters, nugget=0.,
                 y_err=None, y_mean=None, x_axis_mean=None,
                 kernel='RBF1D', devices=None, gather_over_nvlink=False):
        """Same arguments and attributes as cosmogp/pull.py:10-40.  `hyperparameters` (and `nugget`) may
        also be per-object arrays of shape (n_object, n_hyp) / (n_object,): each object is then
        pulled with its own fit, as in the reference's per-object notebook loop.
        devices ('all', an int or a list of device ids): the objects are sharded over those GPUs of the box inside
        this process (cosmogp_b200.multi.ShardedBatch; shared hyperparameters); gather_over_nvlink=True collects
        the per-object outputs on GPU 0 with NCCL before they leave the box's GPUs (False: every GPU's own PCIe link)."""
        self._devices, self._gather = devices, bool(gather_over_nvlink)
        self.y = y
        self.x = x
        self.hyperparameters = hyperparameters

        self.y_err = y_err
        self.y_mean = y_mean
        self.x_axis_mean = x_axis_mean

        self.kernel = kernel
        self.nugget = nugget

        self.n_object = len(y)

        # results stay on the device until somebody reads them: one entry per compute_pull call
        # (the reference's lists grow with every call); see the properties below
        self._results = []
        self._host = {}

        self.pull_average = None
        self.pull_std = None
        self.flags = 0

    def compute_pull(self, diff=None, svd_method=True, substract_mean=False):
        """Pulls and residuals (pull.py:43-102).  Mean handling, per object sn:
          no y_mean, substract_mean False : plain leave-one-out of y              (mode A)
          y_mean, diff None               : offset re-estimated on the kept points (mode B)
          y_mean, diff given              : fixed offset diff[sn]                  (mode C)
          no y_mean, substract_mean True  : the mean of the FIRST object becomes the
                                            template for all (pull.py:71-73, quirk Q8)  (mode D)
        pred_var = |cov_tt| and the pull denominator counts nugget^2 twice (pull.py:90-93)."""
        assert self.kernel in ['RBF1D', 'RBF2D'], '%s is not in implemented kernel' % (self.kernel)
        dim = 1 if self.kernel == 'RBF1D' else 2
        x_flat, off = pack_csr(self.x, dim)
        y_flat, _ = pack_csr(self.y, 1)
        ye_flat = pack_csr(self.y_err, 1)[0] if self.y_err is not None else None

        if self.y_mean is None and substract_mean and self.n_object:
            self.y_mean = np.ones_like(self.y[0]) * np.mean(self.y[0])
            self.x_axis_mean = self.x[0]

        template = None
        mode = _lib.CGP_LOO_PLAIN
        if self.y_mean is not None:
            template = (_mean.interpolate_mean_1d if dim == 1 else _mean.interpolate_mean_2d)(
                self.x_axis_mean, self.y_mean, x_flat)
            if diff is None:
                mode = _lib.CGP_LOO_RECENTER
            else:
                template = template + np.repeat(np.asarray(diff, dtype=float), np.diff(off))

        if self._devices is not None:
            from .multi import ShardedBatch
            assert np.ndim(self.hyperparameters) == 1, "with devices=... the hyperparameters are shared by all objects"
            sb = ShardedBatch(x_flat, y_flat, off, y0=template, y_err=ye_flat, dim=dim, devices=self._devices)
            pred, pvar, pull, resid, info, mom = sb.loo(self.hyperparameters, self.nugget, mode=mode, flags=self.flags,
                                                        gather=self._gather)
            self.shard_ranges = sb.ranges
            sb.close()
            bad = np.nonzero(info)[0]
            if len(bad):
                raise np.linalg.LinAlgError("covariance of object %d is not positive definite" % int(bad[0]))
            self._results.append({"batch": None, "off": off, "pull": pull, "residual": resid, "prediction": pred,
                                  "prediction_variance": pvar, "sums": mom, "n": len(pull)})
        else:
            # one upload; the shared-memory kernel runs once per run of consecutive small objects, in place, with their
            # own largest size as max_n; the large objects read and write their slices of the same arrays
            split = SizeSplit(off)
            batch = DeviceBatch(x_flat, y_flat, off, y0=template, y_err=ye_flat, dim=dim, max_n=split.small_max_n)
            hyp, nug = self.hyperparameters, self.nugget
            outs = batch.loo_dev(hyp, nug, mode=mode, flags=self.flags, ranges=split.runs)
            if len(split.large) == 1:
                # one large object alone: LargeLoo keeps large_potrf's look-ahead side stream, which the grouped
                # factorisation does not use (DESIGN §9: 187 against 212 ms at N = 20 000)
                from .dense import LargeLoo
                i = int(split.large[0])
                p0, p1 = int(off[i]), int(off[i + 1])
                x, y, m, e = (None if t is None else t[p0:p1] for t in (batch.x, batch.y, batch.y0, batch.y_err))
                LargeLoo(p1 - p0, dim, flags=self.flags).run(x, y, m, e, np.asarray(hyp)[i] if np.ndim(hyp) == 2 else hyp,
                                                             np.asarray(nug)[i] if np.ndim(nug) == 1 else nug, mode,
                                                             outs[4][i:i + 1], [o[p0:p1] for o in outs[:4]])
            elif len(split.large):
                from .dense import loo_grouped
                large = split.large
                loo_grouped(batch, large, np.asarray(hyp)[large] if np.ndim(hyp) == 2 else hyp,
                            np.asarray(nug)[large] if np.ndim(nug) == 1 else nug, mode, outs, flags=self.flags)
            pred, pvar, pull, resid = outs[:4]
            info = batch._down(outs[4])            # every object's status, checked once after everything is launched
            bad = np.nonzero(info)[0]
            if len(bad):
                raise np.linalg.LinAlgError("covariance of object %d is not positive definite" % int(bad[0]))
            self._results.append({"batch": batch, "off": off, "pull": pull, "residual": resid, "prediction": pred,
                                  "prediction_variance": pvar, "n": int(pull.numel())})
        self._host = {}

        # scipy.stats.norm.fit (pull.py:102) = sample mean and population standard deviation, over every pull
        # computed so far; reduced on the device (two passes: the mean, then the spread about it)
        def moments(r, center):
            """(sum (v - c), sum (v - c)^2) of one call's pulls: reduced on the device, or from the sums the GPUs
            of a sharded call already reduced"""
            if r["batch"] is not None:
                return r["batch"].moments(r["pull"], center)
            s1, s2 = r["sums"]
            return s1 - r["n"] * center, s2 - 2.0 * center * s1 + r["n"] * center * center

        n_tot = sum(r["n"] for r in self._results)
        if n_tot:
            total = sum(moments(r, 0.0)[0] for r in self._results)
            self.pull_average = total / n_tot
            parts = [moments(r, self.pull_average) for r in self._results]
            self.pull_average += sum(p[0] for p in parts) / n_tot          # second-pass correction of the mean
            self.pull_std = float(np.sqrt(sum(p[1] for p in parts) / n_tot
                                          - (sum(p[0] for p in parts) / n_tot) ** 2))
        else:
            self.pull_average = self.pull_std = float("nan")

    # ---- results, brought to the host when read (10^6 x 40 pulls are 320 MB per array)
    def _flat(self, name):
        if name not in self._host:
            parts = [r[name] if r["batch"] is None else r["batch"]._down(r[name]) for r in self._results]
            self._host[name] = parts[0] if len(parts) == 1 else (np.concatenate(parts) if parts else np.zeros(0))
        return self._host[name]

    def _offsets(self):
        off = np.zeros(1, dtype=np.int64)
        for r in self._results:
            off = np.concatenate([off, off[-1] + r["off"][1:]])
        return off

    @property
    def pull(self):
        """flat array of all pulls, grows with every compute_pull call like the reference list"""
        return self._flat("pull")

    @property
    def residual(self):
        return self._flat("residual")

    @property
    def _pull(self):
        """per object, list-like (views, no 10^6-element list)"""
        return RaggedView(self._flat("pull"), self._offsets())

    @property
    def prediction(self):
        return RaggedView(self._flat("prediction"), self._offsets())

    @property
    def prediction_variance(self):
        """|cov_tt| of the most recent compute_pull call"""
        if not self._results:
            return None
        r = self._results[-1]
        return r["prediction_variance"] if r["batch"] is None else r["batch"]._down(r["prediction_variance"])
