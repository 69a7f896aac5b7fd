"""Per-object fits and predictions of objects above CGP_SMALL_MAX_N points: the grouped likelihood entry point
cgp_large_ll_rows_dev (every object of a wave factored by the same launches, each with its own hyperparameter row)
against the single-object path and the oracle, its group invariance, and the facade over batches that mix such
objects with small ones."""
from fractions import Fraction

import numpy as np
import pytest
from scipy.optimize import fmin

from conftest import assert_close
from oracle import gp_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cg():
    import cosmogp_b200
    from cosmogp_b200 import _lib
    _lib.require_device()
    return cosmogp_b200


def _object(rng, n, dim):
    """Seeded object with cond(K) of order 1e3 under _hyp(dim)."""
    if dim == 1:
        x = np.sort(rng.uniform(0, n / 5.0, n))
        y = np.sin(x) + 0.2 * rng.standard_normal(n)
    else:
        s = 3.0 * np.sqrt(n)
        x = rng.uniform(0, s, (n, 2))
        y = np.sin((x[:, 0] - x[:, 1]) / 5) + 0.2 * rng.standard_normal(n)
    return x, y, rng.uniform(0.1, 0.3, n)


def _hyp(dim):
    return [0.8, 1.5] if dim == 1 else [1.1, 4.0, 3.0, 1.0]


def _ws(n):
    from cosmogp_b200 import _lib
    return int(_lib.lib().cgp_large_ll_ws_doubles(int(n)))


class Group:
    """A batch on the device and direct calls of cgp_large_ll_rows_dev on it."""

    def __init__(self, xs, ys, dim, y_err=None, y0=None):
        import torch
        from cosmogp_b200.batch import DeviceBatch, pack_csr
        xf, off = pack_csr(xs, dim)
        self.b = DeviceBatch(xf, pack_csr(ys)[0], off, y0=None if y0 is None else pack_csr(y0)[0],
                             y_err=None if y_err is None else pack_csr(y_err)[0], dim=dim)
        self.dim, self.torch = dim, torch

    def run(self, hyp_rows, order, nug_rows=None, work_doubles=None, nugget=0.0):
        """-> (rc, ll, info) for the objects `order` (host), row k of hyp_rows / nug_rows belonging to order[k]
        (nugget: the shared one, without nug_rows)."""
        from cosmogp_b200 import _lib
        t = self.torch
        dev = self.b.device
        k = len(order)
        order = np.ascontiguousarray(order, dtype=np.int32)
        if work_doubles is None:
            work_doubles = sum(_ws(self.b.off_host[i + 1] - self.b.off_host[i]) for i in order) or 2
        work = t.empty(int(work_doubles), dtype=t.float64, device=dev)
        hr = np.ascontiguousarray(hyp_rows, dtype=np.float64).reshape(max(k, 1), -1)
        nr = None if nug_rows is None else np.ascontiguousarray(nug_rows, dtype=np.float64)
        ll = t.full((max(k, 1),), -1.0, dtype=t.float64, device=dev)
        info = t.full((max(k, 1),), -7, dtype=t.int32, device=dev)
        p = lambda v: None if v is None else v.data_ptr()
        n0 = _lib.lib().cgp_launch_count()
        rc = _lib.lib().cgp_large_ll_rows_dev(self.b.n_obj, _lib.hptr(self.b.off_host), self.dim, p(self.b.x), p(self.b.y),
                                              p(self.b.y0), p(self.b.y_err), _lib.hptr(hr), _lib.hptr(nr), float(nugget), 0.0, 0,
                                              order.ctypes.data, k, p(ll), p(info), p(work), int(work_doubles),
                                              t.cuda.current_stream(dev).cuda_stream)
        self.launches = _lib.lib().cgp_launch_count() - n0
        t.cuda.synchronize()
        return rc, ll.cpu().numpy()[:k], info.cpu().numpy()[:k]


SIZES = (225, 255, 256, 257, 383, 384, 385, 1000, 2000)


def _fused_det_differs(row):
    """Whether lx^2 ly^2 - lxy^2 of a 2D row rounds differently when the first product is fused into the subtraction
    (one rounding, as a device compiler may contract it) than with every operation rounded (the host's cov_from_hyp)."""
    lx2, ly2, lxy2 = row[1] * row[1], row[2] * row[2], row[3] * row[3]
    return float(Fraction(lx2) * Fraction(ly2) - Fraction(lxy2)) != lx2 * ly2 - lxy2


@pytest.mark.parametrize("dim", [1, 2])
@pytest.mark.parametrize("extras", [False, True])
def test_rows_entry_matches_single_object_path(cg, dim, extras):
    """Every size of SIZES in one grouped call against dense.LargeObject.factor (bit for bit) and the oracle (1e-9);
    with extras: y0, y_err and per-object nuggets and hyperparameters, in 2D with rows whose metric determinant rounds
    differently when contracted into one FMA; without: a shared nugget keeps cond(K) near 1e3."""
    from cosmogp_b200.dense import LargeObject
    rng = np.random.default_rng(7 + dim + 10 * extras)
    objs = [_object(rng, n, dim) for n in SIZES]
    xs, ys = [o[0] for o in objs], [o[1] for o in objs]
    ye = [o[2] for o in objs] if extras else None
    y0 = [0.1 * np.cos(np.arange(len(y))) for y in ys] if extras else None
    base = np.array([1.1, 4.3, 3.7, 0.9] if dim == 2 and extras else _hyp(dim))
    hyp = np.array([base * (1.0 + 0.05 * i) for i in range(len(SIZES))]) if extras else np.tile(base, (len(SIZES), 1))
    if dim == 2 and extras:
        assert any(_fused_det_differs(h) for h in hyp)
    nug = 0.02 + 0.01 * np.arange(len(SIZES)) if extras else None
    g = Group(xs, ys, dim, y_err=ye, y0=y0)
    rc, ll, info = g.run(hyp, np.arange(len(SIZES)), nug, nugget=0.2)
    assert rc == 0 and not info.any()
    for i, n in enumerate(SIZES):
        nu = 0.2 if nug is None else nug[i]
        lo = LargeObject(xs[i], ys[i], None if ye is None else ye[i], None if y0 is None else y0[i], dim=dim)
        np.testing.assert_array_equal(ll[i], lo.factor(hyp[i], nu), "n=%d vs LargeObject" % n)
        ref = O.log_likelihood(ys[i], xs[i], hyp[i], nu, None if ye is None else ye[i], None if y0 is None else y0[i],
                               kind="1d" if dim == 1 else "2d")
        assert_close(ll[i], ref, 1e-9, 0.0, "n=%d vs oracle" % n)


def test_rows_entry_group_invariance_bitwise(cg):
    """An object's ll is bit-identical alone, in a group of other sizes, in reversed order and across waves."""
    rng = np.random.default_rng(11)
    sizes = [1000, 300, 1000, 257, 1000, 385, 100, 2000]
    objs = [_object(rng, n, 1) for n in sizes]
    g = Group([o[0] for o in objs], [o[1] for o in objs], 1, y_err=[o[2] for o in objs])
    hyp = np.array([[0.8 + 0.02 * i, 1.5 - 0.03 * i] for i in range(len(sizes))])
    nug = 0.01 * np.arange(len(sizes))
    alone = np.array([g.run(hyp[i:i + 1], [i], nug[i:i + 1])[1][0] for i in range(len(sizes))])
    order = np.arange(len(sizes))
    rc, together, info = g.run(hyp, order, nug)
    assert rc == 0 and not info.any()
    np.testing.assert_array_equal(together, alone)
    rev = order[::-1]
    rc, back, _ = g.run(hyp[rev], rev, nug[rev])
    np.testing.assert_array_equal(back, alone[rev])
    # waves: [1000, 300] [1000, 257] [1000] [385, 100]: boundaries between objects of different n_pad
    w = _ws(1000) + _ws(300)
    assert w < _ws(1000) + _ws(385)
    first = order[:7]
    rc, waves, _ = g.run(hyp[first], first, nug[first], work_doubles=w)
    assert rc == 0
    np.testing.assert_array_equal(waves, alone[first])
    one_wave_launches = Group([o[0] for o in objs[:7]], [o[1] for o in objs[:7]], 1, y_err=[o[2] for o in objs[:7]])
    one_wave_launches.run(hyp[first], first, nug[first])
    assert g.launches > one_wave_launches.launches            # more waves, more launch sequences


def test_rows_entry_failures_stay_local(cg):
    """A non-positive-definite object in the middle gets info != 0 and NaN; its neighbours keep their bits.  A workspace
    below the largest object's need is refused before anything is launched; no active object returns 0."""
    from cosmogp_b200 import _lib
    rng = np.random.default_rng(5)
    sizes = [300, 600, 400]
    objs = [_object(rng, n, 1) for n in sizes]
    xs, ys, ye = [o[0] for o in objs], [o[1] for o in objs], [o[2] for o in objs]
    xs[1] = xs[1].copy(); xs[1][1] = xs[1][0]                 # duplicate epoch, no noise: the second pivot is 0
    ye[1] = np.zeros(sizes[1])
    g = Group(xs, ys, 1, y_err=ye)
    hyp = np.array([[0.8, 1.5], [1.0, 1.5], [0.9, 1.4]])
    rc, ll, info = g.run(hyp, [0, 1, 2])
    assert rc == 0 and info[1] != 0 and np.isnan(ll[1])
    assert info[0] == 0 and info[2] == 0
    _, ll_ok, _ = g.run(hyp[[0, 2]], [0, 2])
    np.testing.assert_array_equal(ll[[0, 2]], ll_ok)
    n0 = _lib.lib().cgp_launch_count()
    rc, ll, info = g.run(hyp, [0, 1, 2], work_doubles=_ws(600) - 2)
    assert rc < 0 and "workspace" in _lib.last_error()
    assert g.launches == 0 and (ll == -1.0).all() and (info == -7).all()
    assert _lib.lib().cgp_launch_count() == n0
    rc, _, _ = g.run(np.zeros((0, 2)), [], work_doubles=2)
    assert rc == 0 and g.launches == 0


def _mixed(rng, dim, n_small=200, large=(225, 300, 480, 1000)):
    sizes = list(rng.integers(5, 225, n_small)) + list(large)
    objs = [_object(rng, int(n), dim) for n in sizes]
    return [o[0] for o in objs], [o[1] for o in objs], [o[2] for o in objs]


def _fit(gp, guess, nugget, optimizer):
    gp.find_hyperparameters_per_object(hyperparameter_guess=guess, nugget=nugget, optimizer=optimizer)
    return (gp.hyperparameters_per_object.copy(), gp.nugget_per_object.copy(), np.array(gp.log_likelihood_per_object),
            gp.fit_iterations.copy(), gp.fit_evaluations.copy())


@pytest.mark.parametrize("dim,nugget", [(1, False), (1, True), (2, False)])
def test_mixed_batch_fits(cg, dim, nugget):
    rng = np.random.default_rng(40 + dim + 3 * nugget)
    xs, ys, ye = _mixed(rng, dim)
    kern = 'RBF1D' if dim == 1 else 'RBF2D'
    guess = _hyp(dim)
    gp = cg.gaussian_process_nobject(ys, xs, y_err=ye, kernel=kern)
    dev = _fit(gp, guess, nugget, 'device')
    host = _fit(gp, guess, nugget, 'host')
    for d, h in zip(dev, host):
        np.testing.assert_array_equal(d, h)
    ns = len(xs) - 4
    alone = _fit(cg.gaussian_process_nobject(ys[:ns], xs[:ns], y_err=ye[:ns], kernel=kern), guess, nugget, 'device')
    for d, a in zip(dev, alone):
        np.testing.assert_array_equal(d[:ns], a)
    if dim == 1 and not nugget:
        for i in (ns, ns + 1):                               # 225 and 300 points against scipy's fmin on the oracle
            ref = np.abs(fmin(lambda h: -O.log_likelihood(ys[i], xs[i], h, 0.0, ye[i]), guess, disp=False))
            assert_close(dev[0][i], ref, 2e-4)
            assert_close(dev[2][i], O.log_likelihood(ys[i], xs[i], ref, 0.0, ye[i]), 1e-7)
        ys_bad = list(ys)
        ys_bad[ns + 2] = np.full(len(ys[ns + 2]), np.nan)     # never positive definite: +inf after maxfun evaluations
        bad = _fit(cg.gaussian_process_nobject(ys_bad, xs, y_err=ye, kernel=kern), guess, nugget, 'device')
        assert np.isinf(bad[2][ns + 2]) and bad[4][ns + 2] >= 400
        keep = np.arange(len(xs)) != ns + 2
        for d, b in zip(dev, bad):
            np.testing.assert_array_equal(d[keep], b[keep])


def test_all_large_batch_c3_scale(cg):
    """Eight 2D objects of 2000 points (per-CCD PSF scale): the fit completes, and every final likelihood is the
    oracle's at the fitted point."""
    rng = np.random.default_rng(3)
    objs = [_object(rng, 2000, 2) for _ in range(8)]
    xs, ys, ye = [o[0] for o in objs], [o[1] for o in objs], [o[2] for o in objs]
    gp = cg.gaussian_process_nobject(ys, xs, y_err=ye, kernel='RBF2D')
    gp.find_hyperparameters_per_object(hyperparameter_guess=_hyp(2))
    assert np.isfinite(gp.log_likelihood_per_object).all()
    for i in range(8):
        ref = O.log_likelihood(ys[i], xs[i], gp.hyperparameters_per_object[i], 0.0, ye[i], kind="2d")
        assert_close(gp.log_likelihood_per_object[i], ref, 1e-9)


@pytest.mark.parametrize("grid", ["own", "shared"])
@pytest.mark.parametrize("template", [False, True])
def test_mixed_batch_predictions(cg, grid, template):
    """Large objects against oracle.predict (1e-9), small ones bit-identical to a batch of the small objects alone;
    build_pull runs on the same batch with the fitted hyperparameters."""
    rng = np.random.default_rng(60 + 2 * template + (grid == "shared"))
    xs, ys, ye = _mixed(rng, 1, n_small=30, large=(225, 400))
    kw = {}
    if template:
        tx = np.linspace(-5, 100, 60)
        kw = dict(Mean_Y=0.3 * np.cos(tx / 7), Time_mean=tx)
    gp = cg.gaussian_process_nobject(ys, xs, y_err=ye, **kw)
    gp.find_hyperparameters_per_object(hyperparameter_guess=_hyp(1))
    new = None if grid == "own" else np.linspace(0, 60, 333)
    gp.get_prediction(new_binning=new, COV='diag', per_object=True)
    ns = len(xs) - 2
    small = cg.gaussian_process_nobject(ys[:ns], xs[:ns], y_err=ye[:ns], **kw)
    small.hyperparameters_per_object = gp.hyperparameters_per_object[:ns]
    small.nugget_per_object = gp.nugget_per_object[:ns]
    small.get_prediction(new_binning=new, COV='diag', per_object=True)
    for i in range(ns):
        np.testing.assert_array_equal(gp.Prediction[i], small.Prediction[i])
        np.testing.assert_array_equal(gp.prediction_variance[i], small.prediction_variance[i])
    from cosmogp_b200 import mean as M
    for i in (ns, ns + 1):
        o0, o1 = gp._off[i], gp._off[i + 1]
        y0 = gp._y0_flat[o0:o1] if template else 0.0
        if grid == "own":
            g, ny0 = xs[i], y0
        else:
            g = new
            ny0 = (M.template_on_grid(new, 1, kw["Mean_Y"], kw["Time_mean"]) + gp._diff_used[i]) if template else 0.0
        m, v = O.predict(ys[i], xs[i], gp.hyperparameters_per_object[i], gp.nugget_per_object[i], g, y_err=ye[i], y0=y0,
                         new_y0=ny0, full_cov=False)
        assert_close(gp.Prediction[i], m, 1e-9, 1e-9, "mean %d" % i)
        assert_close(gp.prediction_variance[i], v, 1e-9, 1e-9, "var %d" % i)
    assert len(gp.Prediction) == len(xs) and gp.as_the_same_time == (grid == "own")
    if grid == "own" and not template:
        bp = cg.build_pull(ys, xs, gp.hyperparameters_per_object, nugget=gp.nugget_per_object, y_err=ye)
        bp.compute_pull(svd_method=False)
        assert np.isfinite(bp.pull).all() and len(bp.pull) == sum(len(y) for y in ys)
