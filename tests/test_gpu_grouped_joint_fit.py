"""Joint (shared-hyperparameter) likelihoods of batches on the blocked path: the grouped entry cgp_large_ll_rows_dev
(host-built covariance functions) against dense.LargeObject.factor bit for bit, its order and wave invariance and local
failures, and the facade's compute_log_likelihood / find_hyperparameters on mixed batches against the loop of
LargeObject.factor they replace."""
import math

import numpy as np
import pytest
from scipy.optimize import fmin

pytestmark = pytest.mark.gpu

SIZES = (0, 1, 7, 60, 128, 129, 224, 225, 257, 1000, 2000)


@pytest.fixture(scope="module")
def cg():
    import cosmogp_b200
    from cosmogp_b200 import _lib
    _lib.require_device()
    return cosmogp_b200


def _object(rng, n, dim):
    """Seeded object with cond(K) of order 1e3 under _hyp(dim) and a nugget of 0.2."""
    if dim == 1:
        x = np.sort(rng.uniform(0, max(n, 1) / 5.0, n))
        y = np.sin(x) + 0.2 * rng.standard_normal(n)
    else:
        s = 3.0 * np.sqrt(max(n, 1))
        x = rng.uniform(0, s, (n, 2))
        y = np.sin((x[:, 0] - x[:, 1]) / 5) + 0.2 * rng.standard_normal(n)
    return x, y, rng.uniform(0.1, 0.3, n)


def _hyp(dim):
    return np.array([0.8, 1.5]) if dim == 1 else np.array([1.1, 4.0, 3.0, 1.0])


def _ws(n):
    from cosmogp_b200 import dense
    return int(dense.ll_ws_doubles(n))


class Group:
    """A DeviceBatch and direct calls of dense.log_likelihoods on it."""

    def __init__(self, xs, ys, dim, y_err=None, y0=None):
        from cosmogp_b200.batch import DeviceBatch, pack_csr
        xf, off = pack_csr(xs, dim)
        self.xs, self.ys, self.ye, self.y0, self.dim = xs, ys, y_err, y0, dim
        self.b = DeviceBatch(xf, pack_csr(ys)[0], off, y0=None if y0 is None else pack_csr(y0)[0],
                             y_err=None if y_err is None else pack_csr(y_err)[0], dim=dim)

    def run(self, hyp, nugget, objects=None, flags=0, work_doubles=None):
        import torch
        from cosmogp_b200 import dense
        work = None
        if work_doubles is not None:
            work = torch.empty(int(work_doubles), dtype=torch.float64, device=self.b.device)
        return dense.log_likelihoods(self.b, objects, hyp, nugget, flags, work)

    def large_object(self, i, flags=0):
        from cosmogp_b200.dense import LargeObject
        pick = lambda v: None if v is None else v[i]
        return LargeObject(self.xs[i], self.ys[i], pick(self.ye), pick(self.y0), dim=self.dim, flags=flags)

    def reference(self, i, hyp, nugget, flags=0):
        """(ll, info) of LargeObject.factor on object i alone; info parsed from its LinAlgError."""
        try:
            return self.large_object(i, flags).factor(hyp, nugget), 0
        except np.linalg.LinAlgError as e:
            return np.nan, int(str(e).split("-th")[0])


def _empty_ll():
    """LargeObject.factor's formula on an object without points, whose padded block is the identity: quad and log det
    are 0.  (LargeObject itself refuses an object without points.)"""
    return -0.5 * (0.0 + 0.0 + 0 * math.log(2.0 * math.pi))


@pytest.mark.parametrize("dim,extras,flags", [(1, False, 0), (1, True, 0), (2, False, 0), (2, True, 0), (2, True, 1)],
                         ids=["1d", "1d-extras", "2d", "2d-extras", "2d-amp"])
def test_entry_matches_large_object(cg, dim, extras, flags):
    """Every size of SIZES in one grouped call, bit for bit LargeObject.factor; with extras: y_err, y0 and per-object
    hyperparameters and nuggets; flags 1: CGP_AMP_ON_AUTOCOV."""
    rng = np.random.default_rng(3 + dim + 10 * extras + 100 * flags)
    objs = [_object(rng, n, dim) for n in SIZES]
    xs, ys = [o[0] for o in objs], [o[1] for o in objs]
    ye = [o[2] for o in objs] if extras else None
    y0 = [0.1 * np.cos(np.arange(len(y))) for y in ys] if extras else None
    k = len(SIZES)
    hyp = np.array([_hyp(dim) * (1.0 + 0.03 * i) for i in range(k)]) if extras else _hyp(dim)
    nug = 0.15 + 0.01 * np.arange(k) if extras else 0.2
    g = Group(xs, ys, dim, y_err=ye, y0=y0)
    ll, info = g.run(hyp, nug, flags=flags)
    assert not info.any()
    for i, n in enumerate(SIZES):
        h = hyp[i] if extras else hyp
        nu = nug[i] if extras else nug
        ref = _empty_ll() if n == 0 else g.large_object(i, flags).factor(h, nu)
        assert ll[i].tobytes() == np.float64(ref).tobytes(), "n=%d: %r vs %r" % (n, ll[i], ref)


def test_order_and_wave_invariance(cg):
    """Reversed order, a subset, and a workspace of the largest need alone (one object per wave) give the same bits."""
    rng = np.random.default_rng(11)
    sizes = [1000, 300, 60, 2000, 257, 129, 1000]
    objs = [_object(rng, n, 2) for n in sizes]
    g = Group([o[0] for o in objs], [o[1] for o in objs], 2, y_err=[o[2] for o in objs])
    hyp = np.array([_hyp(2) * (1.0 + 0.02 * i) for i in range(len(sizes))])
    nug = 0.01 * np.arange(len(sizes))
    ll, info = g.run(hyp, nug)
    assert not info.any()
    rev = np.arange(len(sizes))[::-1]
    back, _ = g.run(hyp[rev], nug[rev], objects=rev)
    np.testing.assert_array_equal(back, ll[rev])
    one, _ = g.run(hyp, nug, work_doubles=_ws(2000))
    np.testing.assert_array_equal(one, ll)
    sub = np.array([5, 0, 3])
    part, _ = g.run(hyp[sub], nug[sub], objects=sub, work_doubles=_ws(2000) + _ws(129))
    np.testing.assert_array_equal(part, ll[sub])
    for i in (1, 3):
        assert ll[i] == g.large_object(i).factor(hyp[i], nug[i])


def test_failures_stay_local(cg):
    """A singular object (duplicate epoch, no noise, unit amplitude) gives NaN and LargeObject's failing pivot; its
    neighbours keep their bits."""
    rng = np.random.default_rng(5)
    sizes = [300, 600, 400, 30]
    objs = [_object(rng, n, 1) for n in sizes]
    xs, ys, ye = [o[0] for o in objs], [o[1] for o in objs], [o[2] for o in objs]
    xs[1] = xs[1].copy(); xs[1][1] = xs[1][0]
    ye[1] = np.zeros(sizes[1])
    g = Group(xs, ys, 1, y_err=ye)
    hyp = np.array([1.0, 1.5])
    ll, info = g.run(hyp, 0.0)
    ref_ll, ref_info = g.reference(1, hyp, 0.0)
    assert ref_info != 0 and info[1] == ref_info and np.isnan(ll[1])
    assert not info[[0, 2, 3]].any()
    ok, _ = g.run(hyp, 0.0, objects=[0, 2, 3])
    np.testing.assert_array_equal(ll[[0, 2, 3]], ok)
    for i in (0, 2, 3):
        assert ll[i] == g.reference(i, hyp, 0.0)[0]


def _mixed(rng, dim, sizes):
    objs = [_object(rng, int(n), dim) for n in sizes]
    return [o[0] for o in objs], [o[1] for o in objs], [o[2] for o in objs]


def _template(dim):
    if dim == 1:
        tx = np.linspace(-5, 100, 60)
        return dict(Mean_Y=0.3 * np.cos(tx / 7), Time_mean=tx)
    g = np.linspace(-5, 140, 9)
    tx = np.array([(a, b) for a in g for b in g])
    return dict(Mean_Y=0.3 * np.cos(tx[:, 0] / 30) * np.sin(tx[:, 1] / 40), Time_mean=tx)


def _nearest_template(old_binning, mean_function, new_binning):
    """Stand-in for mean.interpolate_mean_2d: the template value at the nearest template point.  interpolate_mean_2d
    calls scipy's bisplrep with task=1 as the reference does, which current scipy refuses on every input; what matters
    here is that the facade's y0 reaches the likelihood, not the interpolation."""
    old, new = np.asarray(old_binning, dtype=float), np.asarray(new_binning, dtype=float)
    d = ((new[:, None, :] - old[None, :, :]) ** 2).sum(-1)
    return np.asarray(mean_function, dtype=float)[np.argmin(d, axis=1)]


def _large_objects(gp):
    from cosmogp_b200.dense import LargeObject
    return [LargeObject(*gp._object_slices(i), dim=gp._dim, flags=gp.flags) for i in range(gp.N_sn)]


def _loop(gp, objs, hyp, nugget):
    """The route the facade took before: LargeObject.factor(hyp, nugget) of every object, the host SVD redo of an
    object whose factorisation fails, and the sum left to right."""
    lls = np.zeros(len(objs))
    for i, o in enumerate(objs):
        try:
            lls[i] = o.factor(hyp, nugget)
        except np.linalg.LinAlgError:
            lls[i] = gp._svd_object(i, hyp, nugget)[0]
    return lls, float(np.add.accumulate(lls)[-1])


@pytest.mark.parametrize("dim", [1, 2])
def test_facade_mixed_batch(cg, monkeypatch, dim):
    """compute_log_likelihood on a batch of small objects and a few large ones, with a mean template and y_err: every
    per-object value and the total bit for bit the LargeObject loop, at two hyperparameter points (the kept workspace)."""
    from cosmogp_b200 import mean as M
    monkeypatch.setattr(M, "interpolate_mean_2d", _nearest_template)
    rng = np.random.default_rng(20 + dim)
    sizes = list(rng.integers(5, 225, 40)) + [225, 600, 300]
    xs, ys, ye = _mixed(rng, dim, sizes)
    gp = cg.gaussian_process_nobject(ys, xs, y_err=ye, kernel='RBF1D' if dim == 1 else 'RBF2D', **_template(dim))
    assert gp._y0_flat is not None and gp._any_large
    objs = _large_objects(gp)
    for scale in (1.0, 1.3):
        hyp = _hyp(dim) * scale
        gp.nugget = 0.05 * scale
        gp.compute_log_likelihood(hyp, svd_method=False)
        per, total = _loop(gp, objs, hyp, 0.05 * scale)
        np.testing.assert_array_equal(gp.log_likelihood_per_object, per)
        assert gp.log_likelihood[0] == total


@pytest.mark.parametrize("dim,nugget", [(1, False), (1, True), (2, False), (2, True)])
def test_find_hyperparameters_matches_the_loop(cg, dim, nugget):
    """The joint fit of a small mixed batch ends where scipy's fmin ends over the LargeObject loop's objective."""
    rng = np.random.default_rng(30 + dim + 2 * nugget)
    xs, ys, ye = _mixed(rng, dim, [20, 50, 8, 230])
    kern = 'RBF1D' if dim == 1 else 'RBF2D'
    gp = cg.gaussian_process_nobject(ys, xs, y_err=ye, kernel=kern)
    start = np.array(gp.hyperparameters, dtype=float)
    gp.find_hyperparameters(nugget=nugget)
    ref = cg.gaussian_process_nobject(ys, xs, y_err=ye, kernel=kern)
    nh = len(start)
    objs = _large_objects(ref)

    def objective(h):
        return -_loop(ref, objs, h[:nh], h[nh] if nugget else 0.0)[1]

    x = fmin(objective, list(start) + ([1.0] if nugget else []), disp=False)
    np.testing.assert_array_equal(gp.hyperparameters, np.sqrt(x[:nh] ** 2))
    assert gp.nugget == (np.sqrt(x[nh] ** 2) if nugget else 0.0)


def test_singular_2d_object(cg):
    """A 2D object with a duplicate star and no noise in a batch with a large object: svd_method=True redoes it by the
    host SVD (bit for bit _svd_object), svd_method=False raises the message of the per-object loop."""
    rng = np.random.default_rng(40)
    xs, ys, ye = _mixed(rng, 2, [30, 12, 300])
    xs[1] = xs[1].copy(); xs[1][1] = xs[1][0]
    ye[1] = np.zeros(len(ye[1]))
    gp = cg.gaussian_process_nobject(ys, xs, y_err=ye, kernel='RBF2D')
    hyp = np.array([1.0, 4.0, 3.0, 1.0])
    with pytest.raises(np.linalg.LinAlgError) as e:
        gp.compute_log_likelihood(hyp, svd_method=False)
    assert str(e.value) == ("1-th leading minor of the covariance of object 1 is not positive definite "
                            "(1 object(s) affected)")
    with pytest.warns(RuntimeWarning):
        gp.compute_log_likelihood(hyp, svd_method=True)
    with pytest.warns(RuntimeWarning):
        ll_svd = gp._svd_object(1, hyp, 0.0)[0]
    assert gp.log_likelihood_per_object[1] == ll_svd
    with pytest.warns(RuntimeWarning):
        per, total = _loop(gp, _large_objects(gp), hyp, 0.0)
    np.testing.assert_array_equal(gp.log_likelihood_per_object, per)
    assert gp.log_likelihood[0] == total


def test_bounded_memory(cg, monkeypatch):
    """With the workspace budget lowered below the batch's sum of n_pad^2 factors, compute_log_likelihood allocates no
    more than the batch upload and one capped workspace, and still gives the loop's values."""
    import torch
    from cosmogp_b200 import dense
    rng = np.random.default_rng(50)
    sizes = [1000] * 6 + [60] * 50
    xs, ys, ye = _mixed(rng, 2, sizes)
    cap = _ws(1000) * 8
    monkeypatch.setattr(dense, "LL_WS_BYTES", cap)
    factors = sum(_ws(n) for n in sizes) * 8
    assert factors > 4 * cap
    gp = cg.gaussian_process_nobject(ys, xs, y_err=ye, kernel='RBF2D')
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    gp.compute_log_likelihood(_hyp(2), svd_method=False)
    torch.cuda.synchronize()
    upload = 8 * 4 * sum(sizes) + 8 * (len(sizes) + 1) + 4 * len(sizes)      # x (2 per point), y, y_err; off; info
    peak = torch.cuda.max_memory_allocated() - base
    assert peak <= upload + cap + (1 << 20), (peak, upload, cap)
    per, total = _loop(gp, _large_objects(gp), _hyp(2), 0.0)
    np.testing.assert_array_equal(gp.log_likelihood_per_object, per)
    assert gp.log_likelihood[0] == total
