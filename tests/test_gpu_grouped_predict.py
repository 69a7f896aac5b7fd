"""Grouped means and variances of objects on the blocked path (cgp_large_predict_objhyp_dev, dense.predictions): bit for
bit dense.LargeObject.factor + .predict object by object, whatever the waves, the object order, the order list or the
variance passes; failures stay with their object; and through the facade, where every object the blocked path takes
now goes through the grouped call."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SIZES = (225, 255, 256, 257, 383, 384, 385, 1000, 2000, 12, 60)
GRID_SIZES = (0, 1, 7, 300, 1000)


@pytest.fixture(scope="module")
def cg():
    import cosmogp_b200
    from cosmogp_b200 import _lib
    _lib.require_device()
    return cosmogp_b200


def _object(rng, n, dim):
    if dim == 1:
        x = np.sort(rng.uniform(0, max(n, 5) / 5.0, n))
    else:
        x = rng.uniform(0, 3.0 * np.sqrt(max(n, 4)), (n, 2))
    y = np.sin(x if dim == 1 else x[:, 0] / 3) + 0.2 * rng.standard_normal(n)
    return x, y, rng.uniform(0.1, 0.3, n), 0.1 * rng.standard_normal(n)


def _rows(rng, k, dim):
    if dim == 1:
        return np.stack([rng.uniform(0.6, 1.2, k), rng.uniform(1.0, 2.0, k)], axis=1)
    lx, ly = rng.uniform(3.0, 5.0, k), rng.uniform(3.0, 5.0, k)
    return np.stack([rng.uniform(0.8, 1.2, k), lx, ly, rng.uniform(-0.3, 0.3, k) * lx * ly], axis=1)


def _grid(rng, dim, m, hi):
    return np.linspace(-1.0, hi, m) if dim == 1 else rng.uniform(0, hi, (m, 2))


class Direct:
    """A batch on the device and direct calls of cgp_large_predict_objhyp_dev on it."""

    def __init__(self, objs, grids, dim, extras=True):
        """objs: (x, y, y_err, y0) per object; grids: one grid per object (list) or one shared grid (array)."""
        import torch
        from cosmogp_b200.batch import pack_csr
        self.torch, self.dim = torch, dim
        self.dev = torch.device("cuda", torch.cuda.current_device())
        up = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64).reshape(-1)).to(self.dev)
        xf, self.off = pack_csr([o[0] for o in objs], dim)
        self.x, self.y = up(xf), up(pack_csr([o[1] for o in objs], 1)[0])
        self.ye = up(pack_csr([o[2] for o in objs], 1)[0]) if extras else None
        self.y0 = up(pack_csr([o[3] for o in objs], 1)[0]) if extras else None
        if isinstance(grids, list):
            gf, self.goff = pack_csr(grids, dim)
            self.m = np.diff(self.goff)
        else:
            gf, self.goff = grids, None
            self.m = np.full(len(objs), len(grids), dtype=np.int64)
        self.g = up(gf if len(gf) else np.zeros(2))
        self.n = np.diff(self.off)
        self.launches = 0

    def need(self, order, want_var=True, chunk_rows=1 << 20):
        from cosmogp_b200 import dense
        return dense.pred_ws_doubles(self.n[order], np.minimum(self.m[order], chunk_rows) if want_var else 0)

    def run(self, hyp_rows, nug_rows, order, new_y0=None, want_var=True, chunk_rows=1 << 20, work_doubles=None):
        """-> rc, means and variances (lists by list position), info.  new_y0: one array per listed object or None."""
        from cosmogp_b200 import _lib
        t = self.torch
        order = np.ascontiguousarray(order, dtype=np.int32)
        k = len(order)
        m = self.m[order]
        moff = np.zeros(k + 1, dtype=np.int64)
        np.cumsum(m, out=moff[1:])
        if work_doubles is None:
            work_doubles = int(self.need(order, want_var, chunk_rows).sum())
        work = t.empty(max(int(work_doubles), 2), dtype=t.float64, device=self.dev)
        mean = t.full((max(int(moff[-1]), 1),), -3.0, dtype=t.float64, device=self.dev)
        var = t.full((max(int(moff[-1]), 1),), -5.0, dtype=t.float64, device=self.dev) if want_var else None
        ny0 = None if new_y0 is None else t.from_numpy(np.concatenate([np.zeros(0)] + list(new_y0))).to(self.dev)
        info = t.full((max(k, 1),), -7, dtype=t.int32, device=self.dev)
        rows = np.ascontiguousarray(hyp_rows, dtype=np.float64)
        nugs = np.ascontiguousarray(nug_rows, dtype=np.float64)
        p = lambda a: None if a is None else a.data_ptr()
        L = _lib.lib()
        n0 = L.cgp_launch_count()
        rc = L.cgp_large_predict_objhyp_dev(len(self.off) - 1, _lib.hptr(self.off), self.dim, p(self.x), p(self.y),
                                            p(self.y0), p(self.ye), _lib.hptr(rows), _lib.hptr(nugs), 0.0, 0.0, 0,
                                            p(self.g), _lib.hptr(self.goff), 0 if self.goff is not None else int(self.m[0]),
                                            p(ny0), order.ctypes.data, k, _lib.hptr(moff), p(mean), p(var), p(info),
                                            int(chunk_rows), p(work), int(work_doubles),
                                            t.cuda.current_stream(self.dev).cuda_stream)
        self.launches = L.cgp_launch_count() - n0
        t.cuda.synchronize()
        mh = mean.cpu().numpy()
        vh = var.cpu().numpy() if want_var else None
        split = lambda h: [h[moff[j]:moff[j + 1]] for j in range(k)]
        return rc, split(mh), (split(vh) if want_var else None), info.cpu().numpy()[:k]


def _reference(obj, grid, hyp, nug, dim, extras, new_y0, want_var=True):
    """LargeObject.factor + .predict of one object; None when the factorisation fails."""
    from cosmogp_b200.dense import LargeObject
    x, y, ye, y0 = obj
    lo = LargeObject(x, y, ye if extras else None, y0 if extras else None, dim=dim)
    try:
        lo.factor(hyp, nug)
    except np.linalg.LinAlgError:
        return None
    if not len(grid):
        return np.zeros(0), np.zeros(0)
    return lo.predict(grid, new_y0=new_y0, want_var=want_var)


def _case(kind, grid, seed):
    dim = 1 if kind == "1d" else 2
    rng = np.random.default_rng(seed)
    objs = [_object(rng, n, dim) for n in SIZES]
    hi = 120.0 if dim == 1 else 60.0
    if grid == "shared":
        g = _grid(rng, dim, 300, hi)
        grids, arg = [g] * len(SIZES), g
    elif grid == "own":
        grids = [o[0] for o in objs]
        arg = grids
    else:
        grids = [_grid(rng, dim, GRID_SIZES[i % len(GRID_SIZES)], hi) for i in range(len(SIZES))]
        arg = grids
    return dim, rng, objs, grids, arg


@pytest.mark.parametrize("extras", [True, False])
@pytest.mark.parametrize("grid", ["shared", "own", "per_object"])
@pytest.mark.parametrize("kind", ["1d", "2d"])
def test_entry_bitwise_large_object(cg, kind, grid, extras):
    """Every size of SIZES (small ones too: the shared route sends them here) in one call, per-object rows and nuggets,
    bit for bit LargeObject.factor + .predict; with and without y0 / new_y0 / y_err; var NULL gives the same means."""
    dim, rng, objs, grids, arg = _case(kind, grid, 10 * (kind == "2d") + 3 * extras + len(grid))
    d = Direct(objs, arg, dim, extras)
    k = len(SIZES)
    hyp, nug = _rows(rng, k, dim), rng.uniform(0.01, 0.1, k)
    ny0 = [0.1 * rng.standard_normal(len(g)) for g in grids] if extras else None
    rc, mean, var, info = d.run(hyp, nug, np.arange(k), new_y0=ny0)
    assert rc == 0 and not info.any()
    rc, mean_only, none, _ = d.run(hyp, nug, np.arange(k), new_y0=ny0, want_var=False)
    assert rc == 0 and none is None
    for i, n in enumerate(SIZES):
        m_ref, v_ref = _reference(objs[i], grids[i], hyp[i], nug[i], dim, extras, ny0[i] if extras else None)
        np.testing.assert_array_equal(mean[i], m_ref, "mean n=%d" % n)
        np.testing.assert_array_equal(var[i], v_ref, "var n=%d" % n)
        np.testing.assert_array_equal(mean_only[i], m_ref, "mean-only n=%d" % n)


def test_invariance(cg):
    """Reversed and shuffled order lists, a workspace of exactly the largest object's need (every object its own wave)
    and variance passes of 128 rows all give the bits of one call over one wave."""
    rng = np.random.default_rng(101)
    sizes = [600, 300, 1000, 12, 257, 2000, 60, 385]
    objs = [_object(rng, n, 1) for n in sizes]
    grids = [_grid(rng, 1, (7, 300, 1000, 1)[i % 4], 120.0) for i in range(len(sizes))]
    d = Direct(objs, grids, 1)
    k = len(sizes)
    hyp, nug = _rows(rng, k, 1), rng.uniform(0.01, 0.1, k)
    order = np.arange(k)
    rc, m1, v1, info = d.run(hyp, nug, order)
    assert rc == 0 and not info.any()
    one_wave = d.launches
    for perm in (order[::-1], rng.permutation(k)):
        rc, m2, v2, _ = d.run(hyp[perm], nug[perm], perm)
        assert rc == 0
        for j, i in enumerate(perm):
            np.testing.assert_array_equal(m2[j], m1[i])
            np.testing.assert_array_equal(v2[j], v1[i])
    rc, m3, v3, _ = d.run(hyp, nug, order, work_doubles=int(d.need(order).max()))
    assert rc == 0 and d.launches > one_wave
    rc, m4, v4, _ = d.run(hyp, nug, order, chunk_rows=128)
    assert rc == 0
    for i in order:
        for m, v in ((m3, v3), (m4, v4)):
            np.testing.assert_array_equal(m[i], m1[i])
            np.testing.assert_array_equal(v[i], v1[i])


def test_launches_do_not_grow_with_objects(cg):
    """A wave of 16 objects takes as many launches as a wave of 2 of the same sizes."""
    rng = np.random.default_rng(150)
    objs = [_object(rng, n, 1) for n in [500, 300] * 8]
    g = _grid(rng, 1, 200, 100.0)
    d = Direct(objs, g, 1)
    hyp, nug = _rows(rng, 16, 1), np.full(16, 0.05)
    rc, _, _, _ = d.run(hyp[:2], nug[:2], [0, 1])
    few = d.launches
    rc2, _, _, _ = d.run(hyp, nug, np.arange(16))
    assert rc == 0 and rc2 == 0 and d.launches == few


def test_long_grid_in_passes(cg):
    """One 2 000-point object on a 10^5-point grid, variances in passes of 16 384 rows, bit for bit LargeObject.predict
    over the whole grid."""
    rng = np.random.default_rng(160)
    obj = _object(rng, 2000, 1)
    g = _grid(rng, 1, 100000, 400.0)
    d = Direct([obj], g, 1)
    hyp, nug = np.array([[0.9, 1.5]]), np.array([0.04])
    rc, mean, var, info = d.run(hyp, nug, [0], chunk_rows=16384)
    assert rc == 0 and not info.any()
    m_ref, v_ref = _reference(obj, g, hyp[0], nug[0], 1, True, None)
    np.testing.assert_array_equal(mean[0], m_ref)
    np.testing.assert_array_equal(var[0], v_ref)


def test_failures_stay_local(cg):
    """A covariance that is not positive definite: that object's info and NaN rows, the others bit for bit a call
    without it.  An empty grid, M = 1 and n_active = 0; a short workspace returns -2 and launches nothing."""
    from cosmogp_b200 import _lib
    rng = np.random.default_rng(170)
    sizes = [300, 250, 400, 90]
    objs = [_object(rng, n, 1) for n in sizes]
    x = objs[1][0].copy(); x[1] = x[0]
    objs[1] = (x, objs[1][1], np.zeros(250), objs[1][3])
    grids = [_grid(rng, 1, 50, 80.0), _grid(rng, 1, 40, 80.0), np.zeros(0), _grid(rng, 1, 1, 80.0)]
    d = Direct(objs, grids, 1)
    hyp = np.array([[0.8, 1.5], [1.0, 1.5], [0.9, 1.4], [1.1, 1.2]])
    nug = np.array([0.05, 0.0, 0.05, 0.05])
    rc, mean, var, info = d.run(hyp, nug, np.arange(4))
    assert rc == 0 and info[1] != 0 and np.count_nonzero(info) == 1
    assert np.isnan(mean[1]).all() and np.isnan(var[1]).all() and len(mean[1]) == 40
    assert len(mean[2]) == 0 and len(mean[3]) == 1
    assert _reference(objs[1], grids[1], hyp[1], nug[1], 1, True, None) is None
    rc, ok_m, ok_v, _ = d.run(hyp[[0, 2, 3]], nug[[0, 2, 3]], [0, 2, 3])
    for j, i in enumerate((0, 2, 3)):
        np.testing.assert_array_equal(mean[i], ok_m[j])
        np.testing.assert_array_equal(var[i], ok_v[j])
        m_ref, v_ref = _reference(objs[i], grids[i], hyp[i], nug[i], 1, True, None)
        np.testing.assert_array_equal(mean[i], m_ref)
        np.testing.assert_array_equal(var[i], v_ref)
    need = d.need(np.arange(4))
    n0 = _lib.lib().cgp_launch_count()
    rc, mean, var, info = d.run(hyp, nug, np.arange(4), work_doubles=int(need.max()) - 2)
    assert rc == -2 and "workspace" in _lib.last_error()
    assert d.launches == 0 and _lib.lib().cgp_launch_count() == n0
    assert (info == -7).all() and all((v == -3.0).all() for v in mean)
    rc, _, _, _ = d.run(np.zeros((0, 2)), np.zeros(0), [], work_doubles=2)
    assert rc == 0 and d.launches == 0


# ---------------------------------------------------------------------------------------------------------- facade
FACADE_SIZES = [12, 300, 40, 257, 7, 400, 60]


def _template():
    tx = np.linspace(-5, 100, 60)
    return dict(Mean_Y=0.3 * np.cos(tx / 7), Time_mean=tx)


@pytest.mark.parametrize("cov", [True, "diag", False])
@pytest.mark.parametrize("grid", ["own", "shared", "per_object"])
@pytest.mark.parametrize("template", [False, True])
def test_facade_per_object(cg, cov, grid, template):
    """get_prediction(per_object=True) on a mixed batch: the large objects bit for bit LargeObject with their own row,
    the small ones bit for bit a batch of the small ones alone."""
    from cosmogp_b200.dense import LargeObject
    from cosmogp_b200 import mean as M
    rng = np.random.default_rng(200 + 7 * template + len(grid) + (0 if cov is True else 1 if cov else 2))
    xs = [np.sort(rng.uniform(0, n / 5.0, n)) for n in FACADE_SIZES]
    ys = [np.sin(x) + 0.3 + 0.2 * rng.standard_normal(len(x)) for x in xs]
    yes = [rng.uniform(0.1, 0.3, len(x)) for x in xs]
    kw = _template() if template else {}
    k = len(FACADE_SIZES)
    hyp, nug = _rows(rng, k, 1), rng.uniform(0.01, 0.1, k)
    if grid == "own":
        new = None
    elif grid == "shared":
        new = np.linspace(0, 80, 97)
    else:
        new = [np.linspace(0, 60, (5, 120, 33, 0)[i % 4]) for i in range(k)]       # object 3 (257 points): empty
    gp = cg.gaussian_process_nobject(ys, xs, y_err=yes, **kw)
    gp.hyperparameters_per_object, gp.nugget_per_object = hyp.copy(), nug.copy()
    gp.get_prediction(new_binning=new, COV=cov, svd_method=False, per_object=True)
    small = [i for i, n in enumerate(FACADE_SIZES) if n <= 224]
    sub = cg.gaussian_process_nobject([ys[i] for i in small], [xs[i] for i in small], y_err=[yes[i] for i in small], **kw)
    sub.hyperparameters_per_object, sub.nugget_per_object = hyp[small].copy(), nug[small].copy()
    sub.get_prediction(new_binning=[new[i] for i in small] if grid == "per_object" else new, COV=cov, svd_method=False,
                       per_object=True)
    for j, i in enumerate(small):
        np.testing.assert_array_equal(gp.Prediction[i], sub.Prediction[j])
        if cov:
            np.testing.assert_array_equal(gp.prediction_variance[i], sub.prediction_variance[j])
    for i, n in enumerate(FACADE_SIZES):
        if n <= 224:
            continue
        g = xs[i] if new is None else (new[i] if grid == "per_object" else new)
        y0 = gp.y0[i] if template else None
        if not template:
            ny0 = None
        elif new is None:
            ny0 = y0
        else:
            ny0 = (M.template_on_grid(g, 1, kw["Mean_Y"], kw["Time_mean"]) if len(g) else np.zeros(0)) + gp._diff_used[i]
        lo = LargeObject(xs[i], ys[i], yes[i], y0, dim=1)
        lo.factor(hyp[i], nug[i])
        m, v = lo.predict(g, new_y0=ny0, want_var=bool(cov)) if len(g) else (np.zeros(0), np.zeros(0))
        np.testing.assert_array_equal(gp.Prediction[i], m, "object %d" % i)
        if cov:
            np.testing.assert_array_equal(gp.prediction_variance[i], v, "object %d" % i)
        else:
            assert gp.prediction_variance is None


@pytest.mark.parametrize("grid", ["shared", "per_object"])
def test_facade_shared_hyperparameters_2d(cg, grid):
    """Shared hyperparameters with an object above 224 points, in 2D: every object bit for bit LargeObject."""
    from cosmogp_b200.dense import LargeObject
    rng = np.random.default_rng(300 + len(grid))
    sizes = [30, 400, 90, 260]
    xs = [rng.uniform(0, 3.0 * np.sqrt(n), (n, 2)) for n in sizes]
    ys = [np.sin(x[:, 0] / 3) + 0.2 * rng.standard_normal(len(x)) for x in xs]
    yes = [rng.uniform(0.1, 0.3, len(x)) for x in xs]
    gp = cg.gaussian_process_nobject(ys, xs, kernel='RBF2D', y_err=yes)
    hyp = np.array([1.0, 4.0, 3.5, 2.0])
    gp.hyperparameters, gp.nugget = hyp.copy(), 0.03
    grids = [rng.uniform(0, 50, (m, 2)) for m in (10, 200, 1, 64)] if grid == "per_object" else rng.uniform(0, 50, (150, 2))
    gp.get_prediction(new_binning=grids, COV='diag', svd_method=False)
    for i in range(len(sizes)):
        lo = LargeObject(xs[i], ys[i], yes[i], None, dim=2)
        lo.factor(hyp, 0.03)
        m, v = lo.predict(grids[i] if grid == "per_object" else grids)
        np.testing.assert_array_equal(gp.Prediction[i], m)
        np.testing.assert_array_equal(gp.prediction_variance[i], v)


def test_facade_singular_large_object(cg):
    """A large object whose covariance is not positive definite: the shared route raises LargeObject.factor's error
    with svd_method=False and redoes it by the host SVD with svd_method=True; the per-object route raises naming it."""
    rng = np.random.default_rng(400)
    sizes = [300, 20, 260]
    xs = [np.sort(rng.uniform(0, n / 5.0, n)) for n in sizes]
    xs[2] = xs[2].copy(); xs[2][1] = xs[2][0]
    ys = [np.sin(x) for x in xs]
    yes = [rng.uniform(0.1, 0.3, n) for n in sizes]
    yes[2] = np.zeros(sizes[2])
    gp = cg.gaussian_process_nobject(ys, xs, y_err=yes)
    hyp = np.array([1.0, 1.5])
    gp.hyperparameters, gp.nugget = hyp.copy(), 0.0
    grid = np.linspace(0, 50, 40)
    with pytest.raises(np.linalg.LinAlgError, match="-th leading minor of the covariance is not positive definite$"):
        gp.get_prediction(new_binning=grid, COV='diag', svd_method=False)
    with pytest.warns(RuntimeWarning):
        gp.get_prediction(new_binning=grid, COV='diag', svd_method=True)
    with pytest.warns(RuntimeWarning):
        _, m, v = gp._svd_object(2, hyp, 0.0, grid, 0.0, True)
    np.testing.assert_array_equal(gp.Prediction[2], m)
    np.testing.assert_array_equal(gp.prediction_variance[2], v)
    gp.hyperparameters_per_object, gp.nugget_per_object = np.tile(hyp, (3, 1)), np.zeros(3)
    with pytest.raises(np.linalg.LinAlgError, match="object 2 "):
        gp.get_prediction(new_binning=grid, COV='diag', svd_method=True, per_object=True)
