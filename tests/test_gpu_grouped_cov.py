"""Grouped predictive covariance matrices of objects above 64 points (cgp_large_covariance_dev,
dense.predictive_covariances): bit for bit a loop of dense.predictive_covariance, whatever the waves, the object order
or the order list; against the oracle; and through the facade, where every such object now takes the grouped call."""
import numpy as np
import pytest

from conftest import assert_close
from oracle import gp_oracle as O

pytestmark = pytest.mark.gpu

SIZES = (1, 63, 64, 65, 128, 129, 224, 225, 256, 257, 600)
GRID_SIZES = (0, 1, 7, 100, 1000)


@pytest.fixture(scope="module")
def cg():
    import cosmogp_b200
    from cosmogp_b200 import _lib
    _lib.require_device()
    return cosmogp_b200


def _object(rng, n, dim):
    """Seeded object with a well-conditioned covariance under _rows(dim)."""
    if dim == 1:
        x = np.sort(rng.uniform(0, max(n, 5) / 5.0, n))
    else:
        s = 3.0 * np.sqrt(max(n, 4))
        x = rng.uniform(0, s, (n, 2))
    return x, rng.uniform(0.1, 0.3, n)


def _rows(rng, k, dim):
    if dim == 1:
        return np.stack([rng.uniform(0.6, 1.2, k), rng.uniform(1.0, 2.0, k)], axis=1)
    lx, ly = rng.uniform(3.0, 5.0, k), rng.uniform(3.0, 5.0, k)
    return np.stack([rng.uniform(0.8, 1.2, k), lx, ly, rng.uniform(-0.3, 0.3, k) * lx * ly], axis=1)


def _grid(rng, dim, m, hi):
    return np.linspace(-1.0, hi, m) if dim == 1 else rng.uniform(0, hi, (m, 2))


def _batch(rng, sizes, dim):
    from cosmogp_b200.batch import pack_csr
    objs = [_object(rng, n, dim) for n in sizes]
    xs, yes = [o[0] for o in objs], [o[1] for o in objs]
    xf, off = pack_csr(xs, dim)
    return xs, yes, xf, off, pack_csr(yes, 1)[0]


def _loop(xs, yes, grids, hyp, nug, dim, flags):
    from cosmogp_b200 import dense
    return [dense.predictive_covariance(xs[i], yes[i], grids[i], hyp[i], nug[i], dim, flags) if len(grids[i])
            else np.zeros((0, 0)) for i in range(len(xs))]


@pytest.mark.parametrize("grid", ["shared", "own", "per_object"])
@pytest.mark.parametrize("rows", ["shared", "per_object"])
@pytest.mark.parametrize("kind", ["1d", "2d", "2d_amp"])
def test_bitwise_loop(cg, kind, rows, grid):
    """Every size of SIZES in one call, bit for bit dense.predictive_covariance object by object: shared rows (one row
    and nugget) or per-object rows and nuggets; a shared grid, the own epochs, or per-object grids of 0..1000 points."""
    from cosmogp_b200 import dense, _lib
    from cosmogp_b200.batch import pack_csr
    dim, flags = (1, 0) if kind == "1d" else (2, _lib.CGP_AMP_ON_AUTOCOV if kind == "2d_amp" else 0)
    rng = np.random.default_rng(["1d", "2d", "2d_amp"].index(kind) * 10 + 3 * (rows == "shared") + len(grid))
    xs, yes, xf, off, yef = _batch(rng, SIZES, dim)
    k = len(SIZES)
    hi = 120.0 if dim == 1 else 75.0
    if rows == "shared":
        h, nu = _rows(rng, 1, dim)[0], 0.05
        hyp, nug = np.tile(h, (k, 1)), np.full(k, nu)
    else:
        hyp, nug = _rows(rng, k, dim), rng.uniform(0.01, 0.1, k)
        h, nu = hyp, nug
    if grid == "shared":
        g = _grid(rng, dim, 97, hi)
        grids, gflat, goff = [g] * k, g, None
    elif grid == "own":
        grids, gflat, goff = xs, xf, off
    else:
        grids = [_grid(rng, dim, GRID_SIZES[i % len(GRID_SIZES)], hi) for i in range(k)]
        gflat, goff = pack_csr(grids, dim)
    mats, info = dense.predictive_covariances(xf, off, yef, gflat, goff, h, nu, dim, flags)
    assert not info.any()
    ref = _loop(xs, yes, grids, hyp, nug, dim, flags)
    for i, n in enumerate(SIZES):
        assert mats[i].shape == ref[i].shape, "n=%d" % n
        np.testing.assert_array_equal(mats[i], ref[i], "n=%d" % n)


class Direct:
    """The batch on the device and direct calls of cgp_large_covariance_dev on it (per-object grids)."""

    def __init__(self, xs, yes, grids, dim):
        import torch
        from cosmogp_b200.batch import pack_csr
        self.torch, self.dim = torch, dim
        xf, self.off = pack_csr(xs, dim)
        gf, self.goff = pack_csr(grids, dim)
        dev = torch.device("cuda", torch.cuda.current_device())
        self.dev = dev
        self.x = torch.from_numpy(np.ascontiguousarray(xf, dtype=np.float64)).to(dev)
        self.ye = torch.from_numpy(pack_csr(yes, 1)[0]).to(dev)
        self.g = torch.from_numpy(np.ascontiguousarray(gf, dtype=np.float64).reshape(-1)).to(dev)
        self.m = np.diff(self.goff)

    def need(self, order):
        from cosmogp_b200 import dense
        return dense.cov_ws_doubles(np.diff(self.off)[order], self.m[order])

    def run(self, hyp_rows, nug_rows, order, work_doubles=None, floor=0.0):
        from cosmogp_b200 import _lib
        t = self.torch
        order = np.ascontiguousarray(order, dtype=np.int32)
        k = len(order)
        m = self.m[order]
        coff = np.zeros(k + 1, dtype=np.int64)
        np.cumsum(m * m, out=coff[1:])
        if work_doubles is None:
            work_doubles = int(self.need(order).sum())
        work = t.empty(int(work_doubles), dtype=t.float64, device=self.dev)
        cov = t.full((max(int(coff[-1]), 1),), -3.0, dtype=t.float64, device=self.dev)
        info = t.full((max(k, 1),), -7, dtype=t.int32, device=self.dev)
        rows = np.ascontiguousarray(hyp_rows, dtype=np.float64)
        nugs = np.ascontiguousarray(nug_rows, dtype=np.float64)
        n0 = _lib.lib().cgp_launch_count()
        rc = _lib.lib().cgp_large_covariance_dev(len(self.off) - 1, _lib.hptr(self.off), self.dim, self.x.data_ptr(),
                                                 self.ye.data_ptr(), _lib.hptr(rows), _lib.hptr(nugs), 0.0, float(floor), 0,
                                                 self.g.data_ptr(), _lib.hptr(self.goff), 0, order.ctypes.data, k,
                                                 cov.data_ptr(), _lib.hptr(coff), info.data_ptr(), work.data_ptr(),
                                                 int(work_doubles), t.cuda.current_stream(self.dev).cuda_stream)
        self.launches = _lib.lib().cgp_launch_count() - n0
        t.cuda.synchronize()
        host = cov.cpu().numpy()
        return rc, [host[coff[j]:coff[j + 1]].reshape(m[j], m[j]) for j in range(k)], info.cpu().numpy()[:k]


def test_waves_and_order(cg):
    """Results do not depend on wave packing, object order or the order list: one wave, waves forced by a small
    workspace, the reversed order, and a subset, all bit for bit."""
    rng = np.random.default_rng(101)
    sizes = [600, 65, 257, 1, 300, 129, 64, 225, 600, 100]
    xs, yes, _, _, _ = _batch(rng, sizes, 1)
    grids = [_grid(rng, 1, (7, 100, 1000, 1)[i % 4], 120.0) for i in range(len(sizes))]
    d = Direct(xs, yes, grids, 1)
    hyp, nug = _rows(rng, len(sizes), 1), rng.uniform(0.01, 0.1, len(sizes))
    order = np.arange(len(sizes))
    rc, one, info = d.run(hyp, nug, order)
    assert rc == 0 and not info.any()
    one_wave = d.launches
    ref = _loop(xs, yes, grids, hyp, nug, 1, 0)
    for i in order:
        np.testing.assert_array_equal(one[i], ref[i])
    small = int(d.need(order).max()) + 1                      # one object per wave at most, for the largest ones
    rc, waves, _ = d.run(hyp, nug, order, work_doubles=small)
    assert rc == 0 and d.launches > one_wave
    rev = order[::-1]
    rc, back, _ = d.run(hyp[rev], nug[rev], rev)
    sub = np.array([8, 3, 5])
    rc2, part, _ = d.run(hyp[sub], nug[sub], sub)
    assert rc == 0 and rc2 == 0
    for i in order:
        np.testing.assert_array_equal(waves[i], one[i])
        np.testing.assert_array_equal(back[len(order) - 1 - i], one[i])
    for j, i in enumerate(sub):
        np.testing.assert_array_equal(part[j], one[i])


@pytest.mark.parametrize("kind", ["1d", "2d", "2d_amp"])
def test_oracle_parity(cg, kind):
    """Against the oracle's covariance_matrix (Gaussian_process.py:356-361) at rtol 1e-9, atol 1e-11."""
    from cosmogp_b200 import dense, _lib
    dim, amp = (1, False) if kind == "1d" else (2, kind == "2d_amp")
    rng = np.random.default_rng(200 + ["1d", "2d", "2d_amp"].index(kind))
    sizes = (65, 200, 300)
    xs, yes, xf, off, yef = _batch(rng, sizes, dim)
    hyp, nug = _rows(rng, len(sizes), dim), rng.uniform(0.01, 0.1, len(sizes))
    g = _grid(rng, dim, 80, 60.0 if dim == 1 else 50.0)
    mats, info = dense.predictive_covariances(xf, off, yef, g, None, hyp, nug, dim,
                                              _lib.CGP_AMP_ON_AUTOCOV if amp else 0)
    assert not info.any()
    for i in range(len(sizes)):
        if dim == 1 or not amp:
            ref = O.predict(np.zeros(len(xs[i])), xs[i], hyp[i], nug[i], g, yes[i], kind="1d" if dim == 1 else "2d")[1]
        else:
            k = O.rbf_2d(xs[i], hyp[i], nugget=nug[i], y_err=yes[i], amp_on_autocov=True)
            h = O.rbf_2d(xs[i], hyp[i], new_x=g)
            ref = O.rbf_2d(g, hyp[i], nugget=nug[i], amp_on_autocov=True) - h @ (O.cholesky_inverse(k) @ h.T)
        assert_close(mats[i], ref, 1e-9, 1e-11, "object %d" % i)


def _facade(cg, rng, sizes, dim=1):
    xs = [np.sort(rng.uniform(0, n / 5.0, n)) for n in sizes]
    ys = [np.sin(x) + 0.2 * rng.standard_normal(len(x)) for x in xs]
    yes = [rng.uniform(0.1, 0.3, len(x)) for x in xs]
    return cg.gaussian_process_nobject(ys, xs, y_err=yes), xs, yes


@pytest.mark.parametrize("per_object", [False, True])
def test_facade_chunks(cg, per_object):
    """Mixed batches whose objects all take the grouped call (an object above 64 points sends every object there under
    shared hyperparameters, every small one with per_object=True): 2 000 000 bytes per matrix on a 500-point grid, so
    the 256 MB chunks end after 134 and 268 objects.  The objects on either side of both boundaries bit for bit
    dense.predictive_covariance; diag(C) against prediction_variance."""
    from cosmogp_b200 import dense
    rng = np.random.default_rng(300 + per_object)
    n_obj, m = 300, 500
    sizes = rng.integers(40, 90, n_obj)
    sizes[5] = 70
    gp, xs, yes = _facade(cg, rng, sizes)
    hyp, nug = _rows(rng, n_obj, 1), rng.uniform(0.01, 0.1, n_obj)
    grid = np.linspace(-1.0, 20.0, m)
    if per_object:
        gp.hyperparameters_per_object, gp.nugget_per_object = hyp.copy(), nug.copy()
    else:
        gp.hyperparameters, gp.nugget = hyp[0].copy(), float(nug[0])
        hyp, nug = np.tile(hyp[0], (n_obj, 1)), np.full(n_obj, nug[0])
    gp.get_prediction(new_binning=grid, COV=True, svd_method=False, per_object=per_object)
    per_chunk = (256 << 20) // (8 * m * m)
    assert per_chunk == 134
    for i in (0, 5, per_chunk - 1, per_chunk, 2 * per_chunk - 1, 2 * per_chunk, n_obj - 1):
        c = gp.covariance_matrix[i]
        np.testing.assert_array_equal(c, dense.predictive_covariance(xs[i], yes[i], grid, hyp[i], nug[i], 1),
                                      "object %d" % i)
        assert_close(np.diag(c), gp.prediction_variance[i], 1e-9, 1e-12, "diag %d" % i)


@pytest.mark.parametrize("grid", ["shared", "own"])
def test_facade_shared_hyp_large(cg, grid):
    """Shared hyperparameters with an object above 224 points: every object through the grouped call, on a shared
    grid and on the own epochs, bit for bit dense.predictive_covariance."""
    from cosmogp_b200 import dense
    rng = np.random.default_rng(310 + (grid == "own"))
    sizes = [70, 300, 20, 150, 5]
    gp, xs, yes = _facade(cg, rng, sizes)
    gp.hyperparameters, gp.nugget = np.array([0.9, 1.4]), 0.03
    g = np.linspace(0, 10, 33)
    gp.get_prediction(new_binning=g if grid == "shared" else None, COV=True, svd_method=False)
    for i in range(len(sizes)):
        gi = g if grid == "shared" else xs[i]
        np.testing.assert_array_equal(gp.covariance_matrix[i],
                                      dense.predictive_covariance(xs[i], yes[i], gi, gp.hyperparameters, 0.03, 1))


def test_not_positive_definite(cg):
    """Duplicate epochs without noise: through the C entry that object's block is NaN with info != 0 and the others
    keep their bits; through the facade only reading that object raises LinAlgError."""
    from cosmogp_b200 import dense
    rng = np.random.default_rng(400)
    sizes = [300, 100, 400, 90]
    xs, yes, _, _, _ = _batch(rng, sizes, 1)
    xs[1] = xs[1].copy(); xs[1][1] = xs[1][0]
    yes[1] = np.zeros(sizes[1])
    grids = [_grid(rng, 1, 50, 80.0)] * len(sizes)
    d = Direct(xs, yes, grids, 1)
    hyp = np.array([[0.8, 1.5], [1.0, 1.5], [0.9, 1.4], [1.1, 1.2]])
    nug = np.array([0.05, 0.0, 0.05, 0.05])
    rc, mats, info = d.run(hyp, nug, np.arange(4))
    assert rc == 0 and info[1] != 0 and np.count_nonzero(info) == 1
    assert np.isnan(mats[1]).all()
    rc, ok, _ = d.run(hyp[[0, 2, 3]], nug[[0, 2, 3]], [0, 2, 3])
    for j, i in enumerate((0, 2, 3)):
        np.testing.assert_array_equal(mats[i], ok[j])
    with pytest.raises(np.linalg.LinAlgError):
        dense.predictive_covariance(xs[1], yes[1], grids[1], hyp[1], 0.0, 1)
    ys = [np.sin(x) for x in xs]
    gp = cg.gaussian_process_nobject(ys, xs, y_err=yes)
    gp.hyperparameters, gp.nugget = np.array([1.0, 1.5]), 0.0
    gp.get_prediction(new_binning=grids[0], COV=True, svd_method=True)      # the SVD redo covers the prediction
    with pytest.raises(np.linalg.LinAlgError):
        gp.covariance_matrix[1]
    for i in (0, 2, 3):
        np.testing.assert_array_equal(gp.covariance_matrix[i],
                                      dense.predictive_covariance(xs[i], yes[i], grids[0], [1.0, 1.5], 0.0, 1))


def test_workspace_error(cg):
    """A workspace below the largest active object's need returns -2 and launches nothing; no active object returns 0."""
    from cosmogp_b200 import _lib
    rng = np.random.default_rng(500)
    sizes = [300, 600, 100]
    xs, yes, _, _, _ = _batch(rng, sizes, 1)
    grids = [_grid(rng, 1, m, 80.0) for m in (10, 200, 1000)]
    d = Direct(xs, yes, grids, 1)
    hyp, nug = _rows(rng, 3, 1), np.full(3, 0.05)
    need = d.need(np.arange(3))
    n0 = _lib.lib().cgp_launch_count()
    rc, mats, info = d.run(hyp, nug, np.arange(3), work_doubles=int(need.max()) - 2)
    assert rc == -2 and "workspace" in _lib.last_error()
    assert d.launches == 0 and _lib.lib().cgp_launch_count() == n0
    assert (info == -7).all() and all((c == -3.0).all() for c in mats)
    rc, _, _ = d.run(np.zeros((0, 2)), np.zeros(0), [], work_doubles=2)
    assert rc == 0 and d.launches == 0


def test_floor_enters_the_data_covariance_only(cg):
    """A floor f adds f^2 to the diagonal of K(x, x) (as y_err^2 does) and never to K(g, g): against the oracle with
    y_err replaced by sqrt(y_err^2 + f^2)."""
    rng = np.random.default_rng(600)
    sizes = [80, 300]
    xs, yes, _, _, _ = _batch(rng, sizes, 1)
    g = _grid(rng, 1, 60, 60.0)
    d = Direct(xs, yes, [g, g], 1)
    hyp, nug, f = _rows(rng, 2, 1), np.array([0.03, 0.07]), 0.3
    rc, mats, info = d.run(hyp, nug, [0, 1], floor=f)
    assert rc == 0 and not info.any()
    for i in range(2):
        ref = O.predict(np.zeros(sizes[i]), xs[i], hyp[i], nug[i], g, np.sqrt(yes[i] ** 2 + f * f), kind="1d")[1]
        assert_close(mats[i], ref, 1e-9, 1e-11, "object %d" % i)


def test_mixed_batch_read_in_order(cg):
    """A per-object batch of objects of <= 64 points (bulk writer) with objects above 224 points (grouped call) in
    between: reading covariance_matrix in index order builds each chunk once -- as many launches as reading every
    small object first and every large one after -- and gives the same matrices."""
    from cosmogp_b200 import _lib
    rng = np.random.default_rng(700)
    sizes = [12, 300, 40, 5, 250, 60, 33, 400, 20, 64]
    gp, xs, yes = _facade(cg, rng, sizes)
    gp.hyperparameters_per_object, gp.nugget_per_object = _rows(rng, len(sizes), 1), rng.uniform(0.01, 0.1, len(sizes))
    grid = np.linspace(-1.0, 60.0, 70)
    L = _lib.lib()

    def read(order):
        gp.get_prediction(new_binning=grid, COV=True, svd_method=False, per_object=True)
        n0 = L.cgp_launch_count()
        mats = {i: gp.covariance_matrix[i] for i in order}
        return L.cgp_launch_count() - n0, mats

    small = [i for i, n in enumerate(sizes) if n <= 64]
    large = [i for i, n in enumerate(sizes) if n > 224]
    in_order, a = read(range(len(sizes)))
    grouped_by_kind, b = read(small + large)
    assert in_order == grouped_by_kind
    for i in range(len(sizes)):
        np.testing.assert_array_equal(a[i], b[i])
