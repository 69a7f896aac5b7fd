"""Per-object predictive covariance matrices: get_prediction(per_object=True, COV=True) and DeviceBatch.covariance with
per-object rows (cgp_covariance_objhyp_dev), against the oracle with each object's own hyperparameters and nugget, across
the facade's 256 MB chunks and the entry's 65 535-object gram launches, on mixed-size batches, and on failures."""
import zlib

import numpy as np
import pytest

from conftest import assert_close
from oracle import gp_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cg():
    import cosmogp_b200
    from cosmogp_b200 import _lib
    _lib.require_device()
    return cosmogp_b200


def _objects(rng, sizes, dim):
    if dim == 1:
        xs = [np.sort(rng.uniform(-10, 40, n)) for n in sizes]
    else:
        xs = [rng.uniform(-50, 50, (n, 2)) for n in sizes]
    ys = [np.sin(x if dim == 1 else x[:, 0] / 10) + 0.2 * rng.standard_normal(len(x)) for x in xs]
    return xs, ys, [rng.uniform(0.1, 0.3, len(x)) for x in xs]


def _rows(rng, n, dim):
    """one row of hyperparameters per object, spread like the outcome of per-object fits"""
    if dim == 1:
        return np.stack([rng.uniform(0.5, 1.5, n), rng.uniform(1.0, 4.0, n)], axis=1)
    lx, ly = rng.uniform(10, 30, n), rng.uniform(10, 30, n)
    return np.stack([rng.uniform(0.5, 1.0, n), lx, ly, rng.uniform(-0.5, 0.5, n) * lx * ly], axis=1)


def _grid(rng, dim, m):
    return np.linspace(-12, 42, m) if dim == 1 else rng.uniform(-50, 50, (m, 2))


def _reference(x, ye, hyp, nug, grid, dim, amp=False):
    """covariance_matrix of one object (Gaussian_process.py:356-361) under its own row"""
    if dim == 1 or not amp:
        return O.predict(np.zeros(len(x)), x, hyp, nug, grid, ye, kind="1d" if dim == 1 else "2d")[1]
    # CGP_AMP_ON_AUTOCOV: sigma^2 on the auto-covariance of the data and of the grid
    k = O.rbf_2d(x, hyp, nugget=nug, y_err=ye, amp_on_autocov=True)
    h = O.rbf_2d(x, hyp, new_x=grid)
    return O.rbf_2d(grid, hyp, nugget=nug, amp_on_autocov=True) - h @ (O.cholesky_inverse(k) @ h.T)


def _gp(cg, xs, ys, yes, dim, hyp, nug, amp=False):
    gp = cg.gaussian_process_nobject(ys, xs, y_err=yes, kernel='RBF1D' if dim == 1 else 'RBF2D')
    if amp:
        from cosmogp_b200 import _lib
        gp.flags = _lib.CGP_AMP_ON_AUTOCOV
    gp.hyperparameters_per_object, gp.nugget_per_object = hyp, nug
    return gp


@pytest.mark.parametrize("n_obj", [40, 400])
@pytest.mark.parametrize("nugget", ["per_object", "shared"])
@pytest.mark.parametrize("grid", ["shared", "own"])
@pytest.mark.parametrize("kind", ["1d", "2d", "2d_amp"])
def test_oracle_parity(cg, kind, grid, nugget, n_obj):
    """Ragged objects of 1..64 points, each matrix against the oracle under the object's own row; fewer objects than
    SMs (several CTAs per object in the factor phase) and more.  Matrices are those of the fit at the call."""
    dim, amp = (1, False) if kind == "1d" else (2, kind == "2d_amp")
    rng = np.random.default_rng(zlib.crc32(("%s %s %s %d" % (kind, grid, nugget, n_obj)).encode()))
    sizes = rng.integers(1, 65, n_obj)
    sizes[:2] = (1, 64)
    xs, ys, yes = _objects(rng, sizes, dim)
    hyp = _rows(rng, n_obj, dim)
    nug = rng.uniform(0.01, 0.1, n_obj) if nugget == "per_object" else np.full(n_obj, 0.05)
    gp = _gp(cg, xs, ys, yes, dim, hyp.copy(), nug.copy(), amp)
    new = None if grid == "own" else _grid(rng, dim, 57)
    gp.get_prediction(new_binning=new, COV=True, svd_method=False, per_object=True)
    gp.hyperparameters_per_object[:] = 9.0                     # later changes do not reach covariance_matrix
    gp.nugget_per_object[:] = 0.5
    assert len(gp.covariance_matrix) == n_obj
    for i in sorted({0, 1, n_obj // 2, n_obj - 1} | set(rng.integers(0, n_obj, 4).tolist())):
        g = xs[i] if grid == "own" else new
        ref = _reference(xs[i], yes[i], hyp[i], nug[i], g, dim, amp)
        assert gp.covariance_matrix[i].shape == (len(g), len(g))
        assert_close(gp.covariance_matrix[i], ref, 1e-9, 1e-11, "object %d" % i)
        assert_close(np.diag(gp.covariance_matrix[i]), gp.prediction_variance[i], 1e-12, 0.0, "diag %d" % i)


def test_fitted_nuggets(cg):
    """Rows and nuggets straight from find_hyperparameters_per_object(nugget=True)."""
    rng = np.random.default_rng(5)
    sizes = rng.integers(8, 65, 60)
    xs, ys, yes = _objects(rng, sizes, 1)
    gp = cg.gaussian_process_nobject(ys, xs, y_err=yes)
    gp.find_hyperparameters_per_object(hyperparameter_guess=[1.0, 3.0], nugget=True)
    grid = np.linspace(-12, 42, 70)
    gp.get_prediction(new_binning=grid, COV=True, svd_method=False, per_object=True)
    for i in (0, 17, 59):
        ref = _reference(xs[i], yes[i], gp.hyperparameters_per_object[i], gp.nugget_per_object[i], grid, 1)
        assert_close(gp.covariance_matrix[i], ref, 1e-9, 1e-11, "object %d" % i)


@pytest.mark.parametrize("grid", ["shared", "own"])
def test_diagonal_is_the_variance(cg, grid):
    """At 2048 objects and more the variance comes from the two-kernel prediction route, the matrices from the
    one-pass kernel's V rows: diag(covariance_matrix[i]) still equals prediction_variance[i]."""
    rng = np.random.default_rng(11 + (grid == "own"))
    n_obj = 3000
    sizes = rng.integers(1, 65, n_obj)
    xs, ys, yes = _objects(rng, sizes, 1)
    gp = _gp(cg, xs, ys, yes, 1, _rows(rng, n_obj, 1), rng.uniform(0.01, 0.1, n_obj))
    gp.get_prediction(new_binning=None if grid == "own" else np.linspace(-12, 42, 90), COV=True, svd_method=False,
                      per_object=True)
    for i in range(0, n_obj, 7):
        assert_close(np.diag(gp.covariance_matrix[i]), gp.prediction_variance[i], 1e-12, 0.0, "object %d" % i)


def test_facade_chunks(cg):
    """8 000 objects on a shared grid of 100 points: 80 kB of matrix each, so the facade's 256 MB chunks end after
    3 355 and 6 710 objects; the objects on either side of both boundaries against the oracle."""
    rng = np.random.default_rng(21)
    n_obj, m = 8000, 100
    sizes = rng.integers(20, 41, n_obj)
    xs, ys, yes = _objects(rng, sizes, 1)
    hyp, nug = _rows(rng, n_obj, 1), rng.uniform(0.01, 0.1, n_obj)
    gp = _gp(cg, xs, ys, yes, 1, hyp, nug)
    grid = np.linspace(-12, 42, m)
    gp.get_prediction(new_binning=grid, COV=True, svd_method=False, per_object=True)
    per_chunk = (256 << 20) // (8 * m * m)
    for i in (0, per_chunk - 1, per_chunk, 2 * per_chunk - 1, 2 * per_chunk, n_obj - 1):
        assert_close(gp.covariance_matrix[i], _reference(xs[i], yes[i], hyp[i], nug[i], grid, 1), 1e-9, 1e-11,
                     "object %d" % i)


def test_gram_launch_chunks(cg):
    """70 000 objects of 5 points on a grid of 3: the entry splits them into gram launches of 65 535 objects, and the
    per-object rows must follow each launch's first object."""
    rng = np.random.default_rng(22)
    n_obj = 70000
    x = np.sort(rng.uniform(0, 10, (n_obj, 5)), axis=1)
    y = np.sin(x) + 0.2 * rng.standard_normal(x.shape)
    ye = rng.uniform(0.1, 0.3, x.shape)
    hyp, nug = _rows(rng, n_obj, 1), rng.uniform(0.01, 0.1, n_obj)
    gp = _gp(cg, x, y, ye, 1, hyp, nug)
    grid = np.array([1.0, 4.5, 9.0])
    gp.get_prediction(new_binning=grid, COV=True, svd_method=False, per_object=True)
    for i in (0, 65534, 65535, 65536, n_obj - 1):
        assert_close(gp.covariance_matrix[i], _reference(x[i], ye[i], hyp[i], nug[i], grid, 1), 1e-9, 1e-11,
                     "object %d" % i)


def _device_batch(xs, ys, yes, dim):
    from cosmogp_b200.batch import DeviceBatch, pack_csr
    xf, off = pack_csr(xs, dim)
    return DeviceBatch(xf, pack_csr(ys, 1)[0], off, y_err=pack_csr(yes, 1)[0], dim=dim)


@pytest.mark.parametrize("dim", [1, 2])
@pytest.mark.parametrize("grid", ["shared", "own"])
def test_invariants(cg, dim, grid):
    """Rows all equal to the shared hyperparameters give the shared writer's matrices (bit for bit in 1D; in 2D the
    device may contract the metric's determinant into an FMA where the host does not); and an object's matrix does
    not depend on the other objects' rows."""
    rng = np.random.default_rng(30 + dim + 2 * (grid == "own"))
    n_obj = 100
    xs, ys, yes = _objects(rng, rng.integers(1, 65, n_obj), dim)
    b = _device_batch(xs, ys, yes, dim)
    g = None if grid == "own" else _grid(rng, dim, 45)
    h = _rows(rng, 1, dim)[0]
    shared, info_s = b.covariance(h, 0.05, g)
    rows, info_r = b.covariance(np.tile(h, (n_obj, 1)), np.full(n_obj, 0.05), g)
    assert not info_s.any() and not info_r.any()
    for i in range(n_obj):
        if dim == 1:
            np.testing.assert_array_equal(rows[i], shared[i])
        else:
            assert_close(rows[i], shared[i], 1e-12, 1e-14, "object %d" % i)
    hyp, nug = _rows(rng, n_obj, dim), rng.uniform(0.01, 0.1, n_obj)
    first, _ = b.covariance(hyp, nug, g)
    k = 37
    other, nug2 = _rows(rng, n_obj, dim), rng.uniform(0.01, 0.1, n_obj)
    other[k], nug2[k] = hyp[k], nug[k]
    second, _ = b.covariance(other, nug2, g)
    np.testing.assert_array_equal(second[k], first[k])
    assert not np.array_equal(second[k + 1], first[k + 1])
    part, _ = b.covariance(hyp, nug, g, objects=(k, k + 5))   # a range of objects takes the rows of that range
    for j in range(5):
        np.testing.assert_array_equal(part[j], first[k + j])


@pytest.mark.parametrize("mid", [False, True])
@pytest.mark.parametrize("grid", ["shared", "own"])
def test_mixed_batch(cg, mid, grid):
    """1D objects of <= 64 and > 224 points (and 65..224 with mid=True) after a per-object fit: every matrix against
    the oracle.  Objects above 224 points, and every object once a small one has more than 64 points, are
    dense.predictive_covariance with the object's row, bit for bit."""
    from cosmogp_b200 import dense
    rng = np.random.default_rng(40 + mid + 2 * (grid == "own"))
    sizes = [12, 64, 230, 5, 40] + ([80, 224] if mid else []) + [300, 33]
    xs = [np.sort(rng.uniform(0, n / 5.0, n)) for n in sizes]
    ys = [np.sin(x) + 0.3 + 0.2 * rng.standard_normal(len(x)) for x in xs]
    yes = [rng.uniform(0.1, 0.3, len(x)) for x in xs]
    gp = cg.gaussian_process_nobject(ys, xs, y_err=yes)
    gp.find_hyperparameters_per_object(hyperparameter_guess=[1.0, 2.0])
    new = None if grid == "own" else np.linspace(0, 60, 97)
    gp.get_prediction(new_binning=new, COV=True, svd_method=False, per_object=True)
    hyp, nug = gp.hyperparameters_per_object, gp.nugget_per_object
    for i, n in enumerate(sizes):
        g = xs[i] if grid == "own" else new
        c = gp.covariance_matrix[i]
        assert_close(c, _reference(xs[i], yes[i], hyp[i], nug[i], g, 1), 1e-9, 1e-11, "object %d" % i)
        assert_close(np.diag(c), gp.prediction_variance[i], 1e-9, 1e-12, "diag %d" % i)
        if n > 224 or mid:
            np.testing.assert_array_equal(c, dense.predictive_covariance(xs[i], yes[i], g, hyp[i], nug[i], 1))


def test_failures(cg):
    """A covariance that is never positive definite raises LinAlgError; through DeviceBatch.covariance only that
    object is flagged and NaN; devices= still refuses per-object predictions."""
    rng = np.random.default_rng(50)
    n_obj = 20
    xs, ys, yes = _objects(rng, rng.integers(5, 40, n_obj), 1)
    hyp, nug = _rows(rng, n_obj, 1), rng.uniform(0.01, 0.1, n_obj)
    bad = hyp.copy()
    bad[7] = (np.nan, 2.0)
    gp = _gp(cg, xs, ys, yes, 1, bad, nug)
    with pytest.raises(np.linalg.LinAlgError):
        gp.get_prediction(new_binning=np.linspace(-12, 42, 30), COV=True, svd_method=False, per_object=True)
    b = _device_batch(xs, ys, yes, 1)
    for g in (np.linspace(-12, 42, 30), None):
        mats, info = b.covariance(bad, nug, g)
        assert info[7] != 0 and np.count_nonzero(info) == 1
        assert np.isnan(mats[7]).all()
        ok, _ = b.covariance(hyp, nug, g)
        for i in range(n_obj):
            if i != 7:
                np.testing.assert_array_equal(mats[i], ok[i])
    gd = cg.gaussian_process_nobject(ys, xs, y_err=yes, devices=[0])
    gd.hyperparameters_per_object, gd.nugget_per_object = hyp, nug
    with pytest.raises(AssertionError):
        gd.get_prediction(new_binning=np.linspace(-12, 42, 30), COV=True, per_object=True)
