"""Per-object prediction grids: get_prediction(new_binning=[one grid per object]).  Every route -- shared and per-object
hyperparameters, COV=False / 'diag' / True, objects above 224 points, the host SVD redo -- against the oracle or bit
for bit against the route it generalises (own epochs, a shared grid, dense.LargeObject); long grids spread over several
CTAs per object (the work table of the prediction entries) bit-identical to one CTA per object (CGP_GRID_PARTS=0)."""
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

from conftest import assert_close
from oracle import gp_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu

HYP = {1: np.array([0.8, 2.0]), 2: np.array([0.8, 20.0, 25.0, 30.0])}
NUG = 0.05
GRID_SIZES = (0, 1, 7, 100, 1000)


@pytest.fixture(scope="module")
def cg():
    import cosmogp_b200
    from cosmogp_b200 import _lib
    _lib.require_device()
    return cosmogp_b200


def _seed(*args):
    return np.random.default_rng(zlib.crc32(repr(args).encode()))


def _objects(rng, sizes, dim):
    if dim == 1:
        xs = [np.sort(rng.uniform(-10, 40, n)) for n in sizes]
    else:
        xs = [rng.uniform(-50, 50, (n, 2)) for n in sizes]
    ys = [np.sin(x if dim == 1 else x[:, 0] / 10) + 0.3 + 0.2 * rng.standard_normal(len(x)) for x in xs]
    return xs, ys, [rng.uniform(0.1, 0.3, len(x)) for x in xs]


def _grid(rng, dim, m):
    """non-uniform: a uniform 1D grid would take the recurrence kernel on the shared-grid side of the identities"""
    return np.sort(rng.uniform(-12, 42, m)) if dim == 1 else rng.uniform(-55, 55, (m, 2))


def _template(dim):
    assert dim == 1
    tx = np.linspace(-20, 60, 50)
    return dict(Mean_Y=0.3 * np.cos(tx / 7), Time_mean=tx)


def _rows(rng, n, dim):
    if dim == 1:
        return np.stack([rng.uniform(0.5, 1.5, n), rng.uniform(1.0, 4.0, n)], axis=1)
    lx, ly = rng.uniform(10, 30, n), rng.uniform(10, 30, n)
    return np.stack([rng.uniform(0.5, 1.0, n), lx, ly, rng.uniform(-0.5, 0.5, n) * lx * ly], axis=1)


def _oracle(x, y, ye, hyp, nug, g, dim, y0, ny0, full):
    """(mean, variance, covariance) of one object on grid g (Gaussian_process.py:332-361)"""
    kind = "1d" if dim == 1 else "2d"
    kern = O.rbf_1d if dim == 1 else O.rbf_2d
    if len(x) == 0:                                   # no data: the prior
        cov = kern(g, hyp, nugget=nug)
        return ny0 + np.zeros(len(g)), np.diag(cov).copy(), cov
    mean, cov = O.predict(y, x, hyp, nug, g, ye, y0=y0, new_y0=ny0, kind=kind, full_cov=True)
    return mean, np.diag(cov).copy(), cov


def _check_against_oracle(gp, xs, ys, yes, grids, dim, hyp_of, nug_of, cov, template):
    from cosmogp_b200 import mean as M
    assert gp.as_the_same_time is False and gp.new_binning is grids
    assert len(gp.Prediction) == len(xs)
    for i, g in enumerate(grids):
        assert gp.Prediction[i].shape == (len(g),)
        if template:
            d = gp._diff_used[i]
            y0 = M.template_on_grid(xs[i], dim, template["Mean_Y"], template["Time_mean"]) + d if len(xs[i]) else 0.0
            ny0 = M.template_on_grid(g, dim, template["Mean_Y"], template["Time_mean"]) + d if len(g) else np.zeros(0)
            np.testing.assert_array_equal(gp.warning_pf[i], ny0)
        else:
            y0, ny0 = 0.0, 0.0
        if len(g) == 0:
            if cov is not False:
                assert gp.prediction_variance[i].shape == (0,)
            if cov is True:
                assert gp.covariance_matrix[i].shape == (0, 0)
            continue
        m, v, c = _oracle(xs[i], ys[i], yes[i], hyp_of(i), nug_of(i), g, dim, y0, ny0, cov is True)
        assert_close(gp.Prediction[i], m, 1e-9, 1e-11, "mean %d" % i)
        if cov is False:
            assert gp.prediction_variance is None
            continue
        assert_close(gp.prediction_variance[i], v, 1e-9, 1e-11, "variance %d" % i)
        if cov is True:
            assert_close(gp.covariance_matrix[i], c, 1e-9, 1e-11, "covariance %d" % i)
    if not template:
        assert gp.warning_pf is None


SIZE_SETS = {"le64": (1, 7, 0, 30, 64, 12, 50), "le224": (1, 7, 0, 30, 64, 100, 224, 150)}


@gpu
@pytest.mark.parametrize("cov", [False, "diag", True])
@pytest.mark.parametrize("sizes", sorted(SIZE_SETS))
@pytest.mark.parametrize("dim,template", [(1, False), (1, True), (2, False)])
def test_oracle_parity(cg, dim, template, sizes, cov):
    """Objects of 1..224 points and an empty one, on grids of 0, 1, 7, 100 and 1 000 points, shared hyperparameters.
    The template runs in 1D: the reference fits a 2D template with bisplrep(task=1), which scipy refuses on a first
    call."""
    rng = _seed("parity", dim, sizes, template, cov)
    sz = SIZE_SETS[sizes]
    xs, ys, yes = _objects(rng, sz, dim)
    grids = [_grid(rng, dim, GRID_SIZES[i % len(GRID_SIZES)]) for i in range(len(sz))]
    tk = _template(dim) if template else None
    kw = dict(tk, diff=list(rng.uniform(-0.2, 0.2, len(sz)))) if template else {}
    gp = cg.gaussian_process_nobject(ys, xs, y_err=yes, kernel="RBF1D" if dim == 1 else "RBF2D", **kw)
    gp.hyperparameters, gp.nugget = HYP[dim].copy(), NUG
    gp.get_prediction(new_binning=grids, COV=cov, svd_method=False)
    _check_against_oracle(gp, xs, ys, yes, grids, dim, lambda i: HYP[dim], lambda i: NUG, cov, tk)


@gpu
@pytest.mark.parametrize("cov", ["diag", True])
@pytest.mark.parametrize("sizes", sorted(SIZE_SETS))
@pytest.mark.parametrize("dim", [1, 2])
def test_per_object_rows(cg, dim, sizes, cov):
    """per_object=True: each object with its own row of hyperparameters and its own nugget."""
    rng = _seed("rows", dim, sizes, cov)
    sz = SIZE_SETS[sizes]
    xs, ys, yes = _objects(rng, sz, dim)
    grids = [_grid(rng, dim, GRID_SIZES[(i + 2) % len(GRID_SIZES)]) for i in range(len(sz))]
    hyp, nug = _rows(rng, len(sz), dim), rng.uniform(0.01, 0.1, len(sz))
    gp = cg.gaussian_process_nobject(ys, xs, y_err=yes, kernel="RBF1D" if dim == 1 else "RBF2D")
    gp.hyperparameters_per_object, gp.nugget_per_object = hyp.copy(), nug.copy()
    gp.get_prediction(new_binning=grids, COV=cov, svd_method=False, per_object=True)
    _check_against_oracle(gp, xs, ys, yes, grids, dim, lambda i: hyp[i], lambda i: nug[i], cov, None)


@gpu
@pytest.mark.parametrize("form", ["list", "ndarray"])
@pytest.mark.parametrize("per_object", [False, True])
def test_grids_equal_to_time(cg, per_object, form):
    """Grids equal to Time give exactly what new_binning=None gives: mean, variance, warning_pf, covariance_matrix."""
    rng = _seed("time", per_object, form)
    n_obj, dim = 40, 1
    if form == "list":
        xs, ys, yes = _objects(rng, rng.integers(1, 65, n_obj), dim)
    else:                                            # equal-length objects as (B, N) arrays
        xs = np.sort(rng.uniform(-10, 40, (n_obj, 30)), axis=1)
        ys, yes = np.sin(xs) + 0.2 * rng.standard_normal(xs.shape), rng.uniform(0.1, 0.3, xs.shape)
    outs = []
    for new in (None, xs):
        gp = cg.gaussian_process_nobject(ys, xs, y_err=yes, **_template(dim))
        gp.hyperparameters, gp.nugget = HYP[dim].copy(), NUG
        gp.hyperparameters_per_object, gp.nugget_per_object = _rows(_seed("r"), n_obj, dim), np.full(n_obj, 0.04)
        gp.get_prediction(new_binning=new, COV=True, svd_method=False, per_object=per_object)
        outs.append(gp)
    own, per = outs
    np.testing.assert_array_equal(per.Prediction.flat, own.Prediction.flat)
    np.testing.assert_array_equal(per.prediction_variance.flat, own.prediction_variance.flat)
    np.testing.assert_array_equal(per.warning_pf.flat, np.asarray(own.warning_pf))
    for i in range(n_obj):
        np.testing.assert_array_equal(per.covariance_matrix[i], own.covariance_matrix[i])


@gpu
@pytest.mark.parametrize("n_obj", [50, 3000])
@pytest.mark.parametrize("dim", [1, 2])
def test_grids_equal_to_a_shared_grid(cg, dim, n_obj):
    """Every grid equal to one non-uniform grid G gives exactly what new_binning=G gives; below 296 objects the shared
    grid is spread by `split`, the per-object grids by the work table; from 2048 objects both take the two-kernel route."""
    rng = _seed("shared", dim, n_obj)
    xs, ys, yes = _objects(rng, rng.integers(1, 65, n_obj), dim)
    G = _grid(rng, dim, 300 if n_obj < 296 else 40)
    outs = []
    for new in (G, [G] * n_obj):
        gp = cg.gaussian_process_nobject(ys, xs, y_err=yes, kernel="RBF1D" if dim == 1 else "RBF2D")
        gp.hyperparameters, gp.nugget = HYP[dim].copy(), NUG
        gp.get_prediction(new_binning=new, COV=True, svd_method=False)
        outs.append(gp)
    shared, per = outs
    assert per.as_the_same_time is False and len(per.Prediction) == n_obj
    np.testing.assert_array_equal(per.Prediction.flat, shared.Prediction.flat)
    np.testing.assert_array_equal(per.prediction_variance.flat, shared.prediction_variance.flat)
    for i in sorted({0, 1, n_obj // 2, n_obj - 1}):
        np.testing.assert_array_equal(per.covariance_matrix[i], shared.covariance_matrix[i])


MIXED = (12, 225, 40, 7, 400, 60)
MIXED_GRIDS = (50, 300, 7, 0, 120, 1000)


@gpu
@pytest.mark.parametrize("template", [False, True])
def test_mixed_sizes_shared_hyperparameters(cg, template):
    """With an object above 224 points every object goes through its own dense.LargeObject: bit for bit equal to
    LargeObject(...).predict(grid_i)."""
    from cosmogp_b200.dense import LargeObject
    rng = _seed("mixed", template)
    xs, ys, yes = _objects(rng, MIXED, 1)
    grids = [_grid(rng, 1, m) for m in MIXED_GRIDS]
    gp = cg.gaussian_process_nobject(ys, xs, y_err=yes, **(_template(1) if template else {}))
    gp.hyperparameters, gp.nugget = HYP[1].copy(), NUG
    gp.get_prediction(new_binning=grids, COV="diag", svd_method=False)
    for i in range(len(MIXED)):
        if not len(grids[i]):
            assert gp.Prediction[i].shape == gp.prediction_variance[i].shape == (0,)
            continue
        lo = LargeObject(xs[i], ys[i], yes[i], gp.y0[i] if template else None, dim=1)
        lo.factor(HYP[1], NUG)
        m, v = lo.predict(grids[i], new_y0=gp.warning_pf[i] if template else None, want_var=True)
        np.testing.assert_array_equal(gp.Prediction[i], m)
        np.testing.assert_array_equal(gp.prediction_variance[i], v)
    _check_against_oracle(gp, xs, ys, yes, grids, 1, lambda i: HYP[1], lambda i: NUG, "diag",
                          _template(1) if template else None)


@gpu
def test_mixed_sizes_per_object(cg):
    """per_object=True on a mixed batch: the small objects equal a batch of the small objects alone, the large ones
    LargeObject with their own row; covariance matrices against the oracle."""
    from cosmogp_b200.dense import LargeObject
    rng = _seed("mixed rows")
    xs, ys, yes = _objects(rng, MIXED, 1)
    grids = [_grid(rng, 1, m) for m in MIXED_GRIDS]
    hyp, nug = _rows(rng, len(MIXED), 1), rng.uniform(0.01, 0.1, len(MIXED))
    gp = cg.gaussian_process_nobject(ys, xs, y_err=yes)
    gp.hyperparameters_per_object, gp.nugget_per_object = hyp.copy(), nug.copy()
    gp.get_prediction(new_binning=grids, COV=True, svd_method=False, per_object=True)
    small = [i for i, n in enumerate(MIXED) if n <= 224]
    alone = cg.gaussian_process_nobject([ys[i] for i in small], [xs[i] for i in small], y_err=[yes[i] for i in small])
    alone.hyperparameters_per_object, alone.nugget_per_object = hyp[small], nug[small]
    alone.get_prediction(new_binning=[grids[i] for i in small], COV="diag", svd_method=False, per_object=True)
    for k, i in enumerate(small):
        np.testing.assert_array_equal(gp.Prediction[i], alone.Prediction[k])
        np.testing.assert_array_equal(gp.prediction_variance[i], alone.prediction_variance[k])
    for i, n in enumerate(MIXED):
        if n > 224 and len(grids[i]):
            lo = LargeObject(xs[i], ys[i], yes[i], None, dim=1)
            lo.factor(hyp[i], nug[i])
            m, v = lo.predict(grids[i], new_y0=None, want_var=True)
            np.testing.assert_array_equal(gp.Prediction[i], m)
            np.testing.assert_array_equal(gp.prediction_variance[i], v)
    _check_against_oracle(gp, xs, ys, yes, grids, 1, lambda i: hyp[i], lambda i: nug[i], True, None)


LONG = {"n64": ((10, 40, 64), (20000, 5, 3000)), "generic": ((40, 100, 200), (20000, 5, 3000))}

_CHILD = r"""
import sys, numpy as np
sys.path.insert(0, sys.argv[1])
import cosmogp_b200 as cg
d = np.load(sys.argv[2], allow_pickle=True)
xs, ys, yes, grids = (list(d[k]) for k in ("xs", "ys", "yes", "grids"))
gp = cg.gaussian_process_nobject(ys, xs, y_err=yes)
gp.hyperparameters, gp.nugget = d["hyp"], float(d["nug"])
gp.get_prediction(new_binning=grids, COV="diag", svd_method=False)
np.savez(sys.argv[3], mean=gp.Prediction.flat, var=gp.prediction_variance.flat)
"""


def _objarray(seq):
    out = np.empty(len(seq), dtype=object)
    out[:] = seq
    return out


@gpu
@pytest.mark.parametrize("kernel", sorted(LONG))
def test_long_grids(cg, kernel, tmp_path):
    """Three objects with grids of 20 000, 5 and 3 000 points: against the oracle (chunked over the grid), and bit for
    bit equal to one work item per object (CGP_GRID_PARTS=0, in a child process: the knob is read once)."""
    rng = _seed("long", kernel)
    sizes, lengths = LONG[kernel]
    xs, ys, yes = _objects(rng, sizes, 1)
    grids = [_grid(rng, 1, m) for m in lengths]
    gp = cg.gaussian_process_nobject(ys, xs, y_err=yes)
    gp.hyperparameters, gp.nugget = HYP[1].copy(), NUG
    gp.get_prediction(new_binning=grids, COV="diag", svd_method=False)
    for i in range(len(sizes)):
        m, v = O.predict_grid_chunked(ys[i], xs[i], HYP[1], NUG, grids[i], yes[i])
        assert_close(gp.Prediction[i], m, 1e-9, 1e-11, "mean %d" % i)
        assert_close(gp.prediction_variance[i], v, 1e-9, 1e-11, "variance %d" % i)
    inp, out = tmp_path / "in.npz", tmp_path / "out.npz"
    np.savez(inp, xs=_objarray(xs), ys=_objarray(ys), yes=_objarray(yes), grids=_objarray(grids), hyp=HYP[1], nug=NUG)
    env = dict(os.environ, CGP_GRID_PARTS="0")
    r = subprocess.run([sys.executable, "-c", _CHILD, ROOT, str(inp), str(out)], cwd=ROOT, env=env,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    one = np.load(out)
    np.testing.assert_array_equal(gp.Prediction.flat, one["mean"])
    np.testing.assert_array_equal(gp.prediction_variance.flat, one["var"])


@gpu
def test_errors(cg):
    """A wrong number of grids and devices=... raise AssertionError; a singular object (duplicate epoch, no noise) is
    redone by the host SVD on its own grid with svd_method=True and raises LinAlgError with svd_method=False."""
    rng = _seed("errors")
    sizes = (12, 30, 20, 8)
    xs, ys, yes = _objects(rng, sizes, 1)
    grids = [_grid(rng, 1, m) for m in (40, 7, 100, 0)]
    gp = cg.gaussian_process_nobject(ys, xs, y_err=yes)
    gp.hyperparameters, gp.nugget = HYP[1].copy(), NUG
    with pytest.raises(AssertionError):
        gp.get_prediction(new_binning=grids[:3], COV="diag")
    gd = cg.gaussian_process_nobject(ys, xs, y_err=yes, devices=[0])
    gd.hyperparameters, gd.nugget = HYP[1].copy(), NUG
    with pytest.raises(AssertionError):
        gd.get_prediction(new_binning=grids, COV="diag")
    bad, hyp = 2, np.array([1.0, 1.5])
    xs[bad] = xs[bad].copy(); xs[bad][1] = xs[bad][0]
    yes[bad] = np.zeros(sizes[bad])
    gs = cg.gaussian_process_nobject(ys, xs, y_err=yes)
    gs.hyperparameters, gs.nugget = hyp.copy(), 0.0
    with pytest.raises(np.linalg.LinAlgError):
        gs.get_prediction(new_binning=grids, COV="diag", svd_method=False)
    with pytest.warns(RuntimeWarning):
        gs.get_prediction(new_binning=grids, COV="diag", svd_method=True)
    with pytest.warns(RuntimeWarning):
        _, m, v = gs._svd_object(bad, hyp, 0.0, grids[bad], 0.0, True)
    np.testing.assert_array_equal(gs.Prediction[bad], m)
    np.testing.assert_array_equal(gs.prediction_variance[bad], v)
    assert all(np.isfinite(gs.Prediction[i]).all() for i in range(len(sizes)))


def test_grid_classification():
    """Which new_binning is one grid per object (CPU only)."""
    from cosmogp_b200.gp import is_per_object_grid as per
    rng = np.random.default_rng(0)
    assert not per(None, 1) and not per(None, 2)
    assert not per(np.linspace(0, 1, 10), 1)
    assert not per([0.0, 0.5, 1.0], 1)
    assert not per(rng.uniform(size=(10, 2)), 2)
    assert per([np.linspace(0, 1, 5), np.linspace(0, 2, 8)], 1)
    assert per([rng.uniform(size=(5, 2)), rng.uniform(size=(0, 2))], 2)
    assert per(rng.uniform(size=(4, 10)), 1)
    assert per(rng.uniform(size=(4, 10, 2)), 2)
    assert per(_objarray([np.linspace(0, 1, 5), np.linspace(0, 2, 8)]), 1)
    assert per(_objarray([rng.uniform(size=(5, 2)), rng.uniform(size=(3, 2))]), 2)
