"""Size routing of the facade under shared hyperparameters (batch.SizeSplit): a 1D batch that mixes small objects with
objects of 225 and 400 points sends every object through its own dense.LargeObject -- the likelihood, predictions on
the objects' epochs and on a shared grid, with and without a mean template -- and redoes a singular object by the host
SVD when svd_method=True."""
import numpy as np
import pytest

from conftest import assert_close
from oracle import gp_oracle as O

pytestmark = pytest.mark.gpu

HYP, NUG = np.array([0.8, 1.5]), 0.05
SIZES = (12, 225, 40, 7, 400, 60)
LARGE = 1                                           # index of the 225-point object


@pytest.fixture(scope="module")
def cg():
    import cosmogp_b200
    from cosmogp_b200 import _lib
    _lib.require_device()
    return cosmogp_b200


def _batch(seed):
    rng = np.random.default_rng(seed)
    xs = [np.sort(rng.uniform(0, n / 5.0, n)) for n in SIZES]
    ys = [np.sin(x) + 0.3 + 0.2 * rng.standard_normal(len(x)) for x in xs]
    return xs, ys, [rng.uniform(0.1, 0.3, len(x)) for x in xs]


def _template():
    tx = np.linspace(-5, 100, 60)
    return dict(Mean_Y=0.3 * np.cos(tx / 7), Time_mean=tx)


@pytest.mark.parametrize("grid", ["own", "shared"])
@pytest.mark.parametrize("template", [False, True])
def test_every_object_through_its_large_object(cg, grid, template):
    """Per-object likelihoods, means and variances bit-identical to direct LargeObject.factor / .predict calls on each
    object's slices; warning_pf is the mean function on the grid and the outputs are RaggedViews."""
    from cosmogp_b200 import mean as M
    from cosmogp_b200.batch import RaggedView
    from cosmogp_b200.dense import LargeObject
    xs, ys, yes = _batch(10 + 2 * template + (grid == "shared"))
    kw = _template() if template else {}
    gp = cg.gaussian_process_nobject(ys, xs, y_err=yes, **kw)
    gp.hyperparameters, gp.nugget = HYP.copy(), NUG
    gp.compute_log_likelihood(HYP, svd_method=False)
    new = None if grid == "own" else np.linspace(0, 80, 97)
    gp.get_prediction(new_binning=new, COV='diag', svd_method=False)
    assert len(gp.Prediction) == len(SIZES) and gp.as_the_same_time == (grid == "own")
    tmpl = M.template_on_grid(new, 1, kw["Mean_Y"], kw["Time_mean"]) if template and new is not None else None
    lls = []
    for i in range(len(SIZES)):
        y0 = gp.y0[i] if template else None
        lo = LargeObject(xs[i], ys[i], yes[i], y0, dim=1)
        lls.append(lo.factor(HYP, NUG))
        if not template:
            ny0 = None
        else:
            ny0 = y0 if new is None else tmpl + gp._diff_used[i]
        m, v = lo.predict(xs[i] if new is None else new, new_y0=ny0, want_var=True)
        assert gp.log_likelihood_per_object[i] == lls[-1], i
        np.testing.assert_array_equal(gp.Prediction[i], m)
        np.testing.assert_array_equal(gp.prediction_variance[i], v)
    assert gp.log_likelihood[0] == np.add.accumulate(lls)[-1]
    if not template:
        assert gp.warning_pf is None
    elif new is None:
        np.testing.assert_array_equal(gp.warning_pf, np.concatenate([gp.y0[i] for i in range(len(SIZES))]))
    else:
        np.testing.assert_array_equal(np.asarray(gp.warning_pf), tmpl[None, :] + gp._diff_used[:, None])
    assert isinstance(gp.Prediction, RaggedView) and isinstance(gp.prediction_variance, RaggedView)


@pytest.mark.parametrize("grid", ["own", "shared"])
def test_singular_object(cg, grid):
    """A small object with a duplicate epoch and no noise: svd_method=True redoes exactly that object by the host SVD
    (bit-identical to _svd_object, with a RuntimeWarning); svd_method=False raises LinAlgError.  A unit amplitude makes
    the second pivot exactly zero."""
    hyp = np.array([1.0, 1.5])
    xs, ys, yes = _batch(20)
    bad = 2
    xs[bad] = xs[bad].copy(); xs[bad][1] = xs[bad][0]
    yes[bad] = np.zeros(SIZES[bad])
    gp = cg.gaussian_process_nobject(ys, xs, y_err=yes)
    gp.hyperparameters, gp.nugget = hyp.copy(), 0.0
    new = None if grid == "own" else np.linspace(0, 80, 97)
    with pytest.raises(np.linalg.LinAlgError):
        gp.compute_log_likelihood(hyp, svd_method=False)
    with pytest.raises(np.linalg.LinAlgError):
        gp.get_prediction(new_binning=new, COV='diag', svd_method=False)
    with pytest.warns(RuntimeWarning):
        gp.compute_log_likelihood(hyp, svd_method=True)
    with pytest.warns(RuntimeWarning):
        gp.get_prediction(new_binning=new, COV='diag', svd_method=True)
    with pytest.warns(RuntimeWarning):
        ll, m, v = gp._svd_object(bad, hyp, 0.0, xs[bad] if new is None else new, 0.0, True)
    assert gp.log_likelihood_per_object[bad] == ll
    np.testing.assert_array_equal(gp.Prediction[bad], m)
    np.testing.assert_array_equal(gp.prediction_variance[bad], v)
    assert np.isfinite(gp.log_likelihood_per_object).all()


def test_matrices_of_a_large_object(cg):
    """kernel_matrix and inv_kernel_matrix of the 225-point object and of a small one against the oracle's K and its
    Cholesky inverse."""
    xs, ys, yes = _batch(30)
    gp = cg.gaussian_process_nobject(ys, xs, y_err=yes)
    gp.hyperparameters, gp.nugget = HYP.copy(), NUG
    gp.get_prediction(COV='diag', svd_method=False)
    for i in (LARGE, 2):
        k = O.rbf_1d(xs[i], HYP, nugget=NUG, y_err=yes[i])
        kinv = O.cholesky_inverse(k)
        assert_close(gp.kernel_matrix[i], k, 1e-9, 1e-12, "K %d" % i)
        assert_close(gp.inv_kernel_matrix[i], kinv, 1e-9, 1e-9 * np.abs(kinv).max(), "K^-1 %d" % i)
