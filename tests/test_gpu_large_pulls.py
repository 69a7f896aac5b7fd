"""Leave-one-out pulls of objects above CGP_SMALL_MAX_N points (blocked factor in HBM, diag(K^-1) by the blocked solve on
identity rows) and build_pull over batches that mix them with small objects, against the oracle.  Tolerance: relative
1e-9 with the absolute floors of the shared-memory LOO tests (1e-9 on predictions, 1e-8 on pulls)."""
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


def _object(rng, n, dim):
    """Seeded object with cond(K) of order 1e3 under _hyp(dim)."""
    if dim == 1:
        x = np.sort(rng.uniform(0, n / 5.0, n))
        y = np.sin(x) + 0.2 * rng.standard_normal(n)
    else:
        s = 3.0 * np.sqrt(n)
        x = rng.uniform(0, s, (n, 2))
        y = np.sin(x[:, 0] / 5) * np.cos(x[:, 1] / 4) + 0.2 * rng.standard_normal(n)
    return x, y, rng.uniform(0.1, 0.3, n)


def _hyp(dim):
    return [0.8, 1.5] if dim == 1 else [1.1, 4.0, 3.0, 1.0]


def _mean_at(dim, tx, ty, x):
    from cosmogp_b200 import mean as M
    return (M.interpolate_mean_1d if dim == 1 else M.interpolate_mean_2d)(tx, ty, x)


def _check(bp, xs, ys, yes, hyp, nug, kind, means=None, diff=None, recenter=False):
    """every object of a single compute_pull call against loo_closed_form"""
    pulls = []
    for i in range(len(ys)):
        po = O.loo_closed_form(ys[i], xs[i], hyp, nug, yes[i], mean=None if means is None else means[i],
                               diff=None if diff is None else diff[i], recenter=recenter, kind=kind)
        assert_close(bp.prediction[i], po[0], 1e-9, 1e-9, "pred %d" % i)
        assert_close(bp._pull[i], po[2], 1e-9, 1e-8, "pull %d" % i)
        pulls.append(po[2])
    return np.concatenate(pulls)


def test_bruteforce_1d_300(cg):
    rng = np.random.default_rng(300)
    x, y, ye = _object(rng, 300, 1)
    hyp, nug = _hyp(1), 0.03
    bp = cg.build_pull([y], [x], hyp, nugget=nug, y_err=[ye])
    bp.compute_pull(svd_method=False)
    bf = O.loo_bruteforce(y, x, hyp, nug, ye)
    cf = O.loo_closed_form(y, x, hyp, nug, ye)
    assert_close(np.asarray(bp.prediction[0]), bf[0], 1e-9, 1e-9, "pred vs refits")
    assert_close(bp.prediction_variance, bf[1], 1e-9, 1e-9, "pred_var vs refits")
    assert_close(bp.pull, bf[2], 1e-9, 1e-8, "pull vs refits")
    assert_close(bp.residual, bf[3], 1e-9, 1e-9, "resid vs refits")
    for got, want, what in zip((np.asarray(bp.prediction[0]), bp.prediction_variance, bp.pull, bp.residual), cf,
                               ("pred", "pred_var", "pull", "resid")):
        assert_close(got, want, 1e-9, 1e-9, what + " vs closed form")


def _large_loo(x, y, m, ye, hyp, nug, dim, mode, chunk_rows=None):
    """one object through dense.LargeLoo (cgp_large_loo_dev) -> host (pred, pred_var, pull, resid)"""
    import torch
    from cosmogp_b200.dense import LargeLoo
    dev = torch.device("cuda", torch.cuda.current_device())
    xd, yd, md, ed = (torch.from_numpy(np.ascontiguousarray(v, dtype=np.float64)).to(dev) for v in (x, y, m, ye))
    outs = [torch.empty(len(y), dtype=torch.float64, device=dev) for _ in range(4)]
    info = torch.ones(1, dtype=torch.int32, device=dev)
    LargeLoo(len(y), dim, chunk_rows=chunk_rows).run(xd, yd, md, ed, hyp, nug, mode, info, outs)
    assert int(info.item()) == 0
    return [o.cpu().numpy() for o in outs]


def _nearest_template(old_binning, mean_function, new_binning):
    """Stand-in for mean.interpolate_mean_2d in the 2D mode tests: the template value at the nearest template point.
    interpolate_mean_2d calls scipy's bisplrep with task=1 as the reference does (mean.py:36-67); scipy 1.18 keeps no
    workspace between calls, so that call fails on every input.  What these tests check is how compute_pull uses the
    template (mode choice, fixed offsets, the first object's mean in mode D), not the interpolation."""
    old, new = np.asarray(old_binning, dtype=float), np.asarray(new_binning, dtype=float)
    d = ((new[:, None, :] - old[None, :, :]) ** 2).sum(-1)
    return np.asarray(mean_function, dtype=float)[np.argmin(d, axis=1)]


@pytest.mark.parametrize("dim", [1, 2])
@pytest.mark.parametrize("n", [225, 255, 256, 257, 383, 384, 385, 1000])
def test_padding_edges_and_modes(cg, monkeypatch, n, dim):
    from cosmogp_b200 import mean as M
    if dim == 2:
        monkeypatch.setattr(M, "interpolate_mean_2d", _nearest_template)
    rng = np.random.default_rng(10 * n + dim)
    kind = "1d" if dim == 1 else "2d"
    kernel = "RBF1D" if dim == 1 else "RBF2D"
    objs = [_object(rng, n, dim), _object(rng, 40, dim)]
    xs, ys, yes = ([o[k] for o in objs] for k in range(3))
    hyp, nug = _hyp(dim), 0.02
    if dim == 1:
        tx = np.linspace(-5, 400, 60)
        ty = 0.3 * np.cos(tx / 7.0)
    else:
        tx = rng.uniform(0, 100, (80, 2))
        ty = 0.2 + 0.3 * np.sin(tx[:, 0] / 30) * np.cos(tx[:, 1] / 25)
    means = [_mean_at(dim, tx, ty, x) for x in xs]
    diff = [0.05, -0.1]
    for name, ctor, ref in (("A", {}, {}),
                            ("B", dict(y_mean=ty, x_axis_mean=tx), dict(means=means, recenter=True)),
                            ("C", dict(y_mean=ty, x_axis_mean=tx), dict(means=means, diff=diff))):
        bp = cg.build_pull(ys, xs, hyp, nugget=nug, y_err=yes, kernel=kernel, **ctor)
        bp.compute_pull(diff=diff if name == "C" else None, svd_method=False)
        allp = _check(bp, xs, ys, yes, hyp, nug, kind, **ref)
        assert_close([bp.pull_average, bp.pull_std], O.norm_fit(allp), 1e-9, 1e-12, "norm.fit mode " + name)
    bp = cg.build_pull(ys, xs, hyp, nugget=nug, y_err=yes, kernel=kernel)
    bp.compute_pull(svd_method=False, substract_mean=True)       # mode D: the first object's mean becomes the template
    md = [_mean_at(dim, xs[0], np.ones_like(ys[0]) * np.mean(ys[0]), x) for x in xs]
    allp = _check(bp, xs, ys, yes, hyp, nug, kind, means=md, recenter=True)
    assert_close([bp.pull_average, bp.pull_std], O.norm_fit(allp), 1e-9, 1e-12, "norm.fit mode D")


def test_diag_inv_chunks_past_the_first_block(cg):
    """N = 1 000 (n_pad = 1 024) in chunks of 384 rows: the chunks start at block columns 0, 3 and 6, run over several
    block-column pairs, end on an unpaired block and have their row counts clipped; all agree with one chunk."""
    from cosmogp_b200 import _lib
    rng = np.random.default_rng(1000)
    for dim, mode in ((1, _lib.CGP_LOO_PLAIN), (2, _lib.CGP_LOO_RECENTER)):
        x, y, ye = _object(rng, 1000, dim)
        m = 0.1 * rng.standard_normal(1000)
        hyp, nug = _hyp(dim), 0.02
        got = [_large_loo(x, y, m, ye, hyp, nug, dim, mode, chunk_rows=c) for c in (384, None)]
        for a, b, what in zip(got[0], got[1], ("pred", "pred_var", "pull", "resid")):
            assert_close(a, b, 1e-12, 1e-12, "%s: chunks of 384 rows vs all rows (dim %d)" % (what, dim))
        po = O.loo_closed_form(y, x, hyp, nug, ye, mean=m, recenter=mode == _lib.CGP_LOO_RECENTER,
                               diff=None if mode == _lib.CGP_LOO_RECENTER else 0.0, kind="1d" if dim == 1 else "2d")
        assert_close(got[0][0], po[0], 1e-9, 1e-9, "pred vs closed form (dim %d)" % dim)
        assert_close(got[0][2], po[2], 1e-9, 1e-8, "pull vs closed form (dim %d)" % dim)


def test_route_cross_check_200_points(cg):
    """One object of 200 points through the batched shared-memory kernel and through cgp_large_loo_dev on its
    256-padded factor; chunks of 128 rows and of all rows give the same outputs."""
    from cosmogp_b200 import _lib
    from cosmogp_b200.batch import DeviceBatch
    rng = np.random.default_rng(200)
    for dim, mode in ((1, _lib.CGP_LOO_PLAIN), (2, _lib.CGP_LOO_RECENTER)):
        x, y, ye = _object(rng, 200, dim)
        m = 0.1 * rng.standard_normal(200)
        hyp, nug = _hyp(dim), 0.04
        small = DeviceBatch(x, y, np.array([0, 200]), y0=m, y_err=ye, dim=dim).loo(hyp, nug, mode=mode)
        assert not small[4].any()
        got = [_large_loo(x, y, m, ye, hyp, nug, dim, mode, chunk_rows=c) for c in (128, 256)]
        for a, b, s, what in zip(got[0], got[1], small[:4], ("pred", "pred_var", "pull", "resid")):
            assert_close(a, s, 1e-11, 1e-11, "%s: large route vs shared-memory route (dim %d)" % (what, dim))
            assert_close(a, b, 1e-12, 1e-12, "%s: chunk 128 vs all rows (dim %d)" % (what, dim))


def _mixed(rng, n_small=300, large=(225, 600, 310, 480, 257, 384)):
    sizes = list(rng.integers(5, 225, n_small))
    for k, n in enumerate(large):
        sizes.insert(int((k + 1) * n_small / (len(large) + 1)) + k, n)
    objs = [_object(rng, n, 1) for n in sizes]
    return sizes, [o[0] for o in objs], [o[1] for o in objs], [o[2] for o in objs]


def test_mixed_batch(cg):
    rng = np.random.default_rng(4)
    sizes, xs, ys, yes = _mixed(rng)
    hyp, nug = _hyp(1), 0.02
    bp = cg.build_pull(ys, xs, hyp, nugget=nug, y_err=yes)
    bp.compute_pull(svd_method=False)
    small = [i for i, n in enumerate(sizes) if n <= 224]
    large = [i for i, n in enumerate(sizes) if n > 224]
    ref = cg.build_pull([ys[i] for i in small], [xs[i] for i in small], hyp, nugget=nug, y_err=[yes[i] for i in small])
    ref.compute_pull(svd_method=False)
    for j, i in enumerate(small):
        assert np.array_equal(bp._pull[i], ref._pull[j]), "small object %d" % i
        assert np.array_equal(bp.prediction[i], ref.prediction[j]), "small object %d" % i
    off = np.concatenate([[0], np.cumsum(sizes)])
    ref_off = np.concatenate([[0], np.cumsum([sizes[i] for i in small])])
    for j, i in enumerate(small):
        s, t = slice(off[i], off[i + 1]), slice(ref_off[j], ref_off[j + 1])
        assert np.array_equal(bp.residual[s], ref.residual[t])
        assert np.array_equal(bp.prediction_variance[s], ref.prediction_variance[t])
    for i in large:
        po = O.loo_closed_form(ys[i], xs[i], hyp, nug, yes[i])
        assert_close(bp.prediction[i], po[0], 1e-9, 1e-9, "large pred %d" % i)
        assert_close(bp._pull[i], po[2], 1e-9, 1e-8, "large pull %d" % i)
    assert [len(p) for p in bp._pull] == sizes
    first = bp.pull.copy()
    bp.compute_pull(svd_method=False)
    assert len(bp._pull) == 2 * len(sizes) and len(bp.pull) == 2 * off[-1]
    assert [len(p) for p in bp._pull] == sizes + sizes
    assert np.array_equal(bp.pull[off[-1]:], first)
    assert_close([bp.pull_average, bp.pull_std], O.norm_fit(np.concatenate([first, first])), 1e-9, 1e-12)


def test_mixed_batch_per_object_hyperparameters(cg):
    rng = np.random.default_rng(5)
    sizes, xs, ys, yes = _mixed(rng, n_small=60, large=(300, 450))
    b = len(sizes)
    hyp = np.column_stack([rng.uniform(0.6, 1.2, b), rng.uniform(1.0, 2.0, b)])
    nug = rng.uniform(0.0, 0.05, b)
    tx = np.linspace(-5, 400, 60)
    ty = 0.3 * np.cos(tx / 7.0)
    diff = rng.uniform(-0.2, 0.2, b)
    bp = cg.build_pull(ys, xs, hyp, nugget=nug, y_err=yes, y_mean=ty, x_axis_mean=tx)
    bp.compute_pull(diff=diff, svd_method=False)
    for i in range(b):
        po = O.loo_closed_form(ys[i], xs[i], hyp[i], nug[i], yes[i], mean=_mean_at(1, tx, ty, xs[i]), diff=diff[i])
        assert_close(bp.prediction[i], po[0], 1e-9, 1e-9, "pred %d" % i)
        assert_close(bp._pull[i], po[2], 1e-9, 1e-8, "pull %d" % i)


def test_2d_amp_on_autocov(cg):
    from cosmogp_b200 import _lib
    rng = np.random.default_rng(22)
    x, y, ye = _object(rng, 300, 2)
    hyp, nug = [1.3, 4.0, 3.0, 1.0], 0.03
    bp = cg.build_pull([y], [x], hyp, nugget=nug, y_err=[ye], kernel="RBF2D")
    bp.flags = _lib.CGP_AMP_ON_AUTOCOV
    bp.compute_pull(svd_method=False)
    # numpy closed form with sigma^2 on the auto-covariance: rho = 1, K** = sigma^2 + nugget^2
    k = O.rbf_2d(x, hyp, nugget=nug, y_err=ye, amp_on_autocov=True)
    inv = O.cholesky_inverse(k)
    d = np.diag(inv)
    pred = y - (inv @ y) / d
    var = np.abs(hyp[0] ** 2 + nug ** 2 - (np.diag(k) - 1.0 / d))
    pull = (pred - y) / np.sqrt(ye ** 2 + var + nug ** 2)
    assert_close(np.asarray(bp.prediction[0]), pred, 1e-9, 1e-9)
    assert_close(bp.prediction_variance, var, 1e-9, 1e-9)
    assert_close(bp.pull, pull, 1e-9, 1e-8)


def test_large_not_positive_definite_names_object(cg):
    rng = np.random.default_rng(7)
    xs = [np.sort(rng.uniform(0, 10, 30)), np.sort(rng.uniform(0, 60, 250)), np.repeat(np.linspace(0, 10, 150), 2)]
    ys = [rng.standard_normal(len(x)) for x in xs]
    yes = [np.full(30, 0.1), np.full(250, 0.1), np.zeros(300)]       # duplicate epochs and no noise in object 2 only
    bp = cg.build_pull(ys, xs, [1.0, 1.0], nugget=0.0, y_err=yes)
    with pytest.raises(np.linalg.LinAlgError, match="object 2 "):
        bp.compute_pull(svd_method=False)


def test_c3_recipe_all_points(cg):
    rng = np.random.default_rng(3)
    n = 2000
    x = rng.uniform(-200, 200, (n, 2)); hyp = [1.0, 30.0, 25.0, 50.0]
    ye = np.full(n, 0.2)
    y = np.sin(x[:, 0] / 60) * np.cos(x[:, 1] / 45) + 0.2 * rng.standard_normal(n)
    bp = cg.build_pull([y], [x], hyp, y_err=[ye], kernel="RBF2D")
    bp.compute_pull(svd_method=False)
    po = O.loo_closed_form(y, x, hyp, 0.0, ye, kind="2d")
    assert_close(np.asarray(bp.prediction[0]), po[0], 1e-9, 1e-9)
    assert_close(bp.prediction_variance, po[1], 1e-9, 1e-9)
    assert_close(bp.pull, po[2], 1e-9, 1e-8)


def test_c4_recipe_sampled_points(cg):
    """N = 20,000 (the C4 recipe of test_c4_large_single_object_at_config_size): 16 points against the host LAPACK
    factorisation, d_t = e_t^T K^-1 e_t and alpha = K^-1 y by cho_solve."""
    from scipy import linalg as sla
    rng = np.random.default_rng(4)
    n = 20000
    x = rng.uniform(0, 1000, (n, 2)); hyp = [1.0, 30.0, 30.0, 0.0]
    ye = np.full(n, 0.3)
    y = np.sin(x[:, 0] / 90) * np.cos(x[:, 1] / 70) + 0.3 * rng.standard_normal(n)
    bp = cg.build_pull([y], [x], hyp, y_err=[ye], kernel="RBF2D")
    bp.compute_pull(svd_method=False)
    k = np.empty((n, n))
    for s in range(0, n, 2000):
        k[s:s + 2000] = O.rbf_2d(x, hyp, new_x=x[s:s + 2000])
    k[np.arange(n), np.arange(n)] = 1.0 + ye ** 2
    low = sla.cholesky(k, lower=True, overwrite_a=True, check_finite=False)
    del k
    t = np.sort(rng.choice(n, 16, replace=False))
    e = np.zeros((n, 16)); e[t, np.arange(16)] = 1.0
    d = np.einsum("ij,ij->j", e, sla.cho_solve((low, True), e, check_finite=False))
    alpha = sla.cho_solve((low, True), y, check_finite=False)[t]
    pred = y[t] - alpha / d                               # sigma = 1: rho = 1
    var = np.abs(1.0 - (1.0 + ye[t] ** 2 - 1.0 / d))
    pull = (pred - y[t]) / np.sqrt(ye[t] ** 2 + var)
    assert_close(np.asarray(bp.prediction[0])[t], pred, 1e-9, 1e-9)
    assert_close(bp.prediction_variance[t], var, 1e-9, 1e-9)
    assert_close(bp.pull[t], pull, 1e-9, 1e-8)
