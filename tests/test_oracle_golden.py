"""Pins oracle/gp_oracle.py (the CPU restatement) against fixtures produced by the
real reference (tests/golden/make_golden.py) and against the notebook numbers the
reference prints.  CPU only."""
import numpy as np
import pytest
from scipy.optimize import fmin

from conftest import assert_close, golden, split
from oracle import gp_oracle as O

RT = 1e-11   # oracle vs reference: same LAPACK, different op order only


def test_kat_1d():
    g = golden("kat_1d")
    x, y, ye, hyp, nug = g["x"], g["y"], g["y_err"], g["hyp"], float(g["nugget"])
    assert_close(O.rbf_1d(x, hyp, nugget=nug, y_err=ye), g["kmat"], 1e-14, what="K")
    assert_close(O.cholesky_inverse(g["kmat"]), g["kinv"], 1e-11, 1e-12, "Kinv")
    assert_close(O.log_likelihood(y, x, hyp, nug, ye), g["ll_chol"], RT)
    assert_close(O.log_likelihood(y, x, hyp, nug, ye, svd_method=True), g["ll_svd"], RT)
    # survey section 9.3 literal values
    assert_close(g["ll_chol"], -3.965348881149514, 1e-15)
    assert_close(O.init_rbf([x], [y]), g["init_rbf"], 1e-15)
    assert_close(g["init_rbf"], [0.7148239865765148, 3.3838834764831844], 1e-15)
    mean, cov = O.predict(y, x, hyp, nug, g["grid"], y_err=ye)
    assert_close(mean, g["mean"], RT); assert_close(cov, g["cov"], 1e-9, 1e-14)
    _, var = O.predict(y, x, hyp, nug, g["grid"], y_err=ye, full_cov=False)
    assert_close(var, np.diag(g["cov"]), 1e-10)
    for fn in (O.loo_bruteforce, O.loo_closed_form):
        pred, _, pull, resid = fn(y, x, hyp, nug, ye)
        assert_close(pull, g["pull"], 1e-9, 1e-13, fn.__name__)
        assert_close(pred, g["pred"], 1e-9, 1e-13); assert_close(resid, g["resid"], 1e-9, 1e-13)
    assert_close(O.norm_fit(g["pull"]), [g["pull_average"], g["pull_std"]], 1e-13)


def test_kat_2d():
    g = golden("kat_2d")
    x, y, ye, hyp, nug = g["x"], g["y"], g["y_err"], g["hyp"], float(g["nugget"])
    k = O.rbf_2d(x, hyp, nugget=nug, y_err=ye)
    assert_close(k, g["kmat"], 1e-13, what="K2d")
    assert_close(k[0, 0], 1.1, 1e-15)                       # sigma^2 absent on the auto branch (Q2)
    assert_close(O.rbf_2d(x, hyp, new_x=g["grid"]), g["hmat"], 1e-13, what="H2d")
    assert_close(O.log_likelihood(y, x, hyp, nug, ye, kind="2d"), g["ll_chol"], RT)
    assert_close(g["ll_chol"], -19.172665221007133, 1e-15)
    assert_close(O.init_rbf([x], [y]), g["init_rbf"][:2], 1e-15)
    mean, cov = O.predict(y, x, hyp, nug, g["grid"], y_err=ye, kind="2d")
    assert_close(mean, g["mean"], 1e-10); assert_close(cov, g["cov"], 1e-9, 1e-13)
    pred, _, pull, resid = O.loo_closed_form(y, x, hyp, nug, ye, kind="2d")
    assert_close(pull, g["pull"], 1e-9, 1e-12); assert_close(pred, g["pred"], 1e-9, 1e-12)


def test_c1_single():
    g = golden("c1_single")
    x, y, ye, hyp, nug = g["x"], g["y"], g["y_err"], g["hyp"], float(g["nugget"])
    assert_close(O.log_likelihood(y, x, hyp, nug, ye), g["ll_chol"], RT)
    assert_close(O.log_likelihood(y, x, hyp, nug, ye, svd_method=True), g["ll_svd"], 1e-10)
    mean, var = O.predict(y, x, hyp, nug, g["grid"], y_err=ye, full_cov=False)
    assert_close(mean, g["mean"], 1e-10, 1e-13); assert_close(var, g["cov_diag"], 1e-9, 1e-13)
    _, cov = O.predict(y, x, hyp, nug, g["grid"], y_err=ye)
    assert_close(cov[100:140, 100:140], g["cov_block"], 1e-9, 1e-13)
    pred, _, pull, resid = O.loo_closed_form(y, x, hyp, nug, ye)
    assert_close(pull, g["pull"], 1e-9, 1e-12); assert_close(resid, g["resid"], 1e-9, 1e-12)


def test_ragged_1d_shared_mean():
    g = golden("ragged_1d")
    off, hyp, nug = g["off"], g["hyp"], float(g["nugget"])
    xs, ys, yes, y0s = (split(g[k], off) for k in ("x", "y", "y_err", "y0"))
    for i in range(len(xs)):
        assert_close(O.return_mean_1d(ys[i], xs[i], g["mean_y"], g["mean_x"]), y0s[i], 1e-15)
        assert_close(O.log_likelihood(ys[i], xs[i], hyp, nug, yes[i], y0s[i]), g["ll_obj"][i], RT)
    assert_close(O.log_likelihood_sum(ys, xs, hyp, nug, yes, y0s), g["ll_sum"], RT)
    assert_close(O.log_likelihood_sum(ys, xs, hyp, 0.07, yes, y0s), g["ll_sum_nugget007"], RT)
    assert_close(O.init_rbf(xs, ys), g["init_rbf"], 1e-15)
    for i in range(len(xs)):
        ny0 = O.return_mean_1d(ys[i], xs[i], g["mean_y"], g["mean_x"], new_x=g["grid"])
        mean, var = O.predict(ys[i], xs[i], hyp, nug, g["grid"], yes[i], y0s[i], ny0, full_cov=False)
        assert_close(mean, g["mean"][i], 1e-10); assert_close(var, g["var"][i], 1e-9, 1e-13)
    mean, cov = O.predict(ys[0], xs[0], hyp, 0.05, xs[0], yes[0], y0s[0], y0s[0])
    assert_close(mean, g["own_mean0"], 1e-10); assert_close(cov, g["own_cov0"], 1e-9, 1e-13)
    # pulls: mode B (mean given, diff None) and mode C (diff given)
    tmpl = [O.return_mean_1d(ys[i], xs[i], g["mean_y"], g["mean_x"], diff=0.0) for i in range(len(xs))]
    pb = [O.loo_closed_form(ys[i], xs[i], hyp, 0.05, yes[i], mean=tmpl[i]) for i in range(len(xs))]
    assert_close(np.concatenate([p[2] for p in pb]), g["pullB"], 1e-8, 1e-11, "pullB")
    assert_close(np.concatenate([p[0] for p in pb]), g["predB"], 1e-9, 1e-11)
    pc = [O.loo_closed_form(ys[i], xs[i], hyp, 0.05, yes[i], mean=tmpl[i], diff=g["diff"][i]) for i in range(len(xs))]
    assert_close(np.concatenate([p[2] for p in pc]), g["pullC"], 1e-8, 1e-11, "pullC")
    assert_close(O.norm_fit(g["pullB"]), [g["pullB_avg"], g["pullB_std"]], 1e-12)


def test_mean_options():
    """Constructor mean options run by the real reference: substract_mean=True without a template, a template with
    the offsets handed in, a single object predicted at its own epochs."""
    g = golden("mean_options")
    off, hyp, nug, grid = g["off"], g["hyp"], float(g["nugget"]), g["grid"]
    xs, ys, yes, y0sub = (split(g[k], off) for k in ("x", "y", "y_err", "y0_sub"))
    b = len(xs)
    # substract_mean=True, no template: y0 = mean(y) and that constant is also the mean on the grid
    for i in range(b):
        assert_close(O.return_mean_1d(ys[i], xs[i]), y0sub[i][0], 1e-15)          # a scalar per object (mean.py:87-90)
    assert_close(O.log_likelihood_sum(ys, xs, hyp, nug, yes, y0sub), g["ll_sub"], RT)
    for i in range(b):
        m, v = O.predict(ys[i], xs[i], hyp, nug, grid, yes[i], y0sub[i], y0sub[i][0], full_cov=False)
        assert_close(m, g["mean_sub"][i], RT); assert_close(v, g["var_sub"][i], RT, 1e-13)
    # template + given offsets
    y0d = [O.return_mean_1d(ys[i], xs[i], g["mean_y"], g["mean_x"], diff=g["diff"][i]) for i in range(b)]
    assert_close(O.log_likelihood_sum(ys, xs, hyp, nug, yes, y0d), g["ll_diff"], RT)
    for i in range(b):
        ny0 = O.return_mean_1d(ys[i], xs[i], g["mean_y"], g["mean_x"], diff=g["diff"][i], new_x=grid)
        m, v = O.predict(ys[i], xs[i], hyp, nug, grid, yes[i], y0d[i], ny0, full_cov=False)
        assert_close(m, g["mean_diff"][i], RT); assert_close(v, g["var_diff"][i], RT, 1e-13)
    # one object, template, offset estimated, own epochs
    y01 = O.return_mean_1d(ys[2], xs[2], g["mean_y"], g["mean_x"])
    assert_close(O.log_likelihood(ys[2], xs[2], hyp, nug, yes[2], y01), g["ll_one"], RT)
    m, v = O.predict(ys[2], xs[2], hyp, nug, xs[2], yes[2], y01, y01, full_cov=False)
    assert_close(m, g["mean_one"], RT); assert_close(v, g["var_one"], RT, 1e-13)


def test_pulls_modes_a_d():
    g = golden("pulls_1d")
    hyp, nug = g["hyp"], float(g["nugget"])
    res = [O.loo_closed_form(g["y"][i], g["x"][i], hyp, nug, g["y_err"][i]) for i in range(len(g["x"]))]
    assert_close(np.concatenate([r[2] for r in res]), g["pullA"], 1e-9, 1e-12)
    assert_close(np.array([r[0] for r in res]), g["predA"], 1e-9, 1e-12)
    assert_close(np.concatenate([r[2] for r in res]), g["pullA_svd"], 1e-8, 1e-11)   # svd path agrees too
    bf = O.loo_bruteforce(g["y"][0], g["x"][0], hyp, nug, g["y_err"][0])
    assert_close(bf[2], g["pullA"][:40], 1e-10, 1e-13)
    sticky = np.ones(40) * np.mean(g["yD"][0])              # pull.py:71-73 freezes object 0's mean
    rd = [O.loo_closed_form(g["yD"][i], g["xD"], hyp, nug, g["y_err"][i], mean=sticky, recenter=True) for i in range(3)]
    assert_close(np.concatenate([r[2] for r in rd]), g["pullD"], 1e-8, 1e-11, "pullD")
    b = O.loo_batched_1d(g["x"], g["y"], g["y_err"], hyp, nug)
    assert_close(b[2].ravel(), g["pullA"], 1e-9, 1e-12)


def test_batch_2d():
    g = golden("batch_2d")
    off, hyp, nug = g["off"], g["hyp"], float(g["nugget"])
    xs, ys, yes = split(g["x"], off), split(g["y"], off), split(g["y_err"], off)
    lls = [O.log_likelihood(ys[i], xs[i], hyp, nug, yes[i], kind="2d") for i in range(3)]
    assert_close(lls, g["ll_obj"], 1e-10); assert_close(sum(lls), g["ll_sum"], 1e-10)
    assert_close(O.rbf_2d(xs[2], hyp, nugget=nug, y_err=yes[2]), g["kmat2"], 1e-12, 1e-300)
    for i in range(3):
        mean, var = O.predict(ys[i], xs[i], hyp, nug, g["grid"], yes[i], kind="2d", full_cov=False)
        assert_close(mean, g["mean"][i], 1e-9, 1e-13); assert_close(var, g["var"][i], 1e-9, 1e-13)
    pred, _, pull, _ = O.loo_closed_form(ys[2], xs[2], hyp, nug, yes[2], kind="2d")
    assert_close(pull, g["pull2"], 1e-9, 1e-12); assert_close(pred, g["pred2"], 1e-9, 1e-12)
    assert_close(O.init_rbf(xs, ys), g["init_rbf"][:2], 1e-15)


def test_batched_helpers_match_per_object():
    g = golden("notebook_with_noise")
    x, y, ye = g["x"][:20], g["y"][:20], g["y_err"][:20]
    hyp = [0.5, 2.0]
    ll = O.ll_batched_1d(x, y, np.zeros_like(y), ye, hyp, 0.03)
    assert_close(ll, [O.log_likelihood(y[i], x[i], hyp, 0.03, ye[i]) for i in range(20)], 1e-11)
    grid = np.linspace(-10, 40, 33)
    m, v = O.predict_batched_1d(x, y, np.zeros_like(y), ye, hyp, 0.03, grid, np.zeros((20, 33)))
    for i in range(20):
        mi, vi = O.predict(y[i], x[i], hyp, 0.03, grid, ye[i], full_cov=False)
        assert_close(m[i], mi, 1e-10, 1e-14); assert_close(v[i], vi, 1e-10, 1e-14)


def test_notebook_known_answers():
    """docs/notebook/1D_kernel_example_with_noise.ipynb cells 9 and 21: the reference at
    HEAD reproduces the printed hyperparameters bit for bit (fixture stores both)."""
    g = golden("notebook_with_noise")
    assert np.array_equal(g["fit_single"], g["printed_single"])
    assert np.array_equal(g["fit_joint"], g["printed_joint"])
    x, y, ye = g["x"], g["y"], g["y_err"]
    neg = lambda h: -O.log_likelihood(y[0], x[0], h, 0.0, ye[0])
    fit = np.abs(fmin(neg, [0.5, 2.0], disp=False))
    assert_close(fit, g["printed_single"], 1e-6)
    assert_close(O.ll_batched_1d(x, y, np.zeros_like(y), ye, g["fit_joint"], 0.0).sum(), g["ll_at_joint"], 1e-11)
    w = golden("notebook_white_noise")
    assert_close(w["fit_single_svd"], w["printed_single"], 1e-11)
    h = w["fit_single_svd"]
    assert_close(O.log_likelihood(w["y"][0], w["x"][0], h[:2], h[2], svd_method=True), w["ll_at_fit_svd"], 1e-10)
    assert_close(O.log_likelihood(w["y"][0], w["x"][0], h[:2], h[2]), w["ll_at_fit_chol"], 1e-10)


def test_oracle_vs_live_reference_random():
    """The kernel matrices and inverses of the oracle against the reference: the reference's own outputs stored in the
    fixtures (60-point 1D object with per-point errors, 30-point 2D object with a nugget; the svd_method=True path is
    pinned by test_oracle_svd_path_against_the_reference_default), and fresh random cases when the reference is installed."""
    from oracle import ref_loader
    g = golden("ragged_1d")
    x0, ye0 = split(g["x"], g["off"])[0], split(g["y_err"], g["off"])[0]
    assert_close(O.rbf_1d(x0, g["hyp"], nugget=float(g["nugget"]), y_err=ye0), g["kmat0"], 1e-14)
    assert_close(O.cholesky_inverse(g["kmat0"]), g["kinv0"], 1e-15, 1e-15)
    b = golden("batch_2d")
    x2, ye2 = split(b["x"], b["off"])[2], split(b["y_err"], b["off"])[2]
    assert_close(O.rbf_2d(x2, b["hyp"], nugget=float(b["nugget"]), y_err=ye2), b["kmat2"], 1e-12, 1e-300)
    if not ref_loader.available():
        return
    ref = ref_loader.load()
    rng = np.random.default_rng(99)
    for n in (3, 17, 64):
        x = np.sort(rng.uniform(0, 30, n)); ye = rng.uniform(0.05, 0.2, n); y = rng.standard_normal(n)
        hyp = [0.8, 3.0]
        assert_close(O.rbf_1d(x, hyp, nugget=0.1, y_err=ye), ref.rbf_kernel_1d(x, hyp, nugget=0.1, y_err=ye), 1e-14)
        x2 = rng.uniform(-5, 5, (n, 2)); h2 = [1.3, 2.0, 3.0, 1.5]
        with ref_loader.quiet():
            assert_close(O.rbf_2d(x2, h2, nugget=0.1, y_err=ye), ref.rbf_kernel_2d(x2, h2, nugget=0.1, y_err=ye), 1e-12, 1e-300)
            assert_close(O.rbf_2d(x2, h2, new_x=x2[:2] + 0.3), ref.rbf_kernel_2d(x2, h2, new_x=x2[:2] + 0.3), 1e-12, 1e-300)
        k = O.rbf_1d(x, hyp, nugget=0.1, y_err=ye)
        assert_close(O.cholesky_inverse(k), ref.cholesky_inverse(k), 1e-15, 1e-15)
        assert_close(O.svd_inverse(k), ref.svd_inverse(k), 1e-15, 1e-15)


def test_chunked_grid_prediction_equals_the_one_shot_formula():
    """predict_grid_chunked (used for BASELINE config 3 at full size) = predict(full_cov=False) slice by slice."""
    rng = np.random.default_rng(8)
    x = rng.uniform(-50, 50, (70, 2)); y = rng.standard_normal(70); ye = np.full(70, 0.2)
    grid = rng.uniform(-50, 50, (333, 2)); hyp = [1.2, 20.0, 15.0, 30.0]
    m1, v1 = O.predict(y, x, hyp, 0.1, grid, ye, 0.0, 0.0, kind="2d", full_cov=False)
    m2, v2 = O.predict_grid_chunked(y, x, hyp, 0.1, grid, ye, kind="2d", chunk=100)
    assert np.max(np.abs(m1 - m2)) < 1e-12 and np.max(np.abs(v1 - v2)) < 1e-12
    x1 = np.sort(rng.uniform(0, 30, 40)); g1 = np.linspace(0, 30, 77)
    m1, v1 = O.predict(y[:40], x1, [0.7, 3.0], 0.05, g1, ye[:40], 0.1, 0.2, full_cov=False)
    m2, v2 = O.predict_grid_chunked(y[:40], x1, [0.7, 3.0], 0.05, g1, ye[:40], 0.1, 0.2, chunk=20)
    assert np.max(np.abs(m1 - m2)) < 1e-12 and np.max(np.abs(v1 - v2)) < 1e-12


def test_oracle_svd_path_against_the_reference_default():
    """The oracle's svd_method=True branch (inv_matrix.py:4-18) on the fixture the real reference produced with its
    default arguments: a singular covariance (12 singular values truncated) beside a well-posed one."""
    g = golden("svd_default")
    ll0 = O.log_likelihood(g["sing_y"], g["sing_x"], g["sing_hyp"], 0.0, np.zeros(len(g["sing_x"])), svd_method=True)
    ll1 = O.log_likelihood(g["ok_y"], g["ok_x"], g["sing_hyp"], 0.0, np.full(len(g["ok_x"]), 0.1), svd_method=True)
    assert_close(ll0, g["sing_ll_per_object"][0], 1e-9); assert_close(ll1, g["sing_ll_per_object"][1], 1e-12)
    assert_close(ll0 + ll1, float(g["sing_ll_total"]), 1e-12)
    with pytest.raises(np.linalg.LinAlgError):
        O.log_likelihood(g["sing_y"], g["sing_x"], g["sing_hyp"], 0.0, np.zeros(len(g["sing_x"])), svd_method=False)
    m, v = O.predict(g["ok_y"], g["ok_x"], g["sing_hyp"], 0.0, g["sing_grid"], np.full(len(g["ok_x"]), 0.1), svd_method=True, full_cov=False)
    assert_close(m, g["sing_pred"][1], 1e-10); assert_close(v, g["sing_var"][1], 1e-9)
    # the noise-free notebook fit (default arguments) is reproduced by the oracle's objective
    r = fmin(lambda h: -O.log_likelihood(g["y"], g["x"], h, 0.0, svd_method=True), [0.5, 1], disp=False)
    assert_close(np.abs(r), g["printed_single"], 1e-12)
