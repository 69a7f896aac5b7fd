"""Host-side mean function (cosmogp/mean.py): the batched evaluation must reproduce the reference's
per-object `return_mean` bit for bit (same scipy calls).  Compared against the reference's outputs stored
in tests/golden, and on fresh random cases against the live reference when it is installed, else against
the oracle restatement."""
import numpy as np
import pytest

from conftest import assert_close, golden
from cosmogp_b200 import mean as M
from oracle import gp_oracle as O, ref_loader


def test_batched_mean_matches_stored_reference():
    """y0 as the reference computed it: the template spline plus one offset per object (ragged_1d), and the plain
    average per object without a template (mean_options, substract_mean=True)."""
    g = golden("ragged_1d")
    y0, _ = M.batched_mean(g["x"], g["y"], g["off"], 1, g["mean_y"], g["mean_x"], np.array([None] * (len(g["off"]) - 1)))
    assert np.array_equal(y0, g["y0"])
    for i in range(len(g["off"]) - 1):
        a, b = g["off"][i], g["off"][i + 1]
        assert np.array_equal(M.return_mean(g["y"][a:b], g["x"][a:b], mean_y=g["mean_y"], mean_xaxis=g["mean_x"]), g["y0"][a:b])
    m = golden("mean_options")
    y0n, _ = M.batched_mean(m["x"], m["y"], m["off"], 1, None, None, np.array([None] * (len(m["off"]) - 1)))
    assert np.array_equal(y0n, m["y0_sub"])


def _objects(rng, b):
    xs = [np.sort(rng.uniform(-10, 40, int(rng.integers(5, 50)))) for _ in range(b)]
    ys = [np.sin(x / 7.0) - 18 + rng.normal(0, 0.3) + 0.1 * rng.standard_normal(len(x)) for x in xs]
    return xs, ys


def test_batched_mean_1d_matches_per_object():
    rng = np.random.default_rng(1)
    xs, ys = _objects(rng, 30)
    tm = np.linspace(-15, 45, 61); ym = -18 + 2 * np.sin(tm / 10)
    off = np.zeros(31, dtype=np.int64); off[1:] = np.cumsum([len(x) for x in xs])
    y0, d = M.batched_mean(np.concatenate(xs), np.concatenate(ys), off, 1, ym, tm, np.array([None] * 30))
    ref = ref_loader.load() if ref_loader.available() else None
    for i in range(30):
        want = ref.return_mean(ys[i], xs[i], mean_y=ym, mean_xaxis=tm) if ref else O.return_mean_1d(ys[i], xs[i], ym, tm)
        assert np.array_equal(y0[off[i]:off[i + 1]], want)
        assert np.array_equal(M.return_mean(ys[i], xs[i], mean_y=ym, mean_xaxis=tm), want)
    # given offsets and a new grid
    diff = [0.25 * i for i in range(30)]
    y0g, dg = M.batched_mean(np.concatenate(xs), np.concatenate(ys), off, 1, ym, tm, diff)
    grid = np.linspace(-10, 40, 17)
    for i in (0, 7, 29):
        want = ref.return_mean(ys[i], xs[i], new_x=grid, mean_y=ym, mean_xaxis=tm, diff=diff[i]) if ref else \
            O.return_mean_1d(ys[i], xs[i], ym, tm, diff=diff[i], new_x=grid)
        assert np.array_equal(M.template_on_grid(grid, 1, ym, tm) + dg[i], want)
    # no template: y0 is the plain average
    y0n, dn = M.batched_mean(np.concatenate(xs), np.concatenate(ys), off, 1, None, None, np.array([None] * 30))
    assert_close(dn, [np.mean(y) for y in ys], 1e-15)
    with pytest.raises(AssertionError):
        M.batched_mean(np.concatenate(xs), np.concatenate(ys), off, 1, ym, None, None)


@pytest.mark.skipif(not ref_loader.available(), reason="reference tree absent")
def test_mean_2d_behaves_like_reference():
    """The reference's 2D template path calls bisplrep(task=1) (mean.py:58), which current scipy
    rejects on a first call ("wrk array too small for iopt=1"); the drop-in makes the same call and
    fails the same way -- a 2D template mean is unusable in both until the reference changes."""
    ref = ref_loader.load()
    rng = np.random.default_rng(2)
    g = np.linspace(0, 10, 8); gx, gy = np.meshgrid(g, g)
    old = np.array([gx.ravel(), gy.ravel()]).T
    fmean = np.cos(old[:, 0] / 3.0) + 0.1 * old[:, 1]
    x = rng.uniform(1, 9, (12, 2)); y = rng.standard_normal(12)
    outcomes = []
    for fn in (ref.return_mean, M.return_mean):
        try:
            outcomes.append(fn(y, x, mean_y=fmean, mean_xaxis=old))
        except Exception as e:                      # noqa: BLE001 - the point is that both fail alike
            outcomes.append(type(e))
    if isinstance(outcomes[0], type):
        assert outcomes[1] is outcomes[0]
    else:
        assert np.array_equal(outcomes[0], outcomes[1])
    # without a template the 2D path works: y0 is the plain average of y
    assert_close(M.return_mean(y, x), ref.return_mean(y, x), 1e-15)
