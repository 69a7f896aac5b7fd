"""bench.py --dump-outputs on the device: the files hold the timed step's outputs for the seeded C2 workload, checked
against the oracle on a few objects."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import assert_close

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_dump_outputs_are_the_step_outputs(tmp_path):
    import bench
    from cosmogp_b200 import mean as M
    from oracle import gp_oracle as O
    b, d = 4096, tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--objects", str(b), "--steps", "2", "--no-cpu",
                        "--dump-outputs", str(d)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    got = {n: np.load(d / (n + ".npy")) for n in ("objects", "ll", "mean", "var")}
    assert np.array_equal(got["objects"], np.arange(b))             # fewer objects than the sample size: all of them
    assert got["ll"].shape == (b,) and got["mean"].shape == got["var"].shape == (b, bench.M_GRID)
    # the same inputs as the benchmark's rank 0: seeded workload, shared mean template plus one offset per object
    x, y, ye, tmean, ymean = bench.make_c2(b, 2)
    off = np.arange(b + 1, dtype=np.int64) * bench.N_EPOCH
    y0, diff = M.batched_mean(x.ravel(), y.ravel(), off, 1, ymean, tmean, None)
    y0 = y0.reshape(b, bench.N_EPOCH)
    grid = np.linspace(-10, 40, bench.M_GRID)
    ny0 = M.template_on_grid(grid, 1, ymean, tmean)[None, :] + diff[:, None]
    sel = np.array([0, 1, 777, 2048, b - 1])
    ll = O.ll_batched_1d(x[sel], y[sel], y0[sel], ye[sel], bench.HYP, bench.NUGGET)
    mean, var = O.predict_batched_1d(x[sel], y[sel], y0[sel], ye[sel], bench.HYP, bench.NUGGET, grid, ny0[sel])
    assert_close(got["ll"][sel], ll, 1e-9, what="ll")
    assert_close(got["mean"][sel], mean, 1e-9, what="mean")
    assert_close(got["var"][sel], var, 1e-9, what="var")
