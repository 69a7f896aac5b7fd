"""CPU-only checks of the host-side logic inside the library (no device calls)."""
import ctypes as C

import numpy as np


def _lib():
    from cosmogp_b200 import build, _lib
    build.build()
    return _lib


def test_uniform_grid_check():
    """The check applied to the CGP_GRID_UNIFORM hint: spacing uniform to a few ulp, l >= spacing > 0."""
    L = _lib()
    ok = lambda g, l: L.lib().cgp_grid_is_uniform(L.hptr(np.ascontiguousarray(g, dtype=np.float64)), len(g),
                                                 L.hptr(np.array([0.5, l])))
    g = np.linspace(-10, 40, 100)
    assert ok(g, 2.0) == 1 and ok(g, -2.0) == 1                  # the sign of l is irrelevant (kernel.py:71 squares it)
    assert ok(g[::-1].copy(), 2.0) == 1                          # descending grids are uniform too
    assert ok(g, 0.5) == 0                                       # l < spacing (0.505): anchors could underflow
    assert ok(g, float("nan")) == 0
    assert ok(np.arange(100) * 0.1 + 3.0, 1.0) == 1              # arange-style grids
    bent = g.copy(); bent[50] += 1e-12
    assert ok(bent, 2.0) == 0
    assert ok(np.sort(np.random.default_rng(0).uniform(0, 1, 50)), 2.0) == 0
    assert ok(np.array([1.0]), 2.0) == 0 and ok(np.array([1.0, 1.0]), 2.0) == 0      # fewer than two points, zero spacing
    assert ok(np.array([0.0, 1.0]), 2.0) == 1
    assert ok(np.array([0.0, np.inf]), 2.0) == 0


def test_streamer_chunk_schedule():
    """Chunk sizes of cgp_streamer_run: they cover the batch exactly, never exceed the buffers, ramp up and down."""
    L = _lib()

    def sched(n_obj, cap, n_pts=60):
        buf = np.zeros(4096, dtype=np.int64)
        k = L.lib().cgp_streamer_schedule(n_obj, cap, n_pts, L.hptr(buf), len(buf))
        assert 0 <= k <= len(buf)
        return buf[:k]

    for n_obj, cap in ((100000, 16667), (100000, 25000), (100000, 2500), (40001, 10001), (5003, 715), (1, 4096),
                       (0, 4096), (9000, 4096), (2049, 2048), (1000000, 50000)):
        s = sched(n_obj, cap)
        assert s.sum() == n_obj and (s > 0).all() and (len(s) == 0 or s.max() <= cap), (n_obj, cap, s)
    s = sched(100000, 16667)
    assert s[0] == 2048 and s[-1] == 2048 and list(s[:4]) == [2048, 3276, 5241, 8385]        # x1.6 up
    assert list(s[-3:]) == [8192, 4096, 2048]                                                  # x2 down
    assert (np.diff(s[:5]) > 0).all()
    assert len(set(sched(100000, 2500))) == 1                       # small buffers: equal chunks
    assert len(set(sched(100000, 16667, n_pts=100))) <= 2           # objects beyond the one-warp kernels: equal chunks
    assert L.lib().cgp_streamer_schedule(10, 0, 60, None, 0) == -1
    assert L.lib().cgp_streamer_schedule(100000, 16667, 60, None, 0) == len(s)


def test_shard_ranges_cover_and_balance():
    """cgp_shard_ranges (host only): contiguous ranges, every object exactly once, sum N^3 balanced."""
    from cosmogp_b200 import multi
    rng = np.random.default_rng(0)
    sizes = rng.integers(1, 200, 5000)
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    for parts in (1, 2, 3, 8):
        r = multi.shard_ranges(off, parts)
        assert r[0][0] == 0 and r[-1][1] == len(sizes) and all(r[i][1] == r[i + 1][0] for i in range(parts - 1))
        cost = [float((sizes[a:b].astype(float) ** 3).sum()) for a, b in r]
        assert max(cost) < 1.1 * sum(cost) / parts + 200.0 ** 3
    assert multi.shard_ranges(np.array([0]), 3) == [(0, 0)] * 3
    assert multi.shard_ranges(np.array([0, 5]), 4)[0] == (0, 1)


def test_reference_arm_times_the_unmodified_reference():
    """`bench.py --impl reference` (the CPU arm): a JSON line with impl == "reference" whose cpu_baseline says
    kind == "reference" exactly when the reference is installed (baseline/_ref, by baseline/fetch_ref.py) -- i.e. the
    numbers then come from the reference's own code -- and kind == "port" (the oracle restatement) otherwise."""
    import importlib.util, json, os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    from oracle import ref_loader
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--cpu-objects", "32"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    kind = "reference" if ref_loader.available() else "port"
    assert line["impl"] == "reference" and line["cpu_baseline"]["kind"] == kind and line["value"] > 0
    assert line["metric"] == "gp_fits_per_sec" and line["unit"] == "objects/s" and line["gpu_launches"] == 0
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["cpu_baseline"]["svd_method_true"]["value"] > 0
    # the installed copy under baseline/_ref is byte-identical to the source tree it was installed from when both are present
    spec = importlib.util.spec_from_file_location("fetch_ref", os.path.join(root, "baseline", "fetch_ref.py"))
    fetch_ref = importlib.util.module_from_spec(spec); spec.loader.exec_module(fetch_ref)
    ref_root, inst = os.path.join(fetch_ref.SOURCE, "cosmogp"), os.path.join(fetch_ref.TARGET, "cosmogp")
    if os.path.isdir(ref_root) and os.path.isdir(inst):
        for name in ("Gaussian_process.py", "kernel.py", "inv_matrix.py", "mean.py", "pull.py", "__init__.py"):
            assert open(os.path.join(ref_root, name), "rb").read() == open(os.path.join(inst, name), "rb").read(), name


def test_bench_dump_outputs(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float64 .npy files of the step's outputs, all objects or a seeded sample of them that
    is the same from run to run, within 64 MB at the workload's size; bad arguments are refused before any work."""
    import os, subprocess, sys
    import torch
    import bench
    assert bench.DUMP_OBJECTS * (2 + 2 * bench.M_GRID) * 8 <= 64 * 2 ** 20
    rng = np.random.default_rng(3)
    b, m = 50, bench.M_GRID
    ll, mean, var = (torch.from_numpy(rng.standard_normal(k)) for k in (b, b * m, b * m))
    monkeypatch.setattr(bench, "DUMP_OBJECTS", 16)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), ll, mean, var)
    got = {n: np.load(tmp_path / "a" / (n + ".npy")) for n in ("objects", "ll", "mean", "var")}
    assert all(a.dtype == np.float64 for a in got.values())
    assert all(np.array_equal(a, np.load(tmp_path / "b" / (n + ".npy"))) for n, a in got.items())
    idx = got["objects"].astype(np.int64)
    assert len(idx) == 16 and len(set(idx)) == 16 and (np.diff(idx) > 0).all()
    assert np.array_equal(got["ll"], ll.numpy()[idx])
    assert np.array_equal(got["mean"], mean.numpy().reshape(b, m)[idx]) and np.array_equal(got["var"], var.numpy().reshape(b, m)[idx])
    monkeypatch.setattr(bench, "DUMP_OBJECTS", 64)
    bench.dump_outputs(str(tmp_path / "c"), ll, mean, var)
    assert np.array_equal(np.load(tmp_path / "c" / "objects.npy"), np.arange(b))
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for bad in (["--steps", "0"], ["--workload", "c5", "--dump-outputs", str(tmp_path / "d")]):
        r = subprocess.run([sys.executable, os.path.join(root, "bench.py")] + bad, capture_output=True, text=True, timeout=120)
        assert r.returncode == 2 and "error" in r.stderr
    assert not (tmp_path / "d").exists()


def test_pack_csr_fast_path_equals_per_object_conversion():
    """pack_csr (what the facade does with the reference's lists of per-object arrays, Gaussian_process.py:156-169)
    skips the per-object conversion when every element already is an ndarray of the right rank; both routes must give
    the same flat float64 array and int64 offsets for ragged, empty, list-valued, float32, integer and xy-flat inputs."""
    from cosmogp_b200.batch import pack_csr, _as_list_of_arrays

    def slow(seq, dim):
        arrs = _as_list_of_arrays(seq, dim)
        off = np.zeros(len(arrs) + 1, dtype=np.int64)
        if not arrs:
            return np.zeros((0, 2) if dim == 2 else (0,)), off
        off[1:] = np.cumsum([len(a) for a in arrs])
        return np.ascontiguousarray(np.concatenate(arrs), dtype=np.float64), off

    rng = np.random.default_rng(0)
    cases = [
        ([rng.standard_normal(n) for n in rng.integers(0, 70, 300)], 1),
        ([rng.standard_normal((n, 2)) for n in rng.integers(0, 70, 300)], 2),
        ([list(rng.standard_normal(n)) for n in rng.integers(1, 9, 40)], 1),
        ([rng.standard_normal(n).astype(np.float32) for n in rng.integers(1, 9, 40)], 1),
        ([rng.standard_normal((2 * n, 2))[::2] for n in rng.integers(1, 9, 40)], 2),        # non-contiguous views
        ([rng.standard_normal(2 * n) for n in rng.integers(1, 9, 40)], 2),                  # flat xy pairs
        ([], 1), ([], 2),
        (tuple(rng.standard_normal(n) for n in (3, 4)), 1),
        ([rng.integers(0, 5, 4) for _ in range(3)], 1),
    ]
    for seq, dim in cases:
        flat, off = pack_csr(seq, dim)
        rf, ro = slow(seq, dim)
        assert flat.dtype == np.float64 and flat.flags.c_contiguous and off.dtype == np.int64
        assert flat.shape == rf.shape and np.array_equal(flat, rf) and np.array_equal(off, ro)
    # an iterator and a list-like view are accepted like a list
    from cosmogp_b200.batch import RaggedView
    arrs = [rng.standard_normal(n) for n in (3, 0, 5)]
    ref = pack_csr(arrs, 1)
    for alt in ((a for a in arrs), RaggedView(ref[0], ref[1])):
        f, o = pack_csr(alt, 1)
        assert np.array_equal(f, ref[0]) and np.array_equal(o, ref[1])
    # equal-length objects handed over as one ndarray
    x = rng.standard_normal((5, 7)); f, o = pack_csr(x, 1)
    assert np.array_equal(f, x.ravel()) and np.array_equal(o, np.arange(6) * 7)


def test_size_split():
    """batch.SizeSplit, the one statement of which objects the shared-memory kernels take (at most 224 points): the mask,
    the large ids, max_n of the small objects, their maximal runs, their points and their CSR offsets alone."""
    from cosmogp_b200.batch import SizeSplit

    def check(sizes, large, runs):
        off = np.concatenate([[0], np.cumsum(sizes, dtype=np.int64)])
        s = SizeSplit(off)
        small = np.array([n <= 224 for n in sizes], dtype=bool)
        assert np.array_equal(s.small, small) and s.small.dtype == bool
        assert list(s.large) == large and s.runs == runs
        assert s.small_max_n == max([n for n in sizes if n <= 224], default=0)
        assert np.array_equal(s.points, np.repeat(small, np.asarray(sizes, dtype=np.int64)))
        assert s.small_off.dtype == np.int64
        assert list(s.small_off) == [0] + list(np.cumsum([n for n in sizes if n <= 224], dtype=np.int64))
        # every small object exactly once, in order, and the runs hold nothing else
        assert [i for a, b in runs for i in range(a, b)] == list(np.nonzero(small)[0])

    check([], [], [])
    check([5, 224, 60], [], [(0, 3)])                                       # all small: one run, max_n 224
    check([225, 400, 1000], [0, 1, 2], [])                                  # all large: no run, max_n 0
    check([300, 5, 7], [0], [(1, 3)])                                       # large first
    check([5, 7, 300], [2], [(0, 2)])                                       # large last
    check([5, 225, 226, 9, 224], [1, 2], [(0, 1), (3, 5)])                  # large ones adjacent; 224 small, 225 large
    check([0, 225, 3, 400, 0], [1, 3], [(0, 1), (2, 3), (4, 5)])            # empty objects are small
    check([224], [], [(0, 1)])
    check([225], [0], [])
