"""Grouped leave-one-out pulls of objects on the blocked path (cgp_large_loo_objhyp_dev, dense.loo_grouped): bit for
bit dense.LargeLoo.run of each object alone at the same chunk_rows, whatever the order, the waves and the other objects
of the call; launch counts that do not grow with the number of objects; failures that stay with their object; and
build_pull, whose large objects go through the grouped call, against a LargeLoo loop."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SENTINEL = 12345.0


@pytest.fixture(scope="module")
def cg():
    import cosmogp_b200
    from cosmogp_b200 import _lib
    _lib.require_device()
    return cosmogp_b200


def _object(rng, n, dim):
    """Seeded object with cond(K) of order 1e3 under the rows of _rows."""
    if dim == 1:
        x = np.sort(rng.uniform(0, n / 5.0, n))
        y = np.sin(x) + 0.2 * rng.standard_normal(n)
    else:
        x = rng.uniform(0, 3.0 * np.sqrt(n), (n, 2))
        y = np.sin(x[:, 0] / 5) * np.cos(x[:, 1] / 4) + 0.2 * rng.standard_normal(n)
    return x, y, rng.uniform(0.1, 0.3, n)


def _rows(rng, dim, k):
    if dim == 1:
        return np.column_stack([rng.uniform(0.6, 1.2, k), rng.uniform(1.0, 2.0, k)])
    return np.column_stack([rng.uniform(0.8, 1.2, k), rng.uniform(3.5, 4.5, k), rng.uniform(2.5, 3.5, k),
                            rng.uniform(0.5, 1.5, k)])


class Batch:
    """Objects on the device and direct calls of cgp_large_loo_objhyp_dev on them; row b of hyp / nug belongs to
    object b."""

    def __init__(self, sizes, dim, seed, with_m=True, with_err=True, flags=0, bad=()):
        import torch
        rng = np.random.default_rng(seed)
        self.dim, self.flags, self.sizes = dim, flags, list(sizes)
        objs = [_object(rng, n, dim) for n in sizes]
        self.x = [o[0] for o in objs]
        self.y = [o[1] for o in objs]
        self.ye = [o[2] for o in objs] if with_err else None
        self.m = [0.1 * rng.standard_normal(n) for n in sizes] if with_m else None
        self.hyp = _rows(rng, dim, len(sizes))
        self.nug = rng.uniform(0.0, 0.05, len(sizes)) if with_err else rng.uniform(0.1, 0.3, len(sizes))
        for b in bad:                       # duplicate epochs, no noise: not positive definite
            n = sizes[b]
            self.x[b] = np.repeat(np.linspace(0, 10, n // 2), 2) if dim == 1 else np.repeat(rng.uniform(0, 10, (n // 2, 2)), 2, 0)
            if with_err:
                self.ye[b] = np.zeros(n)
            self.hyp[b] = [1.0, 1.0] if dim == 1 else [1.0, 1.0, 1.0, 0.0]
            self.nug[b] = 0.0
        self.off = np.zeros(len(sizes) + 1, dtype=np.int64)
        np.cumsum(sizes, out=self.off[1:])
        self.dev = torch.device("cuda", torch.cuda.current_device())

        def up(parts):
            return None if parts is None else torch.from_numpy(np.ascontiguousarray(np.concatenate(parts)).reshape(-1)).to(self.dev)
        self.xd, self.yd, self.yed, self.md = up(self.x), up(self.y), up(self.ye), up(self.m)

    def chunk(self, ids=None):
        from cosmogp_b200 import dense
        return dense.loo_chunk_rows(dense.pad128(max(self.sizes[b] for b in (ids if ids is not None else range(len(self.sizes))))))

    def need(self, ids, chunk_rows):
        from cosmogp_b200 import dense
        return dense.loo_ws_doubles(np.asarray([self.sizes[b] for b in ids]), chunk_rows)

    def run(self, mode, order=None, chunk_rows=None, work_doubles=None, shared=None):
        """-> rc, (pred, pred_var, pull, resid) over all points (SENTINEL where not written), info (compact)"""
        import torch
        from cosmogp_b200 import _lib
        ids = list(range(len(self.sizes))) if order is None else list(order)
        chunk_rows = self.chunk(ids) if chunk_rows is None else chunk_rows
        if work_doubles is None:
            work_doubles = int(self.need(ids, chunk_rows).sum()) if ids else 2
        outs = [torch.full((int(self.off[-1]),), SENTINEL, dtype=torch.float64, device=self.dev) for _ in range(4)]
        info = torch.full((max(len(ids), 1),), -7, dtype=torch.int32, device=self.dev)
        work = torch.empty(max(int(work_doubles), 2), dtype=torch.float64, device=self.dev)
        if shared is None:
            hr, nr = np.ascontiguousarray(self.hyp[ids]), np.ascontiguousarray(self.nug[ids])
        else:
            hr, nr = np.ascontiguousarray(np.tile(np.asarray(shared[0], dtype=float), (len(ids), 1))), None
        o = None if order is None else np.ascontiguousarray(order, dtype=np.int32)
        p = lambda t: None if t is None else t.data_ptr()
        rc = _lib.lib().cgp_large_loo_objhyp_dev(
            len(self.sizes), _lib.hptr(self.off), self.dim, p(self.xd), p(self.yd), p(self.md), p(self.yed), _lib.hptr(hr),
            _lib.hptr(nr), 0.0 if shared is None else float(shared[1]), 0.0, self.flags, int(mode), _lib.hptr(o), len(ids),
            p(info), *[p(t) for t in outs], int(chunk_rows), p(work), int(work_doubles),
            torch.cuda.current_stream(self.dev).cuda_stream)
        torch.cuda.synchronize()
        return rc, [t.cpu().numpy() for t in outs], info.cpu().numpy()[:len(ids)]

    def ref(self, b, mode, chunk_rows, hyp=None, nug=None):
        """object b alone through dense.LargeLoo.run -> host (pred, pred_var, pull, resid), info"""
        import torch
        from cosmogp_b200.dense import LargeLoo
        p0, p1 = int(self.off[b]), int(self.off[b + 1])
        sl = lambda t: None if t is None else t[p0:p1] if self.dim == 1 or t is not self.xd else t[2 * p0:2 * p1]
        outs = [torch.empty(p1 - p0, dtype=torch.float64, device=self.dev) for _ in range(4)]
        info = torch.full((1,), -7, dtype=torch.int32, device=self.dev)
        LargeLoo(p1 - p0, self.dim, flags=self.flags, chunk_rows=chunk_rows).run(
            sl(self.xd), sl(self.yd), sl(self.md), sl(self.yed), self.hyp[b] if hyp is None else hyp,
            self.nug[b] if nug is None else nug, mode, info, outs)
        return [t.cpu().numpy() for t in outs], int(info.item())

    def assert_matches_loop(self, got, info, mode, order=None, chunk_rows=None):
        ids = list(range(len(self.sizes))) if order is None else list(order)
        chunk_rows = self.chunk(ids) if chunk_rows is None else chunk_rows
        for j, b in enumerate(ids):
            want, wi = self.ref(b, mode, chunk_rows)
            assert info[j] == wi, "object %d: info %d vs %d" % (b, info[j], wi)
            s = slice(int(self.off[b]), int(self.off[b + 1]))
            for g, w, what in zip(got, want, ("pred", "pred_var", "pull", "resid")):
                np.testing.assert_array_equal(g[s], w, err_msg="%s of object %d (%d points)" % (what, b, self.sizes[b]))


SIZES = [225, 255, 256, 257, 383, 384, 385, 1000, 2000, 12, 60]


@pytest.mark.parametrize("extras", [True, False], ids=["m_and_yerr", "no_m_no_yerr"])
@pytest.mark.parametrize("mode", [0, 1], ids=["plain", "recenter"])
@pytest.mark.parametrize("dim", [1, 2])
def test_entry_bit_for_bit(cg, dim, mode, extras):
    bt = Batch(SIZES, dim, seed=100 * dim + 10 * mode + extras, with_m=extras, with_err=extras)
    rc, got, info = bt.run(mode)
    assert rc == 0 and not info.any()
    bt.assert_matches_loop(got, info, mode)


@pytest.mark.parametrize("mode", [0, 1], ids=["plain", "recenter"])
def test_entry_2d_amp_on_autocov(cg, mode):
    from cosmogp_b200 import _lib
    bt = Batch(SIZES, 2, seed=7 + mode, flags=_lib.CGP_AMP_ON_AUTOCOV)
    rc, got, info = bt.run(mode)
    assert rc == 0 and not info.any()
    bt.assert_matches_loop(got, info, mode)


def test_entry_shared_hyperparameters(cg):
    """A scalar nugget (nugget_rows NULL) with one row repeated: each object as LargeLoo with that row and nugget."""
    bt = Batch([300, 12, 700], 1, seed=9)
    rc, got, info = bt.run(1, shared=([0.9, 1.4], 0.03))
    assert rc == 0 and not info.any()
    for b in range(3):
        want, _ = bt.ref(b, 1, bt.chunk(), hyp=[0.9, 1.4], nug=0.03)
        s = slice(int(bt.off[b]), int(bt.off[b + 1]))
        for g, w in zip(got, want):
            np.testing.assert_array_equal(g[s], w)


@pytest.mark.parametrize("dim", [1, 2])
def test_order_and_wave_invariance(cg, dim):
    """Reversed and shuffled order lists, and a workspace of exactly the largest need (several waves), give the bits
    of one call over all objects in their own order."""
    bt = Batch(SIZES, dim, seed=31 + dim)
    rc, base, info = bt.run(1)
    assert rc == 0 and not info.any()
    ids = np.arange(len(SIZES))
    chunk = bt.chunk()
    rng = np.random.default_rng(dim)
    for order, wd in ((ids[::-1], None), (rng.permutation(ids), None), (None, int(bt.need(ids, chunk).max())),
                      (rng.permutation(ids), int(bt.need(ids, chunk).max()))):
        rc, got, inf = bt.run(1, order=order, chunk_rows=chunk, work_doubles=wd)
        assert rc == 0 and not inf.any()
        for g, w in zip(got, base):
            np.testing.assert_array_equal(g, w)


@pytest.mark.parametrize("chunk_rows", [128, 384])
def test_chunk_rows(cg, chunk_rows):
    """Passes of 128 and 384 identity rows over objects of 1 000 and 2 000 points (passes that start past the first
    block, run over several block-column pairs and end on an unpaired block) give LargeLoo's bits at that chunk_rows."""
    for dim, mode in ((1, 0), (2, 1)):
        bt = Batch([1000, 2000, 300, 1000], dim, seed=chunk_rows + dim)
        rc, got, info = bt.run(mode, chunk_rows=chunk_rows)
        assert rc == 0 and not info.any()
        bt.assert_matches_loop(got, info, mode, chunk_rows=chunk_rows)


def test_launch_count_does_not_grow_with_objects(cg):
    from cosmogp_b200 import _lib
    L = _lib.lib()
    counts = []
    for reps in (1, 8):
        bt = Batch([300, 700] * reps, 1, seed=reps)
        for mode in (0, 1):
            n0 = L.cgp_launch_count()
            rc, _, info = bt.run(mode)
            assert rc == 0 and not info.any()
            counts.append(L.cgp_launch_count() - n0)
    assert counts[0] == counts[2] and counts[1] == counts[3], counts


def test_failures_stay_local(cg):
    """A non-positive-definite object gets info != 0 and NaN outputs; the other objects keep the bits of a call without
    it; the points of objects not listed keep their values; no active object launches nothing; a short workspace is
    refused with nothing launched."""
    from cosmogp_b200 import _lib
    L = _lib.lib()
    sizes = [300, 12, 600, 400, 257]
    bt = Batch(sizes, 1, seed=5, bad=(2,))
    order = [4, 2, 0, 1]                                    # object 3 is not listed
    rc, got, info = bt.run(1, order=order)
    assert rc == 0
    assert info[1] != 0 and not info[[0, 2, 3]].any()
    s = slice(int(bt.off[2]), int(bt.off[3]))
    for g in got:
        assert np.isnan(g[s]).all()
        assert (g[int(bt.off[3]):int(bt.off[4])] == SENTINEL).all()
    rc, clean, inf = bt.run(1, order=[4, 0, 1])
    assert rc == 0 and not inf.any()
    for g, w in zip(got, clean):
        for b in (4, 0, 1):
            np.testing.assert_array_equal(g[int(bt.off[b]):int(bt.off[b + 1])], w[int(bt.off[b]):int(bt.off[b + 1])])
    want, wi = bt.ref(2, 1, bt.chunk(order))
    assert wi == info[1]
    n0 = L.cgp_launch_count()
    rc, empty, _ = bt.run(1, order=[], chunk_rows=128)
    assert rc == 0 and all((g == SENTINEL).all() for g in empty)
    rc, _, _ = bt.run(1, order=[0, 3], work_doubles=int(bt.need([0, 3], bt.chunk([0, 3])).max()) - 1)
    assert rc == -2 and "workspace" in _lib.last_error()
    assert L.cgp_launch_count() == n0


# ---- the facade
def _loop(batch, objects, hyp, nugget, mode, outs, flags=0, chunk_rows=None, work_doubles=None):
    """dense.loo_grouped's reference: one LargeLoo, sized for the largest object, run on each object in turn."""
    from cosmogp_b200.dense import LargeLoo
    ids = np.asarray(objects, dtype=np.int64)
    off = batch.off_host
    loo = LargeLoo(int((off[ids + 1] - off[ids]).max()), batch.dim, flags=flags, chunk_rows=chunk_rows)
    h, g = np.asarray(hyp, dtype=float), np.asarray(nugget, dtype=float)
    for j, i in enumerate(ids):
        p0, p1 = int(off[i]), int(off[i + 1])
        x, y, m, e = (None if t is None else t[p0:p1] for t in (batch.x, batch.y, batch.y0, batch.y_err))
        loo.run(x, y, m, e, h[j] if h.ndim == 2 else h, g[j] if g.ndim == 1 else g, mode, outs[4][i:i + 1],
                [o[p0:p1] for o in outs[:4]])


def _mixed(rng, n_small=300, large=(225, 600, 310, 480, 257, 384, 512, 450)):
    sizes = list(rng.integers(5, 225, n_small))
    for k, n in enumerate(large):
        sizes.insert(int((k + 1) * n_small / (len(large) + 1)) + k, n)
    objs = [_object(rng, n, 1) for n in sizes]
    return sizes, [o[0] for o in objs], [o[1] for o in objs], [o[2] for o in objs]


@pytest.mark.parametrize("per_object", [False, True], ids=["shared", "per_object"])
def test_build_pull_matches_loop(cg, monkeypatch, per_object):
    """build_pull over ~300 small objects and 8 large ones, modes A-D: every large object's outputs equal those of the
    same call with its large objects sent through a LargeLoo loop.  In modes A and C every output, pull_average and
    pull_std are equal too; in the recentred modes B and D the shared-memory kernel adds the small objects' residual
    sum with shared-memory atomics, so their outputs (and the moments over all pulls) can differ in the last bits
    from one call to the next, and are compared to 1e-12."""
    from cosmogp_b200 import dense
    rng = np.random.default_rng(11 + per_object)
    sizes, xs, ys, yes = _mixed(rng)
    b = len(sizes)
    if per_object:
        hyp = np.column_stack([rng.uniform(0.6, 1.2, b), rng.uniform(1.0, 2.0, b)])
        nug = rng.uniform(0.0, 0.05, b)
    else:
        hyp, nug = [0.8, 1.5], 0.02
    tx = np.linspace(-5, 200, 60)
    ty = 0.3 * np.cos(tx / 7.0)
    diff = rng.uniform(-0.2, 0.2, b)
    for name, ctor, call in (("A", {}, {}), ("B", dict(y_mean=ty, x_axis_mean=tx), {}),
                             ("C", dict(y_mean=ty, x_axis_mean=tx), dict(diff=diff)), ("D", {}, dict(substract_mean=True))):
        res = []
        for route in ("grouped", "loop"):
            with monkeypatch.context() as mp:
                if route == "loop":
                    mp.setattr(dense, "loo_grouped", _loop)
                bp = cg.build_pull(ys, xs, hyp, nugget=nug, y_err=yes, **ctor)
                bp.compute_pull(svd_method=False, **call)
                res.append((bp.pull, bp.residual, np.concatenate(list(bp.prediction)), bp.prediction_variance,
                            bp.pull_average, bp.pull_std))
        off = np.concatenate([[0], np.cumsum(sizes)])
        big = np.concatenate([np.arange(off[i], off[i + 1]) for i in range(b) if sizes[i] > 224])
        for g, w, what in zip(res[0], res[1], ("pull", "residual", "prediction", "prediction_variance", "pull_average",
                                               "pull_std")):
            if np.ndim(g):
                np.testing.assert_array_equal(g[big], w[big], err_msg="mode %s: %s of the large objects" % (name, what))
            if name in "AC":
                np.testing.assert_array_equal(g, w, err_msg="mode %s: %s" % (name, what))
            else:
                np.testing.assert_allclose(g, w, rtol=1e-12, atol=1e-15, err_msg="mode %s: %s" % (name, what))


def test_compute_pull_launch_count_does_not_grow(cg):
    from cosmogp_b200 import _lib
    L = _lib.lib()
    rng = np.random.default_rng(21)
    counts = []
    for reps in (2, 8):
        sizes = list(rng.integers(5, 225, 100)) + [300, 500] * reps      # the large objects last: one small-object run
        objs = [_object(rng, n, 1) for n in sizes]
        bp = cg.build_pull([o[1] for o in objs], [o[0] for o in objs], [0.8, 1.5], nugget=0.02, y_err=[o[2] for o in objs])
        n0 = L.cgp_launch_count()
        bp.compute_pull(svd_method=False)
        counts.append(L.cgp_launch_count() - n0)
    assert counts[0] == counts[1], counts
