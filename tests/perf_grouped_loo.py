"""Grouped leave-one-out pulls on the blocked path (dense.loo_grouped -> cgp_large_loo_objhyp_dev) on one GPU, five shapes:
  1d_300_objhyp      : 10^4 1D objects of 300 points, per-object rows and nuggets
  2d_1000_shared     : 256 2D objects of 1 000 points, shared hyperparameters
  c5_mixed           : 10^5 1D objects of 40 points plus 1 000 of 225..600 points, shared hyperparameters
  2d_2000_shared     : 8 2D objects of 2 000 points, shared hyperparameters
  c4_single_20000    : the C4 recipe, one 2D object of 20 000 points
Per shape: the device time of the grouped call over the large objects (CUDA events, the workspace and chunk_rows
dense.loo_grouped chooses) and of the dense.LargeLoo loop it replaces (timed on a stated subset where the whole loop would
take long, and extrapolated), both alternated in this run; model FLOPs sum 2 n_pad^3 / 3 (factorisation and diag(K^-1)) over
the DMMA ceiling cgp_fp64_peak(1) measured in this run; the wall time of build_pull.compute_pull over the whole batch; and
bitwise equality of every timed output of the grouped call with the loop's.  Writes profiles/bench_grouped_loo_r01.json.
   python tests/perf_grouped_loo.py [--out profiles/bench_grouped_loo_r01.json]"""
import argparse, json, os, subprocess, sys, time, zlib
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import cosmogp_b200 as cg
from cosmogp_b200 import _lib, dense
from cosmogp_b200.batch import DeviceBatch, SizeSplit, pack_csr

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_grouped_loo_r01.json"))
args = ap.parse_args()

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
peak = _lib.fp64_peak(1)
out = {"gpu": smi[0] if smi else torch.cuda.get_device_name(), "dmma_peak_tflops_measured": peak,
       "flop_model": "per large object, on the padded size the kernels run: 2 n_pad^3/3 (factorisation n_pad^3/3, "
                     "diag(K^-1) by the blocked solve on identity rows n_pad^3/3)",
       "mode": "CGP_LOO_PLAIN (mode A)", "shapes": {}}
dev = torch.device("cuda", torch.cuda.current_device())


def pad(v):
    return max((int(v) + 127) // 128, 1) * 128


def make(rng, dim, sizes):
    if dim == 1:
        x = [np.sort(rng.uniform(0, n / 5.0, n)) for n in sizes]
        y = [np.sin(v) + 0.2 * rng.standard_normal(len(v)) for v in x]
    else:
        x = [rng.uniform(0, 3.0 * np.sqrt(n), (n, 2)) for n in sizes]
        y = [np.sin(v[:, 0] / 5) * np.cos(v[:, 1] / 4) + 0.2 * rng.standard_normal(len(v)) for v in x]
    return x, y, [rng.uniform(0.1, 0.3, n) for n in sizes]


def loop(batch, ids, hyp, nug, outs):
    """the per-object reference: one LargeLoo sized for the largest object of the call, run on each object in turn"""
    off = batch.off_host
    all_large = SizeSplit(off).large
    loo = dense.LargeLoo(int((off[all_large + 1] - off[all_large]).max()), batch.dim)
    h, g = np.asarray(hyp, dtype=float), np.asarray(nug, dtype=float)
    for i in ids:
        p0, p1 = int(off[i]), int(off[i + 1])
        x, y, m, e = (None if t is None else t[p0:p1] for t in (batch.x, batch.y, batch.y0, batch.y_err))
        loo.run(x, y, m, e, h[i] if h.ndim == 2 else h, g[i] if g.ndim == 1 else g, _lib.CGP_LOO_PLAIN, outs[4][i:i + 1],
                [o[p0:p1] for o in outs[:4]])


def events(fn, reps):
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    return ts


def shape(name, dim, sizes, per_object, subset, reps=3, pull_reps=3):
    """subset: the large objects the loop is timed on (None: all of them)."""
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    B = len(sizes)
    x, y, ye = make(rng, dim, sizes)
    if per_object:
        hyp = (np.column_stack([rng.uniform(0.6, 1.2, B), rng.uniform(1.0, 2.0, B)]) if dim == 1 else
               np.column_stack([rng.uniform(0.8, 1.2, B), rng.uniform(3.5, 4.5, B), rng.uniform(2.5, 3.5, B),
                                rng.uniform(0.5, 1.5, B)]))
        nug = rng.uniform(0.01, 0.05, B)
    else:
        hyp, nug = (np.array([0.8, 1.5]) if dim == 1 else np.array([1.0, 4.0, 3.0, 1.0])), 0.02
    xf, off = pack_csr(x, dim)
    split = SizeSplit(off)
    large = split.large
    n_large = off[large + 1] - off[large]
    r = {"objects": B, "large_objects": len(large), "large_points": sorted(set(int(n) for n in n_large))
         if len(set(n_large)) < 4 else [int(n_large.min()), int(n_large.max())], "dim": dim,
         "hyperparameters": "per-object rows" if per_object else "shared"}
    batch = DeviceBatch(xf, pack_csr(y, 1)[0], off, y_err=pack_csr(ye, 1)[0], dim=dim, max_n=split.small_max_n)
    n_pts = int(off[-1])
    mk = lambda: [torch.full((n_pts,), np.nan, dtype=torch.float64, device=dev) for _ in range(4)] + \
        [torch.full((B,), -7, dtype=torch.int32, device=dev)]
    hl = np.asarray(hyp)[large] if per_object else hyp
    nl = np.asarray(nug)[large] if per_object else nug
    g_outs, l_outs = mk(), mk()
    sub = large if subset is None else np.asarray(subset)
    grouped = lambda: dense.loo_grouped(batch, large, hl, nl, _lib.CGP_LOO_PLAIN, g_outs)
    looped = lambda: loop(batch, sub, hyp, nug, l_outs)
    grouped(); looped(); torch.cuda.synchronize()            # warm-up: first launches, allocator
    tg, tl = [], []
    for _ in range(reps):                                    # alternated
        tg += events(grouped, 1)
        tl += events(looped, 1)
    flops = sum(2.0 * pad(n) ** 3 / 3.0 for n in n_large)
    t = float(np.median(tg)) * 1e-3
    r["grouped_ms"] = sorted(tg)
    r["grouped_ms_median"] = t * 1e3
    r["model_tflop"] = flops * 1e-12
    r["tflops"] = flops / t * 1e-12
    r["frac_of_dmma_peak"] = flops / t * 1e-12 / peak
    r["loop_ms_timed"] = sorted(tl)
    r["loop_timed_objects"] = int(len(sub))
    r["loop_ms_extrapolated"] = float(np.median(tl)) * len(large) / len(sub)
    r["loop_note"] = ("all %d large objects timed" % len(large) if subset is None else
                      "%d of %d large objects timed, extrapolated by count" % (len(sub), len(large)))
    r["speedup_vs_loop"] = r["loop_ms_extrapolated"] / r["grouped_ms_median"]
    pts = np.concatenate([np.arange(off[i], off[i + 1]) for i in sub])
    same = all(np.array_equal(a.cpu().numpy()[pts], b.cpu().numpy()[pts], equal_nan=False) for a, b in zip(g_outs[:4], l_outs[:4]))
    same &= bool(np.array_equal(g_outs[4].cpu().numpy()[sub], l_outs[4].cpu().numpy()[sub]))
    assert same, name + ": grouped outputs differ from the LargeLoo loop"
    assert not g_outs[4].cpu().numpy()[large].any()
    r["bitwise_grouped_equals_loop_on_timed_objects"] = same
    del g_outs, l_outs, batch
    torch.cuda.empty_cache()

    def pull():
        bp = cg.build_pull(y, x, hyp, nugget=nug, y_err=ye, kernel="RBF1D" if dim == 1 else "RBF2D")
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        bp.compute_pull(svd_method=False)
        torch.cuda.synchronize()
        return time.perf_counter() - t0
    pull()
    r["compute_pull_s"] = sorted(pull() for _ in range(pull_reps))
    out["shapes"][name] = r
    print(name, json.dumps(r), flush=True)


shape("1d_300_objhyp", 1, [300] * 10000, True, list(range(0, 10000, 50)))
shape("2d_1000_shared", 2, [1000] * 256, False, list(range(0, 256, 4)))
rng = np.random.default_rng(5)
sizes5 = [40] * 100000
big5 = [int(v) for v in np.linspace(0, 100999, 1000)]
for i, n in zip(sorted(big5), rng.integers(225, 601, 1000)):
    sizes5.insert(i, int(n))
shape("c5_mixed", 1, sizes5, False, [i for i in sorted(big5)][::10])
shape("2d_2000_shared", 2, [2000] * 8, False, None)
shape("c4_single_20000", 2, [20000], False, None, reps=5, pull_reps=2)

os.makedirs(os.path.dirname(args.out), exist_ok=True)
with open(args.out, "w") as f:
    json.dump(out, f, indent=1)
print("wrote", args.out)
