"""Joint (shared-hyperparameter) likelihoods of batches with objects on the blocked path, on one GPU, four shapes:
  1d_60x1e4_400x8_template : 10^4 1D objects of 60 points plus 8 of 400, own epochs, a Mean_Y template
  2d_1000x256              : 256 2D objects of 1 000 points
  2d_2000x64               : 64 2D objects of 2 000 points
  1d_60x1e5_300x1          : 10^5 1D objects of 60 points plus one of 300
One large object sends the whole batch to the blocked path, so every object of each shape is factored there.  Per
shape: the wall time of one Gaussian_process.compute_log_likelihood by the grouped route (dense.log_likelihoods, one
cgp_large_ll_rows_dev call) against the per-object loop of dense.LargeObject.factor it replaces, alternated (on the two
shapes with the most objects the loop is timed on an evenly spaced subset and scaled by object count); the device time of
the grouped call alone (CUDA events) with model FLOPs sum n_pad^3 / 3 over the DMMA ceiling cgp_fp64_peak(1) measured in
this run; the wall time of a whole find_hyperparameters; and bitwise equality of every timed grouped output with the
loop's.  Writes profiles/bench_joint_fit_r01.json.
   python tests/perf_joint_fit.py [--out profiles/bench_joint_fit_r01.json]"""
import argparse, json, os, subprocess, sys, time, zlib
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import cosmogp_b200 as cg
from cosmogp_b200 import _lib, dense

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_joint_fit_r01.json"))
args = ap.parse_args()

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
peak = _lib.fp64_peak(1)
out = {"gpu": smi[0] if smi else torch.cuda.get_device_name(), "dmma_peak_tflops_measured": peak,
       "flop_model": "per object, on the padded size the kernels run: n_pad^3/3 (the blocked factorisation)",
       "workspace_bytes_cap": dense.LL_WS_BYTES, "shapes": {}}


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


def wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, r


def shape(name, dim, sizes, subset, template=False, reps=3):
    """subset: the objects the loop is timed on (None: all of them)."""
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    B = len(sizes)
    x, y, ye = make(rng, dim, sizes)
    kw = {}
    if template:
        tx = np.linspace(-5, 90, 80)
        kw = dict(Mean_Y=0.3 * np.cos(tx / 7), Time_mean=tx)
    kern = "RBF1D" if dim == 1 else "RBF2D"
    hyp = np.array([0.8, 1.5]) if dim == 1 else np.array([1.0, 4.0, 3.0, 1.0])
    gp = cg.gaussian_process_nobject(y, x, y_err=ye, kernel=kern, **kw)
    gp.nugget = 0.02
    assert gp._any_large
    r = {"objects": B, "points": sorted(set(int(n) for n in sizes)), "dim": dim, "mean_template": template,
         "sum_npad2_factor_bytes": int(8 * sum(pad(n) ** 2 for n in sizes))}

    # the route the facade took before: one LargeObject per object, kept, factor() each, summed left to right
    sub = np.arange(B) if subset is None else np.asarray(subset)
    objs = [dense.LargeObject(*gp._object_slices(int(i)), dim=dim, flags=gp.flags) for i in sub]

    def loop():
        lls = np.array([o.factor(hyp, gp.nugget) for o in objs])
        return lls, float(np.add.accumulate(lls)[-1])

    def grouped():
        gp.compute_log_likelihood(hyp, svd_method=False)
        return np.array(gp.log_likelihood_per_object), float(gp.log_likelihood[0])

    (_, (g_ll, g_tot)), (_, (l_ll, l_tot)) = wall(grouped), wall(loop)         # warm-up: first launches, allocator
    tg, tl = [], []
    for _ in range(reps):                                                     # alternated
        t, (g_ll, g_tot) = wall(grouped); tg.append(t * 1e3)
        t, (l_ll, l_tot) = wall(loop); tl.append(t * 1e3)
    same = bool(np.array_equal(g_ll[sub], l_ll))
    if subset is None:
        same &= g_tot == l_tot
    assert same, name + ": grouped likelihoods differ from the LargeObject loop"
    r["bitwise_grouped_equals_loop_on_timed_objects"] = same
    r["compute_log_likelihood_ms"] = sorted(tg)
    r["loop_ms_timed"] = sorted(tl)
    r["loop_timed_objects"] = int(len(sub))
    r["loop_ms_scaled"] = float(np.median(tl)) * B / len(sub)
    r["loop_note"] = ("all %d objects timed" % B if subset is None else
                      "%d of %d objects timed (evenly spaced, every large object included), scaled by object count"
                      % (len(sub), B))
    r["speedup_vs_loop"] = r["loop_ms_scaled"] / float(np.median(tg))
    del objs
    torch.cuda.empty_cache()

    # the grouped call alone on the device: cgp_large_ll_rows_dev on the facade's batch and workspace
    batch, work = gp._blocked
    L = _lib.lib()
    rows = np.ascontiguousarray(np.broadcast_to(hyp, (B, len(hyp))))
    nug = np.full(B, gp.nugget)
    ll_d = torch.empty(B, dtype=torch.float64, device=batch.device)
    info_d = torch.empty(B, dtype=torch.int32, device=batch.device)

    def call():
        _lib.check(L.cgp_large_ll_rows_dev(batch.n_obj, _lib.hptr(batch.off_host), dim, batch.x.data_ptr(),
                                           batch.y.data_ptr(), None if batch.y0 is None else batch.y0.data_ptr(),
                                           batch.y_err.data_ptr(), _lib.hptr(rows), _lib.hptr(nug), 0.0, 0.0, 0, None, B,
                                           ll_d.data_ptr(), info_d.data_ptr(), work.data_ptr(), int(work.numel()),
                                           batch._stream()), "cgp_large_ll_rows_dev")
    call(); torch.cuda.synchronize()
    te = []
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); call(); e1.record(); e1.synchronize()
        te.append(e0.elapsed_time(e1))
    assert np.array_equal(ll_d.cpu().numpy(), g_ll) and not info_d.cpu().numpy().any()
    flops = sum(pad(n) ** 3 / 3.0 for n in sizes)
    t = float(np.median(te)) * 1e-3
    r["device_ms"] = sorted(te)
    r["model_tflop"] = flops * 1e-12
    r["tflops"] = flops / t * 1e-12
    r["frac_of_dmma_peak"] = flops / t * 1e-12 / peak
    r["workspace_bytes"] = int(work.numel() * 8)

    fit = cg.gaussian_process_nobject(y, x, y_err=ye, kernel=kern, **kw)
    fit.hyperparameters = hyp.copy()
    n0 = [0]
    inner = fit.compute_log_likelihood

    def counted(*a, **k):
        n0[0] += 1
        return inner(*a, **k)
    fit.compute_log_likelihood = counted
    try:
        t, _ = wall(lambda: fit.find_hyperparameters(svd_method=False))
        r["find_hyperparameters_s"] = t
        r["find_hyperparameters_evaluations"] = n0[0]
        r["fitted_hyperparameters"] = [float(v) for v in fit.hyperparameters]
    except np.linalg.LinAlgError as e:
        r["find_hyperparameters_s"] = None
        r["find_hyperparameters_note"] = "stopped at a non-positive-definite trial point: %s" % e
    out["shapes"][name] = r
    print(name, json.dumps(r), flush=True)
    del gp, fit, batch, work
    torch.cuda.empty_cache()


s1 = [60] * 10000
for i in np.linspace(0, 10000, 8).astype(int):
    s1.insert(int(i), 400)
big1 = [i for i, n in enumerate(s1) if n == 400]
shape("1d_60x1e4_400x8_template", 1, s1, sorted(set(list(range(0, len(s1), 20)) + big1)), template=True)
shape("2d_1000x256", 2, [1000] * 256, None)
shape("2d_2000x64", 2, [2000] * 64, None)
s4 = [60] * 100000
s4.insert(50000, 300)
shape("1d_60x1e5_300x1", 1, s4, sorted(set(list(range(0, len(s4), 100)) + [50000])))

os.makedirs(os.path.dirname(args.out), exist_ok=True)
with open(args.out, "w") as f:
    json.dump(out, f, indent=1)
print("wrote", args.out)
