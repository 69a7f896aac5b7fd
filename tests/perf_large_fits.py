"""Per-object fits of large objects on one GPU: one likelihood evaluation of K objects of N points through the grouped
entry point (cgp_large_ll_objhyp_dev) against a loop of dense.LargeObject.factor, K in {1, 8, 64}, N in {300, 1000,
2000}, 1D and 2D; a whole per-object fit of 64 2D objects of 2000 points, with the time the loop would take for the
same evaluation count; a torch.profiler kernel breakdown of one grouped evaluation at K = 64, N = 1000.
Writes profiles/bench_large_fits_r01.json.
   python tests/perf_large_fits.py [--out profiles/bench_large_fits_r01.json] [--skip-fit]"""
import argparse, json, os, subprocess, sys, time
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import cosmogp_b200 as cg
from cosmogp_b200 import _lib, dense
from cosmogp_b200.batch import DeviceBatch, pack_csr

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_large_fits_r01.json"))
ap.add_argument("--skip-fit", action="store_true")
args = ap.parse_args()

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
out = {"gpu": smi[0] if smi else torch.cuda.get_device_name(), "dmma_peak_tflops": _lib.fp64_peak(1),
       "flops_convention": "K N^3 / 3 per evaluation (the factorisation)", "evaluation": []}


def objects(rng, k, n, dim):
    xs, ys, ye = [], [], []
    for _ in range(k):
        if dim == 1:
            x = np.sort(rng.uniform(0, n / 5.0, n)); y = np.sin(x) + 0.2 * rng.standard_normal(n)
        else:                                         # C3 recipe
            x = rng.uniform(-200, 200, (n, 2)); y = np.sin(x[:, 0] / 60) * np.cos(x[:, 1] / 45) + 0.2 * rng.standard_normal(n)
        xs.append(x); ys.append(y); ye.append(np.full(n, 0.2))
    return xs, ys, ye


def hyp_of(dim):
    return [0.8, 1.5] if dim == 1 else [1.0, 30.0, 25.0, 50.0]


def timed(fn, reps):
    fn(); torch.cuda.synchronize()
    best = 1e30
    for _ in range(3):
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        best = min(best, (time.perf_counter() - t0) / reps)
    return best


def grouped_call(k, n, dim, rng):
    xs, ys, ye = objects(rng, k, n, dim)
    xf, off = pack_csr(xs, dim)
    b = DeviceBatch(xf, pack_csr(ys)[0], off, y_err=pack_csr(ye)[0], dim=dim)
    hyp = torch.tensor(np.tile(hyp_of(dim), (k, 1)), dtype=torch.float64, device=b.device)
    need = k * int(_lib.lib().cgp_large_ll_ws_doubles(n))
    work = torch.empty(need, dtype=torch.float64, device=b.device)
    ll = torch.empty(k, dtype=torch.float64, device=b.device); info = torch.empty(k, dtype=torch.int32, device=b.device)
    order = np.arange(k, dtype=np.int32)
    st = torch.cuda.current_stream().cuda_stream
    L = _lib.lib()

    def run():
        _lib.check(L.cgp_large_ll_objhyp_dev(k, _lib.hptr(b.off_host), dim, b.x.data_ptr(), b.y.data_ptr(), None,
                                             b.y_err.data_ptr(), hyp.data_ptr(), None, 0.0, 0.0, 0, order.ctypes.data, k,
                                             ll.data_ptr(), info.data_ptr(), work.data_ptr(), need, st),
                   "cgp_large_ll_objhyp_dev")
    los = [dense.LargeObject(xs[i], ys[i], ye[i], dim=dim) for i in range(k)]

    def loop():
        for o in los:
            o.factor(hyp_of(dim))
    run(); torch.cuda.synchronize()
    ref = np.array([o.factor(hyp_of(dim)) for o in los])
    got = ll.cpu().numpy()
    return run, loop, float(np.max(np.abs(got - ref) / np.abs(ref)))


rng = np.random.default_rng(0)
peak = out["dmma_peak_tflops"]
for dim in (1, 2):
    for n in (300, 1000, 2000):
        for k in (1, 8, 64):
            run, loop, rel = grouped_call(k, n, dim, rng)
            reps = max(1, int(64 // k))
            tg = timed(run, reps * 4)
            tl = timed(loop, reps)
            fl = k * n ** 3 / 3.0
            row = {"dim": dim, "n": n, "k": k, "grouped_ms": tg * 1e3, "loop_ms": tl * 1e3, "speedup": tl / tg,
                   "grouped_tflops": fl / tg * 1e-12, "loop_tflops": fl / tl * 1e-12,
                   "grouped_frac_of_dmma_peak": fl / tg * 1e-12 / peak, "max_rel_diff_vs_loop": rel}
            out["evaluation"].append(row)
            print(json.dumps(row), flush=True)

# kernel breakdown of one grouped evaluation, K = 64, N = 1000, 2D (profiler in a run of its own)
run, _, _ = grouped_call(64, 1000, 2, rng)
run(); torch.cuda.synchronize()
with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
    for _ in range(5):
        run()
    torch.cuda.synchronize()
kern = {}
for e in prof.key_averages():
    us = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
    if us > 0:
        kern[e.key[:90]] = {"us_per_eval": us / 5.0, "calls_per_eval": e.count / 5.0}
out["profile_k64_n1000_2d"] = dict(sorted(kern.items(), key=lambda kv: -kv[1]["us_per_eval"])[:12])

if not args.skip_fit:
    k, n = 64, 2000
    xs, ys, ye = objects(np.random.default_rng(1), k, n, 2)
    gp = cg.gaussian_process_nobject(ys, xs, y_err=ye, kernel='RBF2D')
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    gp.find_hyperparameters_per_object(hyperparameter_guess=hyp_of(2))
    wall = time.perf_counter() - t0
    lo = dense.LargeObject(xs[0], ys[0], ye[0], dim=2)
    t_one = timed(lambda: lo.factor(hyp_of(2)), 5)
    ev = gp.fit_evaluations
    out["fit_64x2000_2d"] = {"wall_s": wall, "evaluations_mean": float(ev.mean()), "evaluations_max": int(ev.max()),
                             "iterations_mean": float(gp.fit_iterations.mean()), "largeobject_factor_ms": t_one * 1e3,
                             "loop_estimate_s": float(ev.sum()) * t_one, "finite": bool(np.isfinite(gp.log_likelihood_per_object).all())}
    print(json.dumps(out["fit_64x2000_2d"]), flush=True)

os.makedirs(os.path.dirname(args.out), exist_ok=True)
with open(args.out, "w") as f:
    json.dump(out, f, indent=1)
print("wrote", args.out)
