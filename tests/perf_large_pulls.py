"""Leave-one-out pulls of large objects on one GPU: stage times (covariance build, blocked Cholesky, diag(K^-1),
vectors + epilogue) at N = 300, 1 000, 2 000 (2D, C3 recipe) and 20 000 (C4 recipe), compute_pull wall time, the
reference's brute force (N refits) timed on a few refits and extrapolated, and a mixed batch (C5 + eight 1D objects
of 2 000 points) against the C5 batch alone.  Writes profiles/bench_large_pulls_r01.json.
   python tests/perf_large_pulls.py [--c5 1000000] [--out profiles/bench_large_pulls_r01.json]"""
import argparse, json, os, subprocess, sys, time
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import cosmogp_b200 as cg
from cosmogp_b200 import _lib, dense
from oracle import gp_oracle as O, ref_loader

ap = argparse.ArgumentParser()
ap.add_argument("--c5", type=int, default=1000000)
ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_large_pulls_r01.json"))
args = ap.parse_args()

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
out = {"gpu": smi[0] if smi else torch.cuda.get_device_name(), "dmma_peak_tflops": _lib.fp64_peak(1),
       "flops_convention": "F = 2N^3/3 + 6N^2 (factor N^3/3 + diag(K^-1) N^3/3)", "sizes": []}


def ev(fn, reps=3):
    fn(); torch.cuda.synchronize(); best = 1e30
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize(); best = min(best, e0.elapsed_time(e1))
    return best


def recipe(n, rng):
    if n == 20000:                                   # C4 (test_c4_large_single_object_at_config_size)
        x = rng.uniform(0, 1000, (n, 2)); hyp = [1.0, 30.0, 30.0, 0.0]; ye = np.full(n, 0.3)
        y = np.sin(x[:, 0] / 90) * np.cos(x[:, 1] / 70) + 0.3 * rng.standard_normal(n)
    else:                                            # C3 recipe
        x = rng.uniform(-200, 200, (n, 2)); hyp = [1.0, 30.0, 25.0, 50.0]; ye = np.full(n, 0.2)
        y = np.sin(x[:, 0] / 60) * np.cos(x[:, 1] / 45) + 0.2 * rng.standard_normal(n)
    return x, y, ye, hyp


def refit_seconds(x, y, ye, hyp, reps):
    """one refit of the reference's build_pull loop (pull.py:66-90): a GP on N-1 points, predicted with its full
    covariance at the N epochs; the unmodified reference when its sources are present, else the oracle port"""
    from threadpoolctl import threadpool_limits
    n = len(y); ts = []
    with threadpool_limits(limits=1):
        for t in range(reps):
            keep = np.arange(n) != t
            t0 = time.perf_counter()
            if ref_loader.available():
                ref = ref_loader.load()
                with ref_loader.quiet():
                    gp = ref.gaussian_process(y[keep], x[keep], kernel="RBF2D", y_err=ye[keep])
                    gp.hyperparameters = np.array(hyp); gp.nugget = 0.0
                    gp.get_prediction(new_binning=x, COV=True, svd_method=False)
            else:
                O.predict(y[keep], x[keep], hyp, 0.0, x, y_err=ye[keep], kind="2d", svd_method=False)
            ts.append(time.perf_counter() - t0)
    return float(np.median(ts))


def categories(prof):
    cat = {"diag_inv": 0.0, "vectors": 0.0, "epilogue": 0.0, "other": 0.0}
    for e in prof.key_averages():
        us = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
        name = e.key
        if "gemm_nt" in name or "identity_rows" in name or "row_norm_var" in name:
            cat["diag_inv"] += us
        elif any(k in name for k in ("fwd_step", "bwd_step", "residual_kernel", "sum_kernel", "ones_kernel")):
            cat["vectors"] += us
        elif "loo_epilogue" in name:
            cat["epilogue"] += us
        elif "Memcpy" in name or "Memset" in name:
            cat["other"] += us
    return {k: v / 1e3 for k, v in cat.items()}


refit_2000 = None
for n in (300, 1000, 2000, 20000):
    rng = np.random.default_rng(n)
    x, y, ye, hyp = recipe(n, rng)
    dev = torch.device("cuda")
    xd, yd, ed = (torch.from_numpy(np.ascontiguousarray(v)).to(dev) for v in (x, y, ye))
    L = _lib.lib(); st = torch.cuda.current_stream().cuda_stream
    n_pad = dense.pad128(n); h = np.ascontiguousarray(hyp, dtype=np.float64)
    loo = dense.LargeLoo(n, 2)
    a = loo.a
    info = torch.zeros(1, dtype=torch.int32, device=dev)
    outs = [torch.empty(n, dtype=torch.float64, device=dev) for _ in range(4)]
    build = lambda: _lib.check(L.cgp_cov_matrix_dev(2, xd.data_ptr(), n, None, 0, ed.data_ptr(), h.ctypes.data, 0.0, 0.0, 0,
                                                    a.data_ptr(), n_pad, n_pad, n_pad, st), "build")
    factor = lambda: _lib.check(L.cgp_potrf_dev(a.data_ptr(), n_pad, n_pad, None, info.data_ptr(), st), "potrf")
    run_loo = lambda: _lib.check(L.cgp_large_loo_dev(a.data_ptr(), n, n_pad, n_pad, 2, yd.data_ptr(), None, ed.data_ptr(),
                                                     h.ctypes.data, 0.0, 0.0, 0, 0, info.data_ptr(), loo.vwork.data_ptr(),
                                                     loo.chunk, *[o.data_ptr() for o in outs], st), "loo")
    reps = 3 if n < 20000 else 2
    t_build = ev(build, reps)
    t_factor = ev(lambda: (build(), factor()), reps) - t_build      # potrf works in place: rebuild K before each
    build(); factor(); torch.cuda.synchronize()
    assert int(info.item()) == 0
    t_loo = ev(run_loo, reps)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        run_loo(); torch.cuda.synchronize()
    cat = categories(prof)
    # compute_pull end to end (host packing, upload, launches, info check, norm.fit)
    cg.build_pull([y], [x], hyp, y_err=[ye], kernel="RBF2D").compute_pull(svd_method=False)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    bp = cg.build_pull([y], [x], hyp, y_err=[ye], kernel="RBF2D"); bp.compute_pull(svd_method=False)
    wall = time.perf_counter() - t0
    # accuracy at the timed size: a few points against the host closed form (all of them up to N = 2 000)
    if n <= 2000:
        po = O.loo_closed_form(y, x, hyp, 0.0, ye, kind="2d")
        err = float(np.max(np.abs(bp.pull - po[2]) / (np.abs(po[2]) + 1e-8)))
    else:
        err = None
    if n <= 2000:
        per_refit = refit_seconds(x, y, ye, hyp, reps=2)
        bf = {"per_refit_s": per_refit, "n_refits_extrapolated_s": per_refit * n,
              "how": "timed %d refits, times N refits (extrapolation)" % 2}
        if n == 2000:
            refit_2000 = per_refit
    else:
        bf = {"per_refit_s": refit_2000 * (n / 2000.0) ** 3, "n_refits_extrapolated_s": refit_2000 * (n / 2000.0) ** 3 * n,
              "how": "not timed at this size: the N = 2000 refit scaled by (N/2000)^3, times N refits (extrapolation)"}
    bf["code"] = "unmodified reference (cosmogp.gaussian_process.get_prediction, COV=True)" if ref_loader.available() \
        else "oracle port of the reference's refit (oracle.gp_oracle.predict, full covariance); reference not installed"
    bf["cores"] = 1
    fl = 2.0 * n ** 3 / 3.0 + 6.0 * n ** 2
    diag_fl = n_pad ** 3 / 3.0
    out["sizes"].append({
        "n": n, "n_pad": n_pad, "recipe": "C4" if n == 20000 else "C3", "chunk_rows": loo.chunk,
        "build_ms": t_build, "factor_ms": t_factor, "loo_call_ms": t_loo,
        "diag_inv_kernels_ms": cat["diag_inv"], "vectors_kernels_ms": cat["vectors"], "epilogue_kernels_ms": cat["epilogue"],
        "diag_over_factor": cat["diag_inv"] / t_factor,
        "diag_inv_tflops": diag_fl / (cat["diag_inv"] * 1e-3) * 1e-12,
        "factor_plus_loo_tflops": fl / ((t_factor + t_loo) * 1e-3) * 1e-12,
        "factor_plus_loo_fraction_of_peak": fl / ((t_factor + t_loo) * 1e-3) * 1e-12 / out["dmma_peak_tflops"],
        "compute_pull_wall_ms": wall * 1e3, "max_rel_pull_err_vs_host_closed_form": err,
        "reference_bruteforce": bf})
    print(json.dumps(out["sizes"][-1]), flush=True)
    del loo, a, outs, xd, yd, ed
    torch.cuda.empty_cache()

# ---- mixed batch: C5 (10^6 x 40, tests/perf_configs.py recipe) plus eight 1D objects of 2 000 points
b, n = args.c5, 40
rng = np.random.default_rng(5)
x5 = np.sort(rng.uniform(-10, 10, (b, n)), axis=1); ye5 = np.full((b, n), 0.1)
y5 = 0.5 * np.sin(x5 / 2.0 + rng.uniform(0, 6.28, (b, 1))) + 0.1 * rng.standard_normal((b, n))
hyp, nug = [0.5, 2.0], 0.0
# epochs of the large objects spread over 400 units: about 40 points within a correlation length, so
# cond(K) ~ 1 + 40 sigma^2 / y_err^2 ~ 1e3
big = [np.sort(rng.uniform(0, 400, 2000)) for _ in range(8)]
ys, xs, yes = list(y5), list(x5), list(ye5)
for k, xb in enumerate(big):
    pos = (k + 1) * b // 9 + k
    xs.insert(pos, xb); ys.insert(pos, 0.5 * np.sin(xb / 2.0) + 0.1 * rng.standard_normal(2000)); yes.insert(pos, np.full(2000, 0.1))


def wall_pull(yy, xx, ee, reps=3):
    cg.build_pull(yy, xx, hyp, nugget=nug, y_err=ee).compute_pull(svd_method=False)
    torch.cuda.synchronize(); best = 1e30
    for _ in range(reps):
        t0 = time.perf_counter()
        cg.build_pull(yy, xx, hyp, nugget=nug, y_err=ee).compute_pull(svd_method=False)
        best = min(best, time.perf_counter() - t0)
    return best


# the same inputs in the same form: compute_pull packs a list of per-object arrays object by object (pack_csr), a 2D
# ndarray of equal-length objects with one reshape, so C5 is timed both ways and the mixed batch against the list form
w5_nd = wall_pull(y5, x5, ye5)
w5 = wall_pull(list(y5), list(x5), list(ye5))
wm = wall_pull(ys, xs, yes)
pos = [(k + 1) * b // 9 + k for k in range(8)]
w8 = wall_pull([ys[p] for p in pos], [xs[p] for p in pos], [yes[p] for p in pos])
t0 = time.perf_counter()
for seq, d in ((xs, 1), (ys, 1), (yes, 1)):
    cg.pack_csr(seq, d)
pack_mixed = time.perf_counter() - t0
out["mixed"] = {"c5_objects": b, "c5_n": n, "large_objects": 8, "large_n": 2000, "large_cond_estimate": "~1e3",
                "c5_alone_ndarray_compute_pull_s": w5_nd, "c5_alone_list_compute_pull_s": w5,
                "c5_plus_large_list_compute_pull_s": wm, "large_alone_compute_pull_s": w8,
                "pack_csr_of_mixed_lists_s": pack_mixed,
                "extra_cost_of_mixing_s": wm - w5 - w8,
                "note": "best of 3 wall times of build_pull(...).compute_pull(); extra cost = mixed - C5 list - large alone"}
print(json.dumps(out["mixed"]), flush=True)
with open(args.out, "w") as f:
    json.dump(out, f, indent=1)
print("wrote", args.out)
