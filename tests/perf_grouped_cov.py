"""Grouped predictive covariance matrices (cgp_large_covariance_dev) on one GPU, four shapes:
  1d_100_shared_rows : 10^4 1D objects of 100 points, shared hyperparameters, a shared 100-point grid
  1d_200_objhyp      : 10^4 1D objects of 200 points, per-object rows and nuggets, a shared 100-point grid
  1d_150_own         : 10^4 1D objects of 150 points on their own epochs, shared hyperparameters
  2d_1000_grid300    : 256 2D objects of 1 000 points on a shared 300-point grid
Per shape: the device time of the entry over all objects (CUDA events, 2 GB workspace as the facade uses), its model
FLOPs over the DMMA ceiling cgp_fp64_peak(1) measured in this run; the wall time of get_prediction(COV=True) and of
reading every covariance_matrix[i] through the facade, against CGP_GROUPED_COV=0 (one dense.predictive_covariance per
object), whose read loop is timed on 200 objects and extrapolated.  Writes profiles/bench_grouped_cov_r01.json.
   python tests/perf_grouped_cov.py [--out profiles/bench_grouped_cov_r01.json]"""
import argparse, json, os, subprocess, sys, time, zlib
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import cosmogp_b200 as cg
from cosmogp_b200 import _lib, dense, gp as gp_mod

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_grouped_cov_r01.json"))
ap.add_argument("--scale", type=float, default=1.0, help="fraction of the object counts (rehearsal)")
args = ap.parse_args()

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
peak = _lib.fp64_peak(1)
out = {"gpu": smi[0] if smi else torch.cuda.get_device_name(), "dmma_peak_tflops_measured": peak,
       "flop_model": "per object, on the padded sizes the kernels run: n_pad^3/3 (factor) + m_pad n_pad^2 (L^-1 H^T) "
                     "+ 2 m_pad^2 n_pad (V V^T, full)",
       "workspace_bytes": 2 << 30, "shapes": {}}
L = _lib.lib()


def pad(v):
    return max((int(v) + 127) // 128, 1) * 128


def shape(name, dim, B, N, M, per_object, own):
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    B = max(int(B * args.scale), 2)
    if dim == 1:
        x = np.sort(rng.uniform(0, N / 5.0, (B, N)), axis=1)
        y = np.sin(x) + 0.2 * rng.standard_normal(x.shape)
        rows = np.stack([rng.uniform(0.6, 1.2, B), rng.uniform(1.0, 2.0, B)], axis=1)
        grid = np.linspace(-1.0, N / 5.0 + 1.0, M)
        shared = np.array([0.9, 1.5])
    else:
        s = 3.0 * np.sqrt(N)
        x = rng.uniform(0, s, (B, N, 2))
        y = np.sin((x[..., 0] - x[..., 1]) / 5) + 0.2 * rng.standard_normal((B, N))
        lx, ly = rng.uniform(3.0, 5.0, B), rng.uniform(3.0, 5.0, B)
        rows = np.stack([rng.uniform(0.8, 1.2, B), lx, ly, rng.uniform(-0.3, 0.3, B) * lx * ly], axis=1)
        grid = rng.uniform(0, s, (M, 2))
        shared = np.array([1.0, 4.0, 4.0, 1.0])
    ye = rng.uniform(0.1, 0.3, (B, N))
    nugs = rng.uniform(0.01, 0.1, B) if per_object else np.full(B, 0.05)
    hyp = rows if per_object else np.tile(shared, (B, 1))
    m = N if own else M
    r = {"objects": B, "points": N, "grid": "own epochs" if own else M, "dim": dim,
         "hyperparameters": "per-object rows" if per_object else "shared"}

    # the entry over all objects, device time by CUDA events
    dev = torch.device("cuda", torch.cuda.current_device())
    xf = x.reshape(-1) if dim == 1 else x.reshape(-1, 2)
    off = np.arange(B + 1, dtype=np.int64) * N
    xd = torch.from_numpy(np.ascontiguousarray(xf).reshape(-1)).to(dev)
    yd = torch.from_numpy(ye.reshape(-1).copy()).to(dev)
    gd = xd if own else torch.from_numpy(np.ascontiguousarray(grid).reshape(-1)).to(dev)
    goff = off if own else None
    coff = np.arange(B + 1, dtype=np.int64) * m * m
    cov = torch.empty(int(coff[-1]), dtype=torch.float64, device=dev)
    info = torch.empty(B, dtype=torch.int32, device=dev)
    work_doubles = (2 << 30) // 8
    work = torch.empty(work_doubles, dtype=torch.float64, device=dev)
    hrows = np.ascontiguousarray(hyp)
    nrows = np.ascontiguousarray(nugs)
    st = torch.cuda.current_stream(dev)

    def entry():
        _lib.check(L.cgp_large_covariance_dev(B, _lib.hptr(off), dim, xd.data_ptr(), yd.data_ptr(), _lib.hptr(hrows),
                                              _lib.hptr(nrows), 0.0, 0.0, 0, gd.data_ptr(), _lib.hptr(goff),
                                              0 if own else M, None, B, cov.data_ptr(), _lib.hptr(coff), info.data_ptr(),
                                              work.data_ptr(), work_doubles, st.cuda_stream), "cgp_large_covariance_dev")
    entry(); torch.cuda.synchronize()
    times = []
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); entry(); e1.record(); e1.synchronize()
        times.append(e0.elapsed_time(e1))
    assert not info.cpu().numpy().any()
    npd, mpd = pad(N), pad(m)
    flops = B * (npd ** 3 / 3.0 + mpd * npd ** 2 + 2.0 * mpd ** 2 * npd)
    t = float(np.median(times)) * 1e-3
    r["entry_ms"] = sorted(times)
    r["entry_ms_median"] = t * 1e3
    r["model_tflop"] = flops * 1e-12
    r["tflops"] = flops / t * 1e-12
    r["frac_of_dmma_peak"] = flops / t * 1e-12 / peak
    # what was timed, against the single-object path, bit for bit
    side = m
    same = True
    for i in (0, B // 2, B - 1):
        got = cov[int(coff[i]):int(coff[i + 1])].cpu().numpy().reshape(side, side)
        ref = dense.predictive_covariance(x[i], ye[i], x[i] if own else grid, hyp[i], nugs[i], dim)
        same &= bool(np.array_equal(got, ref))
    r["bitwise_equal_to_dense_3_objects"] = same
    del cov, work, xd, yd, gd
    torch.cuda.empty_cache()

    # the facade: get_prediction(COV=True) then every covariance_matrix[i]
    gpo = cg.gaussian_process_nobject(list(y), list(x), y_err=list(ye), kernel="RBF1D" if dim == 1 else "RBF2D")
    if per_object:
        gpo.hyperparameters_per_object, gpo.nugget_per_object = rows.copy(), nugs.copy()
    else:
        gpo.hyperparameters, gpo.nugget = shared.copy(), 0.05

    def facade(k):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        gpo.get_prediction(new_binning=None if own else grid, COV=True, svd_method=False, per_object=per_object)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        for i in range(k):
            gpo.covariance_matrix[i]
        t2 = time.perf_counter()
        return t1 - t0, t2 - t1

    facade(min(B, 2))                                    # warm-up: uploads, first launches
    pred, read = [], []
    for _ in range(2):
        a, b = facade(B)
        pred.append(a); read.append(b)
    k = min(200, B)
    gp_mod._GROUPED_COV = False
    try:
        facade(2)
        la, lb = facade(k)
    finally:
        gp_mod._GROUPED_COV = True
    r["facade"] = {"get_prediction_s": pred, "read_all_matrices_s": read,
                   "grouped_total_s": float(min(p + q for p, q in zip(pred, read))),
                   "loop_read_timed_objects": k, "loop_read_timed_s": lb,
                   "loop_total_s_extrapolated": float(min(pred)) + lb * B / k,
                   "note": "CGP_GROUPED_COV=0 read loop timed on %d objects and extrapolated to %d; get_prediction "
                           "itself does not depend on the knob" % (k, B)}
    r["facade"]["speedup_total"] = r["facade"]["loop_total_s_extrapolated"] / r["facade"]["grouped_total_s"]
    out["shapes"][name] = r
    print(name, json.dumps(r), flush=True)


shape("1d_100_shared_rows", 1, 10000, 100, 100, False, False)
shape("1d_200_objhyp", 1, 10000, 200, 100, True, False)
shape("1d_150_own", 1, 10000, 150, 150, False, True)
shape("2d_1000_grid300", 2, 256, 1000, 300, False, False)

os.makedirs(os.path.dirname(args.out), exist_ok=True)
with open(args.out, "w") as f:
    json.dump(out, f, indent=1)
print("wrote", args.out)
