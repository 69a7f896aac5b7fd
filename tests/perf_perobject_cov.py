"""Per-object predictive covariance matrices on one GPU: 2*10^4 1D objects of 60 points, every covariance_matrix written
by cgp_covariance_objhyp_dev (each object with its own row) against cgp_covariance_batched_dev (shared hyperparameters)
on the same batch, calls alternated, each timed to a device synchronisation; on a shared grid of 100 points and on the
objects' own epochs.  Also: the facade materialising every matrix on the host (get_prediction(per_object=True,
COV=True), then covariance_matrix[i] for all i), and a loop of dense.predictive_covariance timed on 200 objects and
extrapolated to the batch.  Writes profiles/bench_perobject_cov_r01.json.
   python tests/perf_perobject_cov.py [--out profiles/bench_perobject_cov_r01.json]"""
import argparse, json, os, subprocess, sys, time
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import cosmogp_b200 as cg
from cosmogp_b200 import _lib, dense
from cosmogp_b200.batch import DeviceBatch

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_perobject_cov_r01.json"))
args = ap.parse_args()

HBM_TBPS = 7.7                                       # HGX B200 data sheet, one GPU: a ceiling, not a measurement
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
B, N, M = 20000, 60, 100
out = {"gpu": smi[0] if smi else torch.cuda.get_device_name(), "objects": B, "points": N, "grid": M,
       "hbm_datasheet_tbps": HBM_TBPS,
       "bytes_convention": "matrices written once + V rows (8 ceil(N/8) doubles per grid point) written by the factor "
                           "phase and read by the gram phase at least once", "runs": {}}

rng = np.random.default_rng(0)
x = np.sort(rng.uniform(0, 50, (B, N)), axis=1)
y = np.sin(x / 5) + 0.2 * rng.standard_normal(x.shape)
ye = rng.uniform(0.1, 0.3, x.shape)
rows = np.stack([rng.uniform(0.5, 1.5, B), rng.uniform(1.0, 4.0, B)], axis=1)
nugs = rng.uniform(0.01, 0.1, B)
shared, shared_nug = np.array([1.0, 2.5]), 0.05
grid = np.linspace(-2, 52, M)

b = DeviceBatch(x.reshape(-1), y.reshape(-1), np.arange(B + 1, dtype=np.int64) * N, y_err=ye.reshape(-1))
L, dev, st = _lib.lib(), b.device, torch.cuda.current_stream().cuda_stream
hyp_d = torch.tensor(rows, dtype=torch.float64, device=dev)
nug_d = torch.tensor(nugs, dtype=torch.float64, device=dev)
info = torch.empty(B, dtype=torch.int32, device=dev)
ldv = 8 * ((N + 7) // 8)


def case(own):
    if own:
        g, goff, goff_host, m = b.x, b.off.data_ptr(), b.off_host.ctypes.data, 0
        coff_h = np.arange(B + 1, dtype=np.int64) * N * N
        coff = torch.tensor(coff_h, device=dev)
        tot, coff_p, grid_rows = int(coff_h[-1]), coff.data_ptr(), B * N
    else:
        g = torch.tensor(grid, device=dev)
        goff = goff_host = coff_p = None
        m, tot, grid_rows, coff = M, B * M * M, B * M, None
    cov = torch.empty(tot, dtype=torch.float64, device=dev)
    head = (B, b.off.data_ptr(), N, 1, b.x.data_ptr(), b.y_err.data_ptr())
    tail = (g.data_ptr(), goff, goff_host, m, cov.data_ptr(), coff_p, info.data_ptr(), st)

    def per_object():
        _lib.check(L.cgp_covariance_objhyp_dev(*head, hyp_d.data_ptr(), nug_d.data_ptr(), 0.0, 0.0, 0, *tail),
                   "cgp_covariance_objhyp_dev")

    def shared_hyp():
        _lib.check(L.cgp_covariance_batched_dev(*head, _lib.hptr(shared), shared_nug, 0.0, 0, *tail),
                   "cgp_covariance_batched_dev")
    return per_object, shared_hyp, cov, tot, grid_rows, coff


def alternated(fa, fb, reps=15):
    fa(); fb(); torch.cuda.synchronize()
    ta, tb = [], []
    for _ in range(reps):
        for f, acc in ((fa, ta), (fb, tb)):
            t0 = time.perf_counter(); f(); torch.cuda.synchronize(); acc.append(time.perf_counter() - t0)
    return np.array(ta), np.array(tb)


for own in (False, True):
    name = "own_epochs" if own else "shared_grid"
    per_object, shared_hyp, cov, tot, grid_rows, _keep = case(own)
    ta, tb = alternated(per_object, shared_hyp)
    # correctness of what was timed: the last per-object call, a few objects against dense.predictive_covariance
    per_object(); torch.cuda.synchronize()
    side = N if own else M
    worst = 0.0
    for i in (0, 9999, B - 1):
        got = cov[i * side * side:(i + 1) * side * side].cpu().numpy().reshape(side, side)
        ref = dense.predictive_covariance(x[i], ye[i], x[i] if own else grid, rows[i], nugs[i], 1)
        worst = max(worst, float(np.max(np.abs(got - ref)) / np.max(np.abs(ref))))
    nbytes = 8 * tot + 2 * 8 * grid_rows * ldv
    r = {"per_object_ms_median": float(np.median(ta)) * 1e3, "per_object_ms_min": float(ta.min()) * 1e3,
         "shared_ms_median": float(np.median(tb)) * 1e3, "shared_ms_min": float(tb.min()) * 1e3,
         "per_object_over_shared_median": float(np.median(ta) / np.median(tb)),
         "matrix_bytes": 8 * tot, "bytes_moved_min": nbytes,
         "per_object_rate_tbps": nbytes / np.median(ta) * 1e-12,
         "per_object_frac_of_hbm_datasheet": nbytes / np.median(ta) * 1e-12 / HBM_TBPS,
         "max_rel_diff_vs_dense_3_objects": worst, "reps": len(ta)}
    out["runs"][name] = r
    print(name, json.dumps(r), flush=True)
    del cov, _keep
    torch.cuda.empty_cache()

# the facade: every matrix materialised on the host, per-object rows against shared hyperparameters
gp = cg.gaussian_process_nobject(y, x, y_err=ye)
gp.hyperparameters_per_object, gp.nugget_per_object = rows, nugs
gp.hyperparameters, gp.nugget = shared.copy(), shared_nug


def facade(per):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    gp.get_prediction(new_binning=grid, COV=True, svd_method=False, per_object=per)
    for i in range(B):
        gp.covariance_matrix[i]
    torch.cuda.synchronize()
    return time.perf_counter() - t0


facade(True); facade(False)                          # warm-up: the batch upload, first launches, pinned buffers
fac = {"per_object_s": [], "shared_s": [], "what": "get_prediction(COV=True) and then covariance_matrix[i] for every i, "
                                                  "alternated after one warm-up call of each"}
for _ in range(3):
    fac["per_object_s"].append(facade(True))
    fac["shared_s"].append(facade(False))
out["facade_all_matrices_on_host_shared_grid"] = fac
print("facade", json.dumps(fac), flush=True)

# a loop of dense.predictive_covariance (one object per call), timed on 200 objects and extrapolated to B
k = 200
dense.predictive_covariance(x[0], ye[0], grid, rows[0], nugs[0], 1)
torch.cuda.synchronize()
t0 = time.perf_counter()
for i in range(k):
    dense.predictive_covariance(x[i], ye[i], grid, rows[i], nugs[i], 1)
torch.cuda.synchronize()
t = time.perf_counter() - t0
out["dense_loop_shared_grid"] = {"timed_objects": k, "timed_s": t,
                                 "extrapolated_to_all_objects_s": t * B / k, "note": "extrapolation, not a measurement"}
print("dense loop", json.dumps(out["dense_loop_shared_grid"]), flush=True)

os.makedirs(os.path.dirname(args.out), exist_ok=True)
with open(args.out, "w") as f:
    json.dump(out, f, indent=1)
print("wrote", args.out)
