"""Per-object prediction grids on one GPU (get_prediction(new_binning=[one grid per object])).
 (a) 10^5 1D objects of 60 points, each on its own non-uniform grid of 100 points, against the same batch on one shared
     non-uniform grid of 100 points: the facade's get_prediction(COV='diag') wall time, and the kernel time of the
     prediction entry (DeviceBatch.predict_dev on device-resident grids) by CUDA events; calls alternated.
 (b) 64 objects of 200 points, each with its own grid of 20 000 points: kernel time with the per-object work table and
     with one work item per object (CGP_GRID_PARTS=0, read once per process: measured in a child process), and whether
     the two give the same bits.
Writes profiles/bench_ragged_grids_r01.json.
   python tests/perf_ragged_grids.py [--out profiles/bench_ragged_grids_r01.json]"""
import argparse, json, os, subprocess, sys, tempfile, time
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import cosmogp_b200 as cg
from cosmogp_b200.batch import DeviceBatch, pack_csr

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_ragged_grids_r01.json"))
ap.add_argument("--long-only", default=None, help=argparse.SUPPRESS)   # child: part (b) only, results to this .npz
args = ap.parse_args()

HYP, NUG = np.array([0.8, 2.0]), 0.05


def events(f, reps):
    """kernel time of f() by CUDA events: median and min over reps calls, after one warm-up call"""
    f(); torch.cuda.synchronize()
    t = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); f(); b.record(); b.synchronize()
        t.append(a.elapsed_time(b))
    return np.array(t)


def long_grids():
    """(b): 64 objects of 200 points, 20 000-point grids -> kernel times (ms), mean, var"""
    rng = np.random.default_rng(1)
    B, N, M = 64, 200, 20000
    x = np.sort(rng.uniform(0, 50, (B, N)), axis=1)
    y = np.sin(x / 5) + 0.2 * rng.standard_normal(x.shape)
    ye = rng.uniform(0.1, 0.3, x.shape)
    grids = [np.sort(rng.uniform(-2, 52, M)) for _ in range(B)]
    b = DeviceBatch(x.reshape(-1), y.reshape(-1), np.arange(B + 1, dtype=np.int64) * N, y_err=ye.reshape(-1))
    gf, goff = pack_csr(grids, 1)
    g, go = b._up(gf), b._up(goff)
    run = lambda: b.predict_dev(HYP, NUG, g, go, want_var=True)
    t = events(run, 20)
    m, v, info = run()
    torch.cuda.synchronize()
    assert not info.cpu().numpy().any()
    return t, m.cpu().numpy(), v.cpu().numpy()


if args.long_only:
    t, m, v = long_grids()
    np.savez(args.long_only, t=t, mean=m, var=v)
    sys.exit(0)

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
out = {"gpu": smi[0] if smi else torch.cuda.get_device_name(), "hyperparameters": HYP.tolist(), "nugget": NUG}

# ---- (a) 10^5 x 60, grids of 100 points: one per object against one shared
rng = np.random.default_rng(0)
B, N, M = 100000, 60, 100
x = np.sort(rng.uniform(0, 50, (B, N)), axis=1)
y = np.sin(x / 5) + 0.2 * rng.standard_normal(x.shape)
ye = rng.uniform(0.1, 0.3, x.shape)
shared = np.sort(rng.uniform(-2, 52, M))
own = np.sort(rng.uniform(-2, 52, (B, M)), axis=1)             # a (B, M) ndarray: one grid per object

gp = cg.gaussian_process_nobject(y, x, y_err=ye)
gp.hyperparameters, gp.nugget = HYP.copy(), NUG


def facade(new):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    gp.get_prediction(new_binning=new, COV="diag", svd_method=False)
    torch.cuda.synchronize()
    return time.perf_counter() - t0


facade(own); facade(shared)
wall = {"per_object_s": [], "shared_s": []}
for _ in range(5):
    wall["per_object_s"].append(facade(own))
    wall["shared_s"].append(facade(shared))
b = gp.batch
g_sh = b._up(shared)
g_own, go_own = b._up(own.reshape(-1)), b._up(np.arange(B + 1, dtype=np.int64) * M)
k_own = lambda: b.predict_dev(HYP, NUG, g_own, go_own, want_var=True)
k_sh = lambda: b.predict_dev(HYP, NUG, g_sh, None, want_var=True)
tk_own, tk_sh = [], []
for _ in range(3):                                              # alternated blocks of 10 calls
    tk_own += list(events(k_own, 10)); tk_sh += list(events(k_sh, 10))
tk_own, tk_sh = np.array(tk_own), np.array(tk_sh)
out["a_1e5x60_grid100"] = {
    "objects": B, "points": N, "grid_points": M,
    "facade_get_prediction_diag_s": {"per_object_grids_median": float(np.median(wall["per_object_s"])),
                                     "shared_grid_median": float(np.median(wall["shared_s"])),
                                     "per_object_grids": wall["per_object_s"], "shared_grid": wall["shared_s"]},
    "kernel_ms": {"per_object_grids_median": float(np.median(tk_own)), "per_object_grids_min": float(tk_own.min()),
                  "shared_grid_median": float(np.median(tk_sh)), "shared_grid_min": float(tk_sh.min()), "reps": len(tk_own)},
    "per_object_over_shared_kernel_median": float(np.median(tk_own) / np.median(tk_sh)),
    "extra_grid_bytes_read": 8 * B * M - 8 * M + 8 * (B + 1),
    "what": "kernel_ms: DeviceBatch.predict_dev (mean + variance) between CUDA events, grids already on the device; "
            "facade: get_prediction(COV='diag') to a device synchronisation, numpy in and out"}
print("a", json.dumps(out["a_1e5x60_grid100"]), flush=True)
del gp, b, g_sh, g_own, go_own
torch.cuda.empty_cache()

# ---- (b) 64 x 200 with 20 000-point grids: work table on, and off in a child process
t_on, m_on, v_on = long_grids()
with tempfile.TemporaryDirectory() as tmp:
    path = os.path.join(tmp, "off.npz")
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--long-only", path],
                       env=dict(os.environ, CGP_GRID_PARTS="0"), capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    off = np.load(path)
    t_off, m_off, v_off = off["t"], off["mean"], off["var"]
out["b_64x200_grid20000"] = {
    "objects": 64, "points": 200, "grid_points_per_object": 20000,
    "kernel_ms": {"work_table_median": float(np.median(t_on)), "work_table_min": float(t_on.min()),
                  "one_item_per_object_median": float(np.median(t_off)), "one_item_per_object_min": float(t_off.min()),
                  "reps": len(t_on)},
    "speedup_median": float(np.median(t_off) / np.median(t_on)),
    "bit_identical": bool(np.array_equal(m_on, m_off) and np.array_equal(v_on, v_off)),
    "what": "DeviceBatch.predict_dev (mean + variance) between CUDA events; one item per object: CGP_GRID_PARTS=0"}
print("b", json.dumps(out["b_64x200_grid20000"]), flush=True)

os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
with open(args.out, "w") as f:
    json.dump(out, f, indent=1)
print("wrote", args.out)
