"""Grouped means and variances on the blocked path (cgp_large_predict_objhyp_dev) on one GPU, four shapes:
  2d_1000_shared_grid300 : 256 2D objects of 1 000 points, shared hyperparameters, a shared 300-point grid
  1d_300_objhyp_grid100  : 10^4 1D objects of 300 points, per-object rows and nuggets, a shared 100-point grid
  1d_mixed_60_400_own    : 2*10^4 1D objects of 60 points plus 8 of 400, shared hyperparameters, own epochs
                           (one object above 224 points sends every object to the blocked path)
  2d_2000_objhyp_grid1e4 : 32 2D objects of 2 000 points, per-object rows and nuggets, a shared 10^4-point grid
Per shape: the device time of the entry over all objects (CUDA events, the 2 GB workspace and the pass length
dense.predictions uses), its model FLOPs (n_pad^3/3 + m_pad n_pad^2 per object) over the DMMA ceiling cgp_fp64_peak(1)
measured in this run; the wall time of get_prediction(COV='diag') against a loop of dense.LargeObject.factor + .predict
over the same objects (timed on a stated subset where the whole loop would take too long, and extrapolated); bitwise
equality of the entry's, the facade's and the loop's outputs.  Writes profiles/bench_grouped_predict_r01.json.
   python tests/perf_grouped_predict.py [--out profiles/bench_grouped_predict_r01.json] [--scale 0.01]"""
import argparse, json, os, subprocess, sys, time, zlib
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import cosmogp_b200 as cg
from cosmogp_b200 import _lib, dense

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_grouped_predict_r01.json"))
ap.add_argument("--scale", type=float, default=1.0, help="fraction of the object counts (rehearsal)")
args = ap.parse_args()

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
peak = _lib.fp64_peak(1)
out = {"gpu": smi[0] if smi else torch.cuda.get_device_name(), "dmma_peak_tflops_measured": peak,
       "flop_model": "per object, on the padded sizes the kernels run: n_pad^3/3 (factor) + m_pad n_pad^2 (L^-1 H^T)",
       "workspace_bytes": 2 << 30, "shapes": {}}
L = _lib.lib()


def pad(v):
    return max((int(v) + 127) // 128, 1) * 128


def make(rng, dim, B, N):
    if dim == 1:
        x = [np.sort(rng.uniform(0, n / 5.0, n)) for n in N]
        y = [np.sin(v) + 0.2 * rng.standard_normal(len(v)) for v in x]
        rows = np.stack([rng.uniform(0.6, 1.2, B), rng.uniform(1.0, 2.0, B)], axis=1)
        shared = np.array([0.9, 1.5])
    else:
        x = [rng.uniform(0, 3.0 * np.sqrt(n), (n, 2)) for n in N]
        y = [np.sin((v[:, 0] - v[:, 1]) / 5) + 0.2 * rng.standard_normal(len(v)) for v in x]
        lx, ly = rng.uniform(3.0, 5.0, B), rng.uniform(3.0, 5.0, B)
        rows = np.stack([rng.uniform(0.8, 1.2, B), lx, ly, rng.uniform(-0.3, 0.3, B) * lx * ly], axis=1)
        shared = np.array([1.0, 4.0, 4.0, 1.0])
    return x, y, [rng.uniform(0.1, 0.3, n) for n in N], rows, shared


def shape(name, dim, sizes, M, per_object, loop_groups):
    """sizes: points per object; M: shared grid points (None: own epochs); loop_groups: [(ids, count)] -- the loop is
    timed on `ids` and stands for `count` objects like them."""
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    B = len(sizes)
    x, y, ye, rows, shared = make(rng, dim, B, sizes)
    nugs = rng.uniform(0.01, 0.1, B) if per_object else np.full(B, 0.05)
    hyp = rows if per_object else np.tile(shared, (B, 1))
    own = M is None
    if own:
        grid = None
    else:
        hi = max(sizes) / 5.0 if dim == 1 else 3.0 * np.sqrt(max(sizes))
        grid = np.linspace(-1.0, hi + 1.0, M) if dim == 1 else rng.uniform(0, hi, (M, 2))
    m = np.array(sizes if own else [M] * B, dtype=np.int64)
    r = {"objects": B, "points": sorted(set(int(n) for n in sizes)), "grid": "own epochs" if own else M, "dim": dim,
         "hyperparameters": "per-object rows" if per_object else "shared"}

    # the entry over all objects, device time by CUDA events
    from cosmogp_b200.batch import pack_csr
    dev = torch.device("cuda", torch.cuda.current_device())
    xf, off = pack_csr(x, dim)
    xd = torch.from_numpy(np.ascontiguousarray(xf).reshape(-1)).to(dev)
    yd = torch.from_numpy(pack_csr(y, 1)[0]).to(dev)
    yed = torch.from_numpy(pack_csr(ye, 1)[0]).to(dev)
    gd = xd if own else torch.from_numpy(np.ascontiguousarray(grid).reshape(-1)).to(dev)
    goff = off if own else None
    moff = np.zeros(B + 1, dtype=np.int64)
    np.cumsum(m, out=moff[1:])
    mean = torch.empty(int(moff[-1]), dtype=torch.float64, device=dev)
    var = torch.empty(int(moff[-1]), dtype=torch.float64, device=dev)
    info = torch.empty(B, dtype=torch.int32, device=dev)
    chunk_rows = max(128, (2 << 30) // (8 * pad(max(sizes)))) // 128 * 128          # dense.predictions' default
    work_doubles = max((2 << 30) // 8, int(dense.pred_ws_doubles(max(sizes), min(int(m.max()), chunk_rows))))
    work = torch.empty(work_doubles, dtype=torch.float64, device=dev)
    hrows, nrows = np.ascontiguousarray(hyp), np.ascontiguousarray(nugs)
    st = torch.cuda.current_stream(dev)

    def entry():
        _lib.check(L.cgp_large_predict_objhyp_dev(B, _lib.hptr(off), dim, xd.data_ptr(), yd.data_ptr(), None,
                                                  yed.data_ptr(), _lib.hptr(hrows), _lib.hptr(nrows), 0.0, 0.0, 0,
                                                  gd.data_ptr(), _lib.hptr(goff), 0 if own else M, None, None, B,
                                                  _lib.hptr(moff), mean.data_ptr(), var.data_ptr(), info.data_ptr(),
                                                  chunk_rows, work.data_ptr(), work_doubles, st.cuda_stream),
                   "cgp_large_predict_objhyp_dev")
    entry(); torch.cuda.synchronize()
    times = []
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); entry(); e1.record(); e1.synchronize()
        times.append(e0.elapsed_time(e1))
    assert not info.cpu().numpy().any()
    flops = sum(pad(n) ** 3 / 3.0 + pad(mm) * pad(n) ** 2 for n, mm in zip(sizes, m))
    t = float(np.median(times)) * 1e-3
    r["entry_ms"] = sorted(times)
    r["entry_ms_median"] = t * 1e3
    r["model_tflop"] = flops * 1e-12
    r["tflops"] = flops / t * 1e-12
    r["frac_of_dmma_peak"] = flops / t * 1e-12 / peak
    entry_mean, entry_var = mean.cpu().numpy(), var.cpu().numpy()
    del mean, var, work, xd, yd, yed, gd
    torch.cuda.empty_cache()

    # the facade, get_prediction(COV='diag'), wall time
    gpo = cg.gaussian_process_nobject(y, x, y_err=ye, kernel="RBF1D" if dim == 1 else "RBF2D")
    if per_object:
        gpo.hyperparameters_per_object, gpo.nugget_per_object = rows.copy(), nugs.copy()
    else:
        gpo.hyperparameters, gpo.nugget = shared.copy(), 0.05

    def facade():
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        gpo.get_prediction(new_binning=grid, COV='diag', svd_method=False, per_object=per_object)
        return time.perf_counter() - t0

    facade()                                             # warm-up: uploads, first launches
    pred = [facade() for _ in range(3)]
    fm =np.concatenate([np.asarray(gpo.Prediction[i]) for i in range(B)])
    fv = np.concatenate([np.asarray(gpo.prediction_variance[i]) for i in range(B)])
    same_entry = bool(np.array_equal(fm, entry_mean) and np.array_equal(fv, entry_var))

    # the loop it replaces: LargeObject.factor + .predict per object
    def loop(ids):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = []
        for i in ids:
            lo = dense.LargeObject(x[i], y[i], ye[i], None, dim=dim)
            lo.factor(hyp[i], nugs[i])
            res.append(lo.predict(x[i] if own else grid))
        return time.perf_counter() - t0, res

    loop(loop_groups[0][0][:2])                          # warm-up
    timed, total, same_loop, note = 0, 0.0, True, []
    for ids, count in loop_groups:
        tl, res = loop(ids)
        total += tl * count / len(ids)
        timed += len(ids)
        note.append("%d objects timed for %d" % (len(ids), count))
        for i, (mm, vv) in zip(ids, res):
            same_loop &= bool(np.array_equal(mm, gpo.Prediction[i]) and np.array_equal(vv, gpo.prediction_variance[i]))
    r["facade"] = {"get_prediction_diag_s": pred, "grouped_s": float(min(pred)),
                   "loop_timed_objects": timed, "loop_s_extrapolated": total, "loop_note": "; ".join(note),
                   "speedup": total / float(min(pred))}
    r["bitwise_entry_equals_facade"] = same_entry
    r["bitwise_facade_equals_loop_on_timed_objects"] = same_loop
    out["shapes"][name] = r
    print(name, json.dumps(r), flush=True)


def n_(v):
    return max(int(v * args.scale), 2)


B1 = n_(256)
shape("2d_1000_shared_grid300", 2, [1000] * B1, 300, False, [(list(range(B1)), B1)])
B2 = n_(10000)
shape("1d_300_objhyp_grid100", 1, [300] * B2, 100, True, [(list(range(0, B2, max(B2 // 500, 1))), B2)])
B3 = n_(20000)
sizes3 = [60] * B3
big3 = [int(v) for v in np.linspace(0, B3 - 1, 8)]
for i in big3:
    sizes3[i] = 400
small3 = [i for i in range(0, B3, max(B3 // 1000, 1)) if i not in big3]
shape("1d_mixed_60_400_own", 1, sizes3, None, False, [(small3, B3 - 8), (big3, 8)])
B4 = n_(32)
shape("2d_2000_objhyp_grid1e4", 2, [2000] * B4, 10000, True, [(list(range(B4)), B4)])

os.makedirs(os.path.dirname(args.out), exist_ok=True)
with open(args.out, "w") as f:
    json.dump(out, f, indent=1)
print("wrote", args.out)
