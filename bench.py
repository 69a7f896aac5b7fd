#!/usr/bin/env python
"""Benchmark of the cosmogp GP hot path on B200.

Workload (BASELINE.json configs[1], "C2"): 10^5 synthetic light curves x 60 epochs with a
shared mean function.  One STEP = one pass of the hot path over the batch:
  one log-likelihood evaluation of all objects (what scipy's optimiser triggers per
  simplex point, cosmogp/Gaussian_process.py:191-213) + one prediction of mean and
  variance on a shared 100-point grid (:270-361; grid of the multi-object notebook cell 22).
metric = objects put through LL+predict per second ("fits/s"), whole job.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--objects B] [--dump-outputs DIR]

--dump-outputs DIR writes what the last timed step computed as DIR/<name>.npy (float64): ll (k,), mean and var (k, 100)
of k = min(objects, 32768) objects, a fixed seeded sample, and their indices in objects.npy.  The inputs are seeded,
so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_EPOCH = 60
M_GRID = 100
HYP = (0.5, 2.0)
NUGGET = 0.0
YERR = 0.2
N_CHECK = 32            # objects per rank whose timed-step outputs are checked against the oracle
DUMP_OBJECTS = 32768    # --dump-outputs: 202 doubles per object (index, ll, mean and var on the grid), 53 MB in all


def flops_ll(n):            # SURVEY.md section 8(d): build + POTRF + forward solve + norms
    return n ** 3 / 3.0 + 3.5 * n ** 2


def flops_predict(n, m):    # build + POTRF + 2 TRSV + per grid point (h build, mean dot, v = L^-1 h, |v|^2)
    return n ** 3 / 3.0 + 4.0 * n ** 2 + m * (n ** 2 + 8.0 * n)


def make_c2(n_obj, seed):
    """SURVEY.md section 8(d) C2 recipe: x = sort(U(-10,40)), truth sigma=0.5 l=2, y_err=0.2,
    template -18+2 sin(t/10) on linspace(-15,45,61), per-object offset N(0,0.3), y = mean + offset + L z."""
    rng = np.random.default_rng(seed)
    tmean = np.linspace(-15, 45, 61)
    ymean = -18 + 2 * np.sin(tmean / 10)
    x = np.empty((n_obj, N_EPOCH)); y = np.empty((n_obj, N_EPOCH))
    from scipy.interpolate import InterpolatedUnivariateSpline
    spline = InterpolatedUnivariateSpline(tmean, ymean)
    eye = np.eye(N_EPOCH)
    for s in range(0, n_obj, 10000):
        e = min(n_obj, s + 10000)
        xs = np.sort(rng.uniform(-10, 40, (e - s, N_EPOCH)), axis=1)
        d = xs[:, None, :] - xs[:, :, None]
        k = HYP[0] ** 2 * np.exp(-0.5 * d * d / HYP[1] ** 2) + YERR ** 2 * eye
        low = np.linalg.cholesky(k)
        z = rng.standard_normal((e - s, N_EPOCH, 1))
        x[s:e] = xs
        y[s:e] = spline(xs) + rng.normal(0, 0.3, (e - s, 1)) + (low @ z)[:, :, 0]
    ye = np.full((n_obj, N_EPOCH), YERR)
    return x, y, ye, tmean, ymean


def dump_outputs(path, ll, mean, var):
    """Write one step's outputs (device tensors: ll (B,), mean and var (B * M_GRID,)) for all objects, or for a sample of
    DUMP_OBJECTS of them drawn from a fixed seed, as path/<name>.npy in float64."""
    import torch
    b = ll.shape[0]
    idx = np.arange(b) if b <= DUMP_OBJECTS else np.sort(np.random.default_rng(0).choice(b, DUMP_OBJECTS, replace=False))
    sel = torch.from_numpy(idx).to(ll.device)
    arrays = {"objects": idx.astype(np.float64), "ll": ll[sel].cpu().numpy(),
              "mean": mean.view(b, M_GRID)[sel].cpu().numpy(), "var": var.view(b, M_GRID)[sel].cpu().numpy()}
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


class ClockSampler(threading.Thread):
    """nvidia-smi clocks and throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.proc = index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
        self.join(timeout=2)
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 6 and r[2 + i] == "Active" for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ----------------------------------------------------------------------------- CPU arm
def reference_available():
    from oracle import ref_loader
    return ref_loader.available()


def _cpu_worker(args):
    """One host core, one BLAS thread.  kind "reference": the UNMODIFIED reference (baseline/_ref, loaded by
    oracle/ref_loader.py) through its own public API -- gaussian_process_nobject(...).compute_log_likelihood(hyp)
    then .get_prediction(new_binning=grid, COV=True) (cosmogp/Gaussian_process.py:191-213, :270-361; COV=True is the
    only way the reference yields a predictive variance).  kind "port": the oracle restatement of the same calls
    (fallback when baseline/_ref is absent).  Only the two calls are timed, not the construction of the object."""
    kind, svd, x, y, ye, tmean, ymean, grid = args
    from threadpoolctl import threadpool_limits
    with threadpool_limits(limits=1):
        if kind == "reference":
            from oracle import ref_loader
            ref = ref_loader.load()
            with ref_loader.quiet():
                gp = ref.gaussian_process_nobject(list(y), list(x), kernel="RBF1D", y_err=list(ye), Mean_Y=ymean, Time_mean=tmean)
                gp.hyperparameters = np.array(HYP); gp.nugget = NUGGET; gp.fit_nugget = False
                t0 = time.perf_counter()
                gp.compute_log_likelihood(np.array(HYP), svd_method=svd)
                gp.get_prediction(new_binning=grid, COV=True, svd_method=svd)
                var0 = np.diag(gp.covariance_matrix[0]).copy()
                dt = time.perf_counter() - t0
            return dt, float(np.ravel(gp.log_likelihood)[0]), gp.Prediction[0].copy(), var0
        from oracle import gp_oracle as O
        from cosmogp_b200 import mean as M
        off = np.arange(len(x) + 1, dtype=np.int64) * x.shape[1]
        y0, d = M.batched_mean(x.ravel(), y.ravel(), off, 1, ymean, tmean, None)
        y0 = y0.reshape(x.shape)
        ny0 = M.template_on_grid(grid, 1, ymean, tmean)[None, :] + d[:, None]
        t0 = time.perf_counter()
        acc = 0.0
        for i in range(len(x)):
            acc += O.log_likelihood(y[i], x[i], HYP, NUGGET, ye[i], y0[i], svd_method=svd)
            m, v = O.predict(y[i], x[i], HYP, NUGGET, grid, ye[i], y0[i], ny0[i], full_cov=False, svd_method=svd)
            if i == 0:
                m0, v0 = m, v
        return time.perf_counter() - t0, acc, m0, v0


def cpu_pass(kind, svd, x, y, ye, tmean, ymean, grid, pool, cores):
    """All host cores, one process each, objects split evenly; the pass takes as long as its slowest worker.
    Returns (objects/s, per-worker results)."""
    parts = [p for p in np.array_split(np.arange(len(x)), cores) if len(p)]
    res = pool.map(_cpu_worker, [(kind, svd, x[p], y[p], ye[p], tmean, ymean, grid) for p in parts])
    return len(x) / max(r[0] for r in res), res


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the step on this box's host cores."""
    if rank != 0:
        return
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    kind = "reference" if reference_available() else "port"
    per_step = args.cpu_objects or 400 * cores
    x, y, ye, tmean, ymean = make_c2(per_step, 2)
    grid = np.linspace(-10, 40, M_GRID)
    if kind == "reference":
        from oracle import ref_loader
        ref_loader.load()                                   # imported once, inherited by the forked workers
    with mp.get_context("fork").Pool(cores) as pool:
        for _ in range(args.warmup):
            cpu_pass(kind, False, x, y, ye, tmean, ymean, grid, pool, cores)
        dt = 0.0
        for _ in range(args.steps):
            v, _r = cpu_pass(kind, False, x, y, ye, tmean, ymean, grid, pool, cores)
            dt += per_step / v
        v_svd, _r = cpu_pass(kind, True, x, y, ye, tmean, ymean, grid, pool, cores)
    val = per_step * args.steps / dt
    what = ("unmodified PFLeget/cosmogp from baseline/_ref: gaussian_process_nobject.compute_log_likelihood + "
            "get_prediction(COV=True), svd_method=False" if kind == "reference" else
            "oracle port of the same calls (baseline/_ref absent), svd_method=False")
    sample = ("%d of the 10^5 objects of the workload per step (N=%d, M=%d), objects/s = sample / slowest worker, no "
              "extrapolation beyond that (the path is linear in the number of objects); %s; %d processes x 1 BLAS thread"
              % (per_step, N_EPOCH, M_GRID, what, cores))
    cfg = workload_config(100000, 1)
    cfg["cpu_sample_objects_per_step"] = per_step
    print(json.dumps({
        "impl": "reference", "metric": "gp_fits_per_sec", "value": val, "unit": "objects/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": val, "unit": "objects/s", "cores": cores, "kind": kind, "sample": sample,
                         "svd_method_true": {"value": v_svd, "unit": "objects/s",
                                             "what": "the same pass with svd_method=True (the reference's default argument)"}},
        "e2e": {"value": val, "unit": "objects/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def workload_config(n_obj, world, scaling="weak"):
    return {"workload": "C2: batched 1D light curves, shared mean; step = one pass of the hot path = log-likelihood of every "
                        "object + predict(mean, var) on a shared grid at the same hyperparameters (one factorisation per "
                        "object serves both); NOT a full fit: a fit repeats the likelihood evaluation ~60-80 times "
                        "(reported as ll_evaluation / facade_e2e)",
            "objects_per_gpu": n_obj, "objects_total": n_obj * world, "epochs": N_EPOCH, "grid_points": M_GRID, "kernel": "RBF1D",
            "hyp": list(HYP), "nugget": NUGGET, "y_err": YERR, "scaling_mode": scaling,
            "sharding": "objects x%d, no data-path collective (LL sum all-reduced)" % world,
            "l2_policy": "inputs+outputs per step (%.0f MB) exceed the 126 MB L2" % (n_obj * (4 * N_EPOCH + 3 * M_GRID) * 8 / 1e6)
            if n_obj * (4 * N_EPOCH + 3 * M_GRID) * 8 > 126e6 else
            "L2 flushed between steps is not needed for the timed kernels' inputs: they are regenerated per object on chip; "
            "inputs+outputs per step are %.0f MB" % (n_obj * (4 * N_EPOCH + 3 * M_GRID) * 8 / 1e6)}


def _facade_worker(args):
    """The reference doing what facade_e2e does: construct, find_hyperparameters, get_prediction (one core)."""
    x, y, ye, tmean, ymean, grid = args
    from threadpoolctl import threadpool_limits
    from oracle import ref_loader
    ref = ref_loader.load()
    with threadpool_limits(limits=1), ref_loader.quiet():
        t0 = time.perf_counter()
        gp = ref.gaussian_process_nobject(list(y), list(x), kernel="RBF1D", y_err=list(ye), Mean_Y=ymean, Time_mean=tmean)
        gp.find_hyperparameters(hyperparameter_guess=[0.4, 3.0], svd_method=False)
        gp.get_prediction(new_binning=grid, COV=True, svd_method=False)
        return time.perf_counter() - t0, [float(v) for v in gp.hyperparameters]


# ----------------------------------------------------------------------------- C5: leave-one-out pulls, sharded
def run_c5(args, rank, world, local):
    """BASELINE config 5: leave-one-out pulls of 10^6 light curves x 40 epochs sharded over the ranks (one per GPU),
    every rank on its own contiguous range, the per-object outputs gathered on rank 0 by NCCL send/recv over NVLink
    (cosmogp_b200.sharding.gather_to_root).  value = objects/s with the shards resident (kernel only, max over ranks);
    e2e = upload of the rank's inputs + kernel + gather of the four output arrays on rank 0 + download there."""
    import torch
    import torch.distributed as dist
    from cosmogp_b200 import _lib, sharding
    from cosmogp_b200.batch import DeviceBatch
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n, total = 40, args.objects if args.objects != 100000 else 1000000
    ranges = sharding.balanced_ranges(np.full(total, n), world)
    a, b = ranges[rank]
    B = b - a
    rng = np.random.default_rng(5 + rank)                              # SURVEY 8(d) C5 recipe
    x = np.sort(rng.uniform(-10, 10, (B, n)), axis=1)
    y = 0.5 * np.sin(x / 2.0 + rng.uniform(0, 2 * np.pi, (B, 1))) + 0.1 * rng.standard_normal((B, n))
    ye = np.full((B, n), 0.1)
    hyp, nug = (0.5, 2.0), 0.0
    off = np.arange(B + 1, dtype=np.int64) * n
    pin = lambda v: torch.from_numpy(np.ascontiguousarray(v)).pin_memory()
    xp, yp, yep = pin(x.ravel()), pin(y.ravel()), pin(ye.ravel())
    batch = DeviceBatch(xp.numpy(), yp.numpy(), off, y_err=yep.numpy(), dim=1)
    for _ in range(max(args.warmup, 3)):
        outs = batch.loo_dev(hyp, nug)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = _lib.lib().cgp_launch_count()
    e0.record()
    for _ in range(args.steps):
        outs = batch.loo_dev(hyp, nug)
    e1.record(); torch.cuda.synchronize()
    launches = _lib.lib().cgp_launch_count() - launches0
    ms = e0.elapsed_time(e1)
    # parity of the timed step on every rank: pulls of the first objects against the oracle
    from oracle import gp_oracle as O
    po = O.loo_batched_1d(x[:N_CHECK], y[:N_CHECK], ye[:N_CHECK], hyp, nug)
    got = outs[2][:N_CHECK * n].cpu().numpy()
    parity = float(np.max(np.abs(got - po[2].ravel()) / np.maximum(np.abs(po[2].ravel()), 1e-3)))

    counts = [(r[1] - r[0]) * n for r in ranges]
    host_all = [torch.empty(total * n, dtype=torch.float64, pin_memory=True) for _ in range(4)] if rank == 0 else None
    host_mine = [torch.empty(B * n, dtype=torch.float64, pin_memory=True) for _ in range(4)]

    def e2e_step(gather):
        """upload this rank's inputs (pinned) -> kernel -> outputs to the host: gather=True collects the four arrays on
        rank 0 with NCCL send/recv over NVLink and downloads them there (north_star's final gather); gather=False lets
        every rank download its own slice over its own PCIe link"""
        bt = DeviceBatch(xp.numpy(), yp.numpy(), off, y_err=yep.numpy(), dim=1)
        pred, pvar, pull, resid, info = bt.loo_dev(hyp, nug)
        for k, t in enumerate((pred, pvar, pull, resid)):
            if gather and world > 1:
                flat = sharding.gather_to_root_dev(t, counts, root=0)
                if rank == 0:
                    host_all[k].copy_(flat, non_blocking=True)
            elif gather:
                host_all[k].copy_(t, non_blocking=True)
            else:
                host_mine[k].copy_(t, non_blocking=True)
        torch.cuda.synchronize()

    def timed_e2e(gather):
        e2e_step(gather)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step(gather)
        if world > 1:
            dist.barrier()
        return time.perf_counter() - t0
    e2e_steps = max(2, min(args.steps, 5))
    e2e_s = timed_e2e(True)
    direct_s = timed_e2e(False)
    if rank == 0:                                           # the gathered pulls are the oracle's on rank 0's own range
        got_g = host_all[2][:N_CHECK * n].numpy()
        parity = max(parity, float(np.max(np.abs(got_g - po[2].ravel()) / np.maximum(np.abs(po[2].ravel()), 1e-3))))
    if world > 1:
        t = torch.tensor([ms, e2e_s, parity, direct_s], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_s, parity, direct_s = (float(v) for v in t.tolist())
    assert parity < 1e-8, "C5 parity %g" % parity
    if rank == 0:
        peak = _lib.fp64_peak(1)
        fl = 2.0 * n ** 3 / 3.0 + 6.0 * n ** 2
        ach = fl * total * args.steps / (ms * 1e-3) * 1e-12 / world
        print(json.dumps({
            "metric": "loo_pull_objects_per_sec", "value": total * args.steps / (ms * 1e-3), "unit": "objects/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "C5: leave-one-out pulls, closed form on K^-1; %d objects x %d epochs in total, sharded x%d by "
                                   "sum N^3, final gather of pred / var / pull / resid on rank 0 by NCCL send/recv" % (total, n, world),
                       "objects_total": total, "epochs": n, "hyp": list(hyp), "y_err": 0.1},
            "e2e": {"value": total * e2e_steps / e2e_s, "unit": "objects/s", "ms_per_step": e2e_s / e2e_steps * 1e3,
                    "h2d_bytes_per_step": int(3 * B * n * 8 + (B + 1) * 8), "d2h_bytes_per_step": int(4 * total * n * 8),
                    "path": "per rank: DeviceBatch upload (pinned) -> cgp_loo_batched_dev -> NCCL gather of 4 arrays on rank 0 -> "
                            "download on rank 0 (h2d bytes are per rank, d2h bytes leave through rank 0's link)",
                    "without_gather": {"value": total * e2e_steps / direct_s, "unit": "objects/s", "ms_per_step": direct_s / e2e_steps * 1e3,
                                       "what": "every rank downloads its own slice over its own PCIe link instead"}},
            "gpu_launches": int(launches), "parity_max_rel_err": parity,
            "roofline": {"bound": "tensor", "kernel": "gp64_kernel<1,LOO,5>", "achieved": ach, "peak": peak, "unit": "TFLOP/s",
                         "frac": ach / peak, "traffic": None, "flop_per_object": fl}}))
    if world > 1:
        dist.destroy_process_group()


# ----------------------------------------------------------------------------- GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of the headline measurement (the ll_evaluation leg runs max(5, K) calls, the e2e leg "
                         "max(3, min(K, 10)) steps)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--objects", type=int, default=100000, help="objects per GPU (weak scaling) or in total (strong)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --objects per GPU (the contract's default); strong: --objects in total, split over the GPUs")
    ap.add_argument("--workload", default="c2", choices=["c2", "c5"])
    ap.add_argument("--cpu-objects", type=int, default=0, help="objects per CPU baseline pass")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's ll, mean and var (rank 0's objects) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.workload != "c2"):
        ap.error("--dump-outputs writes the outputs of the C2 workload of the GPU implementation")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        return run_reference(args, rank, world)
    if args.workload == "c5":
        return run_c5(args, rank, world, local)

    import torch
    import torch.distributed as dist
    from cosmogp_b200 import _lib, mean as M
    from cosmogp_b200.batch import DeviceBatch, pinned_like

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.require_device()

    B = args.objects if args.scaling == "weak" else args.objects // world
    x, y, ye, tmean, ymean = make_c2(B, 2 + rank)
    off = np.arange(B + 1, dtype=np.int64) * N_EPOCH
    y0, d = M.batched_mean(x.ravel(), y.ravel(), off, 1, ymean, tmean, None)      # host prep, outside the path
    grid = np.linspace(-10, 40, M_GRID)
    # shared mean: template on the grid + one offset per object (the reference's Mean_Y / diff, mean.py:92-101);
    # the device adds them, so M + B doubles travel instead of B x M
    tmpl = M.template_on_grid(grid, 1, ymean, tmean)
    ny0 = tmpl[None, :] + d[:, None]                                    # the same thing materialised, for the checker
    packed_mean = np.concatenate([tmpl, d])
    (xp, _k1), (yp, _k2), (y0p, _k3), (yep, _k4), (ny0p, _k5) = (pinned_like(a) for a in (x.ravel(), y.ravel(), y0, ye.ravel(), packed_mean))

    batch = DeviceBatch(xp, yp, off, y0=y0p, y_err=yep, dim=1)
    g_dev = torch.from_numpy(grid).to(dev)
    ny0_dev = torch.from_numpy(ny0p).to(dev)
    peak_dmma = _lib.fp64_peak(1)
    peak_dfma = _lib.fp64_peak(0)

    def step():
        # one factorisation per object: the factor kernel also emits the log-likelihood, the grid kernel predicts from the
        # factor (what cgp_step_batched_dev runs; called as its two halves so that each kernel is timed on its own)
        fac = batch.factor_dev(HYP, NUGGET, want_ll=True)
        if world > 1:
            tot = fac["ll"].sum()
            dist.all_reduce(tot)          # the one exchange a likelihood evaluation needs
        e_mid.record()
        mean, var, _ = batch.predict_factored_dev(fac, g_dev, None, ny0_dev, True, template_mean=True, uniform_grid=True)
        return fac["ll"], mean, var

    e_mid = torch.cuda.Event(enable_timing=True)
    for _ in range(args.warmup):
        out = step()
    torch.cuda.synchronize()

    sampler = ClockSampler(local); sampler.start()
    time.sleep(0.3)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    launches0 = _lib.lib().cgp_launch_count()
    for k in range(args.steps):
        ev[k][0].record()
        e_mid = ev[k][1]
        out = step()
        ev[k][2].record()
    torch.cuda.synchronize()
    launches = _lib.lib().cgp_launch_count() - launches0
    if world > 1:
        dist.barrier()
    total_ms = ev[0][0].elapsed_time(ev[-1][2])
    fa_ms = float(np.mean([e[0].elapsed_time(e[1]) for e in ev]))
    pr_ms = float(np.mean([e[1].elapsed_time(e[2]) for e in ev]))
    clocks = sampler.stop()
    # parity of the TIMED step, on every rank: LL, mean and variance of the first N_CHECK objects against the oracle
    from oracle import gp_oracle as O              # the checker, never the thing measured
    y0m = y0.reshape(B, N_EPOCH)
    sel = slice(0, N_CHECK)
    ll_o = O.ll_batched_1d(x[sel], y[sel], y0m[sel], ye[sel], HYP, NUGGET)
    mean_o, var_o = O.predict_batched_1d(x[sel], y[sel], y0m[sel], ye[sel], HYP, NUGGET, grid, ny0[sel])
    chk = {"ll": out[0][:N_CHECK].cpu().numpy(), "mean": out[1][:N_CHECK * M_GRID].cpu().numpy().reshape(N_CHECK, M_GRID),
           "var": out[2][:N_CHECK * M_GRID].cpu().numpy().reshape(N_CHECK, M_GRID)}
    rel = lambda a, b: float(np.max(np.abs(a - b) / np.abs(b)))
    parity = max(rel(chk["ll"], ll_o), rel(chk["mean"], mean_o), rel(chk["var"], var_o))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *out)

    # the likelihood evaluation alone, as the optimiser drives it: the compact LL kernel (its own factorisation, rows retired)
    # + the device reduction + 16 bytes back; kernel time by CUDA events, wall time of the whole call
    batch.log_likelihood_total(HYP, NUGGET)
    for _ in range(3):
        batch.ll_dev(HYP, NUGGET)
    torch.cuda.synchronize()
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_ll = max(5, args.steps)
    k0.record()
    for _ in range(n_ll):
        batch.ll_dev(HYP, NUGGET)
    k1.record(); torch.cuda.synchronize()
    ll_ms = k0.elapsed_time(k1) / n_ll
    t0 = time.perf_counter()
    for _ in range(n_ll):
        ll_tot, _bad = batch.log_likelihood_total(HYP, NUGGET)
    ll_wall_ms = (time.perf_counter() - t0) / n_ll * 1e3
    parity = max(parity, abs(ll_tot - float(out[0].sum().item())) / abs(ll_tot))
    if world > 1:
        t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())

    # ---- end to end through the numpy-in/numpy-out layer: every step uploads the step's inputs from
    # pinned host memory, runs LL + predict and downloads ll/mean/var; chunks of objects (ramping up from
    # 2048 to a sixteenth of the batch and down again) are pipelined: one upload stream, one download stream,
    # kernels of consecutive chunks on 8 compute streams -- one native call per step (cgp_streamer_run); a chunk of
    # x | y | y_err travels as ONE two-dimensional copy, mean | var likewise, the per-object scalars once per run
    from cosmogp_b200.batch import StreamedEvaluator
    n_chunks = int(os.environ.get("CGP_E2E_CHUNKS", "0")) or max(1, min(16, B // 4096))     # chunks stay on the two-kernel route (>= 2048 objects)
    ev_e2e = StreamedEvaluator(B, N_EPOCH, M_GRID, dim=1, n_chunks=n_chunks, n_streams=int(os.environ.get("CGP_E2E_STREAMS", "8")), shared_mean=True)
    for name, arr in (("x", x), ("y", y), ("y_err", ye), ("template", tmpl), ("diff", d)):
        ev_e2e.host(name)[...] = arr
    # the mean at the epochs (template spline + offset, cosmogp/mean.py:84-90) is evaluated on the device from the
    # template itself -- the reference's own inputs (Mean_Y, Time_mean, diff) -- instead of uploading y0
    ev_e2e.set_mean_template(tmean, ymean)

    def e2e_step():
        tot, ll_h, mean, var, info = ev_e2e.run(HYP, NUGGET, grid)
        return ev_e2e.h2d_bytes, ev_e2e.d2h_bytes, tot
    e2e_steps = max(3, min(args.steps, 10))
    e2e_step(); e2e_step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        h2d, d2h, _ = e2e_step()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    parity = max(parity, rel(ev_e2e.host("ll")[sel], ll_o), rel(ev_e2e.host("mean")[sel], mean_o), rel(ev_e2e.host("var")[sel], var_o))
    # what the box's host side gives N ranks moving data in both directions at the same time (the bound of the end-to-end
    # leg beyond one GPU: tools/pcie_probe.py is the long form of this)
    npb = 8 * 1024 * 1024
    hb_in = torch.empty(npb, dtype=torch.float64, pin_memory=True).fill_(1.0); hb_out = torch.empty(npb, dtype=torch.float64, pin_memory=True)
    db_in = torch.empty(npb, dtype=torch.float64, device=dev); db_out = torch.ones(npb, dtype=torch.float64, device=dev)
    sa, sb = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    def duplex(reps):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            with torch.cuda.stream(sa): db_in.copy_(hb_in, non_blocking=True)
            with torch.cuda.stream(sb): hb_out.copy_(db_out, non_blocking=True)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / reps
    duplex(2)
    duplex_s = duplex(6)
    if world > 1:
        t = torch.tensor([parity, e2e_s, duplex_s], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        parity, e2e_s, duplex_s = (float(v) for v in t.tolist())
    duplex_gbs = npb * 8 / duplex_s / 1e9
    assert parity < 1e-9, "rank %d: parity check of the timed step failed: %g" % (rank, parity)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    traffic, traffic_src = None, None   # DRAM bytes per launch of the dominant kernel: the committed ncu --set full capture
    try:
        if B == 100000:
            tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
            traffic, traffic_src = tj["predict_f"]["traffic"], tj.get("source", "profiles/ncu_traffic.json")
    except Exception:
        pass
    value = B * world * args.steps / (total_ms * 1e-3)
    # dominant kernel = the grid kernel: per grid point h build + mean dot + v = L^-1 h + |v|^2 (SURVEY 8d)
    fl_grid = M_GRID * (N_EPOCH ** 2 + 8.0 * N_EPOCH)
    fl_factor = flops_predict(N_EPOCH, M_GRID) - fl_grid + 2.0 * N_EPOCH       # + |z|^2 for the likelihood
    fl_step = fl_grid + fl_factor
    achieved = fl_grid * B / (pr_ms * 1e-3) * 1e-12
    line = {
        "metric": "gp_fits_per_sec", "value": value, "unit": "objects/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(B, world, args.scaling),
        "clocks": clocks,
        "e2e": {"value": B * world * e2e_steps / e2e_s, "unit": "objects/s", "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_s / e2e_steps * 1e3, "steps": e2e_steps,
                "path": "StreamedEvaluator.run -> cgp_streamer_run: pinned host in, pinned host out; chunks of objects "
                        "pipelined over upload / compute / download streams; the same two kernels per chunk as the resident step",
                "host_link": {"duplex_GBps_per_rank_each_direction": duplex_gbs, "ranks_at_once": world,
                              "transfer_bound_ms_per_step": max(int(h2d), int(d2h)) / (duplex_gbs * 1e9) * 1e3,
                              "what": "64 MB pinned copies in both directions on every rank at the same time, measured in this run: "
                                      "the step cannot be faster than its larger direction at this rate"}},
        "gpu_launches": int(launches),
        "roofline": {"bound": "tensor", "kernel": "gp64_kernel<1,PREDICT_FU,8>: predictive mean+variance on the (uniform) grid by block forward "
                     "substitution against the TMA-staged Cholesky factor (FP64 tensor pipe, DMMA.8x8x4)", "achieved": achieved,
                     "peak": peak_dmma, "unit": "TFLOP/s", "frac": achieved / peak_dmma, "traffic": traffic,
                     "traffic_source": traffic_src,
                     "peak_source": "FP64 DMMA m8n8k4 ceiling measured in this run (cgp_fp64_peak); MEASURED_PEAKS.json "
                                    "has no FP64 entry; DFMA ceiling %.2f" % peak_dfma,
                     "flop_per_object": fl_grid, "ms_per_launch": pr_ms,
                     "factor_kernel": {"ms_per_launch": fa_ms, "flop_per_object": fl_factor,
                                       "achieved": fl_factor * B / (fa_ms * 1e-3) * 1e-12,
                                       "frac": fl_factor * B / (fa_ms * 1e-3) * 1e-12 / peak_dmma,
                                       "what": "covariance + Cholesky + z = L^-1 r + log-likelihood; block rows written to the grid kernel's workspace as they retire"},
                     "whole_step": {"flop_per_object": fl_step, "achieved": fl_step * B * args.steps / (total_ms * 1e-3) * 1e-12,
                                    "frac": fl_step * B * args.steps / (total_ms * 1e-3) * 1e-12 / peak_dmma}},
        "ll_evaluation": {"kernel_ms": ll_ms, "wall_ms": ll_wall_ms, "flop_per_object": flops_ll(N_EPOCH),
                          "achieved": flops_ll(N_EPOCH) * B / (ll_ms * 1e-3) * 1e-12,
                          "frac": flops_ll(N_EPOCH) * B / (ll_ms * 1e-3) * 1e-12 / peak_dmma,
                          "what": "one simplex point of find_hyperparameters: compact LL kernel; wall = kernel + reduction on the "
                                  "device + 16 bytes back (DeviceBatch.log_likelihood_total)"},
    }
    line["parity_max_rel_err"] = parity
    line["parity"] = ("every rank: LL, mean and variance of %d objects of its timed resident step and of its end-to-end "
                      "step against the numpy oracle; max relative error over ranks, asserted < 1e-9" % N_CHECK)
    if not args.no_cpu and world == 1:
        import multiprocessing as mp
        cores = os.cpu_count() or 1
        kind = "reference" if reference_available() else "port"
        n_cpu = args.cpu_objects or 1000 * cores
        if kind == "reference":
            from oracle import ref_loader
            ref_loader.load()
        n_fac = 16 * cores
        with mp.get_context("fork").Pool(cores) as pool:
            cpu_pass(kind, False, x[:4 * cores], y[:4 * cores], ye[:4 * cores], tmean, ymean, grid, pool, cores)
            v, res = cpu_pass(kind, False, x[:n_cpu], y[:n_cpu], ye[:n_cpu], tmean, ymean, grid, pool, cores)
            v_svd, _r = cpu_pass(kind, True, x[:n_cpu // 2], y[:n_cpu // 2], ye[:n_cpu // 2], tmean, ymean, grid, pool, cores)
            fac_ref = None
            if kind == "reference":
                parts = np.array_split(np.arange(n_fac), cores)
                fr = pool.map(_facade_worker, [(x[q], y[q], ye[q], tmean, ymean, grid) for q in parts])
                fac_ref = n_fac / max(r[0] for r in fr)
        # the CPU leg doubles as a second checker: object 0's prediction by the reference itself against the timed step
        m_ref, v_ref = res[0][2], res[0][3]
        line["parity_vs_cpu_arm"] = float(max(np.max(np.abs(chk["mean"][0] - m_ref) / np.abs(m_ref)),
                                              np.max(np.abs(chk["var"][0] - v_ref) / np.abs(v_ref))))
        assert line["parity_vs_cpu_arm"] < 1e-9, "object 0 differs from the CPU arm: %g" % line["parity_vs_cpu_arm"]
        line["cpu_baseline"] = {"value": v, "unit": "objects/s", "cores": cores, "kind": kind,
                                "sample": "first %d of the %d objects, one pass (compute_log_likelihood + get_prediction with "
                                          "COV=True per object, svd_method=False), %s, %d processes x 1 BLAS thread, "
                                          "objects/s = sample / slowest worker" % (
                                              n_cpu, B, "unmodified reference from baseline/_ref" if kind == "reference"
                                              else "oracle port (baseline/_ref absent)", cores),
                                "svd_method_true": {"value": v_svd, "unit": "objects/s",
                                                    "what": "the reference's default argument, %d objects" % (n_cpu // 2)}}
        # the public facade used the way a cosmogp user would: construct -> find_hyperparameters -> get_prediction -> numpy (wall)
        import cosmogp_b200 as cg
        def facade():
            gp = cg.gaussian_process_nobject(y, x, y_err=ye, Mean_Y=ymean, Time_mean=tmean)
            gp.find_hyperparameters(hyperparameter_guess=[0.4, 3.0], svd_method=False)
            gp.get_prediction(new_binning=grid, COV='diag', svd_method=False)
            return gp
        facade()
        t0 = time.perf_counter()
        gp = facade()
        np.asarray(gp.Prediction); np.asarray(gp.prediction_variance)
        fs = time.perf_counter() - t0
        line["facade_e2e"] = {"value": B / fs, "unit": "objects/s", "seconds": fs, "fit_hyperparameters": [float(v) for v in gp.hyperparameters],
                              "what": "gaussian_process_nobject(numpy lists) -> find_hyperparameters (scipy fmin on the host, one device "
                                      "launch per simplex point) -> get_prediction -> numpy arrays; wall clock, all %d objects" % B,
                              "reference": None if fac_ref is None else {
                                  "value": fac_ref, "unit": "objects/s", "cores": cores,
                                  "what": "the unmodified reference doing the same calls (svd_method=False, COV=True) on %d objects, "
                                          "%d processes" % (n_fac, cores)}}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
