#!/usr/bin/env python
"""bench.py -- the reference's headline hot path on B200: MF-GP posterior over the grid + coverage step.

One "step" = one coverage iteration of the workload (default: BASELINE.json config 4 -- synthetic 1024x1024 grid,
4096 MF training samples, 64 agents), i.e. what simulator.todescato does per iteration (simulator.py:888-904), through the
product's own stepper (simulator._Sim.step on one GPU, sharding.ShardedSim.step on a shard):
    refit from scratch: K assembly -> ONE tile-dataflow kernel (tiled Cholesky + forward substitution of the Chebyshev-factored
    posterior's right-hand sides + their Gram product) -> quadratic forms -> mean + variance at every grid point
    -> both bounded-Voronoi partitions clipped on the device, one fused pass (loss, weighted centroids, per-cell max-variance
    arg-max), O(agents) finishing on the device, ONE packed copy home (results, Cholesky status, clip flags, tie count).
`value` = grid points / s with everything resident in HBM; `e2e` = the same iteration through the drop-in Python API
with HOST numpy buffers (grid upload, mu/var download, re-upload into the coverage functions) inside the timed region.
N > 1 (torchrun, one rank per GPU): the FIXED grid of the named config is split into whole-column slices (strong scaling,
BASELINE config 4); every rank factorises the (small) training system itself and forward-substitutes only the right-hand
sides of its own x-interval; per-cell partial sums / arg-max come home through ONE all-gather.  The weak-scaling figure
(every GPU owns a full 1024x1024 shard of a wider grid) is measured in the same run and reported as `other_scaling`;
`--scaling weak|strong` forces one mode for `value`.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c4|c3|c2] [--dump-outputs DIR]

`--dump-outputs DIR` writes what the last timed step returned to its caller as DIR/<name>.npy (float64, at most 64 MB in
all); the inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import sys
import threading
import time

if "reference" in sys.argv:       # --impl reference: the CPU arm uses every host core, also under torchrun (which exports
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):     # OMP_NUM_THREADS=1 to its workers)
        os.environ[_v] = str(os.cpu_count() or 1)

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tests import synth  # noqa: E402

WORKLOADS = {
    # name: (grid side, N training, agents, description)
    "c4": (1024, 4096, 64, "c4: synthetic 1024x1024 grid, 4096 MF samples (1024 lofi + 3072 hifi), 64 agents"),
    "c3": (256, 1024, 16, "c3: synthetic 256x256 grid, 1024 MF samples, 16 agents"),
    "c2": (51, 309, 8, "c2-like: 51x51 grid, 309 MF samples, 8 agents"),
}
# DRAM bytes (read + write) of ONE posterior_kernel launch on the full c4 grid, from the ncu --set full capture in
# profiles/r01_posterior_v3_ncu_summary.txt (18.883 GB read + 0.040 GB written); algorithmic minimum 32 G + 8 N^2 = 0.17 GB:
# W (67 MB used) is re-read from L2 by every CTA and only partly stays resident next to the factor tables.
POSTERIOR_TRAFFIC_C4_1GPU = 18.883344e9 + 39.72864e6
# DRAM bytes (read + write) of ONE chol_dataflow_kernel launch at c4 (N = 4096, 832 right-hand-side columns after the truncation of
# the Chebyshev block, Gram product in the same launch): mean over the 11 step launches of the ncu pass over this command,
# profiles/r02_bench_c4_launches.csv (dram__bytes_read.sum 96.8 MB + dram__bytes_write.sum 46.3 MB).  Algorithmic: lower
# triangle of K in and L out (2 x 69 MB) + B in and Y out (2 x 27 MB) + lower tiles of M out (3 MB) = 195 MB; the measured
# traffic is lower because part of L, Y and M is still in the 126 MB L2 when the kernel ends (and B arrives from it).
CHOL_TRAFFIC_C4_1GPU = 96.788829e6 + 46.284102e6
DGEMM_PEAK_TFLOPS = 35.41   # cuBLAS DGEMM 8192^3 measured on this pool's B200 (profiles/r01_dgemm_peak.json);
#                             MEASURED_PEAKS.json carries no FP64 figure.  DMMA issue peak: 37.15 (r01_fp64_pipes.log)
DUMP_LIMIT = 64 << 20       # bytes written by --dump-outputs, all arrays together


def dump_outputs(path, arrays):
    """Writes every array as path/<name>.npy in float64."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit(f"bench: --dump-outputs would write {total} bytes, more than {DUMP_LIMIT}")
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


def make_workload(name, world=1, rank=0, scaling="weak"):
    """Synthetic inputs of one rank.  Weak scaling (default, SURVEY 8e: the grid points are independent units): every
    rank owns n columns x n rows of an (n * world) x n tensor-product grid over the unit square -- the per-GPU shard is
    the BASELINE grid, the whole grid grows with the number of GPUs.  Strong scaling: the n x n grid is split into
    whole-column slices.  Training set and agents are the same on every rank."""
    n, N, A, desc = WORKLOADS[name]
    base = synth.grid(n)
    fbase = synth.truth_function(base)
    X_L, y_L, X_H, y_H = synth.training_set(base, fbase, N)
    if scaling == "weak":
        ux, uy = np.linspace(0, 1, n * world), np.linspace(0, 1, n)
        c0, c1 = rank * n, (rank + 1) * n
    else:
        ux, uy = np.linspace(0, 1, n), np.linspace(0, 1, n)
        c0, c1 = (rank * n) // world, ((rank + 1) * n) // world
    xy = np.stack(np.meshgrid(ux[c0:c1], uy, indexing="ij"), axis=-1).reshape(-1, 2)
    # the truth function is normalised over the points it is given: evaluate it on the WHOLE grid and take the rank's slice, so
    # that every rank count sees the same global function (and the strong-scaling runs report the 1-GPU loss)
    f = synth.truth_function(np.stack(np.meshgrid(ux, uy, indexing="ij"), axis=-1).reshape(-1, 2))[c0 * n:c1 * n] if world > 1 \
        else synth.truth_function(xy)
    return dict(name=name, desc=desc, n=n, N=N, A=A, xy=xy, f=f, ux=ux, uy=uy, lo=c0 * n, hi=c1 * n,
                G_total=ux.size * uy.size, X_L=X_L, y_L=y_L, X_H=X_H, y_H=y_H, pos=synth.agents(A, 7), cen=synth.agents(A, 8))


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag = index, [], set(), False
        self.max_mhz = None
        self.active = False          # samples are taken only while set (the timed region); NVML is initialised before that --
        self.ready = threading.Event()   # nvmlInit takes driver locks that would stall the launches of a short timed region

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
                     nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                     nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake"}
            self.ready.set()
            while not self.stop_flag:
                if self.active:
                    self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    for bit, nm in names.items():
                        if r & bit:
                            self.reasons.add(nm)
                time.sleep(0.005 if self.active else 0.001)      # (idle wake-ups make no NVML call)
        except Exception as e:   # NVML missing: report that rather than fake numbers
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")
            self.ready.set()

    def result(self):
        self.active = False
        self.stop_flag = True
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


# ---------------------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port of the reference path on the host cores
# ---------------------------------------------------------------------------------------------------------------------

def cpu_step(w, sample_pts, threads=None):
    """The same iteration with the oracle (numpy/scipy) on a bounded sample of the grid: the first `sample_pts` points.
    Returns a dict: seconds of the fit (K assembly + Cholesky, paid once per iteration whatever the grid size), of the
    posterior over the sample, of the coverage step over the sample; the oracle's mu / var on the sample (bench.py checks
    the device results against them); BLAS threads in use."""
    from threadpoolctl import threadpool_info, threadpool_limits
    from oracle import coverage as ocov
    from oracle import gp as ogp
    p = ogp.GPParams.from_hyp(synth.MF_HYP)
    xy = w["xy"][:sample_pts]
    truth = np.column_stack((xy, w["f"][:sample_pts]))
    with threadpool_limits(limits=threads or (os.cpu_count() or 1)):
        blas = max([i.get("num_threads", 1) for i in threadpool_info() if i.get("user_api") == "blas"] or [1])
        t0 = time.perf_counter()
        L = ogp.cholesky(ogp.train_cov(p, w["X_L"], w["X_H"]))
        t1 = time.perf_counter()
        mu, var = ogp.posterior(p, xy, w["X_L"], w["y_L"], w["X_H"], w["y_H"], L=L, chunk=4096)
        t2 = time.perf_counter()
        bbox = ocov.bounding_box_of(w["xy"])
        ocov.compute_loss(ocov.voronoi_bounded(w["pos"], bbox), truth)
        lv = ocov.voronoi_bounded(w["cen"], bbox)
        ocov.compute_centroids(lv, xy, mu)
        try:
            ocov.compute_max_var(lv, truth, var)
        except ValueError:      # a bounded sample can leave cells empty; the reference raises there
            pass
        t3 = time.perf_counter()
    return {"fit_s": t1 - t0, "posterior_s": t2 - t1, "coverage_s": t3 - t2, "total_s": t3 - t0, "mu": mu, "var": var,
            "blas_threads": int(blas), "k0": p.k0}


def cpu_rate(w, r, sample_pts):
    """Whole-grid rate of the CPU arm from a bounded sample: the fit is paid once per iteration, posterior + coverage
    scale with the number of grid points -> G / (fit + (G / sample) * (posterior + coverage)).  (sample / total would
    charge the N^3/3 factorisation to every 16 K points and bias the per-point rate low.)"""
    G = float(w["G_total"])
    return G / (r["fit_s"] + G / sample_pts * (r["posterior_s"] + r["coverage_s"]))


def cpu_sample_points(w):
    return {"c4": 16384, "c3": 16384, "c2": 2601}[w["name"]]


def cpu_baseline_entry(w, r, pts, r1=None):
    e = {"value": cpu_rate(w, r, pts), "unit": "grid-points/s", "cores": os.cpu_count(), "blas_threads": r["blas_threads"],
         "kind": "port",
         "sample": f"one step on the first {pts} of {int(w['G_total'])} grid points with the full N={w['N']} training set "
                   f"(fit {r['fit_s']:.2f} s + posterior {r['posterior_s']:.2f} s + coverage {r['coverage_s']:.2f} s); value = "
                   "G / (fit + G/sample * (posterior + coverage)); oracle = numpy/scipy restatement of the reference (its own "
                   "G x G predict cannot run at this size)",
         "sample_rate_incl_fit": pts / r["total_s"]}
    if r1 is not None:
        e["value_1_thread"] = cpu_rate(w, r1, r1["pts"])
        e["sample_1_thread"] = f"same, BLAS limited to 1 thread, first {r1['pts']} points"
    return e


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = make_workload(args.workload, 1, 0, "strong")
    pts = cpu_sample_points(w)
    for _ in range(min(args.warmup, 1)):
        cpu_step(w, pts)
    runs = [cpu_step(w, pts) for _ in range(args.steps)]
    mean = {k: float(np.mean([r[k] for r in runs])) for k in ("fit_s", "posterior_s", "coverage_s", "total_s")}
    mean["blas_threads"] = runs[0]["blas_threads"]
    value = cpu_rate(w, mean, pts)
    line = base_line(args, w, value, mean["total_s"] * 1e3)        # ms_per_step: one bounded-sample step as it was timed
    line.update({"impl": "reference", "extrapolated_full_grid_ms_per_step": w["G_total"] / value * 1e3, "dtype": "f64", "gpu_launches": 0,
                 "cpu_baseline": cpu_baseline_entry(w, mean, pts),
                 "e2e": {"value": value, "unit": "grid-points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
    print(json.dumps(line))


def base_line(args, w, value, ms, world=None, scaling=None):
    """Keys shared by both arms; `config` is a function of (workload, number of GPUs, scaling mode) only, so the reference arm
    launched with the same flags prints the same config."""
    world = int(os.environ.get("WORLD_SIZE", "1")) if world is None else world
    scaling = getattr(args, "scaling", "strong") if scaling is None else scaling
    n = w["n"]
    G = n * n * (world if scaling == "weak" else 1)
    shard = (f"weak scaling: every GPU owns a {n}x{n}-point shard (whole columns) of a {n * world}x{n} grid"
             if scaling == "weak" else f"strong scaling: the fixed {n}x{n} grid split into whole-column slices")
    return {"metric": "GP posterior mean+var + coverage step, grid-points/s (coverage iterations/s = 1000/ms_per_step)",
            "value": value, "unit": "grid-points/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "data": "synthetic",
            "config": {"workload": w["desc"], "grid_points": int(G), "grid_points_per_gpu": int(G // world),
                       "train_points": int(w["N"]), "agents": int(w["A"]), "parallelism": f"grid-sharded x{world} ({shard})",
                       "l2_policy": "L2 flushed between steps (256 MB write)"}}


# ---------------------------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------------------------

def run_ours(args):
    import torch
    import torch.distributed as dist
    from mfgp_coverage_b200 import _native as nat
    from mfgp_coverage_b200 import _coverage as cv
    from mfgp_coverage_b200 import sharding
    from mfgp_coverage_b200 import simulator as sim
    from mfgp_coverage_b200._engine import TensorAxes

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    bbox = np.array([0.0, 1.0, 0.0, 1.0])
    flush = torch.empty(64 << 20, dtype=torch.float32, device=dev)     # 256 MB > 126 MB L2
    empty_x, empty_y = np.empty((0, 2)), np.empty((0, 1))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed_region(fn, steps):
        """K steps between barriers; device timeline (CUDA events), max over ranks."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = None
        for _ in range(steps):
            out = fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps, out

    class Arm:
        """One workload on this rank: model, device-resident grid (shard), and the step the product runs per iteration:
        simulator._Sim.step on one GPU, sharding.ShardedSim.step on a grid shard."""

        def __init__(self, scaling):
            self.w = w = make_workload(args.workload, world, rank, scaling)
            self.model = sim.init_MFGP(synth.MF_HYP, np.column_stack((w["X_L"], w["y_L"])))
            self.model.updt_info(w["X_L"], w["y_L"], w["X_H"], w["y_H"])      # uploads the training set once
            self.eng = self.model.engine
            self.eng.profile_events = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            self.chol_ms = []
            if world == 1:
                self.state = sim._Sim(np.column_stack((w["xy"], w["f"])))
            else:
                axes = TensorAxes(w["ux"], w["uy"], dev)
                self.state = sharding.ShardedSim(w["xy"], w["f"], axes, w["lo"], bbox)

        def step(self, timed=False):
            w = self.w
            flush.zero_()
            self.eng.refactor(check=False)         # the reference refits every iteration (simulator.py:888-891): factor stale
            if world == 1:
                loss, cent, axy, mv, _, _ = self.state.step(self.model, w["pos"], w["cen"])
                out = (loss, cent, axy, mv)
            else:
                loss, cent, idx, mv = self.state.step(self.model, w["pos"], w["cen"])
                out = (loss, cent, idx, mv)
            if timed and self.eng.profile_events[1].query():
                try:
                    self.chol_ms.append(self.eng.profile_events[0].elapsed_time(self.eng.profile_events[1]))
                except Exception:                  # never recorded (non-fused path)
                    pass
            return out

    main_scaling = args.scaling          # default "strong": BASELINE config 4 is the FIXED grid, sharded at 2 / 4 / 8 GPUs
    arm = Arm(main_scaling)
    w, eng, model = arm.w, arm.eng, arm.model
    G_total, npts = w["G_total"], w["hi"] - w["lo"]
    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(args.warmup):
        arm.step()
    eng.check_factor(force=True)
    sampler.ready.wait(timeout=10)
    sampler.active = True
    l0 = nat.lib().mfgp_launch_count()
    ms_dev, out = timed_region(lambda: arm.step(True), args.steps)
    # layout and route of the TIMED steps' fused fit (later sections -- incremental mode -- use other settings)
    timed_rhs_cols = getattr(arm.eng, "rhs_cols", None)
    timed_fused_gram = bool(getattr(arm.eng, "fused_gram", False))
    launches = nat.lib().mfgp_launch_count() - l0
    clocks = sampler.result()
    chk = min(npts, 1 << 16)
    mu_timed, var_timed = arm.state.mu[:chk].cpu().numpy(), arm.state.var[:chk].cpu().numpy()      # results of the last TIMED step
    if args.dump_outputs and rank == 0:         # N > 1: mu / var of rank 0's grid slice, the merged per-cell results
        dump_outputs(args.dump_outputs, {"mu": arm.state.mu.cpu().numpy(), "var": arm.state.var.cpu().numpy(), "loss": out[0],
                                         "centroids": out[1], "argmax_xy" if world == 1 else "argmax_index": out[2],
                                         "max_var": out[3]})
    plan = eng._fplan[1] if eng._fplan is not None else None

    # the other scaling mode at N > 1, reported inside the same line (never as `value`)
    other = None
    if world > 1 and not args.scaling_given:
        arm2 = Arm("weak")
        for _ in range(args.warmup):
            arm2.step()
        ms2, _ = timed_region(lambda: arm2.step(True), args.steps)
        other = {"scaling": "weak", "grid_points": int(arm2.w["G_total"]), "ms_per_step": ms2,
                 "value": arm2.w["G_total"] / (ms2 * 1e-3), "unit": "grid-points/s",
                 "note": f"every GPU owns a {w['n']}x{w['n']}-point shard of a {w['n'] * world}x{w['n']} grid (the per-GPU work of the "
                         "1-GPU line; the training system is the same)"}
        del arm2

    # instrumented steps (outside the timed region): where the step's time goes
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    bd = {"posterior (incl. the fused fit)": [], "cells + coverage kernels + finish": [], "host tail (copy home, O(A) finishing)": []}
    grid, state = arm.state.grid, arm.state
    k0 = float(eng.params["s_H"] + eng.params["rho"] ** 2 * eng.params["s_L"])
    for _ in range(3):
        flush.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        eng.refactor(check=False)
        ev[0].record()
        model.predict_device(grid.xy, state.mu, state.var, grid=grid)
        ev[1].record()
        lv, pv = cv.HybridVoronoi(w["cen"], bbox), cv.HybridVoronoi(w["pos"], bbox)
        res = grid.assign_reduce(lv, pv, w=state.mu, var=state.var, amax_k0=k0, amax_rel=cv.AMAX_REL)
        if world == 1:
            grid.finish(res, lv, pv, bbox, info=eng.info, with_ties=True)
        ev[2].record()
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        bd["posterior (incl. the fused fit)"].append(ev[0].elapsed_time(ev[1]))
        bd["cells + coverage kernels + finish"].append(ev[1].elapsed_time(ev[2]))
        bd["host tail (copy home, O(A) finishing)"].append(max(0.0, (t1 - t0) * 1e3 - ev[0].elapsed_time(ev[2])))
    pm = float(np.mean(bd["posterior (incl. the fused fit)"]))

    # SURVEY 8(d) metric 1, "factor cached" variant: the posterior alone with the factor standing (a second predict without new data)
    cached = None
    if plan is not None:
        eng.defer_fit = False
        eng.refactor(check=True)                 # eager: L, W and z standing
        eng.posterior(grid.xy, state.mu, state.var, axes=grid.axes, g_lo=w["lo"])
        torch.cuda.synchronize()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 5
        c0.record()
        for _ in range(reps):
            eng.posterior(grid.xy, state.mu, state.var, axes=grid.axes, g_lo=w["lo"])
        c1.record()
        torch.cuda.synchronize()
        cms = c0.elapsed_time(c1) / reps
        cerr = (float((state.var[:chk].cpu() - torch.from_numpy(var_timed)).abs().max().item()) / k0,
                float((state.mu[:chk].cpu() - torch.from_numpy(mu_timed)).abs().max().item()))
        cached = {"what": "posterior only, factor (L, W, z) standing: tables + Y = W [B | z] + Gram product + quadratic forms + evaluation",
                  "ms": cms, "grid_points_per_s": npts * world / (cms * 1e-3) if world == 1 else npts / (cms * 1e-3),
                  "max_diff_vs_timed_steps": {"var_rel_k0": cerr[0], "mu_abs": cerr[1]}}
        eng.defer_fit = True

    # the dense DMMA posterior kernel on a 64-column sub-grid, for reference (it is the path of arbitrary point lists)
    dense = None
    axes = grid.axes
    if plan is not None:
        sub = min(64, npts // axes.ny) * axes.ny
        eng.use_factored = False
        for _ in range(2):
            eng.posterior(grid.xy[:sub], state.mu[:sub], state.var[:sub], axes=axes, g_lo=w["lo"])
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        eng.posterior(grid.xy[:sub], state.mu[:sub], state.var[:sub], axes=axes, g_lo=w["lo"])
        e1.record()
        torch.cuda.synchronize()
        eng.use_factored = True
        dms = e0.elapsed_time(e1)
        dfl = float(sub) * w["N"] * w["N"] + 4.0 * sub * w["N"]
        dense = {"kernel": "posterior_kernel (dense DMMA path, arbitrary point lists)", "grid_points": int(sub), "ms": dms,
                 "achieved": dfl / (dms * 1e-3) * 1e-12, "unit": "TFLOP/s", "frac": dfl / (dms * 1e-3) * 1e-12 / DGEMM_PEAK_TFLOPS,
                 "grid_points_per_s": sub / (dms * 1e-3)}

    # end-to-end through the reference-style call sequence with HOST buffers: updt_hifi -> predict(x_star) ->
    # voronoi_bounded + compute_loss / compute_centroids / compute_max_var (simulator.py:888-904); host arrays in and out
    xs_host = np.ascontiguousarray(w["xy"])
    truth_host = np.ascontiguousarray(np.column_stack((w["xy"], w["f"])))

    def e2e_step():
        model.updt_hifi(empty_x, empty_y)                 # the reference refits every iteration (simulator.py:888-891)
        mu_h, var_h = model.predict(xs_host)              # D2H mean + variance (the grid upload is cached by identity)
        loss_vor = sim.voronoi_bounded(w["pos"], bbox)
        loss = sim.compute_loss(loss_vor, truth_host)
        lloyd_vor = sim.voronoi_bounded(w["cen"], bbox)
        cent = sim.compute_centroids(lloyd_vor, xs_host, mu_h)            # H2D mean
        try:
            axy, mv = sim.compute_max_var(lloyd_vor, truth_host, var_h)   # H2D variance
        except ValueError:          # N > 1: a rank's shard need not hold points of every cell (np.amax([]) in the reference)
            if world == 1:
                raise
            axy = None
        return loss, cent, axy

    e2e_step()
    ms_e2e, out_e2e = timed_region(e2e_step, max(1, min(args.steps, 5)))
    h2d = npts * (8 + 8) + w["A"] * 2 * 16
    d2h = npts * 16 + w["A"] * 8 * 8

    # incremental iteration (SURVEY 8f rank 1, reported separately -- never as `value`): every agent takes one new
    # hifi sample; the factor is bordered (mfgp_cholesky_append) instead of refactored, then posterior + coverage step.
    npad_main = eng.npad
    rng_inc = np.random.default_rng(5)
    pool = rng_inc.permutation(w["n"] * w["n"])
    basegrid = synth.grid(w["n"])
    used = {tuple(r) for r in w["X_H"]}
    pool = [i for i in pool if tuple(basegrid[i]) not in used]
    inc_steps = max(1, min(args.steps, 5))
    inc = None
    if world == 1:
        mu, var = state.mu, state.var
        eng.incremental = True
        eng.refactor(check=False)
        eng.posterior(grid.xy, mu, var, axes=axes, g_lo=w["lo"])
        cursor = [0]
        clip = [None, None]

        def inc_step():
            idx = pool[cursor[0]:cursor[0] + w["A"]]
            cursor[0] += w["A"]
            x_new = basegrid[idx]
            y_new = (synth.truth_function(x_new) + rng_inc.normal(0, 0.1, len(idx))).reshape(-1, 1)
            eng.append_hifi(x_new, y_new, check=False)                 # H2D of the new samples + bordered factor update
            eng.posterior(grid.xy, mu, var, axes=axes, g_lo=w["lo"])   # factored: only the new rows of Y = W B
            clip[0] = cv.ClippedVoronoi(w["pos"], bbox, reuse=clip[0])
            clip[1] = cv.ClippedVoronoi(w["cen"], bbox, reuse=clip[1])
            res = grid.assign_reduce(clip[1], clip[0], w=mu, var=var)
            loss, cent, _, out3 = grid.finish(res, clip[1], clip[0], bbox, info=eng.info)
            return loss, cent, out3

        inc_step()                                                     # warm-up (grows the factor buffers once)
        ms_inc, out_inc = timed_region(inc_step, inc_steps)
        eng.check_factor(force=True)
        mu_i, var_i = mu.clone(), var.clone()
        eng.incremental = False
        eng.defer_fit = False
        eng.refactor(check=True)                                       # from-scratch factor of the grown model
        eng.posterior(grid.xy, mu, var, axes=axes, g_lo=w["lo"])
        inc_err = (float((var_i - var).abs().max().item()) / k0, float((mu_i - mu).abs().max().item()))
        inc = {"ms_per_step": ms_inc, "value": G_total / (ms_inc * 1e-3), "unit": "grid-points/s",
               "iterations_per_s": 1000.0 / ms_inc, "appended_per_step": int(w["A"]), "steps": inc_steps,
               "train_points_end": int(eng.N), "max_err_vs_refit": {"var_rel_k0": inc_err[0], "mu_abs": inc_err[1]},
               "note": "throughput mode: bordered Cholesky append + incremental (factored) posterior + coverage step on "
                       "device-built Voronoi cells, one D2H per iteration; the reference refits from scratch every iteration "
                       "(that is `value`)"}

    if rank == 0:
        value = G_total / (ms_dev * 1e-3)
        N = w["N"]
        line = base_line(args, w, value, ms_dev, world, main_scaling)
        chol_ms = arm.chol_ms
        if plan is not None:
            wv = max(plan["ryL"], plan["ryH"])                 # both kernel parts share one Chebyshev basis
            R = wv * max(plan["rxL"], plan["rxH"])
            if timed_rhs_cols:                                 # truncated column layout: the columns actually carried
                R = int(timed_rhs_cols[0])
            ncols = plan["ncols"]
            macs = 0.5 * N * N * R + float(ncols) * N * R + float(ncols) * N * wv * wv + float(npts) * wv * wv
            flops = 2.0 * macs + N ** 3 / 3.0
            call = {"what": "whole posterior call: covariance + Chebyshev tables + tiled Cholesky/substitution + per-column Gram + evaluation",
                    "ms": pm, "share_of_step": pm / ms_dev, "algorithmic_flops": flops,
                    "achieved": flops / (pm * 1e-3) * 1e-12, "unit": "TFLOP/s",
                    "frac": flops / (pm * 1e-3) * 1e-12 / DGEMM_PEAK_TFLOPS,
                    "algorithmic_flops_note": "N^3/3 (Cholesky) + 2 (N^2 R / 2 + n_col N R + n_col N w^2 + G w^2), "
                                              "R = max rx * max ry, w = max ry",
                    "dense_equivalent_tflops": (float(npts) * N * N + 4.0 * npts * N) / (pm * 1e-3) * 1e-12}
            if chol_ms:
                # the dominant kernel of the step: ONE launch factors K and forward-substitutes [B | y - m] (R + 1 columns)
                km = float(np.mean(chol_ms))
                kfl = N ** 3 / 3.0 + float(N) * N * (R + 1)
                fused_gram = timed_fused_gram
                note = "N^3/3 + N^2 (R + 1), R = expansion columns carried (<= max rx * max ry: product-magnitude truncation)"
                kname = ("chol_dataflow_kernel (tiled Cholesky of K fused with the forward substitution of the R + 1 "
                         "right-hand sides of the factored posterior; persistent tile-dataflow kernel, FP64 DMMA)")
                if fused_gram:         # the same launch also accumulates M = Y^T Y (symmetric: N R (R + 1) / 2 MAC)
                    kfl += float(N) * R * (R + 1)
                    note = ("N^3/3 + N^2 (R + 1) + N R (R + 1), R = expansion columns carried (<= max rx * max ry: product-magnitude "
                            "truncation); the last term: the Gram product M = Y^T Y")
                    kname = ("chol_dataflow_kernel (tiled Cholesky of K fused with the forward substitution of the R + 1 "
                             "right-hand sides of the factored posterior AND their Gram product M = Y^T Y; persistent "
                             "tile-dataflow kernel, warp-specialised, FP64 DMMA)")
                roof = {"bound": "tensor",
                        "kernel": kname,
                        "achieved": kfl / (km * 1e-3) * 1e-12, "peak": DGEMM_PEAK_TFLOPS, "unit": "TFLOP/s",
                        "frac": kfl / (km * 1e-3) * 1e-12 / DGEMM_PEAK_TFLOPS,
                        "traffic": CHOL_TRAFFIC_C4_1GPU if (w["name"] == "c4" and N == 4096 and world == 1) else None,
                        "traffic_unit": "bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum)",
                        "algorithmic_flops": kfl, "algorithmic_flops_note": note,
                        "algorithmic_bytes": 8.0 * (N * (N + 64.0) + 2.0 * N * (R + 64)) + (4.0 * (R + 64) ** 2 if fused_gram else 0.0),
                        "fused_gram": fused_gram,
                        "kernel_ms": km, "kernel_share_of_step": km / ms_dev}
            else:
                roof = {"bound": "tensor", "kernel": "factored posterior (FP64 DMMA)", "achieved": call["achieved"],
                        "peak": DGEMM_PEAK_TFLOPS, "unit": "TFLOP/s", "frac": call["frac"], "traffic": None,
                        "algorithmic_flops": flops, "kernel_ms": pm, "kernel_share_of_step": pm / ms_dev}
            roof.update({"chebyshev_orders": [plan["rxL"], plan["ryL"], plan["rxH"], plan["ryH"]],
                         "rhs_columns": {"expansion": int(R), "full_tensor_block": int(wv * max(plan["rxL"], plan["rxH"])),
                                         "padded": int(timed_rhs_cols[1]) if timed_rhs_cols else None},
                         "posterior_call": call, "posterior_factor_cached": cached,
                         "peak_source": "cuBLAS DGEMM 8192^3 measured on this pool (profiles/r01_dgemm_peak.json); "
                                        "MEASURED_PEAKS.json has no FP64 figure; DMMA issue peak 37.15",
                         "dense_kernel": dense})
        else:
            flops = float(npts) * N * N + 4.0 * npts * N        # algorithmic: triangular solve + mean + column norm
            achieved = flops / (pm * 1e-3) * 1e-12
            roof = {"bound": "tensor", "kernel": "posterior_kernel (DMMA fp64)", "achieved": achieved,
                    "peak": DGEMM_PEAK_TFLOPS, "unit": "TFLOP/s", "frac": achieved / DGEMM_PEAK_TFLOPS, "traffic": None,
                    "kernel_ms": pm, "kernel_share_of_step": pm / ms_dev,
                    "peak_source": "cuBLAS DGEMM 8192^3 measured on this pool (profiles/r01_dgemm_peak.json)"}
        line.update({
            "dtype": "f64", "clocks": clocks, "gpu_launches": int(launches),
            "e2e": {"value": G_total / (ms_e2e * 1e-3), "unit": "grid-points/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": ms_e2e,
                    "api": "MFGP.updt_hifi + MFGP.predict(x_star) + voronoi_bounded + compute_loss / compute_centroids / "
                           "compute_max_var, numpy arrays in and out"},
            "roofline": roof,
            "breakdown_ms": {k: float(np.mean(v)) for k, v in bd.items()},
            "check": {"loss": float(out[0]), "loss_e2e": float(out_e2e[0]) if world == 1 else None, "npad": int(npad_main),
                      "posterior_path": "factored" if plan is not None else "dense",
                      "step": "simulator._Sim.step" if world == 1 else "sharding.ShardedSim.step"},
        })
        if inc is not None:
            line["incremental"] = inc
        if other is not None:
            line["other_scaling"] = other
        if world > 1:
            line["scaling_note"] = ("strong scaling of the fixed grid: every rank factorises the N x N training covariance itself "
                                    "(N^3/3 flop, a serial chain of N/64 diagonal blocks that more GPUs cannot shorten) and "
                                    "forward-substitutes only the right-hand sides of ITS x-interval; Amdahl bound of the step = "
                                    "t_cholesky / t_step(1 GPU)")
        parity_ok = True
        if world == 1:
            pts = cpu_sample_points(w)
            r = cpu_step(w, pts)
            p1 = max(256, pts // 16)
            r1 = cpu_step(w, p1, threads=1)
            r1["pts"] = p1
            line["cpu_baseline"] = cpu_baseline_entry(w, r, pts, r1)
            # parity of the exact path that was timed: device mu / var of the timed steps vs the oracle on the CPU sample
            err_var = float(np.max(np.abs(var_timed[:pts] - r["var"]))) / r["k0"]
            err_mu = float(np.max(np.abs(mu_timed[:pts] - r["mu"]))) / max(1.0, float(np.max(np.abs(r["mu"]))))
            parity_ok = err_var <= 1e-9 and err_mu <= 1e-9
            line["check"]["max_err_vs_oracle"] = {"var_rel_k0": err_var, "mu_rel": err_mu, "points": int(pts), "tolerance": 1e-9,
                                                  "ok": parity_ok,
                                                  "what": "posterior of the TIMED device steps (fused fit + factored posterior) vs "
                                                          "the oracle on the cpu_baseline sample points"}
        print(json.dumps(line))
        if not parity_ok:
            raise SystemExit("bench: the timed path disagrees with the oracle beyond 1e-9 -- the line above is INVALID")
    if world > 1:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------------------
# config c5: replicate sweep of independent periodic_hmf runs on 64x64 grids, run-sharded (no collective)
# ---------------------------------------------------------------------------------------------------------------------

C5 = dict(n=64, agents=8, iterations=120, lattice=6, sigma_n=0.1, total_runs=512,
          desc="c5: replicate sweep, independent periodic_hmf runs on 64x64 (4096-point) grids, 8 agents, 120 iterations, "
               "36-point lofi prior lattice (512 runs in the full sweep; a step is ONE whole run)")
C5_AGENT_COLS = ("X", "Y", "XMax", "YMax", "VarMax", "Var0", "XCentroid", "YCentroid", "ProbExplore", "Explore", "Distance")
C5_DUMP_RUNS = 256          # --dump-outputs keeps the logs of at most this many runs: 512 whole runs exceed DUMP_LIMIT


def c5_inputs():
    xy = synth.grid(C5["n"])
    truth_arr = np.column_stack((xy, synth.truth_function(xy)))
    g = (np.arange(C5["lattice"]) + 0.5) / C5["lattice"]
    lat = np.stack(np.meshgrid(g, g, indexing="ij"), axis=-1).reshape(-1, 2) + 0.013 * np.random.default_rng(11).random((36, 2))
    near = np.argmin(((xy[None, :, :] - lat[:, None, :]) ** 2).sum(axis=2), axis=1)
    prior_arr = np.column_stack((lat, 0.8 * truth_arr[near, 2] + 0.02))
    return truth_arr, prior_arr


def c5_log_arrays(logs):
    """The (loss_log, agent_log, sample_log) rows of the timed runs as arrays, for a fixed, seeded sample of at most
    C5_DUMP_RUNS runs: runs[R'] (the sampled run indices), loss[R', T], agent[R', T, A, 11] (the numeric columns of an
    agent row, in C5_AGENT_COLS order), samples[S, 6] (run index, Iteration, Agent, X, Y, Sample)."""
    R, T = len(logs), len(logs[0][0])
    runs = np.arange(R) if R <= C5_DUMP_RUNS else np.sort(np.random.default_rng(0).choice(R, C5_DUMP_RUNS, replace=False))
    num = lambda v: np.nan if isinstance(v, str) else float(v)       # noqa: E731   ("NA" cells of the reference's rows)
    loss = [[num(r["Loss"]) for r in logs[k][0]] for k in runs]
    agent = [[[num(r[c]) for c in C5_AGENT_COLS] for r in logs[k][1]] for k in runs]
    samples = [[k] + [num(r[c]) for c in ("Iteration", "Agent", "X", "Y", "Sample")] for k in runs for r in logs[k][2]]
    return {"runs": runs, "loss": np.array(loss), "agent": np.array(agent).reshape(len(runs), T, -1, len(C5_AGENT_COLS)),
            "samples": np.array(samples).reshape(-1, 6)}


def run_c5(args):
    """Each step is one complete periodic_hmf run (120 coverage iterations) through the drop-in simulator; every rank
    works through its own runs (run sharding: weak scaling, no data-path collective)."""
    import contextlib
    import io
    import random
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    truth_arr, prior_arr = c5_inputs()
    T, A = C5["iterations"], C5["agents"]
    if args.impl == "reference":
        if rank != 0:
            return
        from oracle import algorithms as oalg
        it = 12                                                    # bounded sample: the first 12 iterations of one run
        times = []
        for s in range(max(1, min(args.steps, 2))):
            t0 = time.perf_counter()
            oalg.periodic(s, it, A, synth.agents(A, 100 + s), truth_arr, C5["sigma_n"], prior_arr, synth.MF_HYP,
                          random.Random(s), np.random.default_rng(s))
            times.append(time.perf_counter() - t0)
        value = it / float(np.mean(times))
        line = {"metric": "coverage iterations/s (periodic_hmf replicate sweep)", "value": value, "unit": "iterations/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(np.mean(times)) * 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "data": "synthetic", "impl": "reference",
                "dtype": "f64", "gpu_launches": 0, "config": {"workload": C5["desc"], "parallelism": "1 host process"},
                "cpu_baseline": {"value": value, "unit": "iterations/s", "cores": os.cpu_count(), "kind": "port",
                                 "sample": f"first {it} iterations of one run (N grows 36 -> {36 + 8 * 5}), oracle loop"},
                "e2e": {"value": value, "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return
    import torch
    import torch.distributed as dist
    from mfgp_coverage_b200 import _native as nat
    from mfgp_coverage_b200 import simulator as sim
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    runs = args.steps                                      # a step is one whole run; the K runs of a rank are stepped TOGETHER

    def sweep(tag, use_graph=False):
        """K periodic_hmf runs on the batched stepper (simulator.run_batched): host arrays in, log rows out."""
        starts = np.stack([synth.agents(A, 100_000 * tag + 1000 * rank + k) for k in range(runs)])
        rngs = [np.random.default_rng(100_000 * tag + 1000 * rank + k) for k in range(runs)]
        logs = sim.run_batched("periodic_hmf", list(range(runs)), T, A, starts, truth_arr, C5["sigma_n"], prior_arr, synth.MF_HYP,
                               noise_rngs=rngs, use_graph=use_graph)
        return logs

    sampler = ClockSampler(local)
    sampler.start()
    for k in range(max(1, min(args.warmup, 2))):
        sweep(10 + k)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler.ready.wait(timeout=10)
    sampler.active = True
    l0 = nat.lib().mfgp_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_host0 = time.perf_counter()
    e0.record()
    logs = sweep(1)
    e1.record()
    torch.cuda.synchronize()
    t_host = time.perf_counter() - t_host0
    launches = nat.lib().mfgp_launch_count() - l0
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    clocks = sampler.result()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, c5_log_arrays(logs))
    # the device loop alone, eager launches vs ONE CUDA graph replay (capture excluded), on fresh state each
    from mfgp_coverage_b200._batched import BatchedRuns
    loop_ms = {}
    for mode in ("eager", "graph"):
        starts = np.stack([synth.agents(A, 7_000_000 + 1000 * rank + k) for k in range(runs)])
        br = BatchedRuns("periodic", truth_arr, prior_arr, synth.MF_HYP, A, T, starts,
                         noise=np.random.default_rng(3).normal(0, C5["sigma_n"], (runs, T * A)))
        if mode == "graph":
            br.capture()
        torch.cuda.synchronize()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        br.run(use_graph=mode == "graph")
        g1.record()
        torch.cuda.synchronize()
        loop_ms[mode] = g0.elapsed_time(g1)
        del br
    # the same run, one simulation at a time through simulator.periodic (the round-1 path), for comparison
    seq = None
    if rank == 0:
        import contextlib
        import io
        import random
        sim.INCREMENTAL = True
        ts = time.perf_counter()
        with contextlib.redirect_stdout(io.StringIO()):
            sim.periodic("periodic_hmf", 0, T, A, synth.agents(A, 100_000 + 1000 * rank), truth_arr, C5["sigma_n"], prior_arr,
                         synth.MF_HYP, False, None, True, rng=random.Random(0), noise_rng=np.random.default_rng(100_000 + 1000 * rank))
        torch.cuda.synchronize()
        seq = T / (time.perf_counter() - ts)
    if rank == 0:
        its = world * runs * T
        value = its / (ms * 1e-3)
        G = truth_arr.shape[0]
        line = {"metric": "coverage iterations/s (periodic_hmf replicate sweep)", "value": value, "unit": "iterations/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / runs,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "data": "synthetic", "dtype": "f64",
                "config": {"workload": C5["desc"], "grid_points": int(G), "agents": A, "iterations_per_run": T,
                           "runs_per_gpu_timed": runs, "parallelism": f"run-sharded x{world} (one process per GPU), {runs} runs "
                           "per GPU stepped together (simulator.run_batched: 3 kernel launches per iteration for all runs)",
                           "l2_policy": f"per-run state {4.0 * runs:.0f} MB per GPU: larger than L2 from ~32 runs on"},
                "clocks": clocks, "gpu_launches": int(launches),
                "e2e": {"value": world * runs * T / t_host, "unit": "iterations/s", "h2d_bytes_per_step": int(G * 24 + 36 * 24 + T * A * 8),
                        "d2h_bytes_per_step": int(T * A * 11 * 8 + T * 8 + T * A * 5 * 8), "host_seconds": t_host,
                        "note": "public API (simulator.run_batched: host arrays in, the reference's log-row dicts out), wall clock "
                                "including the construction of the log rows on the host"},
                "sweep_512_runs_s": {"device": 512.0 / (world * runs) * (ms * 1e-3), "with_host_log_rows": 512.0 / (world * runs) * t_host},
                "sequential_single_run_iterations_per_s": seq,
                "device_loop_ms": {"eager_launches": loop_ms["eager"], "one_cuda_graph": loop_ms["graph"],
                                   "what": f"{T} iterations x 3 launches for {runs} runs, device time of the loop only"},
                "grid_points_per_s": value * G,
                "check": {"final_loss_run0": float(logs[0][0][-1]["Loss"]), "samples_run0": len(logs[0][2])}}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS) + ["c5"])
    ap.add_argument("--scaling", default="strong", choices=["weak", "strong"],
                    help="N > 1: the fixed grid split over the GPUs (strong, default: BASELINE config 4) or a fixed per-GPU shard (weak)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned to DIR/<name>.npy (float64, at most 64 MB in all; --impl ours)")
    args = ap.parse_args()
    args.scaling_given = any(a.startswith("--scaling") for a in sys.argv[1:])
    if args.steps is None:      # c5: a step is one whole run and the runs of a rank are stepped together -> the full sweep
        args.steps = max(1, C5["total_runs"] // max(1, int(os.environ.get("WORLD_SIZE", "1")))) if args.workload == "c5" else 5
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the device path (--impl ours)")
    if args.workload == "c5":
        run_c5(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
