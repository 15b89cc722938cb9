"""Batched Thompson-sampling sweep on the c5 inputs (bench.c5_inputs(): 64x64 grid, 36-point lofi prior, synth.MF_HYP, 8 agents,
120 iterations), against the single-run simulator.thompson and the batched periodic_hmf sweep, with a replay check of sampled
batched runs against simulator.thompson (VORONOI = "clip") at the runs' device normals and noise.

    python profiles/tools/bench_thompson_batched.py --runs 512 --seq-runs 2 --parity-runs 2 --out profiles/<name>.json

Reports the device-loop time (CUDA events around BatchedRuns.run, eager launches and one CUDA graph replay, capture
excluded, fresh state each), the per-kernel split of an eager loop from torch.profiler (a run of its own), the wall time
including the log rows, the sequential rate over a handful of runs (not extrapolated), lower bounds computed from counts,
and the card's name and power limit."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from tests import synth  # noqa: E402

COPY_TBS = 6.54          # device copy rate this project measured (TB/s), for the W-streaming bound
DGEMM_TFLOPS = 35.4      # DGEMM rate this project measured (TFLOP/s, profiles/r09_posterior_sample.json), for the MAC bound


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": out.stdout.strip().splitlines()[:1]}


def timed(make, use_graph):
    br = make()
    if use_graph:
        br.capture()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    br.run(use_graph=use_graph)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), br


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=512)
    ap.add_argument("--seq-runs", type=int, default=2)
    ap.add_argument("--parity-runs", type=int, default=2)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    from mfgp_coverage_b200 import simulator as sim
    from mfgp_coverage_b200._batched import BatchedRuns, _NoiseRow
    from tests.test_gpu_batched_thompson import _DeviceNormals, _compare
    from oracle import sample_centroids as osc
    torch.cuda.set_device(0)
    truth_arr, prior_arr = bench.c5_inputs()
    A, T, sigma, R = bench.C5["agents"], bench.C5["iterations"], bench.C5["sigma_n"], args.runs
    starts = np.stack([synth.agents(A, 1000 + r) for r in range(R)])
    noise = np.stack([np.random.default_rng(5000 + r).normal(0, sigma, T * A) for r in range(R)])
    seeds = [0x9E3779B97F4A7C15 ^ r for r in range(R)]
    out = {"workload": f"thompson_hmf on the c5 inputs: {R} runs, {A} agents, {T} iterations, 64x64 grid, 36-point lofi prior, "
                       "synth.MF_HYP", "card": card()}
    make = lambda algo="thompson", n=R: BatchedRuns(algo, truth_arr, prior_arr, synth.MF_HYP, A, T, starts[:n],  # noqa: E731
                                                    noise=noise[:n], seeds=seeds[:n] if algo == "thompson" else None)
    make(n=8).run()                                                       # warm-up (modules, allocator)
    make(n=8).run(use_graph=True)
    loops = {"eager": [], "graph": [], "periodic_graph": [], "periodic_eager": []}
    for _ in range(args.reps):
        for key, algo, g in (("eager", "thompson", False), ("graph", "thompson", True), ("periodic_eager", "periodic", False),
                             ("periodic_graph", "periodic", True)):
            loops[key].append(timed(lambda: make(algo), g)[0])
    med = {k: float(np.median(v)) for k, v in loops.items()}
    out["device_loop_ms"] = {k: {"reps": v, "median": med[k]} for k, v in loops.items()}
    out["iterations_per_s"] = {k: R * T / (med[k] * 1e-3) for k in med}

    t0 = time.perf_counter()
    br = make()
    br.run()
    t1 = time.perf_counter()
    logs = br.logs()
    t2 = time.perf_counter()
    out["wall"] = {"setup_and_run_s": t1 - t0, "logs_s": t2 - t1, "iterations_per_s_with_logs": R * T / (t2 - t0)}

    # per-kernel split of one eager loop (a profiled run of its own; profiling slows the host, not the kernels)
    from torch.profiler import ProfilerActivity, profile
    br_p = make()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        br_p.run()
        torch.cuda.synchronize()
    kern = {}
    for ev in prof.key_averages():
        if ev.device_type is not None and "CUDA" in str(ev.device_type) and ev.self_device_time_total > 0:
            kern[ev.key] = {"ms": ev.self_device_time_total / 1e3, "calls": ev.count}
    stage = {"append": "batch_append_kernel", "posterior": "batch_posterior", "coverage": "batch_coverage_kernel",
             "draw_prior": "bt_prior_kernel", "draw_beta": "bt_beta_kernel", "draw_cell": "bt_cell_kernel"}
    out["kernels_profiled_eager"] = kern
    out["stage_ms_profiled"] = {s: sum(v["ms"] for k, v in kern.items() if n in k) for s, n in stage.items()}

    # counts-based lower bounds
    N0 = br.N0
    Ns = np.array([N0 + A * t for t in range(T)], dtype=np.float64)
    w_bytes = float(np.sum(Ns * Ns) * 8 * R)         # two passes over the lower triangle = one full N x N matrix of reads
    rxL, ryL, rxH, ryH = br.splan["orders"]
    rx, ry, G = max(rxL, rxH), max(ryL, ryH), br.G
    mac_prior = A * (rxL * ryL * (rxL + ryL) + rxH * ryH * (rxH + ryH)) * T * R
    mac_hc = A * 64 * ry * rx * T * R
    mac_beta = float(np.sum(Ns * Ns)) * A * R
    mac_cell = float(np.sum(Ns)) * G * (2 if br.params["multi"] else 1) * R + G * ry * T * R
    macs = {"prior_coef": mac_prior, "grid_eval_Hc": mac_hc, "beta": mac_beta, "cell": mac_cell}
    out["bounds_from_counts"] = {
        "W_stream_bytes": w_bytes, "W_stream_ms_at_copy_rate": w_bytes / (COPY_TBS * 1e12) * 1e3,
        "macs": macs, "mac_total": float(sum(macs.values())),
        "mac_ms_at_dgemm_rate": {k: 2 * v / (DGEMM_TFLOPS * 1e12) * 1e3 for k, v in macs.items()},
        "note": "not measured: computed from shapes; W bound at the measured copy rate, MAC bound at the measured DGEMM rate"}

    # sequential simulator.thompson on a few of the same runs
    seq_times = []
    for r in range(args.seq_runs + 1):
        pos = starts[r].copy()
        torch.cuda.synchronize()
        s0 = time.perf_counter()
        sim.thompson("thompson_hmf", r, T, A, pos, truth_arr, sigma, prior_arr, synth.MF_HYP, False, None, True,
                     rng=np.random.default_rng(seeds[r]), noise_rng=_NoiseRow(noise[r]))
        torch.cuda.synchronize()
        seq_times.append(time.perf_counter() - s0)
    seq_times = seq_times[1:]                                               # the first run warms up
    out["sequential"] = {"runs": args.seq_runs, "s_per_run": seq_times, "iterations_per_s": T * args.seq_runs / sum(seq_times)}
    out["speedup_graph_loop_vs_sequential"] = out["iterations_per_s"]["graph"] / out["sequential"]["iterations_per_s"]

    # replay: sampled batched runs against simulator.thompson (clip) at their device normals and noise
    sim.VORONOI = "clip"
    ux, uy = osc.tensor_axes(truth_arr[:, :2])
    parity = []
    for r in np.sort(np.random.default_rng(0).choice(R, args.parity_runs, replace=False)).tolist():
        ref = sim.thompson("thompson_hmf", r, T, A, starts[r].copy(), truth_arr, sigma, prior_arr, synth.MF_HYP, False, None,
                           True, rng=_DeviceNormals(br, r), noise_rng=_NoiseRow(noise[r]))
        try:
            n = _compare(logs[r], ref, A, ux, uy)
            parity.append({"run": r, "match": True, "iterations_compared": n})
        except AssertionError as e:
            parity.append({"run": r, "match": False, "failure": repr(e)[:300]})
    out["replay_vs_clip_thompson"] = {"all_match": all(p["match"] for p in parity), "runs": parity}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("card", "iterations_per_s", "stage_ms_profiled", "replay_vs_clip_thompson")}))


if __name__ == "__main__":
    main()
