"""Batched Choi replicate sweep on the c5 inputs (bench.c5_inputs(): 64x64 grid, 36-point lofi prior, synth.MF_HYP, 8 agents,
120 iterations) against the single-run simulator.choi, with a parity check of sampled batched runs against the oracle loop.

    python profiles/tools/bench_choi_batched.py --runs 512 --seq-runs 3 --parity-runs 2 --out profiles/<name>.json

Reports coverage iterations/s of the batched sweep (device time split into planning / clustering + tours / stepping by CUDA
events, wall time of run() which ends in a device synchronise), the number of runs re-run on the single-run path for a
clustering tie, the sequential rate over a handful of runs (not extrapolated), and the card's name and power limit."""
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


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": out.stdout.strip().splitlines()[:1]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=512)
    ap.add_argument("--seq-runs", type=int, default=3)
    ap.add_argument("--parity-runs", type=int, default=2)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    from mfgp_coverage_b200 import simulator as sim
    from mfgp_coverage_b200._batched import BatchedRuns, _NoiseRow, choi_schedule
    from oracle import algorithms as oalg
    from tests.test_gpu_algorithms import _compare
    from tests.test_gpu_batched import _rows_to_arrays
    torch.cuda.set_device(0)
    truth_arr, prior_arr = bench.c5_inputs()
    A, T, sigma = bench.C5["agents"], bench.C5["iterations"], bench.C5["sigma_n"]
    T_logged = len(choi_schedule(T))
    R = args.runs
    starts = np.stack([synth.agents(A, 1000 + r) for r in range(R)])
    noise = np.stack([np.random.default_rng(5000 + r).normal(0, sigma, T_logged * A) for r in range(R)])
    out = {"workload": f"choi_hmf on the c5 inputs: {R} runs, {A} agents, {T} iterations ({T_logged} logged), 64x64 grid, "
                       "36-point lofi prior, synth.MF_HYP", "card": card()}

    BatchedRuns("choi", truth_arr, prior_arr, synth.MF_HYP, A, T, starts[:8], noise=noise[:8]).run()       # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    br = BatchedRuns("choi", truth_arr, prior_arr, synth.MF_HYP, A, T, starts, noise=noise)
    t1 = time.perf_counter()
    br.run()
    t2 = time.perf_counter()
    logs = br.logs(list(range(R)), exact_tie_loss=True)
    t3 = time.perf_counter()
    dev_ms = sum(br.phase_ms.values())
    out["batched"] = {
        "runs": R, "coverage_iterations": R * T_logged,
        "iterations_per_s_run": R * T_logged / (t2 - t1), "run_wall_s": t2 - t1, "setup_wall_s": t1 - t0,
        "device_ms": dict(br.phase_ms, total=dev_ms), "iterations_per_s_device": R * T_logged / (dev_ms * 1e-3),
        "tie_reruns": len(br.tie_reruns), "tie_rerun_rate": len(br.tie_reruns) / R, "logs_and_reruns_wall_s": t3 - t2,
        "iterations_per_s_with_logs_and_reruns": R * T_logged / (t3 - t1), "final_cap": br.cap}

    seq = lambda r, pos: sim.choi("choi_hmf", r, T, A, pos, truth_arr, sigma, prior_arr, synth.MF_HYP, False, None, True,  # noqa: E731
                                  noise_rng=np.random.default_rng(9000 + r))
    seq(0, starts[0].copy())                                                                            # warm-up
    seq_times = []
    for r in range(args.seq_runs):
        pos = starts[r].copy()
        torch.cuda.synchronize()
        s0 = time.perf_counter()
        seq(r, pos)
        torch.cuda.synchronize()
        seq_times.append(time.perf_counter() - s0)
    out["sequential"] = {"runs": args.seq_runs, "s_per_run": seq_times,
                         "iterations_per_s": T_logged * args.seq_runs / sum(seq_times)}
    out["speedup_iterations_per_s_run_vs_sequential"] = out["batched"]["iterations_per_s_run"] / out["sequential"]["iterations_per_s"]

    sample = np.sort(np.random.default_rng(0).choice(R, args.parity_runs, replace=False)).tolist()
    parity = []
    for r in sample:        # the oracle loop with the literal refit-per-pick planner; the test suite's tie-aware comparison
        ref = oalg.choi(r, T, A, starts[r].copy(), truth_arr, sigma, prior_arr, synth.MF_HYP, None,
                        _NoiseRow(noise[r]), fast_planner=False)
        l, a, s = _rows_to_arrays(logs[r], A)
        lo, ao, so = _rows_to_arrays(ref, A)
        try:
            _compare(l, a, s, lo, ao, so, truth_arr)
            ok, why = True, ""
        except AssertionError as e:
            ok, why = False, repr(e)[:300]
        parity.append({"run": r, "rerun": r in br.tie_reruns, "samples": int(s.shape[0]), "match": ok, "failure": why,
                       "max_abs_agent_diff_excl_xmax": float(np.max(np.abs(np.delete(a - ao, 2, axis=2))))
                       if a.shape == ao.shape else None})
    out["parity_vs_oracle"] = {"runs_checked": sample, "all_match": all(p["match"] for p in parity), "runs": parity}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
