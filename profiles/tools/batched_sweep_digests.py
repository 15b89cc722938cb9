"""Digests of the batched stepper's log buffers for seeded periodic_hmf and choi_hmf sweeps on the c5 inputs, and the device
time of the periodic_hmf loop.  Run it on two versions of the library and compare the JSON files: equal digests mean the two
versions compute the same bits for these algorithms.

    python profiles/tools/batched_sweep_digests.py --runs 512 --reps 3 --out profiles/<name>.json

The loop time is the stepper alone (BatchedRuns.run, eager launches and one CUDA graph replay, capture excluded), on fresh
state each repetition, with the card's name and power limit."""
import argparse
import hashlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from tests import synth  # noqa: E402

LOG_BUFFERS = ("log_loss", "log_agent", "log_sample", "nsamples", "pos")


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": out.stdout.strip().splitlines()[:1]}


def digests(br):
    return {name: hashlib.sha256(getattr(br, name).cpu().numpy().tobytes()).hexdigest() for name in LOG_BUFFERS}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=512)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    from mfgp_coverage_b200._batched import BatchedRuns, choi_schedule
    torch.cuda.set_device(0)
    truth_arr, prior_arr = bench.c5_inputs()
    A, T, sigma, R = bench.C5["agents"], bench.C5["iterations"], bench.C5["sigma_n"], args.runs
    starts = np.stack([synth.agents(A, 1000 + r) for r in range(R)])
    Tc = len(choi_schedule(T))
    noise = np.stack([np.random.default_rng(5000 + r).normal(0, sigma, Tc * A) for r in range(R)])
    out = {"workload": f"c5 inputs: {R} runs, {A} agents, {T} iterations, 64x64 grid, 36-point lofi prior, synth.MF_HYP",
           "card": card(), "digests": {}}
    make = lambda algo: BatchedRuns(algo, truth_arr, prior_arr, synth.MF_HYP, A, T, starts,  # noqa: E731
                                    noise=noise[:, :(Tc if algo == "choi" else T) * A])
    for algo in ("periodic", "choi"):
        out["digests"][algo] = digests(make(algo).run())
    make("periodic").run()                                   # warm-up of both modes
    make("periodic").run(use_graph=True)
    loop = {"eager": [], "graph": []}
    for _ in range(args.reps):                               # alternating, fresh state each time
        for mode in ("eager", "graph"):
            br = make("periodic")
            if mode == "graph":
                br.capture()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            br.run(use_graph=mode == "graph")
            e1.record()
            torch.cuda.synchronize()
            loop[mode].append(e0.elapsed_time(e1))
    out["periodic_loop_ms"] = {m: {"reps": v, "median": float(np.median(v))} for m, v in loop.items()}
    out["periodic_iterations_per_s_graph"] = R * T / (out["periodic_loop_ms"]["graph"]["median"] * 1e-3)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
