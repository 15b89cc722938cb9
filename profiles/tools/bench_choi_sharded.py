"""Grid-sharded Choi planner (sharding.ShardPlanner, choi_shard_*) on the c4 inputs: 1024x1024 grid, 4096 MF training
points (tests/synth.py, as bench.make_workload builds them), the grid split into whole-column slices, one rank per GPU.

    torchrun --nproc_per_node K profiles/tools/bench_choi_sharded.py --picks 256 --out profiles/<name>_K.json

One planning round through sharding.plan_shards at the fixed threshold 0, which every variance exceeds, stopped after
`--picks` picks (the V cache holds N + picks rows, so it never grows): every rank count makes the same picks.  Reports, per run: the time to fill the cache (dense posterior
with the V cache, host clock around work that ends in a device synchronise, max over ranks), the picks and ms per pick
(CUDA events around the whole pick loop, max over ranks), the bytes one pick streams per rank (8 n G_local, n averaged over
the round) over that time against the 6542 GB/s copy rate (DESIGN.md section 4), the peak memory per rank, and the card's
name and power limit.  A round on a 64x64 grid first loads the kernels and warms the collective."""
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
import torch.distributed as dist  # noqa: E402

from tests import synth  # noqa: E402

COPY_GBS = 6542.0


def card(dev):
    out = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(dev), "nvidia_smi": out.stdout.strip().splitlines()[:1]}


def planning_round(model, n, picks, world, rank):
    from mfgp_coverage_b200 import sharding
    from mfgp_coverage_b200._coverage import CoverageGrid
    from mfgp_coverage_b200._engine import TensorAxes
    xy = synth.grid(n)
    lo, hi, ux, uy = sharding.column_split(xy, world, rank)
    grid = CoverageGrid(xy[lo:hi], base_index=lo, axes=TensorAxes(ux, uy, torch.device("cuda", torch.cuda.current_device())))
    model.engine.ensure_factor()
    torch.cuda.synchronize()
    dist.barrier()
    t0 = time.perf_counter()
    p = sharding.ShardPlanner(model, grid, chunk=picks)            # fills the cache; ends in a device synchronise
    fill_s = time.perf_counter() - t0

    def exchange(slots):
        recv = torch.empty((world, slots[0].numel()), dtype=slots[0].dtype, device=slots[0].device)
        dist.all_gather_into_tensor(recv, slots[0])
        return recv

    torch.cuda.synchronize()
    dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    idx = sharding.plan_shards([p], exchange, 0.0, chunk=picks, max_picks=picks)
    e1.record()
    torch.cuda.synchronize()
    k = len(idx)
    t = torch.tensor([fill_s, e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    fill_s, loop_ms = t.tolist()
    n_avg = p.n0 + (k - 1) / 2.0
    bytes_pick = 8.0 * n_avg * grid.G
    ms_pick = loop_ms / max(k, 1)
    return {"grid": f"{n}x{n}", "N": p.n0, "G_local": grid.G, "columns": [lo // n, hi // n], "fill_s": fill_s, "picks": k,
            "loop_ms": loop_ms, "ms_per_pick": ms_pick, "bytes_per_pick_per_rank": bytes_pick,
            "GBs_per_rank": bytes_pick / (ms_pick * 1e6), "fraction_of_copy_rate": bytes_pick / (ms_pick * 1e6) / COPY_GBS,
            "cache_GB_per_rank": p.Vc.numel() * 8 / 1e9}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--picks", type=int, default=256)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    world, rank = dist.get_world_size(), dist.get_rank()
    from mfgp_coverage_b200 import simulator as sim
    try:
        base = synth.grid(1024)
        X_L, y_L, X_H, y_H = synth.training_set(base, synth.truth_function(base), 4096)
        model = sim.init_MFGP(synth.MF_HYP, np.column_stack((X_L, y_L)))
        model.updt_info(X_L, y_L, X_H, y_H)
        planning_round(model, 64, 32, world, rank)                  # warm-up: kernels loaded, collective set up
        torch.cuda.reset_peak_memory_stats()
        res = planning_round(model, 1024, args.picks, world, rank)
        peak = torch.tensor([torch.cuda.max_memory_allocated() / 1e9], dtype=torch.float64, device="cuda")
        dist.all_reduce(peak, op=dist.ReduceOp.MAX)
        res.update(world=world, peak_GB_per_rank=float(peak.item()), copy_rate_GBs=COPY_GBS, card=card(local),
                   workload="c4 inputs (tests/synth.py): 1024x1024 grid, 4096 MF samples, synth.MF_HYP; threshold 0, "
                            f"one round of {args.picks} picks")
        if rank == 0:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as fh:
                json.dump(res, fh, indent=1)
            print(json.dumps(res))
    finally:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
