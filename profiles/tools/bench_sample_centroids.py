"""Per-cell centroids of joint posterior draws (CoverageGrid.sample_centroids: cov_cell_moments, cov_cell_moments_centroids)
against the per-draw route built from existing kernels, timed alternately in the same run, plus Thompson-sampling iterations.

    python profiles/tools/bench_sample_centroids.py --out profiles/r11_sample_centroids.json

Workload c4 (tests/synth.py MF hyper-parameters): the 1024 x 1024 grid, N = 4096, A = 64 cells (HybridVoronoi of
synth.agents(64, 4)), S = 1, 64, 256 draws.  Per S, after a warm-up of every shape, `rounds` alternating rounds of:
  * call_ms       the whole sample_centroids call (coefficients, moments, centroids, the tie-count read and the area upload)
  * coef_ms       the draws' coefficients (mfgp_grid_sample_coef, via DeviceGP.posterior_sample_grid_coef)
  * moments_ms    cov_cell_moments (CoverageGrid.cell_moments)
  * centroid_ms   cov_cell_moments_centroids
  * per_draw_ms   the per-draw route: the same coefficients, then per draw mfgp_grid_sample_eval of that draw (S = 1; the
                  evaluator's even row pitch leaves F_s strided, so it is copied to a contiguous vector) and one
                  cov_assign_reduce_grid pass with w = F_s
Each number is the median over the rounds of CUDA-event times of `reps` back-to-back calls.  Outputs are checked against the
per-draw route (max relative error of the partials over the sum of their terms' magnitudes, max centroid difference).
thompson_iter_s: wall time per iteration of simulator.thompson at c4 with 64 agents (runs of 1 and 6 iterations, the
difference over 5: the set-up cancels).  The card's name and power limit are read in the same run."""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from tests import synth  # noqa: E402


def card():
    out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()),
                          "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": out.stdout.strip().splitlines()[:1]}


def timed(fn, reps):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def model(xy, N):
    from mfgp_coverage_b200.gaussian_process import MFGP
    X_L, y_L, X_H, y_H = synth.training_set(xy, synth.truth_function(xy), N)
    m = MFGP(X_L, y_L, X_H, y_H, 1, 1)
    m.hyp = synth.MF_HYP
    m.updt_info(X_L, y_L, X_H, y_H)
    m.engine.ensure_factor()
    m.engine.check_factor(force=True)
    return m


def run_c4(S_values, reps, rounds):
    from mfgp_coverage_b200 import _native as nat
    from mfgp_coverage_b200._coverage import CoverageGrid, HybridVoronoi
    lib = nat.lib()
    xy = synth.grid(1024)
    m = model(xy, 4096)
    eng = m.engine
    g = CoverageGrid(xy)
    axes = g.axes
    bb = (0.0, 1.0, 0.0, 1.0)
    vor = HybridVoronoi(synth.agents(64, 4), bb)
    plan = eng._grid_sample_plan(axes)
    rx, ry = plan["rx"], plan["ry"]
    box = [ctypes.c_double(v) for v in plan["box"]]
    d = eng.grid_sample_dim(axes)
    f64 = dict(dtype=torch.float64, device=eng.device)
    g.sample_centroids(m, vor, torch.randn((d, 1), **f64))          # builds Qhull's cells if the pass meets ties
    A = len(vor)
    areas = torch.from_numpy(np.ascontiguousarray(vor.areas())).to(eng.device)
    mean = ctypes.c_double(eng.params["mean_H"])
    out = []
    for S in S_values:
        E = torch.randn((d, S), **f64)
        C, _ = eng.posterior_sample_grid_coef(axes, E)
        mom, ties, _ = g.cell_moments(vor, plan["box"], (rx, ry))
        cent = torch.empty((S, A, 4), **f64)
        cen = torch.empty((S, A, 2), **f64)
        Fs = torch.empty((g.G, 2), **f64)
        ew = int(lib.mfgp_grid_sample_eval_workspace_bytes(axes.nx, axes.ny, rx, ry, 1))
        ework = torch.empty(ew // 8 + 2, **f64)
        res = g.assign_reduce(lloyd_vor=vor, w=Fs[:, 0])
        pd_cent = torch.empty((S, A, 4), **f64)

        def centroid():
            nat.check(lib.cov_cell_moments_centroids(nat.ptr(mom), A, rx, ry, nat.ptr(C), S, mean, nat.ptr(areas),
                                                     *(ctypes.c_double(v) for v in bb), nat.ptr(cent), nat.ptr(cen), None, 0,
                                                     nat.stream_ptr()), "centroids")

        def per_draw():
            Cd, _ = eng.posterior_sample_grid_coef(axes, E)
            for s in range(S):
                nat.check(lib.mfgp_grid_sample_eval(nat.ptr(axes.ux), axes.nx, nat.ptr(axes.uy), axes.ny, 0, axes.nx, *box, rx,
                                                    ry, nat.ptr(Cd[s]), 1, mean, nat.ptr(Fs), 2, nat.ptr(ework), ew,
                                                    nat.stream_ptr()), "eval")
                w = Fs[:, 0].contiguous()
                g.assign_reduce(lloyd_vor=vor, w=w, out=res)
                pd_cent[s].copy_(res["cent"])

        stages = dict(call_ms=lambda: g.sample_centroids(m, vor, E), coef_ms=lambda: eng.posterior_sample_grid_coef(axes, E),
                      moments_ms=lambda: g.cell_moments(vor, plan["box"], (rx, ry)), centroid_ms=centroid,
                      per_draw_ms=per_draw)
        for fn in stages.values():                                # warm-up of every shape
            fn()
        t = {k: [] for k in stages}
        for _ in range(rounds):
            for k, fn in stages.items():
                t[k].append(timed(fn, reps if k != "per_draw_ms" else max(1, reps // 4)))
        cent_new, cen_new = g.sample_centroids(m, vor, E)
        per_draw()
        scale = torch.empty((S, A), **f64)
        for s in range(S):                                        # sums of |F_s| per cell: the scale of the partials
            nat.check(lib.mfgp_grid_sample_eval(nat.ptr(axes.ux), axes.nx, nat.ptr(axes.uy), axes.ny, 0, axes.nx, *box, rx, ry,
                                                nat.ptr(C[s]), 1, mean, nat.ptr(Fs), 2, nat.ptr(ework), ew, nat.stream_ptr()),
                      "eval")
            g.assign_reduce(lloyd_vor=vor, w=Fs[:, 0].abs().contiguous(), out=res)
            scale[s].copy_(res["cent"][:, 0])
        from mfgp_coverage_b200._coverage import centroids_from_partials
        pdc = pd_cent.cpu().numpy()
        ref_cen = np.stack([centroids_from_partials(pdc[s], vor.areas(), *bb) for s in range(S)])
        diff = (cent_new - pd_cent)[..., :3].abs()
        rel = (diff / scale[..., None]).max().item()
        r = dict(workload="c4", G=g.G, N=eng.N, A=A, S=S, orders=list(plan["orders"]), ties=int(ties.item()),
                 **{k: statistics.median(v) for k, v in t.items()}, spread={k: [min(v), max(v)] for k, v in t.items()},
                 check_partials_max_rel=rel, check_partials_max_abs=diff.max().item(),
                 check_cell0_draw0=[cent_new[0, 0].tolist(), pd_cent[0, 0].tolist()], check_counts_equal=bool(torch.equal(cent_new[..., 3], pd_cent[..., 3])),
                 check_centroids_max_abs=float(np.nanmax(np.abs(cen_new.cpu().numpy() - ref_cen))))
        r["speedup_vs_per_draw"] = r["per_draw_ms"] / r["call_ms"]
        print(json.dumps(r), flush=True)
        out.append(r)
        del E, C, mom, cent, cen
        torch.cuda.empty_cache()
    return out


def thompson_iteration():
    import pandas as pd
    from mfgp_coverage_b200 import simulator as sim
    xy = synth.grid(1024)
    f = synth.truth_function(xy)
    X_L, y_L, _, _ = synth.training_set(xy, f, 4096)
    truth = pd.DataFrame(np.column_stack((xy, f)), columns=["X", "Y", "f_H"])
    prior = pd.DataFrame(np.column_stack((X_L, y_L)), columns=["X", "Y", "f_prior"])
    hyp = pd.DataFrame([synth.MF_HYP])
    wall = {}
    for T in (1, 6, 1, 6):
        pos = synth.agents(64, 4)
        t0 = time.perf_counter()
        sim.thompson("thompson_hmf", 0, T, 64, pos, truth, 0.1, prior, hyp, False, None, True,
                     rng=np.random.default_rng(1), noise_rng=np.random.default_rng(2))
        torch.cuda.synchronize()
        wall.setdefault(T, []).append(time.perf_counter() - t0)
    return dict(thompson_runs_s={str(k): v for k, v in wall.items()}, thompson_iter_s=(min(wall[6]) - min(wall[1])) / 5)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r11_sample_centroids.json"))
    ap.add_argument("--reps", type=int, default=8)
    ap.add_argument("--rounds", type=int, default=5)
    a = ap.parse_args()
    torch.cuda.set_device(0)
    res = dict(card=card(), results=run_c4((1, 64, 256), a.reps, a.rounds))
    torch.cuda.empty_cache()
    res.update(thompson_iteration())
    res["card_after"] = card()
    print(json.dumps({k: v for k, v in res.items() if k != "results"}), flush=True)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
