"""Joint posterior draws over whole tensor-product grids (DeviceGP.posterior_sample_grid: mfgp_grid_sample_coef,
mfgp_grid_sample_eval), with DGEMM and a device copy timed in the same run for the bounds.

    python profiles/tools/bench_posterior_sample_grid.py --out profiles/r10_posterior_sample_grid.json

Workloads (MF model, tests/synth.py hyper-parameters):
  * c4          the 1024 x 1024 grid, N = 4096 (the c4 training set); S = 1, 64, 256
  * c4_16384    a 128 x 128 grid, N = 4096, S = 64, side by side with sample_posterior_device (Cholesky of the covariance)
                on the same points
  * ref_2601    the reference's scale: the 51 x 51 grid, N = 259; S = 1, 64
Per workload and S, each timed with CUDA events after a warm-up call of every shape:
  * call_ms     the whole posterior_sample_grid call (allocations included), normals and output preallocated
  * coef_ms     mfgp_grid_sample_coef (prior coefficients, residual at the training points, W^T W R, B^T alpha)
  * eval_ms     mfgp_grid_sample_eval (basis tables, Hc = Ux C^T, grid_sample_eval_kernel) over every column
  * kernel_ms   grid_sample_eval_kernel alone, from a torch.profiler pass of its own (c4 only)
For the evaluation: MAC = G S ry + ncols S ry kpad, bytes = 8 G S (F's stores; the inputs are L2-resident), the bound is the
larger of 2 MAC / DGEMM rate and bytes / copy rate (a 2 GiB device-to-device copy, read + write), and `of_bound` = bound / time.
F is 0.5 / 2.1 GB at c4 with S = 64 / 256, far past the 126 MB L2.  The card's name and power limit are read in the same run."""
import argparse
import ctypes
import json
import os
import subprocess
import sys

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
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def dgemm_tflops():
    a = torch.randn((8192, 8192), dtype=torch.float64, device="cuda")
    c = torch.empty_like(a)
    return 2 * 8192 ** 3 / timed(lambda: torch.mm(a, a, out=c), 10) / 1e9


def copy_gbs():
    a = torch.empty(1 << 28, dtype=torch.float64, device="cuda")
    b = torch.empty_like(a)
    return 2 * 8 * a.numel() / timed(lambda: b.copy_(a), 10) / 1e6


def model(n, N):
    from mfgp_coverage_b200.gaussian_process import MFGP
    xy = synth.grid(n)
    X_L, y_L, X_H, y_H = synth.training_set(xy, synth.truth_function(xy), N)
    m = MFGP(X_L, y_L, X_H, y_H, 1, 1)
    m.hyp = synth.MF_HYP
    m.updt_info(X_L, y_L, X_H, y_H)
    m.engine.ensure_factor()
    m.engine.check_factor(force=True)
    return m


def kernel_ms(fn, name, reps=5):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    us = 0.0
    for e in prof.key_averages():
        if name in e.key:
            us += getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
    return us / reps / 1e3


def run(name, m, xy, s_values, reps, rates, compare=False, profile_kernel=False):
    from mfgp_coverage_b200 import _native as nat
    from mfgp_coverage_b200._coverage import CoverageGrid
    eng = m.engine
    lib = nat.lib()
    g = CoverageGrid(xy)
    axes = g.axes
    G, N = g.G, eng.N
    d = eng.grid_sample_dim(axes)
    plan = eng._grid_sample_plan(axes)
    rxL, ryL, rxH, ryH = plan["orders"]
    rx, ry = plan["rx"], plan["ry"]
    kpad = -(-rx // 4) * 4
    f64 = dict(dtype=torch.float64, device=eng.device)
    out = []
    for S in s_values:
        lde = S + S % 2
        E = torch.randn((d, lde), **f64)[:, :S]
        F = torch.empty((G, lde), **f64)[:, :S]
        call_ms = timed(lambda: eng.posterior_sample_grid(axes, E, out=F), reps)
        C = torch.empty(S * ry * kpad, **f64)
        cw = int(lib.mfgp_grid_sample_coef_workspace_bytes(N, rxL, ryL, rxH, ryH, S))
        ew = int(lib.mfgp_grid_sample_eval_workspace_bytes(axes.nx, axes.ny, rx, ry, S))
        work = torch.empty(max(cw, ew) // 8 + 2, **f64)
        Q = plan["Q"]
        box = [ctypes.c_double(v) for v in plan["box"]]

        def coef():
            nat.check(lib.mfgp_grid_sample_coef(nat.ptr(eng.Xt), nat.ptr(eng.y), eng.NL, eng.NH, nat.ptr(eng.W), eng.npad, eng.cap,
                                                ctypes.byref(eng.pstruct), rxL, ryL, rxH, ryH, *box, nat.ptr(Q.get("Lx")),
                                                nat.ptr(Q.get("Ly")), nat.ptr(Q["Hx"]), nat.ptr(Q["Hy"]), nat.ptr(E), lde, S,
                                                nat.ptr(C), nat.ptr(work), work.numel() * 8, nat.stream_ptr()), "coef")

        def evaluate():
            nat.check(lib.mfgp_grid_sample_eval(nat.ptr(axes.ux), axes.nx, nat.ptr(axes.uy), axes.ny, 0, axes.nx, *box, rx, ry,
                                                nat.ptr(C), S, ctypes.c_double(eng.params["mean_H"]), nat.ptr(F), lde,
                                                nat.ptr(work), work.numel() * 8, nat.stream_ptr()), "eval")

        coef_ms = timed(coef, reps)
        eval_ms = timed(evaluate, reps)
        mac = G * S * ry + axes.nx * S * ry * kpad
        nbytes = 8 * G * S
        t_flop = 2 * mac / (rates["dgemm_tflops"] * 1e9)
        t_byte = nbytes / (rates["copy_gbs"] * 1e6)
        bound = max(t_flop, t_byte)
        r = dict(workload=name, G=G, N=N, S=S, d=d, orders=[rxL, ryL, rxH, ryH], call_ms=call_ms, coef_ms=coef_ms,
                 eval_ms=eval_ms, eval_mac=mac, eval_bytes=nbytes, eval_tflops=2 * mac / eval_ms / 1e9,
                 eval_gbs=nbytes / eval_ms / 1e6, eval_bound_ms=bound, eval_bound_by="compute" if t_flop >= t_byte else "stores",
                 eval_of_bound=bound / eval_ms)
        if profile_kernel:
            k = kernel_ms(evaluate, "grid_sample_eval_kernel")
            r.update(kernel_ms=k, kernel_of_bound=bound / k if k > 0 else None)
        if compare:
            xs = g.xy
            En = torch.randn((G, lde), **f64)[:, :S]
            Fn = torch.empty((G, lde), **f64)[:, :S]
            r["sample_posterior_ms"] = timed(lambda: eng.posterior_sample(xs, En, axes=axes, out=Fn), max(2, reps // 2))
            del En, Fn
        print(json.dumps(r), flush=True)
        out.append(r)
        del E, F, C, work
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_posterior_sample_grid.json"))
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    torch.cuda.set_device(0)
    rates = dict(dgemm_tflops=dgemm_tflops(), copy_gbs=copy_gbs())
    torch.cuda.empty_cache()
    res = dict(card=card(), rates=rates, results=[])
    m = model(1024, 4096)
    res["results"] += run("c4", m, synth.grid(1024), (1, 64, 256), a.reps, rates, profile_kernel=True)
    gx = np.linspace(0, 1, 128)
    res["results"] += run("c4_16384", m, np.stack(np.meshgrid(gx, gx, indexing="ij"), axis=-1).reshape(-1, 2), (64,), a.reps,
                          rates, compare=True)
    del m
    torch.cuda.empty_cache()
    res["results"] += run("ref_2601", model(51, 259), synth.grid(51), (1, 64), a.reps, rates)
    res["card_after"] = card()
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
