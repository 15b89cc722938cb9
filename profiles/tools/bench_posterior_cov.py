"""Joint / cross posterior covariance (mfgp_posterior_cov, DeviceGP.posterior_cov) against cuBLAS DGEMM in the same run.

    python profiles/tools/bench_posterior_cov.py --out profiles/r08_posterior_cov.json

Workloads (MF model, tests/synth.py hyper-parameters; training sets as bench.make_workload builds them):
  * sym_2601   the reference's scale: the 51 x 51 grid, N = 259 (the size of ref_gp_cases' largest model)
  * sym_16384  a 128 x 128 grid, N = 4096 (the c4 training set)
  * sym_32768  a 256 x 128 grid, N = 4096
  * cross_c4   one c4 block row: the first 1024 points of the 1024 x 1024 grid against all 1,048,576, N = 4096
Per workload, each timed with CUDA events over `reps` launches after one warm-up launch of every call:
  * v_ms       forming V (posterior with the V cache: the separable mfgp_posterior_grid on these grids), A and B
  * kernel_ms  mfgp_posterior_cov alone on the resident V
  * prior_ms   mfgp_posterior_cov with N = 0: the epilogue alone (k** with one or two fp64 exp per element, the stores)
  * call_ms    the whole predict_cov_device call (V, the kernel, the allocations)
  * dgemm_ms   torch.mm(V_A^T, V_B), cuBLAS DGEMM on the same operands: the reference rate
Work is counted from shapes (`work` below): the symmetric form needs N Ga (Ga + 1) / 2 MAC (the lower triangle), the cross
form N Ga Gb; DGEMM does N Ga Gb either way.  rate_vs_dgemm = (kernel MAC / kernel time) / (DGEMM MAC / DGEMM time).
V of the large workloads (0.5 to 34 GB) exceeds the 126 MB L2, so neither side runs from cache.  The card's name and power
limit are read in the same run."""
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


def work(Ga, Gb, N, sym):
    """(MAC, bytes) the algorithm needs: the lower triangle when symmetric; V read once, C written once."""
    macs = N * Ga * (Ga + 1) // 2 if sym else N * Ga * Gb
    return macs, 8 * N * (Ga + (0 if sym else Gb)) + 8 * Ga * Gb


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


def tensor_grid(nx, ny):
    gx, gy = np.linspace(0, 1, nx), np.linspace(0, 1, ny)
    return np.stack(np.meshgrid(gx, gy, indexing="ij"), axis=-1).reshape(-1, 2)


def model(train_n, N):
    from mfgp_coverage_b200.gaussian_process import MFGP
    xy = synth.grid(train_n)
    X_L, y_L, X_H, y_H = synth.training_set(xy, synth.truth_function(xy), N)
    m = MFGP(X_L, y_L, X_H, y_H, 1, 1)
    m.hyp = synth.MF_HYP
    m.updt_info(X_L, y_L, X_H, y_H)
    m.engine.ensure_factor()
    m.engine.check_factor(force=True)
    return m


def run(name, m, xy_a, xy_b, reps):
    from mfgp_coverage_b200 import _native as nat
    from mfgp_coverage_b200._coverage import CoverageGrid
    eng = m.engine
    lib = nat.lib()
    sym = xy_b is None
    N = eng.N
    g_full = CoverageGrid(xy_a if sym else xy_b)
    if sym:
        ga = gb = g_full
    else:       # A: the first Ga points of the grid of B, a whole-column range of its tensor axes
        gb = g_full
        ga = CoverageGrid(xy_a, base_index=0, axes=g_full.axes)
    Ga, Gb = ga.G, gb.G
    lda, ldb = Ga + Ga % 2, Gb + Gb % 2
    f64 = dict(dtype=torch.float64, device=eng.device)
    Va = torch.empty((N, lda), **f64)
    Vb = Va if sym else torch.empty((N, ldb), **f64)
    C = torch.empty((Ga, ldb), **f64)

    def form_v():
        eng.posterior(ga.xy, vcache=Va, axes=ga.axes, g_lo=0)
        if not sym:
            eng.posterior(gb.xy, vcache=Vb, axes=gb.axes, g_lo=0)

    def kernel(n=N):
        nat.check(lib.mfgp_posterior_cov(nat.ptr(ga.xy), Ga, nat.ptr(Va), lda, None if sym else nat.ptr(gb.xy), Gb,
                                         None if sym else nat.ptr(Vb), ldb, n, ctypes.byref(eng.pstruct), nat.ptr(C), ldb,
                                         nat.stream_ptr()), "mfgp_posterior_cov")

    def dgemm():
        torch.mm(Va[:, :Ga].T, Vb[:, :Gb], out=D)

    v_ms = timed(form_v, reps)
    kernel_ms = timed(kernel, reps)
    prior_ms = timed(lambda: kernel(0), reps)
    D = torch.empty((Ga, Gb), **f64)
    dgemm_ms = timed(dgemm, reps)
    del D
    torch.cuda.empty_cache()
    out = C[:, :Gb]
    call_ms = timed(lambda: m.predict_cov_device(ga.xy, None if sym else gb.xy, grid=ga, grid2=None if sym else gb, out=out),
                    reps)
    macs, nbytes = work(Ga, Gb, N, sym)
    dmacs = N * Ga * Gb
    r = dict(name=name, form="symmetric" if sym else "cross", Ga=Ga, Gb=Gb, N=N, reps=reps, macs=macs, bytes=nbytes,
             v_ms=v_ms, kernel_ms=kernel_ms, prior_ms=prior_ms, call_ms=call_ms, dgemm_ms=dgemm_ms,
             kernel_tflops=2 * macs / kernel_ms / 1e9, dgemm_tflops=2 * dmacs / dgemm_ms / 1e9,
             kernel_gbs=nbytes / kernel_ms / 1e6)
    r["rate_vs_dgemm"] = r["kernel_tflops"] / r["dgemm_tflops"]
    r["time_vs_dgemm"] = kernel_ms / dgemm_ms
    print(json.dumps(r), flush=True)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--only", default=None, help="comma-separated workload names")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark measures the GPU"
    torch.cuda.set_device(0)
    info = card()
    print(json.dumps(info), flush=True)
    want = None if args.only is None else set(args.only.split(","))
    results = []
    if want is None or "sym_2601" in want:
        results.append(run("sym_2601", model(51, 259), synth.grid(51), None, 50))
    if want is None or want & {"sym_16384", "sym_32768", "cross_c4"}:
        m = model(1024, 4096)
        if want is None or "sym_16384" in want:
            results.append(run("sym_16384", m, synth.grid(128), None, 10))
        if want is None or "sym_32768" in want:
            results.append(run("sym_32768", m, tensor_grid(256, 128), None, 5))
        if want is None or "cross_c4" in want:
            full = synth.grid(1024)
            results.append(run("cross_c4", m, full[:1024], full, 3))
    doc = dict(card=info, tool="profiles/tools/bench_posterior_cov.py", results=results)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(doc, fh, indent=1)


if __name__ == "__main__":
    main()
