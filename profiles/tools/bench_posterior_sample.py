"""Joint posterior draws (DeviceGP.posterior_sample: mfgp_posterior_cov, mfgp_posterior_cov_factor, mfgp_posterior_sample)
against cuBLAS / cuSOLVER in the same run.

    python profiles/tools/bench_posterior_sample.py --out profiles/r09_posterior_sample.json

Workloads (MF model, tests/synth.py hyper-parameters; training sets as bench_posterior_cov.py builds them):
  * ref_2601    the reference's scale: the 51 x 51 grid, N = 259; S = 1, 64
  * c4_16384    a 128 x 128 grid, N = 4096 (the c4 training set); S = 1, 64, 1024
  * max_32768   a 256 x 128 grid, N = 4096 (npad = 32768, the largest factor accepted); S = 64
Per workload and S, each timed with CUDA events after a warm-up call of every shape:
  * cov_ms       the joint covariance C (posterior_cov into the factor's buffer: V and mfgp_posterior_cov)
  * factor_ms    mfgp_posterior_cov_factor (jitter, identity padding, the fused tiled Cholesky); flop = G^3 / 3, set
                 against dgemm_tflops, a square 8192 DGEMM timed in the same run
  * cusolver_ms  torch.linalg.cholesky on the same matrix (cuSOLVER): a reference point only
  * sample_ms    mfgp_posterior_sample on the factor: MAC = S G (G + 1) / 2
  * dgemm_ref_ms torch.mm(tril(L), E): the same product as a dense DGEMM (twice the MACs)
  * call_ms      the whole sample_posterior_device call (allocations included)
L is 54 MB at G = 2601 (within the 126 MB L2 after the first pass) and 2.1 / 8.6 GB at G = 16384 / 32768 (far past it).
The card's name and power limit are read in the same run."""
import argparse
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


def timed(fn, reps, setup=None):
    """Mean device time of fn() over reps calls (after one warm-up call); setup() runs before each call, outside the timing."""
    if setup:
        setup()
    fn()
    torch.cuda.synchronize()
    total = 0.0
    for _ in range(reps):
        if setup:
            setup()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        total += e0.elapsed_time(e1)
    return total / reps


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


def dgemm_tflops():
    a = torch.randn((8192, 8192), dtype=torch.float64, device="cuda")
    c = torch.empty_like(a)
    ms = timed(lambda: torch.mm(a, a, out=c), 10)
    return 2 * 8192 ** 3 / ms / 1e9


def run(name, m, xy, s_values, reps, dgemm_rate):
    from mfgp_coverage_b200 import _native as nat
    from mfgp_coverage_b200._coverage import CoverageGrid
    eng = m.engine
    lib = nat.lib()
    g = CoverageGrid(xy)
    G, N = g.G, eng.N
    npad = nat.npad(G)
    p = eng.params
    tau = 1e-8 * ((p["rho"] ** 2 * p["s_L"] + p["s_H"]) if p["multi"] else p["s_H"])
    f64 = dict(dtype=torch.float64, device=eng.device)
    C0 = torch.empty((npad, npad), **f64)
    cov_ms = timed(lambda: eng.posterior_cov(g.xy, axes_a=g.axes, g_lo_a=g.base_index, out=C0[:G, :G]), reps)
    mu = eng.posterior_cov(g.xy, axes_a=g.axes, g_lo_a=g.base_index, out=C0[:G, :G])[0]
    C = torch.empty_like(C0)
    W = torch.empty_like(C0)
    work = torch.empty(int(lib.mfgp_workspace_bytes(npad)) // 8 + 1, **f64)
    info = torch.zeros(1, dtype=torch.int32, device=eng.device)

    def factor():
        nat.check(lib.mfgp_posterior_cov_factor(nat.ptr(C), G, npad, npad, tau, nat.ptr(W), npad, nat.ptr(info),
                                                nat.ptr(work), nat.stream_ptr()), "mfgp_posterior_cov_factor")

    factor_ms = timed(factor, reps, setup=lambda: C.copy_(C0))
    assert int(info.item()) == 0, int(info.item())
    del W, work
    A = C0[:G, :G] + tau * torch.eye(G, **f64)
    cusolver_ms = timed(lambda: torch.linalg.cholesky(A), reps)
    del A
    torch.cuda.empty_cache()
    Lt = torch.tril(C[:G, :G])
    out = []
    for S in s_values:
        E = torch.randn((G, S + S % 2), **f64)[:, :S]
        F = torch.empty((G, S + S % 2), **f64)[:, :S]

        def sample():
            nat.check(lib.mfgp_posterior_sample(nat.ptr(C), G, npad, nat.ptr(mu), nat.ptr(E), int(E.stride(0)), S, nat.ptr(F),
                                                int(F.stride(0)), nat.stream_ptr()), "mfgp_posterior_sample")

        sample_ms = timed(sample, reps)
        D = torch.empty((G, S), **f64)
        dgemm_ref_ms = timed(lambda: torch.mm(Lt, E, out=D), reps)
        err = float((D + mu[:, None] - F).abs().max())
        del D
        call_ms = timed(lambda: m.sample_posterior_device(g.xy, E, grid=g), reps)
        macs = S * G * (G + 1) // 2
        r = dict(name=name, G=G, N=N, S=S, npad=npad, reps=reps, jitter=tau,
                 cov_ms=cov_ms, factor_ms=factor_ms, cusolver_ms=cusolver_ms, sample_ms=sample_ms, dgemm_ref_ms=dgemm_ref_ms,
                 call_ms=call_ms, factor_tflops=G ** 3 / 3 / factor_ms / 1e9, dgemm_tflops=dgemm_rate,
                 sample_macs=macs, sample_tflops=2 * macs / sample_ms / 1e9,
                 sample_gbs=8 * (G * (G + 1) / 2 + 2 * G * S) / sample_ms / 1e6,
                 sample_vs_dgemm_ref_time=sample_ms / dgemm_ref_ms, max_abs_diff_vs_dgemm_ref=err)
        r["factor_rate_vs_dgemm"] = r["factor_tflops"] / dgemm_rate
        print(json.dumps(r), flush=True)
        out.append(r)
        del E, F
    return out


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
    rate = dgemm_tflops()
    results = []
    if want is None or "ref_2601" in want:
        results += run("ref_2601", model(51, 259), synth.grid(51), (1, 64), 20, rate)
    if want is None or want & {"c4_16384", "max_32768"}:
        m = model(1024, 4096)
        if want is None or "c4_16384" in want:
            results += run("c4_16384", m, synth.grid(128), (1, 64, 1024), 5, rate)
        if want is None or "max_32768" in want:
            results += run("max_32768", m, tensor_grid(256, 128), (64,), 3, rate)
    doc = dict(card=info, tool="profiles/tools/bench_posterior_sample.py", dgemm_8192_tflops=rate, results=results)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(doc, fh, indent=1)


if __name__ == "__main__":
    main()
