"""Correctness + device time of the tiled dataflow Cholesky (+ fused forward substitution) against numpy.
usage: diag_dataflow_chol.py [N=4096] [R list, default 0,64,1792]"""
import sys, os, ctypes
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import numpy as np, torch
from tests import synth
from mfgp_coverage_b200 import simulator as sim, _native as nat
N = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
base = synth.grid(256)
X_L, y_L, X_H, y_H = synth.training_set(base, synth.truth_function(base), N)
m = sim.init_MFGP(synth.MF_HYP, np.column_stack((X_L, y_L)))
m.updt_info(X_L, y_L, X_H, y_H)
e = m.engine
lib = nat.lib(); st = nat.stream_ptr(); pp = ctypes.byref(e.pstruct); npad, ld = e.npad, e.cap
def ev(): return torch.cuda.Event(enable_timing=True)
def build():
    lib.mfgp_build_train_cov(nat.ptr(e.Xt), e.NL, e.NH, pp, nat.ptr(e.K), npad, ld, nat.ptr(e.Tt), st)
build(); torch.cuda.synchronize()
Kh = e.K.view(ld, ld)[:npad, :npad].cpu().numpy().copy()
Lref = np.linalg.cholesky(Kh)
RS = tuple(int(x) for x in sys.argv[2].split(",")) if len(sys.argv) > 2 else (0, 64, 1792)
for R in RS:
    B0 = torch.randn(npad, max(R, 64), dtype=torch.float64, device="cuda")
    sw = torch.empty(int(lib.mfgp_cholesky_solve_workspace_bytes(npad, max(R, 64))) // 8 + 8, dtype=torch.float64, device="cuda")
    ts = []
    for rep in range(4):
        build(); B = B0.clone(); torch.cuda.synchronize()
        a, b = ev(), ev(); a.record()
        if R == 0:
            rc = lib.mfgp_cholesky(nat.ptr(e.K), npad, ld, nat.ptr(e.W), ld, nat.ptr(e.info), nat.ptr(e.work), st)
        else:
            rc = lib.mfgp_cholesky_solve(nat.ptr(e.K), npad, ld, nat.ptr(e.W), ld, nat.ptr(e.info), nat.ptr(B), R, R, nat.ptr(sw), sw.numel() * 8, st)
        b.record(); torch.cuda.synchronize(); ts.append(a.elapsed_time(b))
    L = np.tril(e.K.view(ld, ld)[:npad, :npad].cpu().numpy())
    errL = np.max(np.abs(L - Lref)) / np.max(np.abs(Lref))
    msg = f"N={N} npad={npad} R={R}: rc={rc} info={int(e.info.item())} device {min(ts):.3f} ms (runs {['%.2f' % t for t in ts]}) errL={errL:.2e}"
    if R:
        import scipy.linalg as sl
        Y = sl.solve_triangular(Lref, B0.cpu().numpy(), lower=True)
        msg += f" errY={np.max(np.abs(B.cpu().numpy() - Y)) / np.max(np.abs(Y)):.2e}"
    W = e.W.view(ld, ld)[:npad, :npad].cpu().numpy()
    d = max(np.max(np.abs(W[j:j+64, j:j+64] @ Lref[j:j+64, j:j+64] - np.eye(64))) for j in range(0, npad, 64))
    print(msg + f" errWdiag={d:.2e}", flush=True)
if os.environ.get("MFGP_DF_TRACE"):
    nbk = npad // 64
    buf = np.zeros((nbk, 16), dtype=np.int64)
    n = lib.mfgp_debug_chol_trace(buf.ctypes.data_as(ctypes.c_void_p), nbk)
    gt, ck = buf[:n, :7].astype(float), buf[:n, 8:15].astype(float)
    names = ["k-loop end -> diag flag seen", "flag -> W loaded", "panel solve (X W^T) + stores", "diag update (L L^T) + S + publish",
             "potrf_diag_body", "fence + flag"]
    sel = slice(2, n)
    print("chain-task phases, median over tasks 2.. (SM clocks | globaltimer ns):")
    for k, nm in enumerate(names):
        print(f"  {nm:38s} {np.median(ck[sel, k + 1] - ck[sel, k]):9.0f} clk | {np.median(gt[sel, k + 1] - gt[sel, k]):8.0f} ns")
    print(f"  flag(d) set -> task d+1 sees it        {np.median(gt[3:n, 1] - gt[2:n - 1, 6]):8.0f} ns   (hop)")
    print(f"  per block column (flag seen -> next flag seen) {np.median(gt[3:n, 1] - gt[2:n - 1, 1]):8.0f} ns")
