"""GPU: the tiled dataflow Cholesky (+ fused forward substitution) behind mfgp_cholesky / mfgp_cholesky_solve against
LAPACK on the same matrices -- np.linalg.cholesky is what the reference calls (gaussian_process.py:254, :529).  Called through
the C-ABI with raw device pointers."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.linalg as sl
import torch

from tests import synth

pytestmark = pytest.mark.gpu


def _lib():
    from mfgp_coverage_b200 import _native as nat
    return nat, nat.lib()


def _spd(n, seed, cond=1e6):
    """Random SPD matrix with a prescribed condition number (kernel matrices of close-by samples are this bad or worse)."""
    rng = np.random.default_rng(seed)
    q, _ = np.linalg.qr(rng.standard_normal((n, n)))
    ev = np.logspace(0, -np.log10(cond), n)
    return (q * ev) @ q.T


def _run(K_host, R, seed=0):
    nat, lib = _lib()
    n = K_host.shape[0]
    npad = int(lib.mfgp_npad(n))
    Kp = np.eye(npad)
    Kp[:n, :n] = K_host
    K = torch.from_numpy(Kp).cuda()
    W = torch.zeros((npad, npad), dtype=torch.float64, device="cuda")
    info = torch.zeros(1, dtype=torch.int32, device="cuda")
    work = torch.empty(int(lib.mfgp_workspace_bytes(npad)) // 8 + 8, dtype=torch.float64, device="cuda")
    st = nat.stream_ptr()
    B0 = None
    if R:
        B0 = np.random.default_rng(seed).standard_normal((npad, R))
        B = torch.from_numpy(B0).cuda()
        sw = torch.empty(int(lib.mfgp_cholesky_solve_workspace_bytes(npad, R)) // 8 + 8, dtype=torch.float64, device="cuda")
        nat.check(lib.mfgp_cholesky_solve(nat.ptr(K), npad, npad, nat.ptr(W), npad, nat.ptr(info), nat.ptr(B), R, R,
                                          nat.ptr(sw), sw.numel() * 8, st), "mfgp_cholesky_solve")
    else:
        B = None
        nat.check(lib.mfgp_cholesky(nat.ptr(K), npad, npad, nat.ptr(W), npad, nat.ptr(info), nat.ptr(work), st), "mfgp_cholesky")
    torch.cuda.synchronize()
    return Kp, np.tril(K.cpu().numpy()), W.cpu().numpy(), int(info.item()), B0, (B.cpu().numpy() if R else None)


@pytest.mark.parametrize("n,R", [(1, 0), (64, 64), (65, 0), (100, 64), (130, 128), (700, 320), (1500, 0), (1500, 192),
                                 (2200, 0), (2200, 192)])
def test_tiled_cholesky_and_solve_match_lapack(n, R):
    Kp, L, W, info, B0, Y = _run(_spd(n, n), R)
    assert info == 0
    Lref = np.linalg.cholesky(Kp)
    assert np.max(np.abs(L - Lref)) <= 1e-11 * np.max(np.abs(Lref))
    npad = Kp.shape[0]
    for j in range(0, npad, 64):            # the diagonal blocks of W hold the inverses of L's diagonal blocks
        blk = W[j:j + 64, j:j + 64]
        assert np.max(np.abs(np.triu(blk, 1))) == 0.0
        assert np.max(np.abs(blk @ Lref[j:j + 64, j:j + 64] - np.eye(64))) <= 1e-9
    if R:
        Yref = sl.solve_triangular(Lref, B0, lower=True)
        assert np.max(np.abs(Y - Yref)) <= 1e-9 * np.max(np.abs(Yref))


def test_kernel_matrix_of_the_workload():
    """The covariance the product builds (multi-fidelity block structure, jitter-limited conditioning), N = 1000."""
    from mfgp_coverage_b200 import simulator as sim
    nat, lib = _lib()
    base = synth.grid(64)
    X_L, y_L, X_H, y_H = synth.training_set(base, synth.truth_function(base), 1000)
    m = sim.init_MFGP(synth.MF_HYP, np.column_stack((X_L, y_L)))
    m.updt_info(X_L, y_L, X_H, y_H)
    e = m.engine
    npad, ld = e.npad, e.cap
    lib.mfgp_build_train_cov(nat.ptr(e.Xt), e.NL, e.NH, ctypes.byref(e.pstruct), nat.ptr(e.K), npad, ld, nat.ptr(e.Tt),
                             nat.stream_ptr())
    Kl = np.tril(e.K.view(ld, ld)[:npad, :npad].cpu().numpy())
    Kfull = Kl + np.tril(Kl, -1).T
    nat.check(lib.mfgp_cholesky(nat.ptr(e.K), npad, ld, nat.ptr(e.W), ld, nat.ptr(e.info), nat.ptr(e.work), nat.stream_ptr()),
              "mfgp_cholesky")
    L = np.tril(e.K.view(ld, ld)[:npad, :npad].cpu().numpy())
    Lref = np.linalg.cholesky(Kfull)
    assert int(e.info.item()) == 0
    assert np.max(np.abs(L - Lref)) <= 1e-10 * np.max(np.abs(Lref))
    assert np.max(np.abs(L @ L.T - Kfull)) <= 1e-13 * np.max(np.abs(Kfull))


@pytest.mark.parametrize("n,R", [(64, 64), (100, 128), (700, 320), (1500, 192), (2100, 448)])
def test_solve_with_fused_gram_product(n, R):
    """mfgp_cholesky_solve_gram: same factor and solution as mfgp_cholesky_solve, plus M = Y^T Y (tiles on and below the
    diagonal; the tiles above are not touched) accumulated by the Gram tasks of the same kernel -- against numpy, and bitwise
    the same on a second call (the groups of block rows are added in a fixed order whatever the scheduling)."""
    nat, lib = _lib()
    Kh = _spd(n, n + 1)
    npad = int(lib.mfgp_npad(n))
    Kp = np.eye(npad)
    Kp[:n, :n] = Kh
    B0 = np.random.default_rng(n).standard_normal((npad, R))
    st = nat.stream_ptr()
    sw = torch.empty(int(lib.mfgp_cholesky_solve_gram_workspace_bytes(npad, R)) // 8 + 8, dtype=torch.float64, device="cuda")
    out = []
    for rep in range(2):
        K = torch.from_numpy(Kp).cuda()
        B = torch.from_numpy(B0).cuda()
        W = torch.zeros((npad, npad), dtype=torch.float64, device="cuda")
        M = torch.full((R, R), np.nan, dtype=torch.float64, device="cuda")
        info = torch.zeros(1, dtype=torch.int32, device="cuda")
        nat.check(lib.mfgp_cholesky_solve_gram(nat.ptr(K), npad, npad, nat.ptr(W), npad, nat.ptr(info), nat.ptr(B), R, R,
                                               nat.ptr(M), R, nat.ptr(sw), sw.numel() * 8, st), "mfgp_cholesky_solve_gram")
        torch.cuda.synchronize()
        assert int(info.item()) == 0
        out.append((np.tril(K.cpu().numpy()), B.cpu().numpy(), M.cpu().numpy()))
    L, Y, M = out[0]
    Lref = np.linalg.cholesky(Kp)
    Yref = sl.solve_triangular(Lref, B0, lower=True)
    assert np.max(np.abs(L - Lref)) <= 1e-11 * np.max(np.abs(Lref))
    assert np.max(np.abs(Y - Yref)) <= 1e-9 * np.max(np.abs(Yref))
    blk = np.arange(R) // 64
    low = blk[:, None] >= blk[None, :]
    Mref = Y.T @ Y
    assert np.all(np.isnan(M[~low]))
    assert np.max(np.abs(M[low] - Mref[low])) <= 1e-12 * np.max(np.abs(Mref))
    assert np.array_equal(M[low], out[1][2][low]) and np.array_equal(Y, out[1][1])
    # and the plain entry point is what M == NULL means
    K = torch.from_numpy(Kp).cuda(); B = torch.from_numpy(B0).cuda()
    W = torch.zeros((npad, npad), dtype=torch.float64, device="cuda")
    info = torch.zeros(1, dtype=torch.int32, device="cuda")
    nat.check(lib.mfgp_cholesky_solve_gram(nat.ptr(K), npad, npad, nat.ptr(W), npad, nat.ptr(info), nat.ptr(B), R, R,
                                           None, 0, nat.ptr(sw), sw.numel() * 8, st), "mfgp_cholesky_solve_gram")
    torch.cuda.synchronize()
    assert np.array_equal(B.cpu().numpy(), Y)


@pytest.mark.parametrize("n,bad", [(64, 0), (64, 5), (64, 38), (200, 70), (200, 129), (500, 448), (500, 499), (2200, 2150)])
def test_first_non_positive_pivot_is_reported_like_lapack(n, bad):
    """np.linalg.cholesky raises on the first non-positive pivot; dpotrf's info names it (1-based) and so does `info` here."""
    K = _spd(n, 7, cond=1e3)
    Lr = np.linalg.cholesky(K)
    # lower the diagonal entry so that pivot `bad` turns negative: pivot = K[bad, bad] - sum_k<bad L[bad, k]^2
    K[bad, bad] = float(np.sum(Lr[bad, :bad] ** 2)) - 0.25
    _, info_ref = sl.lapack.dpotrf(K, lower=1)
    assert info_ref == bad + 1
    _, _, _, info, _, _ = _run(K, 0)
    assert info == info_ref


@pytest.mark.parametrize("mg,lead", [("8", "32"), ("2", "0")])
def test_random_sizes_terminate_and_agree(mg, lead):
    """Stress of the fused kernel (profiles/tools/stress_solve_gram.py): 40 random (block columns, right-hand-side tiles) pairs per
    queue setting -- every launch terminates (the subprocess has a time-out: a scheduling deadlock fails the test instead of
    hanging the suite), info = 0, L / Y / M against LAPACK, the Gram tasks leave L and Y bitwise untouched, and the canaries around
    every buffer the kernel writes (its workspace sized exactly as the library asks) stay intact."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, MFGP_DF_MG=mg, MFGP_DF_MLEAD=lead)
    out = subprocess.run([sys.executable, os.path.join(root, "profiles", "tools", "stress_solve_gram.py"), "40"], env=env,
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "40 cases ok" in out.stdout, (out.stdout[-500:], out.stderr[-2000:])
