"""GPU: the tiled dataflow Cholesky (+ fused forward substitution) behind mfgp_cholesky / mfgp_cholesky_solve against
LAPACK on the same matrices -- np.linalg.cholesky is what the reference calls (gaussian_process.py:254, :529).  Called through
the C-ABI with raw device pointers, on the buffer layouts the engine runs: leading dimensions above npad (DeviceGP grows its
buffers to 1.5x), uninitialised (here: NaN) W and upper tiles of K, every buffer inside a canary margin."""
import ctypes
import functools
import os
import subprocess
import sys
import threading

import numpy as np
import pytest
import scipy.linalg as sl
import torch

from tests import synth

pytestmark = pytest.mark.gpu
GUARD = 512                 # doubles of canary on either side of every buffer a call may write
CANARY = -7.25e300


def _lib():
    from mfgp_coverage_b200 import _native as nat
    return nat, nat.lib()


@functools.lru_cache(maxsize=4)
def _spd_cached(n, seed, cond):
    rng = np.random.default_rng(seed)
    q, _ = np.linalg.qr(rng.standard_normal((n, n)))
    ev = np.logspace(0, -np.log10(cond), n)
    return (q * ev) @ q.T


def _spd(n, seed, cond=1e6):
    """Random SPD matrix with a prescribed condition number (kernel matrices of close-by samples are this bad or worse)."""
    return _spd_cached(n, seed, cond).copy()


def _padded(K_host):
    """K in its npad x npad frame, the padding rows / columns holding the identity (as mfgp_build_train_cov writes it)."""
    n = K_host.shape[0]
    Kp = np.eye(int(_lib()[1].mfgp_npad(n)))
    Kp[:n, :n] = K_host
    return Kp


def _rows(npad, seed=0):
    """All rows up to 32 block columns, a seeded sample of 256 above (keeps the O(n^3) CPU references short)."""
    if npad <= 2048:
        return np.arange(npad)
    return np.sort(np.random.default_rng(seed).choice(npad, 256, replace=False))


def _layouts(npad, R):
    """(ld, ldw, ldb, ldm) per layout: `tight` is what a caller with exact-size buffers passes; `padded` has every stride
    different and above its minimum; `grown` is the engine's: K and W at the capacity DeviceGP._reserve grows to when the
    model outgrows npad - 64 rows (npad = 4160 inside 6144), right-hand sides and M at R."""
    from mfgp_coverage_b200 import _native as nat
    cap = max(npad, nat.npad(int(1.5 * (npad - 64))))
    out = {"tight": (npad, npad, R, R), "padded": (npad + 64, npad + 128, R + 2, R + 64)}
    if cap > npad:
        out["grown"] = (cap, cap, R, R)
    return out


def _guarded(shape, fill):
    """A buffer of `shape` doubles inside a larger allocation whose margins hold the canary; `fill`: array or scalar."""
    n = int(np.prod(shape))
    big = torch.full((n + 2 * GUARD,), CANARY, dtype=torch.float64, device="cuda")
    buf = big[GUARD:GUARD + n].view(*shape)
    if np.isscalar(fill):
        buf.fill_(fill)
    else:
        buf.copy_(torch.from_numpy(np.ascontiguousarray(fill)))
    return big, buf


def _intact(big):
    h = big.cpu().numpy()
    return bool(np.all(h[:GUARD] == CANARY) and np.all(h[-GUARD:] == CANARY))


def _same_bits(a, b):
    """Bitwise equality (NaN payloads and signed zeros count)."""
    return np.array_equal(np.ascontiguousarray(a).view(np.int64), np.ascontiguousarray(b).view(np.int64))


def _block_upper(rows, cols):
    """Mask of the 64x64 tiles strictly above the block diagonal of a rows x cols matrix."""
    return (np.arange(cols)[None, :] // 64) > (np.arange(rows)[:, None] // 64)


def _run(Kp, B0=None, layout="tight", gram=False):
    """One fused factorisation of Kp (npad x npad) through the C-ABI: mfgp_cholesky (B0 None), mfgp_cholesky_solve or, with
    `gram`, mfgp_cholesky_solve_gram, on the strides of `layout` (see _layouts).  Before the call every element the kernel
    must not read is NaN: the tiles of K above the block diagonal, the gap columns of K / W / B, all of W and all of M.
    Checks that the canaries around K, W, B, M and the workspace (sized exactly as the library asks) are intact and that
    every element the call must not write kept its bits.  Returns (info, L, W[:, :npad], Y, M[:, :R]) as host arrays."""
    nat, lib = _lib()
    npad = Kp.shape[0]
    R = 0 if B0 is None else B0.shape[1]
    ld, ldw, ldb, ldm = _layouts(npad, R)[layout]
    Kh = np.full((npad, ld), np.nan)
    Kh[:, :npad] = np.where(_block_upper(npad, npad), np.nan, Kp)
    gK, K = _guarded((npad, ld), Kh)
    gW, W = _guarded((npad, ldw), np.nan)
    info = torch.full((1,), 12345, dtype=torch.int32, device="cuda")
    st = nat.stream_ptr()
    guards = [gK, gW]
    if R:
        Bh = np.full((npad, ldb), np.nan)
        Bh[:, :R] = B0
        gB, B = _guarded((npad, ldb), Bh)
        gM, M = _guarded((R, ldm), np.nan)
        nwork = int((lib.mfgp_cholesky_solve_gram_workspace_bytes if gram else lib.mfgp_cholesky_solve_workspace_bytes)(npad, R))
        gS, work = _guarded((nwork // 8,), 0.0)
        guards += [gB, gM, gS]
        if gram:
            rc = lib.mfgp_cholesky_solve_gram(nat.ptr(K), npad, ld, nat.ptr(W), ldw, nat.ptr(info), nat.ptr(B), ldb, R,
                                              nat.ptr(M), ldm, nat.ptr(work), nwork, st)
        else:
            rc = lib.mfgp_cholesky_solve(nat.ptr(K), npad, ld, nat.ptr(W), ldw, nat.ptr(info), nat.ptr(B), ldb, R,
                                         nat.ptr(work), nwork, st)
    else:
        nwork = int(lib.mfgp_workspace_bytes(npad))
        gS, work = _guarded((nwork // 8,), 0.0)
        guards.append(gS)
        rc = lib.mfgp_cholesky(nat.ptr(K), npad, ld, nat.ptr(W), ldw, nat.ptr(info), nat.ptr(work), st)
    torch.cuda.synchronize()
    assert rc == 0, (rc, nat.last_error())
    assert all(_intact(g) for g in guards), "a write landed outside its buffer"
    Ko, Wo = K.cpu().numpy(), W.cpu().numpy()
    keepK = np.zeros((npad, ld), bool)
    keepK[:, :npad] = _block_upper(npad, npad)
    keepK[:, npad:] = True
    assert _same_bits(Ko[keepK], Kh[keepK]), "K changed above the block diagonal or in its gap columns"
    keepW = np.ones((npad, ldw), bool)
    keepW[:, :npad] = (np.arange(npad)[None, :] // 64) != (np.arange(npad)[:, None] // 64)
    assert _same_bits(Wo[keepW], np.full(int(keepW.sum()), np.nan)), "W changed outside its diagonal blocks"
    Y = Mo = None
    if R:
        Bo, Mo = B.cpu().numpy(), M.cpu().numpy()
        assert _same_bits(Bo[:, R:], Bh[:, R:]), "B changed in its gap columns"
        keepM = np.ones((R, ldm), bool)
        keepM[:, :R] = _block_upper(R, R) if gram else True
        assert _same_bits(Mo[keepM], np.full(int(keepM.sum()), np.nan)), "M changed outside its lower tiles"
        Y, Mo = Bo[:, :R], Mo[:, :R]
    return int(info.item()), np.tril(Ko[:, :npad]), Wo[:, :npad], Y, Mo


def _check_factor(Kp, L, W, cond):
    """L against LAPACK (forward error where it is defined, backward error always), the diagonal blocks of W against the
    inverses of L's diagonal blocks.  Returns the LAPACK factor."""
    npad = Kp.shape[0]
    Lref = np.linalg.cholesky(Kp)
    if cond <= 1e6:
        assert np.max(np.abs(L - Lref)) <= 1e-11 * np.max(np.abs(Lref))
    rows = _rows(npad)
    berr = lambda F: np.max(np.abs(F[rows] @ F.T - Kp[rows]))       # the same rows for both factors
    e_dev, e_ref = berr(L), berr(Lref)
    assert e_dev <= 10 * e_ref and e_dev <= 1e-13 * np.max(np.abs(Kp)), (e_dev, e_ref)
    for j in range(0, npad, 64):            # the diagonal blocks of W hold the inverses of L's diagonal blocks
        blk, Ljj = W[j:j + 64, j:j + 64], L[j:j + 64, j:j + 64]
        assert np.all(np.triu(blk, 1) == 0.0)
        tol = 1e-9 if cond <= 1e6 else 1e-9 * max(1.0, np.max(np.abs(blk) @ np.abs(Ljj)))
        assert np.max(np.abs(blk @ Ljj - np.eye(64))) <= tol
    return Lref


def _check_solve(Lref, L, B0, Y, cond):
    """Y = L^-1 B0 against scipy's triangular solve (with LAPACK's L where the forward error is defined, else with the
    device's own L)."""
    Yref = sl.solve_triangular(Lref if cond <= 1e6 else L, B0, lower=True)
    assert np.max(np.abs(Y - Yref)) <= 1e-9 * np.max(np.abs(Yref))


def _case_id(c):
    n, R, cond = c
    return f"{n}-{R}" if cond == 1e6 else f"{n}-{R}-cond{cond:g}"


# block columns 1, 2, 3, 11, 24, 32 (the last cp.async size), 33 (the first TMA size), 35 and 65 (a c4 model plus one block)
FACTOR_CASES = [(1, 0, 1e6), (64, 64, 1e6), (65, 0, 1e6), (100, 64, 1e6), (130, 128, 1e6), (700, 320, 1e6), (1500, 0, 1e6),
                (1500, 192, 1e6), (2048, 192, 1e6), (2049, 0, 1e6), (2049, 320, 1e6), (2200, 0, 1e6), (2200, 192, 1e6),
                (4100, 0, 1e6), (4100, 448, 1e6), (2049, 192, 1e10), (4100, 0, 1e10), (4100, 192, 1e10)]


@pytest.mark.parametrize("n,R,cond", FACTOR_CASES, ids=[_case_id(c) for c in FACTOR_CASES])
def test_tiled_cholesky_and_solve_match_lapack(n, R, cond):
    """Every layout gives the same bits as the tight one: the strides must not change the arithmetic."""
    Kp = _padded(_spd(n, n, cond))
    npad = Kp.shape[0]
    B0 = np.random.default_rng(0).standard_normal((npad, R)) if R else None
    ref = None
    for layout in _layouts(npad, R):
        info, L, W, Y, _ = _run(Kp, B0, layout)
        assert info == 0
        Wd = np.where((np.arange(npad)[None, :] // 64) == (np.arange(npad)[:, None] // 64), W, 0.0)
        if ref is None:
            ref = (L, Wd, Y)
            continue
        assert _same_bits(L, ref[0]) and _same_bits(Wd, ref[1]), layout
        assert R == 0 or _same_bits(Y, ref[2]), layout
    L, Wd, Y = ref
    Lref = _check_factor(Kp, L, Wd, cond)
    if R:
        _check_solve(Lref, L, B0, Y, cond)


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


@pytest.mark.parametrize("n,R", [(64, 64), (100, 128), (700, 320), (1500, 192), (2048, 320), (2100, 448), (4100, 192)])
def test_solve_with_fused_gram_product(n, R):
    """mfgp_cholesky_solve_gram: same factor and solution as mfgp_cholesky_solve, plus M = Y^T Y (tiles on and below the
    diagonal; the tiles above are not touched) accumulated by the Gram tasks of the same kernel -- against numpy, bitwise
    the same on a second call (the groups of block rows are added in a fixed order whatever the scheduling) and on every
    layout."""
    nat, lib = _lib()
    Kp = _padded(_spd(n, n + 1))
    npad = Kp.shape[0]
    B0 = np.random.default_rng(n).standard_normal((npad, R))
    layouts = ["tight"] + list(_layouts(npad, R))
    out = []
    for layout in layouts:
        info, L, W, Y, M = _run(Kp, B0, layout, gram=True)
        assert info == 0
        out.append((L, Y, M))
    L, Y, M = out[0]
    Lref = np.linalg.cholesky(Kp)
    Yref = sl.solve_triangular(Lref, B0, lower=True)
    assert np.max(np.abs(L - Lref)) <= 1e-11 * np.max(np.abs(Lref))
    assert np.max(np.abs(Y - Yref)) <= 1e-9 * np.max(np.abs(Yref))
    low = ~_block_upper(R, R)
    Mref = Y.T @ Y
    assert np.max(np.abs(M[low] - Mref[low])) <= 1e-12 * np.max(np.abs(Mref))
    for layout, (L2, Y2, M2) in zip(layouts[1:], out[1:]):
        assert _same_bits(L2, L) and _same_bits(Y2, Y) and _same_bits(M2[low], M[low]), layout
    # and the plain entry point is what M == NULL means
    K = torch.from_numpy(Kp).cuda(); B = torch.from_numpy(B0).cuda()
    W = torch.zeros((npad, npad), dtype=torch.float64, device="cuda")
    info = torch.zeros(1, dtype=torch.int32, device="cuda")
    sw = torch.empty(int(lib.mfgp_cholesky_solve_gram_workspace_bytes(npad, R)) // 8 + 8, dtype=torch.float64, device="cuda")
    nat.check(lib.mfgp_cholesky_solve_gram(nat.ptr(K), npad, npad, nat.ptr(W), npad, nat.ptr(info), nat.ptr(B), R, R,
                                           None, 0, nat.ptr(sw), sw.numel() * 8, nat.stream_ptr()), "mfgp_cholesky_solve_gram")
    torch.cuda.synchronize()
    assert _same_bits(B.cpu().numpy(), Y)


@pytest.mark.parametrize("n,bad", [(64, 0), (64, 5), (64, 38), (200, 70), (200, 129), (500, 448), (500, 499), (2200, 2150)])
def test_first_non_positive_pivot_is_reported_like_lapack(n, bad):
    """np.linalg.cholesky raises on the first non-positive pivot; dpotrf's info names it (1-based) and so does `info` here."""
    K = _spd(n, 7, cond=1e3)
    Lr = np.linalg.cholesky(K)
    # lower the diagonal entry so that pivot `bad` turns negative: pivot = K[bad, bad] - sum_k<bad L[bad, k]^2
    K[bad, bad] = float(np.sum(Lr[bad, :bad] ** 2)) - 0.25
    _, info_ref = sl.lapack.dpotrf(K, lower=1)
    assert info_ref == bad + 1
    info = _run(_padded(K))[0]
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


# ---- the rest of the fit: explicit inverse, whitening, the unfused factorisation ----------------------------------------------

def _factor(n, ld, ldw, seed=None):
    """mfgp_cholesky of an n x n SPD matrix on strides ld / ldw (W NaN beforehand, inside a canary margin); returns
    (Kp, K, W, W's allocation with the canaries, work), all but Kp on the device."""
    nat, lib = _lib()
    Kp = _padded(_spd(n, n if seed is None else seed))
    npad = Kp.shape[0]
    Kh = np.full((npad, ld), np.nan)
    Kh[:, :npad] = Kp
    K = torch.from_numpy(Kh).cuda()
    gW, W = _guarded((npad, ldw), np.nan)
    work = torch.empty(int(lib.mfgp_workspace_bytes(npad)) // 8, dtype=torch.float64, device="cuda")
    info = torch.zeros(1, dtype=torch.int32, device="cuda")
    nat.check(lib.mfgp_cholesky(nat.ptr(K), npad, ld, nat.ptr(W), ldw, nat.ptr(info), nat.ptr(work), nat.stream_ptr()),
              "mfgp_cholesky")
    torch.cuda.synchronize()
    assert int(info.item()) == 0
    return Kp, K, W, gW, work


@pytest.mark.parametrize("nb", [1, 2, 3, 5, 7, 33, 35, 65])
@pytest.mark.parametrize("pad", [(0, 0), (64, 192)])
def test_tri_inverse_after_cholesky(nb, pad):
    """mfgp_tri_inverse: W = L^-1 by block doubling.  nb = 1 runs no doubling level; 3, 5, 7 and 35 block columns leave a
    remainder pass at different levels.  W starts as NaN except for the diagonal blocks mfgp_cholesky wrote: every element of
    the strict upper triangle must come out exactly zero, the gap columns untouched, L (const) unchanged."""
    nat, lib = _lib()
    n = 64 * nb - 7
    npad = 64 * nb
    ld, ldw = npad + pad[0], npad + pad[1]
    Kp, K, W, gW, work = _factor(n, ld, ldw)
    K0 = K.cpu().numpy()
    nat.check(lib.mfgp_tri_inverse(nat.ptr(K), npad, ld, nat.ptr(W), ldw, nat.ptr(work), nat.stream_ptr()), "mfgp_tri_inverse")
    torch.cuda.synchronize()
    assert _intact(gW)
    assert _same_bits(K.cpu().numpy(), K0)
    Wo = W.cpu().numpy()
    assert np.all(np.isnan(Wo[:, npad:]))
    Wn = Wo[:, :npad]
    assert np.all(np.triu(Wn, 1) == 0.0)
    L = np.tril(K0[:, :npad])
    rows = _rows(npad, seed=nb)
    assert np.max(np.abs(Wn[rows] @ L - np.eye(npad)[rows])) <= 1e-9


@pytest.mark.parametrize("n,NL", [(130, 0), (700, 250), (2100, 700)])
def test_whiten_matches_triangular_solve(n, NL):
    """mfgp_whiten: z = W (y - mean) with the lofi mean on the first NL rows and the hifi mean on the rest (single fidelity:
    NL = 0, one mean), against solve_triangular(L, y - mean); the padding rows of z are exactly zero."""
    nat, lib = _lib()
    npad = int(lib.mfgp_npad(n))
    ld, ldw = npad + 64, npad + 128
    Kp, K, W, _, work = _factor(n, ld, ldw)
    nat.check(lib.mfgp_tri_inverse(nat.ptr(K), npad, ld, nat.ptr(W), ldw, nat.ptr(work), nat.stream_ptr()), "mfgp_tri_inverse")
    y = np.random.default_rng(n).standard_normal(n) + 0.5
    p = nat.MfgpParams(0.3, 0.5, 0.7, 0.2, 1.1, 0.01, 0.1, -0.4 if NL else 0.0, 0.35, 1e-8, 1 if NL else 0, 0)
    zd = torch.full((npad,), np.nan, dtype=torch.float64, device="cuda")
    nat.check(lib.mfgp_whiten(nat.ptr(W), npad, ldw, nat.ptr(torch.from_numpy(y).cuda()), NL, n - NL, ctypes.byref(p),
                              nat.ptr(zd), nat.stream_ptr()), "mfgp_whiten")
    z = zd.cpu().numpy()
    yc = y - np.where(np.arange(n) < NL, p.mean_L, p.mean_H)
    zref = sl.solve_triangular(np.linalg.cholesky(Kp)[:n, :n], yc, lower=True)
    assert np.max(np.abs(z[:n] - zref)) <= 1e-9 * np.max(np.abs(zref))
    assert np.all(z[n:] == 0.0)


@pytest.mark.parametrize("n,bad", [(60, None), (190, None), (2100, None), (200, 129)])
def test_cholesky_without_w(n, bad):
    """mfgp_cholesky(W = NULL): the per-block path (potrf_diag_kernel + panel GEMMs) on a padded ld, with NaN above the
    block diagonal and in the gap; L against LAPACK, a non-positive pivot reported as dpotrf's info."""
    nat, lib = _lib()
    K = _spd(n, 7 if bad else n, cond=1e3 if bad else 1e6)
    info_ref = 0
    if bad is not None:
        Lr = np.linalg.cholesky(K)
        K[bad, bad] = float(np.sum(Lr[bad, :bad] ** 2)) - 0.25
        info_ref = sl.lapack.dpotrf(K, lower=1)[1]
        assert info_ref == bad + 1
    Kp = _padded(K)
    npad = Kp.shape[0]
    ld = npad + 64
    Kh = np.full((npad, ld), np.nan)
    Kh[:, :npad] = np.where(_block_upper(npad, npad), np.nan, Kp)
    gK, Kd = _guarded((npad, ld), Kh)
    work = torch.empty(int(lib.mfgp_workspace_bytes(npad)) // 8, dtype=torch.float64, device="cuda")
    info = torch.full((1,), 12345, dtype=torch.int32, device="cuda")
    nat.check(lib.mfgp_cholesky(nat.ptr(Kd), npad, ld, None, 0, nat.ptr(info), nat.ptr(work), nat.stream_ptr()), "mfgp_cholesky")
    torch.cuda.synchronize()
    assert int(info.item()) == info_ref
    assert _intact(gK)
    Ko = Kd.cpu().numpy()
    keep = np.zeros((npad, ld), bool)
    keep[:, :npad] = _block_upper(npad, npad)
    keep[:, npad:] = True
    assert _same_bits(Ko[keep], Kh[keep])
    if bad is None:
        Lref = np.linalg.cholesky(Kp)
        assert np.max(np.abs(np.tril(Ko[:, :npad]) - Lref)) <= 1e-11 * np.max(np.abs(Lref))


# ---- argument checks ------------------------------------------------------------------------------------------------------

BAD_ARGS = ["odd_ld", "odd_ldw", "odd_ldb", "odd_ldm", "K_plus_1", "M_plus_1", "short_work", "short_work_gram", "R_not_64",
            "odd_ld_cholesky"]


@pytest.mark.parametrize("nb", [3, 35])          # cp.async and TMA form
@pytest.mark.parametrize("bad", BAD_ARGS)
def test_rejected_arguments_leave_buffers_alone(bad, nb):
    """A call the library rejects returns MFGP_ERR_INVALID and enqueues nothing: K, W, B, M and info keep their contents."""
    nat, lib = _lib()
    npad, R = 64 * nb, 128
    ld, ldw, ldb, ldm = npad + 64, npad + 64, R, R
    if bad == "odd_ld" or bad == "odd_ld_cholesky":
        ld += 1
    if bad == "odd_ldw":
        ldw += 1
    if bad == "odd_ldb":
        ldb += 1
    if bad == "odd_ldm":
        ldm += 1
    if bad == "R_not_64":
        R = ldb = ldm = 96
    Kp = _padded(_spd(npad, 5))
    Kh = np.full((npad + 1, ld), np.nan)
    Kh[:npad, :npad] = Kp
    K = torch.from_numpy(Kh).cuda()
    W = torch.full((npad, ldw), 3.0, dtype=torch.float64, device="cuda")
    B = torch.from_numpy(np.random.default_rng(1).standard_normal((npad, ldb))).cuda()
    M = torch.full((R + 1, ldm), 5.0, dtype=torch.float64, device="cuda")
    info = torch.full((1,), 12345, dtype=torch.int32, device="cuda")
    gram = bad in ("odd_ldm", "M_plus_1", "short_work_gram")
    nwork = int((lib.mfgp_cholesky_solve_gram_workspace_bytes if gram else lib.mfgp_cholesky_solve_workspace_bytes)(npad, R))
    if bad in ("short_work", "short_work_gram"):
        nwork -= 1
    work = torch.full((max(int(lib.mfgp_workspace_bytes(npad)), nwork) // 8 + 1,), 7.0, dtype=torch.float64, device="cuda")
    before = [t.cpu().numpy().copy() for t in (K, W, B, M, info, work)]
    Kptr = ctypes.c_void_p(K.data_ptr() + 8) if bad == "K_plus_1" else nat.ptr(K)
    Mptr = ctypes.c_void_p(M.data_ptr() + 8) if bad == "M_plus_1" else nat.ptr(M)
    st = nat.stream_ptr()
    if bad == "odd_ld_cholesky":
        rc = lib.mfgp_cholesky(Kptr, npad, ld, nat.ptr(W), ldw, nat.ptr(info), nat.ptr(work), st)
    elif gram:
        rc = lib.mfgp_cholesky_solve_gram(Kptr, npad, ld, nat.ptr(W), ldw, nat.ptr(info), nat.ptr(B), ldb, R, Mptr, ldm,
                                          nat.ptr(work), nwork, st)
    else:
        rc = lib.mfgp_cholesky_solve(Kptr, npad, ld, nat.ptr(W), ldw, nat.ptr(info), nat.ptr(B), ldb, R, nat.ptr(work),
                                     nwork, st)
    torch.cuda.synchronize()
    assert rc == nat.MFGP_ERR_INVALID
    for name, t, h in zip("K W B M info work".split(), (K, W, B, M, info, work), before):
        assert _same_bits(t.cpu().numpy(), h) if t.dtype == torch.float64 else np.array_equal(t.cpu().numpy(), h), name


# ---- concurrency ----------------------------------------------------------------------------------------------------------

def test_concurrent_factorisations_on_two_host_threads():
    """Calls with different work buffers may overlap (include/mfgp_b200.h).  The TMA form caches its tensor maps per device;
    two host threads, each with its own stream, buffers and matrix (35 block columns), alternate their calls so that the
    cache changes hands on every call: every result must equal that matrix's serial result bit for bit."""
    nat, lib = _lib()
    n, R, calls = 2200, 192, 10
    npad = int(lib.mfgp_npad(n))
    nwork = int(lib.mfgp_cholesky_solve_workspace_bytes(npad, R))

    def state(seed):
        K0 = torch.from_numpy(_padded(_spd(n, seed))).cuda()
        B0 = torch.from_numpy(np.random.default_rng(seed).standard_normal((npad, R))).cuda()
        return dict(K0=K0, B0=B0, K=torch.empty_like(K0), B=torch.empty_like(B0), W=torch.zeros_like(K0),
                    info=torch.zeros(1, dtype=torch.int32, device="cuda"),
                    work=torch.empty(nwork // 8, dtype=torch.float64, device="cuda"), stream=torch.cuda.Stream())

    def call(s):
        with torch.cuda.stream(s["stream"]):
            s["K"].copy_(s["K0"]); s["B"].copy_(s["B0"])
            rc = lib.mfgp_cholesky_solve(nat.ptr(s["K"]), npad, npad, nat.ptr(s["W"]), npad, nat.ptr(s["info"]), nat.ptr(s["B"]),
                                         R, R, nat.ptr(s["work"]), nwork, nat.stream_ptr(s["stream"]))
            out = (rc, s["info"].clone(), torch.tril(s["K"]), s["B"].clone())
        s["stream"].synchronize()
        return out[0], int(out[1].item()), out[2], out[3]

    states = [state(11), state(12)]
    serial = [call(s) for s in states]
    assert all(r[0] == 0 and r[1] == 0 for r in serial)
    bad = []
    start = threading.Barrier(2)

    def worker(k):
        start.wait()
        for i in range(calls):
            rc, info, L, Y = call(states[k])
            if rc != 0 or info != 0 or not torch.equal(L, serial[k][2]) or not torch.equal(Y, serial[k][3]):
                bad.append((k, i, rc, info))

    threads = [threading.Thread(target=worker, args=(k,)) for k in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not bad, bad
