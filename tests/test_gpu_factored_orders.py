"""GPU: the kernels of the Chebyshev-factored posterior (csrc/gp_factored.cu) at chosen orders, layouts and geometries,
called through the C-ABI with raw device pointers and compared with the term-by-term restatement of oracle/factored.py.

The engine's planner only ever asks for the orders that the synthetic length scales give (~24-36 terms), so the engine-level
tests (test_gpu_factored.py) reach one instantiation of each kernel.  Here the orders are explicit: every qform_kernel<NT>,
gram_eval_kernel<WM> with both shared-memory pitches and its store / update forms, geval_mma_kernel<WM>, one and several
column chunks, truncated layouts, ix0 > 0, ny from 1 to 200.  The length scales are short, so every kept term is
significant and the comparison is against the expansion itself, not against the exact GP; each case asserts that dropping
its highest kept term moves the restatement by more than 100x the tolerance.  Every output and workspace is NaN before the
call and sits inside a canary margin sized exactly as the library asks.  The direct-route cases run with
MFGP_DEBUG_POISON_SMEM=1: gram_eval_kernel then NaN-fills its dynamic shared memory, so a read of a word it did not
initialise shows up as NaN in the output.  Not covered here: the FMA form of the evaluation (MFGP_GEVAL=fma, chosen once per
process)."""
import ctypes
import functools
import math

import numpy as np
import pytest
import torch

from oracle import factored as ofac
from oracle import gp as ogp
from tests import synth

GUARD = 512                 # doubles of canary on either side of every buffer a call may write
CANARY = -7.25e300
TOL = 1e-11
SHORT = (0.03, 0.02)         # (l_L, l_H): at these every term up to order 64 is significant on the unit square

# ---- the cases ------------------------------------------------------------------------------------------------------------
# route: direct  -- standing factor, mfgp_posterior_grid_factored, MFGP_GRAM=direct (Y' per column, gram_eval_kernel)
#        gram    -- standing factor, mfgp_posterior_grid_factored_trunc, MFGP_GRAM=m (M = Y^T Y, qform_kernel, geval_mma_kernel)
#        fdirect -- mfgp_factored_prepare -> mfgp_cholesky_solve -> mfgp_posterior_grid_factored_solved (direct route)
#        fgram   -- mfgp_factored_prepare_trunc -> mfgp_cholesky_solve_gram at mfgp_factored_gram_target -> _solved_gram
#        incr    -- standing full form with Gstore / Hz_store, mfgp_cholesky_append, mfgp_posterior_grid_factored_update
#        fincr   -- fgram with Gstore / Hz_store, mfgp_cholesky_append, mfgp_posterior_grid_factored_update
# layout (Gram routes): None (uniform), "kpad" (kx = kpad everywhere), "four" (all 4s), "zigzag" (non-monotone), "planner"
# (the engine's own orders and kx for the synthetic length scales, run at the short ones)
# N: training rows (incremental: rows before the append, then `add` more)


class Case:
    def __init__(self, cid, multi, orders, route, N, nx, ix0, ncols, ny, chunk=256, layout=None, add=0):
        self.cid, self.multi, self.orders, self.route, self.N = cid, multi, orders, route, N
        self.nx, self.ix0, self.ncols, self.ny, self.chunk, self.layout, self.add = nx, ix0, ncols, ny, chunk, layout, add

    def __repr__(self):
        return self.cid


CASES = [
    Case("d_ry4", False, (0, 0, 6, 4), "direct", 500, 40, 3, 1, 7, chunk=64),
    Case("d_ry8", False, (0, 0, 9, 8), "direct", 70, 63, 0, 63, 33),
    Case("d_ry12", True, (5, 12, 10, 8), "direct", 500, 70, 5, 65, 7, chunk=64),
    Case("d_ry28", True, (13, 28, 7, 20), "direct", 500, 130, 0, 130, 200, chunk=64),
    Case("d_ry32", False, (0, 0, 16, 32), "direct", 70, 64, 0, 64, 33),
    Case("d_ry36", True, (24, 36, 20, 36), "direct", 70, 80, 16, 64, 1),
    Case("d_ry40", True, (30, 40, 31, 24), "direct", 500, 63, 0, 63, 33),
    Case("d_ry44", True, (17, 44, 33, 44), "direct", 500, 70, 6, 64, 7),
    Case("d_ry48", False, (0, 0, 40, 48), "direct", 500, 65, 0, 65, 33, chunk=64),
    Case("d_ry52", True, (45, 28, 50, 52), "direct", 500, 63, 0, 63, 7),
    Case("d_ry60", True, (60, 60, 58, 60), "direct", 70, 64, 0, 64, 33),
    Case("d_ry64", True, (64, 64, 61, 64), "direct", 500, 64, 0, 64, 33),
    Case("fd_ry20", True, (11, 16, 9, 20), "fdirect", 500, 140, 10, 130, 33, chunk=64),
    Case("fd_ry24", False, (0, 0, 22, 24), "fdirect", 70, 64, 0, 64, 7),
    Case("fd_ry56", True, (50, 56, 55, 40), "fdirect", 500, 63, 0, 63, 33),
    Case("g_nt1", False, (0, 0, 3, 4), "gram", 70, 64, 0, 64, 33),
    Case("g_nt2_four", True, (10, 8, 14, 12), "gram", 500, 65, 0, 65, 7, layout="four"),
    Case("g_nt3_kpad", True, (22, 16, 19, 8), "gram", 70, 140, 9, 130, 1, layout="kpad"),
    Case("g_nt4_zigzag", False, (0, 0, 29, 20), "gram", 500, 63, 0, 63, 33, layout="zigzag"),
    Case("g_planner", True, None, "gram", 500, 70, 6, 64, 33, layout="planner"),
    Case("g_nt6", True, (46, 44, 41, 32), "gram", 70, 64, 0, 64, 200),
    Case("g_nt7_zigzag", False, (0, 0, 53, 56), "gram", 500, 30, 17, 1, 33, layout="zigzag"),
    Case("g_nt8", True, (64, 64, 64, 64), "gram", 500, 64, 0, 64, 7),
    Case("fg_nt1_four", False, (0, 0, 7, 64), "fgram", 500, 64, 0, 64, 33, layout="four"),
    Case("fg_nt5", False, (0, 0, 38, 12), "fgram", 500, 63, 0, 63, 200),
    Case("fg_planner", True, None, "fgram", 500, 130, 0, 130, 33, layout="planner"),
    Case("fg_nt8_zigzag", True, (62, 60, 57, 52), "fgram", 70, 65, 0, 65, 7, layout="zigzag"),
    Case("i_ry20", True, (18, 20, 21, 16), "incr", 450, 64, 0, 64, 33, add=64),
    Case("i_ry24", False, (0, 0, 15, 24), "incr", 130, 70, 2, 65, 7, chunk=64, add=70),
    Case("i_ry48", True, (35, 48, 42, 40), "incr", 130, 63, 0, 63, 33, add=70),
    Case("i_ry60", False, (0, 0, 47, 60), "incr", 450, 64, 0, 64, 7, add=64),
    Case("fi_ry32", True, (26, 32, 30, 28), "fincr", 130, 64, 0, 64, 33, add=70),
    Case("fi_ry64", False, (0, 0, 44, 64), "fincr", 450, 64, 0, 64, 7, add=64),
]
DIRECT_ROUTES = ("direct", "fdirect", "incr")


def host_shape(orders):
    """The host formulas of gp_factored.cu that pick the instantiations: kpad, nt8 (f_tail_gram), wm and pitch (f_tail)."""
    rxL, ryL, rxH, ryH = orders
    ry, kpad = max(ryL, ryH), ofac.round_up(max(rxL, rxH), 4)
    pitch = ry if ry % 8 == 4 else ry + 4
    nstage = min(6, max(2, 73728 // (64 * pitch * 8)))
    return dict(ry=ry, kpad=kpad, nt8=(kpad + 7) // 8, wm=40 if ry <= 40 else 64, pitch=pitch, nstage=nstage)


def instantiations(case, orders):
    """Kernel instantiations (and forms) the case reaches, from the same host formulas."""
    h = host_shape(orders)
    ge = f"gram_eval_kernel<{h['wm']}> P={'ry' if h['pitch'] == h['ry'] else 'ry+4'}"
    qf = f"qform_kernel<{h['nt8']}, {'true' if h['nt8'] <= 6 else 'false'}>"
    gm = f"geval_mma_kernel<{h['wm']}>"
    chunks = "chunks>1" if case.route in DIRECT_ROUTES and case.ncols > ofac.round_up(case.chunk, 64) else "chunks=1"
    return {"direct": {ge + " eval", chunks}, "fdirect": {ge + " eval", chunks},
            "gram": {qf, gm}, "fgram": {qf, gm},
            "incr": {ge + " store", ge + " accumulate", gm, chunks},
            "fincr": {qf, gm, ge + " accumulate"}}[case.route]


def poison_reads_past_ring(case, orders, npad):
    """Whether gram_eval_kernel's fragment loads reach past the zero-filled ring when its slack is only 8 doubles: the last
    ring slot is used (npad / 64 chunks >= nstage) and the last row's column WM - 1 lies beyond it (P <= WM - 9)."""
    h = host_shape(orders)
    return case.route in ("direct", "fdirect") and npad // 64 >= h["nstage"] and h["pitch"] <= h["wm"] - 9


def test_cases_reach_every_instantiation():
    """The case table reaches every instantiation of the kernels it tests (planner cases: their orders are at most 40)."""
    seen = set()
    for c in CASES:
        if c.orders is not None:
            seen |= instantiations(c, c.orders)
    need = {f"qform_kernel<{nt}, {'true' if nt <= 6 else 'false'}>" for nt in range(1, 9)}
    need |= {f"geval_mma_kernel<{wm}>" for wm in (40, 64)} | {"chunks=1", "chunks>1"}
    need |= {f"gram_eval_kernel<{wm}> P={p} {form}" for wm in (40, 64) for p in ("ry", "ry+4")
             for form in ("eval", "store", "accumulate")}
    assert need <= seen, sorted(need - seen)
    rys = {host_shape(c.orders)["ry"] for c in CASES if c.orders is not None}
    assert {4, 8, 12, 28, 32, 36, 40, 44, 48, 52, 60, 64} <= rys
    assert {c.ncols for c in CASES} >= {1, 63, 64, 65, 130} and {c.ny for c in CASES} >= {1, 7, 33, 200}
    assert any(c.orders and c.multi and c.orders[0] < c.orders[2] and c.orders[1] > c.orders[3] for c in CASES)
    assert any(c.orders and c.multi and c.orders[0] > c.orders[2] and c.orders[1] < c.orders[3] for c in CASES)
    assert any(c.orders and c.multi and c.orders[1] == c.orders[3] == 64 for c in CASES)
    npads = {ofac.round_up(c.N, 64) // 64 - host_shape(c.orders)["nstage"] for c in CASES if c.route == "direct" and c.orders}
    assert min(npads) < 0 < max(npads)                      # ring slots left unused, and the ring wrapped
    past = {host_shape(c.orders)["ry"] for c in CASES if c.orders and poison_reads_past_ring(c, c.orders, ofac.round_up(c.N, 64))}
    assert {44, 48, 52} <= past and min(past) <= 28         # the poisoned cases include every kind whose loads left the ring


# ---- device plumbing --------------------------------------------------------------------------------------------------------
def _lib():
    from mfgp_coverage_b200 import _native as nat
    return nat, nat.lib()


def _guarded(n, fill):
    big = torch.full((int(n) + 2 * GUARD,), CANARY, dtype=torch.float64, device="cuda")
    buf = big[GUARD:GUARD + int(n)]
    buf.fill_(fill)
    return big, buf


def _intact(big):
    h = big.cpu().numpy()
    return bool(np.all(h[:GUARD] == CANARY) and np.all(h[-GUARD:] == CANARY))


def _bits(t):
    return t.cpu().numpy().view(np.int64).copy()


def _hyp(multi, lens):
    h = (synth.MF_HYP if multi else synth.SF_HYP).copy()
    if multi:
        h[2], h[5] = math.log(lens[0]), math.log(lens[1])
    else:
        h[2] = math.log(lens[1])
    return h


@functools.lru_cache(maxsize=None)
def _data(multi, N, seed=11):
    """Training points uniform on the unit square (a quarter lofi for MF), observations of the synthetic truth plus noise."""
    rng = np.random.default_rng(seed + N + (1000 if multi else 0))
    NL = N // 4 if multi else 0
    X = rng.random((N, 2))
    y = synth.truth_function(X) + rng.normal(0, 0.05, N)
    y[:NL] = 0.8 * y[:NL] + 0.05
    return X[:NL], y[:NL].reshape(-1, 1), X[NL:], y[NL:].reshape(-1, 1)


def _device_model(multi, X_L, y_L, X_H, y_H, lens, incremental=False):
    """A DeviceGP with the factor standing (eager refit): K -> L -> W = L^-1 -> z."""
    from mfgp_coverage_b200._engine import DeviceGP
    from mfgp_coverage_b200.gaussian_process import evaluate_hyp
    e = DeviceGP()
    e.incremental = incremental
    e.fit(np.vstack((X_L, X_H)), np.vstack((y_L, y_H)), X_L.shape[0], X_H.shape[0], evaluate_hyp(_hyp(multi, lens)))
    return e


@functools.lru_cache(maxsize=None)
def _standing(multi, N):
    X_L, y_L, X_H, y_H = _data(multi, N)
    return _device_model(multi, X_L, y_L, X_H, y_H, SHORT)


@functools.lru_cache(maxsize=None)
def _reference_factor(multi, N, n_use=None):
    X_L, y_L, X_H, y_H = _data(multi, N)
    n = X_H.shape[0] if n_use is None else n_use
    p = ogp.GPParams.from_hyp(_hyp(multi, SHORT))
    return p, ofac.factor(p, X_L, X_H[:n], y_L, y_H[:n])


def _grid(case):
    ux = np.linspace(0.0, 1.0, case.nx)
    uy = np.linspace(0.0, 1.0, case.ny) if case.ny > 1 else np.array([0.37])
    xs = ux[case.ix0:case.ix0 + case.ncols]
    box = (float(xs.min()), float(xs.max())) if case.ncols > 1 else (0.0, 1.0)
    return ux, uy, box + (0.0, 1.0)


def _planner_layout(case, ux, uy, box):
    """The orders and kx the engine's planner picks on this grid for the same training points at the synthetic scales."""
    from mfgp_coverage_b200._engine import DeviceGP, TensorAxes
    from mfgp_coverage_b200.gaussian_process import evaluate_hyp
    X_L, y_L, X_H, y_H = _data(case.multi, case.N)
    e = DeviceGP()
    e.fit(np.vstack((X_L, X_H)), np.vstack((y_L, y_H)), X_L.shape[0], X_H.shape[0],
          evaluate_hyp(synth.MF_HYP if case.multi else synth.SF_HYP))
    axes = TensorAxes(ux, uy, torch.device("cuda", torch.cuda.current_device()))
    orders = e._cheb_orders(axes, e.params, box[0], box[1])
    assert orders is not None and e._ftrunc is not None
    return tuple(int(o) for o in orders), np.ascontiguousarray(e._ftrunc, dtype=np.int32)


def _layout(case, orders):
    h = host_shape(orders)
    ry, kpad = h["ry"], h["kpad"]
    if case.layout == "kpad":
        return np.full(ry, kpad, dtype=np.int32)
    if case.layout == "four":
        return np.full(ry, 4, dtype=np.int32)
    if case.layout == "zigzag":             # non-monotone, every multiple of 4 up to kpad, ending on kpad
        k = np.array([4 + 4 * ((5 * l + 3) % (kpad // 4)) for l in range(ry)], dtype=np.int32)
        k[-1] = kpad
        return k
    return None


class Call:
    """Guarded buffers and the C-ABI calls of one case."""

    def __init__(self, case, orders, ux, uy, box, kx):
        self.nat, self.lib = _lib()
        self.case, self.orders, self.box, self.kx = case, orders, box, kx
        self.kxp = None if kx is None else ctypes.c_void_p(kx.ctypes.data)
        self.ux = torch.from_numpy(ux).cuda()
        self.uy = torch.from_numpy(uy).cuda()
        self.G = case.ncols * case.ny
        self.guards = []
        self.st = self.nat.stream_ptr()

    def buf(self, n, fill=np.nan):
        big, b = _guarded(n, fill)
        self.guards.append(big)
        return b

    def outputs(self):
        return self.buf(self.G), self.buf(self.G), self.buf(self.G)

    def work(self, npad):
        n = int(self.lib.mfgp_factored_workspace_bytes(npad, self.case.ncols, self.case.ny, *self.orders, self.case.chunk))
        return self.buf(n // 8), n

    def geom(self):
        c = self.case
        return (self.nat.ptr(self.ux), c.nx, self.nat.ptr(self.uy), c.ny, c.ix0, c.ncols)

    def intact(self):
        torch.cuda.synchronize()
        return all(_intact(g) for g in self.guards)

    def standing(self, e, mu, var, qred, Gs=None, Hs=None, trunc=False):
        nat = self.nat
        work, nb = self.work(e.npad)
        return self.lib.mfgp_posterior_grid_factored_trunc(
            *self.geom(), nat.ptr(e.Xt), e.NL, e.NH, nat.ptr(e.W), e.npad, e.cap, nat.ptr(e.z), ctypes.byref(e.pstruct),
            *self.orders, *self.box, self.case.chunk, self.kxp if trunc else None, nat.ptr(mu), nat.ptr(var), nat.ptr(qred),
            nat.ptr(Gs), nat.ptr(Hs), nat.ptr(work), nb, self.st)

    def fused(self, e, mu, var, qred, gram, Gs=None, Hs=None):
        """build_train_cov -> prepare -> the fused factorisation with the right-hand sides -> the solved form."""
        nat, lib, c = self.nat, self.lib, self.case
        npad = e.npad
        pp = ctypes.byref(e.pstruct)
        work, nb = self.work(npad)
        R = int(lib.mfgp_factored_rhs_cols_trunc(len(self.kx), self.kxp) if self.kx is not None else lib.mfgp_factored_rhs_cols(*self.orders))
        K, W, Tt = self.buf(npad * npad), self.buf(npad * npad), self.buf(npad * 4)
        Ball, zout = self.buf(npad * R), self.buf(npad)
        info = torch.full((1,), 12345, dtype=torch.int32, device="cuda")
        assert lib.mfgp_build_train_cov(nat.ptr(e.Xt), e.NL, e.NH, pp, nat.ptr(K), npad, npad, nat.ptr(Tt), self.st) == 0
        rc = lib.mfgp_factored_prepare_trunc(*self.geom(), nat.ptr(e.Xt), nat.ptr(e.y), e.NL, e.NH, npad, pp, *self.orders, *self.box,
                                             c.chunk, self.kxp, nat.ptr(Ball), R, nat.ptr(work), nb, self.st)
        assert rc == 0, nat.last_error()
        if gram:
            M = lib.mfgp_factored_gram_target(c.nx, c.ny, c.ix0, c.ncols, e.NL, e.NH, npad, pp, *self.orders, c.chunk, self.kxp, R,
                                              nat.ptr(work), nb)
            assert M, "mfgp_factored_gram_target declined the Gram route"
            nw = int(lib.mfgp_cholesky_solve_gram_workspace_bytes(npad, R))
            cw = self.buf(nw // 8, 0.0)
            rc = lib.mfgp_cholesky_solve_gram(nat.ptr(K), npad, npad, nat.ptr(W), npad, nat.ptr(info), nat.ptr(Ball), R, R,
                                              ctypes.c_void_p(M), R, nat.ptr(cw), nw, self.st)
        else:
            nw = int(lib.mfgp_cholesky_solve_workspace_bytes(npad, R))
            cw = self.buf(nw // 8, 0.0)
            rc = lib.mfgp_cholesky_solve(nat.ptr(K), npad, npad, nat.ptr(W), npad, nat.ptr(info), nat.ptr(Ball), R, R, nat.ptr(cw),
                                         nw, self.st)
        assert rc == 0, nat.last_error()
        solved = lib.mfgp_posterior_grid_factored_solved_gram if gram else lib.mfgp_posterior_grid_factored_solved
        args = (*self.geom(), nat.ptr(e.Xt), e.NL, e.NH, npad, pp, *self.orders, *self.box, c.chunk) + \
               ((self.kxp,) if gram else ()) + \
               (nat.ptr(Ball), R, nat.ptr(zout), nat.ptr(mu), nat.ptr(var), nat.ptr(qred), nat.ptr(Gs), nat.ptr(Hs),
                nat.ptr(work), nb, self.st)
        rc = solved(*args)
        torch.cuda.synchronize()
        assert int(info.item()) == 0
        return rc

    def update(self, e, row_lo, mu, var, qred, Gs, Hs):
        nat = self.nat
        work, nb = self.work(e.npad)
        return self.lib.mfgp_posterior_grid_factored_update(
            *self.geom(), nat.ptr(e.Xt), e.NL, e.NH, row_lo, nat.ptr(e.W), e.npad, e.cap, nat.ptr(e.z), ctypes.byref(e.pstruct),
            *self.orders, *self.box, self.case.chunk, nat.ptr(mu), nat.ptr(var), nat.ptr(qred), nat.ptr(Gs), nat.ptr(Hs),
            nat.ptr(work), nb, self.st)


def _compare(case, p, ref, mu, var, qred, drop_ref, what):
    """Device (mu, var, qred) against the restatement; the restatement without its highest term must be far outside."""
    mu, var, qred = (t.cpu().numpy() for t in (mu, var, qred))
    mu_r, var_r, q_r = ref
    tv = TOL * max(p.k0, float(np.max(np.abs(q_r))))
    tm = TOL * max(1.0, float(np.max(np.abs(mu_r))))
    assert np.all(np.isfinite(mu)) and np.all(np.isfinite(var)) and np.all(np.isfinite(qred)), (what, "non-finite output")
    assert np.array_equal(p.k0 - qred, var), what
    ev, eq, em = (float(np.max(np.abs(a - b))) for a, b in ((var, var_r), (qred, q_r), (mu, mu_r)))
    print(f"\n[{case.cid} {what}] err var {ev / p.k0:.2e} k0, q {eq / p.k0:.2e} k0, mu {em:.2e} "
          f"(tol {tv / p.k0:.1e} k0 / {tm:.1e})")
    assert ev <= tv and eq <= tv and em <= tm, (what, ev, eq, em, tv, tm)
    sens = max(float(np.max(np.abs(drop_ref[1] - var_r))) / tv, float(np.max(np.abs(drop_ref[0] - mu_r))) / tm)
    assert sens > 100.0, (what, "the case cannot tell its highest term apart", sens)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=repr)
def test_factored_kernels_match_the_restatement(case, monkeypatch):
    monkeypatch.setenv("MFGP_DEBUG_POISON_SMEM", "1")
    monkeypatch.setenv("MFGP_GRAM", "direct" if case.route in DIRECT_ROUTES else "m")
    ux, uy, box = _grid(case)
    if case.layout == "planner":
        orders, kx = _planner_layout(case, ux, uy, box)
    else:
        orders, kx = case.orders, None
        kx = _layout(case, orders)
    X_L, y_L, X_H, y_H = _data(case.multi, case.N + case.add)
    nh0 = X_H.shape[0] - case.add
    call = Call(case, orders, ux, uy, box, kx)

    def reference(n_h):
        p, fac = _reference_factor(case.multi, case.N + case.add, n_h)
        args = (p, X_L, y_L, X_H[:n_h], y_H[:n_h], ux, uy, case.ix0, case.ncols, orders, box, kx)
        ref = ofac.posterior(*args, fac=fac)
        drop = ofac.posterior(*args, drop=ofac.highest_term(p, orders, kx), fac=fac)
        return p, ref, drop

    mu, var, qred = call.outputs()
    if case.route in ("direct", "gram"):
        e = _standing(case.multi, case.N)
        rc = call.standing(e, mu, var, qred, trunc=True)
    elif case.route in ("fdirect", "fgram"):
        e = _standing(case.multi, case.N)
        rc = call.fused(e, mu, var, qred, gram=case.route == "fgram")
    else:
        e = _device_model(case.multi, X_L, y_L, X_H[:nh0], y_H[:nh0], SHORT, incremental=True)
        Gs = call.buf(case.ncols * 64 * 64)
        Hs = call.buf(call.lib.mfgp_factored_rhs_cols(*orders))
        rc = call.standing(e, mu, var, qred, Gs, Hs) if case.route == "incr" else call.fused(e, mu, var, qred, True, Gs, Hs)
    torch.cuda.synchronize()
    assert rc == 0, call.nat.last_error()
    assert call.intact(), "a write landed outside its buffer"
    p, ref, drop = reference(nh0)
    _compare(case, p, ref, mu, var, qred, drop, "full")
    if case.add:
        row_lo = e.N
        e.append_hifi(X_H[nh0:], y_H[nh0:])
        assert e.N == row_lo + case.add
        mu, var, qred = call.outputs()
        rc = call.update(e, row_lo, mu, var, qred, Gs, Hs)
        torch.cuda.synchronize()
        assert rc == 0, call.nat.last_error()
        assert call.intact(), "a write landed outside its buffer"
        p, ref, drop = reference(X_H.shape[0])
        _compare(case, p, ref, mu, var, qred, drop, "update")


@pytest.mark.gpu
def test_invalid_arguments_are_rejected_untouched(monkeypatch):
    """MFGP_ERR_INVALID (NULL from mfgp_factored_gram_target) for arguments outside the contract, with every output and the
    workspace keeping their bits: nothing is enqueued."""
    monkeypatch.setenv("MFGP_GRAM", "m")
    nat, lib = _lib()
    case = Case("reject", True, (8, 8, 8, 8), "gram", 70, 20, 2, 16, 9)
    ux, uy, box = _grid(case)
    call = Call(case, case.orders, ux, uy, box, None)
    eM, eS = _standing(True, 70), _standing(False, 70)
    npad, ok = eM.npad, case.orders
    nb = int(lib.mfgp_factored_workspace_bytes(npad, case.ncols, case.ny, 64, 64, 64, 64, case.chunk))    # room for any order
    need = int(lib.mfgp_factored_workspace_bytes(npad, case.ncols, case.ny, *ok, case.chunk))
    R = int(lib.mfgp_factored_rhs_cols(*ok))
    mu, var, qred = call.outputs()
    work, Y = call.buf(nb // 8), call.buf(npad * (R + 64))
    Gs, Hs = call.buf(case.ncols * 64 * 64), call.buf(R)
    watched = (mu, var, qred, work, Y, Gs, Hs)
    st, P = call.st, nat.ptr
    kxs = {"kx 0": [8, 8, 0, 8, 8, 8, 8, 8], "kx 6": [8, 6, 8, 8, 8, 8, 8, 8], "kx > kpad": [8, 8, 8, 8, 8, 8, 8, 12]}
    kxs = {k: np.array(v, dtype=np.int32) for k, v in kxs.items()}
    kp = lambda kx: None if kx is None else ctypes.c_void_p(kx.ctypes.data)

    def standing(e, orders, NL=None, ix0=case.ix0, wb=nb, kx=None, stores=False):
        NL = e.NL if NL is None else NL
        return lib.mfgp_posterior_grid_factored_trunc(
            P(call.ux), case.nx, P(call.uy), case.ny, ix0, case.ncols, P(e.Xt), NL, e.N - NL, P(e.W), npad, e.cap, P(e.z),
            ctypes.byref(e.pstruct), *orders, *box, case.chunk, kp(kx), P(mu), P(var), P(qred), P(Gs) if stores else None,
            P(Hs) if stores else None, P(work), wb, st)

    def prepare(e, orders, NL=None, wb=nb, kx=None):
        NL = e.NL if NL is None else NL
        return lib.mfgp_factored_prepare_trunc(P(call.ux), case.nx, P(call.uy), case.ny, case.ix0, case.ncols, P(e.Xt), P(e.y), NL,
                                               e.N - NL, npad, ctypes.byref(e.pstruct), *orders, *box, case.chunk, kp(kx), P(Y), R,
                                               P(work), wb, st)

    def solved(ldY, gram, wb=nb, kx=None):
        fn = lib.mfgp_posterior_grid_factored_solved_gram if gram else lib.mfgp_posterior_grid_factored_solved
        return fn(P(call.ux), case.nx, P(call.uy), case.ny, case.ix0, case.ncols, P(eM.Xt), eM.NL, eM.NH, npad,
                  ctypes.byref(eM.pstruct), *ok, *box, case.chunk, *((kp(kx),) if gram else ()), P(Y), ldY, None, P(mu), P(var),
                  P(qred), None, None, P(work), wb, st)

    def target(ldY, wb=nb, kx=None):
        return lib.mfgp_factored_gram_target(case.nx, case.ny, case.ix0, case.ncols, eM.NL, eM.NH, npad, ctypes.byref(eM.pstruct),
                                             *ok, case.chunk, kp(kx), ldY, P(work), wb)

    calls = {
        "ryH not a multiple of 4": lambda: standing(eS, (0, 0, 8, 6)),
        "ryL not a multiple of 4": lambda: standing(eM, (8, 6, 8, 8)),
        "rxH above 64": lambda: standing(eS, (0, 0, 65, 8)),
        "ryH above 64": lambda: standing(eS, (0, 0, 8, 68)),
        "ryL above 64": lambda: standing(eM, (8, 68, 8, 8)),
        "ix0 + ncols > nx": lambda: standing(eM, ok, ix0=case.nx - case.ncols + 1),
        "short work": lambda: standing(eM, ok, wb=need - 8),
        "short work, stores": lambda: standing(eM, ok, wb=need - 8, stores=True),
        "short work, prepare": lambda: prepare(eM, ok, wb=need - 8),
        "short work, solved": lambda: solved(R, False, wb=need - 8),
        "MF with rxL = 0": lambda: standing(eM, (0, 8, 8, 8)),
        "MF with rxL = 0, prepare": lambda: prepare(eM, (0, 8, 8, 8)),
        "SF with NL > 0": lambda: standing(eS, (0, 0, 8, 8), NL=5),
        "SF with NL > 0, prepare": lambda: prepare(eS, (0, 0, 8, 8), NL=5),
        "ldY > Rp, solved": lambda: solved(R + 64, False),
        "ldY > Rp, solved_gram": lambda: solved(R + 64, True),
    }
    for name, kx in kxs.items():
        calls[name] = functools.partial(standing, eM, ok, kx=kx)
        calls[name + ", prepare"] = functools.partial(prepare, eM, ok, kx=kx)
        calls[name + ", solved_gram"] = functools.partial(solved, R, True, kx=kx)
    torch.cuda.synchronize()
    before = [_bits(b) for b in watched]
    for name, fn in calls.items():
        rc = fn()
        torch.cuda.synchronize()
        assert rc == nat.MFGP_ERR_INVALID, (name, rc)
        assert all(np.array_equal(_bits(b), x) for b, x in zip(watched, before)), (name, "a rejected call wrote")
    assert target(R) is not None                                          # the valid geometry has a Gram target
    for name, ptr_ in {"ldY > Rp": target(R + 64), "short work": target(R, wb=need - 8),
                       **{n: target(R, kx=kx) for n, kx in kxs.items()}}.items():
        assert ptr_ is None, name
    assert call.intact()
