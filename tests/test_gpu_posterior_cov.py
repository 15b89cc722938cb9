"""GPU: the joint / cross posterior covariance (mfgp_posterior_cov, predict(full_cov=True), predict_cov_device) against the
oracle's full-matrix restatement (oracle.gp_cov.posterior_cov), and its structural guarantees: exact symmetry, bitwise
reproducibility, cross blocks that match the joint matrix, stride rules and canaries around C."""
import ctypes
import os

import numpy as np
import pytest

from oracle import gp as ogp
from oracle import gp_cov as ogc
from tests import synth

pytestmark = pytest.mark.gpu
TOL = 1e-9
CANARY = -7.25e300


def _models(hyp, X_L, y_L, X_H, y_H, raw_means=False):
    from mfgp_coverage_b200.gaussian_process import MFGP, SFGP
    p = ogp.GPParams.from_hyp(hyp, raw_means=raw_means)
    if p.multi:
        m = MFGP(X_L, y_L, X_H, y_H, 1, 1)
        m.raw_means, m.hyp = raw_means, hyp
        m.updt_info(X_L, y_L, X_H, y_H)
    else:
        m = SFGP(X_H, y_H, 1)
        m.raw_means, m.hyp = raw_means, hyp
        m.updt_info(X_H, y_H)
    return p, m


def _case(n, N, multi, seed=1234):
    xy = synth.grid(n)
    f = synth.truth_function(xy)
    X_L, y_L, X_H, y_H = synth.training_set(xy, f, N, seed=seed, multi=multi)
    p, m = _models(synth.MF_HYP if multi else synth.SF_HYP, X_L, y_L, X_H, y_H)
    return xy, (X_L, y_L, X_H, y_H), p, m


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()


@pytest.mark.parametrize("n,N,multi", [(51, 9, True), (51, 40, True), (51, 130, True), (64, 300, True),
                                       (51, 64, False), (51, 200, False), (96, 700, True), (64, 1100, True)])
def test_full_cov_matches_oracle(n, N, multi):
    xy, data, p, m = _case(n, N, multi)
    mu, cov = m.predict(xy, full_cov=True)
    mu_o, cov_o = ogc.posterior_cov(p, xy, *data)
    assert mu.shape == (xy.shape[0], 1) and cov.shape == (xy.shape[0], xy.shape[0])
    assert np.max(np.abs(cov - cov_o)) <= TOL * p.k0
    assert np.max(np.abs(mu[:, 0] - mu_o)) <= TOL * max(1.0, np.max(np.abs(mu_o)))
    # the diagonal is the default predict's variance
    _, var = m.predict(xy)
    assert np.max(np.abs(np.diag(cov) - var)) <= 1e-12 * p.k0


@pytest.mark.parametrize("multi,N", [(True, 300), (False, 130)])
def test_scattered_points_match_oracle(multi, N):
    xy, data, p, m = _case(40, N, multi)
    pts = np.random.default_rng(3).random((3001, 2))
    mu, cov = m.predict(pts, full_cov=True)
    mu_o, cov_o = ogc.posterior_cov(p, pts, *data)
    assert np.max(np.abs(cov - cov_o)) <= TOL * p.k0
    assert np.max(np.abs(mu[:, 0] - mu_o)) <= TOL * max(1.0, np.max(np.abs(mu_o)))
    _, var = m.predict(pts)
    assert np.max(np.abs(np.diag(cov) - var)) <= 1e-12 * p.k0


def test_exactly_symmetric_and_reproducible():
    import torch
    xy, data, p, m = _case(51, 259, True)       # 2601 points: 21 tiles per side, the last one partial
    from mfgp_coverage_b200._coverage import CoverageGrid
    g = CoverageGrid(xy)
    _, C1 = m.predict_cov_device(g.xy, grid=g)
    _, C2 = m.predict_cov_device(g.xy, grid=g)
    torch.cuda.synchronize()
    assert C1.shape == (2601, 2601) and C1.stride(0) % 2 == 0
    assert torch.equal(C1, C1.T)
    assert torch.equal(C1, C2)
    pts = _dev(np.random.default_rng(9).random((700, 2)))
    _, S1 = m.predict_cov_device(pts)
    _, S2 = m.predict_cov_device(pts)
    assert torch.equal(S1, S1.T) and torch.equal(S1, S2)


@pytest.mark.parametrize("multi,N", [(True, 201), (False, 77)])
def test_cross_blocks_match_the_joint_matrix(multi, N):
    import torch
    from mfgp_coverage_b200._coverage import CoverageGrid
    xy, data, p, m = _case(51, N, multi)
    rng = np.random.default_rng(11)
    sets = {1: rng.random((1, 2)), 63: rng.random((63, 2)), 65: rng.random((65, 2))}
    g = CoverageGrid(xy)                         # 2601 points of a tensor grid: V from the separable kernel
    for ga, gb in ((1, 63), (65, 1), (63, 65), (65, 2601), (2601, 63)):
        A = xy if ga == 2601 else sets[ga]
        B = xy if gb == 2601 else sets[gb]
        dA, dB = (g.xy if ga == 2601 else _dev(A)), (g.xy if gb == 2601 else _dev(B))
        gA, gB = (g if ga == 2601 else None), (g if gb == 2601 else None)
        mu_a, C_ab = m.predict_cov_device(dA, dB, grid=gA, grid2=gB)
        _, C_ba = m.predict_cov_device(dB, dA, grid=gB, grid2=gA)
        _, J = m.predict_cov_device(_dev(np.vstack((A, B))))
        torch.cuda.synchronize()
        assert C_ab.shape == (ga, gb)
        assert torch.equal(C_ab, C_ba.T), (ga, gb)
        blk = J[:ga, ga:]
        assert float((C_ab - blk).abs().max()) <= 1e-12 * p.k0, (ga, gb)
        _, C_o = ogc.posterior_cov(p, A, *data, X_b=B)
        assert np.max(np.abs(C_ab.cpu().numpy() - C_o)) <= TOL * p.k0, (ga, gb)
        assert mu_a.shape == (ga,)


@pytest.mark.parametrize("multi", [True, False])
def test_empty_model_is_the_prior(multi):
    from mfgp_coverage_b200.gaussian_process import MFGP, SFGP
    xy = synth.grid(20)
    e = np.empty([0, 2]), np.empty([0, 1])
    m = MFGP(e[0], e[1], e[0], e[1], 1, 1) if multi else SFGP(e[0], e[1], 1)
    m.hyp = synth.MF_HYP if multi else synth.SF_HYP
    p = ogp.GPParams.from_hyp(m.hyp)
    for pts in (xy, np.random.default_rng(1).random((333, 2))):
        mu, cov = m.predict(pts, full_cov=True)
        assert np.all(mu == p.mean_H)
        assert np.max(np.abs(cov - ogc.prior_cov(p, pts, pts))) <= 1e-14 * p.k0
        assert np.array_equal(cov, cov.T)


def test_logged_ex_gp_hyper_parameters(golden_dir):
    """Ill-conditioned: the reference's logged ex_gp hyper-parameters and 25-point lofi prior (2020 raw-mean convention)."""
    g = np.load(os.path.join(golden_dir, "logged_ex_gp.npz"), allow_pickle=False)
    pr = g["prior"]
    e = np.empty((0, 2)), np.empty((0, 1))
    p, m = _models(g["hyp"], pr[:, :2], pr[:, 2:3], e[0], e[1], raw_means=True)
    mu, cov = m.predict(g["xs"], full_cov=True)
    mu_o, cov_o = ogc.posterior_cov(p, g["xs"], pr[:, :2], pr[:, 2:3], e[0], e[1])
    assert np.max(np.abs(cov - cov_o)) <= TOL * p.k0
    assert np.max(np.abs(mu[:, 0] - mu_o)) <= TOL * max(1.0, np.max(np.abs(mu_o)))


def test_c4_scale_rows_against_the_oracle_cross_form():
    """N = 4096 training points (the c4 training set), 16384 points: 256 sampled rows of the joint matrix."""
    import torch
    from mfgp_coverage_b200._coverage import CoverageGrid
    big = synth.grid(1024)
    f = synth.truth_function(big)
    data = synth.training_set(big, f, 4096)
    p, m = _models(synth.MF_HYP, *data)
    xy = synth.grid(128)
    g = CoverageGrid(xy)
    _, C = m.predict_cov_device(g.xy, grid=g)
    torch.cuda.synchronize()
    rows = np.sort(np.random.default_rng(4).choice(xy.shape[0], 256, replace=False))
    got = C[torch.from_numpy(rows).cuda()].cpu().numpy()
    _, C_o = ogc.posterior_cov(p, xy[rows], *data, X_b=xy)
    assert np.max(np.abs(got - C_o)) <= TOL * p.k0
    assert torch.equal(C, C.T)


def test_stride_rules_and_canaries():
    """Nothing outside C[Ga][Gb] changes, with ldc > Gb; odd ldc / ldv are MFGP_ERR_INVALID and leave C untouched."""
    import torch
    from mfgp_coverage_b200 import _native as nat
    xy, data, p, m = _case(30, 150, True)
    eng = m.engine
    eng.ensure_factor()
    lib = nat.lib()
    rng = np.random.default_rng(2)
    Ga, Gb, N = 65, 63, eng.N
    Xa, Xb = _dev(rng.random((Ga, 2))), _dev(rng.random((Gb, 2)))
    lda, ldb = 66, 64
    Va = torch.empty((N, lda), dtype=torch.float64, device="cuda")
    Vb = torch.empty((N, ldb), dtype=torch.float64, device="cuda")
    eng.posterior(Xa, vcache=Va)
    eng.posterior(Xb, vcache=Vb)
    pp = ctypes.byref(eng.pstruct)
    st = nat.stream_ptr()
    pad = 256

    def run(sym, ldc, ldva=lda, ldvb=ldb):
        rows, cols = (Ga, Ga) if sym else (Ga, Gb)
        buf = torch.full((2 * pad + rows * ldc,), CANARY, dtype=torch.float64, device="cuda")
        C = buf[pad:pad + rows * ldc]
        rc = lib.mfgp_posterior_cov(nat.ptr(Xa), Ga, nat.ptr(Va), ldva, None if sym else nat.ptr(Xb), rows if sym else Gb,
                                    None if sym else nat.ptr(Vb), ldvb, N, pp, nat.ptr(C), ldc, st)
        torch.cuda.synchronize()
        return rc, buf.cpu().numpy(), cols

    for sym in (True, False):
        cols = Ga if sym else Gb
        ldc = cols + 8 - cols % 2          # even, 7-8 doubles of margin after each row
        rc, buf, cols = run(sym, ldc)
        assert rc == nat.MFGP_OK
        inner = buf[pad:pad + Ga * ldc].reshape(Ga, ldc)
        assert np.all(buf[:pad] == CANARY) and np.all(buf[pad + Ga * ldc:] == CANARY)
        assert np.all(inner[:, cols:] == CANARY) and not np.any(inner[:, :cols] == CANARY)
        _, C_o = ogc.posterior_cov(p, Xa.cpu().numpy(), *data, X_b=None if sym else Xb.cpu().numpy())
        assert np.max(np.abs(inner[:, :cols] - C_o)) <= TOL * p.k0
        bad = [dict(ldc=ldc + 1), dict(ldc=ldc, ldva=lda - 1)] + ([] if sym else [dict(ldc=ldc, ldvb=ldb - 1)])
        for kw in bad:
            rc, buf, _ = run(sym, **kw)
            assert rc == nat.MFGP_ERR_INVALID, kw
            assert np.all(buf == CANARY), kw


def test_non_spd_full_cov_raises_linalgerror():
    """Deferred fit: the non-SPD covariance surfaces from predict(full_cov=True) as LinAlgError, as it does from predict."""
    from mfgp_coverage_b200.gaussian_process import SFGP, evaluate_hyp
    X = np.array([[0.1, 0.1], [0.4, 0.2], [0.5, 0.5]])
    m = SFGP(X, np.zeros((3, 1)), 1)
    m.hyp = synth.SF_HYP
    m.params = lambda: dict(evaluate_hyp(synth.SF_HYP), noise_H=-1.0)    # diagonal = scale - 1 < 0: indefinite on purpose
    m.updt_info(X, np.zeros((3, 1)))
    xy = synth.grid(9)
    with pytest.raises(np.linalg.LinAlgError):
        m.predict(xy, full_cov=True)
    with pytest.raises(np.linalg.LinAlgError):
        m.predict(xy)
