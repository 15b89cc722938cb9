"""GPU: joint posterior draws (mfgp_posterior_cov_factor, mfgp_posterior_sample, sample_posterior[_device]).  The factor
reproduces the oracle's covariance plus jitter; the product kernel matches numpy for every tile edge, reads only the
lower triangle of L and writes only F[G][S]; draws are causal, reproducible and match the oracle's draws for the same
normals; the default jitter factors the ill-conditioned cases; status and argument errors."""
import ctypes
import os

import numpy as np
import pytest

from oracle import gp as ogp
from oracle import gp_cov as ogc
from oracle import gp_sample as ogs
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


def _factor_by_identity(m, xs_dev, grid=None):
    """E = I: F - mu = L (the whole G x G factor, strict upper part included)."""
    import torch
    G = int(xs_dev.shape[0])
    mu, F = m.sample_posterior_device(xs_dev, torch.eye(G, dtype=torch.float64, device="cuda"), grid=grid)
    return mu, F - mu[:, None]


@pytest.mark.parametrize("n,N,multi", [(51, 9, True), (51, 130, True), (51, 259, True), (51, 64, False), (51, 200, False),
                                       ("scattered", 300, True)])
def test_factor_reproduces_the_oracle_covariance(n, N, multi):
    import torch
    from mfgp_coverage_b200._coverage import CoverageGrid
    xy, data, p, m = _case(51 if n == "scattered" else n, N, multi)
    if n == "scattered":
        xy = np.random.default_rng(3).random((3001, 2))
        mu, L = _factor_by_identity(m, _dev(xy))
    else:
        g = CoverageGrid(xy)
        mu, L = _factor_by_identity(m, g.xy, grid=g)
    torch.cuda.synchronize()
    G = xy.shape[0]
    tau = 1e-8 * p.k0
    _, C_o = ogc.posterior_cov(p, xy, *data)
    LLt = torch.mm(L, L.T).cpu().numpy()
    assert np.max(np.abs(LLt - (C_o + tau * np.eye(G)))) <= TOL * p.k0
    assert torch.count_nonzero(torch.triu(L, 1)) == 0


def _lower_with_nan(G, ldl, rng):
    import torch
    L = rng.standard_normal((G, G))
    L = np.tril(L) + np.diag(np.abs(np.diag(L)) + 1.0)
    buf = np.full((G, ldl), np.nan)
    buf[:, :G] = np.where(np.tril(np.ones((G, G), dtype=bool)), L, np.nan)
    buf[np.triu_indices(G, 1)] = np.inf if G % 2 else np.nan
    return np.tril(L), torch.from_numpy(buf).cuda()


@pytest.mark.parametrize("G", [1, 63, 64, 65, 127, 129, 2601])
def test_product_kernel_matches_numpy(G):
    """F = mu + tril(L) E through the C-ABI with NaN / Inf in L's strict upper part, tight and padded strides, canaries
    around F and in its padding columns."""
    import torch
    from mfgp_coverage_b200 import _native as nat
    lib = nat.lib()
    st = nat.stream_ptr()
    rng = np.random.default_rng(G)
    pad = 64
    for S in (1, 2, 63, 64, 65, 1000):
        for extra in (0, 6):
            ldl, lde, ldf = G + (G & 1) + extra, S + (S & 1) + extra, S + (S & 1) + extra
            Lh, L = _lower_with_nan(G, ldl, rng)
            mu_h = rng.standard_normal(G) * 3.0
            E_h = rng.standard_normal((G, S))
            E = torch.full((G, lde), np.nan, dtype=torch.float64, device="cuda")
            E[:, :S] = torch.from_numpy(E_h).cuda()
            mu = _dev(mu_h)
            buf = torch.full((2 * pad + G * ldf,), CANARY, dtype=torch.float64, device="cuda")
            F = buf[pad:pad + G * ldf]
            rc = lib.mfgp_posterior_sample(nat.ptr(L), G, ldl, nat.ptr(mu), nat.ptr(E), lde, S, nat.ptr(F), ldf, st)
            assert rc == nat.MFGP_OK
            torch.cuda.synchronize()
            b = buf.cpu().numpy()
            assert np.all(b[:pad] == CANARY) and np.all(b[pad + G * ldf:] == CANARY), (G, S, extra)
            inner = b[pad:pad + G * ldf].reshape(G, ldf)
            assert np.all(inner[:, S:] == CANARY), (G, S, extra)
            ref = mu_h[:, None] + Lh @ E_h
            bound = 1e-12 * (np.abs(mu_h)[:, None] + np.abs(Lh) @ np.abs(E_h))
            assert np.all(np.abs(inner[:, :S] - ref) <= bound), (G, S, extra)
            if extra == 0 and S in (1, 64):
                snapshot = buf.clone()
                bad = [dict(ldl=ldl + 1), dict(lde=lde + 1), dict(ldf=ldf + 1), dict(Loff=1), dict(Eoff=1), dict(Foff=1)]
                for kw in bad:
                    Lp = L.view(-1)[kw.get("Loff", 0):]
                    Ep = E.view(-1)[kw.get("Eoff", 0):]
                    Fp = F[kw.get("Foff", 0):]
                    rc = lib.mfgp_posterior_sample(nat.ptr(Lp), G, kw.get("ldl", ldl), nat.ptr(mu), nat.ptr(Ep),
                                                   kw.get("lde", lde), S, nat.ptr(Fp), kw.get("ldf", ldf), st)
                    assert rc == nat.MFGP_ERR_INVALID, kw
                torch.cuda.synchronize()
                assert torch.equal(buf, snapshot)


def test_draws_are_causal():
    """A normal vector that is non-zero only in row r moves no row before r, exactly."""
    import torch
    xy, data, p, m = _case(51, 130, True)
    xs = _dev(xy)
    G = xy.shape[0]
    for r in (0, 1, 63, 64, 1000, G - 1):
        E = torch.zeros((G, 3), dtype=torch.float64, device="cuda")
        E[r] = torch.tensor([1.0, -2.5, 1e3], dtype=torch.float64)
        mu, F = m.sample_posterior_device(xs, E)
        D = (F - mu[:, None]).cpu().numpy()
        assert np.all(D[:r] == 0.0), r
        assert np.all(D[r] != 0.0), r


@pytest.mark.parametrize("n,N,multi", [(51, 130, True), (51, 64, False), ("scattered", 300, True)])
def test_draws_match_the_oracle_for_the_same_normals(n, N, multi):
    """jitter 1e-2 k(0): the factor is well determined (condition number <= ~100 G), so the device's and LAPACK's agree."""
    xy, data, p, m = _case(51 if n == "scattered" else n, N, multi)
    if n == "scattered":
        xy = np.random.default_rng(8).random((1500, 2))
    tau = 1e-2 * p.k0
    F = m.sample_posterior(xy, n_samples=16, rng=np.random.default_rng(17), jitter=tau)
    E = np.random.default_rng(17).standard_normal((xy.shape[0], 16))
    F_o = ogs.posterior_samples(p, xy, *data, E, tau)
    mu_o, _ = ogc.posterior_cov(p, xy, *data)
    assert F.shape == (xy.shape[0], 16)
    assert np.max(np.abs(F - F_o)) <= TOL * max(1.0, np.max(np.abs(mu_o)), np.sqrt(p.k0))


def test_reproducible():
    import torch
    xy, data, p, m = _case(51, 259, True)
    a = m.sample_posterior(xy, n_samples=70, rng=np.random.default_rng(5))
    b = m.sample_posterior(xy, n_samples=70, rng=np.random.default_rng(5))
    c = m.sample_posterior(xy, n_samples=70, rng=np.random.default_rng(6))
    assert np.array_equal(a, b) and not np.array_equal(a, c)
    from mfgp_coverage_b200._coverage import CoverageGrid
    g = CoverageGrid(xy)
    E = torch.from_numpy(np.random.default_rng(1).standard_normal((xy.shape[0], 129))).cuda()
    mu1, F1 = m.sample_posterior_device(g.xy, E, grid=g)
    mu2, F2 = m.sample_posterior_device(g.xy, E, grid=g)
    assert torch.equal(F1, F2) and torch.equal(mu1, mu2)


def test_default_jitter_on_the_logged_ex_gp_hyper_parameters(golden_dir):
    """Ill-conditioned: the reference's logged ex_gp hyper-parameters and 25-point lofi prior (2020 raw-mean convention)."""
    import torch
    g = np.load(os.path.join(golden_dir, "logged_ex_gp.npz"), allow_pickle=False)
    pr = g["prior"]
    e = np.empty((0, 2)), np.empty((0, 1))
    p, m = _models(g["hyp"], pr[:, :2], pr[:, 2:3], e[0], e[1], raw_means=True)
    _, L = _factor_by_identity(m, _dev(g["xs"]))
    _, C_o = ogc.posterior_cov(p, g["xs"], pr[:, :2], pr[:, 2:3], e[0], e[1])
    G = C_o.shape[0]
    assert np.max(np.abs(torch.mm(L, L.T).cpu().numpy() - (C_o + 1e-8 * p.k0 * np.eye(G)))) <= TOL * p.k0
    F = m.sample_posterior(g["xs"], n_samples=4, rng=np.random.default_rng(0))
    assert np.all(np.isfinite(F))


@pytest.mark.parametrize("multi", [True, False])
def test_empty_model_draws_from_the_prior(multi):
    import torch
    from mfgp_coverage_b200.gaussian_process import MFGP, SFGP
    xy = synth.grid(20)
    e = np.empty([0, 2]), np.empty([0, 1])
    m = MFGP(e[0], e[1], e[0], e[1], 1, 1) if multi else SFGP(e[0], e[1], 1)
    m.hyp = synth.MF_HYP if multi else synth.SF_HYP
    p = ogp.GPParams.from_hyp(m.hyp)
    mu, L = _factor_by_identity(m, _dev(xy))
    assert torch.all(mu == p.mean_H)
    K = ogc.prior_cov(p, xy, xy) + 1e-8 * p.k0 * np.eye(xy.shape[0])
    assert np.max(np.abs(torch.mm(L, L.T).cpu().numpy() - K)) <= TOL * p.k0
    assert np.all(np.isfinite(m.sample_posterior(xy, n_samples=3, rng=np.random.default_rng(1))))


def _factor_rows_residual(m, p, xy, rows):
    """Factor the joint covariance of the grid xy at the default jitter through the C-ABI sequence and return
    (info, max |L[rows] L^T - (C + tau I)[rows]|), with C kept from before the factorisation (all on the device)."""
    import torch
    from mfgp_coverage_b200 import _native as nat
    from mfgp_coverage_b200._coverage import CoverageGrid
    g = CoverageGrid(xy)
    eng = m.engine
    G = xy.shape[0]
    npad = nat.npad(G)
    tau = 1e-8 * p.k0
    C = torch.empty((npad, npad), dtype=torch.float64, device="cuda")
    eng.posterior_cov(g.xy, axes_a=g.axes, g_lo_a=g.base_index, out=C[:G, :G])
    r = torch.from_numpy(rows).cuda()
    C_rows = C[r, :G].clone()
    C_rows[torch.arange(len(rows), device="cuda"), r] += tau
    W = torch.empty((npad, npad), dtype=torch.float64, device="cuda")
    work = torch.empty(int(nat.lib().mfgp_workspace_bytes(npad)) // 8 + 1, dtype=torch.float64, device="cuda")
    info = torch.zeros(1, dtype=torch.int32, device="cuda")
    nat.check(nat.lib().mfgp_posterior_cov_factor(nat.ptr(C), G, npad, npad, tau, nat.ptr(W), npad, nat.ptr(info),
                                                  nat.ptr(work), nat.stream_ptr()), "mfgp_posterior_cov_factor")
    del W, work
    L = torch.tril(C[:G, :G])
    del C
    res = float((torch.mm(L[r], L.T) - C_rows).abs().max())
    return int(info.item()), res


@pytest.mark.parametrize("nx,ny", [(128, 128), (256, 128)])
def test_default_jitter_at_c4_scale_and_the_largest_size(nx, ny):
    """N = 4096 (the c4 training set); 16384 points, and 32768 (npad = 32768, the largest factor accepted)."""
    import torch
    big = synth.grid(1024)
    f = synth.truth_function(big)
    data = synth.training_set(big, f, 4096)
    p, m = _models(synth.MF_HYP, *data)
    gx, gy = np.linspace(0, 1, nx), np.linspace(0, 1, ny)
    xy = np.stack(np.meshgrid(gx, gy, indexing="ij"), axis=-1).reshape(-1, 2)
    rows = np.sort(np.random.default_rng(4).choice(xy.shape[0], 256, replace=False))
    info, res = _factor_rows_residual(m, p, xy, rows)
    assert info == 0
    assert res <= TOL * p.k0
    torch.cuda.empty_cache()
    if nx == 128:
        F = m.sample_posterior(xy, n_samples=8, rng=np.random.default_rng(2))
        assert F.shape == (xy.shape[0], 8) and np.all(np.isfinite(F))


@pytest.mark.parametrize("k", [0, 63, 64, 137, 199])
def test_non_positive_pivot_is_reported_like_lapack(k):
    import scipy.linalg
    import torch
    from mfgp_coverage_b200 import _native as nat
    G, npad = 200, 256
    A = np.eye(G) + 0.01 * np.ones((G, G))
    A[k, k] = -1.0
    info_ref = scipy.linalg.lapack.dpotrf(A, lower=1)[1]
    C = torch.full((npad, npad), np.nan, dtype=torch.float64, device="cuda")
    C[:G, :G] = _dev(A)
    W = torch.empty((npad, npad), dtype=torch.float64, device="cuda")
    work = torch.empty(int(nat.lib().mfgp_workspace_bytes(npad)) // 8 + 1, dtype=torch.float64, device="cuda")
    info = torch.zeros(1, dtype=torch.int32, device="cuda")
    rc = nat.lib().mfgp_posterior_cov_factor(nat.ptr(C), G, npad, npad, 0.0, nat.ptr(W), npad, nat.ptr(info),
                                             nat.ptr(work), nat.stream_ptr())
    assert rc == nat.MFGP_OK
    assert int(info.item()) == 1 + k == info_ref
    # rejected calls enqueue nothing
    for kw in (dict(npad=npad + 1), dict(npad=32768 + 64), dict(ld=npad + 1), dict(jitter=-1.0), dict(G=npad + 1)):
        info.fill_(-5)
        rc = nat.lib().mfgp_posterior_cov_factor(nat.ptr(C), kw.get("G", G), kw.get("npad", npad), kw.get("ld", npad),
                                                 kw.get("jitter", 0.0), nat.ptr(W), npad, nat.ptr(info), nat.ptr(work),
                                                 nat.stream_ptr())
        assert rc == nat.MFGP_ERR_INVALID, kw
        assert int(info.item()) == -5, kw


def test_non_spd_training_covariance_raises_linalgerror():
    from mfgp_coverage_b200.gaussian_process import SFGP, evaluate_hyp
    X = np.array([[0.1, 0.1], [0.4, 0.2], [0.5, 0.5]])
    m = SFGP(X, np.zeros((3, 1)), 1)
    m.hyp = synth.SF_HYP
    m.params = lambda: dict(evaluate_hyp(synth.SF_HYP), noise_H=-1.0)    # diagonal = scale - 1 < 0: indefinite on purpose
    m.updt_info(X, np.zeros((3, 1)))
    with pytest.raises(np.linalg.LinAlgError):
        m.sample_posterior(synth.grid(9), n_samples=2, rng=np.random.default_rng(0))


def test_argument_errors(monkeypatch):
    import torch
    xy, data, p, m = _case(20, 40, True)
    for n in (0, -1, 1.5):
        with pytest.raises(ValueError):
            m.sample_posterior(xy, n_samples=n)
    with pytest.raises(ValueError):
        m.sample_posterior(xy, n_samples=2, jitter=-1e-9)
    with pytest.raises(ValueError):
        m.sample_posterior(np.random.default_rng(0).random((32769, 2)), n_samples=1)
    # a point set whose covariance alone exceeds the free device memory: MemoryError before anything is allocated
    m.engine.ensure_factor()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    pts = np.random.default_rng(1).random((16384, 2))
    xs = _dev(pts)
    E = torch.zeros((16384, 1), dtype=torch.float64, device="cuda")
    total = torch.cuda.mem_get_info()[1]
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda *a, **k: (1 << 30, total))
    before = torch.cuda.memory_allocated()
    with pytest.raises(MemoryError):
        m.sample_posterior_device(xs, E)
    assert torch.cuda.memory_allocated() == before
