"""GPU: joint posterior draws over tensor-product grids by pathwise conditioning (mfgp_grid_sample_coef / _eval,
sample_posterior_grid[_device]).  With the identity as normals the draws' linear map A has A A^T = the oracle's posterior
covariance; at equal normals (and the product's own node roots) the draws equal the dense restatement's; at c4 scale column
slices reproduce predict_cov_device; whole grid and column slices give the same bits; the evaluation kernel matches numpy
through the C-ABI for every tile edge; argument, memory and factorisation errors."""
import os

import numpy as np
import pytest

from oracle import gp as ogp
from oracle import gp_cov as ogc
from oracle import gp_sample_grid as osg
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


def _tensor(ux, uy):
    return np.stack(np.meshgrid(ux, uy, indexing="ij"), axis=-1).reshape(-1, 2)


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()


def _identity_draws(m, g):
    """E = [I_d | 0]: returns (mu, A) with F = mu + A E."""
    import torch
    d = m.grid_sample_dim(g)
    E = torch.zeros((d, d + 1), dtype=torch.float64, device="cuda")
    E[:, :d] = torch.eye(d, dtype=torch.float64, device="cuda")
    F = m.sample_posterior_grid_device(g, E)
    mu = F[:, d].clone()
    return mu, F[:, :d] - mu[:, None]


CASES = [("51", 9, True), ("51", 130, True), ("51", 259, True), ("51", 64, False), ("51", 200, False), ("51", 0, True),
         ("offset", 130, True), ("two_corners", 130, True)]


@pytest.mark.parametrize("grid,N,multi", CASES)
def test_identity_normals_reproduce_the_oracle_covariance(golden_dir, grid, N, multi):
    import torch
    from mfgp_coverage_b200._coverage import CoverageGrid
    from mfgp_coverage_b200.gaussian_process import MFGP, SFGP
    if grid == "offset":                      # non-square, off the unit square: catches x / y mix-ups
        ux, uy = np.linspace(-0.5, 1.0, 40), np.linspace(0.5, 1.5, 57)
    else:
        ux = uy = np.linspace(0.0, 1.0, 51)
    xy = _tensor(ux, uy)
    hyp, raw = (synth.MF_HYP if multi else synth.SF_HYP), False
    if grid == "two_corners":
        hyp, raw = np.load(os.path.join(golden_dir, "inputs_two_corners.npz"))["mf_hyp"], True
    if N:
        data = synth.training_set(xy, synth.truth_function(xy), N, multi=multi)
        p, m = _models(hyp, *data, raw_means=raw)
    else:
        e2, e1 = np.empty((0, 2)), np.empty((0, 1))
        data = (e2, e1, e2, e1)
        m = MFGP(*data, 1, 1) if multi else SFGP(e2, e1, 1)
        m.hyp = hyp
        p = ogp.GPParams.from_hyp(hyp)
    g = CoverageGrid(xy)
    mu, A = _identity_draws(m, g)
    cov = torch.mm(A, A.T).cpu().numpy()
    _, C_o = ogc.posterior_cov(p, xy, *data)
    assert np.max(np.abs(cov - C_o)) <= TOL * p.k0
    mu_p = m.predict(xy)[0][:, 0]
    assert np.max(np.abs(mu.cpu().numpy() - mu_p)) <= TOL * max(1.0, np.max(np.abs(mu_p)))


@pytest.mark.parametrize("N,multi", [(130, True), (200, False)])
def test_draws_match_the_oracle_at_equal_normals(N, multi):
    """The product's own node roots into the dense restatement: equal draws for the same random normals, so the normals' rows
    are consumed in the documented layout (a permutation of them would leave the covariance unchanged)."""
    import torch
    from mfgp_coverage_b200._coverage import CoverageGrid
    ux, uy = np.linspace(-0.5, 1.0, 40), np.linspace(0.5, 1.5, 57)
    xy = _tensor(ux, uy)
    data = synth.training_set(xy, synth.truth_function(xy), N, multi=multi)
    p, m = _models(synth.MF_HYP if multi else synth.SF_HYP, *data)
    g = CoverageGrid(xy)
    d = m.grid_sample_dim(g)
    plan = m.engine._grid_sample_plan(g.axes)
    Q = tuple(plan["Q"][k].cpu().numpy() if k in plan["Q"] else None for k in ("Lx", "Ly", "Hx", "Hy"))
    E = np.random.default_rng(3).standard_normal((d, 7))
    F = m.sample_posterior_grid_device(g, _dev(E)).cpu().numpy()
    mean, A = osg.pathwise_map(p, ux, uy, *data, plan["box"], plan["orders"], Q)
    F_o = mean[:, None] + A @ E
    assert np.max(np.abs(F - F_o)) <= TOL * max(1.0, np.max(np.abs(F_o)))
    torch.cuda.synchronize()


def test_c4_column_slices_reproduce_predict_cov():
    """1024 x 1024 grid, N = 4096: columns [0, 2) and [512, 514) with E = [I_d | 0] (d ~ 6000) against the dense joint
    covariance of those 4096 points, and the mean column against predict."""
    import torch
    from mfgp_coverage_b200._coverage import CoverageGrid
    xy = synth.grid(1024)
    f = synth.truth_function(xy)
    p, m = _models(synth.MF_HYP, *synth.training_set(xy, f, 4096))
    g = CoverageGrid(xy)
    d = m.grid_sample_dim(g)
    E = torch.zeros((d, d + 1), dtype=torch.float64, device="cuda")
    E[:, :d] = torch.eye(d, dtype=torch.float64, device="cuda")
    As, mus, rows = [], [], []
    for ix0 in (0, 512):
        F = m.sample_posterior_grid_device(g, E, ix0=ix0, ncols=2)
        mus.append(F[:, d].clone())
        As.append(F[:, :d] - mus[-1][:, None])
        rows.append(np.arange(ix0 * 1024, (ix0 + 2) * 1024))
        del F
    del E
    A = torch.cat(As)
    del As
    cov = torch.mm(A, A.T)
    del A
    rows = np.concatenate(rows)
    _, C = m.predict_cov_device(_dev(xy[rows]))
    assert float((cov - C).abs().max()) <= TOL * p.k0
    mu_p = m.predict(xy)[0][rows, 0]
    assert np.max(np.abs(torch.cat(mus).cpu().numpy() - mu_p)) <= TOL
    torch.cuda.empty_cache()


def test_slices_and_repeats_give_the_same_bits():
    import torch
    from mfgp_coverage_b200._coverage import CoverageGrid
    xy = synth.grid(51)
    p, m = _models(synth.MF_HYP, *synth.training_set(xy, synth.truth_function(xy), 130))
    g = CoverageGrid(xy)
    d = m.grid_sample_dim(g)
    E = torch.from_numpy(np.random.default_rng(1).standard_normal((d, 70))).cuda()
    F = m.sample_posterior_grid_device(g, E)
    assert torch.equal(F, m.sample_posterior_grid_device(g, E))
    parts = [m.sample_posterior_grid_device(g, E, ix0=a, ncols=b - a) for a, b in ((0, 20), (20, 21), (21, 51))]
    assert torch.equal(torch.cat(parts), F)
    out = torch.full((51 * 51, 72), np.nan, dtype=torch.float64, device="cuda")
    m.sample_posterior_grid_device(g, E, out=out[:, :70])
    assert torch.equal(out[:, :70], F) and bool(torch.isnan(out[:, 70:]).all())
    H = m.sample_posterior_grid(xy, n_samples=5, rng=np.random.default_rng(9))
    E5 = np.random.default_rng(9).standard_normal((d, 5))
    assert np.array_equal(H, m.sample_posterior_grid_device(g, _dev(E5)).cpu().numpy())
    assert not np.array_equal(H, m.sample_posterior_grid(xy, n_samples=5, rng=np.random.default_rng(10)))


@pytest.mark.parametrize("ny", [2, 63, 64, 65, 1024])
def test_eval_kernel_matches_numpy(ny):
    """F = mean + Uy C_s^T Ux through the C-ABI, canaries around F and in its padding columns; odd ldf or a misaligned F is
    rejected without writing anything."""
    import torch
    from mfgp_coverage_b200 import _native as nat
    from oracle.factored import cheb_basis
    lib = nat.lib()
    st = nat.stream_ptr()
    rng = np.random.default_rng(ny)
    nx, ix0, ncols, rx, ry, kpad = 5, 1, 3, 13, 12, 16
    box = (-1.0, 2.0, 0.5, 1.5)
    ux, uy = np.sort(rng.uniform(-1.0, 2.0, nx)), np.sort(rng.uniform(0.5, 1.5, ny))
    Ux, Uy = cheb_basis(ux[ix0:ix0 + ncols], box[0], box[1], rx), cheb_basis(uy, box[2], box[3], ry)
    ux_d, uy_d = _dev(ux), _dev(uy)
    rows, pad, mean = ncols * ny, 64, 0.75
    for S in (1, 2, 63, 64, 65, 130):
        C_h = rng.standard_normal((S, ry, kpad))
        C = _dev(C_h)
        ldf = S + (S & 1) + 4
        work = torch.empty(int(lib.mfgp_grid_sample_eval_workspace_bytes(ncols, ny, rx, ry, S)) // 8 + 1, dtype=torch.float64,
                           device="cuda")
        buf = torch.full((2 * pad + rows * ldf,), CANARY, dtype=torch.float64, device="cuda")
        F = buf[pad:pad + rows * ldf]

        def call(Fp, ld):
            return lib.mfgp_grid_sample_eval(nat.ptr(ux_d), nx, nat.ptr(uy_d), ny, ix0, ncols, *box, rx, ry, nat.ptr(C), S, mean,
                                             nat.ptr(Fp), ld, nat.ptr(work), work.numel() * 8, st)
        assert call(F, ldf) == nat.MFGP_OK
        b = buf.cpu().numpy()
        assert np.all(b[:pad] == CANARY) and np.all(b[pad + rows * ldf:] == CANARY), S
        inner = b[pad:pad + rows * ldf].reshape(rows, ldf)
        assert np.all(inner[:, S:] == CANARY), S
        ref = mean + np.einsum("ik,slk,jl->ijs", Ux, C_h[:, :, :rx], Uy).reshape(rows, S)
        bound = 1e-12 * (mean + np.einsum("ik,slk,jl->ijs", np.abs(Ux), np.abs(C_h[:, :, :rx]), np.abs(Uy)).reshape(rows, S))
        assert np.all(np.abs(inner[:, :S] - ref) <= bound), S
        snapshot = buf.clone()
        assert call(F, ldf + 1) == nat.MFGP_ERR_INVALID
        assert call(buf[pad + 1:], ldf) == nat.MFGP_ERR_INVALID
        assert call(F, S - 1 if S > 2 else -2) == nat.MFGP_ERR_INVALID
        torch.cuda.synchronize()
        assert torch.equal(buf, snapshot)


def test_argument_errors(monkeypatch):
    import torch
    from mfgp_coverage_b200._coverage import CoverageGrid
    from mfgp_coverage_b200.gaussian_process import SFGP
    xy = synth.grid(40)
    p, m = _models(synth.MF_HYP, *synth.training_set(xy, synth.truth_function(xy), 60))
    with pytest.raises(ValueError):
        m.sample_posterior_grid(np.random.default_rng(0).random((1600, 2)))
    with pytest.raises(ValueError):
        m.sample_posterior_grid(xy, n_samples=0)
    g = CoverageGrid(xy)
    d = m.grid_sample_dim(g)
    for E in (torch.zeros((d + 1, 3), dtype=torch.float64, device="cuda"), torch.zeros((d, 3), dtype=torch.float32, device="cuda"),
              torch.zeros((d, 0), dtype=torch.float64, device="cuda"), torch.zeros((d, 3), dtype=torch.float64)):
        with pytest.raises(ValueError):
            m.sample_posterior_grid_device(g, E)
    E = torch.zeros((d, 3), dtype=torch.float64, device="cuda")
    for out in (torch.empty((1600, 4), dtype=torch.float64, device="cuda"),
                torch.empty((1600, 5), dtype=torch.float64, device="cuda")[:, :3],
                torch.empty((3, 1600), dtype=torch.float64, device="cuda").T):
        with pytest.raises(ValueError):
            m.sample_posterior_grid_device(g, E, out=out)
    for ix0, ncols in ((-1, 2), (39, 2), (0, 0)):
        with pytest.raises(ValueError):
            m.sample_posterior_grid_device(g, E, ix0=ix0, ncols=ncols)
    # too short a length scale for 64 Chebyshev terms over the box
    short = SFGP(xy[:10], np.zeros((10, 1)), 1)
    short.hyp = np.array([0.0, 0.0, np.log(0.004), np.log(0.01)])
    short.updt_info(xy[:10], np.zeros((10, 1)))
    with pytest.raises(ValueError):
        short.sample_posterior_grid(xy)
    # memory: MemoryError before anything is allocated
    big = CoverageGrid(synth.grid(512))
    d = m.grid_sample_dim(big)
    E = torch.zeros((d, 64), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    total = torch.cuda.mem_get_info()[1]
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda *a, **k: (1 << 20, total))
    monkeypatch.setattr(torch.cuda, "memory_reserved", lambda *a, **k: 0)
    before = torch.cuda.memory_allocated()
    with pytest.raises(MemoryError):
        m.sample_posterior_grid_device(big, E)
    assert torch.cuda.memory_allocated() == before


def test_non_spd_training_covariance_raises_linalgerror():
    from mfgp_coverage_b200.gaussian_process import SFGP, evaluate_hyp
    X = np.array([[0.1, 0.1], [0.4, 0.2], [0.5, 0.5]])
    m = SFGP(X, np.zeros((3, 1)), 1)
    m.hyp = synth.SF_HYP
    m.params = lambda: dict(evaluate_hyp(synth.SF_HYP), noise_H=-1.0)    # diagonal = scale - 1 < 0: indefinite on purpose
    m.updt_info(X, np.zeros((3, 1)))
    with pytest.raises(np.linalg.LinAlgError):
        m.sample_posterior_grid(synth.grid(9), n_samples=2, rng=np.random.default_rng(0))
