"""GPU parity of the incremental path (SURVEY.md section 8f rank 1): bordered Cholesky append (mfgp_cholesky_append) +
incremental posterior (mfgp_posterior[_grid]_update) against the oracle's refit-from-scratch, which is what the
reference does every iteration (gaussian_process.py:266-268, :540-542)."""
import random

import numpy as np
import pytest
import torch
from scipy.linalg import solve_triangular

from oracle import algorithms as oalg
from oracle import gp as ogp
from tests import synth
from tests.test_gpu_algorithms import _agent_array, _compare

pytestmark = pytest.mark.gpu
TOL = 1e-9


def _oracle(hyp, X_L, y_L, X_H, y_H, xy):
    om = ogp.Model(ogp.GPParams.from_hyp(hyp), X_L, y_L, X_H, y_H)
    om.updt_info()
    return om, om.predict(xy)


def _check_model(m, om, p, mu, var, mu_o, var_o):
    """Posterior, L, z = L^-1 (y - mean) and W = L^-1 (all rows up to N = 2048, a seeded sample of 256 above) of the
    device model against the oracle's refit."""
    assert np.max(np.abs(var - var_o)) <= TOL * p.k0
    assert np.max(np.abs(mu - mu_o)) <= TOL * max(1.0, np.max(np.abs(mu_o)))
    L = m.factor()
    assert np.max(np.abs(L - om.L)) <= 1e-10 * np.max(np.abs(om.L))
    N = om.L.shape[0]
    e = m.engine
    e.ensure_factor()
    zref = solve_triangular(om.L, ogp.centered_y(om.p, om.y_L, om.y_H)[:, 0], lower=True)
    assert np.max(np.abs(e.z[:N].cpu().numpy() - zref)) <= TOL * max(1.0, np.max(np.abs(zref)))
    rows = np.arange(N) if N <= 2048 else np.sort(np.random.default_rng(N).choice(N, 256, replace=False))
    W = torch.tril(e.W[:N, :N]).cpu().numpy()[rows]
    assert np.max(np.abs(W @ om.L - np.eye(N)[rows])) <= 1e-9


@pytest.mark.parametrize("n,N0,adds,multi,separable", [
    (40, 30, [3, 0, 5, 1, 40, 7], True, True),         # inside one 64-block, across the 64 boundary, empty appends
    (40, 128, [64, 64, 1], True, False),               # block-aligned starts, general (non-separable) posterior path
    (48, 500, [8, 8, 70, 130], True, True),            # across the 512-row block of the posterior kernel, multi-block appends
    (40, 20, [5, 60, 9], False, True),                 # single fidelity
    (32, 120, [200], True, True),                      # one large append spanning several 64-blocks
    (64, 2100, [1, 63, 130], True, True),              # past 2048 rows (TMA form of the fit), capacity 2112 -> 3200
    (72, 4096, [64], True, True),                      # a c4 model taking its first samples: capacity 4096 -> 6144
])
def test_append_and_incremental_posterior_match_refit(n, N0, adds, multi, separable):
    """Past 2048 rows the split-K products of the append run 16-way, W is checked on sampled rows and the posterior on a
    seeded subset of the grid; the grown model is then refactored from scratch through the fused path (mfgp_cholesky_solve_gram
    on ld = capacity) and checked against the oracle as well."""
    from mfgp_coverage_b200 import simulator as sim
    from mfgp_coverage_b200._coverage import CoverageGrid
    xy = synth.grid(n)
    sub = np.arange(xy.shape[0]) if xy.shape[0] <= 2500 else np.sort(np.random.default_rng(n).choice(xy.shape[0], 512, replace=False))
    f = synth.truth_function(xy)
    total = N0 + sum(adds)
    X_L, y_L, X_H, y_H = synth.training_set(xy, f, total + (total // 3 if multi else 0), multi=multi)
    X_H, y_H = X_H[:total - X_L.shape[0]] if multi else X_H[:total], y_H[:total - X_L.shape[0]] if multi else y_H[:total]
    hyp = synth.MF_HYP if multi else synth.SF_HYP
    nh0 = N0 - X_L.shape[0]
    assert nh0 > 0
    if multi:
        m = sim.init_MFGP(hyp, np.column_stack((X_L, y_L)))
        m.updt_info(X_L, y_L, X_H[:nh0], y_H[:nh0])
    else:
        m = sim.init_SFGP(hyp, np.empty((0, 3)))
        m.updt_info(X_H[:nh0], y_H[:nh0])
    m.incremental = True
    m.use_separable = separable
    grid = CoverageGrid(xy)
    mu = torch.empty(grid.G, dtype=torch.float64, device=grid.device)
    var = torch.empty(grid.G, dtype=torch.float64, device=grid.device)
    m.predict_device(grid.xy, mu, var, grid=grid)
    p = ogp.GPParams.from_hyp(hyp)
    nh = nh0
    launches = []
    from mfgp_coverage_b200 import _native as nat
    for k in adds:
        l0 = nat.lib().mfgp_launch_count()
        (m.updt_hifi if multi else m.updt)(X_H[nh:nh + k], y_H[nh:nh + k])
        nh += k
        m.predict_device(grid.xy, mu, var, grid=grid)
        launches.append(nat.lib().mfgp_launch_count() - l0)
        om, (mu_o, var_o) = _oracle(hyp, X_L, y_L, X_H[:nh], y_H[:nh], xy[sub])
        _check_model(m, om, p, mu.cpu().numpy()[sub], var.cpu().numpy()[sub], mu_o, var_o)
    # an empty append costs nothing on the device (the reference refits even then)
    for k, nl in zip(adds, launches):
        if k == 0:
            assert nl == 0
    # a from-scratch evaluation of the same model agrees with the incrementally maintained one
    mu2, var2 = m.predict(xy)
    assert np.max(np.abs(var2 - var.cpu().numpy())) <= 1e-11 * p.k0
    assert np.max(np.abs(mu2[:, 0] - mu.cpu().numpy())) <= 1e-11 * max(1.0, np.max(np.abs(mu2)))
    if N0 > 2048:
        e = m.engine
        e.defer_fit = True
        e.refactor(check=False)
        mu3, var3 = torch.empty_like(mu), torch.empty_like(var)
        m.predict_device(grid.xy, mu3, var3, grid=grid)
        assert e._w_partial and e.cap > e.npad          # the fused fit ran, on leading dimension cap
        _check_model(m, om, p, mu3.cpu().numpy()[sub], var3.cpu().numpy()[sub], mu_o, var_o)


def test_incremental_survives_capacity_growth_and_deepcopy():
    import copy
    from mfgp_coverage_b200 import simulator as sim
    from mfgp_coverage_b200._coverage import CoverageGrid
    xy = synth.grid(36)
    f = synth.truth_function(xy)
    X_L, y_L, X_H, y_H = synth.training_set(xy, f, 400)
    m = sim.init_MFGP(synth.MF_HYP, np.column_stack((X_L, y_L)))
    m.updt_info(X_L, y_L, X_H[:10], y_H[:10])
    m.incremental = True
    grid = CoverageGrid(xy)
    mu = torch.empty(grid.G, dtype=torch.float64, device=grid.device)
    var = torch.empty(grid.G, dtype=torch.float64, device=grid.device)
    m.predict_device(grid.xy, mu, var, grid=grid)
    cap0 = m.engine.cap
    nh = 10
    while m.engine.cap == cap0:                       # append until the device buffers had to be reallocated
        m.updt_hifi(X_H[nh:nh + 37], y_H[nh:nh + 37])
        nh += 37
        m.predict_device(grid.xy, mu, var, grid=grid)
    twin = copy.deepcopy(m)                           # simulator.py:339 deep-copies the model
    assert twin.incremental
    m.updt_hifi(X_H[nh:nh + 5], y_H[nh:nh + 5])
    m.predict_device(grid.xy, mu, var, grid=grid)
    p = ogp.GPParams.from_hyp(synth.MF_HYP)
    _, (mu_o, var_o) = _oracle(synth.MF_HYP, X_L, y_L, X_H[:nh + 5], y_H[:nh + 5], xy)
    assert np.max(np.abs(var.cpu().numpy() - var_o)) <= TOL * p.k0
    assert np.max(np.abs(mu.cpu().numpy() - mu_o)) <= TOL * max(1.0, np.max(np.abs(mu_o)))
    mu_t, var_t = twin.predict(xy)                    # the copy still holds the model as of the copy
    _, (mu_c, var_c) = _oracle(synth.MF_HYP, X_L, y_L, X_H[:nh], y_H[:nh], xy)
    assert np.max(np.abs(var_t - var_c)) <= TOL * p.k0 and np.max(np.abs(mu_t[:, 0] - mu_c)) <= TOL * max(1.0, np.max(np.abs(mu_c)))


def test_append_reports_non_spd():
    """A non-positive pivot in a bordered block surfaces as LinAlgError, like np.linalg.cholesky (gaussian_process.py:254)."""
    from mfgp_coverage_b200 import simulator as sim
    xy = synth.grid(12)
    m = sim.init_SFGP(synth.SF_HYP, np.empty((0, 3)))
    e = m.engine
    e.defer_fit = e.lazy_check = False       # engine-level test: the status is read back by every call (MFGP_EAGER_FIT behaviour)
    m.updt_info(xy[[3, 50, 77]], np.ones((3, 1)))
    m.incremental = True
    bad = dict(e.params)
    bad["noise_H"] = -1.0          # new diagonal entries k(0) + noise < 0: the Schur complement of the border is not SPD
    e.set_params(bad)
    with pytest.raises(np.linalg.LinAlgError):
        e.append_hifi(xy[[5, 9]], np.ones((2, 1)))


@pytest.mark.parametrize("algo,n,A,T,multi", [("todescato", 40, 6, 12, True), ("periodic", 32, 5, 12, False),
                                              ("choi", 36, 4, 24, True)])
def test_incremental_runs_vs_oracle_loops(algo, n, A, T, multi, monkeypatch):
    """Whole control loops with the incremental path switched on agree with the oracle loops (refit every iteration)."""
    from mfgp_coverage_b200 import simulator as sim
    monkeypatch.setattr(sim, "INCREMENTAL", True)
    xy = synth.grid(n)
    truth_arr = np.column_stack((xy, synth.truth_function(xy)))
    hyp = synth.MF_HYP if multi else synth.SF_HYP
    lat_xy = np.random.default_rng(99).random((9, 2))
    near = np.argmin(((xy[None, :, :] - lat_xy[:, None, :]) ** 2).sum(axis=2), axis=1)
    prior_arr = np.column_stack((lat_xy, 0.8 * truth_arr[near, 2] + 0.02))
    seed = 21
    pos0 = synth.agents(A, seed)
    lo, ao, so = getattr(oalg, algo)(0, T, A, pos0.copy(), truth_arr, 0.1, prior_arr, hyp, random.Random(seed),
                                     np.random.default_rng(seed))
    lg, ag, sg = getattr(sim, algo)(algo, 0, T, A, pos0.copy(), truth_arr, 0.1, prior_arr, hyp, False, None, True,
                                    rng=random.Random(seed), noise_rng=np.random.default_rng(seed))
    to_s = lambda s: np.array([[float(r["Iteration"]), float(r["Agent"]), float(r["X"]), float(r["Y"]), float(r["Sample"])]
                               for r in s]).reshape(-1, 5)
    _compare(np.array([r["Loss"] for r in lg]), _agent_array(ag, len(lg), A), to_s(sg),
             np.array([r["Loss"] for r in lo]), _agent_array(ao, len(lo), A), to_s(so), truth_arr)


@pytest.mark.parametrize("algo,n,A,T,multi", [("todescato", 40, 6, 12, True), ("periodic", 32, 5, 12, False)])
def test_throughput_mode_runs_vs_oracle_loops(algo, n, A, T, multi, monkeypatch):
    """Throughput mode (config c5): incremental factor + posterior AND device-built Voronoi cells + device finishing --
    no host Qhull, one D2H per iteration -- still reproduces the oracle loops on tie-free inputs."""
    from mfgp_coverage_b200 import simulator as sim
    monkeypatch.setattr(sim, "INCREMENTAL", True)
    monkeypatch.setattr(sim, "VORONOI", "clip")
    xy = synth.grid(n)
    truth_arr = np.column_stack((xy, synth.truth_function(xy)))
    hyp = synth.MF_HYP if multi else synth.SF_HYP
    lat_xy = np.random.default_rng(99).random((9, 2))
    near = np.argmin(((xy[None, :, :] - lat_xy[:, None, :]) ** 2).sum(axis=2), axis=1)
    prior_arr = np.column_stack((lat_xy, 0.8 * truth_arr[near, 2] + 0.02))
    seed = 21
    pos0 = synth.agents(A, seed)
    lo, ao, so = getattr(oalg, algo)(0, T, A, pos0.copy(), truth_arr, 0.1, prior_arr, hyp, random.Random(seed),
                                     np.random.default_rng(seed))
    lg, ag, sg = getattr(sim, algo)(algo, 0, T, A, pos0.copy(), truth_arr, 0.1, prior_arr, hyp, False, None, True,
                                    rng=random.Random(seed), noise_rng=np.random.default_rng(seed))
    to_s = lambda s: np.array([[float(r["Iteration"]), float(r["Agent"]), float(r["X"]), float(r["Y"]), float(r["Sample"])]
                               for r in s]).reshape(-1, 5)
    _compare(np.array([r["Loss"] for r in lg]), _agent_array(ag, len(lg), A), to_s(sg),
             np.array([r["Loss"] for r in lo]), _agent_array(ao, len(lo), A), to_s(so), truth_arr, replay_ties=False)
