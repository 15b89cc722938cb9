"""CPU: the oracle's joint posterior draws (oracle.gp_sample.posterior_samples): its factor reproduces C + jitter I, and
seeded draws have the posterior mean and covariance within bounds set by their standard errors."""
import numpy as np

from oracle import gp as ogp
from oracle import gp_cov as ogc
from oracle import gp_sample as ogs
from tests import synth


def _case(N=40, n_pts=30, seed=5):
    xy = synth.grid(20)
    f = synth.truth_function(xy)
    data = synth.training_set(xy, f, N)
    p = ogp.GPParams.from_hyp(synth.MF_HYP)
    pts = np.random.default_rng(seed).random((n_pts, 2))
    return p, pts, data


def test_factor_reproduces_the_jittered_covariance():
    p, pts, data = _case()
    tau = 1e-8 * p.k0
    mu, C = ogc.posterior_cov(p, pts, *data)
    G = pts.shape[0]
    F = ogs.posterior_samples(p, pts, *data, np.eye(G), tau)      # E = I: F - mu = L
    L = F - mu[:, None]
    assert np.array_equal(np.triu(L, 1), np.zeros((G, G)))
    assert np.max(np.abs(L @ L.T - (C + tau * np.eye(G)))) <= 1e-13 * p.k0


def test_draws_have_the_posterior_mean_and_covariance():
    p, pts, data = _case()
    tau = 1e-8 * p.k0
    mu, C = ogc.posterior_cov(p, pts, *data)
    Ct = C + tau * np.eye(C.shape[0])
    n = 200_000
    E = np.random.default_rng(2024).standard_normal((pts.shape[0], n))
    F = ogs.posterior_samples(p, pts, *data, E, tau)
    d = np.diag(Ct)
    # sample mean: standard error sqrt(C_ii / n); sample covariance: sqrt((C_ii C_jj + C_ij^2) / n) for Gaussian draws
    assert np.all(np.abs(F.mean(axis=1) - mu) <= 6.0 * np.sqrt(d / n))
    S = np.cov(F)
    assert np.all(np.abs(S - Ct) <= 6.0 * np.sqrt((np.outer(d, d) + Ct ** 2) / n))
    # the bounds are tight enough to see a wrong factor: the transpose (upper) factor gives the wrong covariance
    wrong = mu[:, None] + np.linalg.cholesky(Ct).T @ E
    assert not np.all(np.abs(np.cov(wrong) - Ct) <= 6.0 * np.sqrt((np.outer(d, d) + Ct ** 2) / n))
