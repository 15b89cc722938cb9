"""CPU: the oracle's full posterior covariance (oracle.gp_cov.posterior_cov) against its diagonal-only posterior, whose
variance is pinned to the live reference's np.diag(cov) by the stored ref_gp_cases.npz, and its own structure: symmetry,
cross blocks, the reference's general solves."""
import os

import numpy as np
import pytest

from oracle import gp as ogp
from oracle import gp_cov as ogc
from tests import synth


def _cases(golden_dir):
    g = np.load(os.path.join(golden_dir, "ref_gp_cases.npz"), allow_pickle=False)
    for k in range(int(g["ncases"])):
        yield (g["xs"], ogp.GPParams.from_hyp(g[f"c{k}_hyp"]), g[f"c{k}_XL"], g[f"c{k}_yL"], g[f"c{k}_XH"], g[f"c{k}_yH"],
               g[f"c{k}_var"], g[f"c{k}_mu"])


def test_diagonal_is_the_variance_on_the_reference_cases(golden_dir):
    seen = set()
    for xs, p, XL, yL, XH, yH, var_ref, mu_ref in _cases(golden_dir):
        pts = xs[::7]                      # 372 of the 2601 points: keeps the G x G matrix small
        mu_d, var_d = ogp.posterior(p, pts, XL, yL, XH, yH)
        mu_c, cov = ogc.posterior_cov(p, pts, XL, yL, XH, yH)
        assert cov.shape == (pts.shape[0], pts.shape[0])
        assert np.max(np.abs(np.diag(cov) - var_d)) <= 1e-13 * p.k0
        assert np.max(np.abs(np.diag(cov) - var_ref[::7])) <= 1e-12 * p.k0
        assert np.max(np.abs(mu_c - mu_d)) <= 1e-12 * max(1.0, np.max(np.abs(mu_d)))
        seen.add((bool(p.multi), XL.shape[0] + XH.shape[0] > 0))
    assert (True, True) in seen and (False, True) in seen


@pytest.mark.parametrize("multi", [True, False])
def test_empty_model_is_the_prior_covariance(multi):
    hyp = synth.MF_HYP if multi else synth.SF_HYP
    p = ogp.GPParams.from_hyp(hyp)
    pts = synth.grid(13)
    e = np.empty((0, 2)), np.empty((0, 1))
    mu, cov = ogc.posterior_cov(p, pts, e[0], e[1], e[0], e[1])
    mu_d, var_d = ogp.posterior(p, pts, e[0], e[1], e[0], e[1])
    assert np.array_equal(mu, mu_d) and np.all(mu == p.mean_H)
    assert np.max(np.abs(np.diag(cov) - var_d)) <= 1e-13 * p.k0
    assert np.array_equal(cov, ogc.prior_cov(p, pts, pts))
    assert np.max(np.abs(cov - cov.T)) == 0.0


@pytest.mark.parametrize("multi,N", [(True, 130), (False, 90)])
def test_symmetric_and_cross_blocks(multi, N):
    xy = synth.grid(24)
    f = synth.truth_function(xy)
    X_L, y_L, X_H, y_H = synth.training_set(xy, f, N, multi=multi)
    p = ogp.GPParams.from_hyp(synth.MF_HYP if multi else synth.SF_HYP)
    pts = np.vstack((xy[::5], np.random.default_rng(5).random((40, 2))))
    _, cov = ogc.posterior_cov(p, pts, X_L, y_L, X_H, y_H)
    assert np.max(np.abs(cov - cov.T)) <= 1e-14 * p.k0
    a, b = slice(0, 70), slice(55, pts.shape[0])
    mu_a, cross = ogc.posterior_cov(p, pts[a], X_L, y_L, X_H, y_H, X_b=pts[b])
    assert cross.shape == (70, pts.shape[0] - 55)
    assert np.max(np.abs(cross - cov[a, b])) <= 1e-13 * p.k0
    _, exact = ogc.posterior_cov(p, pts[a], X_L, y_L, X_H, y_H, X_b=pts[b], exact_solve=True)
    assert np.max(np.abs(exact - cross)) <= 1e-11 * p.k0
    mu_d, _ = ogp.posterior(p, pts[a], X_L, y_L, X_H, y_H)
    assert np.max(np.abs(mu_a - mu_d)) <= 1e-12 * max(1.0, np.max(np.abs(mu_d)))
