"""CPU: the pathwise grid sampler's restatement (oracle.gp_sample_grid).  Its linear map A from the normals to the draws
has A A^T = the exact posterior covariance (oracle.gp_cov) and its offset is the posterior mean (oracle.gp); with no data
A A^T is the prior covariance; the node roots Q reproduce DCT K_nodes DCT^T."""
import os

import numpy as np
import pytest

from oracle import gp as ogp
from oracle import gp_cov as ogc
from oracle import gp_sample_grid as osg
from tests import synth


def _orders(p, box):
    from mfgp_coverage_b200._engine import chebyshev_order
    xlo, xhi, ylo, yhi = box
    o = [chebyshev_order(p.l_H, xlo, xhi, xlo, xhi), chebyshev_order(p.l_H, ylo, yhi, ylo, yhi)]
    if p.multi:
        o = [chebyshev_order(p.l_L, xlo, xhi, xlo, xhi), chebyshev_order(p.l_L, ylo, yhi, ylo, yhi)] + o
    else:
        o = [0, 0] + o
    assert all(r is not None for r in o)
    return tuple(o)


def _check(p, ux, uy, data, tol):
    X_L, y_L, X_H, y_H = data
    xy = np.stack(np.meshgrid(ux, uy, indexing="ij"), axis=-1).reshape(-1, 2)
    X = np.vstack((np.asarray(X_L).reshape(-1, 2), np.asarray(X_H).reshape(-1, 2)))
    pts = np.vstack((xy, X))
    box = (pts[:, 0].min(), pts[:, 0].max(), pts[:, 1].min(), pts[:, 1].max())
    orders = _orders(p, box)
    mean, A = osg.pathwise_map(p, ux, uy, X_L, y_L, X_H, y_H, box, orders, osg.node_roots(p, box, orders))
    N = X.shape[0]
    assert A.shape == (xy.shape[0], orders[0] * orders[1] + orders[2] * orders[3] + N)
    mu_o, C_o = ogc.posterior_cov(p, xy, X_L, y_L, X_H, y_H)
    assert np.max(np.abs(A @ A.T - C_o)) <= tol * p.k0
    if N:
        mu_d, _ = ogp.posterior(p, xy, X_L, y_L, X_H, y_H)
        assert np.max(np.abs(mean - mu_d)) <= 1e-9 * max(1.0, np.max(np.abs(mu_d)))
    else:
        assert np.all(mean == p.mean_H)


@pytest.mark.parametrize("n,N,multi", [(31, 9, True), (41, 130, True), (41, 259, True), (41, 200, False)])
def test_map_reproduces_the_posterior_covariance(n, N, multi):
    xy = synth.grid(n)
    data = synth.training_set(xy, synth.truth_function(xy), N, multi=multi)
    p = ogp.GPParams.from_hyp(synth.MF_HYP if multi else synth.SF_HYP)
    g = np.linspace(0, 1, n)
    _check(p, g, g, data, 1e-12)


def test_map_on_an_offset_non_square_grid():
    ux, uy = np.linspace(-0.5, 1.0, 23), np.linspace(0.5, 1.5, 31)
    xy = np.stack(np.meshgrid(ux, uy, indexing="ij"), axis=-1).reshape(-1, 2)
    data = synth.training_set(xy, synth.truth_function(xy), 60)
    _check(ogp.GPParams.from_hyp(synth.MF_HYP), ux, uy, data, 1e-12)


def test_map_with_the_near_zero_noise_two_corners_hyper_parameters(golden_dir):
    hyp = np.load(os.path.join(golden_dir, "inputs_two_corners.npz"))["mf_hyp"]
    p = ogp.GPParams.from_hyp(hyp, raw_means=True)
    g = np.linspace(0, 1, 31)
    xy = synth.grid(31)
    data = synth.training_set(xy, synth.truth_function(xy), 130)
    _check(p, g, g, data, 1e-9)


@pytest.mark.parametrize("multi", [True, False])
def test_without_data_the_map_is_the_prior(multi):
    p = ogp.GPParams.from_hyp(synth.MF_HYP if multi else synth.SF_HYP)
    g = np.linspace(0, 1, 25)
    e2, e1 = np.empty((0, 2)), np.empty((0, 1))
    _check(p, g, g, (e2, e1, e2, e1), 1e-12)


@pytest.mark.parametrize("length,r", [(0.58, 20), (0.2, 36), (0.05, 64)])
def test_node_root_reproduces_the_node_kernel_in_coefficient_space(length, r):
    Q = osg.node_root(length, -0.3, 1.7, r)
    D = osg.dct_matrix(r)
    K = osg.node_kernel(length, -0.3, 1.7, r)
    assert np.max(np.abs(Q @ Q.T - D @ K @ D.T)) <= 1e-13
