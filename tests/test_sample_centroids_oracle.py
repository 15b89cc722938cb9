"""CPU: the coefficient-space route to the centroids of posterior draws (oracle.sample_centroids).  The draws' coefficient
matrices reproduce the dense pathwise draws; the partials <C'_s, Mom_i^w> equal the dense per-draw partials of the same draws
within 1e-12 of the sum of their terms' magnitudes, and the centroids equal compute_centroids draw by draw -- for MF, SF and
no data, and on a grid with points on the bisectors.  Thompson sampling's move rule, in the oracle and in the product."""
import numpy as np
import pytest

from oracle import coverage as ocov
from oracle import gp as ogp
from oracle import gp_sample_grid as osg
from oracle import sample_centroids as osc
from tests import synth


def orders_of(p, box):
    from mfgp_coverage_b200._engine import chebyshev_order
    xlo, xhi, ylo, yhi = box
    o = [chebyshev_order(p.l_H, xlo, xhi, xlo, xhi), chebyshev_order(p.l_H, ylo, yhi, ylo, yhi)]
    if p.multi:
        o = [chebyshev_order(p.l_L, xlo, xhi, xlo, xhi), chebyshev_order(p.l_L, ylo, yhi, ylo, yhi)] + o
    else:
        o = [0, 0] + o
    assert all(r is not None for r in o)
    return tuple(o)


def _case(n, N, multi, seeds, S=5, seed=3):
    g = np.linspace(0.0, 1.0, n)
    xy = np.stack(np.meshgrid(g, g, indexing="ij"), axis=-1).reshape(-1, 2)
    p = ogp.GPParams.from_hyp(synth.MF_HYP if multi else synth.SF_HYP)
    if N:
        X_L, y_L, X_H, y_H = synth.training_set(xy, synth.truth_function(xy), N, multi=multi)
    else:
        X_L = X_H = np.empty((0, 2))
        y_L = y_H = np.empty((0, 1))
    box = osc.sample_box(g, g, np.vstack((X_L.reshape(-1, 2), X_H.reshape(-1, 2))))
    orders = orders_of(p, box)
    Q = osg.node_roots(p, box, orders)
    mean, A = osg.pathwise_map(p, g, g, X_L, y_L, X_H, y_H, box, orders, Q)
    E = np.random.default_rng(seed).standard_normal((A.shape[1], S))
    C = osc.draw_coefficients(p, X_L, y_L, X_H, y_H, box, orders, Q, E)
    return p, g, xy, box, orders, C, mean[:, None] + A @ E, seeds


BISECTOR_SEEDS = np.array([[0.25, 0.25], [0.75, 0.25], [0.25, 0.75], [0.75, 0.75], [0.5, 0.5]])


@pytest.mark.parametrize("n,N,multi,seeds", [(31, 60, True, "agents"), (31, 60, False, "agents"), (31, 0, True, "agents"),
                                             (31, 0, False, "agents"), (41, 40, True, "bisectors")])
def test_coefficient_partials_equal_the_dense_per_draw_partials(n, N, multi, seeds):
    p, g, xy, box, orders, C, F_path, _ = _case(n, N, multi, seeds)
    k0 = p.k0
    F = osc.evaluate(C, p.mean_H, g, g, box)
    assert np.max(np.abs(F - F_path)) <= 1e-9 * max(1.0, k0)       # the coefficients are the pathwise draws
    pts = synth.agents(8, 5) if seeds == "agents" else BISECTOR_SEEDS
    bbox = ocov.bounding_box_of(xy)
    vor = ocov.voronoi_bounded(pts, bbox)
    member = ocov.membership(vor, xy)
    if seeds == "bisectors":
        assert np.any(member.sum(axis=0) != 1)                      # points on bisectors: in 0 or several cells
    ry, kpad = C.shape[1], C.shape[2]
    mom = osc.moments(member, g, g, box, ry, kpad)
    cent_c = osc.coefficient_partials(mom, C, p.mean_H)
    cent_d, scale = osc.dense_partials(member, xy, F)
    assert np.array_equal(cent_c[..., 3], cent_d[..., 3])
    assert np.all(np.abs(cent_c[..., :3] - cent_d[..., :3]) <= 1e-12 * scale + 1e-300)
    areas = np.array([ocov.poly_area(v[:, 0], v[:, 1]) for v in (vor.cell_vertices(i) for i in range(len(pts)))])
    cen = osc.centroids_from_partials(cent_c, areas, *bbox)
    cen_d = osc.dense_centroids(vor, xy, F)
    assert np.max(np.abs(cen - cen_d)) <= 1e-9


def test_an_empty_cell_gives_nan():
    p, g, xy, box, orders, C, F, _ = _case(11, 0, False, "agents", S=2)
    member = np.zeros((2, xy.shape[0]), dtype=bool)
    member[0] = True
    mom = osc.moments(member, g, g, box, C.shape[1], C.shape[2])
    cen = osc.centroids_from_partials(osc.coefficient_partials(mom, C, p.mean_H), np.array([1.0, 1.0]), 0, 1, 0, 1)
    assert np.all(np.isfinite(cen[:, 0])) and np.all(np.isnan(cen[:, 1]))


def _snap_cases():
    ux = np.arange(9) * 0.125                     # binary fractions: the midpoints below are exact ties
    uy = np.arange(17) * 0.125 - 1.0
    pos = np.array([[0.375, 0.0], [0.5, 0.5], [0.875, -0.875], [0.125, 0.25]])
    targets = np.array([[0.52, 0.48],              # -> (0.5, 0.5)
                        [0.49, 0.52],              # the same grid point, taken by agent 0 -> nearest to its position
                        [np.nan, 0.3],             # NaN target -> nearest to its position
                        [0.1875, -0.0625]])        # exact midpoints on both axes -> the lower indices
    expect = np.array([[0.5, 0.5], [0.5, 0.5], [0.875, -0.875], [0.125, -0.125]])
    return ux, uy, pos, targets, expect


def test_oracle_snapping_rules():
    ux, uy, pos, targets, expect = _snap_cases()
    assert np.array_equal(osc.snap_to_grid(targets, pos, ux, uy), expect)


def test_product_snapping_equals_the_oracle():
    from mfgp_coverage_b200.simulator import snap_to_grid
    ux, uy, pos, targets, _ = _snap_cases()
    rng = np.random.default_rng(11)
    for _ in range(20):
        t = np.vstack((targets, rng.uniform(-0.2, 1.2, (6, 2)), np.round(rng.uniform(0, 1, (4, 2)) * 20) / 20 + 0.025))
        p = np.vstack((pos, rng.uniform(0, 1, (10, 2))))
        t[rng.integers(0, t.shape[0])] = np.nan
        assert np.array_equal(snap_to_grid(t, p, ux, uy), osc.snap_to_grid(t, p, ux, uy))
