"""CPU: the term-by-term restatement of the factored posterior (oracle/factored.py) is the exact GP at the orders the engine's
planner picks, and is far from it at under-resolved orders -- which is what lets tests/test_gpu_factored_orders.py compare
the kernels with the restatement at orders where every term matters."""
import numpy as np
import pytest

from oracle import factored as ofac
from oracle import gp as ogp
from tests import synth


def _setup(multi, N, nx=40, ny=36, seed=3):
    gx, gy = np.linspace(0.0, 1.0, nx), np.linspace(0.0, 1.0, ny)
    xy = np.stack(np.meshgrid(gx, gy, indexing="ij"), axis=-1).reshape(-1, 2)
    X_L, y_L, X_H, y_H = synth.training_set(xy, synth.truth_function(xy), N, seed=seed, multi=multi)
    p = ogp.GPParams.from_hyp(synth.MF_HYP if multi else synth.SF_HYP)
    return gx, gy, xy, p, X_L, y_L, X_H, y_H


def _planner(p, X_L, X_H, box):
    """Orders and truncated layout as DeviceGP._cheb_orders picks them for the grid box (training hull plus its margin)."""
    from mfgp_coverage_b200._engine import chebyshev_envelope, chebyshev_order, chebyshev_truncation
    X = np.vstack((X_L.reshape(-1, 2), X_H.reshape(-1, 2)))
    xlo, xhi, ylo, yhi = box
    mx, my = 0.05 * (xhi - xlo), 0.05 * (yhi - ylo)
    hull = (min(X[:, 0].min(), xlo) - mx, max(X[:, 0].max(), xhi) + mx, min(X[:, 1].min(), ylo) - my, max(X[:, 1].max(), yhi) + my)
    ls = [("H", p.l_H)] + ([("L", p.l_L)] if p.multi else [])
    o, env = {}, []
    for name, l in ls:
        o["rx" + name] = chebyshev_order(l, xlo, xhi, hull[0], hull[1])
        o["ry" + name] = chebyshev_order(l, ylo, yhi, hull[2], hull[3])
        env.append((o["rx" + name], o["ry" + name], l))
    orders = (o.get("rxL", 0), o.get("ryL", 0), o["rxH"], o["ryH"])
    kp = ofac.round_up(max(orders[0], orders[2]), 4)
    parts = [(np.pad(chebyshev_envelope(l, xlo, xhi, hull[0], hull[1], rx), (0, kp - rx)),
              chebyshev_envelope(l, ylo, yhi, hull[2], hull[3], ry)) for rx, ry, l in env]
    return orders, chebyshev_truncation(parts, kp, max(orders[1], orders[3]))


@pytest.mark.parametrize("multi,truncated", [(True, False), (True, True), (False, False), (False, True)])
def test_restatement_is_the_exact_gp_at_converged_orders(multi, truncated):
    gx, gy, xy, p, X_L, y_L, X_H, y_H = _setup(multi, 300 if multi else 200)
    box = (0.0, 1.0, 0.0, 1.0)
    orders, kx = _planner(p, X_L, X_H, box)
    assert 16 <= max(orders) <= 40                          # the synth scales: the orders every engine test runs
    if truncated:
        assert kx.sum() < max(orders[1], orders[3]) * ofac.round_up(max(orders[0], orders[2]), 4)
    mu, var, q = ofac.posterior(p, X_L, y_L, X_H, y_H, gx, gy, 0, gx.size, orders, box, kx if truncated else None)
    mu_o, var_o = ogp.posterior(p, xy, X_L, y_L, X_H, y_H)
    assert np.max(np.abs(var - var_o)) <= 1e-12 * p.k0
    assert np.max(np.abs(mu - mu_o)) <= 1e-12 * max(1.0, np.max(np.abs(mu_o)))
    assert np.array_equal(p.k0 - q, var)


@pytest.mark.parametrize("multi,orders", [(True, (8, 8, 12, 4)), (True, (13, 20, 7, 12)), (False, (0, 0, 10, 8))])
def test_restatement_at_under_resolved_orders_is_not_the_exact_gp(multi, orders):
    """The GPU comparison is at 1e-11 k(0); an under-resolved expansion is orders of magnitude further from the exact GP, so
    the comparison there is against the expansion itself."""
    gx, gy, xy, p, X_L, y_L, X_H, y_H = _setup(multi, 240)
    mu, var, _ = ofac.posterior(p, X_L, y_L, X_H, y_H, gx, gy, 0, gx.size, orders, (0.0, 1.0, 0.0, 1.0))
    mu_o, var_o = ogp.posterior(p, xy, X_L, y_L, X_H, y_H)
    assert np.max(np.abs(var - var_o)) >= 1e-6 * p.k0
    assert np.max(np.abs(mu - mu_o)) >= 1e-6 * max(1.0, np.max(np.abs(mu_o)))


def test_chebyshev_tables_interpolate_at_the_nodes():
    """The DCT coefficients and the recurrence basis of the restatement reproduce the axis factor exactly at the r Chebyshev
    nodes of an off-centre interval (interpolation, whatever the order), and the truncated sum drops exactly the given term."""
    lo, hi, l, r = -0.3, 1.4, 0.07, 12
    u = np.array([-0.5, 0.2, 0.9, 1.6])
    nodes = 0.5 * (lo + hi) + 0.5 * (hi - lo) * np.cos(np.pi * (np.arange(r) + 0.5) / r)
    C = ofac.cheb_coef(u, lo, hi, 1.0 / l, r)
    T = ofac.cheb_basis(nodes, lo, hi, r)
    f = np.exp(-0.5 * ((nodes[:, None] - u[None, :]) / l) ** 2)
    assert np.max(np.abs(T @ C - f)) <= 1e-14
    p = ogp.GPParams.from_hyp(synth.SF_HYP)
    X_H = np.array([[0.1, 0.2], [0.7, 0.4]])
    full = ofac.factored_psi(p, np.empty((0, 2)), X_H, nodes, nodes[:5], 0, 3, (0, 0, 7, 8), (lo, hi, lo, hi))
    l, k = ofac.highest_term(p, (0, 0, 7, 8))
    assert (l, k) == (7, 6)
    cut = ofac.factored_psi(p, np.empty((0, 2)), X_H, nodes, nodes[:5], 0, 3, (0, 0, 7, 8), (lo, hi, lo, hi), drop=(l, k))
    Cx = ofac.cheb_coef(X_H[:, 0], lo, hi, 1.0 / p.l_H, 7)
    Cy = ofac.cheb_coef(X_H[:, 1], lo, hi, 1.0 / p.l_H, 8)
    term = p.s_H * np.einsum("x,y,n->xyn", ofac.cheb_basis(nodes[:3], lo, hi, 7)[:, k], ofac.cheb_basis(nodes[:5], lo, hi, 8)[:, l],
                             Cy[l] * Cx[k]).reshape(15, 2)
    assert np.max(np.abs((full - cut) - term)) <= 1e-15
