"""Oracle: joint posterior draws over a tensor-product grid by pathwise conditioning (numpy restatement; TEST
INFRASTRUCTURE).  Dense companion of csrc/gp_sample_grid.cu.

Matheron's rule: with f a prior draw and eps ~ N(0, diag(noise + jitter)),
    f_post(.) = mean_H + f(.) + k(., X) K^-1 (y - m - f(X) - eps)
is a draw from the posterior of the latent f_H.  The prior draw is, per kernel part P, the Chebyshev interpolant on `box` of
a draw g_P ~ N(0, s_P K_P,x (x) K_P,y) at the r_x x r_y tensor of Chebyshev nodes: in coefficient space
C_P = sqrt(s_P) Qx_P Xi_P Qy_P^T with Q = DCT K_nodes^(1/2) (node_root).  The parts combine as the AR1 model:
f_L = g_L, f_H = rho f_L + g_H; lofi training rows see f_L, hifi rows and the grid see f_H.

Here everything is a dense linear map of the normals E[d] (d = rxL ryL + rxH ryH + N, layout of include/mfgp_b200.h:
mfgp_grid_sample_coef): F = mean + A E, with the EXACT cross-covariance k(., X) and training covariance K (oracle.gp), not
the Chebyshev re-expansion the library uses for the update term.
"""
import numpy as np
from scipy.linalg import cho_solve

from . import gp as ogp
from .factored import cheb_basis


def dct_matrix(r):
    """D[k][j] = (k ? 2 : 1) / r cos(pi k (j + 1/2) / r): node values -> Chebyshev coefficients (cheb_coef_kernel)."""
    j = np.arange(r) + 0.5
    return np.cos(np.pi * np.outer(np.arange(r), j) / r) * np.where(np.arange(r) == 0, 1.0, 2.0)[:, None] / r


def node_kernel(length, lo, hi, r):
    """exp(-0.5 ((node_i - node_j) / l)^2) at the r Chebyshev nodes mid + half cos(pi (j + 1/2) / r) of [lo, hi]."""
    mid, half = 0.5 * (lo + hi), 0.5 * (hi - lo)
    node = mid + half * np.cos(np.pi * (np.arange(r) + 0.5) / r)
    d = (node[:, None] - node[None, :]) / length
    return np.exp(-0.5 * d * d)


def node_root(length, lo, hi, r):
    """Q[r, r] = DCT V sqrt(max(Lambda, 0)) V^T: the coefficients of the interpolant of a unit-scale prior draw at the nodes
    are Q xi, xi ~ N(0, I)."""
    lam, V = np.linalg.eigh(node_kernel(length, lo, hi, r))
    return dct_matrix(r) @ ((V * np.sqrt(np.maximum(lam, 0.0))) @ V.T)


def node_roots(p, box, orders):
    """(QxL, QyL, QxH, QyH); the lofi pair is None for a single-fidelity model."""
    xlo, xhi, ylo, yhi = box
    rxL, ryL, rxH, ryH = orders
    QL = (node_root(p.l_L, xlo, xhi, rxL), node_root(p.l_L, ylo, yhi, ryL)) if p.multi else (None, None)
    return QL + (node_root(p.l_H, xlo, xhi, rxH), node_root(p.l_H, ylo, yhi, ryH))


def _prior_rows(x, y, box, Qx, Qy):
    """Rows of the map xi_P -> g_P(x, y) (unit scale), column i ry + j for normal (i, j)."""
    xlo, xhi, ylo, yhi = box
    ax = cheb_basis(x, xlo, xhi, Qx.shape[0]) @ Qx
    ay = cheb_basis(y, ylo, yhi, Qy.shape[0]) @ Qy
    return (ax[:, :, None] * ay[:, None, :]).reshape(ax.shape[0], ax.shape[1] * ay.shape[1])


def pathwise_map(p, ux, uy, X_L, y_L, X_H, y_H, box, orders, Q):
    """(mean[G], A[G, d]) of the draws F = mean + A E over the grid [[x, y] for x in ux for y in uy] (G = nx ny, x-major).
    Q = (QxL, QyL, QxH, QyH) as node_roots gives (or any square roots of the node kernels, for parity with a caller's)."""
    ux = np.asarray(ux, dtype=np.float64).reshape(-1)
    uy = np.asarray(uy, dtype=np.float64).reshape(-1)
    X_L = np.asarray(X_L, dtype=np.float64).reshape(-1, 2)
    X_H = np.asarray(X_H, dtype=np.float64).reshape(-1, 2)
    NL, NH = X_L.shape[0], X_H.shape[0]
    N = NL + NH
    QxL, QyL, QxH, QyH = Q
    multi = bool(p.multi)
    xy = np.stack(np.meshgrid(ux, uy, indexing="ij"), axis=-1).reshape(-1, 2)
    G = xy.shape[0]
    X = np.vstack((X_L, X_H))
    blocks_grid, blocks_X = [], []
    if multi:
        gL = np.sqrt(p.s_L) * _prior_rows(xy[:, 0], xy[:, 1], box, QxL, QyL)
        xL = np.sqrt(p.s_L) * _prior_rows(X[:, 0], X[:, 1], box, QxL, QyL)
        blocks_grid.append(p.rho * gL)
        blocks_X.append(np.where((np.arange(N) < NL)[:, None], xL, p.rho * xL))
    gH = np.sqrt(p.s_H) * _prior_rows(xy[:, 0], xy[:, 1], box, QxH, QyH)
    xH = np.sqrt(p.s_H) * _prior_rows(X[:, 0], X[:, 1], box, QxH, QyH)
    blocks_grid.append(gH)
    blocks_X.append(np.where((np.arange(N) < NL)[:, None], 0.0, xH))
    sigma = np.sqrt(np.where(np.arange(N) < NL, p.noise_L, p.noise_H) + ogp.JITTER)
    A = np.hstack(blocks_grid + [np.zeros((G, N))])
    if N == 0:
        return np.full(G, p.mean_H), A
    PX = np.hstack(blocks_X + [np.diag(sigma)])
    L = ogp.cholesky(ogp.train_cov(p, X_L, X_H))
    psi = ogp.cross_cov(p, xy, X_L, X_H)
    yc = ogp.centered_y(p, y_L, y_H)
    mean = p.mean_H + (psi @ cho_solve((L, True), yc))[:, 0]
    return mean, A - psi @ cho_solve((L, True), PX)
