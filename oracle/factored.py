"""Oracle: the Chebyshev-factored grid posterior of csrc/gp_factored.cu, restated term by term (numpy; TEST INFRASTRUCTURE).

For explicit orders (rxL, ryL, rxH, ryH), the interval [xlo, xhi] x [ylo, yhi] and an optional truncated column layout kx,
every grid point (ix, iy) of the columns [ix0, ix0 + ncols) gets the approximate cross-covariance
    psi~[n] = sum_P coef_P[n] sum_{l < ry_P} sum_{k < min(rx_P, kx[l])} T_l(t_y) T_k(t_x) Cy_P[l][n] Cx_P[k][n]
and the posterior built from it with LAPACK's factor of the exact training covariance (oracle.gp.train_cov):
    q = |L^-1 psi~|^2,   var = k0 - q,   mu = mean_H + psi~ . K^-1 (y - m).
Nothing here forms W B, Y', M = Y^T Y, G'(ix) or z^T Y: the routes of steps 3-6 are what this checks, not what it repeats.
At converged orders psi~ is the exact cross-covariance to ~5e-15 and this is oracle.gp.posterior; at under-resolved orders
every kept term matters, which is where a kernel that drops or mis-indexes one can be told apart.
"""
import numpy as np
from scipy.linalg import solve_triangular

from . import gp as ogp


def round_up(v, m):
    return -(-int(v) // m) * m


def cheb_coef(u, lo, hi, inv_l, r):
    """C[k][n]: order-r Chebyshev coefficients of t -> exp(-0.5 ((x(t) - u_n) / l)^2) on [lo, hi], by the DCT at the r
    Chebyshev nodes -- cheb_coef_kernel (gp_factored.cu:58-92): node_j = mid + half cos(pi (j + 1/2) / r),
    C[k][n] = (k ? 2 : 1) / r * sum_j cos(pi k (j + 1/2) / r) f_n(node_j)."""
    u = np.asarray(u, dtype=np.float64).reshape(-1)
    if r == 0:
        return np.zeros((0, u.size))
    mid, half = 0.5 * (lo + hi), 0.5 * (hi - lo)
    j = np.arange(r) + 0.5
    node = mid + half * np.cos(np.pi * j / r)
    D = np.cos(np.pi * np.outer(np.arange(r), j) / r) * np.where(np.arange(r) == 0, 1.0, 2.0)[:, None] / r
    d = (node[:, None] - u[None, :]) * inv_l
    return D @ np.exp(-0.5 * d * d)


def cheb_basis(u, lo, hi, r):
    """T[i][k] = T_k(t(u_i)), t = (2 u - (lo + hi)) / (hi - lo), by the three-term recurrence of cheb_basis_kernel
    (gp_factored.cu:95-111)."""
    t = (2.0 * np.asarray(u, dtype=np.float64).reshape(-1) - (lo + hi)) / (hi - lo)
    T = np.empty((t.size, r))
    t0, t1 = np.ones_like(t), t
    for k in range(r):
        T[:, k] = t0
        t0, t1 = t1, 2.0 * t * t1 - t0
    return T


def parts(p, NL, NH, orders):
    """Per kernel part: (rx, ry, l, coef[N]) -- the tables f_carve adds (gp_factored.cu:808-814) and the weights
    f_tables_and_B gives build_B_merged_kernel (:853-854): lofi part rho s_L on lofi rows and rho^2 s_L on hifi rows,
    hifi part 0 on lofi rows and s_H on hifi rows.  A single-fidelity model has the hifi part only."""
    rxL, ryL, rxH, ryH = orders
    lofi = np.arange(NL + NH) < NL
    out = []
    if p.multi:
        out.append((rxL, ryL, p.l_L, np.where(lofi, p.rho * p.s_L, p.rho ** 2 * p.s_L)))
    out.append((rxH, ryH, p.l_H, np.where(lofi, 0.0, p.s_H)))
    return out


def layout(orders, kx=None):
    """kx[l] for every y term l of the merged expansion (ry = max(ryL, ryH), kpad = round_up(max(rxL, rxH), 4)): the
    given truncated layout or kpad everywhere (f_set_trunc, gp_factored.cu:768-783)."""
    rxL, ryL, rxH, ryH = orders
    ry, kpad = max(ryL, ryH), round_up(max(rxL, rxH), 4)
    if kx is None:
        return np.full(ry, kpad, dtype=np.int64)
    kx = np.asarray(kx, dtype=np.int64).reshape(-1)
    assert kx.size == ry and np.all((kx >= 4) & (kx <= kpad) & (kx % 4 == 0)), "not a layout the library accepts"
    return kx


def highest_term(p, orders, kx=None):
    """The (l, k) term of largest l, and of largest k for that l, that carries a non-zero coefficient in some part: the far
    corner of the kept block, where a kernel that loses the last x term of the last y term would differ."""
    kxl = layout(orders, kx)
    l = kxl.size - 1
    k = max(min(rx, int(kxl[l])) for rx, ry, _, _ in parts(p, 0, 1, orders) if l < ry) - 1
    return l, k


def factored_psi(p, X_L, X_H, ux, uy, ix0, ncols, orders, box, kx=None, drop=None):
    """psi~[g][n] for the grid points g = (ix - ix0) * ny + iy of the columns [ix0, ix0 + ncols) (the flat output order of
    the library), training points [X_L; X_H].  box = (xlo, xhi, ylo, yhi).  drop: an (l, k) term left out of every part."""
    X_L = np.asarray(X_L, dtype=np.float64).reshape(-1, 2)
    X_H = np.asarray(X_H, dtype=np.float64).reshape(-1, 2)
    X = np.vstack((X_L, X_H))
    NL, N = X_L.shape[0], X.shape[0]
    xlo, xhi, ylo, yhi = box
    kxl = layout(orders, kx)
    ux = np.asarray(ux, dtype=np.float64)[ix0:ix0 + ncols]
    uy = np.asarray(uy, dtype=np.float64).reshape(-1)
    psi = np.zeros((ncols, uy.size, N))
    for rx, ry, length, coef in parts(p, NL, N - NL, orders):
        Cx = cheb_coef(X[:, 0], xlo, xhi, 1.0 / length, rx)                 # [rx][N]
        Cy = cheb_coef(X[:, 1], ylo, yhi, 1.0 / length, ry)                 # [ry][N]
        Tx, Ty = cheb_basis(ux, xlo, xhi, rx), cheb_basis(uy, ylo, yhi, ry)
        # Sx[n][ix][l] = sum_{k < min(rx, kx[l])} T_k(tx) Cx[k][n]: the x sum that y term l keeps
        Sx = np.empty((N, ncols, ry))
        for l in range(ry):
            kk = min(rx, int(kxl[l]))
            cx = Cx[:kk].copy()
            if drop is not None and drop[0] == l and drop[1] < kk:
                cx[drop[1]] = 0.0
            Sx[:, :, l] = (Tx[:, :kk] @ cx).T
        Sy = Ty[None, :, :] * Cy.T[:, None, :]                                 # [N][iy][l] = T_l(ty) Cy[l][n]
        psi += coef[None, None, :] * np.moveaxis(Sx @ np.swapaxes(Sy, 1, 2), 0, 2)
    return psi.reshape(ncols * uy.size, N)


def factor(p, X_L, X_H, y_L, y_H):
    """(L, alpha): LAPACK's Cholesky factor of K + jitter I (oracle.gp.train_cov) and K^-1 (y - m)."""
    L = ogp.cholesky(ogp.train_cov(p, X_L, X_H))
    yc = ogp.centered_y(p, y_L, y_H)
    alpha = solve_triangular(L.T, solve_triangular(L, yc, lower=True), lower=False)
    return L, alpha[:, 0]


def posterior_from_psi(p, L, alpha, psi):
    """(mu, var, q) of the cross-covariances psi[G][N]."""
    v = solve_triangular(L, psi.T, lower=True)
    q = np.einsum("ij,ij->j", v, v)
    return p.mean_H + psi @ alpha, p.k0 - q, q


def posterior(p, X_L, y_L, X_H, y_H, ux, uy, ix0, ncols, orders, box, kx=None, drop=None, fac=None):
    """(mu, var, q) of the factored expansion for the columns [ix0, ix0 + ncols), flat in the library's output order.
    fac: (L, alpha) of `factor`, when the caller already has it."""
    L, alpha = factor(p, X_L, X_H, y_L, y_H) if fac is None else fac
    psi = factored_psi(p, X_L, X_H, ux, uy, ix0, ncols, orders, box, kx, drop)
    return posterior_from_psi(p, L, alpha, psi)
