"""Oracle: per-cell centroids of joint posterior draws over a tensor-product grid (numpy restatement; TEST INFRASTRUCTURE).
Companion of csrc/coverage.cu: cov_cell_moments / cov_cell_moments_centroids.

Two routes to the same numbers:
  * dense: draws F = mean + A E from oracle.gp_sample_grid.pathwise_map (or any draws over the grid), then the reference's
    compute_centroids (oracle.coverage) once per draw;
  * coefficient space: the draws as Chebyshev coefficient matrices C_s (draw_coefficients, the restatement of
    mfgp_grid_sample_coef), F_s(ix, iy) = mean + sum_l sum_k Ty[iy][l] Tx[ix][k] C_s[l][k], and the Lloyd partials of cell i
        sum_{p in cell i} w(p) F_s(p) = <C'_s, Mom_i^w>,  Mom_i^w[l][k] = sum_{p in cell i} w(p) Ty[iy_p][l] Tx[ix_p][k],
    w in {1, x, y}, C' = C with mean added to term (0, 0) (T_0 = 1).  Membership is the crossings test of every point
    against every cell polygon (oracle.coverage.membership).
`thompson` is the Thompson-sampling control loop built on the dense route.
"""
import numpy as np

from . import coverage as cov
from . import gp as ogp
from .factored import cheb_basis, cheb_coef, parts, round_up


def tensor_axes(x_star):
    """(ux, uy) of an x-major tensor-product grid [[x, y] for x in ux for y in uy]."""
    x_star = np.asarray(x_star, dtype=np.float64)
    ny = int(np.argmax(x_star[:, 0] != x_star[0, 0])) or x_star.shape[0]
    return x_star[::ny, 0].copy(), x_star[:ny, 1].copy()


def sample_box(ux, uy, X):
    """The sampler's box: the grid and the training points X[N, 2]."""
    X = np.asarray(X, dtype=np.float64).reshape(-1, 2)
    xs, ys = np.concatenate((ux, X[:, 0])), np.concatenate((uy, X[:, 1]))
    return (float(xs.min()), float(xs.max()), float(ys.min()), float(ys.max()))


def draw_coefficients(p, X_L, y_L, X_H, y_H, box, orders, Q, E):
    """C[S, ry, kpad] of the pathwise draws at the normals E[d, S] (layout of include/mfgp_b200.h: mfgp_grid_sample_coef):
    prior coefficients sqrt(s_P) (Qx Xi_P Qy^T)^T, combined as the AR1 model, plus the update B^T K^-1 (y - m - f(X) - eps)
    with B the Chebyshev coefficients of the cross-covariance (oracle.factored), K LAPACK's factor of the exact training
    covariance."""
    rxL, ryL, rxH, ryH = orders
    rx, ry = max(rxL, rxH), max(ryL, ryH)
    kpad = round_up(rx, 4)
    QxL, QyL, QxH, QyH = Q
    E = np.asarray(E, dtype=np.float64)
    S = E.shape[1]
    X_L = np.asarray(X_L, dtype=np.float64).reshape(-1, 2)
    X_H = np.asarray(X_H, dtype=np.float64).reshape(-1, 2)
    X = np.vstack((X_L, X_H))
    NL, N = X_L.shape[0], X.shape[0]
    xlo, xhi, ylo, yhi = box

    def prior(Qx, Qy, off, scale):
        r_x, r_y = Qx.shape[0], Qy.shape[0]
        Xi = E[off:off + r_x * r_y].reshape(r_x, r_y, S)
        C = np.zeros((S, ry, kpad))
        C[:, :r_y, :r_x] = scale * np.einsum("ki,ijs,lj->slk", Qx, Xi, Qy)
        return C

    CH = prior(QxH, QyH, rxL * ryL, np.sqrt(p.s_H))
    if p.multi:
        CL = prior(QxL, QyL, 0, np.sqrt(p.s_L))
        Cp = p.rho * CL + CH
    else:
        CL, Cp = np.zeros_like(CH), CH
    if N == 0:
        return Cp
    Tx, Ty = cheb_basis(X[:, 0], xlo, xhi, kpad), cheb_basis(X[:, 1], ylo, yhi, ry)
    Tx[:, rx:] = 0.0
    fX = np.where((np.arange(N) < NL)[:, None], np.einsum("nl,slk,nk->ns", Ty, CL, Tx), np.einsum("nl,slk,nk->ns", Ty, Cp, Tx))
    sd = np.sqrt(np.where(np.arange(N) < NL, p.noise_L, p.noise_H) + ogp.JITTER)
    R = ogp.centered_y(p, y_L, y_H) - fX - sd[:, None] * E[rxL * ryL + rxH * ryH:]
    L = ogp.cholesky(ogp.train_cov(p, X_L, X_H))
    from scipy.linalg import cho_solve
    alpha = cho_solve((L, True), R)                                          # [N, S]
    B = np.zeros((N, ry, kpad))
    for r_x, r_y, length, coef in parts(p, NL, N - NL, orders):
        Cx = cheb_coef(X[:, 0], xlo, xhi, 1.0 / length, r_x)               # [r_x][N]
        Cy = cheb_coef(X[:, 1], ylo, yhi, 1.0 / length, r_y)
        B[:, :r_y, :r_x] += coef[:, None, None] * Cy.T[:, :, None] * Cx.T[:, None, :]
    return Cp + np.einsum("nlk,ns->slk", B, alpha)


def evaluate(C, mean, ux, uy, box):
    """F[G, S] = mean + sum_l sum_k Ty[iy][l] Tx[ix][k] C[s][l][k] over the grid (x-major)."""
    S, ry, kpad = C.shape
    Tx, Ty = cheb_basis(ux, box[0], box[1], kpad), cheb_basis(uy, box[2], box[3], ry)
    return mean + np.einsum("xk,slk,yl->xys", Tx, C, Ty).reshape(-1, S)


def moments(member, ux, uy, box, ry, kpad):
    """Mom[A, 3, ry, kpad] of the membership member[A, G] (x-major grid), w = 1, x, y; Tx is zero for k >= rx only through
    the caller's coefficients (the basis itself is full)."""
    nx, ny = ux.size, uy.size
    Tx, Ty = cheb_basis(ux, box[0], box[1], kpad), cheb_basis(uy, box[2], box[3], ry)
    M = np.asarray(member, dtype=np.float64).reshape(-1, nx, ny)
    out = np.empty((M.shape[0], 3, ry, kpad))
    out[:, 0] = np.einsum("axy,yl,xk->alk", M, Ty, Tx)
    out[:, 1] = np.einsum("axy,yl,xk->alk", M, Ty, ux[:, None] * Tx)
    out[:, 2] = np.einsum("axy,yl,xk->alk", M, uy[:, None] * Ty, Tx)
    return out


def coefficient_partials(mom, C, mean):
    """cent[S, A, 4] = (<C'_s, Mom_i^1>, <C'_s, Mom_i^x>, <C'_s, Mom_i^y>, n_i), C' = C + mean on term (0, 0)."""
    Cp = np.array(C, dtype=np.float64)
    Cp[:, 0, 0] += mean
    kp = mom.shape[3]
    s = np.einsum("slk,awlk->saw", Cp[:, :, :kp], mom)
    n = np.broadcast_to(mom[None, :, 0, 0, 0, None], (Cp.shape[0], mom.shape[0], 1))
    return np.concatenate((s, n), axis=2)


def dense_partials(member, x_star, F):
    """(cent[S, A, 4], scale[S, A, 3]): the Lloyd partials of every draw F[:, s] over the membership member[A, G], and the
    sums of the magnitudes of their terms (the scale a relative tolerance refers to)."""
    M = np.asarray(member, dtype=np.float64)
    x_star = np.asarray(x_star, dtype=np.float64)
    W = np.stack((np.ones(x_star.shape[0]), x_star[:, 0], x_star[:, 1]), axis=1)        # [G, 3]
    terms = F[:, :, None] * W[:, None, :]                                                 # [G, S, 3]
    sums = np.einsum("ag,gsw->saw", M, terms)
    scale = np.einsum("ag,gsw->saw", M, np.abs(terms))
    n = np.broadcast_to(M.sum(axis=1)[None, :, None], (F.shape[1], M.shape[0], 1))
    return np.concatenate((sums, n), axis=2), scale


def centroids_from_partials(cent, areas, xmin, xmax, ymin, ymax):
    """compute_centroids' arithmetic on partials cent[..., 4]: ((m/n) area) / ((m0/n) area), then the one-sided clamps."""
    with np.errstate(invalid="ignore", divide="ignore"):
        n = cent[..., 3]
        f_int = (cent[..., 0] / n) * areas
        cx = ((cent[..., 1] / n) * areas) / f_int
        cy = ((cent[..., 2] / n) * areas) / f_int
    cx = np.where(cx < xmin, xmin, cx)
    cx = np.where(cx > xmax, xmax, cx)
    cy = np.where(cy < ymin, ymin, cy)
    cy = np.where(cy > ymax, ymax, cy)
    return np.stack((cx, cy), axis=-1)


def dense_centroids(vor, x_star, F):
    """centroids[S, A, 2]: the reference's compute_centroids with w = F[:, s], draw by draw."""
    return np.stack([cov.compute_centroids(vor, x_star, F[:, s]) for s in range(F.shape[1])])


def snap_to_grid(targets, positions, ux, uy):
    """Thompson sampling's move rule, in agent order: the grid point nearest the target per axis (ties to the lower index);
    the grid point nearest the current position when a lower-index agent already took it or the target is NaN."""
    taken = []
    out = np.empty((targets.shape[0], 2))
    for i in range(targets.shape[0]):
        t = targets[i]
        g = None
        if not np.isnan(t).any():
            g = (int(np.argmin(np.abs(ux - t[0]))), int(np.argmin(np.abs(uy - t[1]))))
        if g is None or g in taken:
            g = (int(np.argmin(np.abs(ux - positions[i, 0]))), int(np.argmin(np.abs(uy - positions[i, 1]))))
        taken.append(g)
        out[i] = (ux[g[0]], uy[g[1]])
    return out


def thompson(sim_num, iterations, agents, positions, truth_arr, sigma_n, prior_arr, hyp, normals_rng, noise_rng, orders_of,
             raw_means=False):
    """Thompson-sampling coverage (simulator.thompson), on the helpers of the oracle's control loops (oracle.algorithms):
    every agent samples at its position (not at iteration 0), the model is updated, loss and cell variances come from the
    step with both partitions seeded by the positions; then one joint posterior draw per agent over the whole grid
    (oracle.gp_sample_grid.pathwise_map at E = normals_rng.standard_normal((d, agents))), agent i's target is the centroid
    of its own cell under draw i (compute_centroids, draw by draw) and the agent moves to the grid point snap_to_grid gives.
    `orders_of(p, box)`: the sampler's Chebyshev orders (rxL, ryL, rxH, ryH) for the box of the grid and the training
    points."""
    from . import algorithms as alg
    from . import gp_sample_grid as osg
    fidelity = alg._fidelity(hyp)
    loss_log, agent_log, sample_log = [], [], []
    p, x_star, max_var_0, model = alg._init_gp(hyp, prior_arr, truth_arr, raw_means)
    bbox = cov.bounding_box_of(x_star)
    ux, uy = tensor_axes(x_star)
    ones = np.ones((agents, 1))
    prev_positions = np.copy(positions)
    for iteration in range(iterations):
        explore_t = ones if iteration else np.zeros((agents, 1))
        x_new, y_new, id_new = alg._take_samples(positions, explore_t, truth_arr, sigma_n, noise_rng)
        distance = np.sqrt(np.sum((positions - prev_positions) ** 2, axis=1)).reshape(-1, 1)
        model.append(x_new, y_new)
        loss_t, _, argmax_var_t, max_var_t = alg._iteration_body(model, positions, positions, truth_arr, x_star, bbox)
        box = sample_box(ux, uy, np.vstack((model.X_L, model.X_H)))
        orders = orders_of(p, box)
        mean, A = osg.pathwise_map(p, ux, uy, model.X_L, model.y_L, model.X_H, model.y_H, box, orders,
                                   osg.node_roots(p, box, orders))
        E = normals_rng.standard_normal((A.shape[1], agents))
        F = mean[:, None] + A @ E
        vor = cov.voronoi_bounded(positions, bbox)
        centroids_t = np.stack([cov.compute_centroids(vor, x_star, F[:, i])[i] for i in range(agents)])
        loss_log.append({"SimNum": sim_num, "Iteration": iteration, "Period": 0, "Fidelity": fidelity, "Loss": loss_t})
        agent_log.extend(alg._agent_rows(sim_num, iteration, 0, fidelity, positions, argmax_var_t, max_var_t, max_var_0,
                                         centroids_t, ones, ones, distance))
        sample_log.extend(alg._sample_rows(sim_num, iteration, 0, fidelity, id_new, x_new, y_new))
        prev_positions = np.copy(positions)
        positions = snap_to_grid(centroids_t, prev_positions, ux, uy)
    return loss_log, agent_log, sample_log
