"""Oracle: the FULL posterior covariance of the single- and two-level multi-fidelity RBF GP (numpy restatement; TEST
INFRASTRUCTURE).  Companion of oracle/gp.py, whose building blocks it uses, for the matrix that
/root/reference/gaussian_process.py returns and oracle.gp.posterior restates diagonal-only:
  prior_cov           <- k(X*, X*') of SFGP.predict :146, MFGP.predict :435-436 (no noise, no jitter)
  posterior_cov       <- SFGP.predict :139-146, MFGP.predict :426-436, the joint covariance or a cross block
"""
import numpy as np
from scipy.linalg import solve_triangular

from .gp import centered_y, cholesky, cross_cov, rbf, train_cov


def prior_cov(p, X_a, X_b):
    """k**(A, B) [Ga, Gb], the prior covariance without noise: gaussian_process.py:146 (SF), :435-436 (MF)."""
    X_a = np.asarray(X_a, dtype=np.float64).reshape(-1, 2)
    X_b = np.asarray(X_b, dtype=np.float64).reshape(-1, 2)
    if not p.multi:
        return rbf(X_a, X_b, p.s_H, p.l_H)
    return p.rho ** 2 * rbf(X_a, X_b, p.s_L, p.l_L) + rbf(X_a, X_b, p.s_H, p.l_H)


def posterior_cov(p, X_a, X_L, y_L, X_H, y_H, X_b=None, L=None, exact_solve=False):
    """Posterior mean [Ga] at X_a and the joint covariance [Ga, Ga] (X_b None) or the cross block [Ga, Gb] between X_a and
    X_b -- the full matrix of SFGP.predict :139-146 / MFGP.predict :426-436:  beta = L^-T L^-1 psi_B^T,
    cov = k**(A, B) - psi_A beta.  `exact_solve=True` keeps the reference's general `np.linalg.solve` calls; the default
    whitens both sides with one triangular solve each, cov = k** - (L^-1 psi_A^T)^T (L^-1 psi_B^T).
    With an empty model the reference returns the constant mean and k**(A, B)."""
    X_a = np.asarray(X_a, dtype=np.float64).reshape(-1, 2)
    X_b = X_a if X_b is None else np.asarray(X_b, dtype=np.float64).reshape(-1, 2)
    X_L = np.asarray(X_L, dtype=np.float64).reshape(-1, 2)
    X_H = np.asarray(X_H, dtype=np.float64).reshape(-1, 2)
    N = X_L.shape[0] + X_H.shape[0]
    cov = prior_cov(p, X_a, X_b)
    if N == 0:
        return np.full(X_a.shape[0], p.mean_H, dtype=np.float64), cov
    if L is None:
        L = cholesky(train_cov(p, X_L, X_H))
    y = centered_y(p, y_L, y_H)
    psi_a = cross_cov(p, X_a, X_L, X_H)
    psi_b = psi_a if X_b is X_a else cross_cov(p, X_b, X_L, X_H)
    if exact_solve:
        alpha = np.linalg.solve(L.T, np.linalg.solve(L, y))
        beta = np.linalg.solve(L.T, np.linalg.solve(L, psi_b.T))
        cov -= psi_a @ beta
    else:
        alpha = solve_triangular(L.T, solve_triangular(L, y, lower=True), lower=False)
        v_a = solve_triangular(L, psi_a.T, lower=True)
        v_b = v_a if psi_b is psi_a else solve_triangular(L, psi_b.T, lower=True)
        cov -= v_a.T @ v_b
    return p.mean_H + (psi_a @ alpha)[:, 0], cov
