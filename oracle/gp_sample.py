"""Oracle: joint posterior draws of the multi-fidelity RBF GP (numpy restatement; TEST INFRASTRUCTURE).  Built on
oracle.gp_cov.posterior_cov, the full-matrix posterior of the reference's SFGP.predict / MFGP.predict; the reference itself
has no sampler, so this states the definition the library's sampler is tested against."""
import numpy as np

from .gp_cov import posterior_cov


def posterior_samples(p, X, X_L, y_L, X_H, y_H, E, jitter):
    """Joint posterior draws of f_H at X[G,2] for the standard normals E[G, S]: mu[:, None] + L E with
    L = cholesky(C + jitter I) (lower), mu and C the mean and joint covariance of posterior_cov.  No observation noise."""
    mu, C = posterior_cov(p, X, X_L, y_L, X_H, y_H)
    L = np.linalg.cholesky(C + jitter * np.eye(C.shape[0]))
    return mu[:, None] + L @ np.asarray(E, dtype=np.float64)
