"""gaussian_process.py -- drop-in for the reference module of the same name, backed by libmfgp_b200 on a B200.

Mirrors the call surface of the reference's `SFGP` (gaussian_process.py:23-268) and `MFGP` (:271-578) that the
coverage algorithms use: construction from arrays, `hyp` assigned after construction (simulator.py:72-73, :99-100),
`updt_info`, `updt` / `updt_hifi`, `predict`, and `copy.deepcopy` support.  Differences, both deliberate:

  * `predict(X_star)` returns `(mu[G,1], var[G])` -- the posterior VARIANCE VECTOR, not the G x G covariance matrix
    (gaussian_process.py:146, :435-436) of which the reference's callers only ever take `np.diag`
    (simulator.py:301, :341, :685, :855).  A 1M-point grid would need an 8 TB matrix.  `predict(X_star, full_cov=True)`
    returns the reference's `(mu[G,1], cov[G,G])`; `predict_cov_device` is its device form, with a cross form for
    block rows of a covariance too large to hold whole.  `sample_posterior` (an addition) draws from that joint
    posterior: mu + chol(cov + jitter I) E, with an absolute jitter (default 1e-8 k(0)) and mu the full_cov mean.
    `sample_posterior_grid` draws over whole tensor-product grids of any size by pathwise conditioning, without a
    covariance or a jitter.
  * `likelihood(hyp)` / `train()` (gaussian_process.py:81-119, :344-399) evaluate the negative log marginal likelihood
    AND its analytic gradient on the device (mfgp_nlml_grad) where the reference differentiates with autograd; the
    optimiser is the same scipy L-BFGS-B call.

Every arithmetic step runs on the GPU through the C-ABI in include/mfgp_b200.h; there is no CPU fallback.
"""
import copy
import os
import weakref

import numpy as np
import torch

from ._engine import DeviceGP

JITTER = 1e-8

# Deferred fit (default): updt_info / updt / updt_hifi upload the data and mark the factor stale; the first consumer
# factorises -- on a tensor-product grid `predict` then runs ONE fused pass (Cholesky + forward substitution + posterior)
# instead of Cholesky, explicit inverse, whitening and a status round trip per update.  A non-SPD covariance raises
# np.linalg.LinAlgError from that consumer (`predict`, `factor`, `likelihood`, the coverage step) instead of from the update
# call.  MFGP_EAGER_FIT=1 (or gaussian_process.EAGER_FIT = True before constructing a model) restores the reference's
# timing of the error: np.linalg.cholesky raises inside updt_info (gaussian_process.py:254, :529).
EAGER_FIT = os.environ.get("MFGP_EAGER_FIT", "0") == "1"


def evaluate_hyp(hyp, raw_means=False):
    """Log-scaled hyper-parameters -> evaluated parameters (dict).

    4 entries [mu, s^2, L, noise] (gaussian_process.py:132, :248-251) or 9 entries
    [mu_lo, s^2_lo, L_lo, mu_hi, s^2_hi, L_hi, rho, noise_lo, noise_hi] (:411-416, :510-514).  `raw_means=True` selects
    the 2020 convention (mean = hyp[0], not exp(hyp[0])) that the reference's older logged runs were produced with."""
    hyp = np.asarray(hyp, dtype=np.float64).reshape(-1)
    if hyp.size == 4:
        mean = hyp[0] if raw_means else np.exp(hyp[0])
        return dict(multi=0, s_L=0.0, l_L=1.0, s_H=float(np.exp(hyp[1])), l_H=float(np.exp(hyp[2])), rho=1.0,
                    noise_L=0.0, noise_H=float(np.exp(hyp[3])), mean_L=0.0, mean_H=float(mean), jitter=JITTER)
    if hyp.size == 9:
        rho = np.exp(hyp[6])
        if raw_means:
            mean_L = hyp[0]
            mean_H = rho * mean_L + hyp[3]
        else:
            mean_L = np.exp(hyp[0])
            mean_H = rho * mean_L + np.exp(hyp[3])
        return dict(multi=1, s_L=float(np.exp(hyp[1])), l_L=float(np.exp(hyp[2])), s_H=float(np.exp(hyp[4])),
                    l_H=float(np.exp(hyp[5])), rho=float(rho), noise_L=float(np.exp(hyp[7])),
                    noise_H=float(np.exp(hyp[8])), mean_L=float(mean_L), mean_H=float(mean_H), jitter=JITTER)
    raise TypeError("Hyperparameters must be of length 4 (single-fidelity) or 9 (multi-fidelity)")


def prior_variance(params):
    """k(x, x) of the empty model: what `np.amax(var_star)` evaluates to at simulator.py:672, :842, :1014."""
    if params["multi"]:
        return params["rho"] ** 2 * params["s_L"] + params["s_H"]
    return params["s_H"]



_PINNED_BUDGET = 1 << 30        # page-locked bytes that results handed to the caller may hold at any one time
_pinned_live = [0]


def _to_host_pinned(t):
    """Device tensor -> numpy array in page-locked memory (asynchronous DMA at PCIe speed instead of a staged pageable
    copy).  The block comes from torch's caching host allocator and goes back to it when the numpy array that wraps it is
    garbage collected, so a loop that calls predict() every iteration reuses the same pages; and because the memory is
    page-locked, handing the array back to compute_centroids / compute_max_var uploads it by DMA as well.  A caller that
    keeps many results alive falls back to ordinary pageable arrays once _PINNED_BUDGET bytes are outstanding."""
    nbytes = t.numel() * t.element_size()
    if _pinned_live[0] + nbytes > _PINNED_BUDGET:
        return t.cpu().numpy()
    h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    h.copy_(t, non_blocking=True)
    a = h.numpy()                       # shares (and keeps alive) the page-locked block; views of `a` keep `a` alive
    _pinned_live[0] += nbytes
    weakref.finalize(a, _release_pinned, nbytes)
    return a


def _release_pinned(nbytes):
    _pinned_live[0] -= nbytes


class _GPBase:
    raw_means = False     # set True to reproduce runs logged with the pre-exp() mean convention
    use_separable = True  # tensor-product grids: per-axis factor tables instead of one exp per (point, sample) pair

    def _init_device(self):
        self._dev = DeviceGP()
        self._dev.defer_fit = self._dev.lazy_check = not EAGER_FIT
        self._grid_key = None
        self._grid_dev = None
        self.L = np.empty([0, 0])

    @property
    def engine(self):
        return self._dev

    @property
    def incremental(self):
        """True: appended samples border the standing factorisation (mfgp_cholesky_append) and a posterior held in the
        caller's device buffers is updated with the new rows only -- same results as the reference's refit-from-scratch
        to ~1e-13 k(0), at a fraction of the work.  False (default): refit + full posterior, as the reference does."""
        return self._dev.incremental

    @incremental.setter
    def incremental(self, flag):
        self._dev.incremental = bool(flag)

    def params(self):
        return evaluate_hyp(self.hyp, self.raw_means)

    def _upload_grid(self, X_star):
        xs = np.ascontiguousarray(X_star, dtype=np.float64).reshape(-1, 2)
        host = torch.from_numpy(xs)
        return host.to(self._dev.device, non_blocking=False)

    def predict_device(self, xs_dev, mu_out=None, var_out=None, vcache=None, grid=None, q_out=None):
        """Posterior on device-resident points; returns device tensors (mu[G], var[G]).  `grid`: the CoverageGrid the
        points belong to -- if it is (a slice of) a tensor-product grid the separable-kernel path is used."""
        if not self._dev.fitted:
            self._refit(check=True)
        axes = getattr(grid, "axes", None) if (grid is not None and self.use_separable) else None
        g_lo = grid.base_index if axes is not None else 0
        return self._dev.posterior(xs_dev, mu_out, var_out, vcache, axes=axes, g_lo=g_lo, q_out=q_out)

    def predict_cov_device(self, xs_dev, xs2_dev=None, grid=None, grid2=None, out=None):
        """Joint posterior covariance on device-resident points; returns device tensors (mu[G], C).  xs2_dev None: C is the
        symmetric G x G matrix of xs_dev; otherwise the G x G2 cross block between xs_dev and xs2_dev.  `grid` / `grid2`:
        the CoverageGrid each point set belongs to, as in predict_device.  See DeviceGP.posterior_cov."""
        if not self._dev.fitted:
            self._refit(check=True)

        def axes_of(g):
            axes = getattr(g, "axes", None) if (g is not None and self.use_separable) else None
            return axes, (g.base_index if axes is not None else 0)

        axes_a, g_lo_a = axes_of(grid)
        axes_b, g_lo_b = axes_of(grid2)
        return self._dev.posterior_cov(xs_dev, xs2_dev, axes_a=axes_a, g_lo_a=g_lo_a, axes_b=axes_b, g_lo_b=g_lo_b, out=out)

    def sample_posterior_device(self, xs_dev, normals, grid=None, jitter=None, out=None):
        """Joint posterior draws of the latent f_H on device-resident points: F[G, S] = mu[:, None] + L normals with
        L = chol(C + jitter I), C the joint covariance of predict_cov_device.  `normals`: a float64 [G, S] device tensor of
        standard normals; `jitter`: absolute, added to C's diagonal (default 1e-8 k(0)); `grid` as in predict_device.
        Returns device tensors (mu[G], F[G, S]).  See DeviceGP.posterior_sample."""
        if not self._dev.fitted:
            self._refit(check=True)
        axes = getattr(grid, "axes", None) if (grid is not None and self.use_separable) else None
        g_lo = grid.base_index if axes is not None else 0
        return self._dev.posterior_sample(xs_dev, normals, axes=axes, g_lo=g_lo, jitter=jitter, out=out)

    def sample_posterior(self, X_star, n_samples=1, rng=None, jitter=None):
        """`n_samples` joint draws of the latent f_H at X_star[G,2] from the posterior (no observation noise): a numpy
        array [G, n_samples], column s = mu + L E[:, s] with E = rng.standard_normal((G, n_samples)) and
        L = chol(C + jitter I), C the covariance of predict(X_star, full_cov=True) and mu its mean.  `rng`: a numpy
        Generator (default np.random.default_rng()), so a seeded generator replays the same draws.  `jitter`: absolute,
        added to C's diagonal, default 1e-8 k(0) (prior_variance).  G <= 32768.  Raises LinAlgError for a non-SPD training
        covariance or when C + jitter I is not positive definite (no retry: pass a larger jitter), MemoryError when C and
        its factor do not fit the device."""
        if int(n_samples) != n_samples or n_samples < 1:
            raise ValueError(f"sample_posterior: n_samples must be a positive integer, got {n_samples}")
        if jitter is not None and not (float(jitter) >= 0.0 and np.isfinite(float(jitter))):
            raise ValueError(f"sample_posterior: jitter must be finite and >= 0, got {jitter}")
        X_star = np.asarray(X_star)
        G = X_star.reshape(-1, 2).shape[0]
        if G > self._dev.SAMPLE_MAX_G:
            raise ValueError(f"sample_posterior: {G} points; at most {self._dev.SAMPLE_MAX_G} can be drawn jointly")
        rng = np.random.default_rng() if rng is None else rng
        E = rng.standard_normal((G, int(n_samples)))
        xs_dev, axes = self._device_points(X_star)
        if not self._dev.fitted:
            self._refit(check=True)
        self._dev.check_factor(force=True)        # LinAlgError for a non-SPD training covariance (deferred fit), as predict
        E_dev = torch.from_numpy(E).to(self._dev.device)
        _, F = self._dev.posterior_sample(xs_dev, E_dev, axes=axes, jitter=jitter)
        return F.cpu().numpy()

    @staticmethod
    def _grid_axes(grid):
        from ._engine import TensorAxes
        axes = grid if isinstance(grid, TensorAxes) else getattr(grid, "axes", None)
        if axes is None or getattr(grid, "base_index", 0):
            raise ValueError("sample_posterior_grid: the points are not a whole x-major tensor-product grid "
                             "[[x, y] for x in ux for y in uy]; use sample_posterior for point sets")
        return axes

    def grid_sample_dim(self, grid):
        """Rows d of the normals sample_posterior_grid_device takes for `grid` (a CoverageGrid of a whole tensor-product grid,
        or its TensorAxes)."""
        if not self._dev.fitted:
            self._refit(check=True)
        return self._dev.grid_sample_dim(self._grid_axes(grid))

    def sample_posterior_grid_device(self, grid, normals, ix0=0, ncols=None, out=None):
        """Joint posterior draws of the latent f_H over a whole tensor-product grid, or its columns [ix0, ix0 + ncols), by
        pathwise conditioning: F = mu + A E with A A^T the posterior covariance, no jitter and no limit on the grid's size.
        `grid`: a CoverageGrid of the whole grid (or its TensorAxes); `normals`: a float64 [grid_sample_dim(grid), S] device
        tensor of standard normals.  Returns F[ncols * ny, S] on the device.  See DeviceGP.posterior_sample_grid."""
        if not self._dev.fitted:
            self._refit(check=True)
        return self._dev.posterior_sample_grid(self._grid_axes(grid), normals, ix0=ix0, ncols=ncols, out=out)

    def sample_posterior_grid(self, X_star, n_samples=1, rng=None):
        """`n_samples` joint draws of the latent f_H over the tensor-product grid X_star[G,2] (x-major,
        `[[x, y] for x in ux for y in uy]`): a numpy array [G, n_samples], F = mu + A E with E = rng.standard_normal((d,
        n_samples)), d = grid_sample_dim, and A A^T the posterior covariance of predict(X_star, full_cov=True).  Pathwise
        conditioning on a prior draw at Chebyshev nodes: unlike sample_posterior, no G x G covariance is formed, so whole 1M-point
        grids can be drawn, and no jitter is added.  `rng`: a numpy Generator (default np.random.default_rng()).  Raises
        ValueError when X_star is not such a grid or the length scales are too short for 64 Chebyshev terms over the grid and the
        training points (sample_posterior covers both), LinAlgError for a non-SPD training covariance, MemoryError when the
        draws do not fit the device."""
        if int(n_samples) != n_samples or n_samples < 1:
            raise ValueError(f"sample_posterior_grid: n_samples must be a positive integer, got {n_samples}")
        X_star = np.asarray(X_star)
        self._device_points(X_star)
        axes = self._grid_dev[1]
        if axes is None:
            raise ValueError("sample_posterior_grid: X_star is not an x-major tensor-product grid [[x, y] for x in ux for y in uy]; "
                             "use sample_posterior for point sets")
        if not self._dev.fitted:
            self._refit(check=True)
        self._dev.check_factor(force=True)        # LinAlgError for a non-SPD training covariance (deferred fit), as predict
        d = self._dev.grid_sample_dim(axes)
        rng = np.random.default_rng() if rng is None else rng
        E = rng.standard_normal((d, int(n_samples)))
        F = self._dev.posterior_sample_grid(axes, torch.from_numpy(E).to(self._dev.device))
        return F.cpu().numpy()

    def _device_points(self, X_star):
        """Device copy of X_star and its tensor-product axes (None if it is not such a grid, or use_separable is off)."""
        from ._engine import TensorAxes, detect_tensor_grid
        # the reference's loops pass the SAME x_star array every iteration (simulator.py:892): its device copy and its
        # tensor-grid analysis are cached on the array's identity (the host array is kept alive by the cache)
        from ._coverage import host_array_key
        key = host_array_key(X_star)
        if self._grid_key == key:
            xs_dev, axes, _ = self._grid_dev
        else:
            xs_dev = self._upload_grid(X_star)
            t = detect_tensor_grid(X_star)
            axes = TensorAxes(t[0], t[1], self._dev.device) if t is not None else None
            self._grid_key, self._grid_dev = key, (xs_dev, axes, X_star)
        return xs_dev, (axes if self.use_separable else None)

    def predict(self, X_star, full_cov=False):
        """Posterior mean [G,1] and variance [G] at X_star[G,2] (host arrays in, host arrays out).

        full_cov=True: the reference's return value (gaussian_process.py:146, :435-436), mean [G,1] and the joint covariance
        [G,G] (8 G^2 bytes on the device and on the host; MemoryError if they do not fit).  That mean comes from the dense
        posterior call that also forms the whitened cross-covariance, so on tensor-product grids where the default call
        takes the Chebyshev-factored path the two means can differ in the last bits; both are within 1e-9 of the exact
        posterior."""
        xs_dev, axes = self._device_points(np.asarray(X_star))
        if not self._dev.fitted:
            self._refit(check=True)
        if full_cov:
            mu, C = self._dev.posterior_cov(xs_dev, axes_a=axes)
            mu_h, C_h = mu.cpu().numpy(), C.cpu().numpy()
            self._dev.check_factor(force=True)    # LinAlgError for a non-SPD covariance (deferred fit), as below
            return mu_h.reshape(-1, 1), C_h
        mu, var = self._dev.posterior(xs_dev, axes=axes)
        mu_h, var_h = _to_host_pinned(mu), _to_host_pinned(var)
        self._dev.check_factor(force=True)        # synchronises; raises LinAlgError for a non-SPD covariance (deferred fit)
        return mu_h.reshape(-1, 1), var_h

    # -- hyper-parameter training (gaussian_process.py:81-119, :344-399) ------------------------------------------------
    def likelihood_and_grad(self, hyp):
        """(NLML, d NLML / d hyp) for log-scaled hyper-parameters `hyp` on the model's current data, on the device: refit
        (K assembly, tiled Cholesky, inverse, whitening) + mfgp_nlml_grad.  Raises np.linalg.LinAlgError where the
        reference's np.linalg.cholesky does.  The exp() mean convention of the reference's likelihood is used whatever
        `raw_means` says (:89, :356-357)."""
        hyp = np.asarray(hyp, dtype=np.float64).reshape(-1)
        if hyp.size != np.asarray(self.hyp).reshape(-1).size:
            raise TypeError("Hyperparameters must be of length 4 (single-fidelity) or 9 (multi-fidelity)")
        keep_hyp, keep_raw = self.hyp, self.raw_means
        self.hyp, self.raw_means = hyp, False
        try:
            self._refit(check=True)
        finally:
            self.hyp, self.raw_means = keep_hyp, keep_raw
        value, grad = self._dev.nlml_grad()
        return value, grad[:hyp.size]

    def likelihood(self, hyp):
        """reference gaussian_process.py:81-105 / :344-384: negative log marginal likelihood (scalar)."""
        return self.likelihood_and_grad(hyp)[0]

    def callback(self, params):
        """reference gaussian_process.py:219-227 / :483-491."""
        print("Log likelihood {}".format(self.likelihood(params)))

    def train(self, callback=True, **options):
        """reference gaussian_process.py:107-119 / :386-399: L-BFGS-B on the NLML from the current `hyp`; the value and the
        gradient come from ONE device evaluation per optimiser step (the reference: autograd's value_and_grad)."""
        from scipy.optimize import minimize
        cb = self.callback if callback is True else (callback or None)
        result = minimize(self.likelihood_and_grad, np.asarray(self.hyp, dtype=np.float64), jac=True, method="L-BFGS-B",
                          callback=cb, options=options or None)
        self.hyp = result.x
        self._refit(check=True)          # leave the device state on the trained hyper-parameters
        return result

    def factor(self):
        """Lower Cholesky factor L[N,N] as a host array (the reference keeps it in `self.L`)."""
        d = self._dev
        if d.N == 0:
            return np.empty([0, 0])
        d.check_factor(force=True)
        return torch.tril(d.K[:d.N, :d.N]).cpu().numpy()

    def __deepcopy__(self, memo):
        cls = self.__class__
        other = cls.__new__(cls)
        memo[id(self)] = other
        for k, v in self.__dict__.items():
            if k == "_dev":
                other._dev = v.clone()
            elif k in ("_grid_dev", "_grid_key"):
                setattr(other, k, None)
            else:
                setattr(other, k, copy.deepcopy(v, memo))
        return other


class SFGP(_GPBase):
    """Single-fidelity GP (reference gaussian_process.py:23-268)."""

    def __init__(self, X, y, len):
        self.D = X.shape[1]
        self.X = X
        self.y = y
        hyp = np.log(np.ones(self.D + 1))
        self.idx_theta = np.arange(hyp.shape[0])
        hyp = np.concatenate([hyp, np.array([-4.0])])
        hyp[0] = -4.0
        hyp[2] = np.log(len)
        self.hyp = hyp
        self.jitter = JITTER
        self._init_device()

    def _refit(self, check=True):
        N = self.X.shape[0]
        self._dev.fit(self.X, self.y, 0, N, self.params(), check=check)

    def updt_info(self, X_new, y_new):
        self.X = X_new
        self.y = y_new
        self._refit()

    def updt(self, X_addition, y_addition):
        self.X = np.vstack((self.X, X_addition))
        self.y = np.vstack((self.y, y_addition))
        d = self._dev
        if d.fitted and d.N + np.asarray(X_addition).reshape(-1, 2).shape[0] == self.X.shape[0]:
            d.set_params(self.params())
            d.append_hifi(X_addition, y_addition)      # device already holds the old rows: upload only the new ones
        else:
            self._refit()


class MFGP(_GPBase):
    """Two-level AR1 multi-fidelity GP (reference gaussian_process.py:271-578)."""

    def __init__(self, X_L, y_L, X_H, y_H, len_L, len_H):
        self.D = X_H.shape[1]
        self.X_L = X_L
        self.y_L = y_L
        self.X_H = X_H
        self.y_H = y_H
        hyp = np.ones(self.D + 1)
        hyp[0] = 0
        self.idx_theta_L = np.arange(hyp.shape[0])
        hyp = np.concatenate((hyp, hyp))
        self.idx_theta_H = np.arange(self.idx_theta_L[-1] + 1, hyp.shape[0])
        hyp = np.concatenate((hyp, np.array([-1.0]), np.array([0, 0])))
        hyp[0] = 0
        hyp[3] = 0
        hyp[2] = np.log(len_L)
        hyp[5] = np.log(len_H)
        self.hyp = hyp
        self.jitter = JITTER
        self._init_device()

    def _refit(self, check=True):
        NL, NH = self.X_L.shape[0], self.X_H.shape[0]
        Xt = np.vstack((np.asarray(self.X_L, dtype=np.float64).reshape(-1, 2),
                        np.asarray(self.X_H, dtype=np.float64).reshape(-1, 2)))
        y = np.vstack((np.asarray(self.y_L, dtype=np.float64).reshape(-1, 1),
                       np.asarray(self.y_H, dtype=np.float64).reshape(-1, 1)))
        self._dev.fit(Xt, y, NL, NH, self.params(), check=check)

    def updt_info(self, X_L_new, y_L_new, X_H_new, y_H_new):
        self.X_L = X_L_new
        self.y_L = y_L_new
        self.X_H = X_H_new
        self.y_H = y_H_new
        self._refit()

    def updt_hifi(self, X_H_addition, y_H_addition):
        self.X_H = np.vstack((self.X_H, X_H_addition))
        self.y_H = np.vstack((self.y_H, y_H_addition))
        d = self._dev
        k = np.asarray(X_H_addition).reshape(-1, 2).shape[0]
        if d.fitted and d.NL == self.X_L.shape[0] and d.NH + k == self.X_H.shape[0]:
            d.set_params(self.params())
            d.append_hifi(X_H_addition, y_H_addition)
        else:
            self._refit()
