"""Device-side state of one GP model and the calls into libmfgp_b200 that operate on it.

`DeviceGP` owns the HBM-resident buffers of a model -- training points Xt[cap,2], observations y[cap], covariance /
Cholesky factor K[npad,npad], its inverse W[npad,npad], scaled coordinates Tt[npad,4], whitened observations z[npad]
-- and sequences the C-ABI calls of include/mfgp_b200.h on the current CUDA stream.  torch provides memory and
streams only.  Layout notes are in DESIGN.md ("Data layout in HBM").
"""
import ctypes
import os
import itertools

import numpy as np
import torch

from . import _native as nat

# MFGP_FUSED_GRAM=0: the Gram product M = Y^T Y of the factored posterior as a separate launch after the factorisation
# (default: accumulated inside the tile-dataflow kernel, see include/mfgp_b200.h: mfgp_cholesky_solve_gram)
FUSED_GRAM = os.environ.get("MFGP_FUSED_GRAM", "1") != "0"


def chebyshev_order(length_scale, lo, hi, centre_lo, centre_hi, tol=5e-15, rmax=64):
    """Smallest Chebyshev order r (multiple of 4) whose interpolant of u -> exp(-0.5 ((u - c) / l)^2) on [lo, hi] has
    converged to `tol` (relative size of the last three coefficients) for every centre c in [centre_lo, centre_hi]
    -- the training coordinates along this axis.  None if rmax does not suffice (short length scale: use the dense path)."""
    half, mid = 0.5 * (hi - lo), 0.5 * (hi + lo)
    if not (half > 0.0) or not (length_scale > 0.0):
        return None
    centres = np.linspace(min(centre_lo, lo), max(centre_hi, hi), 17)
    for r in range(8, rmax + 1, 4):
        j = np.arange(r)
        nodes = mid + half * np.cos(np.pi * (j + 0.5) / r)
        f = np.exp(-0.5 * ((nodes[:, None] - centres[None, :]) / length_scale) ** 2)
        c = (np.cos(np.pi * np.outer(np.arange(r), j + 0.5) / r) @ f) * (2.0 / r)
        scale = max(float(np.abs(c).max()), 1e-300)
        if float(np.abs(c[-3:]).max()) <= tol * scale:
            return r
    return None


def chebyshev_envelope(length_scale, lo, hi, centre_lo, centre_hi, r):
    """|c_k| / max|c|, k < r, of the order-r Chebyshev interpolant of u -> exp(-0.5 ((u - c) / l)^2) on [lo, hi], maximised over
    the centres c in [centre_lo, centre_hi] (the same sampling as chebyshev_order)."""
    half, mid = 0.5 * (hi - lo), 0.5 * (hi + lo)
    centres = np.linspace(min(centre_lo, lo), max(centre_hi, hi), 17)
    j = np.arange(r)
    nodes = mid + half * np.cos(np.pi * (j + 0.5) / r)
    f = np.exp(-0.5 * ((nodes[:, None] - centres[None, :]) / length_scale) ** 2)
    c = np.abs((np.cos(np.pi * np.outer(np.arange(r), j + 0.5) / r) @ f) * (2.0 / r))
    return c.max(axis=1) / max(float(c.max()), 1e-300)


def chebyshev_truncation(parts, kpad, ry, tol=1e-16):
    """Truncated column layout of the factored posterior's right-hand sides (include/mfgp_b200.h: kx).  `parts`: per kernel
    part (envelope over k of the x factor, envelope over l of the y factor).  Term (l, k) is kept while ANY part's bound
    a_y[l] a_x[k] exceeds `tol`; per y term l the kept x terms are rounded up to a multiple of 4.  The dropped terms of a row
    decay super-exponentially behind the first one (<= ~1.5 tol per row, ry rows): with tol = 1e-16 their sum stays below the
    5e-15 the orders themselves were chosen for.  Returns an int32 array of ry entries."""
    kx = np.empty(ry, dtype=np.int32)
    for l in range(ry):
        last = -1
        for ax, ay in parts:
            if l < ay.size:
                keep = np.nonzero(ay[l] * ax > tol)[0]
                if keep.size:
                    last = max(last, int(keep[-1]))
        kx[l] = min(kpad, max(4, -(-(last + 1) // 4) * 4))
    return kx


# MFGP_GUARD=1 (tests): every workspace of the factored / fused path is allocated inside canary margins and sized EXACTLY as the
# library asks; check_guards() then proves that no kernel wrote outside what it was given (compute-sanitizer stand-in)
GUARD = os.environ.get("MFGP_GUARD", "0") != "0"
_CANARY = -7.25e300


# MFGP_TRUNC=0: keep the full rx x ry tensor block of Chebyshev terms (default: product-magnitude truncation, ~1/3 fewer columns)
TRUNCATE = os.environ.get("MFGP_TRUNC", "1") != "0"


class TensorAxes:
    """Axis values of a tensor-product grid `[[x, y] for x in ux for y in uy]` (x-major, distribution.py:337-339)."""

    _uids = itertools.count(1)

    def __init__(self, ux_host, uy_host, device):
        # never reused, unlike id(): plan / order caches key on it, so a collected grid cannot alias a new one
        self.uid = next(TensorAxes._uids)
        self.ux_host = np.ascontiguousarray(ux_host, dtype=np.float64)
        self.uy_host = np.ascontiguousarray(uy_host, dtype=np.float64)
        self.nx, self.ny = int(len(ux_host)), int(len(uy_host))
        self.xlo, self.xhi = float(self.ux_host.min()), float(self.ux_host.max())
        self.ylo, self.yhi = float(self.uy_host.min()), float(self.uy_host.max())
        self.ux = torch.from_numpy(np.ascontiguousarray(ux_host, dtype=np.float64)).to(device)
        self.uy = torch.from_numpy(np.ascontiguousarray(uy_host, dtype=np.float64)).to(device)


def detect_tensor_grid(xy):
    """(ux, uy) if xy[G,2] is exactly `[[x, y] for x in ux for y in uy]` (bitwise), else None.  O(G), vectorised."""
    xy = np.asarray(xy, dtype=np.float64)
    G = xy.shape[0]
    if G < 4:
        return None
    change = np.nonzero(xy[1:, 0] != xy[0, 0])[0]
    ny = int(change[0]) + 1 if change.size else G
    if ny < 2 or G % ny:
        return None
    nx = G // ny
    ux, uy = xy[::ny, 0].copy(), xy[:ny, 1].copy()
    if nx * ny != G or not np.array_equal(xy[:, 0], np.repeat(ux, ny)) or not np.array_equal(xy[:, 1], np.tile(uy, nx)):
        return None
    return ux, uy


def node_root(length, lo, hi, r):
    """Q[r, r] = DCT V sqrt(max(Lambda, 0)) V^T for the unit-scale RBF kernel matrix V Lambda V^T at the r Chebyshev nodes
    mid + half cos(pi (j + 1/2) / r) of [lo, hi], DCT[k][j] = (k ? 2 : 1) / r cos(pi k (j + 1/2) / r) (cheb_coef_kernel's
    node-values-to-coefficients map): Q xi, xi ~ N(0, I), are the Chebyshev coefficients of the interpolant of a prior draw."""
    j = np.arange(r) + 0.5
    node = 0.5 * (lo + hi) + 0.5 * (hi - lo) * np.cos(np.pi * j / r)
    d = (node[:, None] - node[None, :]) / length
    lam, V = np.linalg.eigh(np.exp(-0.5 * d * d))
    dct = np.cos(np.pi * np.outer(np.arange(r), j) / r) * np.where(np.arange(r) == 0, 1.0, 2.0)[:, None] / r
    return np.ascontiguousarray(dct @ ((V * np.sqrt(np.maximum(lam, 0.0))) @ V.T))


def grid_sample_orders(p, box):
    """Chebyshev orders {"Lx", "Ly" (multi-fidelity only), "Hx", "Hy"} of the pathwise grid sampler on `box` (xlo, xhi, ylo,
    yhi) for the evaluated parameters `p`.  ValueError when the box spans no area or an order would exceed 64."""
    if not (box[1] > box[0] and box[3] > box[2]):
        raise ValueError("sample_posterior_grid: the grid and the training points span no area; use sample_posterior")
    orders = {}
    for part, length in ((("L", p["l_L"]), ("H", p["l_H"])) if p["multi"] else (("H", p["l_H"]),)):
        for ax, lo, hi in (("x", box[0], box[1]), ("y", box[2], box[3])):
            r = chebyshev_order(length, lo, hi, lo, hi)
            if r is None:
                raise ValueError(f"sample_posterior_grid: length scale {length:.4g} needs more than 64 Chebyshev terms over "
                                 f"[{lo:.4g}, {hi:.4g}]; draw at point sets of up to {DeviceGP.SAMPLE_MAX_G} points with "
                                 "sample_posterior instead")
            orders[part + ax] = r
    return orders


def params_struct(p):
    """p: dict with the evaluated parameters (see gaussian_process.evaluate_hyp)."""
    return nat.MfgpParams(p["s_L"], p["l_L"], p["s_H"], p["l_H"], p["rho"], p["noise_L"], p["noise_H"],
                          p["mean_L"], p["mean_H"], p["jitter"], int(p["multi"]), 0)


class DeviceGP:
    def __init__(self, device=None):
        nat.require_cuda()
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.NL = 0
        self.NH = 0
        self.npad = 0
        self.cap = 0          # allocated padded size of K / W
        self.Xt = self.y = self.K = self.W = self.Tt = self.z = self.work = None
        self.info = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.params = None
        self.pstruct = None
        self.fitted = False
        self.fit_id = 0               # bumped by every refactor / append: grid tables are rebuilt lazily when stale
        self._tab = None              # (axes key, fit_id, TLx, TLy, THx, THy, ldt)
        # incremental mode (SURVEY 8f rank 1): appended samples border the standing factor instead of a from-scratch
        # refit, and a posterior that was computed into the same (mu, var) buffers is updated with the new rows only
        self.use_factored = True      # tensor-product grids: Chebyshev-factored posterior when it is cheaper (gp_factored.cu)
        self.factored_min_gain = 2.0  # ... i.e. when its MAC count is at least this factor below the dense kernel's
        self._fplan = None            # (key, plan, orders) of the last factored-posterior plan
        self._forders = None          # (key, hull, orders): Chebyshev orders and the training-point hull they cover
        self._ftrunc = None           # truncated column layout (kx per y term) that goes with _forders, or None
        self.rhs_cols = None          # (expansion columns, padded right-hand-side count) of the last fused fit
        self._fwork = None
        self._xrange = None           # (xmin, xmax, ymin, ymax) of the training points, refreshed by fit / append
        self.defer_fit = False        # True: refactor(check=False) only marks the factor stale; the first consumer factorises --
        self._dirty = False           #   a factored posterior then fuses fit + forward substitution (mfgp_cholesky_solve)
        self._w_partial = False       # True: W holds only the diagonal-block inverses (mfgp_tri_inverse still to run)
        self._fB = None               # right-hand-side matrix of the fused fit
        self._twork = None            # workspace of mfgp_nlml_grad (hyper-parameter training)
        self._cwork = None            # ticket counter + tile flags of mfgp_cholesky_solve (caller-owned, per model)
        self._fG = None               # per-column Gram matrices G'(ix) [ncols, 64, 64] and z^T Y: state of the incremental
        self._fHz = None              #   factored update (mfgp_posterior_grid_factored_update)
        self._fstate = None           # (plan key, epoch, rows covered, output buffer key) the stores are valid for
        self.incremental = False
        self.profile_events = None    # optional (start, stop) torch.cuda.Event pair recorded around mfgp_cholesky_solve
        self.lazy_check = False       # True: the caller reads `info` itself (cov_finish carries it home): no sync per fit
        self.epoch = 0                # bumped by every FULL refactor: standing posteriors become stale
        self._post = None             # (buffer key, epoch, N covered)
        self._splan = None            # plan of the pathwise grid sampler (_grid_sample_plan)

    # -- memory -------------------------------------------------------------------------------------------------------
    def _reserve(self, n, keep_factor=False):
        need = nat.npad(n)
        if need <= self.cap:
            return
        cap = max(need, nat.npad(int(self.cap * 1.5)))
        f64 = dict(dtype=torch.float64, device=self.device)
        old = (self.K, self.W, self.Tt, self.z, self.npad) if (keep_factor and self.K is not None) else None
        self.K = torch.empty((cap, cap), **f64)
        self.W = torch.empty((cap, cap), **f64)
        self.Tt = torch.empty((cap, 4), **f64)
        self.z = torch.empty(cap, **f64)
        self.Xt = torch.empty((cap, 2), **f64)
        self.y = torch.empty(cap, **f64)
        lib = nat.lib()
        self.work = torch.empty(max(int(lib.mfgp_workspace_bytes(cap)), int(lib.mfgp_append_workspace_bytes(cap))) // 8 + 8,
                                **f64)
        self.cap = cap
        if old is not None:           # the standing factorisation moves into the larger buffers
            K0, W0, T0, z0, n0 = old
            self.K[:n0, :n0].copy_(K0[:n0, :n0])
            self.W[:n0, :n0].copy_(W0[:n0, :n0])
            self.Tt[:n0].copy_(T0[:n0])
            self.z[:n0].copy_(z0[:n0])

    @property
    def N(self):
        return self.NL + self.NH

    def set_params(self, params):
        self.params = dict(params)
        self.pstruct = params_struct(params)

    # -- fit ----------------------------------------------------------------------------------------------------------
    def fit(self, Xt_host, y_host, NL, NH, params, check=True):
        """Upload the training set ([X_L; X_H], [y_L; y_H]) and factorise.  Replaces updt_info
        (gaussian_process.py:229-255, :493-529)."""
        N = NL + NH
        self.params = dict(params)
        self.pstruct = params_struct(params)
        self.NL, self.NH = int(NL), int(NH)
        self.fitted = True
        if N == 0:
            self.npad = 0
            return
        self._reserve(N)
        xt = torch.from_numpy(np.ascontiguousarray(Xt_host, dtype=np.float64).reshape(N, 2))
        yy = torch.from_numpy(np.ascontiguousarray(y_host, dtype=np.float64).reshape(N))
        xh = xt.numpy()
        self._xrange = (float(xh[:, 0].min()), float(xh[:, 0].max()), float(xh[:, 1].min()), float(xh[:, 1].max()))
        self.Xt[:N].copy_(xt, non_blocking=False)
        self.y[:N].copy_(yy, non_blocking=False)
        self.refactor(check=check)

    def refactor(self, check=True):
        """K assembly -> Cholesky -> inverse -> whitening for the data already resident in Xt / y."""
        if self.defer_fit and (not check or self.lazy_check):
            self.npad = nat.npad(self.N)
            self._dirty = True
            self._w_partial = False
            self.fit_id += 1
            self.epoch += 1
            return
        self._dirty = False
        self._w_partial = False
        N = self.N
        lib = nat.lib()
        st = nat.stream_ptr()
        npad = nat.npad(N)
        self.npad = npad
        ld = self.cap
        pp = ctypes.byref(self.pstruct)
        nat.check(lib.mfgp_build_train_cov(nat.ptr(self.Xt), self.NL, self.NH, pp, nat.ptr(self.K), npad, ld,
                                           nat.ptr(self.Tt), st), "mfgp_build_train_cov")
        nat.check(lib.mfgp_cholesky(nat.ptr(self.K), npad, ld, nat.ptr(self.W), ld, nat.ptr(self.info),
                                    nat.ptr(self.work), st), "mfgp_cholesky")
        nat.check(lib.mfgp_tri_inverse(nat.ptr(self.K), npad, ld, nat.ptr(self.W), ld, nat.ptr(self.work), st),
                  "mfgp_tri_inverse")
        nat.check(lib.mfgp_whiten(nat.ptr(self.W), npad, ld, nat.ptr(self.y), self.NL, self.NH, pp, nat.ptr(self.z),
                                  st), "mfgp_whiten")
        self.fit_id += 1
        self.epoch += 1
        if check:
            self.check_factor()

    def ensure_factor(self, need_inverse=True):
        """Bring a deferred / partially finished factorisation up to date (no-op otherwise)."""
        if self._dirty:
            self.defer_fit, keep = False, self.defer_fit
            try:
                self.fit_id -= 1
                self.epoch -= 1
                self.refactor(check=False)
            finally:
                self.defer_fit = keep
        if need_inverse and self._w_partial:
            nat.check(nat.lib().mfgp_tri_inverse(nat.ptr(self.K), self.npad, self.cap, nat.ptr(self.W), self.cap,
                                                 nat.ptr(self.work), nat.stream_ptr()), "mfgp_tri_inverse")
            self._w_partial = False

    def _append_factor(self, NH_old, check=True):
        """Bordered update of L, W, z for the rows appended since NH_old (mfgp_cholesky_append)."""
        lib = nat.lib()
        self.npad = nat.npad(self.N)
        nat.check(lib.mfgp_cholesky_append(nat.ptr(self.Xt), self.NL, int(NH_old), self.NH, ctypes.byref(self.pstruct),
                                           nat.ptr(self.K), self.cap, nat.ptr(self.W), self.cap, nat.ptr(self.y),
                                           nat.ptr(self.z), nat.ptr(self.Tt), nat.ptr(self.info), nat.ptr(self.work),
                                           self.work.numel() * 8, nat.stream_ptr()), "mfgp_cholesky_append")
        self.fit_id += 1
        if check:
            self.check_factor()

    def grid_tables(self, axes):
        """Per-axis factor tables of the separable kernel for a tensor-product grid (`axes` = TensorAxes), rebuilt
        after every refit (mfgp_grid_tables)."""
        self.ensure_factor(need_inverse=False)
        if self._tab is not None and self._tab[0] is axes and self._tab[1] == self.fit_id:
            return self._tab[2:]
        ldt = self.cap
        need = (axes.nx + axes.ny) * ldt * 2
        buf = self._tab[7] if (self._tab is not None and self._tab[7].numel() >= need) else \
            torch.empty(need, dtype=torch.float64, device=self.device)
        TLx = buf[:axes.nx * ldt]
        TLy = buf[axes.nx * ldt:(axes.nx + axes.ny) * ldt]
        THx = buf[(axes.nx + axes.ny) * ldt:(2 * axes.nx + axes.ny) * ldt]
        THy = buf[(2 * axes.nx + axes.ny) * ldt:need]
        nat.check(nat.lib().mfgp_grid_tables(nat.ptr(axes.ux), axes.nx, nat.ptr(axes.uy), axes.ny, nat.ptr(self.Tt),
                                             self.NL, self.NH, self.npad, ctypes.byref(self.pstruct), nat.ptr(TLx),
                                             nat.ptr(TLy), nat.ptr(THx), nat.ptr(THy), ldt, nat.stream_ptr()),
                  "mfgp_grid_tables")
        self._tab = (axes, self.fit_id, TLx, TLy, THx, THy, ldt, buf)
        return self._tab[2:]

    def check_factor(self, force=False):
        if self.lazy_check and not force:
            return
        self.ensure_factor(need_inverse=False)
        self.raise_for_info(int(self.info.item()))

    @staticmethod
    def raise_for_info(info):
        """The Cholesky status word as the exception the reference raises (np.linalg.cholesky, gaussian_process.py:254, :529)."""
        if info < 0:
            raise RuntimeError("libmfgp_b200: the tiled Cholesky kernel gave up waiting for a tile (internal error)")
        if info != 0:
            raise np.linalg.LinAlgError(f"Matrix is not positive definite (pivot {info - 1})")

    def append_hifi(self, X_new_host, y_new_host, check=True):
        """updt / updt_hifi (gaussian_process.py:257-268, :531-542): new points go to the END of [X_L; X_H]; the factor
        is rebuilt from scratch, as in the reference (which does so even when nothing was added)."""
        k = 0 if X_new_host is None else int(np.asarray(X_new_host).reshape(-1, 2).shape[0])
        border = self.incremental and self.fitted and self.N > 0 and self.npad == nat.npad(self.N)
        if border:
            self.ensure_factor()
        NH_old = self.NH
        if k:
            N = self.N
            if N + k > self.cap:
                old_x, old_y = self.Xt, self.y
                self._reserve(N + k, keep_factor=border)
                if N:
                    self.Xt[:N].copy_(old_x[:N])
                    self.y[:N].copy_(old_y[:N])
            xn = np.ascontiguousarray(X_new_host, dtype=np.float64).reshape(k, 2)
            r = self._xrange
            self._xrange = (float(xn[:, 0].min()), float(xn[:, 0].max()), float(xn[:, 1].min()), float(xn[:, 1].max())) if r is None \
                else (min(r[0], float(xn[:, 0].min())), max(r[1], float(xn[:, 0].max())),
                      min(r[2], float(xn[:, 1].min())), max(r[3], float(xn[:, 1].max())))
            self.Xt[N:N + k].copy_(torch.from_numpy(xn))
            self.y[N:N + k].copy_(torch.from_numpy(np.ascontiguousarray(y_new_host, dtype=np.float64).reshape(k)))
            self.NH += k
        if not self.N:
            return
        if border:
            if k:
                self._append_factor(NH_old, check=check)      # nothing appended: the standing factor is still exact
        else:
            self.refactor(check=check)

    # -- posterior ----------------------------------------------------------------------------------------------------
    def posterior(self, xs_dev, mu_out=None, var_out=None, vcache=None, axes=None, g_lo=0, q_out=None):
        """Posterior mean / variance for device-resident points xs_dev[G,2].  Replaces predict
        (gaussian_process.py:121-148, :401-438), diagonal only.  Returns device tensors (mu[G], var[G]).
        If `axes` (TensorAxes) is given the points are the flat x-major range [g_lo, g_lo+G) of that tensor-product
        grid and the separable-kernel path (mfgp_posterior_grid) is used."""
        G = int(xs_dev.shape[0])
        f64 = dict(dtype=torch.float64, device=self.device)
        mu = torch.empty(G, **f64) if mu_out is None else mu_out
        var = torch.empty(G, **f64) if var_out is None else var_out
        lib = nat.lib()
        ldv = 0 if vcache is None else int(vcache.shape[1])
        # incremental mode: the caller's (mu, var) buffers still hold the posterior of the first `covered` rows of the
        # standing factorisation -> add the appended rows only
        key = (mu.data_ptr(), var.data_ptr(), xs_dev.data_ptr(), G, 0 if q_out is None else q_out.data_ptr(), int(g_lo))
        row_lo = 0
        eligible = self.incremental and vcache is None and mu_out is not None and var_out is not None
        if eligible:
            if self._post is not None and self._post[0] == key and self._post[1] == self.epoch \
                    and 0 < self._post[2] <= self.N:
                row_lo = self._post[2]
            self._post = (key, self.epoch, self.N) if self.N > 0 else None
        if row_lo == self.N and row_lo > 0:
            return mu, var                       # nothing was appended since the standing posterior was computed
        plan = None
        if axes is not None and self.N > 0 and vcache is None and self.use_factored:
            plan = self._factored_plan(axes, int(g_lo), G)
        if plan is not None:
            # state key of the stored G'(ix): same geometry / orders / buffers, only appended rows since
            skey = (axes.uid, int(g_lo), G, plan["rxL"], plan["ryL"], plan["rxH"], plan["ryH"], key)
            if self._dirty:
                self._fit_and_posterior_fused(axes, plan, mu, var, q_out)
            else:
                self.ensure_factor()
                upd = row_lo if (row_lo > 0 and self._fstate is not None and self._fstate[0] == skey
                                 and self._fstate[1] == self.epoch and self._fstate[2] == row_lo) else 0
                self._posterior_factored(axes, plan, mu, var, q_out, row_lo=upd)
            self._fstate = (skey, self.epoch, self.N) if self.incremental else None
            return mu, var
        self.ensure_factor()
        if row_lo > 0:
            if axes is not None:
                TLx, TLy, THx, THy, ldt, _ = self.grid_tables(axes)
                nat.check(lib.mfgp_posterior_grid_update(axes.ny, int(g_lo), G, nat.ptr(TLx), nat.ptr(TLy), nat.ptr(THx),
                                                         nat.ptr(THy), ldt, self.NL, self.NH, nat.ptr(self.W), self.npad,
                                                         self.cap, nat.ptr(self.z), ctypes.byref(self.pstruct), row_lo,
                                                         nat.ptr(mu), nat.ptr(var), nat.ptr(q_out), None, 0,
                                                         nat.stream_ptr()), "mfgp_posterior_grid_update")
            else:
                nat.check(lib.mfgp_posterior_update(nat.ptr(xs_dev), G, nat.ptr(self.Tt), self.NL, self.NH, nat.ptr(self.W),
                                                    self.npad, self.cap, nat.ptr(self.z), ctypes.byref(self.pstruct),
                                                    row_lo, nat.ptr(mu), nat.ptr(var), nat.ptr(q_out), None, 0,
                                                    nat.stream_ptr()), "mfgp_posterior_update")
            return mu, var
        if axes is not None and self.N > 0:
            TLx, TLy, THx, THy, ldt, _ = self.grid_tables(axes)
            nat.check(lib.mfgp_posterior_grid(axes.ny, int(g_lo), G, nat.ptr(TLx), nat.ptr(TLy), nat.ptr(THx),
                                              nat.ptr(THy), ldt, self.NL, self.NH, nat.ptr(self.W), self.npad, self.cap,
                                              nat.ptr(self.z), ctypes.byref(self.pstruct), nat.ptr(mu), nat.ptr(var),
                                              nat.ptr(q_out), nat.ptr(vcache), ldv, nat.stream_ptr()),
                      "mfgp_posterior_grid")
            return mu, var
        nat.check(lib.mfgp_posterior(nat.ptr(xs_dev), G, nat.ptr(self.Tt), self.NL, self.NH, nat.ptr(self.W),
                                     self.npad, self.cap, nat.ptr(self.z), ctypes.byref(self.pstruct), nat.ptr(mu),
                                     nat.ptr(var), nat.ptr(q_out), nat.ptr(vcache), ldv, nat.stream_ptr()),
                  "mfgp_posterior")
        return mu, var

    def posterior_cov(self, xs_a, xs_b=None, axes_a=None, g_lo_a=0, axes_b=None, g_lo_b=0, out=None):
        """Joint posterior covariance of the points xs_a[Ga,2] (xs_b None: the symmetric Ga x Ga matrix, exactly symmetric)
        or the cross block between xs_a and xs_b[Gb,2] -- the cov[G,G] of the reference's predict (gaussian_process.py:146,
        :435-436), which the default `posterior` keeps only the diagonal of.  Returns device tensors (mu_a[Ga], C[Ga,Gb]).

        V = W psi^T of each point set comes from `posterior(..., vcache=)` (on a tensor-product grid given by `axes_*` /
        `g_lo_*`: the separable mfgp_posterior_grid), then mfgp_posterior_cov forms C = k** - V_A^T V_B.  mu_a comes from
        that same dense call, so on a grid where `posterior` would take the Chebyshev-factored path it can differ from it in
        the last bits.  C is a view with an even row pitch (the kernel's stores and TMA want 16-byte rows); `out`: a float64
        [Ga, Gb] device tensor with unit column stride and an even row stride to write instead.
        Raises MemoryError, before allocating anything, when V and C do not fit the free device memory; a covariance too
        large to hold whole can be formed in block rows with the cross form, posterior_cov(xs_a[rows], xs_b=xs_a)."""
        self.ensure_factor()
        cross = xs_b is not None
        Ga = int(xs_a.shape[0])
        Gb = int(xs_b.shape[0]) if cross else Ga
        N = self.N
        lda, ldb = Ga + (Ga & 1), Gb + (Gb & 1)
        if out is not None and (tuple(out.shape) != (Ga, Gb) or out.dtype != torch.float64 or out.device != self.device
                                or (Gb > 1 and out.stride(1) != 1) or (Ga > 1 and out.stride(0) % 2)):
            raise ValueError(f"posterior_cov: out must be a float64 [{Ga}, {Gb}] tensor on {self.device} with unit column "
                             "stride and an even row stride")
        need = 8 * ((0 if out is not None else Ga * ldb) + N * (lda + (ldb if cross else 0)) + 2 * (Ga + (Gb if cross else 0)))
        free, _ = torch.cuda.mem_get_info(self.device)
        free += torch.cuda.memory_reserved(self.device) - torch.cuda.memory_allocated(self.device)
        if need > free:
            raise MemoryError(f"posterior_cov: the {Ga} x {Gb} covariance and its V factors need {need / 1e9:.2f} GB, "
                              f"{free / 1e9:.2f} GB of device memory is free; compute it in block rows with the cross form, "
                              "posterior_cov(xs_a[rows], xs_b=xs_a)")
        f64 = dict(dtype=torch.float64, device=self.device)
        Va = torch.empty((N, lda), **f64)
        mu_a, _ = self.posterior(xs_a, vcache=Va, axes=axes_a, g_lo=g_lo_a)
        Vb = None
        if cross:
            Vb = torch.empty((N, ldb), **f64)
            self.posterior(xs_b, vcache=Vb, axes=axes_b, g_lo=g_lo_b)
        C = torch.empty((Ga, ldb), **f64)[:, :Gb] if out is None else out
        ldc = int(C.stride(0)) if Ga > 1 else ldb
        nat.check(nat.lib().mfgp_posterior_cov(nat.ptr(xs_a), Ga, nat.ptr(Va) if N else None, lda,
                                               nat.ptr(xs_b) if cross else None, Gb, nat.ptr(Vb) if (cross and N) else None,
                                               ldb if cross else 0, N, ctypes.byref(self.pstruct), nat.ptr(C), ldc,
                                               nat.stream_ptr()), "mfgp_posterior_cov")
        return mu_a, C

    SAMPLE_MAX_G = 32768      # largest point set posterior_sample factors (mfgp_posterior_cov_factor's npad limit)

    def posterior_sample(self, xs, normals, axes=None, g_lo=0, jitter=None, out=None):
        """Joint posterior draws of the latent f_H at xs[G,2]: F = mu[:, None] + L E with L = chol(C + jitter I) and
        C = k** - V^T V, the symmetric matrix of `posterior_cov`.  `normals`: E, a float64 [G, S] device tensor of
        standard normals.  Returns device tensors (mu[G], F[G, S]); `out`: a float64 [G, S] device tensor with unit column
        stride and an even row stride to write F into.  `jitter` (absolute, default 1e-8 k(0)) is added to C's diagonal.

        Needs C and the factor's scratch (about 16 mfgp_npad(G)^2 bytes) besides V and F: raises MemoryError before
        allocating anything when they do not fit the free device memory, LinAlgError when C + jitter I has a non-positive
        pivot (no retry: pass a larger `jitter`)."""
        self.ensure_factor()
        G = int(xs.shape[0])
        if G > self.SAMPLE_MAX_G:
            raise ValueError(f"posterior_sample: {G} points; at most {self.SAMPLE_MAX_G} can be drawn jointly")
        if normals.dtype != torch.float64 or normals.device != self.device or normals.dim() != 2 or normals.shape[0] != G:
            raise ValueError(f"posterior_sample: normals must be a float64 [{G}, S] tensor on {self.device}")
        S = int(normals.shape[1])
        if out is not None and (tuple(out.shape) != (G, S) or out.dtype != torch.float64 or out.device != self.device
                                or (S > 1 and out.stride(1) != 1) or (G > 1 and out.stride(0) % 2)):
            raise ValueError(f"posterior_sample: out must be a float64 [{G}, {S}] tensor on {self.device} with unit column "
                             "stride and an even row stride")
        p = self.params
        if jitter is None:
            jitter = 1e-8 * ((p["rho"] ** 2 * p["s_L"] + p["s_H"]) if p["multi"] else p["s_H"])
        jitter = float(jitter)
        if not (jitter >= 0.0 and np.isfinite(jitter)):
            raise ValueError(f"posterior_sample: jitter must be finite and >= 0, got {jitter}")
        if S < 1:
            raise ValueError("posterior_sample: normals must have at least one column")
        f64 = dict(dtype=torch.float64, device=self.device)
        if G == 0:
            return torch.empty(0, **f64), (torch.empty((0, S), **f64) if out is None else out)
        lib = nat.lib()
        npad = nat.npad(G)
        work_bytes = int(lib.mfgp_workspace_bytes(npad))
        lde = S + (S & 1)
        need = (8 * (2 * npad * npad + self.N * (G + (G & 1)) + 2 * G + (0 if out is not None else G * lde))
                + work_bytes)
        free, _ = torch.cuda.mem_get_info(self.device)
        free += torch.cuda.memory_reserved(self.device) - torch.cuda.memory_allocated(self.device)
        if need > free:
            raise MemoryError(f"posterior_sample: {G} points x {S} draws need {need / 1e9:.2f} GB (covariance, its factor's "
                              f"scratch, V, F), {free / 1e9:.2f} GB of device memory is free")
        C = torch.empty((npad, npad), **f64)
        mu, _ = self.posterior_cov(xs, axes_a=axes, g_lo_a=g_lo, out=C[:G, :G])
        W = torch.empty((npad, npad), **f64)
        work = torch.empty(work_bytes // 8 + 1, **f64)
        info = torch.zeros(1, dtype=torch.int32, device=self.device)
        st = nat.stream_ptr()
        nat.check(lib.mfgp_posterior_cov_factor(nat.ptr(C), G, npad, npad, jitter, nat.ptr(W), npad, nat.ptr(info),
                                                nat.ptr(work), st), "mfgp_posterior_cov_factor")
        del W, work
        code = int(info.item())
        if code < 0:
            self.raise_for_info(code)
        if code > 0:
            raise np.linalg.LinAlgError(f"posterior_sample: the posterior covariance plus jitter {jitter:.3g} is not positive "
                                        f"definite (pivot {code - 1}); pass a larger jitter")
        F = torch.empty((G, lde), **f64)[:, :S] if out is None else out
        # the kernel's TMA reads E with a 16-byte aligned base and an even row pitch; other layouts are copied once
        if (S == 1 or normals.stride(1) == 1) and (G == 1 or normals.stride(0) % 2 == 0) and normals.data_ptr() % 16 == 0:
            E, ld_e = normals, (int(normals.stride(0)) if G > 1 else lde)
        else:
            E = torch.empty((G, lde), **f64)[:, :S].copy_(normals)
            ld_e = lde
        ldf = int(F.stride(0)) if G > 1 else lde
        nat.check(lib.mfgp_posterior_sample(nat.ptr(C), G, npad, nat.ptr(mu), nat.ptr(E), ld_e, S, nat.ptr(F), ldf, st),
                  "mfgp_posterior_sample")
        return mu, F

    # -- pathwise posterior draws on tensor-product grids (gp_sample_grid.cu) -------------------------------------------------
    def _grid_sample_plan(self, axes):
        """Box (the grid and the training points), Chebyshev orders and node roots Q = DCT K_nodes^(1/2) of the pathwise grid
        sampler, uploaded; cached per grid, hyper-parameters and training hull.  ValueError when an order would exceed 64."""
        p = self.params
        if self.N:
            t = self._training_range()
            box = (min(axes.xlo, t[0]), max(axes.xhi, t[1]), min(axes.ylo, t[2]), max(axes.yhi, t[3]))
        else:
            box = (axes.xlo, axes.xhi, axes.ylo, axes.yhi)
        key = (axes.uid, box, p["l_L"], p["l_H"], int(p["multi"]))
        if self._splan is not None and self._splan["key"] == key:
            return self._splan
        orders = grid_sample_orders(p, box)
        f64 = dict(dtype=torch.float64, device=self.device)
        Q = {}
        for part, length in ((("L", p["l_L"]), ("H", p["l_H"])) if p["multi"] else (("H", p["l_H"]),)):
            for ax, lo, hi in (("x", box[0], box[1]), ("y", box[2], box[3])):
                Q[part + ax] = torch.from_numpy(node_root(length, lo, hi, orders[part + ax])).to(**f64)
        rxL, ryL = orders.get("Lx", 0), orders.get("Ly", 0)
        rxH, ryH = orders["Hx"], orders["Hy"]
        self._splan = dict(key=key, box=box, orders=(rxL, ryL, rxH, ryH), Q=Q, d0=rxL * ryL + rxH * ryH,
                           rx=max(rxL, rxH), ry=max(ryL, ryH))
        return self._splan

    def grid_sample_dim(self, axes):
        """Rows d of the normals that posterior_sample_grid takes for the tensor-product grid `axes` (TensorAxes)."""
        self.ensure_factor(need_inverse=False)
        return self._grid_sample_plan(axes)["d0"] + self.N

    def posterior_sample_grid(self, axes, normals, ix0=0, ncols=None, out=None):
        """Joint posterior draws of the latent f_H over the whole columns [ix0, ix0 + ncols) of the tensor-product grid `axes`
        (TensorAxes), by pathwise conditioning (mfgp_grid_sample_coef, mfgp_grid_sample_eval): F = mu + A E with A A^T the
        posterior covariance of the whole grid.  `normals`: E, a float64 [d, S] device tensor of standard normals,
        d = grid_sample_dim(axes) (layout: include/mfgp_b200.h).  Returns F[ncols * ny, S] (row (ix - ix0) * ny + iy); `out`: a
        float64 tensor of that shape with unit column stride and an even row stride to write it into.  The same E gives the
        same bits for the whole grid and for any column slice of it.
        Raises MemoryError before allocating anything when the draws and the scratch do not fit the free device memory."""
        self.ensure_factor(need_inverse=True)
        plan = self._grid_sample_plan(axes)
        ix0 = int(ix0)
        ncols = axes.nx - ix0 if ncols is None else int(ncols)
        if not (0 <= ix0 and ncols >= 1 and ix0 + ncols <= axes.nx):
            raise ValueError(f"posterior_sample_grid: columns [{ix0}, {ix0 + ncols}) are not inside the grid's {axes.nx}")
        d = plan["d0"] + self.N
        if (normals.dtype != torch.float64 or normals.device != self.device or normals.dim() != 2 or normals.shape[0] != d
                or normals.shape[1] < 1):
            raise ValueError(f"posterior_sample_grid: normals must be a float64 [{d}, S] tensor on {self.device}, S >= 1")
        S = int(normals.shape[1])
        rows = ncols * axes.ny
        if out is not None and (tuple(out.shape) != (rows, S) or out.dtype != torch.float64 or out.device != self.device
                                or (S > 1 and out.stride(1) != 1) or (rows > 1 and out.stride(0) % 2) or out.data_ptr() % 16):
            raise ValueError(f"posterior_sample_grid: out must be a float64 [{rows}, {S}] tensor on {self.device} with unit "
                             "column stride, an even row stride and a 16-byte aligned base")
        lib = nat.lib()
        rxL, ryL, rxH, ryH = plan["orders"]
        rx, ry = plan["rx"], plan["ry"]
        lde = S + (S & 1)
        copy_e = not ((S == 1 or normals.stride(1) == 1) and (d == 1 or normals.stride(0) % 2 == 0)
                      and normals.data_ptr() % 16 == 0)
        cw = int(lib.mfgp_grid_sample_coef_workspace_bytes(self.N, rxL, ryL, rxH, ryH, S))
        ew = int(lib.mfgp_grid_sample_eval_workspace_bytes(ncols, axes.ny, rx, ry, S))
        ncoef = S * ry * (-(-rx // 4) * 4)
        need = cw + ew + 8 * (ncoef + (rows * lde if out is None else 0) + (d * lde if copy_e else 0)) + 1024
        free, _ = torch.cuda.mem_get_info(self.device)
        free += torch.cuda.memory_reserved(self.device) - torch.cuda.memory_allocated(self.device)
        if need > free:
            raise MemoryError(f"posterior_sample_grid: {ncols} columns x {axes.ny} rows x {S} draws need {need / 1e9:.2f} GB "
                              f"(draws, coefficients, scratch), {free / 1e9:.2f} GB of device memory is free; draw the grid in "
                              "column slices (ix0, ncols) with the same normals")
        f64 = dict(dtype=torch.float64, device=self.device)
        if copy_e:
            E, lde_e = torch.empty((d, lde), **f64), lde
            E[:, :S].copy_(normals)
        else:
            E, lde_e = normals, (int(normals.stride(0)) if d > 1 else lde)
        F = torch.empty((rows, lde), **f64)[:, :S] if out is None else out
        ldf = int(F.stride(0)) if rows > 1 else lde
        C = torch.empty(ncoef + 2, **f64)
        work = torch.empty(max(cw, ew) // 8 + 2, **f64)
        Q = plan["Q"]
        st = nat.stream_ptr()
        xlo, xhi, ylo, yhi = (ctypes.c_double(v) for v in plan["box"])
        N = self.N
        nat.check(lib.mfgp_grid_sample_coef(nat.ptr(self.Xt) if N else None, nat.ptr(self.y) if N else None, self.NL, self.NH,
                                            nat.ptr(self.W) if N else None, self.npad if N else 0, self.cap if N else 0,
                                            ctypes.byref(self.pstruct), rxL, ryL, rxH, ryH, xlo, xhi, ylo, yhi,
                                            nat.ptr(Q.get("Lx")), nat.ptr(Q.get("Ly")), nat.ptr(Q["Hx"]), nat.ptr(Q["Hy"]),
                                            nat.ptr(E), lde_e, S, nat.ptr(C), nat.ptr(work), work.numel() * 8, st),
                  "mfgp_grid_sample_coef")
        nat.check(lib.mfgp_grid_sample_eval(nat.ptr(axes.ux), axes.nx, nat.ptr(axes.uy), axes.ny, ix0, ncols, xlo, xhi, ylo, yhi,
                                            rx, ry, nat.ptr(C), S, ctypes.c_double(self.params["mean_H"]), nat.ptr(F), ldf,
                                            nat.ptr(work), work.numel() * 8, st), "mfgp_grid_sample_eval")
        return F

    def posterior_sample_grid_coef(self, axes, normals, extra_bytes=0):
        """The coefficients of the draws posterior_sample_grid evaluates, without evaluating them: C[S, ry * kpad] (term (l, k) in
        column l * kpad + k, kpad = rx rounded up to 4) with F_s = mean_H + sum T_l(ty) T_k(tx) C[s][l][k] on plan["box"].
        Returns (C, plan).  `extra_bytes`: the caller's own allocations, included in the memory check (MemoryError before
        anything is allocated)."""
        self.ensure_factor(need_inverse=True)
        plan = self._grid_sample_plan(axes)
        d = plan["d0"] + self.N
        if (normals.dtype != torch.float64 or normals.device != self.device or normals.dim() != 2 or normals.shape[0] != d
                or normals.shape[1] < 1):
            raise ValueError(f"posterior_sample_grid: normals must be a float64 [{d}, S] tensor on {self.device}, S >= 1")
        S = int(normals.shape[1])
        lib = nat.lib()
        rxL, ryL, rxH, ryH = plan["orders"]
        R = plan["ry"] * (-(-plan["rx"] // 4) * 4)
        lde = S + (S & 1)
        copy_e = not ((S == 1 or normals.stride(1) == 1) and (d == 1 or normals.stride(0) % 2 == 0)
                      and normals.data_ptr() % 16 == 0)
        cw = int(lib.mfgp_grid_sample_coef_workspace_bytes(self.N, rxL, ryL, rxH, ryH, S))
        need = cw + int(extra_bytes) + 8 * (S * R + (d * lde if copy_e else 0)) + 1024
        free, _ = torch.cuda.mem_get_info(self.device)
        free += torch.cuda.memory_reserved(self.device) - torch.cuda.memory_allocated(self.device)
        if need > free:
            raise MemoryError(f"posterior_sample_grid: {S} draws need {need / 1e9:.2f} GB (coefficients, moments, scratch), "
                              f"{free / 1e9:.2f} GB of device memory is free")
        f64 = dict(dtype=torch.float64, device=self.device)
        if copy_e:
            E, lde_e = torch.empty((d, lde), **f64), lde
            E[:, :S].copy_(normals)
        else:
            E, lde_e = normals, (int(normals.stride(0)) if d > 1 else lde)
        C = torch.empty((S, R), **f64)
        work = torch.empty(cw // 8 + 2, **f64)
        Q = plan["Q"]
        xlo, xhi, ylo, yhi = (ctypes.c_double(v) for v in plan["box"])
        N = self.N
        nat.check(lib.mfgp_grid_sample_coef(nat.ptr(self.Xt) if N else None, nat.ptr(self.y) if N else None, self.NL, self.NH,
                                            nat.ptr(self.W) if N else None, self.npad if N else 0, self.cap if N else 0,
                                            ctypes.byref(self.pstruct), rxL, ryL, rxH, ryH, xlo, xhi, ylo, yhi,
                                            nat.ptr(Q.get("Lx")), nat.ptr(Q.get("Ly")), nat.ptr(Q["Hx"]), nat.ptr(Q["Hy"]),
                                            nat.ptr(E), lde_e, S, nat.ptr(C), nat.ptr(work), work.numel() * 8,
                                            nat.stream_ptr()), "mfgp_grid_sample_coef")
        return C, plan

    # -- factored posterior on tensor-product grids (gp_factored.cu) ---------------------------------------------------------
    def _training_range(self):
        """(xmin, xmax, ymin, ymax) of the training points, tracked on the host by fit / append_hifi."""
        if self._xrange is None:
            xt = self.Xt[:self.N]
            lo, hi = xt.min(dim=0).values.tolist(), xt.max(dim=0).values.tolist()
            self._xrange = (lo[0], hi[0], lo[1], hi[1])
        return self._xrange

    def _cheb_orders(self, axes, p, xlo, xhi):
        """(rxL, ryL, rxH, ryH) or None for the column range whose x values span [xlo, xhi]; cached while the training
        points stay inside the hull the orders were computed for."""
        ylo, yhi = axes.ylo, axes.yhi
        t = self._training_range()
        c = self._forders
        if c is not None and c[0] == (axes.uid, xlo, xhi, p["l_L"], p["l_H"], p["multi"]) and c[1][0] <= t[0] and c[1][1] >= t[1] \
                and c[1][2] <= t[2] and c[1][3] >= t[3]:
            return c[2]
        mx, my = 0.05 * (axes.xhi - axes.xlo), 0.05 * (yhi - ylo)      # a margin, so that a few new samples do not invalidate it
        hull = (min(t[0], axes.xlo) - mx, max(t[1], axes.xhi) + mx, min(t[2], ylo) - my, max(t[3], yhi) + my)
        rxH = chebyshev_order(p["l_H"], xlo, xhi, hull[0], hull[1])
        ryH = chebyshev_order(p["l_H"], ylo, yhi, hull[2], hull[3])
        rxL = ryL = 0
        ok = rxH is not None and ryH is not None
        if ok and p["multi"]:
            rxL = chebyshev_order(p["l_L"], xlo, xhi, hull[0], hull[1])
            ryL = chebyshev_order(p["l_L"], ylo, yhi, hull[2], hull[3])
            ok = rxL is not None and ryL is not None
        orders = (rxL, ryL, rxH, ryH) if ok else None
        self._ftrunc = None
        if ok and TRUNCATE:
            parts = [(chebyshev_envelope(p["l_H"], xlo, xhi, hull[0], hull[1], rxH),
                      chebyshev_envelope(p["l_H"], ylo, yhi, hull[2], hull[3], ryH))]
            if p["multi"]:
                parts.append((chebyshev_envelope(p["l_L"], xlo, xhi, hull[0], hull[1], rxL),
                              chebyshev_envelope(p["l_L"], ylo, yhi, hull[2], hull[3], ryL)))
            kp = -(-max(rxL, rxH) // 4) * 4
            parts = [(np.pad(ax, (0, kp - ax.size)), ay) for ax, ay in parts]
            self._ftrunc = chebyshev_truncation(parts, kp, max(ryL, ryH))
        self._forders = ((axes.uid, xlo, xhi, p["l_L"], p["l_H"], p["multi"]), hull, orders)
        return orders

    def _factored_plan(self, axes, g_lo, G):
        """Chebyshev orders + cost model.  None: keep the dense kernel (range is not whole columns, orders too large for
        the 64-term budget, or the dense triangular products are cheaper -- small grids).
        The x expansion covers only the interval of the REQUESTED columns: a grid shard (whole-column slice, grid sharding)
        needs a lower order in x than the whole grid, so its right-hand-side count R = ry * rx -- and with it the forward
        substitution, the one part of the fit that is not replicated work -- shrinks with the number of ranks."""
        ny = axes.ny
        if ny < 2 or axes.nx < 2 or g_lo % ny or G % ny:
            return None
        p = self.params
        N = self.npad
        dense = 0.5 * G * N * N
        if self.factored_min_gain > 0 and dense < 4e9:      # the dense kernel needs well under a millisecond: no plan
            return None
        ix0, ncols = g_lo // ny, G // ny
        if ncols < 2:
            return None
        xs = axes.ux_host[ix0:ix0 + ncols]
        xlo, xhi = float(xs.min()), float(xs.max())
        if not (xhi > xlo):
            return None
        key = (axes.uid, g_lo, G, self.npad, p["l_L"], p["l_H"], p["multi"], self.factored_min_gain)
        orders = self._cheb_orders(axes, p, xlo, xhi)
        if self._fplan is not None and self._fplan[0] == key and self._fplan[2] == orders and self._fplan[3] is self._ftrunc:
            return self._fplan[1]          # (same orders AND the truncation table they were cached with)
        plan = None
        if orders is not None:
            rxL, ryL, rxH, ryH = orders
            ry, kp = max(ryL, ryH), -(-max(rxL, rxH) // 4) * 4         # both kernel parts share one Chebyshev basis
            R = ry * kp
            fact = 0.5 * N * N * R + ncols * N * R + ncols * N * 64 * 64 + G * 64 * 64
            if fact * self.factored_min_gain < dense:
                chunk = max(64, min(-(-ncols // 64) * 64, ((1 << 28) // max(self.cap * max(ryL, ryH), 1)) // 64 * 64))   # <= 2 GiB of Y'
                plan = dict(rxL=rxL, ryL=ryL, rxH=rxH, ryH=ryH, xlo=xlo, xhi=xhi, ylo=axes.ylo, yhi=axes.yhi,
                            ix0=ix0, ncols=ncols, chunk=chunk, macs=fact, dense_macs=dense, kx=self._ftrunc)
        self._fplan = (key, plan, orders, self._ftrunc)
        return plan


    def _wsalloc(self, n, slack=8):
        """n doubles of workspace (+ `slack`); with GUARD: exactly n, inside canary margins that check_guards() inspects."""
        if not GUARD:
            return torch.empty(n + slack, dtype=torch.float64, device=self.device)
        big = torch.full((n + 1024,), _CANARY, dtype=torch.float64, device=self.device)
        self._guards = [g for g in getattr(self, "_guards", []) if g[0] is not None]
        self._guards.append((big, n))
        return big[512:512 + n]

    def check_guards(self):
        """True iff no canary of a GUARD-mode workspace has been overwritten."""
        torch.cuda.synchronize(self.device)
        return all(bool((big[:512] == _CANARY).all().item()) and bool((big[512 + n:] == _CANARY).all().item())
                   for big, n in getattr(self, "_guards", []))

    def _factored_work(self, axes, plan):
        # sized for the CAPACITY of the factor buffers, so appended samples do not reallocate gigabytes every iteration
        need = int(nat.lib().mfgp_factored_workspace_bytes(self.cap, plan["ncols"], axes.ny, plan["rxL"], plan["ryL"],
                                                           plan["rxH"], plan["ryH"], plan["chunk"]))
        if self._fwork is None or self._fwork.numel() * 8 < need:
            self._fwork = self._wsalloc(need // 8)
        return self._fwork

    def _factored_stores(self, plan):
        """Persistent G'(ix) / z^T Y buffers of the incremental factored update (only kept in incremental mode)."""
        if not self.incremental:
            return None, None
        lib = nat.lib()
        nG = plan["ncols"] * 64 * 64
        nH = int(lib.mfgp_factored_rhs_cols(plan["rxL"], plan["ryL"], plan["rxH"], plan["ryH"]))     # >= ry * kpad
        if self._fG is None or self._fG.numel() < nG:
            self._fG = self._wsalloc(nG, 0)
        if self._fHz is None or self._fHz.numel() < nH:
            self._fHz = self._wsalloc(nH, 0)
        return self._fG, self._fHz

    def _fit_and_posterior_fused(self, axes, plan, mu, var, q_out):
        """From-scratch iteration on a tensor grid in one pass: K -> (L, diagonal-block inverses) with the right-hand sides
        [B | y - mean] forward-substituted inside the same tile-dataflow kernel -> steps 4-6 (see include/mfgp_b200.h)."""
        lib = nat.lib()
        st = nat.stream_ptr()
        pp = ctypes.byref(self.pstruct)
        npad, ld = self.npad, self.cap
        o = (plan["rxL"], plan["ryL"], plan["rxH"], plan["ryH"])
        work = self._factored_work(axes, plan)
        geom = (ctypes.c_double(plan["xlo"]), ctypes.c_double(plan["xhi"]), ctypes.c_double(plan["ylo"]),
                ctypes.c_double(plan["yhi"]), plan["chunk"])
        # Gram route of steps 4 + 5: M = Y^T Y is accumulated inside the factorisation kernel (NULL: direct route), and the
        # right-hand sides may use the truncated column layout (not with the incremental stores, which keep the uniform one)
        kx = plan.get("kx") if (FUSED_GRAM and not self.incremental) else None
        M, R = None, 0
        if FUSED_GRAM:
            if kx is not None:
                kxp = ctypes.c_void_p(kx.ctypes.data)
                R = int(lib.mfgp_factored_rhs_cols_trunc(int(kx.size), kxp))
                M = lib.mfgp_factored_gram_target(axes.nx, axes.ny, plan["ix0"], plan["ncols"], self.NL, self.NH, npad, pp, *o,
                                                  plan["chunk"], kxp, R, nat.ptr(work), work.numel() * 8)
            if not M:
                kx, kxp = None, None
                R = int(lib.mfgp_factored_rhs_cols(*o))
                M = lib.mfgp_factored_gram_target(axes.nx, axes.ny, plan["ix0"], plan["ncols"], self.NL, self.NH, npad, pp, *o,
                                                  plan["chunk"], None, R, nat.ptr(work), work.numel() * 8)
        else:
            kx, kxp = None, None
            R = int(lib.mfgp_factored_rhs_cols(*o))
        if self._fB is None or self._fB.numel() < self.cap * R:
            self._fB = self._wsalloc(self.cap * R, 0)
        nat.check(lib.mfgp_build_train_cov(nat.ptr(self.Xt), self.NL, self.NH, pp, nat.ptr(self.K), npad, ld,
                                           nat.ptr(self.Tt), st), "mfgp_build_train_cov")
        nat.check(lib.mfgp_factored_prepare_trunc(nat.ptr(axes.ux), axes.nx, nat.ptr(axes.uy), axes.ny, plan["ix0"], plan["ncols"],
                                                  nat.ptr(self.Xt), nat.ptr(self.y), self.NL, self.NH, npad, pp, *o, *geom,
                                                  kxp if kx is not None else None, nat.ptr(self._fB), R, nat.ptr(work),
                                                  work.numel() * 8, st), "mfgp_factored_prepare")
        ev = self.profile_events          # bench.py: (start, stop) CUDA events around the dominant kernel
        if ev is not None:
            ev[0].record()
        cneed = int(lib.mfgp_cholesky_solve_gram_workspace_bytes(self.cap, R))
        if self._cwork is None or self._cwork.numel() * 8 < cneed:
            self._cwork = self._wsalloc(cneed // 8)
        nat.check(lib.mfgp_cholesky_solve_gram(nat.ptr(self.K), npad, ld, nat.ptr(self.W), ld, nat.ptr(self.info),
                                               nat.ptr(self._fB), R, R, ctypes.c_void_p(M), R, nat.ptr(self._cwork),
                                               self._cwork.numel() * 8, st), "mfgp_cholesky_solve_gram")
        if ev is not None:
            ev[1].record()
        Gs, Hs = self._factored_stores(plan)
        if M:
            nat.check(lib.mfgp_posterior_grid_factored_solved_gram(
                nat.ptr(axes.ux), axes.nx, nat.ptr(axes.uy), axes.ny, plan["ix0"], plan["ncols"], nat.ptr(self.Xt), self.NL,
                self.NH, npad, pp, *o, *geom, kxp if kx is not None else None, nat.ptr(self._fB), R, nat.ptr(self.z), nat.ptr(mu),
                nat.ptr(var), nat.ptr(q_out), nat.ptr(Gs), nat.ptr(Hs), nat.ptr(work), work.numel() * 8, st),
                "mfgp_posterior_grid_factored_solved_gram")
        else:
            nat.check(lib.mfgp_posterior_grid_factored_solved(
                nat.ptr(axes.ux), axes.nx, nat.ptr(axes.uy), axes.ny, plan["ix0"], plan["ncols"], nat.ptr(self.Xt), self.NL,
                self.NH, npad, pp, *o, *geom, nat.ptr(self._fB), R, nat.ptr(self.z), nat.ptr(mu), nat.ptr(var), nat.ptr(q_out),
                nat.ptr(Gs), nat.ptr(Hs), nat.ptr(work), work.numel() * 8, st), "mfgp_posterior_grid_factored_solved")
        self.rhs_cols = (int(kx.sum()) if kx is not None else max(plan["ryL"], plan["ryH"]) * (-(-max(plan["rxL"], plan["rxH"]) // 4) * 4), R)
        self.fused_gram = bool(M)
        self._dirty = False
        self._w_partial = True

    def _posterior_factored(self, axes, plan, mu, var, q_out, row_lo=0):
        """Full factored posterior from W, or (row_lo > 0, stores valid) the incremental update with the appended rows."""
        lib = nat.lib()
        work = self._factored_work(axes, plan)
        Gs, Hs = self._factored_stores(plan)
        geom = (ctypes.c_double(plan["xlo"]), ctypes.c_double(plan["xhi"]), ctypes.c_double(plan["ylo"]),
                ctypes.c_double(plan["yhi"]), plan["chunk"])
        o = (plan["rxL"], plan["ryL"], plan["rxH"], plan["ryH"])
        if row_lo > 0 and Gs is not None:
            nat.check(lib.mfgp_posterior_grid_factored_update(
                nat.ptr(axes.ux), axes.nx, nat.ptr(axes.uy), axes.ny, plan["ix0"], plan["ncols"], nat.ptr(self.Xt), self.NL,
                self.NH, int(row_lo), nat.ptr(self.W), self.npad, self.cap, nat.ptr(self.z), ctypes.byref(self.pstruct), *o, *geom,
                nat.ptr(mu), nat.ptr(var), nat.ptr(q_out), nat.ptr(Gs), nat.ptr(Hs), nat.ptr(work), work.numel() * 8,
                nat.stream_ptr()), "mfgp_posterior_grid_factored_update")
            return
        kx = plan.get("kx") if Gs is None else None      # truncated column layout (not with the incremental stores)
        nat.check(lib.mfgp_posterior_grid_factored_trunc(
            nat.ptr(axes.ux), axes.nx, nat.ptr(axes.uy), axes.ny, plan["ix0"], plan["ncols"], nat.ptr(self.Xt), self.NL, self.NH,
            nat.ptr(self.W), self.npad, self.cap, nat.ptr(self.z), ctypes.byref(self.pstruct), *o, *geom,
            ctypes.c_void_p(kx.ctypes.data) if kx is not None else None, nat.ptr(mu), nat.ptr(var),
            nat.ptr(q_out), nat.ptr(Gs), nat.ptr(Hs), nat.ptr(work), work.numel() * 8, nat.stream_ptr()),
            "mfgp_posterior_grid_factored")

    # -- hyper-parameter training ------------------------------------------------------------------------------------
    def nlml_grad(self):
        """(NLML, gradient[10]) of the standing fit (mfgp_nlml_grad; gaussian_process.py:81-105, :344-384 and the autograd
        gradient behind train :107-119, :386-399).  Host floats / numpy array; one device->host copy."""
        if self.N == 0:
            raise ValueError("likelihood of an empty model")
        self.ensure_factor(need_inverse=True)
        self.check_factor(force=True)             # LinAlgError where the reference's np.linalg.cholesky raises (:100, :380)
        lib = nat.lib()
        need = int(lib.mfgp_nlml_workspace_bytes(self.npad))
        if self._twork is None or self._twork.numel() * 8 < need:
            self._twork = torch.empty(need // 8 + 8, dtype=torch.float64, device=self.device)
        out = torch.empty(10, dtype=torch.float64, device=self.device)
        nat.check(lib.mfgp_nlml_grad(nat.ptr(self.K), self.npad, self.cap, nat.ptr(self.W), self.cap, nat.ptr(self.z),
                                     nat.ptr(self.Tt), self.NL, self.NH, ctypes.byref(self.pstruct), nat.ptr(out),
                                     nat.ptr(self._twork), self._twork.numel() * 8, nat.stream_ptr()), "mfgp_nlml_grad")
        h = out.cpu().numpy()
        return float(h[0]), h[1:].copy()

    def clone(self):
        self.ensure_factor()
        other = DeviceGP(self.device)
        other.NL, other.NH, other.npad, other.cap = self.NL, self.NH, self.npad, self.cap
        other.params = None if self.params is None else dict(self.params)
        other.pstruct = None if self.params is None else params_struct(self.params)
        other.fitted = self.fitted
        for name in ("Xt", "y", "K", "W", "Tt", "z", "work"):
            t = getattr(self, name)
            setattr(other, name, None if t is None else t.clone())
        other.info = self.info.clone()
        other.fit_id = self.fit_id
        other.incremental = self.incremental
        other.use_factored = self.use_factored
        other.factored_min_gain = self.factored_min_gain
        other.lazy_check = self.lazy_check
        other.defer_fit = self.defer_fit
        other.epoch = self.epoch
        return other
