"""simulator.py -- drop-in for the reference module of the same name with the hot path on a B200.

Same public names and signatures as the reference's simulator.py: the model factories (`init_MFGP`, `init_SFGP`,
:47-102), the coverage functions (`in_polygon`, `poly_area`, `in_box`, `voronoi_bounded`, `compute_loss`,
`compute_centroids`, `compute_max_var`, `compute_sample_points`, `compute_sample_clusters`, `compute_sample_tsp`,
:105-454), the decision rules (:457-500) and the four control algorithms (`lloyd`, `periodic`, `todescato`, `choi`,
:508-1161) with their 12-argument signature and list-of-dict log rows.

What runs where: the iteration loops, the O(agents) decision rules, Qhull (scipy.spatial.Voronoi, as in the
reference) and CSV/log bookkeeping stay host Python; the GP fit + posterior over the grid, the membership of every
grid point in the Voronoi cells, the per-cell sums / max-variance arg-max and the Choi greedy planner run in
libmfgp_b200 (include/mfgp_b200.h).  The grid stays resident in HBM for the whole simulation; per iteration only the
new samples and O(agents) results cross PCIe.  There is no CPU fallback for any of the device steps.

Deliberate differences from the reference (documented in DESIGN.md):
  * `var_star` is the posterior variance VECTOR (the reference passes a G x G covariance and takes np.diag);
    `compute_max_var` accepts either.
  * optional keyword arguments `rng=` (object with .random(), default: the `random` module) and `noise_rng=`
    (numpy Generator, default: a fresh `np.random.default_rng()` per sample as in the reference) make runs replayable.
  * the Choi TSP tour comes from a deterministic device planner (nearest neighbour + 2-opt, csrc/tsp.cu) instead of
    mlrose's genetic algorithm, whose tours are not reproducible (unpinned third-party routine); MFGP_TSP=mlrose
    selects mlrose when it is installed.
"""
import copy
import os
import random
import sys

import numpy as np
import torch

from . import _coverage as cv
from . import _native as nat
from ._coverage import BoundedVoronoi, CoverageGrid
from .gaussian_process import MFGP, SFGP, prior_variance

eps = cv.EPS

line_break = "\n" + "".join(["-" for i in range(100)]) + "\n"
slash_break = "\n" + "".join(["/" for i in range(100)]) + "\n"


#######################################################################################################################
# Helper functions
#######################################################################################################################

def _prior_arrays(prior):
    if prior is not None and len(prior) > 0:
        p = np.vstack(prior.values.tolist()) if hasattr(prior, "values") else np.asarray(prior, dtype=np.float64)
        return np.reshape(p[:, [0, 1]], (-1, 2)), np.reshape(p[:, 2], (-1, 1))
    return np.empty([0, 2]), np.empty([0, 1])


def _hyp_array(hyp):
    return np.array(hyp.values.tolist()[0]) if hasattr(hyp, "values") else np.asarray(hyp, dtype=np.float64).reshape(-1)


def _hyp_len(hyp):
    return len(hyp.columns) if hasattr(hyp, "columns") else np.asarray(hyp).reshape(-1).size


def init_MFGP(hyp, prior):
    """reference simulator.py:47-75 -- the prior, if any, conditions the LOFI level."""
    X_L, y_L = _prior_arrays(prior)
    model = MFGP(X_L, y_L, np.empty([0, 2]), np.empty([0, 1]), 1, 1)
    model.hyp = _hyp_array(hyp)
    return model


def init_SFGP(hyp, prior):
    """reference simulator.py:78-102."""
    X, y = _prior_arrays(prior)
    model = SFGP(X, y, 1)
    model.hyp = _hyp_array(hyp)
    return model


_grid_cache = {}


def _grid_for(arr):
    """Device-resident copy of a grid given as x_star[G,2] or truth_arr[G,3] (third column = ground truth), cached on
    the identity of the host array so the reference-style free functions (which receive `truth_arr` / `x_star` on every
    call) do not re-upload it.  The host array is kept alive by the cache so its address cannot be recycled."""
    arr = np.asarray(arr)
    key = cv.host_array_key(arr)
    hit = _grid_cache.get(key)
    if hit is not None:
        return hit[0]
    if len(_grid_cache) > 8:
        _grid_cache.clear()
    g = CoverageGrid(arr[:, [0, 1]], arr[:, 2] if arr.shape[1] >= 3 else None)
    # extent of the grid (simulator.py:264-271 clamps the centroids to it), computed once per grid, not per call
    g.extent = (np.amin(arr[:, 0]), np.amax(arr[:, 0]), np.amin(arr[:, 1]), np.amax(arr[:, 1]))
    _grid_cache[key] = (g, arr)
    return g


def in_polygon(xq, yq, xv, yv):
    """reference simulator.py:105-124 (matplotlib crossings test), evaluated on the device."""
    shape = np.asarray(xq).shape
    pts = np.column_stack((np.asarray(xq, dtype=np.float64).reshape(-1), np.asarray(yq, dtype=np.float64).reshape(-1)))
    poly = np.column_stack((np.asarray(xv, dtype=np.float64).reshape(-1), np.asarray(yv, dtype=np.float64).reshape(-1)))
    if pts.shape[0] == 0:
        return np.zeros(shape, dtype=bool)
    part = cv.polygon_partition(np.zeros((1, 2)), [poly])
    res = CoverageGrid(pts).assign_reduce(lloyd_vor=part, want_members=True, tie_tol=float("inf"))
    return (res["members"][:, 0].cpu().numpy() & 1).astype(bool).reshape(shape)


def poly_area(x, y):
    """reference simulator.py:127-136."""
    return 0.5 * np.abs(np.dot(x, np.roll(y, 1)) - np.dot(y, np.roll(x, 1)))


in_box = cv.in_box


# How the bounded Voronoi cells are built (MFGP_VORONOI / simulator.VORONOI):
#   "auto"  (default) cells clipped ON THE DEVICE (cov_voronoi_clip); scipy/Qhull -- the reference's builder -- runs on the
#           host only for the passes that meet a grid point within TIE_TOL of a bisector (its membership is decided by the
#           polygon vertices, and tie parity is defined by live Qhull, SURVEY 7.4) or when the host reads the vertices.
#           Without tie points the two builders give the same memberships; cell areas agree to 1e-11.
#   "qhull" always Qhull on the host, polygons uploaded (the round-1 default; bitwise the reference's areas);
#   "clip"  never Qhull: grid points EXACTLY on a bisector may be classified differently (throughput mode).
VORONOI = os.environ.get("MFGP_VORONOI", "auto")


def voronoi_bounded(points, bounding_box):
    """reference simulator.py:154-191."""
    if VORONOI == "clip":
        return cv.ClippedVoronoi(points, bounding_box)
    if VORONOI == "qhull":
        return BoundedVoronoi(points, bounding_box)
    return cv.HybridVoronoi(points, bounding_box)


def compute_loss(vor, truth_arr):
    """reference simulator.py:194-228."""
    grid = _grid_for(truth_arr)
    host = grid.reduce_to_host(loss_vor=vor)
    return cv.loss_from_partials(host["lossp"], vor.areas())


def compute_centroids(vor, x_star, mu_star):
    """reference simulator.py:231-283.  `mu_star` may be a host array [G,1] or a device tensor [G]."""
    x_star = np.asarray(x_star)
    grid = _grid_for(x_star)
    w = mu_star if torch.is_tensor(mu_star) else torch.from_numpy(
        np.ascontiguousarray(mu_star, dtype=np.float64).reshape(-1)).to(grid.device)
    host = grid.reduce_to_host(lloyd_vor=vor, w=w)
    return cv.centroids_from_partials(host["cent"], vor.areas(), *grid.extent)


def _as_var_vector(var_star, device):
    if torch.is_tensor(var_star):
        return var_star
    v = np.asarray(var_star, dtype=np.float64)
    if v.ndim == 2 and v.shape[0] == v.shape[1] and v.shape[0] > 1:
        v = np.diag(v)          # the reference's callers pass the full covariance (simulator.py:301)
    return torch.from_numpy(np.ascontiguousarray(v.reshape(-1))).to(device)


def _max_var_from(res, truth_arr):
    """`res`: an assign_reduce result (device tensors) or its host copy (CoverageGrid.results_to_host)."""
    if torch.is_tensor(res["amax_idx"]):
        res = cv.CoverageGrid.results_to_host(res)
    idx = res["amax_idx"]
    if np.any(idx < 0):
        raise ValueError("zero-size array to reduction operation maximum which has no identity")   # np.amax([])
    return truth_arr[idx][:, [0, 1]], np.array(res["amax_val"]).reshape(-1, 1), idx


def compute_max_var(vor, truth_arr, var_star):
    """reference simulator.py:286-323; returns (argmax_xy[A,2], max_var[A,1])."""
    truth_arr = np.asarray(truth_arr)
    grid = _grid_for(truth_arr)
    host = grid.reduce_to_host(lloyd_vor=vor, var=_as_var_vector(var_star, grid.device))
    xy, mv, _ = _max_var_from(host, truth_arr)
    return xy, mv


def compute_sample_points(model, x_star, threshold, console=False, return_indices=False):
    """reference simulator.py:326-374: greedy max-variance planning, on the device (V-cached bordered updates instead
    of a refit + full predict per pick; see csrc/choi.cu).  The model is left unchanged."""
    if not isinstance(model, (SFGP, MFGP)):
        raise TypeError("Invalid model type: must be SFGP or MFGP")
    x_star = np.asarray(x_star, dtype=np.float64)
    grid = _grid_for(x_star)
    dev = grid.device
    G = grid.G
    eng = model.engine
    if not eng.fitted:
        model._refit()
    n = eng.N
    chunk = 128
    cap = n + chunk
    Vc = torch.empty((cap, G), dtype=torch.float64, device=dev)
    q = torch.empty(G, dtype=torch.float64, device=dev)
    _, var = model.predict_device(grid.xy, vcache=Vc if n else None, grid=grid, q_out=q)
    eng.check_factor(force=True)
    lib = cv.nat.lib()
    work = torch.empty(int(lib.cov_workspace_bytes(G, 1, 0)) // 8 + (G // 256 + 2) * 2 + 64 + (1 << 15), dtype=torch.float64,
                       device=dev)
    picks = []
    import ctypes
    while True:
        room = cap - n
        buf = (ctypes.c_int64 * room)()
        k = lib.choi_greedy(cv.nat.ptr(grid.xy), G, cv.nat.ptr(Vc), G, n, cap, cv.nat.ptr(var), cv.nat.ptr(q),
                            ctypes.byref(eng.pstruct), ctypes.c_double(float(threshold)),
                            ctypes.c_double(cv.AMAX_REL), room, buf,
                            cv.nat.ptr(work), work.numel() * 8, cv.nat.stream_ptr())
        if k < 0:
            cv.nat.check(int(k), "choi_greedy")
        picks.extend(buf[i] for i in range(k))
        n += k
        print(f"Found {len(picks)} sample points so far") if console else None
        if k < room:
            break
        bigger = torch.empty((cap + chunk * 2, G), dtype=torch.float64, device=dev)     # V cache full: grow, resume
        bigger[:n].copy_(Vc[:n])
        Vc, cap = bigger, cap + chunk * 2
    idx = np.asarray(picks, dtype=np.int64)
    pts = x_star[idx].reshape(-1, 2) if idx.size else np.empty([0, 2])
    return (pts, idx) if return_indices else pts


def compute_sample_clusters(vor, sample_points):
    """reference simulator.py:377-412."""
    clusters = [np.empty((0, 2)) for i in range(len(vor.filtered_regions))]
    if sample_points.shape[0] == 0:
        return clusters
    if isinstance(vor, cv.HybridVoronoi):
        vor = vor.qhull()       # sample points are grid points: bisector ties are common here, Qhull's vertices decide them
    res = CoverageGrid(sample_points).assign_reduce(lloyd_vor=vor, want_members=True)
    m = res["members"].cpu().numpy().view(np.uint64)
    for i in range(len(clusters)):
        sel = ((m[:, i // 64] >> np.uint64(i % 64)) & np.uint64(1)).astype(bool)
        clusters[i] = sample_points[sel, :]
    return clusters


# MFGP_TSP=mlrose (or simulator.TSP = "mlrose"): the reference's mlrose genetic algorithm, if mlrose is installed.
TSP = os.environ.get("MFGP_TSP", "2opt")


def plan_tours(clusters):
    """Visiting order (index arrays) of every cluster: nearest-neighbour + best-improvement 2-opt on the device
    (choi_tsp_tours, csrc/tsp.cu), all clusters of a period in one launch."""
    lens = [int(c.shape[0]) for c in clusters]
    n_total = sum(lens)
    if n_total == 0:
        return [np.empty(0, dtype=np.int64) for _ in clusters]
    nat = cv.nat
    nat.require_cuda()
    dev = torch.device("cuda", torch.cuda.current_device())
    off = np.zeros(len(clusters) + 1, dtype=np.int32)
    np.cumsum(lens, out=off[1:])
    pts = np.ascontiguousarray(np.concatenate([np.asarray(c, dtype=np.float64).reshape(-1, 2) for c in clusters], axis=0))
    d_pts = torch.from_numpy(pts).to(dev)
    d_off = torch.from_numpy(off).to(dev)
    d_ord = torch.empty(n_total, dtype=torch.int32, device=dev)
    n_max = max(lens)
    lib = nat.lib()
    work = None
    if n_max > 4096:
        work = torch.empty(int(lib.choi_tsp_workspace_bytes(n_total)) // 8 + 8, dtype=torch.float64, device=dev)
    nat.check(lib.choi_tsp_tours(nat.ptr(d_pts), nat.ptr(d_off), len(clusters), n_total, n_max, nat.ptr(d_ord), None,
                                 nat.ptr(work), 0 if work is None else work.numel() * 8, nat.stream_ptr()), "choi_tsp_tours")
    order = d_ord.cpu().numpy().astype(np.int64)
    return [order[off[i]:off[i + 1]] for i in range(len(clusters))]


def compute_sample_tsp(clusters):
    """reference simulator.py:415-454.  The reference's mlrose genetic algorithm (an unpinned third-party host routine
    whose tours are not reproducible) is replaced by a deterministic planner for the same objective -- nearest neighbour
    + 2-opt on the closed tour, on the device (see plan_tours); TSP = "mlrose" selects mlrose itself when installed."""
    if TSP == "mlrose":
        import six
        sys.modules['sklearn.externals.six'] = six
        import mlrose
        tours = []
        for cluster in clusters:
            tour = np.empty((0, 2))
            if cluster.shape[0] > 0:
                coords_list = [tuple(coord) for coord in cluster]
                problem = mlrose.TSPOpt(length=len(coords_list), coords=coords_list, maximize=False)
                solution, _ = mlrose.genetic_alg(problem, mutation_prob=0.2, max_attempts=100, random_state=2)
                tour = cluster[solution]
            tours.append(tour)
        return tours
    orders = plan_tours(clusters)
    return [cluster[o] if cluster.shape[0] > 0 else np.empty((0, 2)) for cluster, o in zip(clusters, orders)]


def todescato_prob(max_var_t, max_var_0):
    """reference simulator.py:457-467."""
    num_agents = max_var_t.shape[0]
    return np.sqrt(max_var_t / (max_var_0 * num_agents))


def choi_threshold(threshold):
    """reference simulator.py:470-478."""
    return 0.82 * threshold


def choi_double(period):
    """reference simulator.py:481-489."""
    return 8 * 2 ** period


def periodic_decision(iteration):
    """reference simulator.py:492-500."""
    return (iteration // 5) % 2 == 0


#######################################################################################################################
# Device-resident simulation state
#######################################################################################################################

class _Sim:
    """Grid, truth and work buffers of one simulation, resident on the device."""

    def __init__(self, truth):
        self.truth_arr = np.vstack(truth.values.tolist()) if hasattr(truth, "values") else np.asarray(truth, dtype=np.float64)
        self.x_star = self.truth_arr[:, [0, 1]]
        self.bounding_box = np.array([np.amin(self.x_star[:, 0]), np.amax(self.x_star[:, 0]),
                                      np.amin(self.x_star[:, 1]), np.amax(self.x_star[:, 1])])
        self.grid = CoverageGrid(self.x_star, self.truth_arr[:, 2])
        f64 = dict(dtype=torch.float64, device=self.grid.device)
        self.mu = torch.empty(self.grid.G, **f64)
        self.var = torch.empty(self.grid.G, **f64)
        self._clip = [None, None]
        self._step_begin = None
        self._index_of = None

    def index_of(self):
        if self._index_of is None:
            self._index_of = _coordinate_index(self.truth_arr) or {}
        return self._index_of or None

    def step(self, model, positions, centroids_t, weights=None):
        """One hot-path iteration: posterior over the grid, then both partitions in one fused pass.
        Returns (loss_t, centroids_t, argmax_var_t, max_var_t, loss_vor, lloyd_vor).

        Nothing on the device waits for the host: the fit is deferred into the posterior call (fused Cholesky + forward
        substitution on tensor grids), the cells are clipped on the device, the O(A) finishing runs on the device and ONE
        packed copy brings the results, the Cholesky status and the pass's tie count home.  Host Qhull -- the reference's
        cell builder -- runs only when that count is non-zero (VORONOI = "auto", see voronoi_bounded) or always
        (VORONOI = "qhull")."""
        bb = self.bounding_box

        def build_cells():
            if VORONOI == "qhull":       # host Qhull; polygons uploaded afterwards
                lv, cvor = BoundedVoronoi(positions, bb), BoundedVoronoi(centroids_t, bb)
                lv.areas()
                cvor.areas()
                return lv, cvor
            # device-built cells (two small kernels per partition), the buffers of the previous iteration are recycled
            cls = cv.ClippedVoronoi if VORONOI == "clip" else cv.HybridVoronoi
            lv = cls(positions, bb, reuse=self._clip[0])
            cvor = cls(centroids_t, bb, reuse=self._clip[1])
            self._clip = [lv, cvor]
            return lv, cvor

        if model is not None:
            eng = model.engine
            if self._step_begin is None:
                self._step_begin = torch.cuda.Event()
            self._step_begin.record()        # the previous iteration's kernels (readers of the recycled cell buffers) are behind it
            eng.lazy_check = True            # cov_finish / the packed results bring the Cholesky status home: no sync per fit
            eng.defer_fit = True             # a refit fuses with the factored posterior on large tensor grids
            model.predict_device(self.grid.xy, self.mu, self.var, grid=self.grid)       # queued first: the host prepares
            if VORONOI != "qhull" and self._clip[0] is not None:                        # the cells while the GPU works
                # recycled device buffers: the clip kernels (4 CTAs each) go to a side stream, where they are placed as soon as
                # the tiled Cholesky's CTAs start to leave the SMs -- inside its tail instead of behind the evaluation kernels
                main, side = torch.cuda.current_stream(), nat.side_stream(self.grid.device)
                side.wait_event(self._step_begin)
                with torch.cuda.stream(side):
                    loss_vor, lloyd_vor = build_cells()
                main.wait_stream(side)
            else:
                loss_vor, lloyd_vor = build_cells()
            kw = dict(w=self.mu, var=self.var, amax_k0=prior_variance(model.params()), amax_rel=cv.AMAX_REL)
            info = eng.info
        else:
            kw = dict(w=weights)
            info = None
            loss_vor, lloyd_vor = build_cells()
        device_cells = isinstance(lloyd_vor, cv.ClippedVoronoi) and len(loss_vor) and len(lloyd_vor) and \
            loss_vor.seeds_inside and lloyd_vor.seeds_inside
        if device_cells:
            res = self.grid.assign_reduce(lloyd_vor, loss_vor, **kw)
            loss_t, centroids, max_var, idx, ties = self.grid.finish(res, lloyd_vor, loss_vor, bb, info=info, with_ties=True)
            if not (ties and VORONOI != "clip"):
                if model is None:
                    return loss_t, centroids, None, None, loss_vor, lloyd_vor
                if np.any(idx < 0):
                    raise ValueError("zero-size array to reduction operation maximum which has no identity")   # np.amax([])
                return loss_t, centroids, self.truth_arr[idx][:, [0, 1]], max_var.reshape(-1, 1), loss_vor, lloyd_vor
            loss_vor.qhull()                 # tie points: the pass below runs on Qhull's polygons, like the reference
            lloyd_vor.qhull()
        host = self.grid.reduce_to_host(lloyd_vor, loss_vor, **kw)     # one device->host copy for all the per-cell results
        if model is not None:
            model.engine.check_factor(force=True)
        loss_t = cv.loss_from_partials(host["lossp"], loss_vor.areas())
        centroids = cv.centroids_from_partials(host["cent"], lloyd_vor.areas(), bb[0], bb[1], bb[2], bb[3])
        if model is None:
            return loss_t, centroids, None, None, loss_vor, lloyd_vor
        argmax_xy, max_var, _ = _max_var_from(host, self.truth_arr)
        return loss_t, centroids, argmax_xy, max_var, loss_vor, lloyd_vor


class _ShardedSim:
    """_Sim on a grid sharded over a process group: this rank keeps its whole-column slice of the grid resident
    (sharding.column_split) and steps through sharding.ShardedSim, whose results are global and the same on every rank."""

    def __init__(self, truth, group):
        import torch.distributed as dist
        from . import sharding
        from ._engine import TensorAxes
        self.truth_arr = np.vstack(truth.values.tolist()) if hasattr(truth, "values") else np.asarray(truth, dtype=np.float64)
        self.x_star = self.truth_arr[:, [0, 1]]
        self.bounding_box = np.array([np.amin(self.x_star[:, 0]), np.amax(self.x_star[:, 0]),
                                      np.amin(self.x_star[:, 1]), np.amax(self.x_star[:, 1])])
        if VORONOI == "clip":
            raise ValueError("MFGP_VORONOI=clip is not available on a sharded grid: its cells fall back to Qhull at "
                             "bisector ties (auto) or always use Qhull (qhull)")
        self.group = group
        lo, hi, ux, uy = sharding.column_split(self.x_star, dist.get_world_size(group), dist.get_rank(group))
        axes = TensorAxes(ux, uy, torch.device("cuda", torch.cuda.current_device()))
        self.state = sharding.ShardedSim(self.x_star[lo:hi], self.truth_arr[lo:hi, 2], axes, lo, self.bounding_box, group)
        self.grid, self.mu, self.var = self.state.grid, self.state.mu, self.state.var
        self._index_of = None

    index_of = _Sim.index_of

    def max_var(self):
        """Global maximum of var (one all-reduce)."""
        import torch.distributed as dist
        v = self.grid.argmax(self.var)[0]
        dist.all_reduce(v, op=dist.ReduceOp.MAX, group=self.group)
        return float(v.item())

    def step(self, model, positions, centroids_t, weights=None):
        """_Sim.step's results; the partitions are not returned (None)."""
        loss_t, centroids, idx, max_var = self.state.step(model, positions, centroids_t, weights=weights,
                                                          voronoi="qhull" if VORONOI == "qhull" else "auto")
        if model is None:
            return loss_t, centroids, None, None, None, None
        if np.any(idx < 0):
            raise ValueError("zero-size array to reduction operation maximum which has no identity")   # np.amax([])
        return loss_t, centroids, self.truth_arr[idx][:, [0, 1]], np.asarray(max_var).reshape(-1, 1), None, None


def _sharded(group):
    import torch.distributed as dist
    return group is not None and dist.get_world_size(group) > 1


def _shared_generators(rng, noise_rng, group):
    """Generators of a sharded run: every rank must consume the same draws.  Given ones are used as passed; for missing
    ones rank 0 draws one 64-bit seed from `random` and broadcasts it, and every rank builds random.Random(seed) /
    np.random.default_rng(seed) from it."""
    import torch.distributed as dist
    if rng is not None and noise_rng is not None:
        return rng, noise_rng
    seed = np.array([random.getrandbits(64) if dist.get_rank(group) == 0 else 0], dtype=np.uint64)
    t = torch.from_numpy(seed.view(np.int64)).to(torch.device("cuda", torch.cuda.current_device()))
    dist.broadcast(t, src=dist.get_global_rank(group, 0), group=group)
    seed = int(t.cpu().numpy().view(np.uint64)[0])
    return (random.Random(seed) if rng is None else rng), (np.random.default_rng(seed) if noise_rng is None else noise_rng)


def _coordinate_index(truth_arr):
    """{(x, y): row} for grids without repeated points (else None): the exact-equality lookup of simulator.py:875 in O(1)."""
    idx = {}
    for r, (x, y) in enumerate(zip(truth_arr[:, 0].tolist(), truth_arr[:, 1].tolist())):
        if (x, y) in idx:
            return None
        idx[(x, y)] = r
    return idx


def _take_samples(agents, positions, explore_t, truth_arr, sigma_n, noise_rng, console, centroids_t, iteration,
                  index_of=None):
    """reference simulator.py:698-713 / :868-883 / :1060-1075: exact-coordinate lookup of the truth + N(0, sigma_n)."""
    x_new = np.empty([0, 2])
    y_new = np.empty([0, 1])
    id_new = np.empty([0, 1])
    for i in range(agents):
        if explore_t[i] == 1:
            x_sample = positions[i, :]
            row = index_of.get((float(x_sample[0]), float(x_sample[1]))) if index_of is not None else None
            if row is not None:
                sample_idx = [row]
            else:
                sample_idx = np.logical_and(truth_arr[:, 0] == x_sample[0], truth_arr[:, 1] == x_sample[1])
            gen = noise_rng if noise_rng is not None else np.random.default_rng()
            y_sample = truth_arr[sample_idx, 2] + gen.normal(loc=0, scale=sigma_n)
            print(f"Robot {i} explored {x_sample} and sampled {y_sample}") if console else None
            x_new = np.vstack((x_new, x_sample))
            y_new = np.vstack((y_new, y_sample))
            id_new = np.vstack((id_new, i))
        elif iteration > 0:
            print(f"Robot {i} exploited to {centroids_t[i, :]}") if console else None
    return x_new, y_new, id_new


def _fidelity_of(hyp):
    n = _hyp_len(hyp)
    if n == 4:
        return "S"
    if n == 9:
        return "M"
    raise TypeError("Hyperparameters must be of length 4 (single-fidelity) or 9 (multi-fidelity)")


# MFGP_INCREMENTAL=1 (or simulator.INCREMENTAL = True): bordered factor updates + incremental posterior in the algorithm
# loops instead of the reference's refit-from-scratch every iteration (gaussian_process.py:266-268, :540-542).
INCREMENTAL = os.environ.get("MFGP_INCREMENTAL", "0") == "1"


def _init_models(fidelity, hyp, prior):
    """reference simulator.py:656-681 / :826-851 / :998-1024: max_var_0 from the EMPTY model (== k(0), evaluated on the
    device through the N = 0 posterior), then the model conditioned on the prior with a forced update."""
    empty = init_SFGP(hyp, prior=None) if fidelity == "S" else init_MFGP(hyp, prior=None)
    max_var_0 = prior_variance(empty.params())
    if fidelity == "S":
        model = init_SFGP(hyp, prior=prior)
        model.updt_info(model.X, model.y)
    else:
        model = init_MFGP(hyp, prior=prior)
        model.updt_info(model.X_L, model.y_L, model.X_H, model.y_H)
    model.incremental = INCREMENTAL
    return model, max_var_0


def _log_rows(log, loss_log, agent_log, sample_log, sim_num, iteration, period, fidelity, agents, positions,
              argmax_var_t, max_var_t, max_var_0, centroids_t, prob_explore_t, explore_t, distance, loss_t, id_new,
              x_new, y_new):
    if not log:
        return
    loss_log.append({"SimNum": sim_num, "Iteration": iteration, "Period": period, "Fidelity": fidelity, "Loss": loss_t})
    for i in range(agents):
        agent_log.append({"SimNum": sim_num, "Iteration": iteration, "Period": period,
                          "Fidelity": fidelity, "Agent": i,
                          "X": positions[i, 0], "Y": positions[i, 1],
                          "XMax": argmax_var_t[i, 0], "YMax": positions[i, 1],      # sic: reference :924 logs positions
                          "VarMax": max_var_t[i, 0], "Var0": max_var_0,
                          "XCentroid": centroids_t[i, 0], "YCentroid": centroids_t[i, 1],
                          "ProbExplore": prob_explore_t[i, 0], "Explore": explore_t[i, 0],
                          "Distance": distance[i, 0]})
    if id_new is not None:
        for i in range(id_new.size):
            sample_log.append({"SimNum": sim_num, "Iteration": iteration, "Period": period, "Fidelity": fidelity,
                               "Agent": id_new[i, 0], "X": x_new[i, 0], "Y": x_new[i, 1], "Sample": y_new[i, 0]})


def _console(console, period, fidelity, loss_t, max_var_t, max_var_0, prob_explore_t, explore_t, iteration):
    if console:
        print(f"Period {period}")
        print(f"Fidelity {fidelity}")
        print(f"Current loss: {loss_t}")
        print(f"Max var by cell: {max_var_t.flatten()}")
        print(f"Normalizing max var: {max_var_0}")
        print(f"Probability of exploration: {prob_explore_t.flatten()}")
        print(f"Decision of exploration: {explore_t.flatten()}")
        print(f"End Iteration {iteration}")


#######################################################################################################################
# Control Algorithms
#######################################################################################################################

def lloyd(title, sim_num, iterations, agents, positions, truth, sigma_n, prior, hyp, console, plotter, log,
          rng=None, noise_rng=None, group=None):
    """reference simulator.py:508-616: Lloyd's algorithm with perfect knowledge (weights = ground truth).
    `group` (torch.distributed process group, all four algorithms): the grid is split into whole-column slices, one per
    rank on its own GPU; every rank returns the same logs.  None or a group of one rank: the single-GPU path."""
    loss_log, agent_log, sample_log = [], [], [] if log else None
    fidelity = "NA"
    max_var_0 = 0
    prob_explore_t = np.zeros((agents, 1))
    explore_t = np.zeros((agents, 1))
    argmax_var_t = np.zeros((agents, 1))
    max_var_t = np.zeros((agents, 1))
    print(line_break + title + line_break)
    sim = _ShardedSim(truth, group) if _sharded(group) else _Sim(truth)
    prev_positions = np.copy(positions)
    centroids_t = np.copy(positions)
    period = 0
    for iteration in range(iterations):
        print(f"\nBegin Iteration {iteration} of Simulation {sim_num} of {title}") if console else None
        distance = np.sqrt(np.sum((positions - prev_positions) ** 2, axis=1)).reshape(-1, 1)
        loss_t, centroids_t, _, _, _, _ = sim.step(None, positions, centroids_t, weights=sim.grid.f)
        _console(console, period, fidelity, loss_t, max_var_t, max_var_0, prob_explore_t, explore_t, iteration)
        if log:
            loss_log.append({"SimNum": sim_num, "Iteration": iteration, "Period": period,
                             "Fidelity": fidelity, "Loss": loss_t})
            sample_log.append({"SimNum": sim_num, "Iteration": iteration, "Period": period, "Fidelity": fidelity,
                               "Agent": "NA", "X": "NA", "Y": "NA", "Sample": "NA"})
            _log_rows(True, [], agent_log, None, sim_num, iteration, period, fidelity, agents, positions, argmax_var_t,
                      max_var_t, max_var_0, centroids_t, prob_explore_t, explore_t, distance, loss_t, None, None, None)
        prev_positions = np.copy(positions)
        positions = np.copy(centroids_t)
    return loss_log, agent_log, sample_log


def _explore_exploit(kind, title, sim_num, iterations, agents, positions, truth, sigma_n, prior, hyp, console, log,
                     rng, noise_rng, group=None):
    loss_log, agent_log, sample_log = [], [], [] if log else None
    fidelity = _fidelity_of(hyp)
    print(line_break + title + line_break)
    sharded = _sharded(group)
    if sharded:
        rng, noise_rng = _shared_generators(rng, noise_rng, group)
    rng = random if rng is None else rng
    model, max_var_0 = _init_models(fidelity, hyp, prior)
    print("Max Initial Predictive Variance: " + str(max_var_0)) if console else None
    sim = _ShardedSim(truth, group) if sharded else _Sim(truth)
    truth_arr = sim.truth_arr
    model.predict_device(sim.grid.xy, sim.mu, sim.var, grid=sim.grid)
    if sharded:
        max_var_t = sim.max_var() * np.ones((agents, 1))
    else:
        max_var_t = float(sim.grid.argmax(sim.var)[0].item()) * np.ones((agents, 1))     # value only: ties irrelevant
    prob_explore_t = todescato_prob(max_var_t, max_var_0) if kind == "todescato" else np.zeros((agents, 1))
    explore_t = np.zeros((agents, 1))
    prev_positions = np.copy(positions)
    centroids_t = np.copy(positions)
    period = 0
    for iteration in range(iterations):
        print(f"\nBegin Iteration {iteration} of Simulation {sim_num} of {title}") if console else None
        x_new, y_new, id_new = _take_samples(agents, positions, explore_t, truth_arr, sigma_n, noise_rng, console,
                                             centroids_t, iteration, sim.index_of())
        distance = np.sqrt(np.sum((positions - prev_positions) ** 2, axis=1)).reshape(-1, 1)
        if fidelity == "S":
            model.updt(x_new, y_new)
        else:
            model.updt_hifi(x_new, y_new)
        loss_t, centroids_t, argmax_var_t, max_var_t, _, _ = sim.step(model, positions, centroids_t)
        _console(console, period, fidelity, loss_t, max_var_t, max_var_0, prob_explore_t, explore_t, iteration)
        _log_rows(log, loss_log, agent_log, sample_log, sim_num, iteration, period, fidelity, agents, positions,
                  argmax_var_t, max_var_t, max_var_0, centroids_t, prob_explore_t, explore_t, distance, loss_t, id_new,
                  x_new, y_new)
        if kind == "todescato":
            prob_explore_t = todescato_prob(max_var_t, max_var_0)
            explore_t = np.array([int(rng.random() < cutoff) for cutoff in prob_explore_t]).reshape(-1, 1)
        else:
            explore_bool = periodic_decision(iteration)
            prob_explore_t = np.array([int(explore_bool) for agent in range(agents)]).reshape(-1, 1)
            explore_t = np.array([int(explore_bool) for agent in range(agents)]).reshape(-1, 1)
        prev_positions = np.copy(positions)
        for i in range(agents):
            if explore_t[i, 0]:
                positions[i, :] = argmax_var_t[i, :]
            else:
                positions[i, :] = centroids_t[i, :]
    return loss_log, agent_log, sample_log


def periodic(title, sim_num, iterations, agents, positions, truth, sigma_n, prior, hyp, console, plotter, log,
             rng=None, noise_rng=None, group=None):
    """reference simulator.py:618-785.  `group`: see lloyd."""
    return _explore_exploit("periodic", title, sim_num, iterations, agents, positions, truth, sigma_n, prior, hyp,
                            console, log, rng, noise_rng, group)


def todescato(title, sim_num, iterations, agents, positions, truth, sigma_n, prior, hyp, console, plotter, log,
              rng=None, noise_rng=None, group=None):
    """reference simulator.py:788-954.  `group`: see lloyd."""
    return _explore_exploit("todescato", title, sim_num, iterations, agents, positions, truth, sigma_n, prior, hyp,
                            console, log, rng, noise_rng, group)


def run_batched(algo, sim_nums, iterations, agents, positions, truth, sigma_n, prior, hyp, uniforms=None, noise=None,
                noise_rngs=None, exact_tie_loss=False, use_graph=False):
    """Many independent runs of ONE experiment stepped together on the device (config c5, the replicate sweeps of
    runner.py:100, :131-147): `algo` names lloyd, periodic, todescato or choi (as runner.run_sim dispatches), `positions[R, A,
    2]` the runs' start positions (updated in place to the final ones, like the single-run functions do).  Returns a list of R
    (loss_log, agent_log, sample_log) triples with the reference's row schemas.  See _batched.BatchedRuns for the
    random-number and tie conventions; `exact_tie_loss=True` re-evaluates the losses that involve exact bisector ties with
    Qhull cells.  Choi runs come back to the host once per period, so `use_graph` is not available for them."""
    from ._batched import BatchedRuns
    kind = "choi" if "choi" in algo else ("todescato" if "todescato" in algo else ("lloyd" if "lloyd" in algo else
                                          ("periodic" if "periodic" in algo else None)))
    if kind is None:
        raise ValueError("run_batched supports lloyd, periodic, todescato and choi")
    if kind == "choi" and use_graph:
        raise ValueError("Choi runs return to the host once per period: use_graph is not available for them")
    truth_arr = np.vstack(truth.values.tolist()) if hasattr(truth, "values") else np.asarray(truth, dtype=np.float64)
    prior_arr = None
    if prior is not None and len(prior) > 0:
        prior_arr = np.vstack(prior.values.tolist()) if hasattr(prior, "values") else np.asarray(prior, dtype=np.float64)
    br = BatchedRuns(kind, truth_arr, prior_arr, hyp, agents, iterations, positions, sigma_n, uniforms, noise, noise_rngs)
    br.run(use_graph=use_graph)          # use_graph: the whole device-resident loop replayed from one CUDA graph
    logs = br.logs(sim_nums, exact_tie_loss)
    np.asarray(positions)[...] = br.final_positions()
    return logs


def choi(title, sim_num, iterations, agents, positions, truth, sigma_n, prior, hyp, console, plotter, log,
         rng=None, noise_rng=None, group=None):
    """reference simulator.py:957-1161.  `group`: see lloyd; the planner's V cache is split with the grid
    (sharding.sharded_sample_points), clustering and tours run on the same inputs on every rank."""
    loss_log, agent_log, sample_log = [], [], [] if log else None
    fidelity = _fidelity_of(hyp)
    print(line_break + title + line_break)
    sharded = _sharded(group)
    if sharded:
        rng, noise_rng = _shared_generators(rng, noise_rng, group)
    model, max_var_0 = _init_models(fidelity, hyp, prior)
    threshold = max_var_0
    print("Max Initial Predictive Variance: " + str(max_var_0)) if console else None
    sim = _ShardedSim(truth, group) if sharded else _Sim(truth)
    truth_arr, x_star, bounding_box = sim.truth_arr, sim.x_star, sim.bounding_box
    iteration = 0
    period = 0
    centroids_t = np.copy(positions)
    prev_positions = np.copy(positions)
    prob_explore_t = np.zeros((agents, 1))
    explore_t = np.zeros((agents, 1))
    while iteration < iterations:
        threshold = choi_threshold(threshold)
        sample_vor = voronoi_bounded(centroids_t, bounding_box)
        if sharded:
            from .sharding import sharded_sample_points
            sample_points, _ = sharded_sample_points(model, sim.grid, threshold, group, console)
        else:
            sample_points = compute_sample_points(model, x_star, threshold, console)
        sample_clusters = compute_sample_clusters(sample_vor, sample_points)
        print("\nBegin TSP Computation") if console else None
        tsp_tours_t = compute_sample_tsp(sample_clusters)
        print("\nEnd TSP Computation") if console else None
        tsp_tours_0 = copy.deepcopy(tsp_tours_t)    # noqa: F841  (kept for parity with the reference's plotter hook)
        period_length = choi_double(period)
        for step in range(period_length):
            print(f"\nBegin Iteration {iteration} of Simulation {sim_num} of {title}") if console else None
            x_new, y_new, id_new = _take_samples(agents, positions, explore_t, truth_arr, sigma_n, noise_rng, console,
                                                 centroids_t, iteration)
            distance = np.sqrt(np.sum((positions - prev_positions) ** 2, axis=1)).reshape(-1, 1)
            if fidelity == "S":
                model.updt(x_new, y_new)
            else:
                model.updt_hifi(x_new, y_new)
            loss_t, centroids_t, argmax_var_t, max_var_t, _, _ = sim.step(model, positions, centroids_t)
            _console(console, period, fidelity, loss_t, max_var_t, max_var_0, prob_explore_t, explore_t, iteration)
            _log_rows(log, loss_log, agent_log, sample_log, sim_num, iteration, period, fidelity, agents, positions,
                      argmax_var_t, max_var_t, max_var_0, centroids_t, prob_explore_t, explore_t, distance, loss_t,
                      id_new, x_new, y_new)
            for i in range(agents):
                if tsp_tours_t[i].shape[0] > 0:
                    prob_explore_t[i] = 1
                    explore_t[i] = 1
                else:
                    prob_explore_t[i] = 0
                    explore_t[i] = 0
            prev_positions = np.copy(positions)
            for i in range(agents):
                if explore_t[i, 0]:
                    positions[i, :] = tsp_tours_t[i][0, :]
                    tsp_tours_t[i] = np.delete(tsp_tours_t[i], 0, axis=0)
                else:
                    positions[i, :] = centroids_t[i, :]
            iteration += 1
        period += 1
    return loss_log, agent_log, sample_log
