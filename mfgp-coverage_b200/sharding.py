"""Multi-GPU sharding of the hot path: one process per GPU, torch.distributed for the plumbing.

Two axes, both taken from the reference's own parallelism (SURVEY.md section 2.1 / 8e):

  * GRID sharding (config c4): the G grid points are split into contiguous slices, one per rank -- the reference's
    experimental `predict_multiproc` slicing (gaussian_process_numba.py:478-503).  The posterior is then
    communication-free.  The training factor is needed by every rank: rank 0 factorises and broadcasts W = L^-1 and
    z (NCCL over NVLink; 134 MB at N = 4096), or every rank factorises redundantly (`replicate_factor=True`, no
    collective at all; chosen by measurement).  The coverage step all-reduces only O(agents) numbers:
    per-cell partial sums (SUM) and the per-cell (max variance, first index) pairs (all-gather + local merge, lowest
    global index wins ties exactly as np.argmax on the unsharded array).
    Whole simulations run this way through simulator.lloyd / periodic / todescato / choi(..., group=); the Choi planner then
    keeps only its slice's V cache on each rank (ShardPlanner, sharded_sample_points: one all-gather of a small slot per pick).
  * RUN sharding (config c5, replicate sweeps): independent simulations, `runner._map_sims` -- no collective.

The merge logic is plain tensor code so that it is exercised on CPU with the gloo backend (tests/test_sharding_gloo.py).
"""
import numpy as np
import torch
import torch.distributed as dist


def shard_bounds(G, world, rank):
    """Contiguous slice [lo, hi) of rank `rank` (sizes differ by at most one, like np.array_split)."""
    base, extra = divmod(G, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def merge_argmax(vals, idxs, k0=0.0, rel=0.0):
    """vals[R, A], idxs[R, A] (global indices, -1 = empty) -> per-cell (max value, LOWEST index attaining it).

    Ranks are folded in rank order with the SAME tie rule the kernels apply inside a shard (csrc/argmax.cuh,
    argmax_combine): two candidates are tied when they differ by at most rel * (k0 - smaller value) -- a tolerance
    relative to the variance reduction -- and a tie goes to the lower global index, carrying the larger value.  With
    rel = 0 this is the plain first-index arg-max.  Without it two mirror-image grid points ~1e-16 apart that land on
    different ranks would be resolved by rounding noise instead of by index (the single-GPU kernel and the reference
    pick the lower index)."""
    R = vals.shape[0]
    bv, bi = vals[0].clone(), idxs[0].clone()
    for r in range(1, R):
        v, i = vals[r], idxs[r]
        a_empty, b_empty = bi < 0, i < 0
        lo = torch.minimum(bv, v)
        tol = torch.clamp(rel * (k0 - lo), min=0.0) if rel > 0.0 else torch.zeros_like(lo)
        d = bv - v
        take_b = (-d > tol)
        tie = ~(d > tol) & ~take_b
        nv = torch.where(take_b, v, torch.where(tie, torch.maximum(bv, v), bv))
        ni = torch.where(take_b, i, torch.where(tie, torch.minimum(bi, i), bi))
        nv = torch.where(b_empty, bv, torch.where(a_empty, v, nv))
        ni = torch.where(b_empty, bi, torch.where(a_empty, i, ni))
        bv, bi = nv, ni
    bv = torch.where(bi < 0, torch.full_like(bv, -float("inf")), bv)
    return bv, bi


def allreduce_partials(res, group=None, amax_k0=0.0, amax_rel=0.0):
    """In-place combination of the outputs of CoverageGrid.assign_reduce across ranks.  (amax_k0, amax_rel): the arg-max
    tie rule the kernels were called with (see merge_argmax)."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return res
    world = dist.get_world_size(group)
    if res.get("cent") is not None:
        dist.all_reduce(res["cent"], op=dist.ReduceOp.SUM, group=group)
    if res.get("lossp") is not None:
        dist.all_reduce(res["lossp"], op=dist.ReduceOp.SUM, group=group)
    if res.get("ties") is not None:
        dist.all_reduce(res["ties"], op=dist.ReduceOp.SUM, group=group)
    if res.get("amax_val") is not None:
        A = res["amax_val"].numel()
        vals = [torch.empty_like(res["amax_val"]) for _ in range(world)]
        idxs = [torch.empty_like(res["amax_idx"]) for _ in range(world)]
        dist.all_gather(vals, res["amax_val"].contiguous(), group=group)
        dist.all_gather(idxs, res["amax_idx"].contiguous(), group=group)
        v, i = merge_argmax(torch.stack(vals).reshape(world, A), torch.stack(idxs).reshape(world, A), amax_k0, amax_rel)
        res["amax_val"].copy_(v)
        res["amax_idx"].copy_(i)
    return res


def merge_argmax_host(vals, idxs, k0=0.0, rel=0.0):
    """numpy twin of merge_argmax for host-side merging: vals[R, A], idxs[R, A] (int64, -1 = empty)."""
    vals = np.asarray(vals, dtype=np.float64)
    idxs = np.asarray(idxs, dtype=np.int64)
    bv, bi = vals[0].copy(), idxs[0].copy()
    for r in range(1, vals.shape[0]):
        v, i = vals[r], idxs[r]
        a_empty, b_empty = bi < 0, i < 0
        with np.errstate(invalid="ignore"):
            lo = np.minimum(bv, v)
            tol = np.maximum(rel * (k0 - lo), 0.0) if rel > 0.0 else np.zeros_like(lo)
            d = bv - v
            take_b = -d > tol
            tie = ~(d > tol) & ~take_b
        nv = np.where(take_b, v, np.where(tie, np.maximum(bv, v), bv))
        ni = np.where(take_b, i, np.where(tie, np.minimum(bi, i), bi))
        bv = np.where(b_empty, bv, np.where(a_empty, v, nv))
        bi = np.where(b_empty, bi, np.where(a_empty, i, ni))
    bv = np.where(bi < 0, -np.inf, bv)
    return bv, bi


def gather_results_to_host(res, group=None, amax_k0=0.0, amax_rel=0.0, extras=None):
    """Global per-cell results of CoverageGrid.assign_reduce on the host with ONE collective and ONE device->host copy:
    the packed result buffers of all ranks are all-gathered, copied home, and combined there -- partial sums added in rank
    order (deterministic), arg-max pairs merged with the lowest-global-index rule.  Every rank gets the same dict of numpy
    arrays (cent, amax_val, amax_idx, lossp).  Cheaper than allreduce_partials (two all-reduces, two all-gathers and a
    handful of small kernels) when the results go to the host anyway, as in the coverage loops.
    `extras`: small float64 device tensors of THIS rank (cell areas, status flags) that ride home in the same copy;
    returned as out["extras"] (list of numpy arrays)."""
    from ._coverage import CoverageGrid
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        out = CoverageGrid.results_to_host(res)
        if extras:
            out["extras"] = [e.detach().cpu().numpy() for e in extras]
        return out
    world = dist.get_world_size(group)
    Ac, Ap = res["pack_shape"]
    pack = res["pack"]
    if pack.is_cuda:
        allp = torch.empty((world,) + tuple(pack.shape), dtype=pack.dtype, device=pack.device)
        dist.all_gather_into_tensor(allp, pack, group=group)
    else:
        parts = [torch.empty_like(pack) for _ in range(world)]
        dist.all_gather(parts, pack, group=group)
        allp = torch.stack(parts)
    ex_host = None
    if allp.is_cuda:
        flat = torch.cat([allp.reshape(-1)] + [e.reshape(-1) for e in extras]) if extras else allp.reshape(-1)
        h = torch.empty(flat.shape, dtype=flat.dtype, pin_memory=True)
        h.copy_(flat, non_blocking=True)
        torch.cuda.current_stream(allp.device).synchronize()
        a = h.numpy()[:allp.numel()].reshape(tuple(allp.shape))
        if extras:
            ex_host, o = [], allp.numel()
            for e in extras:
                ex_host.append(h.numpy()[o:o + e.numel()])
                o += e.numel()
    else:
        a = allp.numpy()
        if extras:
            ex_host = [e.numpy().reshape(-1) for e in extras]
    out = {"cent": None, "amax_val": None, "amax_idx": None, "lossp": None,
           "ties": int(a[:, 6 * Ac + 2 * Ap:].copy().view(np.int32)[:, 0].sum())}
    if Ac:
        cent = np.zeros((Ac, 4))
        for r in range(world):                                   # rank order: the same sum on every rank, every run
            cent += a[r, :4 * Ac].reshape(Ac, 4)
        out["cent"] = cent
        out["amax_val"], out["amax_idx"] = merge_argmax_host(a[:, 4 * Ac:5 * Ac], a[:, 5 * Ac:6 * Ac].copy().view(np.int64),
                                                             amax_k0, amax_rel)
    if Ap:
        lossp = np.zeros((Ap, 2))
        for r in range(world):
            lossp += a[r, 6 * Ac:6 * Ac + 2 * Ap].reshape(Ap, 2)
        out["lossp"] = lossp
    if ex_host is not None:
        out["extras"] = ex_host
    return out


def broadcast_partitions(seed_sets, bounding_box, device, src=0, group=None):
    """Bounded Voronoi partitions for every rank from ONE host: rank `src` runs Qhull on each seed set and broadcasts the
    packed cells (seeds, areas, offsets, vertices: ~0.1 KB per cell) over NCCL; the other ranks only queue the receive.
    The partitions are global (every rank classifies its own grid shard against the same cells), so building them once
    removes N - 1 redundant Qhull runs per step and, more importantly, the wait for the slowest host of the N.
    Returns a list of PackedPartition (accepted by CoverageGrid.assign_reduce; .areas() for the host finishing)."""
    from . import _coverage as cv
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    heads = [cv.seeds_summary(p, bounding_box) for p in seed_sets]            # (A, seeds_inside): cheap, every rank
    sizes = [cv.partition_doubles(A) for A, _ in heads]
    total = sum(sizes)
    if rank == src:
        stage = torch.empty(total, dtype=torch.float64, pin_memory=torch.device(device).type == "cuda")
        host = stage.numpy()
        o = 0
        for p, n in zip(seed_sets, sizes):
            cv.pack_partition(cv.BoundedVoronoi(p, bounding_box), host[o:o + n])
            o += n
        buf = stage.to(device, non_blocking=True)
    else:
        buf = torch.empty(total, dtype=torch.float64, device=device)
    if world > 1:
        dist.broadcast(buf, src=src, group=group)
    out, o = [], 0
    for (A, inside), n in zip(heads, sizes):
        out.append(cv.PackedPartition(buf[o:o + n], A, inside))
        o += n
    return out


def broadcast_factor(engine, src=0, group=None):
    """Broadcast the fitted factor state (W, z, Tt) of `engine` (a DeviceGP) from rank `src` to all ranks."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return
    engine.ensure_factor()        # a fused / deferred fit leaves only the diagonal-block inverses in W: complete it first
    n = engine.npad
    for t in (engine.W[:n], engine.z[:n], engine.Tt[:n]):
        dist.broadcast(t, src=src, group=group)


class ShardedGrid:
    """Rank-local slice of the grid plus the collectives that turn rank-local reductions into global ones."""

    def __init__(self, xy_host, f_host=None, group=None):
        from ._coverage import CoverageGrid
        from ._engine import TensorAxes, detect_tensor_grid
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        xy_host = np.asarray(xy_host, dtype=np.float64).reshape(-1, 2)
        self.G_total = xy_host.shape[0]
        self.lo, self.hi = shard_bounds(self.G_total, self.world, self.rank)
        tg = detect_tensor_grid(xy_host)
        axes = TensorAxes(tg[0], tg[1], torch.device("cuda", torch.cuda.current_device())) if tg is not None else None
        self.local = CoverageGrid(xy_host[self.lo:self.hi], None if f_host is None else np.asarray(f_host)[self.lo:self.hi],
                                  base_index=self.lo, axes=axes)

    def assign_reduce(self, *a, **k):
        return allreduce_partials(self.local.assign_reduce(*a, **k), self.group, k.get("amax_k0", 0.0), k.get("amax_rel", 0.0))


class ShardedSim:
    """Grid-sharded twin of simulator._Sim (config c4: the fixed grid split into whole-column slices, one per rank).

    Every rank keeps its slice of the grid resident, factorises the (small) training system itself -- the fused
    Cholesky + forward substitution of the factored posterior; the x expansion covers only the slice's interval, so the
    right-hand-side count shrinks with the number of ranks -- and clips the SAME global Voronoi cells on its own device
    (deterministic: identical on every rank, no broadcast).  One step needs ONE collective: the all-gather of the packed
    per-cell results (6 A_c + 2 A_p + 1 doubles per rank), merged on the host in rank order with the kernels' arg-max tie
    rule.  Tie points (grid points within TIE_TOL of a bisector, counted over all ranks) send every rank to Qhull's
    polygons for that step, exactly like the single-GPU path."""

    def __init__(self, xy_shard, f_shard, axes, base_index, bounding_box, group=None):
        from ._coverage import CoverageGrid
        self.group = group
        self.bounding_box = np.asarray(bounding_box, dtype=np.float64)
        self.grid = CoverageGrid(xy_shard, f_shard, base_index=base_index, axes=axes)
        f64 = dict(dtype=torch.float64, device=self.grid.device)
        self.mu = torch.empty(self.grid.G, **f64)
        self.var = torch.empty(self.grid.G, **f64)
        self._clip = [None, None]

    def step(self, model, positions, centroids_t, voronoi="auto", weights=None):
        """(loss, centroids[A,2], argmax grid indices[A], max variance[A]) -- global results, the same on every rank.
        Lloyd form (model=None): the centroids are weighted by `weights` (this shard's slice, e.g. its truth) and no
        variance is evaluated; the last two results are None."""
        from . import _coverage as cv
        from .gaussian_process import prior_variance
        bb = self.bounding_box
        eng = None if model is None else model.engine
        if eng is not None:
            eng.lazy_check = eng.defer_fit = True
            model.predict_device(self.grid.xy, self.mu, self.var, grid=self.grid)   # queued first; the host builds the cells meanwhile
        if voronoi == "qhull":
            loss_vor, lloyd_vor = cv.BoundedVoronoi(positions, bb), cv.BoundedVoronoi(centroids_t, bb)
        else:
            loss_vor = cv.HybridVoronoi(positions, bb, reuse=self._clip[0])
            lloyd_vor = cv.HybridVoronoi(centroids_t, bb, reuse=self._clip[1])
            self._clip = [loss_vor, lloyd_vor]
        if eng is not None:
            k0 = prior_variance(model.params())
            kw = dict(w=self.mu, var=self.var, amax_k0=k0, amax_rel=cv.AMAX_REL)
            info = eng.info.reshape(1)
        else:
            k0 = 0.0
            kw = dict(w=weights)
            info = torch.zeros(1, dtype=torch.int32, device=self.grid.device)
        extras = None
        if voronoi != "qhull" and self.grid.xy.is_cuda and len(loss_vor) and len(lloyd_vor):
            # this rank's cell areas, the clip flags and the Cholesky status ride home in the gathered results' copy
            extras = [lloyd_vor.dev_areas[:len(lloyd_vor)], loss_vor.dev_areas[:len(loss_vor)],
                      torch.cat([info, lloyd_vor.flag.reshape(1), loss_vor.flag.reshape(1)]).to(torch.float64)]
        host = gather_results_to_host(self.grid.assign_reduce(lloyd_vor, loss_vor, **kw), self.group, k0, cv.AMAX_REL, extras)
        if extras is not None:
            ac, ap, st = host["extras"]
            if eng is not None:
                eng.raise_for_info(int(st[0]))
            if st[1] != 0 or st[2] != 0:
                raise RuntimeError("cov_voronoi_clip: polygon capacity exceeded")
            lloyd_vor._areas_host, loss_vor._areas_host = ac.copy(), ap.copy()
        if host["ties"] and voronoi != "qhull":
            loss_vor.qhull(), lloyd_vor.qhull()
            host = gather_results_to_host(self.grid.assign_reduce(lloyd_vor, loss_vor, **kw), self.group, k0, cv.AMAX_REL)
        if extras is None and eng is not None:
            eng.check_factor(force=True)
        loss = cv.loss_from_partials(host["lossp"], loss_vor.areas())
        cent = cv.centroids_from_partials(host["cent"], lloyd_vor.areas(), bb[0], bb[1], bb[2], bb[3])
        if eng is None:
            return loss, cent, None, None
        return loss, cent, host["amax_idx"], host["amax_val"]


def column_split(xy_host, world, rank):
    """Whole-column slice of rank `rank` of the x-major tensor-product grid xy_host[G,2], split as the strong-scaling
    benchmark splits it (columns [rank nx / world, (rank + 1) nx / world)).  Returns (lo, hi, ux, uy): the flat index range
    [lo, hi) -- a multiple of ny, as the column-sweep coverage kernel needs -- and the grid's axes.  ValueError for a grid
    that is not tensor-product or has fewer columns than ranks."""
    from ._engine import detect_tensor_grid
    tg = detect_tensor_grid(xy_host)
    if tg is None:
        raise ValueError("grid sharding needs an x-major tensor-product grid [[x, y] for x in ux for y in uy]")
    ux, uy = tg
    nx, ny = ux.size, uy.size
    if world > nx:
        raise ValueError(f"grid sharding needs at least one grid column per rank ({nx} columns, {world} ranks)")
    c0, c1 = (rank * nx) // world, ((rank + 1) * nx) // world
    return c0 * ny, c1 * ny, ux, uy


# ---- grid-sharded Choi planner (csrc/choi.cu, choi_shard_*) ------------------------------------------------------------

PLAN_BATCH = 16          # picks enqueued per host read of the planner's `done` flag, as choi_greedy does


class ShardPlanner:
    """Greedy-planner state of one grid shard: the V cache Vc[cap, G] of the shard's slice, q, var and the workspace.
    One pick is append() -> propose() -> exchange of the send slots of all ranks (rank order) -> select(recv); see
    include/mfgp_b200.h, choi_shard_*.  `grid`: the shard's CoverageGrid (base_index = global index of its first point,
    axes = those of the whole grid).  The model is not changed."""

    def __init__(self, model, grid, chunk=128):
        from . import _native as nat
        from ._coverage import AMAX_REL
        eng = model.engine
        if not eng.fitted:
            model._refit()
        self.nat, self.lib, self.eng, self.grid = nat, nat.lib(), eng, grid
        self.G, self.base, self.tie_rel = grid.G, grid.base_index, AMAX_REL
        self.n0 = eng.N
        self.cap = self.n0 + chunk
        f64 = dict(dtype=torch.float64, device=grid.device)
        self.Vc = torch.empty((self.cap, self.G), **f64)
        self.q = torch.empty(self.G, **f64)
        _, self.var = model.predict_device(grid.xy, vcache=self.Vc if self.n0 else None, grid=grid, q_out=self.q)
        eng.check_factor(force=True)
        self._buffers()

    def _buffers(self):
        f64 = dict(dtype=torch.float64, device=self.grid.device)
        self.work = torch.empty(int(self.lib.choi_shard_workspace_bytes(self.G, self.cap)) // 8 + 1, **f64)
        self.send = torch.empty(self.cap + 4, **f64)

    def _w(self):
        return self.nat.ptr(self.work), self.work.numel() * 8, self.nat.stream_ptr()

    def begin(self, n):
        """Start planning with rows [0, n) of the cache valid: arg-max of the slice's var and the first send slot."""
        import ctypes
        nat = self.nat
        nat.check(self.lib.choi_shard_begin(nat.ptr(self.grid.xy), self.G, self.base, nat.ptr(self.Vc), self.G, n, self.cap,
                                            nat.ptr(self.var), ctypes.byref(self.eng.pstruct), ctypes.c_double(self.tie_rel),
                                            nat.ptr(self.send), *self._w()), "choi_shard_begin")
        return self.send

    def append(self):
        import ctypes
        nat = self.nat
        nat.check(self.lib.choi_shard_append(nat.ptr(self.grid.xy), self.G, self.base, nat.ptr(self.Vc), self.G, self.cap,
                                             nat.ptr(self.var), nat.ptr(self.q), ctypes.byref(self.eng.pstruct),
                                             ctypes.c_double(self.tie_rel), *self._w()), "choi_shard_append")

    def propose(self):
        """The shard's send slot (cap + 4 doubles) after the last append."""
        import ctypes
        nat = self.nat
        nat.check(self.lib.choi_shard_propose(nat.ptr(self.grid.xy), self.G, self.base, nat.ptr(self.Vc), self.G, self.cap,
                                              ctypes.byref(self.eng.pstruct), ctypes.c_double(self.tie_rel),
                                              nat.ptr(self.send), *self._w()), "choi_shard_propose")
        return self.send

    def select(self, recv, threshold, max_picks):
        """recv[world, cap + 4]: the send slots of all ranks in rank order."""
        import ctypes
        nat = self.nat
        recv = recv.contiguous()
        nat.check(self.lib.choi_shard_select(nat.ptr(recv), recv.shape[0], self.G, self.cap, ctypes.byref(self.eng.pstruct),
                                             ctypes.c_double(float(threshold)), ctypes.c_double(self.tie_rel), int(max_picks),
                                             *self._w()), "choi_shard_select")

    def status(self, with_picks=False):
        """(n, picks, done[, pick list]) -- synchronises the stream."""
        import ctypes
        st = (ctypes.c_int64 * 3)()
        buf = (ctypes.c_int64 * self.cap)() if with_picks else None
        self.nat.check(self.lib.choi_shard_status(self.G, self.cap, *self._w()[:2], st, buf, self.nat.stream_ptr()),
                       "choi_shard_status")
        out = (st[0], st[1], bool(st[2]))
        return out + ([buf[i] for i in range(st[1])],) if with_picks else out

    def grow(self, n, rows):
        """Cache full: a larger one with rows [0, n) kept (every rank decides this from the same n)."""
        bigger = torch.empty((self.cap + rows, self.G), dtype=torch.float64, device=self.grid.device)
        bigger[:n].copy_(self.Vc[:n])
        self.Vc, self.cap = bigger, self.cap + rows
        self._buffers()


def plan_shards(planners, exchange, threshold, chunk=128, console=False, max_picks=None):
    """Greedy picks (global grid indices, selection order) of the shards of one grid.  `planners`: the ShardPlanners this
    process drives (one per rank in a process group; all shards when one process emulates the group); `exchange(slots)`
    turns their send slots into the slots of every rank, recv[world, cap + 4] in rank order (an all-gather).  Every shard
    gets the same picks; the cache grows in lockstep since every shard sees the same n.  `max_picks`: stop after that many
    picks even while the maximum variance is still above the threshold (None: no limit)."""
    picks = []
    n = planners[0].n0
    while True:
        room = planners[0].cap - n
        limit = room if max_picks is None else min(room, max_picks - len(picks))
        recv = exchange([p.begin(n) for p in planners])
        for p in planners:
            p.select(recv, threshold, limit)
        while True:
            for _ in range(PLAN_BATCH):
                for p in planners:
                    p.append()
                recv = exchange([p.propose() for p in planners])
                for p in planners:
                    p.select(recv, threshold, limit)
            _, _, done = planners[0].status()
            if done:
                break
        n, k, _, got = planners[0].status(with_picks=True)
        picks.extend(got)
        print(f"Found {len(picks)} sample points so far") if console else None
        if k < room or (max_picks is not None and len(picks) >= max_picks):
            break
        for p in planners:                  # V cache full: grow, resume
            p.grow(n, chunk * 2)
    return np.asarray(picks, dtype=np.int64)


def sharded_sample_points(model, shard_grid, threshold, group=None, console=False):
    """compute_sample_points on a grid sharded over `group`: this rank plans on its slice `shard_grid` (a CoverageGrid with
    the base index and axes of a whole-column slice, see column_split), one all-gather of the shards' send slots per pick.
    Returns (points[k, 2], global grid indices[k]), the same on every rank."""
    world = dist.get_world_size(group)
    planner = ShardPlanner(model, shard_grid)

    def exchange(slots):
        recv = torch.empty((world, slots[0].numel()), dtype=slots[0].dtype, device=slots[0].device)
        dist.all_gather_into_tensor(recv, slots[0], group=group)
        return recv

    idx = plan_shards([planner], exchange, threshold, console=console)
    axes = shard_grid.axes
    pts = np.column_stack((axes.ux_host[idx // axes.ny], axes.uy_host[idx % axes.ny])) if idx.size else np.empty([0, 2])
    return pts, idx
