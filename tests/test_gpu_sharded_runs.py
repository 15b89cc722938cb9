"""Grid-sharded simulations: the sharded Choi planner (choi_shard_*, sharding.ShardPlanner) with K shards emulated in one
process -- the all-gather of the send slots done with torch.stack -- against the single-GPU planner and the oracle, and
whole runs of the four algorithms over real NCCL process groups (`group=`) against the oracle loops and the single-GPU run."""
import ctypes
import os
import pickle
import random
import socket

import numpy as np
import pytest
import torch

from oracle import algorithms as oalg
from tests import synth

pytestmark = pytest.mark.gpu


def _model(n_grid, N):
    from mfgp_coverage_b200 import simulator as sim
    xy = synth.grid(n_grid)
    f = synth.truth_function(xy)
    X_L, y_L, X_H, y_H = synth.training_set(xy, f, N)
    m = sim.init_MFGP(synth.MF_HYP, np.column_stack((X_L, y_L)))
    m.updt_info(X_L, y_L, X_H, y_H)
    return xy, m


def _shard_grids(xy, cols):
    """CoverageGrids of whole-column slices with `cols` columns each (left to right)."""
    from mfgp_coverage_b200._coverage import CoverageGrid
    from mfgp_coverage_b200._engine import TensorAxes, detect_tensor_grid
    ux, uy = detect_tensor_grid(xy)
    assert sum(cols) == ux.size
    axes = TensorAxes(ux, uy, torch.device("cuda", torch.cuda.current_device()))
    grids, c = [], 0
    for k in cols:
        lo, hi = c * uy.size, (c + k) * uy.size
        grids.append(CoverageGrid(xy[lo:hi], base_index=lo, axes=axes))
        c += k
    return grids


def _emulated(model, xy, cols, thr, chunk=128, max_picks=None):
    """Picks of K emulated shards and the shards' planners (their var after planning)."""
    from mfgp_coverage_b200 import sharding
    planners = [sharding.ShardPlanner(model, g, chunk) for g in _shard_grids(xy, cols)]
    return sharding.plan_shards(planners, torch.stack, thr, chunk, max_picks=max_picks), planners


def _single(model, xy, thr, rows):
    """choi_greedy as compute_sample_points calls it, with room for `rows` picks: (picks, var after planning)."""
    from mfgp_coverage_b200 import _coverage as cv
    from mfgp_coverage_b200 import _native as nat
    grid = cv.CoverageGrid(xy)
    eng = model.engine
    n, G = eng.N, grid.G
    Vc = torch.empty((n + rows, G), dtype=torch.float64, device=grid.device)
    q = torch.empty(G, dtype=torch.float64, device=grid.device)
    _, var = model.predict_device(grid.xy, vcache=Vc, grid=grid, q_out=q)
    lib = nat.lib()
    work = torch.empty(int(lib.cov_workspace_bytes(G, 1, 0)) // 8 + (G // 256 + 2) * 2 + 64 + (1 << 15), dtype=torch.float64,
                       device=grid.device)
    buf = (ctypes.c_int64 * rows)()
    k = lib.choi_greedy(nat.ptr(grid.xy), G, nat.ptr(Vc), G, n, n + rows, nat.ptr(var), nat.ptr(q), ctypes.byref(eng.pstruct),
                        ctypes.c_double(float(thr)), ctypes.c_double(cv.AMAX_REL), rows, buf, nat.ptr(work), work.numel() * 8,
                        nat.stream_ptr())
    assert k >= 0
    return np.array(buf[:k], dtype=np.int64), var.cpu().numpy()


@pytest.fixture(scope="module")
def planner_case():
    """The 30x30 inputs of test_choi_planner_matches_reference_greedy and the oracle's picks."""
    from oracle import coverage as ocov, gp as ogp
    xy, m = _model(30, 40)
    f = synth.truth_function(xy)
    X_L, y_L, X_H, y_H = synth.training_set(xy, f, 40)
    om = ogp.Model(ogp.GPParams.from_hyp(synth.MF_HYP), X_L, y_L, X_H, y_H)
    om.updt_info()
    _, var = om.predict(xy)
    thr = 0.55 * var.max()
    _, idx_o = ocov.compute_sample_points(om, xy, thr)
    return xy, m, thr, np.asarray(idx_o, dtype=np.int64)


@pytest.mark.parametrize("cols", [[30], [1, 29], [7, 11, 12], [7, 8, 7, 8]])
def test_sharded_planner_matches_single_gpu(planner_case, cols):
    from mfgp_coverage_b200 import simulator as sim
    from mfgp_coverage_b200.gaussian_process import prior_variance
    xy, m, thr, idx_o = planner_case
    mu0, var0 = m.predict(xy)
    idx_s, var_s = _single(m, xy, thr, 128)
    idx_k, planners = _emulated(m, xy, cols, thr)
    pts_g, idx_g = sim.compute_sample_points(m, xy, thr, False, return_indices=True)
    assert len(idx_o) > 5
    assert np.array_equal(idx_k, idx_o) and np.array_equal(idx_k, idx_g) and np.array_equal(idx_k, idx_s)
    k0 = prior_variance(m.params())
    var_k = np.concatenate([p.var.cpu().numpy() for p in planners])
    assert np.max(np.abs(var_k - var_s)) <= 1e-12 * k0
    mu1, var1 = m.predict(xy)                                    # the model is untouched
    assert m.engine.N == 40
    assert np.max(np.abs(mu1 - mu0)) <= 1e-12 and np.max(np.abs(var1 - var0)) <= 1e-12 * k0


def test_sharded_planner_odd_column_length():
    """ny = 31: the V cache's row stride is odd, so the append pass takes its scalar loads on every shard."""
    from mfgp_coverage_b200 import simulator as sim
    from mfgp_coverage_b200.gaussian_process import prior_variance
    xy, m = _model(31, 40)
    thr = 0.55 * m.predict(xy)[1].max()
    idx_s, var_s = _single(m, xy, thr, 128)
    idx_k, planners = _emulated(m, xy, [7, 11, 13], thr)
    assert len(idx_s) > 5
    assert np.array_equal(idx_k, idx_s)
    assert np.array_equal(idx_k, sim.compute_sample_points(m, xy, thr, False, return_indices=True)[1])
    var_k = np.concatenate([p.var.cpu().numpy() for p in planners])
    assert np.max(np.abs(var_k - var_s)) <= 1e-12 * prior_variance(m.params())


def test_sharded_planner_ties_go_to_lowest_global_index():
    """A prior mirror-symmetric in x on a 31 x 31 grid, split [15 | 16] columns: mirror-image grid points lie on
    different shards.  The data cover x <= 0.2 and x >= 0.8, so the picks start on the mirror axis (column 15),
    which keeps the posterior symmetric, and later picks meet mirror twins tied under the arg-max rule in the proposes
    of two shards after earlier appends.  Every such tie must go to the lower global index, as on one GPU."""
    from mfgp_coverage_b200 import _coverage as cv
    from mfgp_coverage_b200 import simulator as sim
    from mfgp_coverage_b200.gaussian_process import prior_variance
    n = 31
    xy = synth.grid(n)
    f = synth.truth_function(xy)
    left = (np.arange(0, 8, 2)[:, None] * n + np.arange(0, n, 3)[None, :]).reshape(-1)   # x <= 0.2, every third row
    y = f[left] + np.random.default_rng(5).normal(0, 0.1, left.size)
    mirrored = np.column_stack((1.0 - xy[left, 0], xy[left, 1]))
    prior = np.vstack([np.column_stack((xy[left], y)), np.column_stack((mirrored, y))])
    model, _ = sim._init_models("S", synth.SF_HYP, prior)
    k0 = prior_variance(model.params())
    picks = 40
    idx_s, _ = _single(model, xy, 0.0, picks)
    idx_k, _ = _emulated(model, xy, [15, 16], 0.0, max_picks=picks)
    assert len(idx_s) == picks
    assert np.array_equal(idx_k, idx_s)
    tied_after_append = 0
    for k, p in enumerate(idx_k.tolist()):
        m = (n - 1 - p // n) * n + p % n
        if m == p:
            continue
        var_k = _single(model, xy, 0.0, k)[1]                      # the variance pick k was chosen from
        a, b = var_k[p], var_k[m]
        if abs(a - b) <= cv.AMAX_REL * (k0 - min(a, b)):          # argmax_combine's tie condition
            assert (p < 15 * n) != (m < 15 * n)                    # twins on different shards
            assert p < m                                           # the lower global index won
            tied_after_append += k >= 1
    assert tied_after_append >= 1


def test_sharded_planner_cache_growth(planner_case):
    """An initial chunk of 4 rows: the V caches of all shards grow several times during planning."""
    from mfgp_coverage_b200 import simulator as sim
    xy, m, thr, idx_o = planner_case
    idx_k, planners = _emulated(m, xy, [7, 11, 12], thr, chunk=4)
    assert len(idx_k) > 12
    assert all(p.cap > p.n0 + 4 for p in planners)
    assert np.array_equal(idx_k, sim.compute_sample_points(m, xy, thr, False, return_indices=True)[1])


def test_sharded_planner_c3_size():
    from mfgp_coverage_b200 import sharding
    from mfgp_coverage_b200 import simulator as sim
    xy, m = _model(256, 1024)
    _, var60 = _single(m, xy, 0.0, 60)                           # max var left after 60 picks: a threshold for >= 60
    thr = float(var60.max()) * (1 - 1e-9)
    idx_g = sim.compute_sample_points(m, xy, thr, False, return_indices=True)[1]
    cols = [(sharding.column_split(xy, 4, r)[1] - sharding.column_split(xy, 4, r)[0]) // 256 for r in range(4)]
    idx_k, _ = _emulated(m, xy, cols, thr)
    assert len(idx_g) >= 50
    assert np.array_equal(idx_k, idx_g)


def test_sharded_planner_rejects_bad_arguments(planner_case):
    from mfgp_coverage_b200 import _native as nat
    from mfgp_coverage_b200 import sharding
    xy, m, thr, _ = planner_case
    p = sharding.ShardPlanner(m, _shard_grids(xy, [10, 20])[1])
    p.begin(p.n0)
    torch.cuda.synchronize()
    lib = nat.lib()
    bufs = [p.send, p.work, p.Vc, p.var, p.q]
    before = [b.clone() for b in bufs]
    prm, rel, wb, s = ctypes.byref(m.engine.pstruct), ctypes.c_double(p.tie_rel), p.work.numel() * 8, nat.stream_ptr()
    X, V, var, send, work = (nat.ptr(t) for t in (p.grid.xy, p.Vc, p.var, p.send, p.work))
    assert lib.choi_shard_begin(X, p.G, p.base, V, p.G - 1, p.n0, p.cap, var, prm, rel, send, work, wb, s) == -1   # ldv < G
    assert lib.choi_shard_begin(X, p.G, p.base, V, p.G, p.n0, p.n0 - 1, var, prm, rel, send, work, wb, s) == -1   # cap < n
    short = int(lib.choi_shard_workspace_bytes(p.G, p.cap)) - 8
    assert lib.choi_shard_begin(X, p.G, p.base, V, p.G, p.n0, p.cap, var, prm, rel, send, work, short, s) == -1
    assert lib.choi_shard_append(X, p.G, p.base, V, p.G, p.cap, var, nat.ptr(p.q), prm, rel, work, short, s) == -1
    assert lib.choi_shard_propose(X, p.G, p.base, V, p.G - 1, p.cap, prm, rel, send, work, wb, s) == -1
    assert lib.choi_shard_select(send, 1, p.G, p.cap, prm, ctypes.c_double(thr), rel, 8, work, short, s) == -1
    torch.cuda.synchronize()
    for a, b in zip(bufs, before):
        assert torch.equal(a.view(torch.int64), b.view(torch.int64))


# ---- whole runs over real process groups -------------------------------------------------------------------------------

RUNS = [("lloyd", 32, 5, 8, False), ("todescato", 40, 6, 10, True), ("periodic", 32, 5, 12, False),
        ("choi", 36, 4, 24, True)]


def _inputs(n, A, multi):
    """The seeded synthetic inputs of test_synthetic_runs_vs_oracle_loops."""
    xy = synth.grid(n)
    truth_arr = np.column_stack((xy, synth.truth_function(xy)))
    hyp = synth.MF_HYP if multi else synth.SF_HYP
    lat_xy = np.random.default_rng(99).random((9, 2))
    near = np.argmin(((xy[None, :, :] - lat_xy[:, None, :]) ** 2).sum(axis=2), axis=1)
    prior_arr = np.column_stack((lat_xy, 0.8 * truth_arr[near, 2] + 0.02))
    return truth_arr, hyp, prior_arr, synth.agents(A, 21)


def _run(algo, n, A, T, multi, group, seeded=True):
    from mfgp_coverage_b200 import simulator as sim
    truth_arr, hyp, prior_arr, pos0 = _inputs(n, A, multi)
    kw = dict(rng=random.Random(21), noise_rng=np.random.default_rng(21)) if seeded else {}
    return getattr(sim, algo)(algo, 0, T, A, pos0.copy(), truth_arr, 0.1, prior_arr, hyp, False, None, True, group=group, **kw)


def _worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        group = dist.group.WORLD
        res = {algo: _run(algo, n, A, T, multi, group) for algo, n, A, T, multi in RUNS}
        res["unseeded"] = _run("todescato", 40, 6, 10, True, group, seeded=False)
        if world == 1:
            res["none"] = {algo: _run(algo, n, A, T, multi, None) for algo, n, A, T, multi in RUNS}
        with open(f"{out}.{rank}", "wb") as fh:
            pickle.dump(res, fh)
    finally:
        dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _spawn(world, tmp_path):
    import torch.multiprocessing as mp
    out = str(tmp_path / f"logs{world}")
    mp.spawn(_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    res = []
    for r in range(world):
        with open(f"{out}.{r}", "rb") as fh:
            res.append(pickle.load(fh))
    return res


def _arrays(logs, A):
    from tests.test_gpu_algorithms import _agent_array
    lg, ag, sg = logs
    loss = np.array([r["Loss"] for r in lg])
    samples = np.array([[float(r["Iteration"]), float(r["Agent"]), float(r["X"]), float(r["Y"]), float(r["Sample"])]
                        for r in sg if r["Agent"] != "NA"]).reshape(-1, 5)
    return loss, _agent_array(ag, len(lg), A), samples


@pytest.mark.parametrize("world", [2, 4])
def test_sharded_runs_match_oracle_and_single_gpu(world, tmp_path):
    from tests.test_gpu_algorithms import _compare
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    res = _spawn(world, tmp_path)
    for r in range(1, world):                                    # every rank returns the same logs
        assert pickle.dumps(res[r]) == pickle.dumps(res[0])
    for algo, n, A, T, multi in RUNS:
        truth_arr, hyp, prior_arr, pos0 = _inputs(n, A, multi)
        if algo == "lloyd":
            ref = oalg.lloyd(0, T, A, pos0.copy(), truth_arr)
        else:
            ref = getattr(oalg, algo)(0, T, A, pos0.copy(), truth_arr, 0.1, prior_arr, hyp, random.Random(21),
                                      np.random.default_rng(21))
        single = _run(algo, n, A, T, multi, None)
        got = _arrays(res[0][algo], A)
        for other in (_arrays(ref, A), _arrays(single, A)):
            _compare(*got, *other, truth_arr)


def test_world_size_one_group_is_the_single_gpu_path(tmp_path):
    res = _spawn(1, tmp_path)[0]
    for algo, *_ in RUNS:
        assert pickle.dumps(res[algo]) == pickle.dumps(res["none"][algo])
