"""GPU: Thompson-sampling runs on the batched stepper (BatchedRuns("thompson"), csrc/batched_thompson.cu) against
simulator.thompson run with VORONOI = "clip" at each run's device normals and noise, against the oracle loop on an irregular
grid, graph replay, batch composition, the device generator, argument errors and the runner's batched mode."""
import ctypes
import os

import numpy as np
import pandas as pd
import pytest

from oracle import sample_centroids as osc
from tests import synth
from tests.test_batched_thompson_generator import device_normals_reference

pytestmark = pytest.mark.gpu


def _uniform(n):
    xy = synth.grid(n)
    return np.column_stack((xy, synth.truth_function(xy)))


def _irregular(nx, ny, seed=3):
    rng = np.random.default_rng(seed)
    ux = np.sort(np.concatenate(([0.0, 1.0], rng.uniform(0.0, 1.0, nx - 2))))
    uy = np.sort(np.concatenate(([0.0, 1.0], rng.uniform(0.0, 1.0, ny - 2))))
    xy = np.array([[x, y] for x in ux for y in uy])
    return np.column_stack((xy, synth.truth_function(xy)))


def _prior(truth_arr, k=9, seed=99):
    lat = np.random.default_rng(seed).random((k, 2))
    near = np.argmin(((truth_arr[None, :, :2] - lat[:, None, :]) ** 2).sum(axis=2), axis=1)
    return np.column_stack((lat, 0.8 * truth_arr[near, 2] + 0.02))


class _DeviceNormals:
    """Stands in for simulator.thompson's numpy Generator: standard_normal((d, A)) returns the normals run r of a batch used
    at the same iteration."""

    def __init__(self, br, r):
        self.br, self.r, self.t = br, r, 0

    def standard_normal(self, shape):
        E = self.br.draw_normals(self.t)[self.r].cpu().numpy()
        assert E.shape == tuple(shape), (E.shape, shape)
        self.t += 1
        return E


def _batched(truth_arr, prior_arr, hyp, A, T, starts, seeds, noise, use_graph=False):
    from mfgp_coverage_b200._batched import BatchedRuns
    return BatchedRuns("thompson", truth_arr, prior_arr, hyp, A, T, starts, noise=noise, seeds=seeds).run(use_graph=use_graph)


def _near_midpoint(t, u, tol=1e-9):
    s = np.sort(u)
    return bool(np.any(np.abs(t - 0.5 * (s[1:] + s[:-1])) <= tol))


def _compare(batched, ref, A, ux, uy):
    """test_seeded_thompson_run_reproduces_the_oracle_loop's rule: positions and samples exact, loss within 1e-9
    relative, VarMax / centroids / Distance within 1e-9; the comparison stops at a position flipped by a target within 1e-9
    of a grid midpoint."""
    (loss, agent, samples), (oloss, oagent, osamples) = batched, ref
    T = len(oloss)
    assert len(loss) == T and len(agent) == T * A
    for t in range(T):
        rows, orows = agent[t * A:(t + 1) * A], oagent[t * A:(t + 1) * A]
        xy = np.array([[r["X"], r["Y"]] for r in rows])
        oxy = np.array([[r["X"], r["Y"]] for r in orows])
        if not np.array_equal(xy, oxy):
            prev = oagent[(t - 1) * A:t * A]
            moved = np.nonzero(np.any(xy != oxy, axis=1))[0]
            assert t > 0 and all(_near_midpoint(prev[i]["XCentroid"], ux) or _near_midpoint(prev[i]["YCentroid"], uy)
                                 for i in moved), (t, moved)
            return t
        assert abs(loss[t]["Loss"] - oloss[t]["Loss"]) <= 1e-9 * abs(oloss[t]["Loss"]), t
        for k in ("VarMax", "XCentroid", "YCentroid", "Distance"):
            a = np.array([r[k] for r in rows], dtype=np.float64)
            b = np.array([r[k] for r in orows], dtype=np.float64)
            scale = max(1.0, abs(float(rows[0]["Var0"]))) if k == "VarMax" else 1.0
            assert np.array_equal(np.isnan(a), np.isnan(b)) and np.nanmax(np.abs(a - b), initial=0.0) <= 1e-9 * scale, (t, k)
        for k in ("Var0", "ProbExplore", "Explore"):
            assert [r[k] for r in rows] == pytest.approx([r[k] for r in orows], rel=1e-12, abs=1e-12), (t, k)
    key = lambda s: (int(s["Iteration"]), int(s["Agent"]), s["X"], s["Y"])         # noqa: E731
    assert [key(s) for s in samples] == [key(s) for s in osamples]
    assert np.allclose([s["Sample"] for s in samples], [s["Sample"] for s in osamples], rtol=0, atol=1e-15)
    return T


CASES = {"hmf_uniform": (lambda: _uniform(32), True, 6, 16),
         "nsf_uniform": (lambda: _uniform(28), False, 5, 14),
         "hmf_irregular": (lambda: _irregular(30, 26), True, 8, 12),
         "nsf_irregular": (lambda: _irregular(27, 31, seed=8), False, 7, 20)}


@pytest.mark.parametrize("case", sorted(CASES))
def test_batched_thompson_runs_match_clip_thompson_run_by_run(case, monkeypatch):
    from mfgp_coverage_b200 import simulator as sim
    from mfgp_coverage_b200._batched import _NoiseRow
    make, multi, A, T = CASES[case]
    truth_arr = make()
    prior_arr, hyp = (_prior(truth_arr), synth.MF_HYP) if multi else (None, synth.SF_HYP)
    R = 4
    starts = np.stack([synth.agents(A, 300 + r) for r in range(R)])
    seeds = [(2 ** 63 + 12345 * r) if r % 2 else 77 + r for r in range(R)]
    noise = np.stack([np.random.default_rng(700 + r).normal(0, 0.1, T * A) for r in range(R)])
    br = _batched(truth_arr, prior_arr, hyp, A, T, starts, seeds, noise)
    logs = br.logs()
    monkeypatch.setattr(sim, "VORONOI", "clip")
    ux, uy = osc.tensor_axes(truth_arr[:, :2])
    compared = []
    for r in range(R):
        pos = starts[r].copy()
        ref = sim.thompson("thompson", r, T, A, pos, truth_arr, 0.1, prior_arr, hyp, False, None, True,
                           rng=_DeviceNormals(br, r), noise_rng=_NoiseRow(noise[r]))
        compared.append(_compare(logs[r], ref, A, ux, uy))
        if compared[-1] == T:
            assert np.array_equal(br.final_positions()[r], pos)
    assert sum(compared) >= R * T // 2, compared          # the midpoint rule cuts at most a few runs short


def test_batched_thompson_matches_the_oracle_loop_on_an_irregular_grid():
    from mfgp_coverage_b200._batched import _NoiseRow
    from tests.test_gpu_sample_centroids import _orders_of
    truth_arr = _irregular(22, 20, seed=5)
    prior_arr, hyp = _prior(truth_arr, 6, seed=4), synth.MF_HYP
    R, A, T = 4, 5, 12
    starts = np.stack([synth.agents(A, 40 + r) for r in range(R)])
    noise = np.stack([np.random.default_rng(90 + r).normal(0, 0.1, T * A) for r in range(R)])
    br = _batched(truth_arr, prior_arr, hyp, A, T, starts, [11, 12, 13, 14], noise)
    logs = br.logs()
    ux, uy = osc.tensor_axes(truth_arr[:, :2])
    for r in (0, 3):
        ref = osc.thompson(r, T, A, starts[r].copy(), truth_arr, 0.1, prior_arr, hyp, _DeviceNormals(br, r),
                           _NoiseRow(noise[r]), _orders_of)
        assert _compare(logs[r], ref, A, ux, uy) == T


def test_thompson_graph_replay_is_bitwise_the_eager_run():
    import torch
    truth_arr = _uniform(32)
    prior_arr = _prior(truth_arr)
    R, A, T = 5, 6, 14
    starts = np.stack([synth.agents(A, 10 + r) for r in range(R)])
    noise = np.random.default_rng(2).normal(0, 0.1, (R, T * A))
    a = _batched(truth_arr, prior_arr, synth.MF_HYP, A, T, starts, list(range(R)), noise)
    b = _batched(truth_arr, prior_arr, synth.MF_HYP, A, T, starts, list(range(R)), noise, use_graph=True)
    assert b.graph is not None
    for name in ("log_loss", "log_agent", "log_sample", "nsamples", "Ncur", "mu", "var", "pos", "pos_idx", "cen"):
        assert torch.equal(getattr(a, name), getattr(b, name)), name
    assert int(a.nsamples.sum()) == R * (T - 1) * A


def test_a_run_gives_the_same_bits_alone_and_inside_a_batch():
    import torch
    truth_arr = _irregular(26, 24)
    prior_arr = _prior(truth_arr)
    A, T = 7, 12
    starts = np.stack([synth.agents(A, 500 + r) for r in range(8)])
    noise = np.random.default_rng(6).normal(0, 0.1, (8, T * A))
    seeds = [1000 + r for r in range(8)]
    batch = _batched(truth_arr, prior_arr, synth.MF_HYP, A, T, starts, seeds, noise)
    for r in (0, 5):
        alone = _batched(truth_arr, prior_arr, synth.MF_HYP, A, T, starts[r:r + 1], seeds[r:r + 1], noise[r:r + 1])
        for name in ("log_loss", "log_agent", "log_sample", "pos"):
            assert torch.equal(getattr(alone, name)[0], getattr(batch, name)[r]), (r, name)
        for t in (0, T - 1):
            assert torch.equal(alone.draw_normals(t)[0], batch.draw_normals(t)[r])
    again = _batched(truth_arr, prior_arr, synth.MF_HYP, A, T, starts, seeds, noise)
    assert torch.equal(again.log_agent, batch.log_agent) and torch.equal(again.log_loss, batch.log_loss)


def test_device_normals_follow_the_documented_generator_and_look_standard_normal():
    truth_arr = _uniform(24)
    from mfgp_coverage_b200._batched import BatchedRuns
    seeds = [3, 2 ** 64 - 5, 123456789123] + [2 ** 40 + k for k in range(5)]
    br = BatchedRuns("thompson", truth_arr, _prior(truth_arr), synth.MF_HYP, 16, 40, np.stack([synth.agents(16, s) for s in
                                                                                              range(8)]), seeds=seeds)
    E = {t: br.draw_normals(t).cpu().numpy() for t in (0, 7, 20, 39)}
    R, d, A = E[39].shape
    assert d == br.d0 + br.N0 + 16 * 39
    for t, e in E.items():          # a restatement of Philox4x32-10 + Box-Muller (tests/test_batched_thompson_generator.py)
        for r in range(R):
            rows = np.arange(e.shape[1])[:, None] * np.ones((1, A), dtype=np.int64)
            ref = device_normals_reference(seeds[r], t, rows, np.arange(A)[None, :] * np.ones_like(rows))
            assert np.max(np.abs(e[r] - ref)) <= 1e-12
    big = np.concatenate([E[t].reshape(-1) for t in E])
    n = big.size
    assert n >= 10 ** 6
    assert abs(big.mean()) <= 5 / np.sqrt(n) and abs(big.var() - 1) <= 6 * np.sqrt(2 / n)
    assert abs(np.mean(big ** 3)) <= 6 * np.sqrt(15 / n) and abs(np.mean(big ** 4) - 3) <= 6 * np.sqrt(96 / n)
    e = E[39]
    corr = lambda a, b: float(np.corrcoef(a.reshape(-1), b.reshape(-1))[0, 1])       # noqa: E731
    lim = 6 / np.sqrt(e[0].size)
    assert abs(corr(e[0][1:], e[0][:-1])) <= lim                       # neighbouring rows
    assert abs(corr(e[0][:, 1:], e[0][:, :-1])) <= 6 / np.sqrt(e[0][:, 1:].size)   # neighbouring agents
    assert abs(corr(e[0], e[1])) <= lim and abs(corr(e[1], e[2])) <= lim          # seeds
    m = E[7].shape[1]
    assert abs(corr(E[7][0], E[39][0][:m])) <= 6 / np.sqrt(E[7][0].size)         # iterations
    assert len(np.unique(big)) == big.size


def test_errors_are_raised_before_any_launch():
    from mfgp_coverage_b200 import _native as nat
    from mfgp_coverage_b200._batched import BatchedRuns
    truth_arr = _uniform(24)
    prior_arr = _prior(truth_arr)
    T = 10
    lib = nat.lib()
    n0 = lib.mfgp_launch_count()
    with pytest.raises(ValueError, match="at most 16 agents"):
        BatchedRuns("thompson", truth_arr, prior_arr, synth.MF_HYP, 17, T, synth.agents(17)[None])
    with pytest.raises(ValueError, match="tensor-product grid"):
        BatchedRuns("thompson", truth_arr[np.random.default_rng(0).permutation(len(truth_arr))], prior_arr, synth.MF_HYP, 4, T,
                    synth.agents(4)[None])
    out = synth.agents(4)[None].copy()
    out[0, 2] = (1.5, 0.5)
    with pytest.raises(ValueError, match="cushioned bounding box"):
        BatchedRuns("thompson", truth_arr, prior_arr, synth.MF_HYP, 4, T, out)
    with pytest.raises(ValueError, match="simulator.thompson"):
        BatchedRuns("thompson", truth_arr, prior_arr, synth.MF_HYP, 16, 60, synth.agents(16)[None])
    short = synth.SF_HYP.copy()
    short[2] = np.log(0.004)
    with pytest.raises(ValueError, match="needs more than 64 Chebyshev terms"):
        BatchedRuns("thompson", truth_arr, None, short, 4, T, synth.agents(4)[None])
    assert lib.mfgp_launch_count() == n0


def test_c_entry_points_reject_bad_arguments_with_buffers_intact():
    import torch
    from mfgp_coverage_b200 import _native as nat
    truth_arr = _uniform(24)
    br = _batched(truth_arr, _prior(truth_arr), synth.MF_HYP, 5, 6, np.stack([synth.agents(5, 1)] * 2), [1, 2], None)
    lib, sp = nat.lib(), nat.stream_ptr()
    keep = {k: getattr(br, k).clone() for k in ("pos", "log_agent", "work", "prev", "cen", "pos_idx")}
    n0 = lib.mfgp_launch_count()
    b, p = br._b, ctypes.byref(br.pstruct)
    run = lambda it=0, work=None, nbytes=None: lib.mfgp_batch_thompson(  # noqa: E731
        ctypes.byref(b), p, it, nat.ptr(br.work) if work is None else work, br.work.numel() * 8 if nbytes is None else nbytes, sp)
    assert run(it=6) == nat.MFGP_ERR_INVALID and run(it=-1) == nat.MFGP_ERR_INVALID
    assert run(nbytes=8) == nat.MFGP_ERR_INVALID
    assert run(work=ctypes.c_void_p(br.work.data_ptr() + 8)) == nat.MFGP_ERR_INVALID
    assert lib.mfgp_batch_thompson(None, p, 0, nat.ptr(br.work), br.work.numel() * 8, sp) == nat.MFGP_ERR_INVALID
    for field, bad in (("algo", 1), ("rxH", 65), ("ryL", 0), ("A", 17), ("bxhi", b.bxlo), ("cmask", None), ("seed", None)):
        old = getattr(b, field)
        setattr(b, field, bad)
        assert run() == nat.MFGP_ERR_INVALID, field
        setattr(b, field, old)
    out = torch.full((2, 10, 5), -7.25, dtype=torch.float64, device=br.dev)
    assert lib.mfgp_batch_thompson_normals(ctypes.byref(b), 0, 0, nat.ptr(out), sp) == nat.MFGP_ERR_INVALID
    assert lib.mfgp_batch_thompson_normals(ctypes.byref(b), 6, 10, nat.ptr(out), sp) == nat.MFGP_ERR_INVALID
    assert lib.mfgp_batch_thompson_normals(ctypes.byref(b), 0, 10, None, sp) == nat.MFGP_ERR_INVALID
    assert lib.mfgp_launch_count() == n0
    torch.cuda.synchronize()
    assert bool((out == -7.25).all())
    for k, v in keep.items():
        assert torch.equal(getattr(br, k), v), k
    assert lib.mfgp_batch_thompson_workspace_bytes(None) == 0
    assert run() == nat.MFGP_OK           # the restored struct is accepted


def test_runner_batched_thompson_writes_the_sequential_csvs(golden_dir, tmp_path):
    """runner.run(batched=True) for Thompson: the sequential mode's columns and shapes, and the same start positions (the
    2 A coordinates, then one random.getrandbits(64) per simulation): iteration 0's loss and agent rows agree except for
    the centroid columns, whose draws come from another generator."""
    from mfgp_coverage_b200 import runner
    from tests.test_gpu_runner import _write_inputs
    name, null = _write_inputs(golden_dir, str(tmp_path))
    kw = dict(name=name, agents=6, iterations=4, simulations=3, sigma_n=0.1, seed=9, null_prior_path=null, n_processors=1)
    try:
        runner.run(prefix=os.path.join(str(tmp_path), "seq"), algorithms=["thompson_hmf"], batched=False, **kw)
        runner.run(prefix=os.path.join(str(tmp_path), "bat"), algorithms=["thompson_hmf"], batched=True, **kw)
    finally:
        runner.BATCHED = False
        os.environ["MFGP_BATCHED"] = "0"
    for kind in ("loss", "agent", "sample"):
        a = pd.read_csv(os.path.join(str(tmp_path), f"seq_thompson_hmf_{kind}.csv"), index_col=0)
        b = pd.read_csv(os.path.join(str(tmp_path), f"bat_thompson_hmf_{kind}.csv"), index_col=0)
        assert list(a.columns) == list(b.columns) and a.shape == b.shape, kind
        if kind == "sample":
            continue
        a, b = a[a.Iteration == 0], b[b.Iteration == 0]
        num = [c for c in a.columns if c not in ("Fidelity", "XCentroid", "YCentroid")]
        assert np.allclose(a[num].values.astype(float), b[num].values.astype(float), rtol=1e-9, atol=1e-12), kind
