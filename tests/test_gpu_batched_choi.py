"""Choi on the batched replicate stepper (_batched.BatchedRuns, csrc/batched.cu): many runs planned, clustered, toured and
stepped together, against the oracle loops and the single-run simulator.choi run by run."""
import os
import random

import numpy as np
import pandas as pd
import pytest

from oracle import algorithms as oalg
from tests import synth
from tests.test_gpu_algorithms import _compare
from tests.test_gpu_batched import _inputs, _rows_to_arrays

gpu = pytest.mark.gpu


def _periods(logs):
    return [row["Period"] for row in logs[0]]


@pytest.mark.parametrize("iterations", [1, 8, 10, 24, 120])
def test_choi_schedule_matches_the_oracle_loop(iterations):
    """The loop checks `iteration < iterations` only between periods: the logged iterations and their periods."""
    from mfgp_coverage_b200._batched import choi_schedule
    xy = synth.grid(5)
    truth_arr = np.column_stack((xy, synth.truth_function(xy)))
    lo, _, _ = oalg.choi(0, iterations, 2, synth.agents(2, 3), truth_arr, 0.1, None, synth.SF_HYP, None,
                         np.random.default_rng(0))
    sched = choi_schedule(iterations)
    assert [r["Iteration"] for r in lo] == list(range(len(sched)))
    assert [r["Period"] for r in lo] == sched.tolist()


@gpu
@pytest.mark.parametrize("n,A,T,multi", [(36, 4, 24, True), (32, 5, 10, False), (30, 8, 56, True)])
def test_batched_choi_matches_the_oracle_loops_run_by_run(n, A, T, multi):
    """Every run against simulator.choi with the same start positions and noise draws, and with a prior also against the oracle
    loop (literal refit-per-pick planner).  Without a prior the period-0 picks are placed symmetrically, so the next period's
    variances tie between mirror-image grid points: bit-identical in the reference, ~1e-16 apart in any other operation order
    (the oracle's numpy included), where the reference's own seeded runs are the yardstick (next test)."""
    from mfgp_coverage_b200 import simulator as sim
    from mfgp_coverage_b200._batched import choi_schedule
    truth_arr, prior_arr, hyp = _inputs(n, multi)
    R = 4
    starts = np.stack([synth.agents(A, 300 + r) for r in range(R)])
    pos = starts.copy()
    logs = sim.run_batched("choi_hmf" if multi else "choi_nsf", list(range(R)), T, A, pos, truth_arr, 0.1, prior_arr, hyp,
                           noise_rngs=[np.random.default_rng(700 + r) for r in range(R)], exact_tie_loss=True)
    assert len(logs) == R
    for r in range(R):
        p0 = starts[r].copy()
        refs = [sim.choi("choi", r, T, A, p0, truth_arr, 0.1, prior_arr, hyp, False, None, True,
                         noise_rng=np.random.default_rng(700 + r))]
        if multi:
            refs.append(oalg.choi(r, T, A, starts[r].copy(), truth_arr, 0.1, prior_arr, hyp, None, np.random.default_rng(700 + r),
                                  fast_planner=False))
        l, a, s = _rows_to_arrays(logs[r], A)
        for ref in refs:
            lo, ao, so = _rows_to_arrays(ref, A)
            _compare(l, a, s, lo, ao, so, truth_arr)
            assert _periods(logs[r]) == _periods(ref) == choi_schedule(T).tolist()
            assert [row["Period"] for row in logs[r][2]] == [row["Period"] for row in ref[2]]
        assert np.allclose(pos[r], p0, atol=1e-9)


@gpu
@pytest.mark.parametrize("ds,name,hyp_key,use_prior", [("australia6", "choi_hmf", "mf_hyp", True),
                                                       ("australia6", "choi_nsf", "sf_hyp", False),
                                                       ("australia3", "choi_nsf", "sf_hyp", False)])
def test_seeded_reference_runs_through_the_batched_stepper(golden_dir, ds, name, hyp_key, use_prior):
    """The seeded runs of the unmodified reference (tests/golden/ref_runs.npz) as run 0 of a batch of two.  choi_nsf plans on
    tied variances far from the data: the test of the planner's k0 - q variance."""
    from mfgp_coverage_b200 import simulator as sim
    g = np.load(os.path.join(golden_dir, "ref_runs.npz"), allow_pickle=False)
    inp = np.load(os.path.join(golden_dir, f"inputs_{ds}.npz"))
    key = f"{ds}_{name}"
    A, T, seed = (int(v) for v in g[f"{key}_meta"])
    truth = pd.DataFrame(inp["truth"], columns=["X", "Y", "f_H"])
    prior = pd.DataFrame(inp["prior"] if use_prior else np.empty((0, 3)), columns=["X", "Y", "f_prior"])
    cols = ["mu_sf", "s^2_sf", "L_sf", "noise_sf"] if hyp_key == "sf_hyp" else \
        ["mu_lo", "s^2_lo", "L_lo", "mu_hi", "s^2_hi", "L_hi", "rho", "noise_lo", "noise_hi"]
    hyp = pd.DataFrame([inp[hyp_key]], columns=cols)
    random.seed(seed)
    pos0 = np.column_stack(([random.random() for _ in range(A)], [random.random() for _ in range(A)]))
    assert np.array_equal(pos0, g[f"{key}_start"])
    pos = np.stack([pos0, np.random.default_rng(seed + 1).random((A, 2))])
    logs = sim.run_batched(name, [0, 1], T, A, pos, truth, 0.1, prior, hyp,
                           noise_rngs=[np.random.default_rng(seed), np.random.default_rng(seed + 1)], exact_tie_loss=True)
    loss, agent, samples = _rows_to_arrays(logs[0], A)
    _compare(loss, agent, samples, g[f"{key}_loss"], g[f"{key}_agent"], g[f"{key}_samples"], inp["truth"])
    assert _periods(logs[0]) == list(g[f"{key}_period"])


def _choi_batch(n, A, R, multi, T=8, cap=None, seed=300):
    from mfgp_coverage_b200._batched import BatchedRuns
    truth_arr, prior_arr, hyp = _inputs(n, multi)
    starts = np.stack([synth.agents(A, seed + r) for r in range(R)])
    br = BatchedRuns("choi", truth_arr, prior_arr, hyp, A, T, starts, noise_rngs=[np.random.default_rng(700 + r) for r in range(R)],
                     cap=cap)
    return br, truth_arr


def _oracle_model(br, r, hyp):
    from oracle import gp as ogp
    N, NL = int(br.Ncur[r]), br.NL
    X, y = br.Xt[r, :N].cpu().numpy(), br.y[r, :N].cpu().numpy().reshape(-1, 1)
    m = ogp.Model(ogp.GPParams.from_hyp(hyp), X[:NL], y[:NL], X[NL:], y[NL:])
    m.updt_info()
    return m


@gpu
def test_batched_planner_matches_the_literal_greedy_and_leaves_the_models_alone():
    """compute_sample_points (simulator.py:326-374) refits and predicts per pick; the batched planner appends temporary rows
    to every run's own factor.  Runs with different training sets (after one period), index for index."""
    import torch
    from oracle import coverage as ocov
    R, A = 3, 4
    br, truth_arr = _choi_batch(30, A, R, True, T=24)
    br.run()
    before = {k: getattr(br, k).clone() for k in ("W", "z", "mu", "var", "Ncur")}
    thr = 0.5 * br.k0
    br.plan(thr)
    nplan = br.nplan.cpu().numpy()
    assert nplan.sum() > 5
    for r in range(R):
        _, idx = ocov.compute_sample_points(_oracle_model(br, r, synth.MF_HYP), truth_arr[:, :2], thr)
        assert np.array_equal(br.picks[r, :nplan[r]].cpu().numpy(), idx), r
        N = int(before["Ncur"][r])
        assert torch.equal(br.W[r, :N, :N], before["W"][r, :N, :N])
        assert torch.equal(br.z[r, :N], before["z"][r, :N])
    for k in ("mu", "var", "Ncur"):
        assert torch.equal(getattr(br, k), before[k]), k
    assert len({br.Xt[r, :int(br.Ncur[r])].cpu().numpy().tobytes() for r in range(R)}) > 1      # the runs did differ


@gpu
def test_capacity_growth_gives_the_same_runs():
    """Null prior: the planner outgrows a one-row capacity every period; the buffers grow between pick rounds."""
    import torch
    small, _ = _choi_batch(32, 5, 3, False, T=24, cap=1)
    ample, _ = _choi_batch(32, 5, 3, False, T=24, cap=400)
    cap0 = small.cap
    small.run()
    ample.run()
    assert small.cap > cap0 and ample.cap == 400
    for k in ("log_loss", "log_agent", "log_sample", "nsamples", "Ncur", "mu", "var", "pos"):
        assert torch.equal(getattr(small, k), getattr(ample, k)), k


@gpu
def test_clusters_and_tours_match_qhull_and_the_tour_oracle():
    """No ties: the clusters of every run's picks equal compute_sample_clusters on Qhull's cells (empty ones included),
    in selection order, and the tours equal oracle/tsp.py's."""
    from oracle import coverage as ocov
    from oracle import tsp as otsp
    R, A = 3, 8
    br, truth_arr = _choi_batch(30, A, R, True, seed=40)
    br.run()
    xy = truth_arr[:, :2]
    bbox = ocov.bounding_box_of(xy)
    empty = picks = 0
    for frac in (0.6, 0.75, 0.9):
        br.plan(frac * br.k0)
        br.cluster_and_tours(0, 16)
        assert br.cluster_ties[:, 0].sum() == 0
        nplan, cen = br.nplan.cpu().numpy(), br.cen.cpu().numpy().reshape(R, A, 2)
        off, tour = br.tour_off.cpu().numpy(), br.tour.cpu().numpy()
        picks += nplan.sum()
        for r in range(R):
            pts = xy[br.picks[r, :nplan[r]].cpu().numpy()]
            clusters = ocov.compute_sample_clusters(ocov.voronoi_bounded(cen[r], bbox), pts)
            tours = otsp.compute_sample_tsp(clusters)
            for c in range(A):
                got = xy[tour[off[r * A + c]:off[r * A + c + 1]]]
                assert np.array_equal(got, tours[c].reshape(-1, 2)), (r, c)
                assert sorted(map(tuple, got)) == sorted(map(tuple, clusters[c]))
                empty += clusters[c].shape[0] == 0
    assert empty > 0 and picks > 0


@gpu
def test_a_hard_clustering_tie_reruns_the_run_on_the_single_run_path():
    """Centroids symmetric about x = 0.5 and y = 0.5 on a grid that holds those lines: planned grid points lie exactly on a
    bisector.  The tie is counted, and the run's logs are simulator.choi's with the same start positions and noise."""
    from mfgp_coverage_b200 import simulator as sim
    from mfgp_coverage_b200._batched import BatchedRuns
    xy = synth.grid(21)
    truth_arr = np.column_stack((xy, synth.truth_function(xy)))
    A, T = 4, 10
    sym = np.array([[0.25, 0.25], [0.75, 0.25], [0.25, 0.75], [0.75, 0.75]])
    starts = np.stack([sym, synth.agents(A, 5)])
    br = BatchedRuns("choi", truth_arr, None, synth.SF_HYP, A, T, starts,
                     noise_rngs=[np.random.default_rng(1), np.random.default_rng(2)]).run()
    assert br.cluster_ties[0].sum() > 0
    logs = br.logs([0, 1])
    assert 0 in br.tie_reruns
    ref = sim.choi("choi", 0, T, A, sym.copy(), truth_arr, 0.1, None, synth.SF_HYP, False, None, True,
                   noise_rng=np.random.default_rng(1))
    for got, want in zip(_rows_to_arrays(logs[0], A), _rows_to_arrays(ref, A)):
        assert np.array_equal(got, want)


@gpu
def test_runner_batched_mode_runs_choi(golden_dir, tmp_path):
    """runner.run(batched=True) on a Choi experiment: same CSV columns and shapes as the sequential mode; with the same seed the
    start positions and iteration 0 (before any sample noise, unseeded as in the reference, can matter) coincide."""
    from mfgp_coverage_b200 import runner
    from tests.test_gpu_runner import _write_inputs
    name, null = _write_inputs(golden_dir, str(tmp_path))
    kw = dict(name=name, agents=8, iterations=6, simulations=4, sigma_n=0.1, seed=9, null_prior_path=null, n_processors=1)
    try:
        runner.run(prefix=os.path.join(str(tmp_path), "seq"), algorithms=["choi_hmf"], batched=False, **kw)
        runner.run(prefix=os.path.join(str(tmp_path), "bat"), algorithms=["choi_hmf"], batched=True, **kw)
    finally:
        runner.BATCHED = False
        os.environ["MFGP_BATCHED"] = "0"
    for kind in ("loss", "agent"):
        a = pd.read_csv(os.path.join(str(tmp_path), f"seq_choi_hmf_{kind}.csv"), index_col=0)
        b = pd.read_csv(os.path.join(str(tmp_path), f"bat_choi_hmf_{kind}.csv"), index_col=0)
        assert list(a.columns) == list(b.columns) and a.shape == b.shape
        a, b = a[a.Iteration == 0], b[b.Iteration == 0]
        num = [c for c in a.columns if c != "Fidelity"]
        assert np.allclose(a[num].values.astype(float), b[num].values.astype(float), rtol=1e-9, atol=1e-12), kind
