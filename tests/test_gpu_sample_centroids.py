"""GPU: per-cell centroids of joint posterior draws reduced in Chebyshev coefficient space (cov_cell_moments,
cov_cell_moments_centroids, CoverageGrid.sample_centroids, simulator.compute_centroids_samples / thompson).  Partials and
centroids agree with the per-draw route built from existing kernels (mfgp_grid_sample_eval, then cov_assign_reduce_grid with
w = F[:, s]) and with the oracle at equal normals; HybridVoronoi ties rerun on Qhull's polygons; empty cells give NaN;
repeats give the same bits; the C-ABI rejects bad arguments and writes nothing outside its outputs; seeded Thompson runs
reproduce the oracle loop."""
import ctypes
import os

import numpy as np
import pandas as pd
import pytest

from oracle import coverage as ocov
from oracle import gp as ogp
from oracle import gp_sample_grid as osg
from oracle import sample_centroids as osc
from tests import synth

pytestmark = pytest.mark.gpu
CANARY = -7.25e300


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()


def _model(kind, xy, N):
    from mfgp_coverage_b200.gaussian_process import MFGP, SFGP
    multi = kind != "SF"
    hyp = synth.MF_HYP if multi else synth.SF_HYP
    if N:
        X_L, y_L, X_H, y_H = synth.training_set(xy, synth.truth_function(xy), N, multi=multi)
    else:
        X_L = X_H = np.empty((0, 2))
        y_L = y_H = np.empty((0, 1))
    if multi:
        m = MFGP(X_L, y_L, X_H, y_H, 1, 1)
        m.hyp = hyp
        m.updt_info(X_L, y_L, X_H, y_H)
    else:
        m = SFGP(X_H, y_H, 1)
        m.hyp = hyp
        m.updt_info(X_H, y_H)
    return m, ogp.GPParams.from_hyp(hyp), (X_L, y_L, X_H, y_H)


def _per_draw(g, vor, F):
    """cent[S, A, 4] and |F|-weighted sums [S, A] of the per-draw route: one cov_assign_reduce_grid pass per draw."""
    import torch
    from mfgp_coverage_b200._coverage import CoverageGrid
    cents, scale = [], []
    for s in range(F.shape[1]):
        w = F[:, s].contiguous()
        cents.append(CoverageGrid.results_to_host(g.assign_reduce(lloyd_vor=vor, w=w))["cent"].copy())
        scale.append(CoverageGrid.results_to_host(g.assign_reduce(lloyd_vor=vor, w=torch.abs(w)))["cent"][:, 0].copy())
    return np.stack(cents), np.stack(scale)


def _check_against_per_draw(m, g, vor, S, seed=1):
    import torch
    from mfgp_coverage_b200 import _coverage as cv
    d = m.grid_sample_dim(g)
    E = torch.from_numpy(np.random.default_rng(seed).standard_normal((d, S))).cuda()
    cent, cen = g.sample_centroids(m, vor, E)
    F = m.sample_posterior_grid_device(g, E)
    ref, scale = _per_draw(g, vor, F)
    cent = cent.cpu().numpy()
    xy = g.xy.cpu().numpy()
    cmax = max(1.0, float(np.abs(xy).max()))
    assert np.array_equal(cent[..., 3], ref[..., 3])
    assert np.all(np.abs(cent[..., :3] - ref[..., :3]) <= 1e-12 * cmax * scale[..., None] + 1e-300)
    bb = ocov.bounding_box_of(xy)
    ref_c = np.stack([cv.centroids_from_partials(ref[s], vor.areas(), *bb) for s in range(S)])
    got = cen.cpu().numpy()
    assert np.array_equal(np.isnan(got), np.isnan(ref_c))
    assert np.nanmax(np.abs(got - ref_c)) <= 1e-9
    return cent, got, F


CASES = [("MF", 120, 1, 1), ("SF", 80, 4, 7), ("MF", 200, 64, 64), ("MF", 0, 256, 7), ("SF", 0, 64, 1), ("MF", 60, 4, 64),
         ("SF", 150, 256, 64)]


@pytest.mark.parametrize("kind,N,A,S", CASES)
def test_matches_the_per_draw_route(kind, N, A, S):
    from mfgp_coverage_b200._coverage import BoundedVoronoi, CoverageGrid
    xy = synth.grid(51)
    m, _, _ = _model(kind, xy, N)
    g = CoverageGrid(xy)
    vor = BoundedVoronoi(synth.agents(A, 3), ocov.bounding_box_of(xy))
    assert len(vor) == A
    _check_against_per_draw(m, g, vor, S)


def test_matches_the_per_draw_route_at_c4():
    from mfgp_coverage_b200._coverage import CoverageGrid, HybridVoronoi
    xy = synth.grid(1024)
    m, _, _ = _model("MF", xy, 4096)
    g = CoverageGrid(xy)
    vor = HybridVoronoi(synth.agents(64, 4), ocov.bounding_box_of(xy))
    _check_against_per_draw(m, g, vor, 64)


@pytest.mark.parametrize("kind,N", [("MF", 60), ("SF", 90), ("MF", 0)])
def test_matches_the_oracle_at_equal_normals(kind, N):
    import torch
    from mfgp_coverage_b200._coverage import BoundedVoronoi, CoverageGrid
    gx = np.linspace(0.0, 1.0, 31)
    xy = synth.grid(31)
    m, p, (X_L, y_L, X_H, y_H) = _model(kind, xy, N)
    g = CoverageGrid(xy)
    seeds = synth.agents(6, 2)
    bb = ocov.bounding_box_of(xy)
    d = m.grid_sample_dim(g)
    E = np.random.default_rng(4).standard_normal((d, 5))
    cent, cen = g.sample_centroids(m, BoundedVoronoi(seeds, bb), torch.from_numpy(E).cuda())
    plan = m.engine._grid_sample_plan(g.axes)
    Q = tuple(plan["Q"][k].cpu().numpy() if k in plan["Q"] else None for k in ("Lx", "Ly", "Hx", "Hy"))
    mean, Amap = osg.pathwise_map(p, gx, gx, X_L, y_L, X_H, y_H, plan["box"], plan["orders"], Q)
    F = mean[:, None] + Amap @ E
    vo = ocov.voronoi_bounded(seeds, bb)
    ref, scale = osc.dense_partials(ocov.membership(vo, xy), xy, F)
    cent = cent.cpu().numpy()
    assert np.array_equal(cent[..., 3], ref[..., 3])
    assert np.all(np.abs(cent[..., :3] - ref[..., :3]) <= 1e-9 * np.maximum(scale, 1.0))
    assert np.max(np.abs(cen.cpu().numpy() - osc.dense_centroids(vo, xy, F))) <= 1e-9


def test_hybrid_partition_reruns_ties_on_qhull_polygons():
    import torch
    from mfgp_coverage_b200._coverage import CoverageGrid, HybridVoronoi
    xy = synth.grid(41)
    m, _, _ = _model("MF", xy, 50)
    g = CoverageGrid(xy)
    seeds = np.array([[0.25, 0.25], [0.75, 0.25], [0.25, 0.75], [0.75, 0.75], [0.5, 0.5]])
    bb = ocov.bounding_box_of(xy)
    vor = HybridVoronoi(seeds, bb)
    E = torch.from_numpy(np.random.default_rng(8).standard_normal((m.grid_sample_dim(g), 3))).cuda()
    cent, cen = g.sample_centroids(m, vor, E)
    assert vor._qhull is not None                                   # the pass met ties: Qhull's polygons decided them
    F = m.sample_posterior_grid_device(g, E).cpu().numpy()
    vo = ocov.voronoi_bounded(seeds, bb)
    member = ocov.membership(vo, xy)
    assert np.any(member.sum(axis=0) != 1)
    ref, scale = osc.dense_partials(member, xy, F)
    cent = cent.cpu().numpy()
    assert np.array_equal(cent[..., 3], ref[..., 3])
    assert np.all(np.abs(cent[..., :3] - ref[..., :3]) <= 1e-12 * scale + 1e-300)
    assert np.max(np.abs(cen.cpu().numpy() - osc.dense_centroids(vo, xy, F))) <= 1e-9


def test_an_empty_cell_gives_nan():
    import torch
    from mfgp_coverage_b200._coverage import BoundedVoronoi, CoverageGrid
    xy = synth.grid(5)                                              # spacing 0.25
    m, _, _ = _model("SF", synth.grid(21), 20)
    g = CoverageGrid(xy)
    seeds = np.array([[0.1, 0.1], [0.11, 0.11], [0.12, 0.12], [0.9, 0.8]])   # cell 1: the strip 0.21 < x + y < 0.23
    bb = ocov.bounding_box_of(xy)
    E = torch.from_numpy(np.random.default_rng(2).standard_normal((m.grid_sample_dim(g), 2))).cuda()
    cent, cen = g.sample_centroids(m, BoundedVoronoi(seeds, bb), E)
    cen = cen.cpu().numpy()
    assert np.all(np.isnan(cen[:, 1])) and np.all(np.isfinite(cen[:, [0, 2, 3]]))
    assert np.all(cent.cpu().numpy()[:, 1] == 0.0)
    F = m.sample_posterior_grid_device(g, E).cpu().numpy()
    ref = osc.dense_centroids(ocov.voronoi_bounded(seeds, bb), xy, F)
    assert np.array_equal(np.isnan(ref), np.isnan(cen))


def test_repeats_give_the_same_bits():
    import torch
    from mfgp_coverage_b200._coverage import CoverageGrid, HybridVoronoi
    xy = synth.grid(200)
    m, _, _ = _model("MF", xy, 300)
    g = CoverageGrid(xy)
    vor = HybridVoronoi(synth.agents(37, 6), ocov.bounding_box_of(xy))
    E = torch.from_numpy(np.random.default_rng(1).standard_normal((m.grid_sample_dim(g), 33))).cuda()
    a = g.sample_centroids(m, vor, E)
    b = g.sample_centroids(m, vor, E)
    for x, y in zip(a, b):
        assert torch.equal(torch.nan_to_num(x, nan=7.0), torch.nan_to_num(y, nan=7.0))


def test_host_form_replays_seeded_draws():
    from mfgp_coverage_b200 import simulator as sim
    xy = synth.grid(41)
    m, _, _ = _model("MF", xy, 70)
    vor = sim.voronoi_bounded(synth.agents(5, 1), ocov.bounding_box_of(xy))
    a = sim.compute_centroids_samples(vor, xy, m, n_samples=4, rng=np.random.default_rng(3))
    b = sim.compute_centroids_samples(vor, xy, m, n_samples=4, rng=np.random.default_rng(3))
    assert a.shape == (4, 5, 2) and np.array_equal(a, b)
    with pytest.raises(ValueError):
        sim.compute_centroids_samples(vor, xy[::-1][:-3].copy(), m)     # not a tensor-product grid


def test_c_abi_rejects_bad_arguments_and_keeps_canaries():
    import torch
    from mfgp_coverage_b200 import _native as nat
    from mfgp_coverage_b200._coverage import BoundedVoronoi, CoverageGrid
    lib = nat.lib()
    xy = synth.grid(33)
    g = CoverageGrid(xy)
    vor = BoundedVoronoi(synth.agents(5, 2), ocov.bounding_box_of(xy))
    P = g.upload(vor)
    A, nx, ny, rx, ry = 5, 33, 33, 10, 12
    kpad = 12
    box = [ctypes.c_double(v) for v in (0.0, 1.0, 0.0, 1.0)]
    wb = int(lib.cov_cell_moments_workspace_bytes(nx, ny, A, rx, ry))
    assert wb > 0 and int(lib.cov_cell_moments_workspace_bytes(nx, ny, 257, rx, ry)) == 0
    n_mom = A * 3 * ry * kpad
    buf = torch.full((n_mom + 8,), CANARY, dtype=torch.float64, device="cuda")
    mom = buf[4:4 + n_mom]
    work = torch.empty(wb // 8 + 4, dtype=torch.float64, device="cuda")
    ties = torch.zeros(2, dtype=torch.int32, device="cuda")
    st = nat.stream_ptr()

    def call(xyp=None, A_=A, rx_=rx, ry_=ry, momp=None, wbytes=wb, tie_tol=1e-9, workp=None, boxv=None):
        return lib.cov_cell_moments(xyp if xyp is not None else nat.ptr(g.xy), nx, ny, nat.ptr(P.seeds), A_, nat.ptr(P.poly),
                                    nat.ptr(P.off), ctypes.c_double(tie_tol), *(boxv or box), rx_, ry_,
                                    momp if momp is not None else nat.ptr(mom), nat.ptr(ties),
                                    workp if workp is not None else nat.ptr(work), wbytes, st)

    bad = [dict(wbytes=wb - 8), dict(A_=0), dict(A_=257), dict(rx_=65), dict(ry_=0), dict(tie_tol=float("nan")),
           dict(xyp=ctypes.c_void_p(g.xy.data_ptr() + 8)), dict(momp=ctypes.c_void_p(mom.data_ptr() + 8)),
           dict(workp=ctypes.c_void_p(work.data_ptr() + 8)), dict(boxv=[ctypes.c_double(v) for v in (1.0, 1.0, 0.0, 1.0)])]
    for kw in bad:
        assert call(**kw) == nat.MFGP_ERR_INVALID, kw
    torch.cuda.synchronize()
    assert torch.all(buf == CANARY)
    assert call() == nat.MFGP_OK
    torch.cuda.synchronize()
    assert torch.all(buf[:4] == CANARY) and torch.all(buf[4 + n_mom:] == CANARY) and torch.all(mom != CANARY)
    # centroid stage
    S = 3
    C = _dev(np.random.default_rng(0).standard_normal((S, ry, kpad)))
    areas = _dev(vor.areas())
    ob = torch.full((S * A * 6 + 16,), CANARY, dtype=torch.float64, device="cuda")
    cent, cen = ob[4:4 + S * A * 4], ob[8 + S * A * 4:8 + S * A * 6]
    assert int(lib.cov_cell_moments_centroids_workspace_bytes(A, rx, ry, S)) == 0

    def ccall(momp=None, A_=A, S_=S, centp=None, cenp=None, Cp=None):
        return lib.cov_cell_moments_centroids(momp if momp is not None else nat.ptr(mom), A_, rx, ry,
                                              Cp if Cp is not None else nat.ptr(C), S_, ctypes.c_double(0.5), nat.ptr(areas),
                                              *box, centp if centp is not None else nat.ptr(cent),
                                              cenp if cenp is not None else nat.ptr(cen), None, 0, st)

    for kw in [dict(A_=0), dict(A_=257), dict(S_=0), dict(momp=ctypes.c_void_p(mom.data_ptr() + 8)),
               dict(Cp=ctypes.c_void_p(C.data_ptr() + 8)), dict(centp=ctypes.c_void_p(cent.data_ptr() + 8)),
               dict(cenp=ctypes.c_void_p(cen.data_ptr() + 8))]:
        assert ccall(**kw) == nat.MFGP_ERR_INVALID, kw
    torch.cuda.synchronize()
    assert torch.all(ob == CANARY)
    assert ccall() == nat.MFGP_OK
    torch.cuda.synchronize()
    assert torch.all(ob[:4] == CANARY) and torch.all(ob[4 + S * A * 4:8 + S * A * 4] == CANARY)
    assert torch.all(ob[8 + S * A * 6:] == CANARY)


def test_sampler_errors_are_raised_unchanged():
    import torch
    from mfgp_coverage_b200._coverage import BoundedVoronoi, CoverageGrid
    xy = synth.grid(21)
    m, _, _ = _model("MF", xy, 30)
    vor = BoundedVoronoi(synth.agents(3, 1), ocov.bounding_box_of(xy))
    pts = np.random.default_rng(0).uniform(0, 1, (300, 2))
    with pytest.raises(ValueError):
        CoverageGrid(pts).sample_centroids(m, vor, torch.zeros((10, 1), dtype=torch.float64, device="cuda"))
    g = CoverageGrid(xy)
    with pytest.raises(ValueError):
        g.sample_centroids(m, vor, torch.zeros((3, 1), dtype=torch.float64, device="cuda"))     # wrong d


def _thompson_inputs(golden_dir, fid):
    inp = np.load(os.path.join(golden_dir, "inputs_australia6.npz"))
    truth = inp["truth"]
    if fid == "hmf":
        hyp, prior = inp["mf_hyp"], inp["prior"]
        cols = ["mu_lo", "s^2_lo", "L_lo", "mu_hi", "s^2_hi", "L_hi", "rho", "noise_lo", "noise_hi"]
    else:
        hyp, prior = inp["sf_hyp"], np.empty((0, 3))
        cols = ["mu_sf", "s^2_sf", "L_sf", "noise_sf"]
    return truth, hyp, prior, cols


def _orders_of(p, box):
    from mfgp_coverage_b200._engine import chebyshev_order
    xlo, xhi, ylo, yhi = box
    o = [chebyshev_order(p.l_H, xlo, xhi, xlo, xhi), chebyshev_order(p.l_H, ylo, yhi, ylo, yhi)]
    if p.multi:
        return (chebyshev_order(p.l_L, xlo, xhi, xlo, xhi), chebyshev_order(p.l_L, ylo, yhi, ylo, yhi), *o)
    return (0, 0, *o)


def _near_midpoint(t, u, tol=1e-9):
    """True when t lies within tol of the midpoint between two neighbouring values of u."""
    s = np.sort(u)
    return bool(np.any(np.abs(t - 0.5 * (s[1:] + s[:-1])) <= tol))


@pytest.mark.parametrize("fid", ["hmf", "nsf"])
def test_seeded_thompson_run_reproduces_the_oracle_loop(golden_dir, fid):
    from mfgp_coverage_b200 import simulator as sim
    truth, hyp, prior, cols = _thompson_inputs(golden_dir, fid)
    A, T = 6, 10
    start = np.random.default_rng(17).uniform(0.0, 1.0, (A, 2))
    bb = ocov.bounding_box_of(truth[:, :2])
    start = bb[[0, 2]] + start * (bb[[1, 3]] - bb[[0, 2]])
    pos = start.copy()
    loss, agent, samples = sim.thompson(f"thompson_{fid}", 0, T, A, pos, pd.DataFrame(truth, columns=["X", "Y", "f_H"]), 0.1,
                                        pd.DataFrame(prior, columns=["X", "Y", "f_prior"]), pd.DataFrame([hyp], columns=cols),
                                        False, None, True, rng=np.random.default_rng(5), noise_rng=np.random.default_rng(9))
    oloss, oagent, osamples = osc.thompson(0, T, A, start.copy(), truth, 0.1, prior, hyp, np.random.default_rng(5),
                                            np.random.default_rng(9), _orders_of)
    ux, uy = osc.tensor_axes(truth[:, :2])
    keys = ("VarMax", "XCentroid", "YCentroid", "Distance")
    for t in range(T):
        rows, orows = agent[t * A:(t + 1) * A], oagent[t * A:(t + 1) * A]
        xy = np.array([[r["X"], r["Y"]] for r in rows])
        oxy = np.array([[r["X"], r["Y"]] for r in orows])
        if not np.array_equal(xy, oxy):
            # a flipped snap: the previous iteration's target of a moved agent lies within 1e-9 of a grid midpoint
            prev = oagent[(t - 1) * A:t * A]
            moved = np.nonzero(np.any(xy != oxy, axis=1))[0]
            assert t > 0 and all(_near_midpoint(prev[i]["XCentroid"], ux) or _near_midpoint(prev[i]["YCentroid"], uy)
                                 for i in moved), (t, moved)
            break
        assert abs(loss[t]["Loss"] - oloss[t]["Loss"]) <= 1e-9 * abs(oloss[t]["Loss"])
        for k in keys:
            a = np.array([r[k] for r in rows], dtype=np.float64)
            b = np.array([r[k] for r in orows], dtype=np.float64)
            assert np.max(np.abs(a - b)) <= 1e-9 * (max(1.0, abs(float(rows[0]["Var0"]))) if k == "VarMax" else 1.0), (t, k)
        assert all(r["ProbExplore"] == 1 and r["Explore"] == 1 for r in rows)
    else:
        assert [(s["Agent"], s["X"], s["Y"]) for s in samples] == [(s["Agent"], s["X"], s["Y"]) for s in osamples]


def test_run_sim_dispatches_thompson(golden_dir):
    import random
    from mfgp_coverage_b200.runner import run_sim
    truth, hyp, prior, cols = _thompson_inputs(golden_dir, "hmf")
    random.seed(3)
    args = ("thompson_hmf", "thompson_hmf", 0, 3, 4, pd.DataFrame(truth, columns=["X", "Y", "f_H"]), 0.1,
            pd.DataFrame(prior, columns=["X", "Y", "f_prior"]), pd.DataFrame([hyp], columns=cols), False, None, True)
    loss, agent, samples = run_sim(args)
    assert len(loss) == 3 and len(agent) == 12 and len(samples) == 8
