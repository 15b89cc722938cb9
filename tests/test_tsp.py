"""The deterministic Choi tour planner that replaces mlrose's genetic algorithm (reference simulator.py:415-454): the CPU
statement oracle/tsp.py (properties + optimality on small clusters) and, on the GPU, bit-identical tours from
choi_tsp_tours (csrc/tsp.cu)."""
import itertools

import numpy as np
import pytest

from oracle import tsp as otsp
from tests import synth


def _clusters(rng, sizes, on_grid=False):
    out = []
    for n in sizes:
        if on_grid:      # sample points of the Choi planner ARE grid points: many exactly equal distances (tie rules matter)
            g = synth.grid(17)
            out.append(g[rng.choice(g.shape[0], n, replace=False)].copy() if n else np.empty((0, 2)))
        else:
            out.append(rng.random((n, 2)))
    return out


def test_tour_is_a_permutation_and_2opt_never_lengthens():
    rng = np.random.default_rng(0)
    for n in (1, 2, 3, 4, 5, 9, 30, 61):
        pts = rng.random((n, 2))
        nn = otsp.nearest_neighbour(pts)
        tour = otsp.plan_tour(pts)
        assert sorted(tour) == list(range(n)) and tour[0] == 0 and nn[0] == 0
        assert otsp.tour_length(pts, tour) <= otsp.tour_length(pts, nn) + 1e-15
        # 2-opt local optimality: no reversal improves by more than the tolerance
        t2, moves = otsp.two_opt(pts, tour)
        assert moves == 0 and t2 == tour
    assert otsp.plan_tour([]) == []


def test_small_clusters_reach_the_optimal_closed_tour():
    """n <= 7: brute force over all tours.  2-opt is a local search, so allow the known worst case (a few %) but demand
    the optimum on the convex cases where 2-opt is exact (points on a circle, a square)."""
    rng = np.random.default_rng(1)
    worst = 1.0
    for _ in range(30):
        n = int(rng.integers(4, 8))
        pts = rng.random((n, 2))
        best = min(otsp.tour_length(pts, (0,) + p) for p in itertools.permutations(range(1, n)))
        worst = max(worst, otsp.tour_length(pts, otsp.plan_tour(pts)) / best)
    assert worst <= 1.10
    ang = np.sort(rng.random(12)) * 2 * np.pi
    circle = np.column_stack((np.cos(ang), np.sin(ang)))[rng.permutation(12)]
    tour = otsp.plan_tour(circle)
    a = np.arctan2(circle[tour, 1], circle[tour, 0])
    steps = np.diff(np.unwrap(np.concatenate((a, a[:1]))))
    assert np.all(steps > 0) or np.all(steps < 0)                 # convex position: the optimal tour is the hull order
    square = np.array([[0.0, 0.0], [1.0, 1.0], [1.0, 0.0], [0.0, 1.0]])
    assert abs(otsp.tour_length(square, otsp.plan_tour(square)) - 4.0) <= 1e-15


@pytest.mark.gpu
@pytest.mark.parametrize("on_grid", [False, True])
def test_device_tours_are_bit_identical_to_the_cpu_statement(on_grid):
    from mfgp_coverage_b200 import simulator as sim
    rng = np.random.default_rng(3)
    clusters = _clusters(rng, (0, 1, 2, 3, 4, 5, 8, 33, 0, 70, 120), on_grid=on_grid)
    orders = sim.plan_tours(clusters)
    for c, o in zip(clusters, orders):
        assert list(o) == otsp.plan_tour([tuple(p) for p in c])
    tours = sim.compute_sample_tsp(clusters)
    for c, t, o in zip(clusters, tours, orders):
        assert t.shape == c.shape and np.array_equal(t, c[o] if len(o) else np.empty((0, 2)))


@pytest.mark.gpu
def test_device_tour_of_a_large_cluster_is_2opt_optimal():
    """n = 1500 (c3-scale Choi periods; the literal oracle is O(n^3) there): the device tour must be a permutation that
    starts at point 0 and admits no improving segment reversal (checked with a vectorised delta matrix)."""
    from mfgp_coverage_b200 import simulator as sim
    pts = np.random.default_rng(4).random((1500, 2))
    (o,) = sim.plan_tours([pts])
    assert sorted(o.tolist()) == list(range(1500)) and o[0] == 0
    t = pts[o]
    n = len(o)
    nxt = np.roll(t, -1, axis=0)
    e = np.sqrt(((t - nxt) ** 2).sum(axis=1))
    i = np.arange(1, n - 1)[:, None]
    j = np.arange(2, n)[None, :]
    d_ac = np.sqrt(((t[i - 1] - t[j]) ** 2).sum(axis=2))
    d_bd = np.sqrt(((t[i] - nxt[j]) ** 2).sum(axis=2))
    delta = (d_ac + d_bd) - (e[i - 1] + e[j])
    delta[j <= i] = 0.0
    assert delta.min() >= -1e-12
    nn = pts[otsp.nearest_neighbour(pts[:300])]       # and it is shorter than plain nearest neighbour (sanity, on a subset)
    (o3,) = sim.plan_tours([pts[:300]])
    assert otsp.tour_length(pts[:300], list(o3)) < otsp.tour_length(pts[:300], otsp.nearest_neighbour(pts[:300]))
