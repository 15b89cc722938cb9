"""Batched replicate runs: many independent simulations of ONE experiment stepped together on the device.

The reference runs its replicate sweeps (100+ simulations of the same algorithm on the same data, runner.py:100, :131-147)
one simulation per worker process; every simulation is a host loop that calls the GP and the coverage functions once per
iteration (simulator.py periodic :618-785, todescato :788-954, lloyd :508-616).  On small grids that loop is launch-bound on
a GPU.  `BatchedRuns` keeps the loop state of all runs on the device and advances every run by one iteration with three
kernel launches (`mfgp_batch_step`, csrc/batched.cu); the host draws the runs' random numbers up front, in the order the
reference consumes them, and reads the log buffers back once at the end.  Results per run: the reference's three lists of
log-row dicts.

Parity: samples, decisions, centroids, arg-max points and variances follow the single-run path (appended samples border the
factor instead of a refit: same results to ~1e-13).  The LOSS of an iteration in which agents sit on grid points can involve
grid points lying exactly on a bisector; the reference resolves those through Qhull's vertex rounding.  The stepper counts
them per (run, iteration); `exact_tie_loss=True` re-evaluates exactly those losses with Qhull cells on the single-run path.

Choi (simulator.py:957-1161) returns to the host once per period.  Period p lasts 8 * 2**p iterations whatever the run, so
all runs share the period boundaries; the loop does not stop inside a period, so `iterations` = 10 logs 24 iterations
(choi_schedule).  At a period start every run plans on the device (greedy max-variance picks on its own factor, the picks
held as temporary rows past Ncur), its picks are clustered by the cells of its centroids, all runs' clusters are ordered
by one tour-planner launch, and the period's iterations run through the stepper with the Choi decision (explore while the
agent's tour has points left).  The buffers grow between pick rounds when a run's picks reach the capacity.  A pick that
lies within TIE_TOL/10 of a bisector of the centroid cells (which agent visits it is then decided by Qhull's vertex
rounding in the single-run path) makes the run's result depend on Qhull: such runs are re-run on the single-run path with
the same start positions and noise draws (`tie_reruns`).
"""
import ctypes

import numpy as np
import torch

from . import _coverage as cv
from . import _native as nat
from .gaussian_process import evaluate_hyp, prior_variance

ALGOS = {"lloyd": 0, "periodic": 1, "todescato": 2, "choi": 3}
LOG_COLS = ("X", "Y", "XMax", "YMax", "VarMax", "Var0", "XCentroid", "YCentroid", "ProbExplore", "Explore", "Distance")
CHOI_ROUNDS = 16          # planner pick rounds launched between two reads of the runs' planning state
CHOI_GROW = 32            # training rows added per run when a planner reaches the capacity
BUFFER_NAMES = ("xy", "f", "ux", "uy", "Xt", "y", "W", "z", "TxL", "TyL", "TxH", "TyH", "mu", "var", "pos", "prev", "cen",
                "pos_idx", "prob", "explore", "Ncur", "knew", "status", "noise_used", "nsamples", "ties", "noise", "unif",
                "log_loss", "log_agent", "log_sample")
CHOI_BUFFER_NAMES = ("q", "picks", "nplan", "plan_state", "pmask", "ccount", "cties", "tour_off", "tour_cur", "tour")


def choi_schedule(iterations):
    """Period index of every iteration a Choi run logs: period p lasts 8 * 2**p iterations (choi_double,
    simulator.py:481-489), and `while iteration < iterations` is only checked between periods (simulator.choi)."""
    period, p = [], 0
    while len(period) < iterations:
        period.extend([p] * (8 * 2 ** p))
        p += 1
    return np.array(period, dtype=np.int64)


class _NoiseRow:
    """Stands in for a numpy Generator: returns the pre-drawn N(0, sigma_n) draws of one run in order (loc 0 and the scale
    are already applied)."""

    def __init__(self, row):
        self.row, self.k = row, 0

    def normal(self, loc=0, scale=1):
        v = self.row[self.k]
        self.k += 1
        return v


class BatchedRuns:
    def __init__(self, algo, truth_arr, prior_arr, hyp, agents, iterations, positions0, sigma_n=0.1, uniforms=None, noise=None,
                 noise_rngs=None, raw_means=False, device=None, cap=None):
        """algo: "lloyd" | "periodic" | "todescato" | "choi".  positions0[R, A, 2]: start positions of the R runs.
        uniforms[R, iterations, A]: todescato's Bernoulli draws (random.random(), simulator.py:943), in consumption order.
        noise[R, iterations * A]: the N(0, sigma_n) sample noise in consumption order -- or `noise_rngs`, one numpy Generator
        per run, from which it is drawn here (the reference draws one normal per sample, :707).  Choi logs
        len(choi_schedule(iterations)) iterations and needs that many times A draws.  cap (Choi): initial training rows per
        run; the buffers grow when the planner needs more."""
        from . import simulator as sim
        from ._engine import TensorAxes, detect_tensor_grid
        nat.require_cuda()
        cap_arg = cap
        self.dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.algo = algo
        self.code = ALGOS[algo]
        truth_arr = np.ascontiguousarray(truth_arr, dtype=np.float64)
        self.truth_arr = truth_arr
        xy = np.ascontiguousarray(truth_arr[:, :2])
        tg = detect_tensor_grid(xy)
        if tg is None:
            raise ValueError("BatchedRuns needs a tensor-product grid (every grid of the reference: distribution.py:337-339)")
        ux, uy = tg
        positions0 = np.ascontiguousarray(positions0, dtype=np.float64)
        R, A = positions0.shape[0], positions0.shape[1]
        if A != agents or A > 16:
            raise ValueError("positions0 must be [runs, agents, 2] with at most 16 agents")
        G, nx, ny, T = xy.shape[0], len(ux), len(uy), int(iterations)
        self.iterations, self.positions0 = T, positions0.copy()
        if self.code == 3:
            self.period = choi_schedule(T)
            T = len(self.period)
        else:
            self.period = np.zeros(T, dtype=np.int64)
        self.R, self.A, self.G, self.T = R, A, G, T
        f64 = dict(dtype=torch.float64, device=self.dev)
        i32 = dict(dtype=torch.int32, device=self.dev)
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(self.dev)
        self.xy, self.f, self.ux, self.uy = t(xy), t(truth_arr[:, 2]), t(ux), t(uy)
        self.bbox = np.array([xy[:, 0].min(), xy[:, 0].max(), xy[:, 1].min(), xy[:, 1].max()])
        # ---- the shared initial model (prior only), fitted and evaluated once by the single-run engine
        self.fidelity = "NA"
        self.prior_arr, self.hyp, self.sigma_n = prior_arr, hyp, sigma_n
        NL = N0 = 0
        cap = 8
        self.params = None
        prob0 = 0.0
        if self.code != 0:
            hyp = np.asarray(hyp.values.tolist()[0] if hasattr(hyp, "values") else hyp, dtype=np.float64).reshape(-1)
            self.fidelity = sim._fidelity_of(hyp)
            model = sim.init_SFGP(hyp, prior_arr) if self.fidelity == "S" else sim.init_MFGP(hyp, prior_arr)
            model.raw_means = raw_means
            if self.fidelity == "S":
                model.updt_info(model.X, model.y)
                X0, y0 = np.asarray(model.X, dtype=np.float64).reshape(-1, 2), np.asarray(model.y, dtype=np.float64).reshape(-1)
            else:
                model.updt_info(model.X_L, model.y_L, model.X_H, model.y_H)
                X0, y0 = np.asarray(model.X_L, dtype=np.float64).reshape(-1, 2), np.asarray(model.y_L, dtype=np.float64).reshape(-1)
                NL = X0.shape[0]
            self.params = evaluate_hyp(hyp, raw_means)
            self.pstruct = model.engine.pstruct
            N0 = X0.shape[0]
            grid = cv.CoverageGrid(xy, truth_arr[:, 2], device=self.dev)
            mu0, var0 = model.predict_device(grid.xy, grid=grid)
            eng = model.engine
            eng.ensure_factor(need_inverse=True)
            eng.check_factor(force=True)
            cap = -(-(N0 + T * A) // 8) * 8
            if self.code == 3:
                cap = -(-max(N0 + CHOI_GROW if cap_arg is None else int(cap_arg), N0 + 1) // 8) * 8
            k0 = prior_variance(self.params)
            self.k0 = k0
            if self.code == 2:
                prob0 = float(np.sqrt(float(var0.max().item()) / (k0 * A)))      # simulator.py:855-857
        else:
            self.pstruct = nat.MfgpParams(0.0, 1.0, 1.0, 1.0, 1.0, 0.0, 0.0, 0.0, 0.0, 1e-8, 0, 0)
        self.cap, self.NL, self.N0 = cap, NL, N0
        self.max_samples = max(T * A, 1)
        z = lambda *shape, **k: torch.zeros(shape, **(k or f64))
        self.Xt, self.y, self.W, self.z = z(R, cap, 2), z(R, cap), torch.empty((R, cap, cap), **f64), z(R, cap)
        self.TxL, self.TyL, self.TxH, self.TyH = z(R, cap, nx), z(R, cap, ny), z(R, cap, nx), z(R, cap, ny)
        self.mu, self.var = z(R, G), z(R, G)
        if self.code != 0:
            if N0:
                self.Xt[:, :N0] = t(X0)
                self.y[:, :N0] = t(y0)
                self.W[:, :N0, :N0] = torch.tril(eng.W[:N0, :N0])
                self.z[:, :N0] = eng.z[:N0]
                p = self.params
                X0d = t(X0)
                for tab, u, col, l in ((self.TxH, self.ux, 0, p["l_H"]), (self.TyH, self.uy, 1, p["l_H"]),
                                       (self.TxL, self.ux, 0, p["l_L"]), (self.TyL, self.uy, 1, p["l_L"])):
                    d = u[None, :] / l - (X0d[:, col] / l)[:, None]          # the division first, as gaussian_process.py:77-78
                    tab[:, :N0] = torch.exp(-0.5 * (d * d))
            self.mu[:] = mu0
            self.var[:] = var0
        pos = t(positions0.reshape(R, A * 2))
        self.pos, self.prev, self.cen = pos.clone(), pos.clone(), pos.clone()
        self.pos_idx = torch.full((R, A), -1, dtype=torch.int64, device=self.dev)
        self.prob = torch.full((R, A), prob0, **f64)
        self.explore, self.Ncur = z(R, A, **i32), torch.full((R,), N0, **i32)
        self.knew, self.status, self.noise_used, self.nsamples = z(R, **i32), z(R, **i32), z(R, **i32), z(R, **i32)
        self.ties = z(R, T, **i32)
        if noise is None:
            gens = noise_rngs if noise_rngs is not None else [np.random.default_rng() for _ in range(R)]
            noise = np.stack([g.normal(loc=0, scale=sigma_n, size=self.max_samples) for g in gens]) if self.code else np.zeros((R, 1))
        self.noise = t(np.asarray(noise, dtype=np.float64).reshape(R, -1))
        if self.noise.shape[1] < self.max_samples and self.code:
            raise ValueError("noise must hold iterations * agents draws per run")
        self.max_samples = int(self.noise.shape[1]) if self.code else 1
        if self.code == 2:
            if uniforms is None:
                raise ValueError("todescato needs the runs' uniform draws (random.random(), simulator.py:943)")
            self.unif = t(np.asarray(uniforms, dtype=np.float64).reshape(R, T, A))
        else:
            self.unif = z(1)
        self.log_loss, self.log_agent = z(R, T), z(R, T, A, len(LOG_COLS))
        self.log_sample = z(R, self.max_samples, 5)
        self.noise_host = np.asarray(noise, dtype=np.float64).reshape(R, -1)
        b = nat.MfgpBatch()
        b.runs, b.G, b.nx, b.ny, b.A, b.NL, b.cap, b.algo, b.iterations, b.max_samples = R, G, nx, ny, A, NL, cap, self.code, T, \
            self.max_samples
        b.xmin, b.xmax, b.ymin, b.ymax = (float(v) for v in self.bbox)
        b.eps, b.tie_tol, b.amax_rel = cv.EPS, cv.TIE_TOL, cv.AMAX_REL
        self._b = b
        self.graph = None
        self.tie_reruns = []
        if self.code == 3:
            self.q = z(R, G)
            self.picks = torch.zeros((R, cap), dtype=torch.int64, device=self.dev)
            self.pmask = z(R, cap, **i32)
            self.nplan, self.plan_state, self.cties = z(R, **i32), z(R, **i32), z(R, **i32)
            self.ccount, self.tour_off, self.tour_cur = z(R, A, **i32), z(R * A + 1, **i32), z(R * A, **i32)
            self.tour = torch.zeros(1, dtype=torch.int64, device=self.dev)
            self.cluster_ties = np.zeros((R, int(self.period[-1]) + 1 if T else 0), dtype=np.int64)
            self.phase_ms = {"plan": 0.0, "cluster_tours": 0.0, "step": 0.0}
        self._bind()

    def _bind(self):
        b = self._b
        b.cap = self.cap
        for name in BUFFER_NAMES + (CHOI_BUFFER_NAMES if self.code == 3 else ()):
            setattr(b, name, getattr(self, name).data_ptr())

    def _grow(self, cap):
        """Choi: room for `cap` training rows per run (the rows in use and the factor are copied over)."""
        cap = -(-int(cap) // 8) * 8
        if 2 * self.A * cap * 8 > 200 * 1024:
            raise ValueError(f"a batched Choi run needs {cap} training rows, more than the stepper's sample append can stage with "
                             f"{self.A} agents ({200 * 1024 // (16 * self.A)} rows); run this experiment with simulator.choi")
        old = self.cap
        for name in ("Xt", "y", "z", "TxL", "TyL", "TxH", "TyH", "picks", "pmask"):
            t = getattr(self, name)
            n = torch.zeros((t.shape[0], cap) + tuple(t.shape[2:]), dtype=t.dtype, device=t.device)
            n[:, :old] = t
            setattr(self, name, n)
        W = torch.zeros((self.R, cap, cap), dtype=torch.float64, device=self.dev)
        W[:, :old, :old] = self.W
        self.W = W
        self.cap = cap
        self._bind()

    def step(self, it):
        nat.check(nat.lib().mfgp_batch_step(ctypes.byref(self._b), ctypes.byref(self.pstruct), int(it), nat.stream_ptr()),
                  "mfgp_batch_step")

    def plan(self, threshold):
        """Choi, every run: greedy picks on the run's own factor until its max variance is <= threshold
        (compute_sample_points, simulator.py:326-374).  Picks: picks[r, :nplan[r]]; the runs' models are unchanged."""
        lib, sp, b = nat.lib(), nat.stream_ptr(), ctypes.byref(self._b)
        nat.check(lib.mfgp_batch_choi_begin(b, ctypes.byref(self.pstruct), sp), "mfgp_batch_choi_begin")
        while True:
            nat.check(lib.mfgp_batch_choi_plan(b, ctypes.byref(self.pstruct), ctypes.c_double(threshold), CHOI_ROUNDS, sp),
                      "mfgp_batch_choi_plan")
            st = self.plan_state.cpu().numpy()
            if (st == 2).any():                 # a planner reached the capacity: grow, resume
                self._grow(self.cap + CHOI_GROW)
                b = ctypes.byref(self._b)
                self.plan_state.masked_fill_(self.plan_state == 2, 0)
            elif not (st == 0).any():
                return

    def cluster_and_tours(self, period, length):
        """Choi: clusters of the planned picks by the cells of each run's centroids (compute_sample_clusters,
        simulator.py:377-412) and their tours (compute_sample_tsp, :415-454) for a period of `length` iterations."""
        lib, sp = nat.lib(), nat.stream_ptr()
        nat.check(lib.mfgp_batch_choi_cluster(ctypes.byref(self._b), sp), "mfgp_batch_choi_cluster")
        cnt = self.ccount.cpu().numpy().reshape(-1).astype(np.int64)
        self.cluster_ties[:, period] = self.cties.cpu().numpy()
        # the period's samples go to rows Ncur, Ncur + 1, ...: the pending explorers' (decided in the previous period) and the
        # tour points visited in this one
        need = int((self.Ncur.cpu().numpy() + self.A + np.minimum(cnt.reshape(self.R, self.A), length).sum(axis=1)).max())
        if need > self.cap:
            self._grow(need)
        off = np.zeros(self.R * self.A + 1, dtype=np.int32)
        np.cumsum(cnt, out=off[1:])
        n_total, n_max = int(off[-1]), int(cnt.max())
        self.tour_off.copy_(torch.from_numpy(off))
        pts = torch.empty((max(n_total, 1), 2), dtype=torch.float64, device=self.dev)
        gidx = torch.empty(max(n_total, 1), dtype=torch.int64, device=self.dev)
        order = torch.empty(max(n_total, 1), dtype=torch.int32, device=self.dev)
        self.tour = torch.empty(max(n_total, 1), dtype=torch.int64, device=self.dev)
        self._b.tour = self.tour.data_ptr()
        work, wbytes = None, 0
        if n_max > 4096:
            wbytes = int(lib.choi_tsp_workspace_bytes(n_total))
            work = torch.empty(wbytes // 8 + 8, dtype=torch.float64, device=self.dev)
        nat.check(lib.mfgp_batch_choi_tours(ctypes.byref(self._b), n_total, n_max, nat.ptr(pts), nat.ptr(gidx), nat.ptr(order),
                                            nat.ptr(work), wbytes, sp), "mfgp_batch_choi_tours")

    def _run_choi(self):
        ev = lambda: torch.cuda.Event(enable_timing=True)        # noqa: E731
        marks = []
        threshold = self.k0                                     # max_var_0 (simulator.choi)
        it = 0
        for period in range(int(self.period[-1]) + 1 if self.T else 0):
            length = 8 * 2 ** period
            threshold = 0.82 * threshold                        # choi_threshold (:470-478)
            e = [ev() for _ in range(4)]
            e[0].record()
            self.plan(threshold)
            e[1].record()
            self.cluster_and_tours(period, length)
            e[2].record()
            for _ in range(length):
                self.step(it)
                it += 1
            e[3].record()
            marks.append(e)
        torch.cuda.current_stream(self.dev).synchronize()
        for e in marks:
            for key, a, b in (("plan", 0, 1), ("cluster_tours", 1, 2), ("step", 2, 3)):
                self.phase_ms[key] += e[a].elapsed_time(e[b])

    def capture(self):
        """Record the whole run -- every iteration's three launches -- into ONE CUDA graph.  Nothing in the loop depends on
        the host (sample counts, explore decisions and the growing training-set sizes live in device memory), so the graph
        is valid for any state the buffers hold when it is replayed."""
        if self.code == 3:
            raise ValueError("Choi runs return to the host once per period: they cannot be captured in one CUDA graph")
        graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(device=self.dev)
        side.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.graph(graph, stream=side):
            for it in range(self.T):
                self.step(it)
        self.graph = graph
        return self

    def run(self, use_graph=False):
        """All iterations, no host round trip in between; returns when the device is done.  `use_graph`: replay the run
        from one CUDA graph (captured on first use) instead of 3 * iterations launches."""
        if use_graph:
            if self.graph is None:
                self.capture()
            self.graph.replay()
        elif self.code == 3:
            self._run_choi()
        else:
            for it in range(self.T):
                self.step(it)
        torch.cuda.current_stream(self.dev).synchronize()
        st = self.status.cpu().numpy()
        bad = np.nonzero(st)[0]
        if bad.size:
            r, code = int(bad[0]), int(st[bad[0]])
            if code > 0:
                raise np.linalg.LinAlgError(f"Matrix is not positive definite (pivot {code - 1}) in run {r}")
            if code == -4:
                raise ValueError("zero-size array to reduction operation maximum which has no identity")      # np.amax([])
            raise RuntimeError(f"mfgp_batch_step: run {r} stopped with status {code}")
        return self

    def logs(self, sim_nums=None, exact_tie_loss=False, rerun_ties=True):
        """The reference's (loss_log, agent_log, sample_log) row lists, one triple per run.  Choi: the runs whose clustering
        met a hard bisector tie are re-run on the single-run path (simulator.choi) with the same start positions and noise
        draws unless `rerun_ties` is False; their indices are in `tie_reruns`."""
        R, T, A = self.R, self.T, self.A
        per = self.period.tolist()
        loss = self.log_loss.cpu().numpy().copy()
        agent = self.log_agent.cpu().numpy()
        samples = self.log_sample.cpu().numpy()
        ns = self.nsamples.cpu().numpy()
        ties = self.ties.cpu().numpy()
        if exact_tie_loss and ties.any():
            from . import simulator as sim
            for r, it in zip(*np.nonzero(ties)):
                vor = cv.BoundedVoronoi(agent[r, it, :, :2], self.bbox)
                loss[r, it] = sim.compute_loss(vor, self.truth_arr)
        self.tie_iterations = ties > 0
        sim_nums = list(range(R)) if sim_nums is None else list(sim_nums)
        fid = self.fidelity
        out = []
        for r in range(R):
            s = sim_nums[r]
            loss_log = [{"SimNum": s, "Iteration": it, "Period": per[it], "Fidelity": fid, "Loss": loss[r, it]} for it in range(T)]
            rows = agent[r].tolist()
            var0 = 0 if self.code == 0 else None
            agent_log = [{"SimNum": s, "Iteration": it, "Period": per[it], "Fidelity": fid, "Agent": i,
                          "X": v[0], "Y": v[1], "XMax": v[2], "YMax": v[3], "VarMax": v[4], "Var0": v[5] if var0 is None else 0,
                          "XCentroid": v[6], "YCentroid": v[7], "ProbExplore": v[8], "Explore": v[9], "Distance": v[10]}
                         for it in range(T) for i, v in enumerate(rows[it])]
            if self.code == 0:
                sample_log = [{"SimNum": s, "Iteration": it, "Period": 0, "Fidelity": fid, "Agent": "NA", "X": "NA", "Y": "NA",
                               "Sample": "NA"} for it in range(T)]
            else:
                sample_log = [{"SimNum": s, "Iteration": int(v[0]), "Period": per[int(v[0])], "Fidelity": fid, "Agent": v[1],
                               "X": v[2], "Y": v[3], "Sample": v[4]} for v in samples[r, :ns[r]].tolist()]
            out.append((loss_log, agent_log, sample_log))
        self._rerun_pos = {}
        if self.code == 3 and rerun_ties:
            from . import simulator as sim
            self.tie_reruns = [int(r) for r in np.nonzero(self.cluster_ties.sum(axis=1))[0]]
            for r in self.tie_reruns:
                pos = self.positions0[r].copy()
                out[r] = sim.choi(f"choi run {sim_nums[r]}", sim_nums[r], self.iterations, A, pos, self.truth_arr, self.sigma_n,
                                  self.prior_arr, self.hyp, False, None, True, noise_rng=_NoiseRow(self.noise_host[r]))
                self._rerun_pos[r] = pos
        return out

    def final_positions(self):
        pos = self.pos.cpu().numpy().reshape(self.R, self.A, 2)
        for r, p in getattr(self, "_rerun_pos", {}).items():
            pos[r] = p
        return pos
