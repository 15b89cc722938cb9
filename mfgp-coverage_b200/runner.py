"""runner.py -- drop-in for the reference's batch driver (reference runner.py:33-171).

`run_sim(args)` keeps the reference's 12-tuple and algorithm-name substring dispatch (runner.py:46-59); `run()` keeps
its experiment literals as keyword defaults (runner.py:80-100), the hyper-parameter / prior selection rules
(`"mf" in algo`, `"_n" in algo`, :119-128) and the three CSVs per algorithm `{prefix}_{algo}_{loss,agent,sample}.csv`
written with pandas' default index column (:150-156), so `analysis.py` keeps working on the output.

The reference fans simulations out over a `multiprocessing.Pool` of CPU workers (:131-141).  Here `n_processors`
worker processes are spawned one per GPU slot (worker r uses device r % #GPUs) and the replicate simulations are
sharded over them -- run-sharding, no communication until the host concatenates the logs (:144-147).
"""
import os
import random
import time

import numpy as np
import pandas as pd

line_break = "\n" + "".join(["-" for i in range(100)]) + "\n"
slash_break = "\n" + "".join(["/" for i in range(100)]) + "\n"

eps = 0.1


def run_sim(args):
    """reference runner.py:33-69."""
    from .simulator import choi, lloyd, periodic, todescato
    (out_name, algo, sim_num, iterations, agents, truth, sigma_n, prior, hyp, console, plotter, log) = args
    print(line_break + f"Start Simulation {sim_num} : {algo}" + line_break)
    sim_start = time.time()
    x_positions = [random.random() for i in range(agents)]
    y_positions = [random.random() for i in range(agents)]
    positions = np.column_stack((x_positions, y_positions))
    if "choi" in algo:
        fn = choi
    elif "todescato" in algo:
        fn = todescato
    elif "lloyd" in algo:
        fn = lloyd
    elif "periodic" in algo:
        fn = periodic
    else:
        raise ValueError("Invalid simulation algorithm specified.")
    loss_log_t, agent_log_t, sample_log_t = fn(algo, sim_num, iterations, agents, positions, truth, sigma_n, prior,
                                               hyp, console, plotter, log)
    plotter.save(f"{out_name}.png") if plotter else None
    sim_end = time.time()
    print(line_break + f"End Simulation {sim_num} : {algo}\nTime : {sim_end - sim_start}" + line_break)
    return loss_log_t, agent_log_t, sample_log_t


# MFGP_BATCHED=1 (or runner.BATCHED = True, or run(batched=True)): the replicate simulations of lloyd / periodic / todescato /
# choi experiments are stepped TOGETHER on the device (simulator.run_batched: three kernel launches advance every run by one
# iteration; Choi plans all runs' tours on the device once per period) instead of one host loop per simulation.  The random
# streams are consumed exactly as the sequential loop consumes them: per simulation the 2 A start coordinates, then
# (todescato) one uniform per agent and iteration.
BATCHED = os.environ.get("MFGP_BATCHED", "0") == "1"
BATCH_RUNS = 512          # simulations per device batch (state: ~4 MB per run at 64x64 points, 520 samples)


def _batchable(args):
    algos = {a[1] for a in args}
    return len(args) > 1 and len(algos) == 1 and \
        any(k in next(iter(algos)) for k in ("choi", "todescato", "lloyd", "periodic")) and all(a[10] is None for a in args)


def run_sims_batched(args):
    """run_sim for a list of argument tuples of ONE experiment, in order, on the batched stepper."""
    from .simulator import run_batched
    out = []
    for b0 in range(0, len(args), BATCH_RUNS):
        chunk = args[b0:b0 + BATCH_RUNS]
        (_, algo, _, iterations, agents, truth, sigma_n, prior, hyp, _, _, _) = chunk[0]
        pos, unif = [], []
        for a in chunk:                                   # the draws of run_sim (:41-43) and of todescato (:943), in order
            x_positions = [random.random() for i in range(agents)]
            y_positions = [random.random() for i in range(agents)]
            pos.append(np.column_stack((x_positions, y_positions)))
            if "todescato" in algo and "choi" not in algo:
                unif.append([[random.random() for i in range(agents)] for t in range(iterations)])
        print(line_break + f"Start Simulations {chunk[0][2]}..{chunk[-1][2]} : {algo} (batched)" + line_break)
        sim_start = time.time()
        logs = run_batched(algo, [a[2] for a in chunk], iterations, agents, np.array(pos), truth, sigma_n, prior, hyp,
                           uniforms=np.array(unif) if unif else None)
        print(line_break + f"End Simulations : {algo}\nTime : {time.time() - sim_start}" + line_break)
        out.extend(logs)
    return out


def _worker(rank, world, args, seed, queue, fn=None):
    """One worker process.  Whatever happens it reports exactly once: ("ok", rank, results) or ("error", rank, exception,
    traceback text) -- Pool.map in the reference (runner.py:131-141) re-raises worker exceptions in the parent too."""
    import traceback
    try:
        import torch
        if torch.cuda.is_available():
            torch.cuda.set_device(rank % max(torch.cuda.device_count(), 1))
        if seed is not None:
            random.seed(seed + rank)
        out = {}
        mine = list(range(rank, len(args), world))    # run-sharding: simulation i goes to worker i mod world
        if fn is None and BATCHED and _batchable([args[i] for i in mine]):
            out = dict(zip(mine, run_sims_batched([args[i] for i in mine])))
        else:
            for i in mine:
                out[i] = (fn or run_sim)(args[i])
        queue.put(("ok", rank, out))
    except BaseException as e:                         # noqa: BLE001 -- everything goes home, the parent re-raises
        tb = traceback.format_exc()
        try:
            queue.put(("error", rank, e, tb))
        except Exception:                              # the exception itself does not pickle
            queue.put(("error", rank, RuntimeError(f"{type(e).__name__}: {e}"), tb))


class WorkerError(RuntimeError):
    """A simulation worker died without reporting (killed, segfault, CUDA abort)."""


def _map_sims(args, n_processors, seed=None, fn=None):
    """Pool.map(run_sim, args) of the reference (runner.py:131-141) over `n_processors` spawned workers (one per GPU slot).
    A worker exception is re-raised here; a worker that dies silently raises WorkerError.  `fn`: stand-in for run_sim
    (a picklable top-level function), used by the tests."""
    if n_processors <= 1:
        if seed is not None:
            random.seed(seed)
        if fn is None and BATCHED and _batchable(args):
            return run_sims_batched(args)
        return [(fn or run_sim)(a) for a in args]
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    queue = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, n_processors, args, seed, queue, fn)) for r in range(n_processors)]
    for p in procs:
        p.start()
    merged, failure, reported = {}, None, set()
    import queue as _q
    while len(reported) < len(procs) and failure is None:
        try:
            msg = queue.get(timeout=1.0)
        except _q.Empty:
            # liveness: a child that exited without putting its report (hard crash) must not block the parent forever
            dead = [r for r, p in enumerate(procs) if r not in reported and p.exitcode is not None]
            if dead:
                try:
                    msg = queue.get(timeout=2.0)      # its report may still be in flight through the pipe
                except _q.Empty:
                    failure = WorkerError(f"simulation worker {dead[0]} exited with code {procs[dead[0]].exitcode} "
                                          "without reporting")
                    break
            else:
                continue
        reported.add(msg[1])
        if msg[0] == "ok":
            merged.update(msg[2])
        else:
            failure = msg[2]
            failure.worker_traceback = msg[3]
    if failure is not None:
        for p in procs:
            if p.is_alive():
                p.terminate()
    for p in procs:
        p.join()
    if failure is not None:
        raise failure
    return [merged[i] for i in range(len(args))]


def run(n_processors=4, name="Data/australia9", prefix="Data/australia9.3", agents=16, iterations=120,
        simulations=100, sigma_n=0.1, console=False, log=True, plotter=None, algorithms=None, seed=None,
        null_prior_path="Data/null_prior.csv", batched=None):
    """reference runner.py:72-161.  Keyword defaults are the literals the reference hard-codes.  `batched`: step the
    replicate simulations of an algorithm together on the device (see BATCHED above; default: the environment's setting)."""
    global BATCHED
    if batched is not None:
        BATCHED = bool(batched)
        os.environ["MFGP_BATCHED"] = "1" if BATCHED else "0"      # spawned workers read the environment
    np.random.seed(1234)
    if algorithms is None:
        algorithms = ["todescato_nsf", "choi_nsf", "todescato_hsf", "choi_hsf", "todescato_hmf", "choi_hmf", "lloyd"]
    truth = pd.read_csv(f"{name}_hifi.csv")
    mf_hyp = pd.read_csv(f"{name}_mf_hyp.csv")
    sf_hyp = pd.read_csv(f"{name}_sf_hyp.csv")
    null_prior = pd.read_csv(null_prior_path)
    human_prior = pd.read_csv(f"{name}_prior.csv")
    for algo in algorithms:
        print(slash_break + f"Start Algorithm : {algo}" + slash_break)
        algo_start = time.time()
        out_name = f"{prefix}_{algo}"
        loss_log, agent_log, sample_log = [], [], []
        hyp = mf_hyp if "mf" in algo else sf_hyp
        prior = null_prior if "_n" in algo else human_prior
        args = [(out_name, algo, sim_num, iterations, agents, truth, sigma_n, prior, hyp, console, plotter, log)
                for sim_num in range(simulations)]
        out = _map_sims(args, n_processors, seed)
        for sim_num in range(simulations):
            loss_log.extend(out[sim_num][0])
            agent_log.extend(out[sim_num][1])
            sample_log.extend(out[sim_num][2])
        if log:
            pd.DataFrame(loss_log).to_csv(f"{out_name}_loss.csv")
            pd.DataFrame(agent_log).to_csv(f"{out_name}_agent.csv")
            pd.DataFrame(sample_log).to_csv(f"{out_name}_sample.csv")
        algo_end = time.time()
        print(slash_break + f"End Algorithm : {algo}\nTime : {algo_end - algo_start}\n"
                            f"Time/Sim : {(algo_end - algo_start) / simulations}" + slash_break)


if __name__ == "__main__":
    start = time.time()
    run(n_processors=4)
    end = time.time()
    print(slash_break + slash_break + f"runner.py Total Time : {end - start}\n" + slash_break + slash_break)
