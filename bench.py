#!/usr/bin/env python
"""bench.py -- converged multi-vehicle OBCA solves/sec (batched) on N B200s of one node; p50 distributed-MPC step ms.

Workload (BASELINE.json configs[3]): ONE global batch of 4096 randomized initial conditions x 4 vehicles, centralised OBCA
(multi_vehicle_planner.py:343-480, K=5, N_per_set=5, shrink_tube=0.5, dmin=0.05, IPOPT tol = constr_viol_tol = 1e-2), sharded
over the N GPUs (strong scaling: global batch fixed, instance b -> rank b % N, no data-path collective).  A "step" = one
batched joint solve of the whole batch from the reference's warm start (single-vehicle solutions + pair duals).

    python bench.py                                   # N = 1, the whole 4096 batch on one GPU
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...              # the CPU restatement (oracle port) on all host cores, full solves

One JSON line on stdout (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

AGENTS = ["vehicle_0", "vehicle_1", "vehicle_2", "vehicle_3"]
HEADINGS = {"vehicle_0": 0.0, "vehicle_1": 3 * np.pi / 2, "vehicle_2": np.pi, "vehicle_3": np.pi / 2}  # multi_vehicle_planner.py:644-649
METRIC = "converged multi-vehicle OBCA solves/sec (batched)"
GLOBAL_BATCH = 4096
# SURVEY.md section 8(d) convention for the 4-vehicle joint problem, per IPM iteration and instance
BYTES_PER_ITER = 3.456e6
FLOPS_PER_ITER_CONVENTION = 767e6
FP64_PEAK_TFLOPS = 37.0  # B200 data sheet (non-tensor FP64); replaced by the measured DFMA figure when available
# ncu --set full capture of k_solve this round (profiles/, see NCU_SOURCE): DRAM bytes per IPM iteration and instance, pipe activity
NCU = {"dram_bytes_per_iter": 21.9e6, "fp64_pipe_pct": 6.7, "issue_active_pct": 20.0, "warps_active_pct": 12.5,
       "source": "profiles/r01c_ncu_full_k_solve_summary_final.txt"}


def load_ncu():
    """The committed ncu summary of the current kernel, if this round produced one (profiles/r02_ncu_k_solve.json)."""
    for name in ("r03m_ncu_k_solve_full_load.json", "r02q_ncu_k_solve.json", "r02g_ncu_k_solve.json", "r02_ncu_k_solve.json"):  # newest first (r03m: one instance on every SM)
        path = os.path.join(ROOT, "profiles", name)
        if os.path.exists(path):
            with open(path) as f:
                d = json.load(f)
            d["source"] = "profiles/" + name
            return d
    return dict(NCU)


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.rows = index, threading.Event(), []

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                for line in out.strip().splitlines():
                    self.rows.append([c.strip() for c in line.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        sm = [float(r[1]) for r in self.rows if len(r) > 2 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for name, val in zip(names, r[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(self.rows)}


# ----------------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port (oracle/ipm.py, SuperLU), FULL converged joint solves, one single-threaded process per core
# ----------------------------------------------------------------------------------------------------------------------
def _cpu_warm_start(fn, offs_b):
    """Joint warm start of one instance on the CPU, the reference's chain with the oracle as the solver: per agent
    tube-following solve (state_ws) -> closed-form obstacle duals (dual_ws) -> single-vehicle OBCA solve; then pair duals."""
    import dataclasses

    from conflict_rez_b200.control import warmstart
    from conflict_rez_b200.control.scenario import build_problem, pose_guess
    from conflict_rez_b200.problem import CollocationGuess
    from oracle import ipm
    from oracle.nlp import CollocationNLP

    opt = ipm.IpmOptions(max_iter=600)
    prob = build_problem(fn, AGENTS, init_offsets=offs_b[None], final_headings=HEADINGS).instance(0)
    V, O, Mmax = prob.V, prob.O, int(prob.nodes.max())
    z, lam, mu, dts = np.zeros((V, Mmax, 7)), np.zeros((V, Mmax, O, 4)), np.zeros((V, Mmax, O, 4)), []
    for ia, agent in enumerate(AGENTS):
        p1 = build_problem(fn, [agent], init_offsets=offs_b[None, ia:ia + 1], final_headings=HEADINGS)
        z0, dt0 = pose_guess(p1, fn, [agent])
        p1 = p1.instance(0)
        M = int(p1.nodes[0])
        p0 = dataclasses.replace(p1, obs_A=np.zeros((0, 4, 2)), obs_b=np.zeros((0, 4)))
        n0 = CollocationNLP(p0)
        g0 = CollocationGuess(z0[0, :, :M], np.zeros((1, M, 0, 4)), np.zeros((1, M, 0, 4)), np.float64(dt0[0, 0]))
        r0 = ipm.solve(n0, n0.init_slacks(n0.pack(g0)), opt)
        zz, dt1 = (n0.unpack(r0.x)["z"], n0.unpack(r0.x)["dt"]) if r0.status >= -2 else (g0.z, float(g0.dt))
        l1, m1 = warmstart.dual_ws_rect(zz[0, :M, 0], zz[0, :M, 1], zz[0, :M, 2], p1.obs_A, p1.obs_b, p1.body_G, p1.body_g)
        n1 = CollocationNLP(p1)
        g1 = CollocationGuess(zz[:, :M], l1[None], m1[None], np.float64(dt1))
        r1 = ipm.solve(n1, n1.init_slacks(n1.pack(g1)), opt)
        u = n1.unpack(r1.x) if r1.status >= -2 else {"z": g1.z, "lam": g1.lam, "mu": g1.mu, "dt": float(g1.dt)}
        z[ia, :M], lam[ia, :M], mu[ia, :M] = u["z"][0, :M], u["lam"][0, :M], u["mu"][0, :M]
        dts.append(u["dt"])
    P = len(prob.pairs)
    pl, pm, ps = np.zeros((P, Mmax, 4)), np.zeros((P, Mmax, 4)), np.zeros((P, Mmax, 2))
    for q, (a, b) in enumerate(prob.pairs):
        m = int(min(prob.nodes[a], prob.nodes[b]))
        pl[q, :m], pm[q, :m], ps[q, :m] = warmstart.joint_dual_ws_rect(z[a, :m, 0], z[a, :m, 1], z[a, :m, 2], z[b, :m, 0], z[b, :m, 1], z[b, :m, 2], prob.body_G, prob.body_g)
    return prob, CollocationGuess(z, lam, mu, np.float64(np.mean(dts)), pl, pm, ps)


def _cpu_full_solve(task):
    """One worker = one core: untimed problem construction (+ warm start when none is given), then ONE timed, full,
    converged joint solve at the reference's tolerance.  Returns measured seconds, iterations, status."""
    os.environ["OMP_NUM_THREADS"] = "1"
    os.environ["OPENBLAS_NUM_THREADS"] = "1"
    fn, offs_b, prob, guess, tol = task
    from oracle import ipm
    from oracle.nlp import CollocationNLP

    t_build = time.perf_counter()
    if guess is None:
        prob, guess = _cpu_warm_start(fn, offs_b)
    nlp = CollocationNLP(prob)  # the analogue of the reference's CasADi graph construction: reported separately
    x0 = nlp.init_slacks(nlp.pack(guess))
    t_build = time.perf_counter() - t_build
    t0 = time.perf_counter()
    res = ipm.solve(nlp, x0, ipm.IpmOptions(tol=tol, constr_viol_tol=tol, max_iter=600))
    return time.perf_counter() - t0, int(res.iters), int(res.status), t_build, float(res.obj)


def cpu_baseline(fn, offs, tol, plan=None, n_proc=None):
    """All host cores, one full converged 4-vehicle solve each (different instances of the same workload)."""
    import multiprocessing as mp

    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        cores = os.cpu_count() or 1
    n_proc = n_proc or cores
    tasks = []
    for b in range(n_proc):
        if plan is not None:
            tasks.append((fn, None, plan.problem.instance(b), plan.guess.instance(b), tol))
        else:
            tasks.append((fn, offs[b], None, None, tol))
    budget = float(os.environ.get("OBCA_CPU_BUDGET_S", "240"))  # wall-clock cap of the pool: keeps the default bench run within minutes
    out, unfinished = [], 0
    with mp.get_context("spawn").Pool(n_proc) as pool:
        t0 = time.perf_counter()
        pending = [pool.apply_async(_cpu_full_solve, (t,)) for t in tasks]
        for r in pending:
            left = budget - (time.perf_counter() - t0)
            try:
                out.append(r.get(timeout=max(left, 0.05)))
            except mp.TimeoutError:
                unfinished += 1
        wall = time.perf_counter() - t0
        pool.terminate()
    if not out:
        return {"value": 0.0, "unit": "solves/s", "cores": n_proc, "kind": "port", "sample": "no CPU solve finished within %.0f s" % budget}
    secs = np.array([o[0] for o in out])
    iters = np.array([o[1] for o in out])
    status = np.array([o[2] for o in out])
    build = np.array([o[3] for o in out])
    conv = int((status >= 0).sum())
    # steady-state throughput of the pool: every core keeps solving back to back at its own measured rate
    value = float(np.sum(1.0 / secs[status >= 0])) if conv else 0.0
    return {
        "value": value, "unit": "solves/s", "cores": n_proc, "kind": "port",
        "sample": "%d full converged 4-vehicle joint solves (one per core, instances 0..%d of the bench batch, tol %.0e) by the oracle port "
        "(oracle/ipm.py: scipy SuperLU, TWO sparse LUs per trial -- the KKT solve and the inertia test); measured per solve: "
        "median %.1f s, max %.1f s, iterations median %d (min %d, max %d), %d/%d converged; untimed per-worker setup "
        "(warm start + sparse NLP assembly) median %.1f s; pool wall %.1f s; %d solve(s) still running at the %.0f s budget are left out "
        "(that favours the CPU figure)"
        % (n_proc, n_proc - 1, tol, float(np.median(secs)), float(secs.max()), int(np.median(iters)), int(iters.min()), int(iters.max()), conv, len(out),
           float(np.median(build)), wall, unfinished, budget),
        "solve_s_median": float(np.median(secs)), "iters_median": float(np.median(iters)), "converged": conv,
        "status_hist": {str(int(k)): int(v) for k, v in zip(*np.unique(status, return_counts=True))},
        "construction_s_median": float(np.median(build)),
    }


# ----------------------------------------------------------------------------------------------------------------------
def mpc_latency(rl_file, device, steps):
    """Second half of BASELINE.json's metric (configs[2]): p50 / p99 latency of one distributed-MPC control step (4 vehicles,
    horizon 30, vehicle_follower.py:main), host parameters in -> first input + predictions on the host."""
    from conflict_rez_b200.control.vehicle_follower import MultiDistributedFollower
    from conflict_rez_b200.pytypes import VehicleState

    mdf = MultiDistributedFollower(rl_file, {a: True for a in AGENTS}, {a: {} for a in AGENTS}, {a: VehicleState() for a in AGENTS}, HEADINGS, device=device)
    mdf.setup_multi_vehicles()
    mdf.solve(num_iter=steps)
    t = 1e3 * np.array(mdf.step_time[5:])  # first steps warm the allocator / pinned buffers
    out = {"p50_step_ms": float(np.percentile(t, 50)), "p99_step_ms": float(np.percentile(t, 99)), "mean_step_ms": float(t.mean()), "steps": int(len(t)),
           "vehicles": len(AGENTS), "solves": int(len(t)) * len(AGENTS), "horizon": 30,
           "failed_solves": int(getattr(mdf, "failed_solves", -1)), "failed_steps": int(getattr(mdf, "failed_steps", -1)),
           "iters_p50": float(np.percentile(mdf.step_iters[5:], 50)), "iters_max": int(np.max(mdf.step_iters[5:])),
           "note": "closed loop of %d control steps, Jacobi exchange of predictions, one batched k_solve launch per control step (4 NLPs); "
           "failed solves fall back to the shifted plan like the reference (vehicle_follower.py:501-524) and are counted, their time is the measured one" % steps}
    # the same closed loop device resident (DeviceMpcLoop): reference window, shifts, solve, fallback and plant step as kernels on
    # one stream; "eager" = one host synchronisation per control step (a controller that has to ship the input), "graph" = one
    # captured step replayed back to back
    try:
        import torch

        from conflict_rez_b200.control.vehicle_follower import DeviceMpcLoop

        np.random.seed(0)
        m2 = MultiDistributedFollower(rl_file, {a: True for a in AGENTS}, {a: {} for a in AGENTS}, {a: VehicleState() for a in AGENTS}, HEADINGS, device=device)
        m2.setup_multi_vehicles()
        loop = DeviceMpcLoop(m2)
        ts = []
        for _ in range(steps):
            ts.append(1e3 * loop.run(1))
        ex = loop.export()
        te = np.array(ts[5:])
        out["device_loop"] = {"p50_step_ms": float(np.percentile(te, 50)), "p99_step_ms": float(np.percentile(te, 99)), "mean_step_ms": float(te.mean()),
                              "steps": int(len(te)), "failed_solves": int(ex["failed_solves"]), "iters_p50": float(np.percentile(ex["iters"].max(1)[5:], 50))}
        np.random.seed(0)
        m3 = MultiDistributedFollower(rl_file, {a: True for a in AGENTS}, {a: {} for a in AGENTS}, {a: VehicleState() for a in AGENTS}, HEADINGS, device=device)
        m3.setup_multi_vehicles()
        g = DeviceMpcLoop(m3)
        g.run(5)  # the restoration-heavy first steps stay out of the replayed average
        out["device_loop"]["graph_mean_step_ms"] = 1e3 * g.run(steps - 5, graph=True)
    except Exception as e:  # the device loop is an extra: report why it is missing instead of losing the bench line
        out["device_loop"] = {"error": repr(e)[:200]}
    return out


def latency_single_instance(fn, device, opts):
    """configs[0] / configs[1]: one single-vehicle plan and one 4-vehicle centralised plan, host buffers in -> host buffers out."""
    import torch

    from conflict_rez_b200.control.batch_planner import prepare_joint_batch
    from conflict_rez_b200.control.scenario import build_guess, build_problem
    from conflict_rez_b200.solver import ObcaSolver

    out = {}
    t0 = time.perf_counter()
    p1 = build_problem(fn, ["vehicle_0"], final_headings=HEADINGS)
    g1 = build_guess(p1, fn, ["vehicle_0"])
    sv = ObcaSolver(p1, opts, device=device)
    torch.cuda.synchronize(device)
    out["config1_setup_ms"] = 1e3 * (time.perf_counter() - t0)
    ts = []
    for _ in range(4):
        t0 = time.perf_counter()
        r = sv.solve(g1)
        ts.append(1e3 * (time.perf_counter() - t0))
    out.update(config1_single_vehicle_ms=float(np.median(ts[1:])), config1_iters=int(r.iters[0]), config1_status=r.return_status(0))
    sv.close()
    offs = np.zeros((1, 4, 3))
    offs[0, 0] = [0.1, 0.0, np.pi / 20]  # multi_vehicle_planner.py:641-642
    t0 = time.perf_counter()
    plan = prepare_joint_batch(fn, AGENTS, offs, opts, device=device, final_headings=HEADINGS)
    torch.cuda.synchronize(device)
    out["config2_warm_start_ms"] = 1e3 * (time.perf_counter() - t0)
    ts = []
    for _ in range(4):
        t0 = time.perf_counter()
        r = plan.solver.solve(plan.guess)
        ts.append(1e3 * (time.perf_counter() - t0))
    out.update(config2_four_vehicle_joint_ms=float(np.median(ts[1:])), config2_iters=int(r.iters[0]), config2_status=r.return_status(0))
    plan.solver.close()
    return out


# (vehicles, obstacles, intervals per move): BASELINE.json configs[4] -- V 2-8 x O 5-20 x N 20-100 at batch 1024.  The parking lot
# has 6 obstacles (fewer is not this scenario), extra ones are seeded rectangles between the tubes; N = n_per_set x 9 moves
SWEEP_CELLS = [(2, 6, 5), (4, 6, 5), (8, 12, 5), (4, 10, 5), (4, 20, 5), (4, 6, 2), (4, 6, 11), (8, 12, 2)]


def sweep_leg(fn, device, tol, batch, cells=None):
    """Scaling sweep: one batched joint solve per cell, device-timed (1 warm-up + 1 timed launch, warm start untimed)."""
    import torch

    from conflict_rez_b200.control.batch_planner import prepare_joint_batch, prepare_replicated_batch, random_init_offsets
    from conflict_rez_b200.control.scenario import random_obstacles
    from conflict_rez_b200.solver import RETURN_STATUS, SolveOptions

    out = []
    opts = SolveOptions(tol=tol, constr_viol_tol=tol, max_iter=600)
    for V, O, nps in cells or SWEEP_CELLS:
        t0 = time.perf_counter()
        copies = 2 if V > 4 else 1
        v1 = V // copies
        agents = AGENTS if v1 == 4 else ["vehicle_1", "vehicle_2"] if v1 == 2 else AGENTS[1:1 + v1]
        idx = [int(a[-1]) for a in agents]
        heads = {a: HEADINGS[a] for a in agents}
        kw = dict(n_per_set=nps, final_headings=heads)
        n_extra = O // copies - 6
        if n_extra > 0:
            kw["obstacles"] = random_obstacles(fn, n_extra, seed=7)
        offs = random_init_offsets(batch, 4 * copies, seed=3).reshape(batch, copies, 4, 3)[:, :, idx].reshape(batch, copies * v1, 3)
        try:
            if copies == 1:
                plan = prepare_joint_batch(fn, agents, offs, opts, device=device, **kw)
            else:
                plan = prepare_replicated_batch(fn, agents, copies, offs, opts, device=device, **kw)
            sv = plan.solver
            sv.set_order(np.sum([r.iters for r in plan.singles[:v1]], axis=0))
            torch.cuda.synchronize(device)
            t_ws = time.perf_counter() - t0
            sv.set_inputs(plan.dev_guess), sv.run(), sv.fetch_stats()
            torch.cuda.synchronize(device)
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            sv.set_inputs(plan.dev_guess)
            a0.record()
            sv.run()
            a1.record()
            st, it, _ = sv.fetch_stats()
            torch.cuda.synchronize(device)
            st, it = st.cpu().numpy(), it.cpu().numpy()
            ms = a0.elapsed_time(a1)
            L = sv.layout()
            out.append({"vehicles": plan.problem.V, "obstacles": plan.problem.O, "intervals": int(plan.problem.nodes.max()) // 6, "batch": batch,
                        "nx": L["nx"], "ny": L["ny"], "solves_per_s": float((st >= 0).sum()) / (ms / 1e3), "k_solve_ms": ms,
                        "converged_fraction": float((st >= 0).mean()), "iters_median": float(np.median(it)), "iters_max": int(it.max()),
                        "ms_per_iteration_and_instance": ms * min(batch, 148) / float(it.sum()),
                        "status_hist": {RETURN_STATUS[int(k)]: int(v) for k, v in zip(*np.unique(st, return_counts=True))},
                        "warm_start_s": t_ws})
            sv.close()
        except Exception as e:  # a cell that does not fit (memory, shape limits) is reported, not hidden
            out.append({"vehicles": V, "obstacles": O, "n_per_set": nps, "batch": batch, "error": "%s: %s" % (type(e).__name__, str(e)[:300])})
        torch.cuda.empty_cache()
    return out


# instances whose whole solution --dump-outputs writes: 64 x 0.6 MB (z, lam, mu, dt, pair duals of 4 vehicles in float64) = 39 MB
DUMP_SAMPLE = 64


def dump_outputs(out_dir, st, it, dbl, sol):
    """What one step of the timed path returns, as float64 ``out_dir/<name>.npy``: the per-instance statistics of the whole batch
    (status, iters, obj, cviol, dual_inf, compl_inf, elastic) and the solution of a fixed, seeded sample of instances (z, lam, mu,
    dt, pair_lam, pair_mu, pair_s; ``instance`` holds their batch indices)."""
    import torch

    os.makedirs(out_dir, exist_ok=True)
    B = st.shape[0]
    idx = np.sort(np.random.default_rng(0).choice(B, min(B, DUMP_SAMPLE), replace=False))
    sel = torch.as_tensor(idx, device=st.device)
    arrays = {"status": st, "iters": it, **dict(zip(("obj", "cviol", "dual_inf", "compl_inf", "elastic"), dbl)), "instance": idx}
    names = {"pl": "pair_lam", "pm": "pair_mu", "ps": "pair_s"}
    arrays.update({names.get(k, k): v.index_select(0, sel) for k, v in sol.items()})
    for name, a in arrays.items():
        a = a.cpu().numpy() if torch.is_tensor(a) else a
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=GLOBAL_BATCH, help="GLOBAL batch (BASELINE.json configs[3]: 4096), sharded over the ranks")
    ap.add_argument("--weak", action="store_true", help="weak scaling instead: --batch instances PER GPU")
    ap.add_argument("--tol", type=float, default=1e-2, help="IPOPT tol / constr_viol_tol of the reference (vehicle.py:651-652)")
    ap.add_argument("--no-pipeline", action="store_true", help="one handle, one stream: every step waits for the previous step's last instance (default: two handles on two streams, conflict_rez_b200.solver.PipelinedSolver)")
    ap.add_argument("--no-lpt", action="store_true", help="process the instances in index order instead of longest-expected-first")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the tight-tolerance leg, the single-instance latencies and the MPC leg")
    ap.add_argument("--mpc-steps", type=int, default=250)
    ap.add_argument("--tight-batch", type=int, default=592)
    ap.add_argument("--sweep", action="store_true", help="add the scaling sweep (BASELINE.json configs[4]) at --sweep-batch instances per cell")
    ap.add_argument("--sweep-batch", type=int, default=1024)
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed to DIR/<name>.npy (float64; "
                    "statistics of every instance, solutions of %d seeded instances) to compare two builds output for output" % DUMP_SAMPLE)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and (args.impl != "ours" or world > 1):
        ap.error("--dump-outputs needs --impl ours in a single process")
    global_batch = args.batch * world if args.weak else args.batch

    from conflict_rez_b200.control.batch_planner import random_init_offsets, shard_instances
    from conflict_rez_b200.control.strategy import write_strategy

    config = {
        "workload": "BASELINE.json configs[3]: batch of %d randomized initial conditions x 4 vehicles, centralized OBCA (multi_vehicle_planner.py "
        "defaults: K=5, N_per_set=5, shrink_tube=0.5, dmin=0.05), parking-lot scenario, synthetic strategy; sharded over the GPUs" % global_batch,
        "global_batch": global_batch,
        "batch_per_gpu": (global_batch + world - 1) // world,
        "vehicles": 4,
        "obstacles": 6,
        "tol": args.tol,
        "queue": "index order" if args.no_lpt else "longest-expected-first (predictor: iterations of the single-vehicle warm-start solves)",
        "pipeline": "none (one handle, one stream)" if args.no_pipeline else "consecutive steps double buffered: two library handles on two CUDA streams (PipelinedSolver); the next batch's CTAs "
        "start on the SMs the previous batch's last wave frees, host<->device copies of the e2e leg overlap the other handle's solve; every step is a full solve of the whole batch",
        "l2": "per-step working set (iterates of the batch, > 2 MB per instance) is larger than the 126 MB L2; no explicit flush",
        "parallelism": "instance b -> GPU b %% %d, no data-path collective" % world,
    }
    fn = os.path.join(tempfile.mkdtemp(), "4v")
    write_strategy(fn)
    offs_all = random_init_offsets(global_batch, 4, seed=0)

    if args.impl == "reference":
        # CPU arm: the oracle port on all host cores (rank 0 only); a step = one full converged solve per core
        if rank != 0:
            return
        t_all = time.perf_counter()
        cb = cpu_baseline(fn, offs_all, args.tol)
        line = {
            "metric": METRIC, "value": cb["value"], "unit": "solves/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * cb["cores"] / max(cb["value"], 1e-12), "higher_is_better": True, "scaling": "weak" if args.weak else "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config, "impl": "reference", "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0,
            "wall_s": time.perf_counter() - t_all,
            "note": "reference arm = CPU restatement of the reference path (oracle port: numpy/scipy SuperLU interior point), measured on full "
            "converged solves from the same kind of warm start (single-vehicle solutions + pair duals, computed by the same port, untimed); one "
            "measured step (a full solve per core) stands for every --steps/--warmup step; CasADi/IPOPT/HSL are not installable in this image",
        }
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist

    from conflict_rez_b200.control.batch_planner import prepare_joint_batch
    from conflict_rez_b200.solver import SolveOptions

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the OBCA solver has no CPU fallback")
    # torchrun sets OMP_NUM_THREADS=1: give every rank its share of the host cores back (the e2e leg stages its buffers with torch's
    # multi-threaded CPU copy)
    torch.set_num_threads(max(1, (os.cpu_count() or 8) // max(1, world)))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL prints its version banner to stdout when the communicator is created: keep stdout for the one JSON line
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=device)
            dist.barrier()
            torch.cuda.synchronize(device)
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    opts = SolveOptions(tol=args.tol, constr_viol_tol=args.tol, max_iter=600)
    mine = shard_instances(global_batch, rank, world)  # interleaved shard: random instances, equal expected load per rank
    offs = offs_all[mine]
    B = len(mine)
    # the warm-start pipeline runs twice: the first call also pays the one-time costs of a process (CUDA context, growth of the device
    # memory pool the handles allocate from, pinned staging buffers); the second one is what a planner that runs continuously sees
    t_ws0 = time.perf_counter()
    plan = prepare_joint_batch(fn, AGENTS, offs, opts, device=device, final_headings=HEADINGS)
    torch.cuda.synchronize(device)
    t_ws0 = time.perf_counter() - t_ws0
    plan.solver.close()
    del plan
    t_ws = time.perf_counter()
    plan = prepare_joint_batch(fn, AGENTS, offs, opts, device=device, final_headings=HEADINGS)  # warm start, device resident
    torch.cuda.synchronize(device)
    t_ws = time.perf_counter() - t_ws
    sv = plan.solver
    cost = np.sum([r.iters for r in plan.singles], axis=0)
    if not args.no_lpt:
        sv.set_order(cost)
    # Consecutive steps are independent batches: by default they are double buffered over two library handles on two streams
    # (PipelinedSolver), so that the next batch's CTAs take over every SM the previous batch's last wave leaves idle.
    pipe = None
    if not args.no_pipeline:
        from conflict_rez_b200.solver import PipelinedSolver

        pipe = PipelinedSolver(plan.problem, opts, device=device, depth=2, first=sv)
        if not args.no_lpt:
            pipe.set_order(cost)
    counter = pipe if pipe is not None else sv

    # ---------------- device-resident timing (value): inputs already in HBM (the warm start never left the device)
    dev_in = plan.dev_guess
    barrier()
    if pipe is not None:
        pipe.run_resident(dev_in, max(args.warmup, 2))
    else:
        for _ in range(args.warmup):
            sv.set_inputs(dev_in)
            sv.run()
            sv.fetch_stats()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = counter.launch_count
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ksolve_ms = []
    pipeline_consistent = True
    ev[0].record()
    if pipe is not None:
        outs = pipe.run_resident(dev_in, args.steps)
        st, it, dbl = outs[-1]
    else:
        for _ in range(args.steps):
            sv.set_inputs(dev_in)
            k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            k0.record()
            sv.run()
            k1.record()
            st, it, dbl = sv.fetch_stats()
            ksolve_ms.append((k0, k1))
    ev[1].record()
    barrier()
    sampler.stop_flag.set()
    if pipe is not None:  # every step solved the same batch: both handles must agree bit for bit
        pipeline_consistent = all(bool(torch.equal(o[0], outs[0][0])) and bool(torch.equal(o[1], outs[0][1])) and bool(torch.equal(o[2][0], outs[0][2][0])) for o in outs)
    launches = counter.launch_count - launches0
    t_dev = ev[0].elapsed_time(ev[1]) / 1e3
    # pipelined: the launches overlap, their individual durations include waiting for SMs -- the kernel time per step is the timed region / steps
    t_kernel = float(np.mean([a.elapsed_time(b) for a, b in ksolve_ms])) / 1e3 if ksolve_ms else t_dev / args.steps
    if args.dump_outputs:  # the solution of the last step stays in the handle that ran it
        last = pipe.solvers[(args.steps - 1) % len(pipe.solvers)] if pipe is not None else sv
        dump_outputs(args.dump_outputs, st, it, dbl, last.fetch_solution())
    st_h, it_h = st.cpu().numpy(), it.cpu().numpy()
    converged = int((st_h >= 0).sum())
    sum_iters = float(it_h.sum())

    # ---------------- end-to-end timing (e2e): host buffers in, host results out, through the public solve() call
    if pipe is not None:
        if args.warmup:
            pipe.solve_many([plan.guess] * 2, want_duals=False)  # one per handle: pinned staging buffers of both exist
    else:
        for _ in range(min(1, args.warmup)):
            sv.solve(plan.guess, want_duals=False)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    if pipe is not None:
        res = pipe.solve_many([plan.guess] * args.steps, want_duals=False)[-1]
    else:
        for _ in range(args.steps):
            res = sv.solve(plan.guess, want_duals=False)
    torch.cuda.synchronize(device)
    e1.record()
    barrier()
    t_e2e = e0.elapsed_time(e1) / 1e3
    g = plan.guess
    h2d = sum(int(np.asarray(a).nbytes) for a in (plan.problem.init_pose, g.z, g.lam, g.mu, g.dt, g.pair_lam, g.pair_mu, g.pair_s))
    d2h = sum(int(a.nbytes) for a in (res.z, res.dt, res.pair_lam, res.pair_mu, res.pair_s, res.status, res.iters, res.obj, res.cviol, res.dual_inf,
                                      res.compl_inf, res.elastic))  # want_duals=False: lam / mu stay on the device
    conv_e2e = int((res.status >= 0).sum())

    # ---------------- reduce over ranks: time = max, counts = sum
    stats = torch.tensor([t_dev, t_e2e, t_kernel], dtype=torch.float64, device=device)
    counts = torch.tensor([converged, conv_e2e, sum_iters, launches, float(B), h2d, d2h], dtype=torch.float64, device=device)
    hist_codes = [0, 1, -1, -2, -3, -4, -5, -6]
    hist = torch.tensor([float((st_h == c).sum()) for c in hist_codes], dtype=torch.float64, device=device)
    per_rank = torch.zeros(world, 3, dtype=torch.float64, device=device)
    per_rank[rank] = torch.tensor([t_kernel, sum_iters, float(it_h.max())], dtype=torch.float64)
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
        dist.all_reduce(counts, op=dist.ReduceOp.SUM)
        dist.all_reduce(hist, op=dist.ReduceOp.SUM)
        dist.all_reduce(per_rank, op=dist.ReduceOp.SUM)
    t_dev, t_e2e, t_kernel = [float(v) for v in stats.cpu()]
    converged, conv_e2e, sum_iters, launches, total, h2d, d2h = [float(v) for v in counts.cpu()]
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    from conflict_rez_b200.solver import RETURN_STATUS

    value = converged * args.steps / t_dev
    e2e_value = conv_e2e * args.steps / t_e2e
    peak, peak_src = load_peaks()
    ncu = load_ncu()
    import ctypes

    fp64_peak = ctypes.c_double(0.0)
    fp64_src = "data sheet"
    if sv.lib.obca_measure_dfma_peak(local_rank, ctypes.byref(fp64_peak)) == 0 and fp64_peak.value > 0:
        fp64_src = "measured (obca_measure_dfma_peak: 8 independent DFMA chains per thread, 8 CTAs of 256 threads per SM)"
    else:
        fp64_peak.value = FP64_PEAK_TFLOPS
    achieved_gbs = sum_iters * BYTES_PER_ITER / t_kernel / 1e9 / world  # per GPU, dominant kernel k_solve
    pr = per_rank.cpu().numpy()
    line = {
        "metric": METRIC,
        "value": value,
        "unit": "solves/s",
        "n_gpus": world,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": 1e3 * t_dev / args.steps,
        "higher_is_better": True,
        "scaling": "weak" if args.weak else "strong",
        "vs_baseline": None,
        "dtype": "f64",
        "data": "synthetic",
        "config": config,
        "converged_fraction": converged / max(1.0, total),
        "iters_median": float(np.median(it_h)),
        "iters_max": int(pr[:, 2].max()),
        "status_hist": {RETURN_STATUS[c]: int(v) for c, v in zip(hist_codes, hist.cpu().numpy()) if v > 0},
        "per_rank": {"k_solve_ms": [round(1e3 * float(v), 2) for v in pr[:, 0]], "sum_iters": [int(v) for v in pr[:, 1]],
                     "k_solve_ms_note": "average launch duration (CUDA events around each launch)" if args.no_pipeline else "timed region / steps (the launches of consecutive steps overlap)"},
        "e2e": {"value": e2e_value, "unit": "solves/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
        "gpu_launches": int(launches),
        "pipeline_consistent": bool(pipeline_consistent),  # the steps of the timed region (alternating handles) returned bit-identical statuses / iterations / objectives
        "clocks": sampler.summary(),
        "roofline": {
            "bound": "hbm",
            "kernel": "k_solve (one CTA per instance: NLP evaluation + structured KKT solve + IPM loop)",
            "achieved": achieved_gbs,
            "peak": peak,
            "unit": "GB/s",
            "frac": achieved_gbs / peak,
            "traffic": ncu["dram_bytes_per_iter"] * sum_iters / world,
            "traffic_note": "%.1f MB of DRAM traffic per IPM iteration and instance (dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full "
            "capture of k_solve, %s) x the iterations of one launch (per GPU); algorithmic bytes are 3.456 MB per iteration" % (ncu["dram_bytes_per_iter"] / 1e6, ncu["source"]),
            "fp64_pipe_pct": ncu["fp64_pipe_pct"],
            "issue_active_pct": ncu["issue_active_pct"],
            "warps_active_pct": ncu["warps_active_pct"],
            "ncu_source": ncu["source"],
            "peak_source": peak_src,
            "note": "algorithmic bytes = 3.456 MB per IPM iteration and instance (one read + one write of the primal-dual iterate, SURVEY.md 8d) "
            "x iterations of all instances / k_solve time; the kernel is FP64-latency bound, not bandwidth bound (DESIGN.md)"
            + ("" if args.no_pipeline else "; pipelined steps: the launches of consecutive steps overlap, so the k_solve time per launch is the timed region / steps "
               "(with --no-pipeline it is the average of CUDA events around each launch: 4592 ms vs 4594 ms per step at batch 4096)"),
            "fp64_convention": {
                "achieved_tflops": sum_iters * FLOPS_PER_ITER_CONVENTION / t_kernel / 1e12 / world,
                "peak_tflops": fp64_peak.value,
                "frac": sum_iters * FLOPS_PER_ITER_CONVENTION / t_kernel / 1e12 / world / fp64_peak.value,
                "peak_source": fp64_src,
                "note": "SURVEY.md 8d counts 767 MFLOP/iteration for a dense block elimination; the null-space Riccati solve needs far fewer flops, "
                "so this is an equivalent-work figure, not executed flops (executed: ncu fp64_pipe_pct)",
            },
        },
    }
    ws_total = t_ws
    line["warm_start"] = {
        "wall_s_rank0": t_ws, "first_call_wall_s_rank0": t_ws0, **plan.timing, "single_vehicle_fail_rank0": int(sum((r.status < 0).sum() for r in plan.singles)),
        "plan_to_plan_solves_per_s": converged / (ws_total + t_dev / args.steps) if world == 1 else None,
        "note": "untimed setup of the step (SURVEY.md 8f rank 1), second call of the pipeline in this process (first_call_wall_s_rank0 = the first, with "
        "the process's one-time costs): kinematic guess on the host, state_ws (Euler NLP) + interp_ws_for_collocation, obstacle and pair "
        "duals by obca_dual_ws / obca_joint_dual_ws on the device, 4 batched single-vehicle solves; the joint warm start stays in HBM. "
        "plan_to_plan = converged plans / (warm-start pipeline + one joint solve), the reference's solve_single_problems -> solve_final_problem_obca chain",
    }
    if world == 1 and not args.no_extras:
        # tight tolerance (BASELINE.md 3.5): same workload at tol = constr_viol_tol = 1e-8 (iterative refinement on), a sub-batch of whole waves
        nb = min(args.tight_batch, B)
        topts = SolveOptions(tol=1e-8, constr_viol_tol=1e-8, max_iter=600)
        from conflict_rez_b200.problem import CollocationGuess
        from conflict_rez_b200.solver import ObcaSolver

        sub = plan.problem
        import copy

        subp = copy.copy(sub)
        subp.init_pose = sub.init_pose[:nb]
        tsv = ObcaSolver(subp, topts, device=device)
        gsub = CollocationGuess(g.z[:nb], g.lam[:nb], g.mu[:nb], g.dt[:nb], g.pair_lam[:nb], g.pair_mu[:nb], g.pair_s[:nb])
        d_in = tsv.upload(gsub)
        tsv.set_inputs(d_in), tsv.run(), tsv.fetch_stats()
        torch.cuda.synchronize(device)
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        tsv.set_inputs(d_in), tsv.run()
        tst, tit, tdbl = tsv.fetch_stats()
        a1.record()
        torch.cuda.synchronize(device)
        tst, tit = tst.cpu().numpy(), tit.cpu().numpy()
        line["tight_tolerance"] = {"tol": 1e-8, "batch": nb, "value": float((tst >= 0).sum()) / (a0.elapsed_time(a1) / 1e3), "unit": "solves/s",
                                   "iters_median": float(np.median(tit)), "iters_max": int(tit.max()),
                                   "status_hist": {RETURN_STATUS[int(k)]: int(v) for k, v in zip(*np.unique(tst, return_counts=True))},
                                   "max_cviol_converged": float(tdbl[1].cpu().numpy()[tst >= 0].max()) if (tst >= 0).any() else None}
        tsv.close()
        line["latency"] = latency_single_instance(fn, device, opts)
        line["mpc"] = mpc_latency(fn, device, args.mpc_steps)
    if world == 1 and args.sweep:
        line["sweep"] = sweep_leg(fn, device, args.tol, args.sweep_batch)
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(fn, offs_all, args.tol, plan=plan)
    sv.close()
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
