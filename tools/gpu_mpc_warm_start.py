"""Warm start from the stored primal-dual iterate (obca_warm_start) in the two workloads that solve nearly the same problem again.

1. Distributed MPC, the 4-vehicle scene of bench.py's MPC leg through DeviceMpcLoop (horizon 30, one batched launch per control
   step).  First a sweep of warm_start_mu_init x push (warm_start_bound_push = warm_start_mult_bound_push) over --sweep-steps steps,
   each configuration on a fresh handle from the same plans and first-step duals.  The push whose worst vehicle-step over all
   mu_init is the smallest is chosen, then the mu_init with the fewest iterations over steps 2.. at that push.  Then --steps control
   steps cold and warm (chosen configuration), the two loops alternated step by step in this process: per-step latency (host clock
   around one synchronised control step), iterations per vehicle and step, failed solves.
2. Loose -> tight on the bench batch (4-vehicle centralised OBCA, --tight-batch instances of bench.py's seeded offsets): a cold
   tol 1e-8 solve against a tol 1e-2 solve followed by a warm tol 1e-8 solve from its iterate, solves/s of both routes (CUDA events),
   alternated over --reps repetitions.

The card's name and power limit are read in the same run.

    python tools/gpu_mpc_warm_start.py --out profiles/r04_mpc_warm_start.json
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

from bench import AGENTS, HEADINGS
from conflict_rez_b200.control import vehicle_follower as vf
from conflict_rez_b200.control.strategy import write_strategy
from conflict_rez_b200.pytypes import VehicleState
from conflict_rez_b200.solver import RETURN_STATUS, ObcaMpcSolver, ObcaSolver, SolveOptions

MU_INITS, PUSHES = (1e-2, 1e-3, 1e-4, 1e-5), (1e-3, 1e-6, 1e-9)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def ws_options(mu_init, push):
    return dict(warm_start_bound_push=push, warm_start_mult_bound_push=push, warm_start_mu_init=mu_init)


class Loop:
    """One DeviceMpcLoop on a fresh handle of the shared scene (same plans, same first-step duals)."""

    def __init__(self, mdf, warm, ws):
        mdf.solver = ObcaMpcSolver(mdf.vehicles[0].mpc_problem(batch=len(mdf.vehicles)), SolveOptions(max_iter=600, **ws), device=mdf.device)
        self.loop = vf.DeviceMpcLoop(mdf, warm_start=warm)
        self.ms = []

    def step(self):
        self.ms.append(1e3 * self.loop.run(1))  # run() synchronises before and after the step

    def summary(self, skip=5):
        ex = self.loop.export()
        it, st = ex["iters"], ex["status"]
        t = np.array(self.ms[skip:])
        return {"steps": int(len(self.ms)), "p50_step_ms": float(np.percentile(t, 50)), "p99_step_ms": float(np.percentile(t, 99)),
                "mean_step_ms": float(t.mean()), "iters_per_vehicle_step_p50": float(np.percentile(it[1:], 50)),
                "iters_per_vehicle_step_max": int(it[1:].max()), "iters_sum_steps_2_on": int(it[1:].sum()),
                "iters_max_vehicle_p50": float(np.percentile(it[1:].max(1), 50)), "failed_solves": int((st < 0).sum()),
                "latency_skips_first_steps": skip}


def mpc_leg(fn, device, steps, sweep_steps):
    np.random.seed(0)
    mdf = vf.MultiDistributedFollower(fn, {a: True for a in AGENTS}, {a: {} for a in AGENTS}, {a: VehicleState() for a in AGENTS}, HEADINGS, device=device)
    mdf.setup_multi_vehicles()
    sweep = []
    cold = Loop(mdf, False, {})
    for _ in range(sweep_steps):
        cold.step()
    base = cold.summary()
    for mu_init in MU_INITS:
        for push in PUSHES:
            lp = Loop(mdf, True, ws_options(mu_init, push))
            for _ in range(sweep_steps):
                lp.step()
            s = lp.summary()
            sweep.append(dict(mu_init=mu_init, push=push, **{k: s[k] for k in ("iters_sum_steps_2_on", "iters_per_vehicle_step_p50", "iters_per_vehicle_step_max",
                                                                               "failed_solves", "p50_step_ms", "p99_step_ms")}))
    # push: the value whose worst vehicle-step (largest iteration count, failures counted as the limit) over every mu_init is the
    # smallest -- tiny pushes leave iterates on their bounds and show heavy tails; then mu_init: fewest iterations at that push
    tail = lambda s: s["iters_per_vehicle_step_max"] + 600 * s["failed_solves"]
    push = min(PUSHES, key=lambda q: max(tail(s) for s in sweep if s["push"] == q))
    best = min((s for s in sweep if s["push"] == push), key=lambda s: (s["failed_solves"], s["iters_sum_steps_2_on"]))
    chosen = ws_options(best["mu_init"], best["push"])
    loops = {"cold": Loop(mdf, False, {}), "warm": Loop(mdf, True, chosen)}
    for _ in range(steps):
        for lp in loops.values():  # alternated step by step
            lp.step()
    return {"sweep_steps": sweep_steps, "sweep_cold": {k: base[k] for k in ("iters_sum_steps_2_on", "iters_per_vehicle_step_p50", "iters_per_vehicle_step_max",
                                                                          "failed_solves", "p50_step_ms", "p99_step_ms")},
            "sweep": sweep, "chosen": chosen, "run": {k: lp.summary() for k, lp in loops.items()}}


def tight_leg(fn, device, nb, reps):
    from conflict_rez_b200.control.batch_planner import prepare_joint_batch, random_init_offsets

    loose_opts = SolveOptions(tol=1e-2, constr_viol_tol=1e-2, max_iter=600)
    tight_opts = SolveOptions(tol=1e-8, constr_viol_tol=1e-8, max_iter=600)
    offs = random_init_offsets(nb, 4, seed=0)  # bench.py's seeded offsets (its first nb instances)
    plan = prepare_joint_batch(fn, AGENTS, offs, loose_opts, device=device, final_headings=HEADINGS)
    d_in, loose = plan.dev_guess, plan.solver
    cold = ObcaSolver(plan.problem, tight_opts, device=device)
    warm = ObcaSolver(plan.problem, tight_opts, device=device)
    warm.set_inputs(d_in)  # the initial poses, once per batch (the guess part of x is replaced by the loose iterate)

    def route_cold():
        cold.set_inputs(d_in)
        cold.run()
        return cold.fetch_stats()

    def route_warm():
        loose.set_inputs(d_in)
        loose.run()
        warm.put_iterate(loose.fetch_iterate())
        warm.arm_warm_start()
        warm.run()
        return warm.fetch_stats()

    out = {"cold": [], "warm": []}
    last = {}
    for rep in range(reps + 1):  # repetition 0 warms up
        for name, fnc in (("cold", route_cold), ("warm", route_warm)):
            torch.cuda.synchronize(device)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            st, it, dbl = fnc()
            e1.record()
            torch.cuda.synchronize(device)
            st, it = st.cpu().numpy(), it.cpu().numpy()
            ms = e0.elapsed_time(e1)
            last[name] = (st, it, dbl[0].cpu().numpy())
            if rep:
                out[name].append({"ms": ms, "solves_per_s": float((st >= 0).sum()) / (ms / 1e3)})
    lst, lit, _ = loose.fetch_stats()
    lit = lit.cpu().numpy()
    res = {"batch": nb, "reps": reps}
    for name in ("cold", "warm"):
        st, it, obj = last[name]
        sps = [r["solves_per_s"] for r in out[name]]
        res[name] = {"solves_per_s_median": float(np.median(sps)), "solves_per_s_min": float(np.min(sps)), "solves_per_s_max": float(np.max(sps)),
                     "ms_median": float(np.median([r["ms"] for r in out[name]])), "tight_iters_median": float(np.median(it)), "tight_iters_max": int(it.max()),
                     "status_hist": {RETURN_STATUS[int(k)]: int(v) for k, v in zip(*np.unique(st, return_counts=True))}}
    res["warm"]["loose_iters_median"] = float(np.median(lit))
    both = (last["cold"][0] == 0) & (last["warm"][0] == 0)
    rel = np.abs(last["warm"][2] - last["cold"][2]) / np.abs(last["cold"][2])
    res["objective_rel_diff_where_both_succeed"] = {"n": int(both.sum()), "median": float(np.median(rel[both])) if both.any() else None,
                                                    "max": float(rel[both].max()) if both.any() else None}
    for s in (loose, cold, warm):
        s.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=250)
    ap.add_argument("--sweep-steps", type=int, default=50)
    ap.add_argument("--tight-batch", type=int, default=592)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gpu_mpc_warm_start.py: no CUDA device")
    device = torch.device("cuda", 0)
    fn = os.path.join(tempfile.mkdtemp(), "4v_rl_traj")
    write_strategy(fn)
    t0 = time.perf_counter()
    out = {"card": card(), "tool": "tools/gpu_mpc_warm_start.py", "args": vars(args)}
    out["mpc"] = mpc_leg(fn, device, args.steps, args.sweep_steps)
    print(json.dumps({"mpc_chosen": out["mpc"]["chosen"], "run": out["mpc"]["run"]}), flush=True)
    out["loose_to_tight"] = tight_leg(fn, device, args.tight_batch, args.reps)
    out["wall_s"] = time.perf_counter() - t0
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out["loose_to_tight"]))


if __name__ == "__main__":
    main()
