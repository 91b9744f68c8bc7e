"""Cost and content of the iteration record on the headline bench batch (BASELINE.json configs[3]: 4096 randomized 4-vehicle
instances, centralised OBCA, tol 1e-2, the bench's warm start and longest-first order).

Solves the same device-resident batch alternately with recording off and with 128 rows per instance, three pairs, and writes one
JSON file: solves/s of each setting and their spread, whether status / iterations / objective / z are bit-identical between the two,
and an event summary of the batch read from the record (barrier resets, inertia corrections, restarts, raised penalty weights,
the heads of the slowest instance).  The card's name and power limit are read in the same run.

    python tools/gpu_history.py --out profiles/r03_history_overhead_b4096.json
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

from bench import AGENTS, GLOBAL_BATCH, HEADINGS
from conflict_rez_b200.control.batch_planner import prepare_joint_batch, random_init_offsets
from conflict_rez_b200.control.strategy import write_strategy
from conflict_rez_b200.solver import (HIST_F_INERTIA, HIST_F_RESET, HIST_FIELDS, BatchResult, ObcaSolver, SolveOptions, format_history)

CAPACITY, PAIRS = 128, 3
F = {n: k for k, n in enumerate(HIST_FIELDS)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def timed_solve(sv, d):
    sv.set_inputs(d)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    sv.run()
    e1.record()
    st, it, dbl = sv.fetch_stats()
    z = sv.fetch_solution()["z"]
    hist, cnt = sv.fetch_history()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    cpu = lambda t: None if t is None else t.cpu().numpy()
    return ms, dict(status=cpu(st), iters=cpu(it), obj=cpu(dbl[0]), z=cpu(z), hist=cpu(hist), cnt=cpu(cnt))


def dist(x):
    x = np.asarray(x)
    if len(x) == 0:
        return {"n": 0}
    return {"n": int(len(x)), "p50": float(np.median(x)), "p90": float(np.percentile(x, 90)), "max": int(x.max()), "mean": float(x.mean())}


def events(out):
    hist, cnt, iters = out["hist"], out["cnt"], out["iters"]
    B = len(cnt)
    flags = np.nan_to_num(hist[:, :, F["flags"]], nan=0).astype(np.int64)
    reset = (flags & HIST_F_RESET).any(axis=1)
    inertia = (flags & HIST_F_INERTIA).any(axis=1)
    attempts = np.nanmax(hist[:, :, F["attempt"]], axis=1) + 1
    rho0 = hist[:, 0, F["rho"]]
    rho_raised = (np.nanmax(hist[:, :, F["rho"]], axis=1) > rho0)
    groups = {"barrier_reset": reset, "inertia_correction": inertia, "more_than_one_attempt": attempts > 1, "rho_raised": rho_raised}
    summ = {k: {"instances": int(m.sum()), "iterations": dist(iters[m])} for k, m in groups.items()}
    summ["all"] = {"instances": B, "iterations": dist(iters)}
    summ["rows_past_capacity"] = int((cnt > CAPACITY).sum())
    summ["barrier_resets_total"] = int(((flags & HIST_F_RESET) > 0).sum())
    slow = int(np.argmax(iters))
    n = min(int(cnt[slow]), CAPACITY)
    res = BatchResult(*([None] * 14), history=hist, history_count=cnt)
    table = format_history(res, slow).split("\n")
    # the last 10 heads of the slowest instance, or its last 10 stored rows when it ran past the capacity
    summ["slowest"] = {"instance": slow, "iters": int(iters[slow]), "heads": int(cnt[slow]), "past_capacity": bool(cnt[slow] > CAPACITY),
                       "last_10_stored_rows": {f: hist[slow, max(0, n - 10):n, k].tolist() for f, k in F.items()},
                       "last_10_stored_table": [table[0]] + table[1 + max(0, n - 10):1 + n]}
    return summ


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=GLOBAL_BATCH)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gpu_history.py: no CUDA device")
    info = card()
    fn = os.path.join(tempfile.mkdtemp(), "4v")
    write_strategy(fn)
    opts = SolveOptions(tol=1e-2, constr_viol_tol=1e-2, max_iter=600)
    plan = prepare_joint_batch(fn, AGENTS, random_init_offsets(args.batch, 4, seed=0), opts, device="cuda:0", final_headings=HEADINGS)
    cost = np.sum([r.iters for r in plan.singles], axis=0)
    plan.solver.close()
    solvers = {0: ObcaSolver(plan.problem, opts), CAPACITY: ObcaSolver(plan.problem, SolveOptions(tol=1e-2, constr_viol_tol=1e-2, max_iter=600, history=CAPACITY))}
    for sv in solvers.values():
        sv.set_order(cost)
        timed_solve(sv, plan.dev_guess)  # warm-up
    times = {0: [], CAPACITY: []}
    outs = {}
    for _ in range(PAIRS):
        for h, sv in solvers.items():
            ms, outs[h] = timed_solve(sv, plan.dev_guess)
            times[h].append(ms)
    a, b = outs[0], outs[CAPACITY]
    identical = {k: bool(np.array_equal(a[k], b[k])) for k in ("status", "iters", "obj", "z")}
    conv = int((a["status"] >= 0).sum())
    rate = {h: [conv / (ms / 1e3) for ms in t] for h, t in times.items()}
    line = {
        "what": "iteration record off vs %d rows per instance, batch %d (BASELINE.json configs[3]), device-resident k_solve timed by CUDA events, "
                "%d alternating pairs after one warm-up solve each" % (CAPACITY, args.batch, PAIRS),
        "card": info,
        "k_solve_ms": {"off": times[0], "on": times[CAPACITY]},
        "solves_per_s": {"off": rate[0], "on": rate[CAPACITY]},
        "solves_per_s_mean": {"off": float(np.mean(rate[0])), "on": float(np.mean(rate[CAPACITY]))},
        "spread_pct": {h: float(100 * (max(r) - min(r)) / np.mean(r)) for h, r in (("off", rate[0]), ("on", rate[CAPACITY]))},
        "overhead_pct": float(100 * (np.mean(times[CAPACITY]) / np.mean(times[0]) - 1)),
        "bit_identical": identical,
        "converged": conv,
        "record_bytes": int(args.batch * CAPACITY * len(HIST_FIELDS) * 8),
        "events": events(b),
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(line, f, indent=1)
    print(json.dumps({k: line[k] for k in ("card", "solves_per_s_mean", "spread_pct", "overhead_pct", "bit_identical")}))
    for sv in solvers.values():
        sv.close()


if __name__ == "__main__":
    main()
