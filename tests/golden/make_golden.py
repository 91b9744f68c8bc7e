"""Regenerates the golden fixtures in this directory from the CPU oracle (oracle/nlp.py + oracle/ipm.py).

    python tests/golden/make_golden.py

The reference ships no golden vectors for the OBCA path and CasADi/IPOPT cannot be installed in this image
(SURVEY.md section 8c), so these fixtures pin the *restated* formulation: problem data, warm start, and the oracle's
solution at tight tolerance.  Parity therefore stays "unpinned" at the CasADi/IPOPT boundary.
"""
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from conflict_rez_b200.control import warmstart  # noqa: E402
from conflict_rez_b200.control.scenario import build_guess, build_problem  # noqa: E402
from conflict_rez_b200.control.strategy import write_strategy  # noqa: E402
from conflict_rez_b200.problem import CollocationGuess  # noqa: E402
from oracle import ipm  # noqa: E402
from oracle.nlp import CollocationNLP  # noqa: E402

PROB_FIELDS = ["n_sets", "obs_A", "obs_b", "tube_A", "tube_b", "init_pose", "final_heading", "body_G", "body_g", "region", "limits"]


def save(name, prob, guess, nlp, res):
    u = nlp.unpack(res.x)
    out = {"p_" + k: getattr(prob, k) for k in PROB_FIELDS}
    out.update(p_wb=prob.wb, p_dmin=prob.dmin, p_shrink=prob.shrink_tube, p_K=prob.K, p_n_per_set=prob.n_per_set)
    out.update(g_z=guess.z, g_lam=guess.lam, g_mu=guess.mu, g_dt=guess.dt)
    if guess.pair_lam is not None:
        out.update(g_pl=guess.pair_lam, g_pm=guess.pair_mu, g_ps=guess.pair_s)
    out.update(s_z=u["z"], s_dt=u["dt"], s_obj=res.obj, s_iters=res.iters, s_status=res.status, s_cviol=res.cviol, s_dual_inf=res.dual_inf)
    out.update(s_lam=u["lam"], s_mu=u["mu"], s_pl=u["pair_lam"], s_pm=u["pair_mu"], s_ps=u["pair_s"])
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    # constraint and bound multipliers in the oracle's own ordering (oracle/nlp.py): with the above the full primal-dual point, input
    # of the KKT certificate of the unmodified reference NLP (oracle/reference_nlp.py).  A file of their own keeps every fixture
    # under 1 MB (the 4-vehicle instance is 1.3 MB in one file).
    np.savez_compressed(os.path.join(HERE, name + "_multipliers.npz"), s_y=res.y, s_zL=res.zL, s_zU=res.zU)
    print(name, res.return_status, res.iters, res.obj, res.cviol)


def main():
    fn = os.path.join(tempfile.mkdtemp(), "4v")
    write_strategy(fn)
    tight = ipm.IpmOptions(tol=1e-8, constr_viol_tol=1e-8, max_iter=500)
    singles = {}
    for agent in ["vehicle_1", "vehicle_2"]:
        prob = build_problem(fn, [agent])
        guess = build_guess(prob, fn, [agent])
        nlp = CollocationNLP(prob)
        res = ipm.solve(nlp, nlp.init_slacks(nlp.pack(guess)), tight)
        singles[agent] = (prob, nlp, res)
        save("single_" + agent, prob, guess, nlp, res)
    # vehicle without a final heading (terminal psi row absent)
    prob = build_problem(fn, ["vehicle_2"], final_headings={"vehicle_2": None})
    guess = build_guess(prob, fn, ["vehicle_2"])
    nlp = CollocationNLP(prob)
    save("single_vehicle_2_free_heading", prob, guess, nlp, ipm.solve(nlp, nlp.init_slacks(nlp.pack(guess)), tight))
    # 2-vehicle joint problem warm-started from the single solutions (ragged horizons: N = 20 and 25)
    agents = ["vehicle_1", "vehicle_2"]
    prob = build_problem(fn, agents)
    V, O, Mmax = 2, prob.O, int(prob.nodes.max())
    z, lam, mu, dts = np.zeros((V, Mmax, 7)), np.zeros((V, Mmax, O, 4)), np.zeros((V, Mmax, O, 4)), []
    for ia, a in enumerate(agents):
        _, n1, r1 = singles[a]
        u = n1.unpack(r1.x)
        M = n1.M[0]
        z[ia, :M], lam[ia, :M], mu[ia, :M] = u["z"][0, :M], u["lam"][0, :M], u["mu"][0, :M]
        dts.append(u["dt"])
    m = int(prob.nodes.min())
    pl, pm, ps = np.zeros((1, Mmax, 4)), np.zeros((1, Mmax, 4)), np.zeros((1, Mmax, 2))
    pl[0, :m], pm[0, :m], ps[0, :m] = warmstart.joint_dual_ws_rect(z[0, :m, 0], z[0, :m, 1], z[0, :m, 2], z[1, :m, 0], z[1, :m, 1], z[1, :m, 2], prob.body_G, prob.body_g)
    guess = CollocationGuess(z, lam, mu, np.float64(np.mean(dts)), pl, pm, ps)
    nlp = CollocationNLP(prob)
    save("joint_vehicle_1_2", prob, guess, nlp, ipm.solve(nlp, nlp.init_slacks(nlp.pack(guess)), tight))
    four_vehicle_headline(fn, tight)


def four_vehicle_headline(fn, tight):
    """BASELINE.json configs[1] / the instance shape of configs[3]: 4-vehicle centralised conflict resolution with the
    initial offsets of multi_vehicle_planner.py:641-642 (vehicle_0: x + 0.1, psi + pi/20), n = 75 601.  The warm start is
    the one the bench pipeline produces (state_ws -> dual_ws -> single OBCA solves -> pair duals,
    control/batch_planner.py) -- run here under the developer host emulation of the kernels, since no GPU is available
    where fixtures are generated; the SOLUTION stored is the oracle's (sparse LU interior point, tol 1e-8) from that start."""
    from conflict_rez_b200 import solver as S
    from conflict_rez_b200.control.batch_planner import prepare_joint_batch
    from conflict_rez_b200.solver import SolveOptions

    emu = S.load_library(os.path.join(ROOT, "tools", "host_emu", "libobca_hostemu.so"))
    agents = ["vehicle_0", "vehicle_1", "vehicle_2", "vehicle_3"]
    heads = {"vehicle_0": 0.0, "vehicle_1": 3 * np.pi / 2, "vehicle_2": np.pi, "vehicle_3": np.pi / 2}   # multi_vehicle_planner.py:644-649
    offs = np.zeros((1, 4, 3))
    offs[0, 0] = [0.1, 0.0, np.pi / 20]
    plan = prepare_joint_batch(fn, agents, offs, SolveOptions(max_iter=600), device="cpu", lib=emu, final_headings=heads)
    plan.solver.close()
    print("warm start: single-vehicle status", [int(r.status[0]) for r in plan.singles], "iters", [int(r.iters[0]) for r in plan.singles])
    prob, guess = plan.problem.instance(0), plan.guess.instance(0)
    nlp = CollocationNLP(prob)
    res = ipm.solve(nlp, nlp.init_slacks(nlp.pack(guess)), tight)
    save("joint_vehicle_0_1_2_3", prob, guess, nlp, res)


if __name__ == "__main__":
    main()
