"""Warm start from the stored primal-dual iterate (obca_get_iterate / obca_set_iterate / obca_shift_iterate / obca_warm_start,
ObcaSolver.fetch_iterate / put_iterate / shift_iterate / arm_warm_start / solve_warm, DeviceMpcLoop(warm_start=True)): unarmed
solves are unchanged bit for bit, the iterate round-trips, the MPC shift moves every node field, a restart at a solution stops at
once, loose -> tight reaches the golden solution, the first iterations match the oracle's warm start, and the closed MPC loop
needs fewer iterations warm than cold."""
import numpy as np
import pytest
import torch

from cases import body_corners, check_solution_properties, load_golden, quad_distance
from layout_map import DeviceLayout, build_maps
from test_history import F, _assert_same_results, _compare_with_oracle
from test_history import joint_case  # noqa: F401  (module fixture)
from test_mpc import _guess as _mpc_guess
from test_mpc import _maps
from test_mpc import mpc_case  # noqa: F401  (module fixture)
from test_refine_and_certificate import _assert_kkt_point, _certificate
from warm_oracle import solve_warm

from conflict_rez_b200.pytypes import VehicleState
from conflict_rez_b200.solver import HIST_F_WARM, MpcProblem, ObcaMpcSolver, ObcaSolver, ObcaStateWsSolver, SolveOptions, format_history
from oracle import ipm

BACKENDS = [pytest.param("emu", id="emu"), pytest.param("cuda", id="cuda", marks=pytest.mark.gpu)]


@pytest.fixture(params=BACKENDS)
def backend(request):
    if request.param == "emu":
        return request.getfixturevalue("emu_lib"), "cpu"
    return request.getfixturevalue("cuda_lib"), "cuda:0"


def _mpc_solver(backend, p, batch=1, **opts):
    lib, dev = backend
    mp = MpcProblem(obs_A=p["obs_A"], obs_b=p["obs_b"], n_others=p["n_others"], N=p["N"], dt=p["dt"], batch=batch)
    return ObcaMpcSolver(mp, SolveOptions(**opts), device=dev, lib=lib)


def test_unarmed_and_masked_solves_are_unchanged(backend, joint_case):  # noqa: F811
    lib, dev = backend
    prob, guess = joint_case
    assert prob.batch == 4
    cold = ObcaSolver(prob, SolveOptions(), device=dev, lib=lib).solve(guess)
    sv = ObcaSolver(prob, SolveOptions(), device=dev, lib=lib)
    sv.arm_warm_start(np.zeros(4, np.int32))  # armed with an all-zero mask
    _assert_same_results(cold, sv.solve(guess))
    _assert_same_results(cold, sv.solve(guess))  # not armed, after solves that left their iterates behind
    sv.arm_warm_start(np.array([1, 0, 1, 0], np.int32))  # instances 0 and 2 start from the guess with the stored multipliers
    mixed = sv.solve(guess)
    for k in ("status", "iters", "obj", "z", "lam", "mu", "dt", "pair_lam", "pair_mu", "pair_s"):
        assert np.array_equal(getattr(mixed, k)[[1, 3]], getattr(cold, k)[[1, 3]]), k
    assert (mixed.status == 0).all()
    _assert_same_results(cold, sv.solve(guess))  # the arm was consumed
    sv.close()


def test_iterate_round_trip_and_errors(backend, joint_case, mpc_case, strategy_file):  # noqa: F811
    from test_state_ws import _case as _ws_case

    lib, dev = backend
    prob, guess = joint_case
    sv = ObcaSolver(prob, SolveOptions(), device=dev, lib=lib)
    res = sv.solve(guess)
    d = sv.fetch_iterate()
    L = sv.layout()
    assert tuple(d["x"].shape) == (4, L["nx"]) and tuple(d["zL"].shape) == (4, L["nx"]) and tuple(d["zU"].shape) == (4, L["nx"])
    assert tuple(d["y"].shape) == (4, L["ny"]) and tuple(d["mu"].shape) == (4,)
    host = {k: v.cpu().numpy() for k, v in d.items()}
    assert np.array_equal(host["x"][1], sv.debug_get_iterate(1)[0])
    assert np.array_equal(host["x"][:, L["oDT"]], res.dt) and (host["mu"] > 0).all()
    other = ObcaSolver(prob, SolveOptions(), device=dev, lib=lib)
    other.put_iterate(d)
    back = {k: v.cpu().numpy() for k, v in other.fetch_iterate().items()}
    for k in ("x", "y", "zL", "zU"):
        assert np.array_equal(back[k], host[k]), k
    other.put_iterate({"y": d["y"] * 0})  # a missing part of the iterate is kept
    part = {k: v.cpu().numpy() for k, v in other.fetch_iterate().items()}
    assert (part["y"] == 0).all() and np.array_equal(part["x"], host["x"])
    with pytest.raises(ValueError, match="shape"):
        other.put_iterate({"x": d["x"][:2]})
    for name, args in (("obca_get_iterate", [None] * 6), ("obca_set_iterate", [None] * 5), ("obca_shift_iterate", [None]), ("obca_warm_start", [None] * 3)):
        assert getattr(lib, name)(None, *args) < 0
        assert b"null handle" in lib.obca_last_error(), name
    with pytest.raises(RuntimeError, match="MPC mode only"):
        sv.shift_iterate()
    p, cur, z0, _ = _ws_case(strategy_file, "vehicle_1")
    ws = ObcaStateWsSolver(p, SolveOptions(max_iter=500), device=dev, lib=lib)
    with pytest.raises(RuntimeError, match="MPC mode only"):
        ws.shift_iterate()
    for s in (sv, other, ws):
        s.close()


def test_shift_moves_every_node_field(backend, mpc_case):  # noqa: F811
    p, par, g = mpc_case
    sv = _mpc_solver(backend, p, batch=2)
    L = sv.layout()
    D = DeviceLayout(L)
    N, B = L["Mv"], 2
    rng = np.random.default_rng(3)
    it = {k: rng.standard_normal((B, L["nx"] if k != "y" else L["ny"])) for k in ("x", "zL", "zU", "y")}
    dev = sv.device
    sv.put_iterate({k: torch.as_tensor(v, device=dev) for k, v in it.items()})
    sv.shift_iterate()
    got = {k: v.cpu().numpy() for k, v in sv.fetch_iterate().items()}
    held = lambda rows, nv: np.concatenate([rows[..., 1:nv], rows[..., nv - 1:nv], rows[..., nv:]], axis=-1)
    for k in ("x", "zL", "zU"):
        want = it[k].copy()
        rows = want[:, : L["oDT"]].reshape(B, -1, N)  # every primal field but dt is node-minor (no tube slacks in MPC mode)
        want[:, : L["oDT"]] = held(rows, N).reshape(B, -1)
        assert np.array_equal(got[k], want), k
    want = it["y"].copy()
    col = slice(L["oYCOL"], L["oYCOL"] + 5 * N)
    want[:, col] = held(want[:, col].reshape(B, 5, N), N - 1).reshape(B, -1)  # node N - 1 of the dynamics rows is padding: untouched
    rest = slice(L["oYOBS"], L["ny"])
    want[:, rest] = held(want[:, rest].reshape(B, -1, N), N).reshape(B, -1)
    assert np.array_equal(got["y"], want)
    # spot checks through the named layout
    assert got["x"][1, D.Z(0, 0, 3)] == it["x"][1, D.Z(0, 0, 4)] and got["x"][1, D.Z(0, 0, N - 1)] == it["x"][1, D.Z(0, 0, N - 1)]
    assert got["y"][0, D.YCOL(0, 2, N - 2)] == it["y"][0, D.YCOL(0, 2, N - 2)] and got["y"][0, D.YCOL(0, 2, N - 1)] == it["y"][0, D.YCOL(0, 2, N - 1)]
    for fixed in (slice(L["oYINIT"], L["oYCOL"]), slice(L["oYCONT"], L["oYOBS"])):
        assert np.array_equal(got["y"][:, fixed], it["y"][:, fixed])
    assert np.array_equal(got["x"][:, L["oDT"]], it["x"][:, L["oDT"]])
    sv.close()


def test_restart_at_a_solution_stops_at_once(backend):
    lib, dev = backend
    prob, guess, _ = load_golden("joint_vehicle_1_2")
    tight = dict(tol=1e-8, constr_viol_tol=1e-8, max_iter=500)
    sv = ObcaSolver(prob, SolveOptions(**tight), device=dev, lib=lib)
    cold = sv.solve(guess)
    assert cold.status[0] == 0
    d = sv.fetch_iterate()
    # pushes of 1e-12: IPOPT's default 1e-3 would move the active bounds (gaps ~ mu / z ~ 1e-9) away from the solution
    w = ObcaSolver(prob, SolveOptions(**tight, history=8, warm_start_bound_push=1e-12, warm_start_mult_bound_push=1e-12), device=dev, lib=lib)
    w.set_inputs(w.upload(guess))  # the initial poses; x is replaced next
    w.put_iterate(d)
    res = w.solve_warm(mu0=d["mu"])
    print(format_history(res, 0))
    assert res.status[0] == 0, res.return_status(0)
    assert res.iters[0] <= 2, res.iters[0]
    assert np.abs(res.z - cold.z).max() <= 1e-8
    row = res.history[0, 0]
    assert row[F["mu"]] == float(d["mu"][0]) and int(row[F["flags"]]) & HIST_F_WARM
    assert "w" in format_history(res, 0).splitlines()[1].split()[-1]
    sv.close(), w.close()


def test_loose_then_tight_reaches_the_golden_solution(backend):
    from oracle.nlp import CollocationNLP

    lib, dev = backend
    prob, guess, gold = load_golden("joint_vehicle_1_2")
    loose = ObcaSolver(prob, SolveOptions(tol=1e-2, constr_viol_tol=1e-2), device=dev, lib=lib)
    r0 = loose.solve(guess)
    assert r0.status[0] == 0
    tight = ObcaSolver(prob, SolveOptions(tol=1e-8, constr_viol_tol=1e-8, max_iter=500), device=dev, lib=lib)
    tight.set_inputs(tight.upload(guess))
    tight.put_iterate(loose.fetch_iterate())
    res = tight.solve_warm()
    print("loose %d + warm tight %d iterations" % (r0.iters[0], res.iters[0]))
    assert res.status[0] == 0, res.return_status(0)
    # the tolerances of test_parity.test_solution_matches_golden
    assert abs(res.obj[0] - gold["obj"]) <= 1e-6 * abs(gold["obj"])
    assert res.cviol[0] <= 1e-6
    assert np.abs(res.z[0] - gold["z"]).max() <= 1e-4
    assert abs(res.dt[0] - gold["dt"]) <= 1e-6
    worst = check_solution_properties(prob, res.z, res.dt, tol=1e-6)
    assert worst["collocation"] <= 1e-6 and worst["continuity"] <= 1e-6 and worst["init"] <= 1e-6 and worst["terminal"] <= 1e-6
    assert worst["tube"] <= 1e-6 and worst["bounds"] <= 1e-9
    assert worst["obstacle_clearance"] >= prob.dmin - 1e-5 and worst["vehicle_clearance"] >= prob.dmin - 1e-5
    # the certificate of the unmodified reference NLP, as test_refine_and_certificate applies it to a solver point
    nlp = CollocationNLP(prob)
    ix, iy = build_maps(tight.layout(), nlp)
    xd, yd, zLd, zUd = tight.debug_get_iterate(0)
    cert = _certificate(prob, nlp, xd[ix], yd[iy], zLd[ix], zUd[ix])
    L = tight.layout()
    s_d = max(100.0, (np.abs(yd).sum() + zLd.sum() + zUd.sum()) / (L["m_active"] + L["nb"])) / 100.0
    _assert_kkt_point(cert, tol=1e-8, s_d=s_d)
    loose.close(), tight.close()


def test_warm_mpc_step_matches_oracle_history(backend, mpc_case):  # noqa: F811
    from oracle.mpc import MpcNLP

    p, par, g = mpc_case
    opts = dict(tol=1e-8, constr_viol_tol=1e-8, max_iter=600)
    sv = _mpc_solver(backend, p, history=64, **opts)
    first = sv.solve_step(par["cur"][None], par["ref"][None], par["others"][None], _mpc_guess(g))
    assert first.status[0] == 0
    it = {k: v.cpu().numpy()[0] for k, v in sv.fetch_iterate().items()}
    cur = par["cur"].copy()
    cur[:2] += 0.3 * p["dt"] * cur[3] * np.array([np.cos(cur[2]), np.sin(cur[2])])  # a third of a step along the heading
    cur[3] += 0.05
    sv.set_params(sv.upload_params(cur[None], par["ref"][None], par["others"][None]))
    res = sv.solve_warm()
    assert res.status[0] == 0, res.return_status(0)
    assert int(res.history[0, 0, F["flags"]]) & HIST_F_WARM
    assert res.history[0, 0, F["mu"]] == 1e-3  # warm_start_mu_init
    nlp = MpcNLP(p, dict(par, cur=cur))
    ix, iy = _maps(sv.layout(), nlp)
    ref = solve_warm(nlp, nlp.init_slacks(it["x"][ix]), it["y"][iy], it["zL"][ix], it["zU"][ix], opts=ipm.IpmOptions(**opts))  # the library's constants
    assert ref.status == 0
    _compare_with_oracle(res.history[0], ref.history)
    sv.close()


def _follower(strategy_file, lib, dev, warm_start):
    from conflict_rez_b200.control.vehicle_follower import MultiDistributedFollower

    agents = ["vehicle_1", "vehicle_2"]
    heads = {"vehicle_1": 3 * np.pi / 2, "vehicle_2": np.pi}
    np.random.seed(0)  # the first-step duals are 0.1 * rand (vehicle_follower.py:401-402)
    m = MultiDistributedFollower(strategy_file, {a: True for a in agents}, {a: {} for a in agents}, {a: VehicleState() for a in agents}, heads, device=dev, lib=lib)
    m.setup_multi_vehicles(warm_start=warm_start)
    return m


def test_warm_closed_loop(backend, strategy_file):
    from conflict_rez_b200.control.vehicle_follower import DeviceMpcLoop

    lib, dev = backend
    steps = 25
    cold = DeviceMpcLoop(_follower(strategy_file, lib, dev, False))
    cold.run(steps)
    warm = DeviceMpcLoop(_follower(strategy_file, lib, dev, True), warm_start=True)
    warm.run(steps)
    oc, ow = cold.export(), warm.export()
    assert (ow["status"] >= 0).all() and ow["failed_solves"] == 0
    # the plans stay collision free (as in test_mpc.test_distributed_mpc_closed_loop)
    tr = ow["traj"]
    ca, cb = (body_corners(tr[:, b, 0], tr[:, b, 1], tr[:, b, 2], None, np.array([3.3, 0.9, 0.6, 0.9])) for b in range(2))
    assert quad_distance(ca, cb).min() >= 0.05 - 1e-2
    it_cold, it_warm = int(oc["iters"][1:].sum()), int(ow["iters"][1:].sum())
    print("iterations over steps 2-%d: cold %d, warm %d" % (steps, it_cold, it_warm))
    assert np.array_equal(ow["iters"][0], oc["iters"][0])  # the first step is cold in both
    assert it_warm < it_cold
    # the host loop with warm_start=True follows the same trajectories.  On the GPU the MPC-mode sums are not bit-deterministic (see
    # test_history._assert_close_results) and the closed loop carries their last bits on: 1e-8 over the 6 steps of
    # test_mpc.test_device_resident_loop_reproduces_the_host_loop, 1e-6 over all 25; the emulation is deterministic, 1e-8 throughout
    host = _follower(strategy_file, lib, dev, True)
    host.solve(num_iter=steps)
    for b, v in enumerate(host.vehicles):
        ft = v.final_traj
        ref = np.stack([ft.x[1:], ft.y[1:], ft.psi[1:], ft.v[1:], ft.u_steer[1:], ft.u_a[1:], ft.u_steer_dot[1:]], axis=1)
        err = np.abs(tr[:, b] - ref).max(axis=1)
        assert err[:6].max() <= 1e-8 and err.max() <= (1e-8 if dev == "cpu" else 1e-6), err
    assert host.failed_solves == 0
    if dev != "cpu":  # replayed from a CUDA graph: the shift and the arm are captured with the step
        g = DeviceMpcLoop(_follower(strategy_file, lib, dev, True), warm_start=True)
        assert g.run(steps, graph=True) > 0
        assert np.abs(g.export()["state"] - ow["state"]).max() <= 1e-8
