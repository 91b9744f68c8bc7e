"""MPC mode (VehicleFollower.setup_controller / step, confrez/control/vehicle_follower.py:146-563): parity of the kernel
with the MPC oracle (oracle/mpc.py) through the C ABI, and the closed loop of the drop-in classes."""
import numpy as np
import pytest

from cases import body_corners, oracle_newton_step, quad_distance
from layout_map import DeviceLayout

from conflict_rez_b200.control import warmstart
from conflict_rez_b200.problem import CollocationGuess
from conflict_rez_b200.pytypes import VehicleState
from conflict_rez_b200.solver import MpcProblem, ObcaMpcSolver, SolveOptions

BACKENDS = [pytest.param("emu", id="emu"), pytest.param("cuda", id="cuda", marks=pytest.mark.gpu)]


@pytest.fixture(params=BACKENDS)
def backend(request):
    if request.param == "emu":
        return request.getfixturevalue("emu_lib"), "cpu"
    return request.getfixturevalue("cuda_lib"), "cuda:0"


@pytest.fixture(scope="module")
def mpc_case():
    """One MPC step of vehicle_1 with vehicle_2 as neighbour, references cut from the golden single-vehicle plans."""
    from cases import load_golden
    from conflict_rez_b200.control.vehicle import collocation_coefficients

    def resample(name, N=30, dt=0.1):
        prob, _, sol = load_golden(name)
        z, dtc = sol["z"][0], float(sol["dt"])
        M = int(prob.nodes[0])
        tau = warmstart.radau_nodes(5)
        t_nodes = (np.arange(M // 6)[:, None] + tau[None, :]).ravel() * dtc
        keep = np.concatenate([[True], np.diff(t_nodes) > 1e-12])
        tq = np.arange(N) * dt
        return np.stack([np.interp(tq, t_nodes[keep], z[:M][keep, c]) for c in range(7)], axis=1), prob

    z1, prob = resample("single_vehicle_1")
    z2, _ = resample("single_vehicle_2")
    p = dict(N=30, dt=0.1, wb=2.5, obs_A=prob.obs_A, obs_b=prob.obs_b, body_G=prob.body_G, body_g=prob.body_g, region=prob.region,
             limits=prob.limits, dmin=0.05, n_others=1)
    par = dict(cur=z1[0, :5].copy(), ref=z1[:, :3].copy(), others=z2[None, :, :3].copy())
    lam, mu = warmstart.dual_ws_rect(z1[:, 0], z1[:, 1], z1[:, 2], p["obs_A"], p["obs_b"], p["body_G"], p["body_g"])
    pl, pm, ps = warmstart.joint_dual_ws_rect(z1[:, 0], z1[:, 1], z1[:, 2], z2[:, 0], z2[:, 1], z2[:, 2], p["body_G"], p["body_g"])
    return p, par, dict(z=z1, lam=lam, mu=mu, pl=pl[None], pm=pm[None], ps=ps[None])


def _maps(L, nlp):
    D = DeviceLayout(L)
    N, O, Vo = nlp.N, nlp.O, nlp.Vo
    ix, iy, n = np.full(nlp.n, -1), np.full(nlp.m, -1), np.arange(N)
    for c in range(7):
        ix[nlp.iz[:, c]] = D.Z(0, c, n)
    for j in range(O):
        for r in range(4):
            ix[nlp.ilam[:, j, r]], ix[nlp.imu[:, j, r]], iy[nlp.r_obs[0][:, j, r]] = D.LAM(0, j, r, n), D.MU(0, j, r, n), D.YOBS(0, j, r, n)
        ix[nlp.isd[:, j]], ix[nlp.iel[:, j]] = D.SD(0, j, n), D.EL(0, j, n)
    for o in range(Vo):
        for r in range(4):
            ix[nlp.ipl[o][:, r]], ix[nlp.ipm[o][:, r]] = D.PAIR("oPL", 4, o, r, n), D.PAIR("oPM", 4, o, r, n)
        for r in range(2):
            ix[nlp.ips[o][:, r]] = D.PAIR("oPS", 2, o, r, n)
        ix[nlp.ipsd[o]], ix[nlp.ipsn[o]], ix[nlp.ipel[o]] = D.PAIR("oPSD", 1, o, 0, n), D.PAIR("oPSN", 1, o, 0, n), D.PAIR("oPEL", 1, o, 0, n)
        for r in range(6):
            iy[nlp.r_pair[o][:, r]] = D.YPAIR(o, r, n)
    for c in range(5):
        iy[nlp.r_init[c]] = L["oYINIT"] + c
        iy[nlp.r_dyn[:, c]] = D.YCOL(0, c, np.arange(N - 1))
    assert (ix >= 0).all() and (iy >= 0).all()
    return ix, iy


def _solver(backend, p, **opts):
    lib, dev = backend
    mp = MpcProblem(obs_A=p["obs_A"], obs_b=p["obs_b"], n_others=p["n_others"], N=p["N"], dt=p["dt"])
    return ObcaMpcSolver(mp, SolveOptions(**opts), device=dev, lib=lib)


def _guess(g):
    return CollocationGuess(g["z"][None, None], g["lam"][None, None], g["mu"][None, None], np.zeros(1), g["pl"][None], g["pm"][None], g["ps"][None])


def test_rk4_dynamics_match_reference_definition():
    """oracle RK4 x 4 (chain-rule Jacobian) against the plain restatement of dynamic_model.py:30-58 and finite differences."""
    from oracle.collocation import f_rk4
    from oracle.mpc import rk4

    rng = np.random.default_rng(0)
    z, u = rng.uniform(-1, 1, (5, 4)), rng.uniform(-1, 1, (2, 4))
    F, J = rk4(z, u, 0.1, 2.5)
    for k in range(4):
        assert np.allclose(F[:, k], f_rk4(z[:, k], u[:, k], 0.1), atol=1e-14)
        for q in range(7):
            d = np.zeros(7)
            d[q] = 1e-6
            fd = (f_rk4(z[:, k] + d[:5], u[:, k] + d[5:], 0.1) - f_rk4(z[:, k] - d[:5], u[:, k] - d[5:], 0.1)) / 2e-6
            assert np.allclose(J[:, q, k], fd, atol=1e-8)


def test_mpc_residuals_step_and_solution_match_oracle(backend, mpc_case):
    from oracle import ipm
    from oracle.mpc import MpcNLP

    p, par, g = mpc_case
    nlp = MpcNLP(p, par)
    sv = _solver(backend, p, max_iter=0)
    sv.set_params(sv.upload_params(par["cur"][None], par["ref"][None], par["others"][None]))
    sv.solve(_guess(g))
    L = sv.layout()
    assert L["m_active"] == nlp.m
    ix, iy = _maps(L, nlp)
    xd, _, zLd, zUd = sv.debug_get_iterate(0)
    x0 = ipm.push_into_bounds(nlp.init_slacks(nlp.pack(g["z"], g["lam"], g["mu"], g["pl"], g["pm"], g["ps"])), nlp.xL, nlp.xU, 1e-2, 1e-2)
    assert np.allclose(xd[ix], x0, rtol=0, atol=1e-11)
    y = 0.3 * np.random.default_rng(5).standard_normal(nlp.m)
    yd = np.zeros(L["ny"])
    yd[iy] = y
    sv.debug_set_iterate(0, y=yd)
    c_d, gl_d, f_d = sv.debug_eval(0)
    dx_o, dy_o, c_o, gl_o, res_o = oracle_newton_step(nlp, x0, y, zLd[ix], zUd[ix], 0.1, 1e-3)
    assert max(res_o[1:]) <= 1e-10  # the reference step solves its system
    assert abs(f_d - nlp.f(x0)) <= 1e-11 * abs(f_d)
    assert np.abs(c_d[iy] - c_o).max() <= 1e-10 and np.abs(gl_d[ix] - gl_o).max() <= 1e-9 * np.abs(gl_o).max()
    dx_d, dy_d, ok = sv.debug_step(0, 0.1, 1e-3)
    assert ok == 1
    assert np.abs(dx_d[ix] - dx_o).max() <= 1e-8 * np.abs(dx_o).max() and np.abs(dy_d[iy] - dy_o).max() <= 1e-8 * np.abs(dy_o).max()
    sv.close()
    for tol in (1e-2, 1e-8):  # the reference's tolerance (vehicle_follower.py:362-363) and a tight one
        sv = _solver(backend, p, tol=tol, constr_viol_tol=tol, max_iter=600)
        res = sv.solve_step(par["cur"][None], par["ref"][None], par["others"][None], _guess(g))
        ref = ipm.solve(nlp, nlp.init_slacks(nlp.pack(g["z"], g["lam"], g["mu"], g["pl"], g["pm"], g["ps"])), ipm.IpmOptions(tol=tol, constr_viol_tol=tol, max_iter=600))
        assert res.status[0] == 0 and ref.status == 0
        assert abs(res.obj[0] - ref.obj) <= 1e-6 * abs(ref.obj)
        assert np.abs(res.z[0, 0] - ref.x[nlp.iz]).max() <= 1e-4
        assert abs(int(res.iters[0]) - ref.iters) <= 3
        sv.close()


def test_distributed_mpc_closed_loop(backend, strategy_file):
    """Two followers, 25 control steps, all vehicles of a step solved in one batched launch: every solve succeeds, the
    plants track their references, the predictions stay collision free."""
    from conflict_rez_b200.control.vehicle_follower import MultiDistributedFollower

    lib, dev = backend
    agents = ["vehicle_1", "vehicle_2"]
    heads = {"vehicle_1": 3 * np.pi / 2, "vehicle_2": np.pi}
    mdf = MultiDistributedFollower(strategy_file, {a: True for a in agents}, {a: {} for a in agents}, {a: VehicleState() for a in agents}, heads, device=dev, lib=lib)
    mdf.setup_multi_vehicles()
    mdf.solve(num_iter=25)
    devs = []
    for v in mdf.vehicles:
        assert len(v.final_traj.x) == 26 and len(v.iter_time) == 25
        t = np.array(v.final_traj.t)
        ref_x = np.interp(t, v.reference_traj.t, v.reference_traj.x)
        ref_y = np.interp(t, v.reference_traj.t, v.reference_traj.y)
        devs.append(np.hypot(np.array(v.final_traj.x) - ref_x, np.array(v.final_traj.y) - ref_y).max())
        assert v.back_up_steps == v.N - 1  # the last step was a successful solve
    # the two single-vehicle references conflict: one vehicle keeps its path, the other yields (but stays close)
    assert min(devs) < 0.1 and max(devs) < 0.8
    a, b = mdf.vehicles
    ca = body_corners(np.array(a.final_traj.x), np.array(a.final_traj.y), np.array(a.final_traj.psi), None, np.array([3.3, 0.9, 0.6, 0.9]))
    cb = body_corners(np.array(b.final_traj.x), np.array(b.final_traj.y), np.array(b.final_traj.psi), None, np.array([3.3, 0.9, 0.6, 0.9]))
    assert quad_distance(ca, cb).min() >= 0.05 - 1e-2
    if dev != "cpu":
        assert mdf.solver.launch_count > 0  # the CUDA kernels ran (the emulation does not count launches)


def test_infeasible_neighbour_is_reported_not_adopted(backend, mpc_case):
    """A neighbour predicted on top of the ego vehicle makes the reference problem infeasible (the distance row cannot reach
    dmin).  IPOPT reports Infeasible_Problem_Detected, Opti raises and VehicleFollower.step keeps the shifted backup plan
    (vehicle_follower.py:478-524).  The elastic formulation must not hide this: the status is negative, the elastic magnitude is
    visible in cviol / elastic, and the planner does not adopt the penetrating plan."""
    p, par, g = mpc_case
    sv = _solver(backend, p, max_iter=600)
    others = par["ref"][None].copy()  # the neighbour sits exactly where the ego reference is
    res = sv.solve_step(par["cur"][None], par["ref"][None], others[None], _guess(g))
    assert res.status[0] < 0, res.return_status(0)
    assert res.return_status(0) in ("Infeasible_Problem_Detected", "Maximum_Iterations_Exceeded", "Restoration_Failed")
    if res.status[0] == -6:
        assert res.elastic[0] > 1e-2 and res.cviol[0] >= res.elastic[0]
    sv.close()


def test_device_resident_loop_reproduces_the_host_loop(backend, strategy_file):
    """DeviceMpcLoop (reference window, neighbour shift, warm-start shift, solve, fallback, plant step all as kernels on one
    stream) follows the same closed-loop trajectories as MultiDistributedFollower.solve, which does those steps in numpy."""
    from conflict_rez_b200.control.vehicle_follower import DeviceMpcLoop, MultiDistributedFollower

    lib, dev = backend
    agents = ["vehicle_1", "vehicle_2"]
    heads = {"vehicle_1": 3 * np.pi / 2, "vehicle_2": np.pi}

    def make():
        np.random.seed(0)  # the first-step duals are 0.1 * rand (vehicle_follower.py:401-402)
        m = MultiDistributedFollower(strategy_file, {a: True for a in agents}, {a: {} for a in agents}, {a: VehicleState() for a in agents}, heads, device=dev, lib=lib)
        m.setup_multi_vehicles()
        return m

    steps = 6
    host = make()
    host.solve(num_iter=steps)
    loop = DeviceMpcLoop(make())
    loop.run(steps)
    out = loop.export()
    assert out["traj"].shape == (steps, 2, 7) and (out["status"] >= 0).all()
    for b, v in enumerate(host.vehicles):
        ft = v.final_traj
        ref = np.stack([ft.x[1:], ft.y[1:], ft.psi[1:], ft.v[1:], ft.u_steer[1:], ft.u_a[1:], ft.u_steer_dot[1:]], axis=1)
        assert np.abs(out["traj"][:, b] - ref).max() <= 1e-8
        assert abs(out["clock"][b] - v.state.t) <= 1e-12
    assert out["failed_solves"] == host.failed_solves
    if dev != "cpu":  # the same loop replayed from a CUDA graph: no host work between the steps
        g = DeviceMpcLoop(make())
        per_step = g.run(steps, graph=True)
        assert per_step > 0
        assert np.abs(g.export()["state"] - out["state"]).max() <= 1e-8


def test_inexact_penalty_is_escalated_and_carried_over(backend, strategy_file):
    """4-vehicle scene (the bench's MPC leg).  vehicle_1's plan passes an obstacle corner so closely that the minimiser of the
    penalised problem (rho = 1e3 against a tracking cost of 100 per m^2 and node) cuts the corner by 7 cm with the *separating*
    duals -- the l1 penalty is not exact there.  The solver must raise the weight and return a feasible plan (round 2: it returned
    Infeasible_Problem_Detected for the first 31 control steps), and the raised weight must carry over to the next control step of
    that vehicle (second step without a second attempt: far fewer iterations than the first)."""
    from conflict_rez_b200.control.vehicle_follower import MultiDistributedFollower

    lib, dev = backend
    agents = ["vehicle_0", "vehicle_1", "vehicle_2", "vehicle_3"]
    heads = {"vehicle_0": 0.0, "vehicle_1": 3 * np.pi / 2, "vehicle_2": np.pi, "vehicle_3": np.pi / 2}
    np.random.seed(0)
    mdf = MultiDistributedFollower(strategy_file, {a: True for a in agents}, {a: {} for a in agents}, {a: VehicleState() for a in agents}, heads, device=dev, lib=lib)
    mdf.setup_multi_vehicles()
    log = []
    orig = mdf.solver.solve_step

    def spy(*a, **k):
        r = orig(*a, **k)
        log.append((r.status.copy(), r.iters.copy(), r.elastic.copy()))
        return r

    mdf.solver.solve_step = spy
    mdf.solve(num_iter=3)
    for st, it, el in log:
        assert (st == 0).all(), st
        assert el.max() <= 1e-2
    assert log[1][1][1] < log[0][1][1] // 2, (log[0][1], log[1][1])
    assert mdf.failed_solves == 0
