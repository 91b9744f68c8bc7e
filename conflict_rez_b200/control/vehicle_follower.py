"""``VehicleFollower`` / ``MultiDistributedFollower`` -- distributed MPC with the reference's method surface
(confrez/control/vehicle_follower.py:36-670).

Each vehicle plans a reference path (``plan_single_path``), builds its horizon-30 OBCA MPC once (``setup_controller``) and
then, every 0.1 s step, sets the parameters (current state, reference, neighbours' shifted predictions), warm-starts
from the previous solution shifted by one step and solves (``step``).  The NLP is solved by the CUDA kernel in MPC mode
(:class:`~conflict_rez_b200.solver.ObcaMpcSolver`); ``MultiDistributedFollower`` solves the independent per-vehicle NLPs
of one control step in **one batched launch** (the reference steps them sequentially, vehicle_follower.py:639-641; they
only depend on the Jacobi snapshot of the previous predictions, :636-637).

Differences from the reference: no pygame window (SURVEY.md App. B item 10); the plant is integrated with a fine fixed-step
RK4 (100 sub-steps, error < 1e-12) instead of IDAS (``dynamic_model.py:61-93``); a failed step records its measured time,
not the constant 0.5 s (``vehicle_follower.py:505``).
"""
import time
from typing import Dict, List, Tuple

import numpy as np

from conflict_rez_b200.control import warmstart
from conflict_rez_b200.control.vehicle import Vehicle
from conflict_rez_b200.obstacle_types import GeofenceRegion
from conflict_rez_b200.problem import CollocationGuess
from conflict_rez_b200.pytypes import VehiclePrediction, VehicleState
from conflict_rez_b200.solver import MpcProblem, ObcaMpcSolver, SolveOptions
from conflict_rez_b200.vehicle_types import VehicleBody, VehicleConfig

np.random.seed(0)  # vehicle_follower.py:29 (seeds the random initial obstacle duals of the first step)

# Warm-start constants of the MPC loops (warm_start=True), from the sweep of tools/gpu_mpc_warm_start.py on the 4-vehicle scene
# (profiles/r04_mpc_warm_start.json, DESIGN.md section 4): IPOPT's push of 1e-3 (pushes of 1e-6 / 1e-9 gave single steps of 97 - 572
# iterations), and mu starting at 1e-5, next to the final mu of a tol 1e-2 solve.  They act only on warm-started solves.
MPC_WARM_START_OPTIONS = dict(warm_start_bound_push=1e-3, warm_start_mult_bound_push=1e-3, warm_start_mu_init=1e-5)


def simulate_plant(state: np.ndarray, u: np.ndarray, dt: float, wb: float, substeps: int = 100) -> np.ndarray:
    """[x, y, psi, v, delta] after dt under constant input [a, w] (the reference integrates the same ODE with IDAS)."""
    z = np.array(state, dtype=float)
    h = dt / substeps

    def f(s):
        return np.array([s[3] * np.cos(s[2]), s[3] * np.sin(s[2]), s[3] / wb * np.tan(s[4]), u[0], u[1]])

    for _ in range(substeps):
        k1 = f(z)
        k2 = f(z + h / 2 * k1)
        k3 = f(z + h / 2 * k2)
        k4 = f(z + h * k3)
        z = z + h / 6 * (k1 + 2 * k2 + 2 * k3 + k4)
    return z


class VehicleFollower(Vehicle):
    def __init__(self, rl_file_name: str, agent: str, color: Dict[str, Tuple[float, float, float]], init_offset: VehicleState,
                 final_heading: float, vehicle_config: VehicleConfig = VehicleConfig(), vehicle_body: VehicleBody = VehicleBody(),
                 region: GeofenceRegion = GeofenceRegion(), printer: callable = None, device="cuda:0") -> None:
        super().__init__(rl_file_name, agent, color, vehicle_config, vehicle_body, region, device=device)
        self.init_offset, self.final_heading = init_offset, final_heading
        self.state: VehicleState = self.init_state
        self.state.t = 0
        self.pred: VehiclePrediction = None
        self.back_up_steps = 0
        self.others: List[str] = []
        self.others_pred: Dict[str, VehiclePrediction] = {}
        self.reference_traj: VehiclePrediction = None
        self.final_traj = VehiclePrediction()
        self.final_traj.t = [self.state.t]
        self.final_traj.x, self.final_traj.y, self.final_traj.psi = [self.state.x.x], [self.state.x.y], [self.state.e.psi]
        self.final_traj.v, self.final_traj.u_steer = [self.state.v.v], [self.state.u.u_steer]
        self.final_traj.u_a, self.final_traj.u_steer_dot = [self.state.u.u_a], [self.state.u.u_steer_dot]
        self.iter_time: List[float] = []
        self.print = print if printer is None else printer
        self.solver = None

    # ------------------------------------------------------------------ reference path (vehicle_follower.py:91-138)
    def plan_single_path(self, N_ws: int = 30, dt_ws: float = 0.1, K: int = 5, N_per_set: int = 5, shrink_tube: float = 0.5,
                         dmin: float = 0.05, spline_ws: bool = True, interp_dt: float = 0.01):
        zu0 = self.state_ws(N=N_ws, dt=dt_ws, init_offset=self.init_offset, final_heading=self.final_heading, shrink_tube=shrink_tube, spline_ws=spline_ws)
        zu0 = self.interp_ws_for_collocation(self.dual_ws(zu0), K=K, N_per_set=N_per_set)
        self.setup_single_final_problem(zu0=zu0, init_offset=self.init_offset, final_heading=self.final_heading, K=K, N_per_set=N_per_set,
                                        shrink_tube=shrink_tube, dmin=dmin)
        result = self.get_solution(self.solve_single_final_problem())
        interp_time = np.linspace(result.t[0], result.t[-1], num=int((result.t[-1] - result.t[0]) / interp_dt), endpoint=True)
        self.reference_traj = self.interpolate_states(interp_time)
        self.reference_xy = np.vstack([self.reference_traj.x, self.reference_traj.y]).T

    def get_others(self, vehicles: List[Vehicle]):
        self.others = [v.agent for v in vehicles if v.agent != self.agent]

    # ------------------------------------------------------------------ controller (vehicle_follower.py:146-368)
    def mpc_problem(self, dt: float = 0.1, N: int = 30, dmin=0.05, batch: int = 1) -> MpcProblem:
        vc, rg = self.vehicle_config, self.region
        A, b = self._obstacle_arrays()
        return MpcProblem(obs_A=A, obs_b=b, n_others=len(self.others), N=N, dt=dt, body_G=np.asarray(self.vehicle_body.A, float),
                          body_g=np.asarray(self.vehicle_body.b, float), wb=self.vehicle_body.wb,
                          region=np.array([rg.x_min, rg.x_max, rg.y_min, rg.y_max]),
                          limits=np.array([vc.v_min, vc.v_max, vc.delta_min, vc.delta_max, vc.a_min, vc.a_max, vc.w_delta_min, vc.w_delta_max], dtype=float),
                          dmin=dmin, batch=batch)

    def setup_controller(self, dt: float = 0.1, N: int = 30, dmin=0.05, solver: ObcaMpcSolver = None):
        """``solver`` may be a shared batched handle (MultiDistributedFollower); otherwise a private one is created."""
        self.N, self.dt = N, dt
        self.horizon_interp_ahead = np.linspace(0, N * dt, N, endpoint=False)
        self.opt_lambda_ij = {o: np.zeros((N, 4)) for o in self.others}
        self.opt_lambda_ji = {o: np.zeros((N, 4)) for o in self.others}
        self.opt_s = {o: np.zeros((N, 2)) for o in self.others}
        if solver is None:
            solver = ObcaMpcSolver(self.mpc_problem(dt, N, dmin), SolveOptions(max_iter=600), device=self.device, lib=getattr(self, "_lib", None))
        self.solver = solver

    def get_current_ref(self):
        min_idx = np.abs(self.reference_traj.t - self.state.t).argmin()
        interp_t_span = self.reference_traj.t[min_idx] + self.horizon_interp_ahead
        result = self.interpolate_states(time=interp_t_span)
        if self.pred is None:
            self.pred = result.copy()
            n_l = 4 * len(self.obstacles)
            self.pred.l = 0.1 * np.random.rand(self.N, n_l)  # vehicle_follower.py:401-402
            self.pred.m = 0.1 * np.random.rand(self.N, n_l)
        return result

    def get_others_pred(self, vehicles: List[Vehicle]):
        for v in vehicles:
            self.others_pred[v.agent] = v.pred.copy()

    @staticmethod
    def _adv_onestep(array: np.ndarray):
        array = np.asarray(array)
        if array.ndim == 1:
            return np.append(array[1:], array[-1])
        if array.ndim == 2:
            return np.vstack([array[1:, :], array[-1, :]])
        raise ValueError("unexpected shape when advancing the array to one step ahead.")

    # ------------------------------------------------------------------ one control step (vehicle_follower.py:428-563)
    def step_inputs(self):
        """Parameters and shifted warm start of this step (what ``opti.set_value`` / ``set_initial`` receive)."""
        cur = np.array([self.state.x.x, self.state.x.y, self.state.e.psi, self.state.v.v, self.state.u.u_steer])
        ref = self.get_current_ref()
        adv = self._adv_onestep
        others = np.stack([np.stack([adv(self.others_pred[o].x), adv(self.others_pred[o].y), adv(self.others_pred[o].psi)], axis=1) for o in self.others]) \
            if self.others else np.zeros((0, self.N, 3))
        z = np.stack([adv(getattr(self.pred, k)) for k in ("x", "y", "psi", "v", "u_steer", "u_a", "u_steer_dot")], axis=1)
        O = len(self.obstacles)
        guess = dict(z=z, lam=adv(self.pred.l).reshape(self.N, O, 4), mu=adv(self.pred.m).reshape(self.N, O, 4),
                     pl=np.stack([adv(self.opt_lambda_ij[o]) for o in self.others]) if self.others else np.zeros((0, self.N, 4)),
                     pm=np.stack([adv(self.opt_lambda_ji[o]) for o in self.others]) if self.others else np.zeros((0, self.N, 4)),
                     ps=np.stack([adv(self.opt_s[o]) for o in self.others]) if self.others else np.zeros((0, self.N, 2)))
        return cur, np.stack([ref.x, ref.y, ref.psi], axis=1), others, guess

    def apply_result(self, ok: bool, res, b: int, solve_time: float):
        """Store the new prediction (or shift the old one on failure), step the plant, log (vehicle_follower.py:478-563)."""
        self.iter_time.append(solve_time)
        adv = self._adv_onestep
        if ok:
            self.back_up_steps = self.N - 1
            z = res.z[b, 0]
            self.pred.x, self.pred.y, self.pred.psi, self.pred.v = z[:, 0].copy(), z[:, 1].copy(), z[:, 2].copy(), z[:, 3].copy()
            self.pred.u_steer, self.pred.u_a, self.pred.u_steer_dot = z[:, 4].copy(), z[:, 5].copy(), z[:, 6].copy()
            self.pred.l, self.pred.m = res.lam[b, 0].reshape(self.N, -1).copy(), res.mu[b, 0].reshape(self.N, -1).copy()
            for io, o in enumerate(self.others):
                self.opt_lambda_ij[o], self.opt_lambda_ji[o], self.opt_s[o] = res.pair_lam[b, io].copy(), res.pair_mu[b, io].copy(), res.pair_s[b, io].copy()
        else:
            self.back_up_steps -= 1
            for k in ("x", "y", "psi", "v", "u_steer", "u_a", "u_steer_dot", "l", "m"):
                setattr(self.pred, k, adv(getattr(self.pred, k)))
            for o in self.others:
                self.opt_lambda_ij[o], self.opt_lambda_ji[o], self.opt_s[o] = adv(self.opt_lambda_ij[o]), adv(self.opt_lambda_ji[o]), adv(self.opt_s[o])
        self.state.t += self.dt
        zint = simulate_plant([self.state.x.x, self.state.x.y, self.state.e.psi, self.state.v.v, self.state.u.u_steer],
                              [self.pred.u_a[0], self.pred.u_steer_dot[0]], self.dt, self.vehicle_body.wb)
        self.state.x.x, self.state.x.y, self.state.e.psi = float(zint[0]), float(zint[1]), float(zint[2])
        self.state.v.v, self.state.u.u_steer = float(zint[3]), float(zint[4])
        self.state.u.u_a, self.state.u.u_steer_dot = float(self.pred.u_a[0]), float(self.pred.u_steer_dot[0])
        ft = self.final_traj
        for lst, val in ((ft.t, self.state.t), (ft.x, self.state.x.x), (ft.y, self.state.x.y), (ft.psi, self.state.e.psi), (ft.v, self.state.v.v),
                         (ft.u_steer, self.state.u.u_steer), (ft.u_a, self.state.u.u_a), (ft.u_steer_dot, self.state.u.u_steer_dot)):
            lst.append(val)

    def step(self):
        cur, ref, others, g = self.step_inputs()
        guess = CollocationGuess(g["z"][None, None], g["lam"][None, None], g["mu"][None, None], np.zeros(1), g["pl"][None], g["pm"][None], g["ps"][None])
        t0 = time.perf_counter()
        res = self.solver.solve_step(cur[None], ref[None], others[None], guess)
        self.apply_result(bool(res.status[0] >= 0), res, 0, time.perf_counter() - t0)


class MultiDistributedFollower(object):
    def __init__(self, rl_file_name: str, spline_ws_config: Dict[str, bool], colors: Dict[str, Tuple[float, float, float]],
                 init_offsets: Dict[str, VehicleState], final_headings: Dict[str, float], device="cuda:0", lib=None) -> None:
        self.rl_file_name, self.spline_ws_config, self.colors = rl_file_name, spline_ws_config, colors
        self.init_offsets, self.final_headings, self.device, self._lib = init_offsets, final_headings, device, lib
        self.agents = sorted(self.spline_ws_config.keys())
        self.vehicles: List[VehicleFollower] = []
        for agent in self.agents:
            v = VehicleFollower(rl_file_name=rl_file_name, agent=agent, color=self.colors[agent], init_offset=self.init_offsets[agent],
                                final_heading=self.final_headings[agent], device=device)
            v._lib = lib
            self.vehicles.append(v)
        self.iter_time = {agent: [] for agent in self.agents}
        self.step_time: List[float] = []
        self.step_iters: List[int] = []
        self.failed_solves = 0  # solves whose status was not a success (the vehicle kept its shifted plan, vehicle_follower.py:501-524)
        self.failed_steps = 0   # control steps with at least one failed solve
        self.single_results: Dict[str, VehiclePrediction] = {}
        self.final_results: Dict[str, VehiclePrediction] = {}
        self.solver = None
        self.warm_start = False

    def setup_multi_vehicles(self, dt: float = 0.1, N: int = 30, dmin: float = 0.05, warm_start: bool = False):
        """``warm_start``: from the second control step on, a vehicle whose previous solve succeeded starts from that solve's
        primal-dual iterate shifted by one node (``ObcaSolver.shift_iterate`` / ``solve_warm``) instead of z = 1, y = 0, mu = 0.1."""
        self.warm_start = warm_start
        for v in self.vehicles:
            v.plan_single_path(spline_ws=self.spline_ws_config[v.agent])
            v.get_others(self.vehicles)
        # one batched handle: instance b = vehicle b (same obstacles, body, horizon; n_others = V - 1)
        self.solver = ObcaMpcSolver(self.vehicles[0].mpc_problem(dt, N, dmin, batch=len(self.vehicles)), SolveOptions(max_iter=600, **MPC_WARM_START_OPTIONS),
                                    device=self.device, lib=self._lib)
        for v in self.vehicles:
            v.setup_controller(dt=dt, N=N, dmin=dmin, solver=self.solver)
            v.get_current_ref()
            self.single_results[v.agent] = v.reference_traj

    def solve(self, num_iter: int = 500):
        sv, ok = self.solver, None
        for _ in range(num_iter):
            for v in self.vehicles:
                v.get_others_pred(self.vehicles)  # Jacobi snapshot (vehicle_follower.py:636-637)
            inputs = [v.step_inputs() for v in self.vehicles]
            cur = np.stack([i[0] for i in inputs])
            ref = np.stack([i[1] for i in inputs])
            others = np.stack([i[2] for i in inputs])
            st = lambda k: np.stack([i[3][k] for i in inputs])
            guess = CollocationGuess(st("z")[:, None], st("lam")[:, None], st("mu")[:, None], np.zeros(len(inputs)), st("pl"), st("pm"), st("ps"))
            t0 = time.perf_counter()
            if self.warm_start and ok is not None:
                # the stored iterates are last step's solutions: shift them, then write the guesses (the same user variables for the
                # vehicles that succeeded, the shifted backup plan for the others), and start only the former warm
                sv.set_params(sv.upload_params(cur, ref, others))
                sv.shift_iterate()
                sv.set_inputs(sv.upload(guess))
                res = sv.solve_warm(ok.astype(np.int32))
            else:
                res = sv.solve_step(cur, ref, others, guess)  # all vehicles of this control step in one launch
            ok = res.status >= 0
            dt_solve = time.perf_counter() - t0
            self.step_time.append(dt_solve)
            self.step_iters.append(int(np.max(res.iters)))
            nfail = int((res.status < 0).sum())
            self.failed_solves += nfail
            self.failed_steps += int(nfail > 0)
            for b, v in enumerate(self.vehicles):
                v.apply_result(bool(res.status[b] >= 0), res, b, dt_solve)
        for v in self.vehicles:
            self.iter_time[v.agent] = v.iter_time
            self.final_results[v.agent] = v.final_traj


class DeviceMpcLoop(object):
    """Device-resident closed loop of ``MultiDistributedFollower`` (SURVEY.md 8f rank 2): every quantity a control step touches
    lives in HBM and every operation of ``VehicleFollower.step`` (vehicle_follower.py:428-563) is a kernel on one stream --

        reference window  get_current_ref (:370-404)      obca_mpc_ref_times + obca_interpolate
        neighbours        get_others_pred / _adv_onestep  obca_shift_horizon of everybody's last prediction (Jacobi snapshot, :636-637)
        warm start        shifted previous solution       obca_shift_horizon
        solve             opti.solve()                    obca_set_mpc_params / obca_set_initial / obca_solve (all vehicles, one launch)
        fallback          except-branch (:501-524)        torch.where on the per-vehicle status: failed vehicles keep the shifted plan
        plant             simulator (dynamic_model.py)    obca_plant_step

    so a control step needs no host round trip: ``run(k)`` enqueues k steps and synchronises once; ``run(k, graph=True)`` captures one
    step in a CUDA graph and replays it.  Built from a ``MultiDistributedFollower`` after ``setup_multi_vehicles()`` so that both
    loops start from the same plans and the same (random) first-step duals; ``export()`` writes the state back."""

    def __init__(self, mdf: "MultiDistributedFollower", warm_start: bool = False):
        """``warm_start``: from the second step on, every vehicle whose previous solve succeeded starts from that solve's primal-dual
        iterate shifted by one node on the device (``obca_shift_iterate`` + ``obca_warm_start``), as in
        ``MultiDistributedFollower.setup_multi_vehicles(warm_start=True)``; a vehicle that failed starts cold from its shifted plan."""
        import torch

        from conflict_rez_b200.solver import TrajectoryOps

        self.torch, self.mdf, self.solver = torch, mdf, mdf.solver
        sv, vs = mdf.solver, mdf.vehicles
        self.dev = sv.device
        self.ops = TrajectoryOps(self.dev, lib=sv.lib)
        V, N, O = len(vs), vs[0].N, len(vs[0].obstacles)
        P = V - 1
        self.V, self.N, self.O, self.P, self.dt = V, N, O, P, vs[0].dt
        self.wb = vs[0].vehicle_body.wb
        f64 = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).to(self.dev)
        # reference plans: collocation solutions of plan_single_path (one per vehicle, own interval count and dt)
        n_ref = [v._interp["N"] for v in vs]
        Mmax = 6 * max(n_ref)
        zref = np.zeros((1, V, Mmax, 7))
        for a, v in enumerate(vs):
            I = v._interp
            M = 6 * I["N"]
            zref[0, a, :M, :5] = I["X"].reshape(M, 5)
            zref[0, a, :M, 5], zref[0, a, :M, 6] = I["u_a"], I["u_w"]
        self.n_ref = n_ref
        self.zref = f64(zref)
        self.dt_ref = f64([[v._interp["dt"] for v in vs]])
        self.grid = f64([[[v.reference_traj.t[0], v.reference_traj.t[-1], len(v.reference_traj.t)] for v in vs]])
        # loop state
        self.state = f64([[v.state.x.x, v.state.x.y, v.state.e.psi, v.state.v.v, v.state.u.u_steer] for v in vs])
        self.clock = f64([[v.state.t for v in vs]])
        self.pred_z = f64([np.stack([getattr(v.pred, k) for k in ("x", "y", "psi", "v", "u_steer", "u_a", "u_steer_dot")], axis=1) for v in vs])
        self.pred_lam = f64([np.asarray(v.pred.l).reshape(N, O, 4) for v in vs])
        self.pred_mu = f64([np.asarray(v.pred.m).reshape(N, O, 4) for v in vs])
        self.pl = f64([[v.opt_lambda_ij[o] for o in v.others] for v in vs]).reshape(V, P, N, 4)
        self.pm = f64([[v.opt_lambda_ji[o] for o in v.others] for v in vs]).reshape(V, P, N, 4)
        self.ps = f64([[v.opt_s[o] for o in v.others] for v in vs]).reshape(V, P, N, 2)
        agents = [v.agent for v in vs]
        self.other_idx = torch.as_tensor([[agents.index(o) for o in v.others] for v in vs], dtype=torch.long, device=self.dev).reshape(V, P)
        self.zero_dt = torch.zeros(V, dtype=torch.float64, device=self.dev)
        self.steps_done = 0
        self.fail_count = torch.zeros(V, dtype=torch.int64, device=self.dev)
        self.iters_log, self.status_log, self.traj_log = [], [], []
        self.warm_start = warm_start
        self.prev_ok = None  # (V,) int32 status >= 0 of the last solve, once there was one (warm_start only)

    def _step(self, log=True):
        torch, sv, ops = self.torch, self.solver, self.ops
        V, N = self.V, self.N
        # parameters: current state, reference window, neighbours' shifted predictions (Jacobi snapshot of the previous solutions)
        times = ops.mpc_ref_times(self.grid, self.clock, N, self.dt)
        ref = ops.interpolate(self.zref, self.dt_ref, self.n_ref, times)[0, :, :, :3].contiguous()
        sh_z = ops.shift_horizon(self.pred_z)
        others = sh_z[self.other_idx][:, :, :, :3].contiguous() if self.P else None
        d = {"z": sh_z.unsqueeze(1), "lam": ops.shift_horizon(self.pred_lam).unsqueeze(1), "mu": ops.shift_horizon(self.pred_mu).unsqueeze(1), "dt": self.zero_dt}
        if self.P:
            d["pl"] = ops.shift_horizon(self.pl.reshape(V * self.P, N, 4)).reshape(V, self.P, N, 4)
            d["pm"] = ops.shift_horizon(self.pm.reshape(V * self.P, N, 4)).reshape(V, self.P, N, 4)
            d["ps"] = ops.shift_horizon(self.ps.reshape(V * self.P, N, 2)).reshape(V, self.P, N, 2)
        warm = self.warm_start and self.prev_ok is not None
        if warm:
            sv.shift_iterate()  # before set_inputs, which writes the same user variables for the vehicles that start warm
        sv.set_params({"cur": self.state, "ref": ref, "others": others})
        sv.set_inputs({k: v.contiguous() for k, v in d.items()})
        if warm:
            sv.arm_warm_start(self.prev_ok)
        sv.run()
        st, it, _ = sv.fetch_stats()
        sol = sv.fetch_solution()
        ok = st >= 0
        pick = lambda new, old: torch.where(ok.view((V,) + (1,) * (old.dim() - 1)), new.reshape(old.shape), old)
        self.pred_z = pick(sol["z"], d["z"].squeeze(1))
        self.pred_lam = pick(sol["lam"], d["lam"].squeeze(1))
        self.pred_mu = pick(sol["mu"], d["mu"].squeeze(1))
        if self.P:
            self.pl, self.pm, self.ps = pick(sol["pl"], d["pl"]), pick(sol["pm"], d["pm"]), pick(sol["ps"], d["ps"])
        self.state = ops.plant_step(self.state, self.pred_z[:, 0, 5:7].contiguous(), self.dt, self.wb)
        self.clock = self.clock + self.dt
        self.fail_count += (~ok).to(torch.int64)
        if self.warm_start:
            self.prev_ok = ok.to(torch.int32)
        if log:
            self.iters_log.append(it)
            self.status_log.append(st)
            self.traj_log.append(torch.cat([self.state, self.pred_z[:, 0, 5:7]], dim=1))
        self.steps_done += 1

    def run(self, num_iter: int, graph: bool = False):
        """Enqueue ``num_iter`` control steps; one synchronisation at the end.  Returns the wall time per step in seconds."""
        torch = self.torch
        if graph and self.dev.type == "cuda":
            side = torch.cuda.Stream(self.dev)
            side.wait_stream(torch.cuda.current_stream(self.dev))
            with torch.cuda.stream(side):  # warm-up on a side stream (allocator), then capture one step
                self._step(log=False)
            torch.cuda.current_stream(self.dev).wait_stream(side)
            torch.cuda.synchronize(self.dev)
            names = ("state", "clock", "pred_z", "pred_lam", "pred_mu", "pl", "pm", "ps") + (("prev_ok",) if self.warm_start else ())
            static = {k: getattr(self, k).clone() for k in names}
            for k in names:
                setattr(self, k, static[k])
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._step(log=False)
                for k in names:  # write the new state back into the static tensors the graph reads on its next replay
                    static[k].copy_(getattr(self, k))
            for k in names:
                setattr(self, k, static[k])
            self.steps_done -= 1  # the capture pass itself does not execute
            torch.cuda.synchronize(self.dev)
            t0 = time.perf_counter()
            for _ in range(num_iter - 1):
                g.replay()
            torch.cuda.synchronize(self.dev)
            self.steps_done += num_iter - 1
            return (time.perf_counter() - t0) / max(1, num_iter - 1)
        if self.dev.type == "cuda":
            torch.cuda.synchronize(self.dev)
        t0 = time.perf_counter()
        for _ in range(num_iter):
            self._step()
        if self.dev.type == "cuda":
            torch.cuda.synchronize(self.dev)
        return (time.perf_counter() - t0) / max(1, num_iter)

    def export(self):
        """Host copies: states (V,5), clock (V), trajectory log (steps,V,7) = state + applied input, statuses, iterations."""
        cpu = lambda t: t.detach().cpu().numpy()
        out = {"state": cpu(self.state), "clock": cpu(self.clock)[0], "failed_solves": int(self.fail_count.sum().item())}
        if self.traj_log:
            out["traj"] = np.stack([cpu(t) for t in self.traj_log])
            out["status"] = np.stack([cpu(t) for t in self.status_log])
            out["iters"] = np.stack([cpu(t) for t in self.iters_log])
        return out


class _RemotePrediction(object):
    """The part of a neighbour's ``VehiclePrediction`` that the controllers read (x, y, psi over the horizon)."""

    def __init__(self, xyp: np.ndarray):
        self.x, self.y, self.psi = xyp[:, 0].copy(), xyp[:, 1].copy(), xyp[:, 2].copy()

    def copy(self):
        return _RemotePrediction(np.stack([self.x, self.y, self.psi], axis=1))


class DistributedFollowerNode(object):
    """One process per GPU (``torch.distributed``): the multi-process form of ``MultiDistributedFollower``.

    The reference runs one ROS node per vehicle and exchanges predictions on the ``/pred`` topic
    (ros2_ws/src/confrez_ros/confrez_ros/vehicle_node.py:80-189, launch/multi_follower.launch.py:37-52); in the
    single-process simulation the exchange is the Jacobi snapshot of vehicle_follower.py:636-637.  Here rank r owns the
    agents ``agents[r::world]`` and solves their MPC problems in one batched launch on its own GPU; the only
    communication is one all-gather per control step of every vehicle's predicted (x, y, psi)[N] -- 720 bytes per
    vehicle -- over NCCL (gloo on CPU).  Trajectories are identical to the single-process closed loop.
    """

    def __init__(self, rl_file_name: str, spline_ws_config: Dict[str, bool], colors: Dict[str, Tuple[float, float, float]],
                 init_offsets: Dict[str, VehicleState], final_headings: Dict[str, float], device="cuda:0", lib=None, group=None) -> None:
        import torch.distributed as dist

        self.dist, self.group = dist, group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.device, self._lib = device, lib
        self.agents = sorted(spline_ws_config.keys())
        if len(self.agents) % self.world:
            raise ValueError("the number of vehicles must be a multiple of the number of ranks")
        self.local_agents = self.agents[self.rank :: self.world]
        self.spline_ws_config = spline_ws_config
        self.vehicles: List[VehicleFollower] = []
        for agent in self.local_agents:
            v = VehicleFollower(rl_file_name=rl_file_name, agent=agent, color=colors[agent], init_offset=init_offsets[agent],
                                final_heading=final_headings[agent], device=device)
            v._lib = lib
            self.vehicles.append(v)
        self.step_time: List[float] = []
        self.exchange_time: List[float] = []
        self.final_results: Dict[str, VehiclePrediction] = {}
        self.solver = None

    def setup_multi_vehicles(self, dt: float = 0.1, N: int = 30, dmin: float = 0.05):
        for v in self.vehicles:
            v.plan_single_path(spline_ws=self.spline_ws_config[v.agent])
            v.others = [a for a in self.agents if a != v.agent]
        self.solver = ObcaMpcSolver(self.vehicles[0].mpc_problem(dt, N, dmin, batch=len(self.vehicles)), SolveOptions(max_iter=600),
                                    device=self.device, lib=self._lib)
        for v in self.vehicles:
            v.setup_controller(dt=dt, N=N, dmin=dmin, solver=self.solver)
            v.get_current_ref()
        self.N = N

    def exchange_predictions(self):
        """All-gather of the predicted poses: (n_local, N, 3) per rank -> every vehicle's ``others_pred``."""
        import torch

        dev = self.solver.device
        mine = torch.as_tensor(np.stack([np.stack([v.pred.x, v.pred.y, v.pred.psi], axis=1) for v in self.vehicles]), dtype=torch.float64).to(dev)
        parts = [torch.empty_like(mine) for _ in range(self.world)]
        self.dist.all_gather(parts, mine.contiguous(), group=self.group)
        full = torch.stack(parts).cpu().numpy()  # [rank][local index][N][3]; agent agents[r + k * world] is local index k of rank r
        for v in self.vehicles:
            for o in v.others:
                g = self.agents.index(o)
                v.others_pred[o] = _RemotePrediction(full[g % self.world, g // self.world])

    def solve(self, num_iter: int = 500):
        for _ in range(num_iter):
            t0 = time.perf_counter()
            self.exchange_predictions()
            t1 = time.perf_counter()
            inputs = [v.step_inputs() for v in self.vehicles]
            cur = np.stack([i[0] for i in inputs])
            ref = np.stack([i[1] for i in inputs])
            others = np.stack([i[2] for i in inputs])
            st = lambda k: np.stack([i[3][k] for i in inputs])
            guess = CollocationGuess(st("z")[:, None], st("lam")[:, None], st("mu")[:, None], np.zeros(len(inputs)), st("pl"), st("pm"), st("ps"))
            t2 = time.perf_counter()
            res = self.solver.solve_step(cur, ref, others, guess)
            dt_solve = time.perf_counter() - t2
            self.exchange_time.append(t1 - t0)
            self.step_time.append(dt_solve)
            for b, v in enumerate(self.vehicles):
                v.apply_result(bool(res.status[b] >= 0), res, b, dt_solve)
        for v in self.vehicles:
            self.final_results[v.agent] = v.final_traj
