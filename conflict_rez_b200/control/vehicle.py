"""``Vehicle`` -- single-vehicle planner with the reference's method surface (confrez/control/vehicle.py:24-829).

Same constructor, method names, keyword arguments and defaults as the reference class; what sits underneath changes:
``setup_single_final_problem`` fills a :class:`~conflict_rez_b200.problem.CollocationProblem` instead of a CasADi graph
and ``solve_single_final_problem`` calls the CUDA solver (:class:`~conflict_rez_b200.solver.ObcaSolver`) instead of IPOPT.
The returned ``sol`` offers what the reference consumes from ``OptiSol``: ``stats()["return_status"]``,
``stats()["t_wall_total"]`` and an exception on non-success.

Warm-start stages (SURVEY.md section 8f-1):
* ``state_ws`` solves the reference's Euler-discretised tube-following NLP (vehicle.py:116-216) on the device, started from the spline
  guess whatever ``spline_ws`` says (the all-zero start needs IPOPT's restoration phase);
* ``dual_ws`` uses the closed-form rectangle-distance duals instead of an IPOPT solve (vehicle.py:250-294) -- the same optimum.
"""
import time
from typing import Dict, Optional, Tuple

import numpy as np

from conflict_rez_b200.control import warmstart
from conflict_rez_b200.control.compute_sets import compute_initial_states, compute_obstacles, compute_sets, interp_along_sets
from conflict_rez_b200.obstacle_types import GeofenceRegion
from conflict_rez_b200.problem import CollocationGuess, CollocationProblem
from conflict_rez_b200.pytypes import VehiclePrediction, VehicleState
from conflict_rez_b200.solver import HIST_FIELDS, HIST_STEP_FIELDS, RETURN_STATUS, ObcaSolver, SolveOptions
from conflict_rez_b200.vehicle_types import VehicleBody, VehicleConfig


def collocation_coefficients(K: int):
    """Lagrange-basis collocation matrices on tau = [0, Radau(K)] (reference: vehicle.py:54-97)."""
    return warmstart.collocation_coefficients(K)


class ObcaSol:
    """What the planners read from CasADi's ``OptiSol``."""

    def __init__(self, result, wall, b=0):
        self.result, self.b, self._wall = result, b, wall

    def stats(self):
        """``iterations`` is present when the solve recorded (``SolveOptions.history`` > 0): IPOPT's per-iteration record as a dict
        of lists, one entry per iterate.  Its key names are those of CasADi's IPOPT plugin as recalled; they could not be checked
        against an installed CasADi.  As in IPOPT's table, the step entries (d_norm, regularization_size, alpha_pr, alpha_du,
        ls_trials) of entry k describe the step that produced iterate k, and entry 0 has zeros there."""
        r, b = self.result, self.b
        out = {
            "return_status": RETURN_STATUS.get(int(r.status[b]), "Unknown"),
            "iter_count": int(r.iters[b]),
            "t_wall_total": self._wall,
            "success": bool(r.status[b] >= 0),
        }
        if r.history is not None:
            rows = r.history[b, : min(int(r.history_count[b]), r.history.shape[1])]
            step = np.zeros((len(rows), 5))  # reg, d_norm, alpha_pr, alpha_du, ls_trials of the step into each iterate
            step[1:] = np.nan_to_num(rows[:-1, HIST_STEP_FIELDS], nan=0.0)
            f = dict(zip(HIST_FIELDS, rows.T))
            out["iterations"] = {
                "obj": f["obj"].tolist(), "inf_pr": f["inf_pr"].tolist(), "inf_du": f["inf_du"].tolist(), "mu": f["mu"].tolist(),
                "d_norm": step[:, 1].tolist(), "regularization_size": step[:, 0].tolist(), "alpha_pr": step[:, 2].tolist(),
                "alpha_du": step[:, 3].tolist(), "ls_trials": step[:, 4].astype(int).tolist(),
            }
        return out


class Vehicle(object):
    def __init__(
        self,
        rl_file_name: str,
        agent: str,
        color: Dict[str, Tuple[float, float, float]],
        vehicle_config: VehicleConfig = VehicleConfig(),
        vehicle_body: VehicleBody = VehicleBody(),
        region: GeofenceRegion = GeofenceRegion(),
        device="cuda:0",
    ) -> None:
        self.rl_file_name, self.agent, self.color = rl_file_name, agent, color
        self.vehicle_config, self.vehicle_body, self.region = vehicle_config, vehicle_body, region
        self.device = device
        self.init_state = compute_initial_states(self.rl_file_name, self.vehicle_body)[self.agent]
        self.obstacles = compute_obstacles()
        self.rl_tube = compute_sets(self.rl_file_name)[self.agent]
        self.num_sets = len(self.rl_tube)
        self.solve_options = SolveOptions()  # tol = constr_viol_tol = 1e-2 like vehicle.py:651-652

    collocation_coefficients = staticmethod(collocation_coefficients)

    # ------------------------------------------------------------------ warm start
    def state_ws(self, N: int = 30, dt: float = 0.1, init_offset: VehicleState = VehicleState(), final_heading: float = None,
                 bounded_input: bool = False, shrink_tube: float = 0.8, spline_ws: bool = False, verbose: int = 0) -> VehiclePrediction:
        """Tube-following state warm start (vehicle.py:99-231): the reference's Euler-discretised NLP -- nodes 0 .. N (num_sets - 1),
        cost sum a^2 + w^2, tube sets at k = N i, a_0 = w_0 = 0, optional final heading, input bounds only with ``bounded_input`` --
        solved on the device (``ObcaStateWsSolver``, OBCA_MODE_STATE_WS).  Initial guess: the Bezier pose guess through the sets
        (what ``spline_ws=True`` passes to ``opti.set_initial``) completed by the speeds of its kinematic reconstruction; the
        all-zero start of ``spline_ws=False`` (outside the region, IPOPT reaches the tube through its restoration phase) is not
        reproduced -- both settings start from the spline.  Output as the reference returns it: uniform grid t, inputs padded by
        their last value (vehicle.py:219-229)."""
        from conflict_rez_b200.solver import ObcaStateWsSolver, StateWsProblem

        path = interp_along_sets(self.rl_file_name, self.vehicle_body, N)[self.agent].copy()
        off = np.array([init_offset.x.x, init_offset.x.y, init_offset.e.psi])
        path += np.clip(1.0 - np.arange(len(path)) / float(N), 0.0, 1.0)[:, None] * off[None, :]
        vc, rg = self.vehicle_config, self.region
        limits = np.array([vc.v_min, vc.v_max, vc.delta_min, vc.delta_max, vc.a_min, vc.a_max, vc.w_delta_min, vc.w_delta_max], dtype=float)
        kin = warmstart.kinematic_guess(path, dt, self.vehicle_body.wb, limits)
        names = ("x", "y", "psi", "v", "delta", "a", "w")
        S = self.num_sets
        tube_A, tube_b = np.zeros((S, 2, 4, 2)), np.zeros((S, 2, 4))
        for q, sets in enumerate(self.rl_tube):
            for ib, body in enumerate(("back", "front")):
                tube_A[q, ib], tube_b[q, ib] = sets[body].A, np.ravel(sets[body].b)
        prob = StateWsProblem(tube_A=tube_A, tube_b=tube_b, N=N, dt=dt, final_heading=final_heading, bounded_input=bounded_input, shrink_tube=shrink_tube,
                              wb=self.vehicle_body.wb, region=np.array([rg.x_min, rg.x_max, rg.y_min, rg.y_max]), limits=limits)
        M = prob.nodes
        assert len(path) == M, (len(path), M)
        z0 = np.stack([kin[k] for k in names], axis=1)
        cur = np.array([path[0, 0], path[0, 1], path[0, 2], 0.0, 0.0])
        sv = ObcaStateWsSolver(prob, SolveOptions(tol=1e-2, constr_viol_tol=1e-2, max_iter=500), device=self.device, lib=getattr(self, "_lib", None))  # vehicle.py:207-213
        res = sv.solve_ws(cur[None], z0[None])
        sv.close()
        self.state_ws_result = res
        if verbose:
            print(res.return_status(0))
        if res.status[0] >= 0:
            kin = {k: res.z[0, 0, :, c].copy() for c, k in enumerate(names)}
        result = VehiclePrediction()
        result.t = np.linspace(0, (M - 1) * dt, M, endpoint=True)
        result.x, result.y, result.psi, result.v = kin["x"], kin["y"], kin["psi"], kin["v"]
        result.u_steer = kin["delta"]
        result.u_a = np.append(kin["a"][:-1], kin["a"][-2])
        result.u_steer_dot = np.append(kin["w"][:-1], kin["w"][-2])
        return result

    def _obstacle_arrays(self):
        return np.stack([o.A for o in self.obstacles]), np.stack([np.ravel(o.b) for o in self.obstacles])

    def dual_ws(self, zu0: VehiclePrediction, verbose: int = 0) -> VehiclePrediction:
        A, b = self._obstacle_arrays()
        lam, mu = warmstart.dual_ws_rect(np.asarray(zu0.x), np.asarray(zu0.y), np.asarray(zu0.psi), A, b,
                                         np.asarray(self.vehicle_body.A, float), np.asarray(self.vehicle_body.b, float))
        zu0.l = lam.reshape(len(zu0.x), -1).T  # (sum h, N) like vehicle.py:252,293
        zu0.m = mu.reshape(len(zu0.x), -1).T
        return zu0

    def interp_ws_for_collocation(self, zu0: VehiclePrediction, K: int = 5, N_per_set: int = 5):
        N = N_per_set * (self.num_sets - 1)
        sig = {"x": zu0.x, "y": zu0.y, "psi": zu0.psi, "v": zu0.v, "u_steer": zu0.u_steer, "u_a": zu0.u_a, "u_steer_dot": zu0.u_steer_dot,
               "l": np.asarray(zu0.l).T, "m": np.asarray(zu0.m).T}
        t_interp, res = warmstart.interp_ws_for_collocation(np.asarray(zu0.t), sig, N, K)
        out = VehiclePrediction()
        out.t = t_interp
        for k in ("x", "y", "psi", "v", "u_steer", "u_a", "u_steer_dot"):
            setattr(out, k, res[k])
        out.l = [[res["l"][i * (K + 1) + k] for k in range(K + 1)] for i in range(N)]
        out.m = [[res["m"][i * (K + 1) + k] for k in range(K + 1)] for i in range(N)]
        return out

    # ------------------------------------------------------------------ final problem
    def _guess_arrays(self, zu0: VehiclePrediction):
        N, K1, O = self.N, self.K + 1, len(self.obstacles)
        z = np.stack([np.asarray(getattr(zu0, k), float) for k in ("x", "y", "psi", "v", "u_steer", "u_a", "u_steer_dot")], axis=1)
        lam = np.array([[zu0.l[i][k] for k in range(K1)] for i in range(N)], float).reshape(N * K1, O, 4)
        mu = np.array([[zu0.m[i][k] for k in range(K1)] for i in range(N)], float).reshape(N * K1, O, 4)
        return z, lam, mu

    def setup_single_final_problem(self, zu0: VehiclePrediction, init_offset: VehicleState = VehicleState(), final_heading: float = None,
                                   opti=None, dt=None, K: int = 5, N_per_set: int = 5, dmin: float = 0.05, shrink_tube: float = 0.8):
        """Fill the problem descriptor.  ``opti`` may be a :class:`JointProblem` (the analogue of sharing one ``ca.Opti``
        between vehicles, multi_vehicle_planner.py:374-384); ``dt`` is then the shared interval length."""
        self.N, self.K = N_per_set * (self.num_sets - 1), K
        z, lam, mu = self._guess_arrays(zu0)
        dt0 = zu0.dt if getattr(zu0, "dt", None) is not None else np.asarray(zu0.t)[-1] / self.N
        pose0 = np.array([self.init_state.x.x + init_offset.x.x, self.init_state.x.y + init_offset.x.y, self.init_state.e.psi + init_offset.e.psi])
        self._block = dict(agent=self.agent, tube=self.rl_tube, pose0=pose0, heading=final_heading, z=z, lam=lam, mu=mu, dt0=float(dt0))
        self._params = dict(K=K, n_per_set=N_per_set, dmin=dmin, shrink_tube=shrink_tube)
        self.opti = opti if opti is not None else JointProblem(self.obstacles, self.vehicle_body, self.vehicle_config, self.region)
        self.opti.add_vehicle(self._block, self._params, dt)
        return self.opti

    def solve_single_final_problem(self, verbose: int = 0):
        sol = self.opti.solve(self.solve_options, self.device, getattr(self, "_lib", None))
        if verbose:
            print(sol.stats()["return_status"])
        return sol

    def get_solution(self, sol: ObcaSol) -> VehiclePrediction:
        r, b = sol.result, sol.b
        ia = sol.agents.index(self.agent)
        M = self.N * (self.K + 1)
        z = r.z[b, ia, :M]
        result = VehiclePrediction()
        result.dt = float(r.dt[b])
        tau = warmstart.radau_nodes(self.K)
        result.t = (np.arange(self.N)[:, None] + tau[None, :]).ravel() * result.dt
        result.x, result.y, result.psi, result.v = z[:, 0].copy(), z[:, 1].copy(), z[:, 2].copy(), z[:, 3].copy()
        result.u_steer, result.u_a, result.u_steer_dot = z[:, 4].copy(), z[:, 5].copy(), z[:, 6].copy()
        lam = r.lam[b, ia, :M].reshape(M, -1)
        mu = r.mu[b, ia, :M].reshape(M, -1)
        K1 = self.K + 1
        result.l = [[lam[i * K1 + k] for k in range(K1)] for i in range(self.N)]
        result.m = [[mu[i * K1 + k] for k in range(K1)] for i in range(self.N)]
        self.get_interpolator(K=self.K, N=self.N, dt=result.dt, opt=result)
        return result

    # ------------------------------------------------------------------ interpolation (vehicle.py:722-829)
    def get_interpolator(self, K: int, N: int, dt: float, opt: VehiclePrediction):
        X = np.stack([np.reshape(getattr(opt, k), (N, K + 1)) for k in ("x", "y", "psi", "v", "u_steer")], axis=-1)
        _, _, D = collocation_coefficients(K)
        self._interp = dict(X=X, lf=np.einsum("k,kl->l", D, X[-1]), tau=warmstart.radau_nodes(K), K=K, N=N, dt=dt,
                            t_in=np.asarray(opt.t), u_a=np.asarray(opt.u_a), u_w=np.asarray(opt.u_steer_dot))

    def interpolate_states(self, time) -> VehiclePrediction:
        """Piecewise degree-K Lagrange interpolation of the states, piecewise-constant inputs, final state held after t_final."""
        I = self._interp
        tq = np.asarray(time, dtype=float)
        tgrid = np.linspace(0, I["N"] * I["dt"], I["N"] + 1)
        idx = np.searchsorted(tgrid[1:], tq, side="right")  # ca.pw_const: interval i while t < tgrid[i+1]
        inside = idx < I["N"]
        ii = np.minimum(idx, I["N"] - 1)
        rel = (tq - tgrid[ii]) / I["dt"]
        tau = I["tau"]
        basis = np.ones((len(tq), I["K"] + 1))
        for j in range(I["K"] + 1):
            for k in range(I["K"] + 1):
                if k != j:
                    basis[:, j] *= (rel - tau[k]) / (tau[j] - tau[k])
        states = np.einsum("tj,tjl->tl", basis, I["X"][ii])
        # beyond the horizon every collocation value is the final state lf, so the interpolant is lf itself
        states[~inside] = I["lf"][None, :] * np.ones((np.count_nonzero(~inside), 1))
        ju = np.clip(np.searchsorted(I["t_in"][1:], tq, side="right"), 0, len(I["u_a"]) - 1)
        res = VehiclePrediction()
        res.t = tq
        res.x, res.y, res.psi, res.v, res.u_steer = states[:, 0], states[:, 1], states[:, 2], states[:, 3], states[:, 4]
        res.u_a, res.u_steer_dot = I["u_a"][ju], I["u_w"][ju]
        return res


class JointProblem:
    """The analogue of one ``ca.Opti`` instance shared by several vehicles (plus the pair blocks)."""

    def __init__(self, obstacles, vehicle_body, vehicle_config, region):
        self.obstacles, self.vb, self.vc, self.region = obstacles, vehicle_body, vehicle_config, region
        self.blocks, self.params, self.dt0, self.pair_guess = [], None, None, None

    def add_vehicle(self, block, params, dt):
        if self.params is not None and params != self.params:
            raise ValueError("all vehicles of a joint problem must share K, N_per_set, dmin and shrink_tube")
        self.params = params
        self.blocks.append(block)
        if dt is not None:
            self.dt0 = float(dt)

    def set_pair_initial(self, pair_lam, pair_mu, pair_s):
        self.pair_guess = (pair_lam, pair_mu, pair_s)

    def build(self):
        V, O = len(self.blocks), len(self.obstacles)
        n_sets = np.array([len(b["tube"]) for b in self.blocks])
        Smax = int(n_sets.max())
        tube_A, tube_b = np.zeros((V, Smax, 2, 4, 2)), np.zeros((V, Smax, 2, 4))
        for ia, blk in enumerate(self.blocks):
            for q, sets in enumerate(blk["tube"]):
                for ib, body in enumerate(("back", "front")):
                    tube_A[ia, q, ib], tube_b[ia, q, ib] = sets[body].A, np.ravel(sets[body].b)
        vc, rg = self.vc, self.region
        prob = CollocationProblem(
            n_sets=n_sets,
            obs_A=np.stack([o.A for o in self.obstacles]) if O else np.zeros((0, 4, 2)),
            obs_b=np.stack([np.ravel(o.b) for o in self.obstacles]) if O else np.zeros((0, 4)),
            tube_A=tube_A, tube_b=tube_b, init_pose=np.stack([b["pose0"] for b in self.blocks]),
            final_heading=np.array([np.nan if b["heading"] is None else float(b["heading"]) for b in self.blocks]),
            body_G=np.asarray(self.vb.A, float), body_g=np.asarray(self.vb.b, float), wb=self.vb.wb,
            region=np.array([rg.x_min, rg.x_max, rg.y_min, rg.y_max]),
            limits=np.array([vc.v_min, vc.v_max, vc.delta_min, vc.delta_max, vc.a_min, vc.a_max, vc.w_delta_min, vc.w_delta_max], dtype=float),
            **self.params,
        )
        Mmax = int(prob.nodes.max())
        z, lam, mu = np.zeros((V, Mmax, 7)), np.zeros((V, Mmax, O, 4)), np.zeros((V, Mmax, O, 4))
        for ia, blk in enumerate(self.blocks):
            M = len(blk["z"])
            z[ia, :M], lam[ia, :M], mu[ia, :M] = blk["z"], blk["lam"], blk["mu"]
        dt0 = self.dt0 if self.dt0 is not None else float(np.mean([b["dt0"] for b in self.blocks]))
        pl = pm = ps = None
        if V > 1:
            if self.pair_guess is None:
                P = len(prob.pairs)
                pl, pm, ps = np.zeros((P, Mmax, 4)), np.zeros((P, Mmax, 4)), np.zeros((P, Mmax, 2))
                for q, (a, b) in enumerate(prob.pairs):
                    m = int(min(prob.nodes[a], prob.nodes[b]))
                    pl[q, :m], pm[q, :m], ps[q, :m] = warmstart.joint_dual_ws_rect(
                        z[a, :m, 0], z[a, :m, 1], z[a, :m, 2], z[b, :m, 0], z[b, :m, 1], z[b, :m, 2], prob.body_G, prob.body_g)
            else:
                pl, pm, ps = self.pair_guess
        return prob, CollocationGuess(z, lam, mu, np.float64(dt0), pl, pm, ps)

    def solve(self, options: Optional[SolveOptions] = None, device="cuda:0", lib=None) -> ObcaSol:
        prob, guess = self.build()
        sv = ObcaSolver(prob, options, device=device, lib=lib)
        t0 = time.perf_counter()
        res = sv.solve(guess)
        wall = time.perf_counter() - t0
        sv.close()
        sol = ObcaSol(res, wall)
        sol.agents = [b["agent"] for b in self.blocks]
        sol.problem = prob
        if res.status[0] < 0:
            # CasADi's Opti raises when IPOPT does not report success (SURVEY.md App. E); so does this drop-in
            err = RuntimeError("OBCA solve failed: " + sol.stats()["return_status"])
            err.sol = sol
            raise err
        return sol
