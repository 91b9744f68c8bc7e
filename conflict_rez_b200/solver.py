"""ctypes binding of ``libobca_b200.so`` (C ABI in ``include/obca.h``) and the batched front door.

This is the drop-in for the ``opti.solver("ipopt", ...); opti.solve()`` call of the reference
(confrez/control/vehicle.py:657-658, multi_vehicle_planner.py:464-465): the planners fill a
:class:`~conflict_rez_b200.problem.CollocationProblem` / ``CollocationGuess`` and call
:meth:`ObcaSolver.solve`.  PyTorch is used for device memory and streams only; every numerical step runs in
the hand-written sm_100a kernels.  There is **no CPU fallback**: a missing library or a missing GPU raises.
"""
import ctypes
import os
from dataclasses import dataclass
from typing import Optional

import numpy as np
import torch

from conflict_rez_b200.problem import CollocationGuess, CollocationProblem

OBCA_MAX_V = 8
_LIB_NAME = "libobca_b200.so"

RETURN_STATUS = {
    0: "Solve_Succeeded",
    1: "Solved_To_Acceptable_Level",
    -1: "Maximum_Iterations_Exceeded",
    -2: "Restoration_Failed",
    -3: "Error_In_Step_Computation",
    -4: "Invalid_Number_Detected",
    -5: "Search_Direction_Becomes_Too_Small",
    -6: "Infeasible_Problem_Detected",
    -100: "Not_Solved",
}


class ObcaDims(ctypes.Structure):
    _fields_ = [
        ("batch", ctypes.c_int32),
        ("V", ctypes.c_int32),
        ("O", ctypes.c_int32),
        ("K", ctypes.c_int32),
        ("n_per_set", ctypes.c_int32),
        ("n_sets", ctypes.c_int32 * OBCA_MAX_V),
        ("mode", ctypes.c_int32),
        ("horizon", ctypes.c_int32),
        ("n_others", ctypes.c_int32),
        ("bounded_input", ctypes.c_int32),
    ]


class ObcaOptions(ctypes.Structure):
    _fields_ = [
        ("tol", ctypes.c_double),
        ("constr_viol_tol", ctypes.c_double),
        ("dual_inf_tol", ctypes.c_double),
        ("compl_inf_tol", ctypes.c_double),
        ("mu_init", ctypes.c_double),
        ("dmin", ctypes.c_double),
        ("shrink_tube", ctypes.c_double),
        ("elastic_weight", ctypes.c_double),
        ("max_iter", ctypes.c_int32),
        ("refine_steps", ctypes.c_int32),
    ]


_dp = ctypes.POINTER(ctypes.c_double)


class ObcaStatic(ctypes.Structure):
    _fields_ = [(n, _dp) for n in ("obs_A", "obs_b", "tube_A", "tube_b", "body_G", "body_g", "region", "limits", "final_heading")] + [
        ("wb", ctypes.c_double),
        ("mpc_dt", ctypes.c_double),
        ("colloc_A", _dp),
        ("colloc_B", _dp),
    ]


EXPORTS = [
    "obca_version",
    "obca_last_error",
    "obca_default_options",
    "obca_create",
    "obca_destroy",
    "obca_set_static",
    "obca_set_options",
    "obca_set_init_pose",
    "obca_set_initial",
    "obca_set_mpc_params",
    "obca_dual_ws",
    "obca_joint_dual_ws",
    "obca_measure_dfma_peak",
    "obca_interpolate",
    "obca_interp_ws",
    "obca_mpc_ref_times",
    "obca_plant_step",
    "obca_shift_horizon",
    "obca_set_order",
    "obca_solve",
    "obca_get_solution",
    "obca_get_stats",
    "obca_set_history",
    "obca_get_history",
    "obca_launch_count",
    "obca_layout",
    "obca_debug_get_iterate",
    "obca_debug_set_iterate",
    "obca_debug_eval",
    "obca_debug_step",
    "obca_debug_kkt_apply",
    "obca_debug_profile",
]


def default_library_path() -> str:
    return os.path.join(os.path.dirname(os.path.abspath(__file__)), _LIB_NAME)


def load_library(path: Optional[str] = None) -> ctypes.CDLL:
    """Load the CUDA library; raises (never falls back) when it has not been built."""
    path = path or default_library_path()
    if not os.path.exists(path):
        raise RuntimeError(
            "%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  conflict_rez_b200 has no CPU fallback." % path
        )
    lib = ctypes.CDLL(path)
    vp, i32p = ctypes.c_void_p, ctypes.POINTER(ctypes.c_int32)
    lib.obca_version.restype = ctypes.c_char_p
    lib.obca_last_error.restype = ctypes.c_char_p
    lib.obca_default_options.argtypes = [ctypes.POINTER(ObcaOptions)]
    lib.obca_create.argtypes = [ctypes.POINTER(ObcaDims), ctypes.POINTER(ObcaOptions), ctypes.c_int, ctypes.POINTER(vp)]
    lib.obca_destroy.argtypes = [vp]
    lib.obca_set_static.argtypes = [vp, ctypes.POINTER(ObcaStatic)]
    lib.obca_set_options.argtypes = [vp, ctypes.POINTER(ObcaOptions)]
    lib.obca_set_init_pose.argtypes = [vp, vp, vp]
    lib.obca_set_initial.argtypes = [vp] + [vp] * 7 + [vp]
    lib.obca_set_mpc_params.argtypes = [vp, vp, vp, vp, vp]
    lib.obca_dual_ws.argtypes = [vp, vp, vp, vp, vp]
    lib.obca_joint_dual_ws.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.obca_measure_dfma_peak.argtypes = [ctypes.c_int, _dp]
    lib.obca_interpolate.argtypes = [ctypes.c_int, vp, vp, i32p, _dp, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp]
    lib.obca_interp_ws.argtypes = [ctypes.c_int, vp, vp, _dp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp]
    lib.obca_mpc_ref_times.argtypes = [ctypes.c_int, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double, vp, vp]
    lib.obca_plant_step.argtypes = [ctypes.c_int, vp, vp, ctypes.c_int, ctypes.c_double, ctypes.c_double, ctypes.c_int, vp, vp]
    lib.obca_shift_horizon.argtypes = [ctypes.c_int, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp]
    lib.obca_set_order.argtypes = [vp, vp, vp]
    lib.obca_solve.argtypes = [vp, vp]
    lib.obca_get_solution.argtypes = [vp] + [vp] * 7 + [vp]
    lib.obca_get_stats.argtypes = [vp] + [vp] * 7 + [vp]
    lib.obca_set_history.argtypes = [vp, ctypes.c_int32]
    lib.obca_get_history.argtypes = [vp, vp, vp, vp]
    lib.obca_launch_count.argtypes = [vp]
    lib.obca_launch_count.restype = ctypes.c_int64
    lib.obca_layout.argtypes = [vp, ctypes.POINTER(ctypes.c_int64), ctypes.c_int]
    lib.obca_debug_get_iterate.argtypes = [vp, ctypes.c_int] + [_dp] * 4
    lib.obca_debug_set_iterate.argtypes = [vp, ctypes.c_int] + [_dp] * 4
    lib.obca_debug_eval.argtypes = [vp, ctypes.c_int, _dp, _dp, _dp]
    lib.obca_debug_step.argtypes = [vp, ctypes.c_int, ctypes.c_double, ctypes.c_double, _dp, _dp, i32p]
    lib.obca_debug_kkt_apply.argtypes = [vp, ctypes.c_int, ctypes.c_double, _dp, _dp, _dp, _dp]
    lib.obca_debug_profile.argtypes = [vp, ctypes.POINTER(ctypes.c_int64), ctypes.c_int]
    return lib


@dataclass
class SolveOptions:
    """IPOPT options the reference passes (vehicle.py:648-656) plus the formulation constants."""

    tol: float = 1e-2
    constr_viol_tol: float = 1e-2
    dual_inf_tol: float = 1.0
    compl_inf_tol: float = 1e-4
    mu_init: float = 0.1
    max_iter: int = 3000
    elastic_weight: float = 1e3
    refine_steps: int = -1  # iterative-refinement solves per Newton system; -1: none at tol > 1e-5, 2 at tight tolerances
    history: int = 0  # rows of the iteration record kept per instance (BatchResult.history); 0: no record


# Fields of one row of the iteration record, in the order of OBCA_HIST_ITER .. OBCA_HIST_RHO (include/obca.h).  Row r describes
# iterate r and the step taken from it; rows without a step have NaN in reg .. ls_trials.
HIST_FIELDS = ("iter", "attempt", "obj", "inf_pr", "theta", "inf_du", "compl", "mu", "err", "reg", "d_norm", "alpha_pr", "alpha_du", "ls_trials",
               "flags", "rho")
HIST_STEP_FIELDS = slice(9, 14)  # reg, d_norm, alpha_pr, alpha_du, ls_trials
HIST_F_MU_LOWERED, HIST_F_INERTIA, HIST_F_TINY_STEP, HIST_F_RESET, HIST_F_ACCEPTABLE = 1, 2, 4, 8, 16


@dataclass
class BatchResult:
    status: np.ndarray  # (B,) int32, see RETURN_STATUS
    iters: np.ndarray
    obj: np.ndarray
    cviol: np.ndarray
    dual_inf: np.ndarray
    compl_inf: np.ndarray
    elastic: np.ndarray  # largest elastic variable of the distance rows (0 at a solution of the reference problem)
    z: np.ndarray  # (B,V,Mmax,7)
    lam: np.ndarray
    mu: np.ndarray
    dt: np.ndarray
    pair_lam: Optional[np.ndarray]
    pair_mu: Optional[np.ndarray]
    pair_s: Optional[np.ndarray]
    history: Optional[np.ndarray] = None  # (B, capacity, len(HIST_FIELDS)) float64 iteration record, None when not recorded
    history_count: Optional[np.ndarray] = None  # (B,) int32 heads evaluated per instance (may exceed the capacity)

    def return_status(self, b: int = 0) -> str:
        return RETURN_STATUS.get(int(self.status[b]), "Unknown")


def format_history(result: BatchResult, b: int = 0) -> str:
    """IPOPT's iteration table of instance ``b`` from its record.  As in IPOPT's output, the step columns of a line (``||d||``,
    ``lg(rg)`` = log10 delta_w, ``alpha_du``, ``alpha_pr``, ``ls`` = line-search trials) describe the step that produced its iterate,
    so line 0 has none.  The last column shows the flags: m = mu lowered and a = acceptable point at this iterate; i = inertia
    correction, t = tiny step and r = barrier reset on the step that led to it."""
    if result.history is None:
        raise ValueError("format_history: the solve did not record (SolveOptions.history = 0)")
    rows, n = result.history[b], int(result.history_count[b])
    lines = ["iter att       objective   inf_pr   inf_du lg(mu)  ||d|| lg(rg) alpha_du alpha_pr   ls      rho flags"]
    head_bits, step_bits = HIST_F_MU_LOWERED | HIST_F_ACCEPTABLE, HIST_F_INERTIA | HIST_F_TINY_STEP | HIST_F_RESET
    prev = None
    for r in rows[: min(n, rows.shape[0])]:
        fl = int(r[14]) & head_bits
        if prev is None or np.isnan(prev[11]):  # first line, or first line of a restarted attempt
            step = "     -      -        -        -    -"
        else:
            fl |= int(prev[14]) & step_bits
            rg = "%6.1f" % np.log10(prev[9]) if prev[9] > 0 else "     -"
            step = "%6.1e %s %8.2e %8.2e %4d" % (prev[10], rg, prev[12], prev[11], int(prev[13]))
        flags = "".join(c for c, bit in zip("mitra", (HIST_F_MU_LOWERED, HIST_F_INERTIA, HIST_F_TINY_STEP, HIST_F_RESET, HIST_F_ACCEPTABLE)) if fl & bit)
        lines.append("%4d %3d %15.8e %8.2e %8.2e %6.2f %s %8.1e %s" % (int(r[0]), int(r[1]), r[2], r[3], r[5], np.log10(r[7]), step, r[15], flags))
        prev = r
    if n > rows.shape[0]:
        lines.append("... %d more iterations past the capacity of %d rows" % (n - rows.shape[0], rows.shape[0]))
    return "\n".join(lines)


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _np_ptr(a: np.ndarray):
    return a.ctypes.data_as(_dp)


class TrajectoryOps:
    """Trajectory-side kernels around the solve (csrc/obca_traj.h): batched evaluation of collocation solutions
    (``Vehicle.interpolate_states``, vehicle.py:722-829), the MPC reference window (``get_current_ref``, vehicle_follower.py:370-404),
    the plant step (``simulator``, dynamic_model.py:61-93) and the one-step horizon shift (``_adv_onestep``).  All arrays are device
    tensors (float64, contiguous) on ``device``; the kernels run on torch's current stream."""

    def __init__(self, device="cuda:0", lib: Optional[ctypes.CDLL] = None):
        self.lib = lib if lib is not None else load_library()
        self.device = torch.device(device)
        self.is_emulation = b"EMULATION" in self.lib.obca_version()
        if self.device.type != "cuda" and not self.is_emulation:
            raise RuntimeError("TrajectoryOps needs a CUDA device (no CPU fallback)")
        self.index = (self.device.index or 0) if self.device.type == "cuda" else 0
        from conflict_rez_b200.control.warmstart import radau_nodes

        self._tau = np.ascontiguousarray(radau_nodes(5))

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream) if self.device.type == "cuda" else None

    def _check(self, rc):
        if rc < 0:
            raise RuntimeError("obca: " + self.lib.obca_last_error().decode())

    def interpolate(self, z: torch.Tensor, dt: torch.Tensor, n_intervals, times: torch.Tensor) -> torch.Tensor:
        """z (B,V,Mmax,7), dt (B) or (B,V), n_intervals (V) ints, times (T) or (B,V,T) -> (B,V,T,7) = x y psi v delta a w."""
        B, V, Mmax, _ = z.shape
        per = times.dim() == 3
        T = times.shape[-1]
        out = torch.empty((B, V, T, 7), dtype=torch.float64, device=z.device)
        ni = (ctypes.c_int32 * V)(*[int(n) for n in n_intervals])
        self._check(self.lib.obca_interpolate(self.index, _ptr(z.contiguous()), _ptr(dt.contiguous()), ni, _np_ptr(self._tau), B, V, Mmax,
                                              _ptr(times.contiguous()), T, int(per), int(dt.dim() == 2), _ptr(out), self._stream()))
        return out

    def interp_ws(self, sig: torch.Tensor, t: torch.Tensor, N: int) -> torch.Tensor:
        """``Vehicle.interp_ws_for_collocation`` (vehicle.py:298-358) for a batch: sig (B,T,C) sampled on t (T) -> (B,N*6,C), linear
        interpolation onto the collocation times (i + tau_k) / N * t[-1]."""
        B, T, C = sig.shape
        out = torch.empty((B, N * 6, C), dtype=torch.float64, device=sig.device)
        self._check(self.lib.obca_interp_ws(self.index, _ptr(sig.contiguous()), _ptr(t.contiguous()), _np_ptr(self._tau), B, T, C, N, _ptr(out), self._stream()))
        return out

    def mpc_ref_times(self, grid: torch.Tensor, clock: torch.Tensor, N: int, dt_mpc: float) -> torch.Tensor:
        """grid (B,V,3) = (t_first, t_last, n_ref) of each dense reference time grid, clock (B,V) -> (B,V,N) sample times."""
        B, V, _ = grid.shape
        out = torch.empty((B, V, N), dtype=torch.float64, device=grid.device)
        self._check(self.lib.obca_mpc_ref_times(self.index, _ptr(grid.contiguous()), _ptr(clock.contiguous()), B, V, N, float(dt_mpc), _ptr(out), self._stream()))
        return out

    def plant_step(self, state: torch.Tensor, u: torch.Tensor, dt: float, wb: float, substeps: int = 100) -> torch.Tensor:
        """state (B,5), u (B,2) -> state after dt under constant input."""
        out = torch.empty_like(state)
        self._check(self.lib.obca_plant_step(self.index, _ptr(state.contiguous()), _ptr(u.contiguous()), state.shape[0], float(dt), float(wb), int(substeps), _ptr(out), self._stream()))
        return out

    def shift_horizon(self, a: torch.Tensor) -> torch.Tensor:
        """(B,N,...) -> shifted by one step along N with the last value held (``_adv_onestep``)."""
        B, N = a.shape[:2]
        W = int(np.prod(a.shape[2:])) if a.dim() > 2 else 1
        out = torch.empty_like(a)
        self._check(self.lib.obca_shift_horizon(self.index, _ptr(a.contiguous()), B, N, W, _ptr(out), self._stream()))
        return out


class ObcaSolver:
    """One handle = one problem shape (V, sets, obstacles) x one batch size on one GPU."""

    def __init__(self, prob: CollocationProblem, options: Optional[SolveOptions] = None, device="cuda:0", lib: Optional[ctypes.CDLL] = None):
        self.lib = lib if lib is not None else load_library()
        self.device = torch.device(device)
        self.is_emulation = b"EMULATION" in self.lib.obca_version()
        if self.device.type != "cuda" and not self.is_emulation:
            raise RuntimeError("ObcaSolver needs a CUDA device (no CPU fallback)")
        if self.device.type == "cuda" and not torch.cuda.is_available():
            raise RuntimeError("ObcaSolver: CUDA is not available on this machine (no CPU fallback)")
        self.prob = prob
        self.opts = options or SolveOptions()
        self.B = prob.batch or 1
        self.V, self.O, self.P = prob.V, prob.O, len(prob.pairs)
        self.Mmax = int(prob.nodes.max())
        dims = ObcaDims(batch=self.B, V=self.V, O=self.O, K=prob.K, n_per_set=prob.n_per_set)
        for a in range(self.V):
            dims.n_sets[a] = int(prob.n_sets[a])
        copts = ObcaOptions()
        self.lib.obca_default_options(ctypes.byref(copts))
        for name in ("tol", "constr_viol_tol", "dual_inf_tol", "compl_inf_tol", "mu_init", "max_iter", "elastic_weight", "refine_steps"):
            setattr(copts, name, getattr(self.opts, name))
        copts.dmin, copts.shrink_tube = prob.dmin, prob.shrink_tube
        self.handle = ctypes.c_void_p()
        dev_index = self.device.index or 0 if self.device.type == "cuda" else 0
        self._check(self.lib.obca_create(ctypes.byref(dims), ctypes.byref(copts), dev_index, ctypes.byref(self.handle)))
        keep = {n: np.ascontiguousarray(getattr(prob, n), dtype=np.float64) for n in ("obs_A", "obs_b", "tube_A", "tube_b", "body_G", "body_g", "region", "limits", "final_heading")}
        from conflict_rez_b200.control.warmstart import collocation_coefficients

        cA, cB, _ = collocation_coefficients(prob.K)  # the reference's own construction (vehicle.py:54-97), bit-identical on both sides
        keep["colloc_A"], keep["colloc_B"] = np.ascontiguousarray(cA), np.ascontiguousarray(cB)
        st = ObcaStatic(wb=float(prob.wb), **{n: _np_ptr(a) for n, a in keep.items()})
        self._check(self.lib.obca_set_static(self.handle, ctypes.byref(st)))
        self._set_history()
        self._stream = None
        self._staging = {}

    # -- helpers -----------------------------------------------------------------------------------
    def _check(self, rc):
        if rc < 0:
            raise RuntimeError("obca: " + self.lib.obca_last_error().decode())
        return rc

    def _stream_ptr(self):
        if self.device.type != "cuda":
            return None
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _to_dev(self, a, shape, name=None):
        """Host array -> device tensor.  With ``name`` the copy goes through a persistent pinned staging buffer and a
        persistent device tensor (one host memcpy + one asynchronous H2D copy per call, no allocation after the first)."""
        if self.device.type != "cuda":
            return torch.from_numpy(np.array(a, dtype=np.float64, order="C", copy=True).reshape(shape)).contiguous()
        if name is None:
            t = torch.from_numpy(np.array(a, dtype=np.float64, order="C", copy=True).reshape(shape))
            return t.pin_memory().to(self.device, non_blocking=True).contiguous()
        shape = tuple(int(v) for v in shape)
        buf = self._staging.get(name)
        if buf is None or tuple(buf[0].shape) != shape:
            buf = (torch.empty(shape, dtype=torch.float64, pin_memory=True), torch.empty(shape, dtype=torch.float64, device=self.device))
            self._staging[name] = buf
        arr = np.ascontiguousarray(a, dtype=np.float64).reshape(shape)
        if not arr.flags.writeable:  # torch.from_numpy warns about read-only arrays (it is only read here)
            arr = arr.copy()
        src = torch.from_numpy(arr)
        if src.is_pinned():  # the caller's array already is page-locked (e.g. allocated through torch.empty(pin_memory=True)): DMA straight from it
            buf[1].copy_(src, non_blocking=True)
        else:
            buf[0].copy_(src)  # torch's CPU copy runs on all intra-op threads: several times the rate of a single-threaded memcpy
            buf[1].copy_(buf[0], non_blocking=True)
        return buf[1]

    def _to_host(self, tensors):
        """Device tensors -> independent numpy arrays: asynchronous D2H copies into persistent pinned buffers, one sync."""
        if self.device.type != "cuda":
            return [None if t is None else t.numpy().copy() for t in tensors]
        pins = []
        for k, t in enumerate(tensors):
            if t is None:
                pins.append(None)
                continue
            key = ("out", k, tuple(t.shape), t.dtype)
            pin = self._staging.get(key)
            if pin is None:
                pin = torch.empty(tuple(t.shape), dtype=t.dtype, pin_memory=True)
                self._staging[key] = pin
            pin.copy_(t, non_blocking=True)
            pins.append(pin)
        torch.cuda.current_stream(self.device).synchronize()  # every copy above is on this stream; other streams (PipelinedSolver) keep running
        return [None if p_ is None else p_.clone().numpy() for p_ in pins]  # independent copies (multi-threaded), the pinned buffers are reused

    def close(self):
        if getattr(self, "handle", None):
            self.lib.obca_destroy(self.handle)
            self.handle = None

    def _set_history(self):
        """Turn the iteration record on for ``self.opts.history`` rows per instance (obca_set_history)."""
        if self.opts.history:  # a negative capacity is rejected by the library
            self._check(self.lib.obca_set_history(self.handle, int(self.opts.history)))

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launch_count(self) -> int:
        return int(self.lib.obca_launch_count(self.handle))

    # -- device-resident API (inputs already on the GPU) -------------------------------------------------
    def upload(self, guess: CollocationGuess, init_pose: Optional[np.ndarray] = None):
        """Host -> device copies of the per-instance data through persistent pinned staging buffers; returns the device
        tensors, which are owned by the solver and overwritten by the next ``upload``."""
        B, V, M, O, P = self.B, self.V, self.Mmax, self.O, self.P
        pose = self.prob.init_pose if init_pose is None else init_pose
        d = {
            "pose": self._to_dev(pose, (B, V, 3), "pose"),
            "z": self._to_dev(guess.z, (B, V, M, 7), "z"),
            "lam": self._to_dev(guess.lam, (B, V, M, O, 4), "lam"),
            "mu": self._to_dev(guess.mu, (B, V, M, O, 4), "mu"),
            "dt": self._to_dev(np.broadcast_to(guess.dt, (B,)), (B,), "dt"),
        }
        if P:
            d["pl"] = self._to_dev(guess.pair_lam, (B, P, M, 4), "pl")
            d["pm"] = self._to_dev(guess.pair_mu, (B, P, M, 4), "pm")
            d["ps"] = self._to_dev(guess.pair_s, (B, P, M, 2), "ps")
        return d

    def dual_ws(self, z):
        """Device warm start of the obstacle duals (replaces ``Vehicle.dual_ws``): z (B,V,Mmax,7) device -> lam, mu."""
        B, V, M, O = self.B, self.V, self.Mmax, self.O
        z = z.contiguous()
        assert tuple(z.shape) == (B, V, M, 7) and z.dtype == torch.float64
        lam = torch.empty((B, V, M, O, 4), dtype=torch.float64, device=z.device)
        mu = torch.empty_like(lam)
        self._check(self.lib.obca_dual_ws(self.handle, _ptr(z), _ptr(lam), _ptr(mu), self._stream_ptr()))
        return lam, mu

    def joint_dual_ws(self, z):
        """Device warm start of the pair duals (replaces ``MultiVehiclePlanner.joint_dual_ws``): z -> pair_lam, pair_mu, pair_s."""
        B, V, M, P = self.B, self.V, self.Mmax, self.P
        z = z.contiguous()
        assert tuple(z.shape) == (B, V, M, 7) and z.dtype == torch.float64
        pl = torch.empty((B, P, M, 4), dtype=torch.float64, device=z.device)
        pm = torch.empty_like(pl)
        ps = torch.empty((B, P, M, 2), dtype=torch.float64, device=z.device)
        self._check(self.lib.obca_joint_dual_ws(self.handle, _ptr(z), _ptr(pl), _ptr(pm), _ptr(ps), self._stream_ptr()))
        return pl, pm, ps

    def set_inputs(self, d):
        s = self._stream_ptr()
        self._check(self.lib.obca_set_init_pose(self.handle, _ptr(d["pose"]), s))
        self._check(
            self.lib.obca_set_initial(self.handle, _ptr(d["z"]), _ptr(d["lam"]), _ptr(d["mu"]), _ptr(d["dt"]), _ptr(d.get("pl")), _ptr(d.get("pm")), _ptr(d.get("ps")), s)
        )

    def set_order(self, predicted_cost=None):
        """Longest-expected-first processing order of the batch (``obca_set_order``): ``predicted_cost`` (B,) array or device
        tensor, e.g. the iteration counts of the single-vehicle solves behind the warm start; None restores 0..B-1."""
        if predicted_cost is None:
            self._check(self.lib.obca_set_order(self.handle, None, self._stream_ptr()))
            return
        cost = torch.as_tensor(predicted_cost, device=self.device)
        self._order = torch.argsort(cost, descending=True, stable=True).to(torch.int32).contiguous()
        self._check(self.lib.obca_set_order(self.handle, _ptr(self._order), self._stream_ptr()))

    def run(self):
        """Launch the batched interior-point solve on the current stream (asynchronous)."""
        self._check(self.lib.obca_solve(self.handle, self._stream_ptr()))

    def fetch_stats(self):
        B = self.B
        dev = self.device
        st = torch.empty(B, dtype=torch.int32, device=dev)
        it = torch.empty(B, dtype=torch.int32, device=dev)
        dbl = [torch.empty(B, dtype=torch.float64, device=dev) for _ in range(5)]  # obj, cviol, dual_inf, compl_inf, elastic
        self._check(self.lib.obca_get_stats(self.handle, _ptr(st), _ptr(it), *[_ptr(t) for t in dbl], self._stream_ptr()))
        return st, it, dbl

    def fetch_history(self):
        """Device copies of the iteration record of the last solve: rows (B, history, 16) float64 and counts (B,) int32, or
        (None, None) when the solver does not record."""
        if self.opts.history <= 0:
            return None, None
        rows = torch.empty((self.B, self.opts.history, len(HIST_FIELDS)), dtype=torch.float64, device=self.device)
        cnt = torch.empty(self.B, dtype=torch.int32, device=self.device)
        self._check(self.lib.obca_get_history(self.handle, _ptr(rows), _ptr(cnt), self._stream_ptr()))
        return rows, cnt

    def fetch_solution(self):
        B, V, M, O, P = self.B, self.V, self.Mmax, self.O, self.P
        dev = self.device
        out = {
            "z": torch.empty((B, V, M, 7), dtype=torch.float64, device=dev),
            "lam": torch.empty((B, V, M, O, 4), dtype=torch.float64, device=dev),
            "mu": torch.empty((B, V, M, O, 4), dtype=torch.float64, device=dev),
            "dt": torch.empty((B,), dtype=torch.float64, device=dev),
        }
        if P:
            out["pl"] = torch.empty((B, P, M, 4), dtype=torch.float64, device=dev)
            out["pm"] = torch.empty((B, P, M, 4), dtype=torch.float64, device=dev)
            out["ps"] = torch.empty((B, P, M, 2), dtype=torch.float64, device=dev)
        self._check(
            self.lib.obca_get_solution(self.handle, _ptr(out["z"]), _ptr(out["lam"]), _ptr(out["mu"]), _ptr(out["dt"]), _ptr(out.get("pl")), _ptr(out.get("pm")), _ptr(out.get("ps")), self._stream_ptr())
        )
        return out

    # -- host-buffer API (the call a planner makes) ------------------------------------------------------
    def solve(self, guess: CollocationGuess, init_pose: Optional[np.ndarray] = None, want_duals: bool = True) -> BatchResult:
        """Host arrays in, host arrays out: H2D copies, batched solve, D2H copies."""
        d = self.upload(guess, init_pose)
        self.set_inputs(d)
        self.run()
        st, it, dbl = self.fetch_stats()
        sol = self.fetch_solution()
        hist, hcnt = self.fetch_history()
        h = self._to_host([st, it, dbl[0], dbl[1], dbl[2], dbl[3], sol["z"], sol["lam"] if want_duals else None, sol["mu"] if want_duals else None,
                           sol["dt"], sol.get("pl"), sol.get("pm"), sol.get("ps"), dbl[4], hist, hcnt])
        return BatchResult(status=h[0], iters=h[1], obj=h[2], cviol=h[3], dual_inf=h[4], compl_inf=h[5], elastic=h[13], z=h[6], lam=h[7], mu=h[8], dt=h[9],
                           pair_lam=h[10], pair_mu=h[11], pair_s=h[12], history=h[14], history_count=h[15])

    # -- introspection for the parity tests --------------------------------------------------------------
    def layout(self):
        buf = (ctypes.c_int64 * 40)()
        n = self._check(self.lib.obca_layout(self.handle, buf, 40))
        names = ["V", "O", "P", "Mv", "Nmax", "Smax", "nx", "ny", "oZ", "oLAM", "oMU", "oSD", "oEL", "oTS", "oPL", "oPM", "oPS", "oPSD", "oPSN", "oPEL", "oDT",
                 "oYINIT", "oYCOL", "oYCONT", "oYTERM", "oYOBS", "oYTUBE", "oYPAIR", "m_active", "nb"]
        assert n == len(names)
        return {k: int(buf[i]) for i, k in enumerate(names)}

    PHASES = ["eval_pairs", "eval_nodes", "pair_eliminate", "node_assemble", "nullspace", "cross", "riccati_bwd", "riccati_fwd",
              "expand+residual", "multipliers", "local_backsub", "ipm_vector_ops", "ric_assemble", "ric_products", "ric_cholesky", "ric_ksolve",
              "ns_setup", "ns_qr", "ns_tcols", "ns_store", "ns_project", "ipm_P1_errors", "ipm_P2_sigma", "ipm_P3_ftb", "ipm_P4_trial", "ipm_theta", "ipm_P5_accept", "ra_zero+prefetch", "ra_Tmaps+sync", "ra_passA", "ra_passB"]

    def debug_profile(self):
        buf = (ctypes.c_int64 * 31)()
        self._check(self.lib.obca_debug_profile(self.handle, buf, 31))
        return {k: int(buf[i]) for i, k in enumerate(self.PHASES)}

    def debug_get_iterate(self, b=0):
        L = self.layout()
        x, zL, zU = (np.zeros(L["nx"]) for _ in range(3))
        y = np.zeros(L["ny"])
        self._check(self.lib.obca_debug_get_iterate(self.handle, b, _np_ptr(x), _np_ptr(y), _np_ptr(zL), _np_ptr(zU)))
        return x, y, zL, zU

    def debug_set_iterate(self, b, x=None, y=None, zL=None, zU=None):
        arrs = [None if a is None else np.ascontiguousarray(a, dtype=np.float64) for a in (x, y, zL, zU)]
        self._check(self.lib.obca_debug_set_iterate(self.handle, b, *[None if a is None else _np_ptr(a) for a in arrs]))

    def debug_eval(self, b=0):
        L = self.layout()
        c, gl, f = np.zeros(L["ny"]), np.zeros(L["nx"]), ctypes.c_double()
        self._check(self.lib.obca_debug_eval(self.handle, b, _np_ptr(c), _np_ptr(gl), ctypes.cast(ctypes.byref(f), _dp)))
        return c, gl, f.value

    def debug_kkt_apply(self, b, delta_w, dx, dy):
        """K [dx; dy] at the stored iterate (internal layout), applied matrix-free on the device (obca_refine.h)."""
        L = self.layout()
        r1, r2 = np.zeros(L["nx"]), np.zeros(L["ny"])
        dx, dy = np.ascontiguousarray(dx, dtype=np.float64), np.ascontiguousarray(dy, dtype=np.float64)
        self._check(self.lib.obca_debug_kkt_apply(self.handle, b, delta_w, _np_ptr(dx), _np_ptr(dy), _np_ptr(r1), _np_ptr(r2)))
        return r1, r2

    def debug_step(self, b, mu, delta_w):
        L = self.layout()
        dx, dy, ok = np.zeros(L["nx"]), np.zeros(L["ny"]), ctypes.c_int32()
        self._check(self.lib.obca_debug_step(self.handle, b, mu, delta_w, _np_ptr(dx), _np_ptr(dy), ctypes.byref(ok)))
        return dx, dy, int(ok.value)


class PipelinedSolver:
    """Consecutive batches of the SAME problem shape, double buffered: ``depth`` library handles on ``depth`` CUDA streams.

    One batch is one persistent ``k_solve`` launch (one CTA per SM pulling instances from a queue); its last wave leaves SMs idle
    (3.46 instances per SM at 512 instances: a fifth of the launch).  With the next batch already launched on another stream, its CTAs
    start on every SM the moment the previous batch's CTA retires, and its host<->device copies overlap the previous solve.  Nothing is
    shared between the handles (own iterates, work areas, queue counter); results are bit-identical to ``ObcaSolver.solve``.

    ``solve_many`` is the host-facing call (host arrays in, host arrays out, one worker thread per handle calling the ordinary
    ``ObcaSolver.solve`` on its stream); ``run_resident`` the device-resident one (inputs already in HBM)."""

    def __init__(self, prob: CollocationProblem, options: Optional[SolveOptions] = None, device="cuda:0", lib: Optional[ctypes.CDLL] = None, depth: int = 2,
                 first: Optional["ObcaSolver"] = None):
        if torch.device(device).type != "cuda":
            raise RuntimeError("PipelinedSolver needs a CUDA device (streams); there is no CPU fallback")
        if depth < 1:
            raise ValueError("PipelinedSolver: depth must be >= 1")
        self.solvers = [first if first is not None else ObcaSolver(prob, options, device=device, lib=lib)]
        self.solvers += [ObcaSolver(prob, options, device=device, lib=lib) for _ in range(depth - 1)]
        self.device = self.solvers[0].device
        self.streams = [torch.cuda.Stream(self.device) for _ in self.solvers]

    @property
    def launch_count(self):
        return sum(s.launch_count for s in self.solvers)

    def set_order(self, predicted_cost=None):
        for s in self.solvers:
            s.set_order(predicted_cost)
        torch.cuda.current_stream(self.device).synchronize()

    def run_resident(self, dev_inputs, steps: int):
        """``steps`` batches with device-resident inputs (the dict of ``ObcaSolver.upload``), alternating over the handles.  Asynchronous:
        returns the per-step (status, iters, [obj, cviol, dual_inf, compl_inf, elastic]) device tensors; the caller's current stream
        waits for all of them."""
        main = torch.cuda.current_stream(self.device)
        for st in self.streams:
            st.wait_stream(main)
        out = []
        for k in range(steps):
            sv, st = self.solvers[k % len(self.solvers)], self.streams[k % len(self.solvers)]
            with torch.cuda.stream(st):
                sv.set_inputs(dev_inputs)
                sv.run()
                out.append(sv.fetch_stats())
        for st in self.streams:
            main.wait_stream(st)
        return out

    def solve_many(self, guesses, want_duals: bool = True):
        """Host arrays in, host arrays out, for a list of batches: list of BatchResult in the order of ``guesses``."""
        import threading

        todo = list(enumerate(guesses))
        out = [None] * len(todo)
        lock = threading.Lock()
        err = []

        def worker(sv, st):
            try:
                torch.cuda.set_device(self.device)  # the current device is per thread
                with torch.cuda.stream(st):
                    while True:
                        with lock:
                            if not todo:
                                return
                            k, g = todo.pop(0)
                        out[k] = sv.solve(g, want_duals=want_duals)
            except BaseException as e:  # surfaced in the calling thread
                err.append(e)

        threads = [threading.Thread(target=worker, args=(sv, st)) for sv, st in zip(self.solvers, self.streams)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        if err:
            raise err[0]
        return out

    def close(self):
        for s in self.solvers:
            s.close()


# ---------------------------------------------------------------------------------------------------------------------
# MPC mode: the NLP of VehicleFollower.setup_controller / step (confrez/control/vehicle_follower.py:146-563)
# ---------------------------------------------------------------------------------------------------------------------
@dataclass
class MpcProblem:
    """Static data of the distributed-MPC controller: horizon, sample time, obstacles, body, limits (vehicle_follower.py:146-368)."""

    obs_A: np.ndarray  # (O,4,2)
    obs_b: np.ndarray  # (O,4)
    n_others: int
    N: int = 30
    dt: float = 0.1
    body_G: np.ndarray = None
    body_g: np.ndarray = None
    wb: float = 2.5
    region: np.ndarray = None
    limits: np.ndarray = None
    dmin: float = 0.05
    batch: int = 1

    def __post_init__(self):
        if self.body_G is None:
            self.body_G = np.array([[1.0, 0], [0, 1], [-1, 0], [0, -1]])
        if self.body_g is None:
            self.body_g = np.array([3.3, 0.9, 0.6, 0.9])
        if self.region is None:
            self.region = np.array([2.5, 32.5, 7.5, 27.5])
        if self.limits is None:
            self.limits = np.array([-2.5, 2.5, -0.85, 0.85, -1.5, 1.5, -1.0, 1.0])


class ObcaMpcSolver(ObcaSolver):
    """One handle per controller shape; ``batch`` instances (e.g. the vehicles of one scene) are solved in one launch."""

    def __init__(self, prob: MpcProblem, options: Optional[SolveOptions] = None, device="cuda:0", lib: Optional[ctypes.CDLL] = None):
        self.lib = lib if lib is not None else load_library()
        self.device = torch.device(device)
        self.is_emulation = b"EMULATION" in self.lib.obca_version()
        if self.device.type != "cuda" and not self.is_emulation:
            raise RuntimeError("ObcaMpcSolver needs a CUDA device (no CPU fallback)")
        if self.device.type == "cuda" and not torch.cuda.is_available():
            raise RuntimeError("ObcaMpcSolver: CUDA is not available on this machine (no CPU fallback)")
        self.prob = prob
        self._staging = {}
        self.opts = options or SolveOptions(max_iter=600)  # vehicle_follower.py:362-364
        self.B, self.V, self.O, self.P, self.Mmax = prob.batch, 1, prob.obs_A.shape[0], prob.n_others, prob.N
        dims = ObcaDims(batch=self.B, V=1, O=self.O, K=5, n_per_set=1, mode=1, horizon=prob.N, n_others=prob.n_others)
        copts = ObcaOptions()
        self.lib.obca_default_options(ctypes.byref(copts))
        for name in ("tol", "constr_viol_tol", "dual_inf_tol", "compl_inf_tol", "mu_init", "max_iter", "elastic_weight", "refine_steps"):
            setattr(copts, name, getattr(self.opts, name))
        copts.dmin = prob.dmin
        self.handle = ctypes.c_void_p()
        dev_index = self.device.index or 0 if self.device.type == "cuda" else 0
        self._check(self.lib.obca_create(ctypes.byref(dims), ctypes.byref(copts), dev_index, ctypes.byref(self.handle)))
        keep = {n: np.ascontiguousarray(getattr(prob, n), dtype=np.float64) for n in ("obs_A", "obs_b", "body_G", "body_g", "region", "limits")}
        st = ObcaStatic(wb=float(prob.wb), mpc_dt=float(prob.dt), **{n: _np_ptr(a) for n, a in keep.items()})
        self._check(self.lib.obca_set_static(self.handle, ctypes.byref(st)))
        self._set_history()

    def upload_params(self, cur, ref, others):
        B, N, P = self.B, self.Mmax, self.P
        d = {"cur": self._to_dev(cur, (B, 5), "cur"), "ref": self._to_dev(ref, (B, N, 3), "ref")}
        d["others"] = self._to_dev(others, (B, P, N, 3), "others") if P else None
        return d

    def set_params(self, d):
        self._check(self.lib.obca_set_mpc_params(self.handle, _ptr(d["cur"]), _ptr(d["ref"]), _ptr(d.get("others")), self._stream_ptr()))

    def upload(self, guess: CollocationGuess, init_pose=None):
        B, M, O, P = self.B, self.Mmax, self.O, self.P
        d = {
            "z": self._to_dev(guess.z, (B, 1, M, 7), "z"),
            "lam": self._to_dev(guess.lam, (B, 1, M, O, 4), "lam"),
            "mu": self._to_dev(guess.mu, (B, 1, M, O, 4), "mu"),
            "dt": self._to_dev(np.zeros(B), (B,), "dt"),
        }
        if P:
            d["pl"] = self._to_dev(guess.pair_lam, (B, P, M, 4), "pl")
            d["pm"] = self._to_dev(guess.pair_mu, (B, P, M, 4), "pm")
            d["ps"] = self._to_dev(guess.pair_s, (B, P, M, 2), "ps")
        return d

    def set_inputs(self, d):
        self._check(
            self.lib.obca_set_initial(self.handle, _ptr(d["z"]), _ptr(d["lam"]), _ptr(d["mu"]), _ptr(d["dt"]), _ptr(d.get("pl")), _ptr(d.get("pm")), _ptr(d.get("ps")), self._stream_ptr())
        )

    def solve_step(self, cur, ref, others, guess: CollocationGuess) -> BatchResult:
        """One MPC solve for every instance: parameters + warm start in (host), solution out (host)."""
        self.set_params(self.upload_params(cur, ref, others))
        return ObcaSolver.solve(self, guess)

    def solve(self, guess, init_pose=None, want_duals=True):  # parameters must have been set with set_params
        return ObcaSolver.solve(self, guess, want_duals=want_duals)


# ---------------------------------------------------------------------------------------------------------------------
# State warm start: the Euler-discretised tube-following NLP of Vehicle.state_ws (confrez/control/vehicle.py:99-231)
# ---------------------------------------------------------------------------------------------------------------------
@dataclass
class StateWsProblem:
    """Static data of ``Vehicle.state_ws``: ``n_sets`` strategy sets, ``N`` Euler steps of ``dt`` per move, tube sets (raw b; the
    solver subtracts ``shrink_tube``), optional final heading, ``bounded_input`` (vehicle.py:99-108)."""

    tube_A: np.ndarray  # (S,2,4,2) [set][back,front][row][x,y]
    tube_b: np.ndarray  # (S,2,4)
    N: int = 30
    dt: float = 0.1
    final_heading: Optional[float] = None
    bounded_input: bool = False
    shrink_tube: float = 0.8
    wb: float = 2.5
    region: np.ndarray = None
    limits: np.ndarray = None
    batch: int = 1

    def __post_init__(self):
        if self.region is None:
            self.region = np.array([2.5, 32.5, 7.5, 27.5])
        if self.limits is None:
            self.limits = np.array([-2.5, 2.5, -0.85, 0.85, -1.5, 1.5, -1.0, 1.0])

    @property
    def n_sets(self):
        return int(np.asarray(self.tube_A).shape[0])

    @property
    def nodes(self):
        return self.N * (self.n_sets - 1) + 1


class ObcaStateWsSolver(ObcaMpcSolver):
    """``batch`` state warm starts of one vehicle shape (same tube, different initial poses) in one launch.  The NLP runs through
    the MPC-mode kernels (stage-wise Riccati over the N (S - 1) + 1 nodes); ``solve_ws`` takes the initial states (B,5) and the
    node-major guess z (B,nodes,7) = (x, y, psi, v, delta, a, w)."""

    def __init__(self, prob: StateWsProblem, options: Optional[SolveOptions] = None, device="cuda:0", lib: Optional[ctypes.CDLL] = None):
        self.lib = lib if lib is not None else load_library()
        self.device = torch.device(device)
        self.is_emulation = b"EMULATION" in self.lib.obca_version()
        if self.device.type != "cuda" and not self.is_emulation:
            raise RuntimeError("ObcaStateWsSolver needs a CUDA device (no CPU fallback)")
        if self.device.type == "cuda" and not torch.cuda.is_available():
            raise RuntimeError("ObcaStateWsSolver: CUDA is not available on this machine (no CPU fallback)")
        self.prob = prob
        self._staging = {}
        self.opts = options or SolveOptions(max_iter=500)  # vehicle.py:207-213
        self.B, self.V, self.O, self.P, self.Mmax = prob.batch, 1, 0, 0, prob.nodes
        dims = ObcaDims(batch=self.B, V=1, O=0, K=5, n_per_set=prob.N, mode=2, horizon=prob.nodes, n_others=0, bounded_input=int(bool(prob.bounded_input)))
        dims.n_sets[0] = prob.n_sets
        copts = ObcaOptions()
        self.lib.obca_default_options(ctypes.byref(copts))
        for name in ("tol", "constr_viol_tol", "dual_inf_tol", "compl_inf_tol", "mu_init", "max_iter", "elastic_weight", "refine_steps"):
            setattr(copts, name, getattr(self.opts, name))
        copts.shrink_tube = float(prob.shrink_tube)
        self.handle = ctypes.c_void_p()
        dev_index = self.device.index or 0 if self.device.type == "cuda" else 0
        self._check(self.lib.obca_create(ctypes.byref(dims), ctypes.byref(copts), dev_index, ctypes.byref(self.handle)))
        S = prob.n_sets
        keep = {
            "obs_A": np.zeros((1, 4, 2)), "obs_b": np.zeros((1, 4)), "body_G": np.array([[1.0, 0], [0, 1], [-1, 0], [0, -1]]), "body_g": np.array([3.3, 0.9, 0.6, 0.9]),
            "tube_A": np.ascontiguousarray(prob.tube_A, dtype=np.float64).reshape(1, S, 2, 4, 2), "tube_b": np.ascontiguousarray(prob.tube_b, dtype=np.float64).reshape(1, S, 2, 4),
            "region": np.ascontiguousarray(prob.region, dtype=np.float64), "limits": np.ascontiguousarray(prob.limits, dtype=np.float64),
            "final_heading": np.array([np.nan if prob.final_heading is None else float(prob.final_heading)]),
        }
        self._keep = keep
        st = ObcaStatic(wb=float(prob.wb), mpc_dt=float(prob.dt), **{n: _np_ptr(a) for n, a in keep.items()})
        self._check(self.lib.obca_set_static(self.handle, ctypes.byref(st)))
        self._set_history()

    def solve_ws(self, init_state, z_guess) -> BatchResult:
        B, M = self.B, self.Mmax
        init_state = np.ascontiguousarray(init_state, dtype=np.float64).reshape(B, 5)
        z = np.ascontiguousarray(z_guess, dtype=np.float64).reshape(B, 1, M, 7)
        guess = CollocationGuess(z, np.zeros((B, 1, M, 0, 4)), np.zeros((B, 1, M, 0, 4)), np.zeros(B))
        return self.solve_step(init_state, np.zeros((B, M, 3)), None, guess)
