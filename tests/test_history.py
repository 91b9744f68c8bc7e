"""Iteration record (obca_set_history / obca_get_history, SolveOptions.history): off by default, bit-identical results with it
on, consistent bookkeeping, the oracle's per-iteration history reproduced row by row, and the CasADi-style stats()["iterations"]."""
import numpy as np
import pytest

from cases import load_golden
from conftest import make_case
from test_mpc import _guess as _mpc_guess
from test_mpc import mpc_case  # noqa: F401  (module fixture)
from test_state_ws import _case as _ws_case

from conflict_rez_b200.solver import (HIST_F_RESET, HIST_FIELDS, HIST_STEP_FIELDS, MpcProblem, ObcaMpcSolver, ObcaSolver, ObcaStateWsSolver,
                                      SolveOptions, format_history)
from oracle import ipm

BACKENDS = [pytest.param("emu", id="emu"), pytest.param("cuda", id="cuda", marks=pytest.mark.gpu)]
F = {n: k for k, n in enumerate(HIST_FIELDS)}
OFFSETS = np.array([[[0, 0, 0], [0, 0, 0]], [[0.1, -0.1, 0.05], [0, 0.1, 0]], [[-0.1, 0.1, 0], [0.05, 0, -0.05]], [[0.0, 0.15, 0.0], [-0.1, 0, 0]]])


@pytest.fixture(params=BACKENDS)
def backend(request):
    if request.param == "emu":
        return request.getfixturevalue("emu_lib"), "cpu"
    return request.getfixturevalue("cuda_lib"), "cuda:0"


@pytest.fixture(scope="module")
def joint_case(strategy_file):
    return make_case(strategy_file, ("vehicle_1", "vehicle_2"), init_offsets=OFFSETS)


def _assert_same_results(a, b):
    for k in ("status", "iters", "obj", "cviol", "dual_inf", "compl_inf", "elastic", "z", "lam", "mu", "dt", "pair_lam", "pair_mu", "pair_s"):
        x, y = getattr(a, k), getattr(b, k)
        assert (x is None) == (y is None), k
        if x is not None:
            assert np.array_equal(x, y), k


def _assert_close_results(a, b):
    """MPC mode sums the objective over task units that the warps of a CTA pull from a shared counter, so its last bits depend
    on warp timing with or without the record: same status and iterations, values equal to rounding."""
    assert np.array_equal(a.status, b.status) and np.array_equal(a.iters, b.iters)
    for k in ("obj", "cviol", "dual_inf", "compl_inf", "elastic", "z", "lam", "mu", "pair_lam", "pair_mu", "pair_s"):
        assert np.allclose(getattr(a, k), getattr(b, k), rtol=1e-10, atol=1e-12), k


def _check_bookkeeping(res):
    """Invariants of the record that hold for every solve."""
    B, cap, nf = res.history.shape
    assert nf == len(HIST_FIELDS) == 16 and res.history_count.shape == (B,)
    for b in range(B):
        n = int(res.history_count[b])
        rows = res.history[b, : min(n, cap)]
        assert np.isnan(res.history[b, min(n, cap):]).all()  # rows past the count read back as NaN
        if rows[:, F["attempt"]].max() == 0:  # single attempt
            assert n == int(res.iters[b]) + 1
            assert np.array_equal(rows[:, F["iter"]], np.arange(len(rows)))
        if n <= cap:
            assert np.isnan(rows[-1, HIST_STEP_FIELDS]).all()  # the terminating head takes no step
            if res.status[b] == 0 and res.elastic[b] == 0:
                last = rows[-1]
                assert last[F["obj"]] == res.obj[b] and last[F["inf_pr"]] == res.cviol[b]
                assert last[F["inf_du"]] == res.dual_inf[b] and last[F["compl"]] == res.compl_inf[b]
        mu = rows[:, F["mu"]]
        for k in range(1, len(rows)):
            if mu[k] > mu[k - 1]:
                assert int(rows[k - 1, F["flags"]]) & HIST_F_RESET, (b, k)


def test_off_means_off(backend, joint_case):
    lib, dev = backend
    prob, guess = joint_case
    sv = ObcaSolver(prob, SolveOptions(), device=dev, lib=lib)
    res = sv.solve(guess)
    assert res.history is None and res.history_count is None
    assert sv.lib.obca_get_history(sv.handle, None, None, None) < 0
    assert b"recording is off" in sv.lib.obca_last_error()
    assert sv.lib.obca_set_history(sv.handle, -1) < 0
    assert b"capacity" in sv.lib.obca_last_error()
    sv.close()
    with pytest.raises(RuntimeError, match="capacity"):
        ObcaSolver(prob, SolveOptions(history=-3), device=dev, lib=lib)


def test_joint_batch_bit_identical_and_bookkeeping(backend, joint_case):
    lib, dev = backend
    prob, guess = joint_case
    assert prob.batch >= 4
    off = ObcaSolver(prob, SolveOptions(), device=dev, lib=lib).solve(guess)
    sv = ObcaSolver(prob, SolveOptions(history=400), device=dev, lib=lib)
    on = sv.solve(guess)
    _assert_same_results(off, on)
    assert (on.status == 0).all()
    _check_bookkeeping(on)
    assert "objective" in format_history(on, 1)
    sv.close()
    # capacity 5: the same count, the first five rows of the full record
    small = ObcaSolver(prob, SolveOptions(history=5), device=dev, lib=lib).solve(guess)
    _assert_same_results(off, small)
    assert np.array_equal(small.history_count, on.history_count)
    assert np.array_equal(small.history, on.history[:, :5], equal_nan=True)
    assert "more iterations past the capacity" in format_history(small, 0)


def _compare_with_oracle(rows, hist):
    """First 8 rows (or all, if fewer) of the device record against the oracle's ``hist``."""
    n = min(8, len(hist), len(rows))
    assert n >= 2
    for k in range(n):
        r, h = rows[k], hist[k]
        assert abs(r[F["mu"]] - h["mu"]) <= 1e-14 * h["mu"], k  # mu^1.5 of the device's pow and numpy's may differ in the last bit
        assert abs(r[F["obj"]] - h["f"]) <= 1e-9 * abs(h["f"]), k
        for fd, fo in (("theta", "theta"), ("inf_pr", "cviol"), ("inf_du", "dual_inf")):
            assert abs(r[F[fd]] - h[fo]) <= 1e-6 * max(1.0, abs(h[fo])), (k, fd, r[F[fd]], h[fo])
        if "alpha" in h:
            for fd, fo in (("alpha_pr", "alpha"), ("alpha_du", "alpha_du"), ("reg", "dw_used")):
                assert abs(r[F[fd]] - h[fo]) <= 1e-6, (k, fd, r[F[fd]], h[fo])


def test_state_ws_matches_oracle_history(backend, strategy_file):
    lib, dev = backend
    p, cur, z0, (nlp,) = _ws_case(strategy_file, "vehicle_1")
    out = {}
    for h in (0, 64):
        sv = ObcaStateWsSolver(p, SolveOptions(tol=1e-8, constr_viol_tol=1e-8, max_iter=500, history=h), device=dev, lib=lib)
        out[h] = sv.solve_ws(cur, z0)
        sv.close()
    _assert_same_results(out[0], out[64])
    res = out[64]
    _check_bookkeeping(res)
    ref = ipm.solve(nlp, nlp.init_slacks(nlp.pack(z0[0, :, :5], z0[0, :-1, 5:])), ipm.IpmOptions(tol=1e-8, constr_viol_tol=1e-8, max_iter=500))
    _compare_with_oracle(res.history[0], ref.history)


def test_mpc_step_matches_oracle_history(backend, mpc_case):  # noqa: F811
    from oracle.mpc import MpcNLP

    lib, dev = backend
    p, par, g = mpc_case
    mp = MpcProblem(obs_A=p["obs_A"], obs_b=p["obs_b"], n_others=p["n_others"], N=p["N"], dt=p["dt"])
    out = {}
    for h in (0, 64):
        sv = ObcaMpcSolver(mp, SolveOptions(tol=1e-8, constr_viol_tol=1e-8, max_iter=600, history=h), device=dev, lib=lib)
        out[h] = sv.solve_step(par["cur"][None], par["ref"][None], par["others"][None], _mpc_guess(g))
        sv.close()
    (_assert_same_results if dev == "cpu" else _assert_close_results)(out[0], out[64])
    res = out[64]
    _check_bookkeeping(res)
    assert (res.history[0, : res.history_count[0], F["rho"]] == 1e3).all()
    nlp = MpcNLP(p, par)
    ref = ipm.solve(nlp, nlp.init_slacks(nlp.pack(g["z"], g["lam"], g["mu"], g["pl"], g["pm"], g["ps"])), ipm.IpmOptions(tol=1e-8, constr_viol_tol=1e-8, max_iter=600))
    _compare_with_oracle(res.history[0], ref.history)


@pytest.mark.parametrize("name", ["single_vehicle_1", "joint_vehicle_1_2"])
def test_collocation_first_row_matches_oracle(backend, name):
    from oracle.nlp import CollocationNLP

    lib, dev = backend
    prob, guess, _ = load_golden(name)
    sv = ObcaSolver(prob, SolveOptions(max_iter=0, history=4), device=dev, lib=lib)
    res = sv.solve(guess)
    sv.close()
    assert int(res.history_count[0]) == 1
    nlp = CollocationNLP(prob)
    x0 = ipm.push_into_bounds(nlp.init_slacks(nlp.pack(guess)), nlp.xL, nlp.xU, 1e-2, 1e-2)
    c = nlp.c(x0)
    row = res.history[0, 0]
    for fd, want in (("obj", nlp.f(x0)), ("theta", np.abs(c).sum()), ("inf_pr", np.abs(c).max())):
        assert abs(row[F[fd]] - want) <= 1e-12 * abs(want), (fd, row[F[fd]], want)


def test_vehicle_stats_iterations(backend, strategy_file):
    from conflict_rez_b200.control.vehicle import Vehicle
    from conflict_rez_b200.pytypes import VehicleState

    lib, dev = backend
    v = Vehicle(rl_file_name=strategy_file, agent="vehicle_1", color={}, device=dev)
    v._lib = lib
    zu0 = v.state_ws(N=30, dt=0.1, init_offset=VehicleState(), final_heading=3 * np.pi / 2, shrink_tube=0.5, spline_ws=True)
    zu0 = v.interp_ws_for_collocation(v.dual_ws(zu0), K=5, N_per_set=5)
    v.setup_single_final_problem(zu0=zu0, init_offset=VehicleState(), final_heading=3 * np.pi / 2, K=5, N_per_set=5, shrink_tube=0.5)
    assert "iterations" not in v.solve_single_final_problem().stats()
    v.solve_options.history = 500
    st = v.solve_single_final_problem().stats()
    it = st["iterations"]
    assert set(it) == {"obj", "inf_pr", "inf_du", "mu", "d_norm", "regularization_size", "alpha_pr", "alpha_du", "ls_trials"}
    assert all(len(vals) == st["iter_count"] + 1 for vals in it.values())
    assert it["alpha_pr"][0] == 0 and it["ls_trials"][0] == 0 and all(a > 0 for a in it["alpha_pr"][1:])


@pytest.mark.gpu
def test_pipelined_histories_equal_serial(cuda_lib):
    from conflict_rez_b200.solver import PipelinedSolver

    prob, guess, _ = load_golden("joint_vehicle_1_2")
    opts = SolveOptions(tol=1e-6, constr_viol_tol=1e-6, history=200)
    g2 = type(guess)(guess.z + 1e-3, guess.lam, guess.mu, guess.dt, guess.pair_lam, guess.pair_mu, guess.pair_s)
    refs = [ObcaSolver(prob, opts, device="cuda:0", lib=cuda_lib).solve(g) for g in (guess, g2)]
    pipe = PipelinedSolver(prob, opts, device="cuda:0", lib=cuda_lib, depth=2)
    out = pipe.solve_many([guess, g2, guess, g2])
    for k, r in enumerate(out):
        want = refs[k % 2]
        assert np.array_equal(r.history_count, want.history_count)
        assert np.array_equal(r.history, want.history, equal_nan=True)
    pipe.close()
