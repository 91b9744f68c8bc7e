"""The device Newton step and inertia decision at every stage shape the structured KKT solve (csrc/obca_kkt.h) specialises on.

The Riccati stage factorisation picks its code by shape.  With nu free directions (about 5 per vehicle still in its horizon)
and nX = 7 V + 1 stage states (poses and dt), ``stage_ldl_fused`` runs ``cta_stage_ldl<LOG2CG, KMAX>``:
  * nu + nX + 1 <= 64:  <6,2> (nu <= 8), <6,4> (<= 16), <6,6> (<= 24), <6,8> (<= 32);
  * above:              <7,16> (nu <= 32), <7,24> (<= 48), <7,32> (<= 64).
For more than four vehicles the stage matrices no longer fit shared memory and the Riccati phase runs from the per-slot
global-memory arena (``riccati_backward<false>``, ``W.ricg``).  The host emulation takes neither path (it factorises with
``stage_ldl_scalar`` in its shared arena), so these cases pin the device against the oracle's assembled K (tests/cases.py):
  * ``ok`` (inertia (n, m, 0), which decides the delta_w escalation of every iteration) equals the negative pivot count
    of a symmetric LDL' of K;
  * where ok = 1, the step's residual in K is at rounding level in every row, collocation rows included;
  * where the oracle's own LU step has a residual at rounding level too (K numerically nonsingular), the two steps agree.
``riccati_factor_generic`` is not reached on the device: nu <= 8 V <= 64 and nu + nX + 1 <= 64 + 58 always pass
``ldl_fast_shape``.  ``<7,32>`` (nu > 48, more than six free directions per vehicle on average at one stage) is not reached
by any case here: it needs rank loss in most of eight vehicles' collocation blocks at the same stage.
"""
import numpy as np
import pytest

from cases import kkt_inertia_ok, kkt_residual, kkt_system, oracle_newton_step
from conftest import make_case
from layout_map import build_maps
from test_mpc import mpc_case  # noqa: F401  (fixture)

from conflict_rez_b200.solver import ObcaSolver, SolveOptions

BACKENDS = [pytest.param("emu", id="emu"), pytest.param("cuda", id="cuda", marks=pytest.mark.gpu)]
AGENTS4 = ("vehicle_0", "vehicle_1", "vehicle_2", "vehicle_3")
STEP_TOL = 1e-10  # residual of the device step relative to |rhs|; the emulation measures 2e-13 .. 6e-13 at the initial point
FWD_TOL = 1e-7  # forward error against a trustworthy oracle step, as in test_parity.py


@pytest.fixture(params=BACKENDS)
def backend(request):
    if request.param == "emu":
        return request.getfixturevalue("emu_lib"), "cpu"
    return request.getfixturevalue("cuda_lib"), "cuda:0"


def _replicated(strategy_file, agents, copies, shift, **kw):
    """``copies`` lots of ``agents`` side by side (``replicate_problem``) with a host-built guess: the single lot's pose guess
    tiled and translated, the duals of all obstacles and pairs from the closed-form warm starts."""
    from conflict_rez_b200.control import warmstart
    from conflict_rez_b200.control.batch_planner import replicate_problem
    from conflict_rez_b200.problem import CollocationGuess

    base, g = make_case(strategy_file, agents, **kw)
    prob = replicate_problem(base, copies, (shift, 0.0))
    V, M = prob.V, int(prob.nodes.max())
    z = np.concatenate([g.z + np.array([c * shift, 0, 0, 0, 0, 0, 0]) for c in range(copies)], axis=0)
    lam, mu = np.zeros((V, M, prob.O, 4)), np.zeros((V, M, prob.O, 4))
    for a in range(V):
        m = int(prob.nodes[a])
        lam[a, :m], mu[a, :m] = warmstart.dual_ws_rect(z[a, :m, 0], z[a, :m, 1], z[a, :m, 2], prob.obs_A, prob.obs_b, prob.body_G, prob.body_g)
    P = len(prob.pairs)
    pl, pm, ps = np.zeros((P, M, 4)), np.zeros((P, M, 4)), np.zeros((P, M, 2))
    for q, (a, b) in enumerate(prob.pairs):
        m = int(min(prob.nodes[a], prob.nodes[b]))
        pl[q, :m], pm[q, :m], ps[q, :m] = warmstart.joint_dual_ws_rect(z[a, :m, 0], z[a, :m, 1], z[a, :m, 2], z[b, :m, 0], z[b, :m, 1], z[b, :m, 2],
                                                                       prob.body_G, prob.body_g)
    return prob, CollocationGuess(z, lam, mu, g.dt, pl, pm, ps)


def case_v4_headline(fn):
    """The benchmarked instance: vehicles 0-3, default n_per_set.  Stage shape (20, 29): <6,6>, shared-memory arena.
    vehicle_0's final approach over-collocates k = 0, so K is singular: residual and inertia checks only."""
    return make_case(fn, AGENTS4)


def case_v4_o32(fn):
    """Vehicles 0-3 with 26 seeded extra rectangles: O = 32 = OBCA_MAX_O, the largest obstacle count the ABI accepts.
    Stage shape (20, 29): <6,6>, shared-memory arena."""
    from conflict_rez_b200.control.scenario import random_obstacles

    return make_case(fn, AGENTS4, obstacles=random_obstacles(fn, 26, seed=7), n_per_set=2)


def case_v5(fn):
    """Five lots of vehicle_1 (35 m apart), n_per_set = 2.  Stage shape (25, 36): nu + nX + 1 = 62, <6,8>, global arena."""
    return _replicated(fn, ("vehicle_1",), 5, 35.0, n_per_set=2)


def case_v6(fn):
    """Two lots of vehicles 1-3 (35 m apart), n_per_set = 2.  Stage shape (30, 43): <7,16>, global arena."""
    return _replicated(fn, ("vehicle_1", "vehicle_2", "vehicle_3"), 2, 35.0, n_per_set=2)


def case_v6_ragged(fn):
    """Three lots of vehicles 1 and 2 (35 m apart), whose horizons differ: nu = 30 (<7,16>) while all six vehicles are in
    their horizons, nu = 15 (<6,4>) at the late stages of the longer vehicle -- both LOG2CG families in one factorisation
    and the zero fill of the finished blocks in ``ric_input_fetch``.  Global arena."""
    return _replicated(fn, ("vehicle_1", "vehicle_2"), 3, 35.0, n_per_set=2)


def case_v8_near(fn):
    """Two lots of vehicles 0-3 only 1.5 m apart: vehicles of different lots interact (active cross-lot pair blocks).
    Stage shape (40, 57): <7,24>, global arena."""
    return _replicated(fn, AGENTS4, 2, 1.5, n_per_set=2)


def case_v8_far(fn):
    """Two lots of vehicles 0-3, 35 m apart (non-interacting lots).  Stage shape (40, 57): <7,24>, global arena."""
    return _replicated(fn, AGENTS4, 2, 35.0, n_per_set=2)


CASES = {f.__name__[5:]: f for f in (case_v4_headline, case_v4_o32, case_v5, case_v6, case_v6_ragged, case_v8_near, case_v8_far)}


@pytest.fixture(scope="module")
def built(strategy_file):
    """(problem, guess, oracle NLP) per case, built once per module."""
    from oracle.nlp import CollocationNLP

    cache = {}

    def get(name):
        if name not in cache:
            prob, guess = CASES[name](strategy_file)
            cache[name] = (prob, guess, CollocationNLP(prob))
        return cache[name]

    return get


def _check_step(sv, nlp, ix, iy, x, y, zL, zU, mu, dw, forward=True, tol=STEP_TOL, backward=False):
    """Inertia, residual and (where the oracle step is trustworthy) forward error of the device step at the stored iterate."""
    dx, dy, ok = sv.debug_step(0, mu, dw)
    assert ok == int(kkt_inertia_ok(nlp, x, y, zL, zU, mu, dw)), (ok, dw)
    if not ok:
        return "dw %.0e: ok = 0 (agrees with the pivot count)" % dw
    rows, r1, r2 = kkt_residual(nlp, x, y, zL, zU, mu, dw, dx[ix], dy[iy], backward=backward)
    cols = np.concatenate([r.ravel() for r in nlp.r_col])
    assert r1 <= tol and r2 <= tol, (dw, r1, r2)
    assert rows[nlp.n + cols].max() <= tol  # the collocation rows, where the implied and dropped rows of [NULLSP] act
    msg = "dw %.0e: ok = 1, %s r1 %.1e r2 %.1e" % (dw, "backward error" if backward else "residual", r1, r2)
    if forward:
        dxo, dyo, _, _, (_, o1, o2) = oracle_newton_step(nlp, x, y, zL, zU, mu, dw)
        if max(o1, o2) <= STEP_TOL:  # K numerically nonsingular: the step is unique
            ex, ey = np.abs(dx[ix] - dxo).max() / np.abs(dxo).max(), np.abs(dy[iy] - dyo).max() / np.abs(dyo).max()
            assert ex <= FWD_TOL and ey <= FWD_TOL, (dw, ex, ey)
            msg += ", forward error dx %.1e dy %.1e" % (ex, ey)
        else:
            msg += ", oracle LU residual %.1e: K singular, no forward comparison" % max(o1, o2)
    return msg


@pytest.mark.parametrize("name", list(CASES))
def test_newton_step_and_inertia_at_the_initial_point(backend, built, name):
    """At the solver's own initial point with y = 0.3 N(0, 1), mu = 0.1 and delta_w in {1e-3, 10} (test_parity.py's recipe)."""
    from oracle import ipm

    lib, dev = backend
    prob, guess, nlp = built(name)
    sv = ObcaSolver(prob, SolveOptions(max_iter=0), device=dev, lib=lib)
    sv.solve(guess)
    L = sv.layout()
    assert L["m_active"] == nlp.m
    ix, iy = build_maps(L, nlp)
    xd, _, zLd, zUd = sv.debug_get_iterate(0)
    x0 = ipm.push_into_bounds(nlp.init_slacks(nlp.pack(guess)), nlp.xL, nlp.xU, 1e-2, 1e-2)
    assert np.allclose(xd[ix], x0, rtol=0, atol=1e-10)
    y = 0.3 * np.random.default_rng(5).standard_normal(nlp.m)
    yd = np.zeros(L["ny"])
    yd[iy] = y
    sv.debug_set_iterate(0, y=yd)
    for dw in (1e-3, 10.0):
        print(name, _check_step(sv, nlp, ix, iy, x0, y, zLd[ix], zUd[ix], 0.1, dw))
    sv.close()


# Mid-solve the multipliers reach 1e8 on nearly dependent collocation rows.  Without iterative refinement (off at the default
# tol = 1e-2) the emulation's backward error reaches 7.8e-10 (8 vehicles, delta_w = 1e4, a pose row of vehicle_0; 4.7e-15 with two
# refinement steps) and stays below 3e-12 at delta_w <= 10.  The bound leaves a margin of 13 for the device's other summation
# order (fused multiply-adds, the CTA-parallel elimination); a wrong term in the factorisation leaves residuals of order 1.
MIDSOLVE_TOL = 1e-8


@pytest.mark.parametrize("name", ["v4_headline", "v8_far"])
def test_newton_step_and_inertia_mid_solve(backend, built, name):
    """After 15 interior-point iterations (Sigma spread over many decades): backward error and inertia of the device step.
    The ABI does not export the solver's mu; the mean complementarity of the read-back iterate stands in for it."""
    lib, dev = backend
    prob, guess, nlp = built(name)
    sv = ObcaSolver(prob, SolveOptions(max_iter=15), device=dev, lib=lib)
    sv.solve(guess)
    L = sv.layout()
    ix, iy = build_maps(L, nlp)
    xd, yd, zLd, zUd = sv.debug_get_iterate(0)
    x, y, zL, zU = xd[ix], yd[iy], zLd[ix], zUd[ix]
    hasL, hasU = np.isfinite(nlp.xL), np.isfinite(nlp.xU)
    mu = (np.sum(zL[hasL] * (x - nlp.xL)[hasL]) + np.sum(zU[hasU] * (nlp.xU - x)[hasU])) / (hasL.sum() + hasU.sum())
    for dw in (1e-3, 10.0, 1e4):  # the 4-vehicle iterate only passes the inertia test at 1e4
        print(name, "mu %.2e" % mu, _check_step(sv, nlp, ix, iy, x, y, zL, zU, mu, dw, forward=False, tol=MIDSOLVE_TOL, backward=True))
    sv.close()


def test_inertia_count_matches_dense_eigenvalues(strategy_file):
    """``kkt_inertia_ok``'s pivot count against numpy.linalg.eigvalsh of the same (delta_c-shifted) K on a tiny instance
    (one vehicle, one interval per move, two moves: n + m ~ 2 000), at a positive definite and at an indefinite delta_w."""
    from oracle import ipm
    from oracle.nlp import CollocationNLP

    prob, guess = make_case(strategy_file, ("vehicle_1",), n_per_set=1)
    nlp = CollocationNLP(prob)
    assert nlp.n + nlp.m < 5000
    x = ipm.push_into_bounds(nlp.init_slacks(nlp.pack(guess)), nlp.xL, nlp.xU, 1e-2, 1e-2)
    rng = np.random.default_rng(1)
    y = 0.3 * rng.standard_normal(nlp.m)
    zL, zU = np.where(np.isfinite(nlp.xL), 0.1, 0.0), np.where(np.isfinite(nlp.xU), 0.1, 0.0)
    seen = set()
    for dw in (1e-3, 10.0, -5.0, -50.0):
        K, _, _, _ = kkt_system(nlp, x, y, zL, zU, 0.1, dw)
        Kd = K.toarray()
        d2 = np.diag(Kd)[nlp.n :].copy()
        Kd[nlp.n :, nlp.n :] -= np.diag(np.where(d2 == 0.0, 1e-10, 0.0))
        ev = np.linalg.eigvalsh(Kd)
        neg = int((ev < 0).sum())
        assert np.abs(ev).min() > 1e-6  # no eigenvalue near the shift: the count is well defined
        assert kkt_inertia_ok(nlp, x, y, zL, zU, 0.1, dw) == (neg == nlp.m), (dw, neg, nlp.m)
        seen.add(neg == nlp.m)
    assert seen == {True, False}  # both answers were exercised


@pytest.mark.gpu
def test_global_arena_slots_are_independent(cuda_lib, strategy_file, built):
    """V = 6 (global-memory Riccati arena) with B = 2 * SMs + 3 distinct initial poses: every slot of the arena is reused by
    another instance while other CTAs still run.  Instances solved alone reproduce their batch results bit for bit, and so
    does another processing order of the batch (``obca_set_order``)."""
    import dataclasses

    import torch

    from conflict_rez_b200.control.batch_planner import random_init_offsets
    from conflict_rez_b200.problem import CollocationGuess

    prob1, g1, _ = built("v6")
    B = 2 * torch.cuda.get_device_properties(0).multi_processor_count + 3
    prob = dataclasses.replace(prob1, init_pose=prob1.init_pose[None] + random_init_offsets(B, prob1.V, seed=2))
    tile = lambda a: np.broadcast_to(a, (B,) + a.shape).copy()
    guess = CollocationGuess(tile(g1.z), tile(g1.lam), tile(g1.mu), np.full(B, float(g1.dt)), tile(g1.pair_lam), tile(g1.pair_mu), tile(g1.pair_s))
    opts = SolveOptions(max_iter=40)
    sv = ObcaSolver(prob, opts, device="cuda:0", lib=cuda_lib)
    r = sv.solve(guess)
    assert (r.iters > 0).all()
    sv.set_order(np.random.default_rng(3).permutation(B).astype(float))
    rp = sv.solve(guess)
    sv.close()
    assert np.array_equal(r.z, rp.z) and np.array_equal(r.iters, rp.iters) and np.array_equal(r.obj, rp.obj)
    for b in (0, B // 2, B - 1):
        s1 = ObcaSolver(prob.instance(b), opts, device="cuda:0", lib=cuda_lib)
        rb = s1.solve(guess.instance(b))
        s1.close()
        assert np.array_equal(rb.z[0], r.z[b]) and rb.iters[0] == r.iters[b] and rb.obj[0] == r.obj[b], b
    print("B = %d, iterations %d .. %d, status" % (B, r.iters.min(), r.iters.max()), np.unique(r.status, return_counts=True))


@pytest.mark.parametrize("n_others", [0, 3, 7])
def test_mpc_newton_step_with_n_neighbours(backend, mpc_case, n_others):
    """MPC-mode step parity beyond one neighbour: n_others = 0 takes the NULL pair-pointer path, 3 is what the device MPC
    loop runs, 7 the most the ABI accepts.  The neighbours are vehicle_2's prediction translated by a few metres each."""
    from test_mpc import _guess, _maps, _solver

    from conflict_rez_b200.control import warmstart
    from oracle import ipm
    from oracle.mpc import MpcNLP

    p0, par0, g0 = mpc_case
    z1, z2 = g0["z"], par0["others"][0]
    others = np.stack([z2 + np.array([0.6 * j, -0.4 * j, 0.0]) for j in range(n_others)]) if n_others else np.zeros((0, p0["N"], 3))
    p, par = dict(p0, n_others=n_others), dict(par0, others=others)
    pd = [warmstart.joint_dual_ws_rect(z1[:, 0], z1[:, 1], z1[:, 2], o[:, 0], o[:, 1], o[:, 2], p["body_G"], p["body_g"]) for o in others]
    N = p["N"]
    g = dict(g0, pl=np.array([d[0] for d in pd]).reshape(n_others, N, 4), pm=np.array([d[1] for d in pd]).reshape(n_others, N, 4),
             ps=np.array([d[2] for d in pd]).reshape(n_others, N, 2))
    nlp = MpcNLP(p, par)
    sv = _solver(backend, p, max_iter=0)
    sv.set_params(sv.upload_params(par["cur"][None], par["ref"][None], others[None]))
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
    for dw in (1e-3, 10.0):
        dx_o, dy_o, _, _, (_, o1, o2) = oracle_newton_step(nlp, x0, y, zLd[ix], zUd[ix], 0.1, dw)
        assert max(o1, o2) <= STEP_TOL  # the MPC system is nonsingular: the reference step is trustworthy
        dx_d, dy_d, ok = sv.debug_step(0, 0.1, dw)
        assert ok == int(kkt_inertia_ok(nlp, x0, y, zLd[ix], zUd[ix], 0.1, dw))
        if ok:
            assert np.abs(dx_d[ix] - dx_o).max() <= 1e-8 * np.abs(dx_o).max() and np.abs(dy_d[iy] - dy_o).max() <= 1e-8 * np.abs(dy_o).max()
        print("n_others %d dw %.0e ok %d" % (n_others, dw, ok))
    sv.close()
