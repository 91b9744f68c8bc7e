"""Independent checks of the Newton system and of returned points.

* ``kkt_apply`` (csrc/obca_refine.h) applies K = [[W + Sigma + dw, J'], [J, -dc]] matrix free on the device; it shares no code
  with the structured elimination and is compared here with the oracle's sparse matrix (sympy derivatives).
* Iterative refinement: the refined Newton step has a residual at rounding level in *every* row (the un-refined
  structured solve leaves ~1e-8 in the dt row, which is what kept tol = 1e-8 out of reach in round 1).
* KKT certificate of the UNMODIFIED reference NLP (oracle/reference_nlp.py: hard inequalities, no slack / elastic variables,
  no clipped multipliers, derivatives by torch.autograd) for every golden solution and for the solver's own output.
"""
import numpy as np
import pytest

from cases import DROPPED_ROW_TOL, kkt_residual, load_golden
from conftest import make_case
from layout_map import build_maps

from conflict_rez_b200.solver import ObcaSolver, SolveOptions

BACKENDS = [pytest.param("emu", id="emu"), pytest.param("cuda", id="cuda", marks=pytest.mark.gpu)]
GOLDEN = ["single_vehicle_1", "single_vehicle_2", "single_vehicle_2_free_heading", "joint_vehicle_1_2", "joint_vehicle_0_1_2_3"]


@pytest.fixture(params=BACKENDS)
def backend(request):
    if request.param == "emu":
        return request.getfixturevalue("emu_lib"), "cpu"
    return request.getfixturevalue("cuda_lib"), "cuda:0"


def _oracle_matrix(nlp, x, y, zL, zU, dw):
    import scipy.sparse as sp

    hasL, hasU = np.isfinite(nlp.xL), np.isfinite(nlp.xU)
    gL, gU = np.where(hasL, x - nlp.xL, 1.0), np.where(hasU, nlp.xU - x, 1.0)
    Sigma = np.where(hasL, zL / gL, 0.0) + np.where(hasU, zU / gU, 0.0)
    J = nlp.jac(x)
    dc = np.zeros(nlp.m)
    for r in nlp.r_obs + nlp.r_pair:
        dc[np.ravel(r)] = 1e-8
    return nlp.hess(x, y) + sp.diags(Sigma + dw), J, dc


@pytest.mark.parametrize("agents", [("vehicle_1",), ("vehicle_1", "vehicle_2"), ("vehicle_3",)], ids=["single", "joint_ragged", "stop_move"])
def test_kkt_apply_and_refined_step(backend, strategy_file, agents):
    from oracle import ipm
    from oracle.nlp import CollocationNLP

    lib, dev = backend
    prob, guess = make_case(strategy_file, agents)
    nlp = CollocationNLP(prob)
    # a few interior-point iterations in: multipliers, slacks and bound multipliers are all non-trivial
    sv = ObcaSolver(prob, SolveOptions(max_iter=6, refine_steps=2), device=dev, lib=lib)
    sv.solve(guess)
    L = sv.layout()
    ix, iy = build_maps(L, nlp)
    xd, yd, zLd, zUd = sv.debug_get_iterate(0)
    x, y, zL, zU = xd[ix], yd[iy], zLd[ix], zUd[ix]
    dw = 0.37
    H, J, dc = _oracle_matrix(nlp, x, y, zL, zU, dw)
    rng = np.random.default_rng(11)
    for trial in range(2):
        dx, dy = rng.standard_normal(nlp.n), rng.standard_normal(nlp.m)
        if trial == 1:  # each half on its own: an error in W cannot hide behind J'dy
            dy[:] = 0
        dxd, dyd = np.zeros(L["nx"]), np.zeros(L["ny"])
        dxd[ix], dyd[iy] = dx, dy
        r1d, r2d = sv.debug_kkt_apply(0, dw, dxd, dyd)
        r1, r2 = H @ dx + J.T @ dy, J @ dx - dc * dy
        scale1 = np.abs(H).max() + np.abs(J).max()
        assert np.abs(r1d[ix] - r1).max() <= 1e-12 * scale1 * max(1.0, np.abs(dx).max())
        assert np.abs(r2d[iy] - r2).max() <= 1e-11 * max(1.0, np.abs(r2).max())
        pad = np.ones(L["nx"], bool)
        pad[ix] = False
        assert not pad.any() or np.abs(r1d[pad]).max() == 0.0
    # the refined Newton step: residual of the full system at rounding level, including the dt row
    mu = 1e-3
    dx_d, dy_d, ok = sv.debug_step(0, mu, dw)
    assert ok == 1
    hasL, hasU = np.isfinite(nlp.xL), np.isfinite(nlp.xU)
    gL, gU = np.where(hasL, x - nlp.xL, 1.0), np.where(hasU, nlp.xU - x, 1.0)
    gl = nlp.grad_f(x) + J.T @ y
    gphi = gl - np.where(hasL, mu / gL, 0.0) + np.where(hasU, mu / gU, 0.0) + 1e-4 * mu * ((hasL & ~hasU).astype(float) - (hasU & ~hasL).astype(float))
    c = nlp.c(x)
    r1 = H @ dx_d[ix] + J.T @ dy_d[iy] + gphi
    r2 = J @ dx_d[ix] - dc * dy_d[iy] + c
    rhs = max(np.abs(gphi).max(), np.abs(c).max())
    if agents == ("vehicle_3",):
        # the stop move makes the collocation rows dependent: the structured solve drops them, everything else is refined.  The
        # dropped rows keep the dependent combination as residual, below the rank tolerance of [NULLSP] (DROPPED_ROW_TOL, cases.py)
        rows, rr1, rr2 = kkt_residual(nlp, x, y, zL, zU, mu, dw, dx_d[ix], dy_d[iy])
        cols = nlp.n + np.concatenate([r.ravel() for r in nlp.r_col])
        mask = np.ones(nlp.n + nlp.m, bool)
        mask[: nlp.n] = mask[cols] = False
        print("stop move, refined: r1 %.1e, r2 %.1e off the collocation rows, %.1e on them" % (rr1, rows[mask].max(), rows[cols].max()))
        assert rr1 <= 2e-10 and rows[mask].max() <= 1e-9
        assert rows[cols].max() <= DROPPED_ROW_TOL
    else:
        assert np.abs(r1).max() <= 2e-10 * rhs and np.abs(r2).max() <= 2e-10 * rhs  # the refinement loop stops at a residual ratio of 1e-10
        assert abs(r1[nlp.idt]) <= 2e-10 * rhs
    sv.close()


def _certificate(prob, nlp, x, y, zL, zU):
    from oracle.reference_nlp import ReferenceNLP, kkt_certificate

    u = nlp.unpack(x)
    ref = ReferenceNLP(prob)
    w = ref.variables(u["z"], u["lam"], u["mu"], u["dt"], u["pair_lam"], u["pair_mu"], u["pair_s"])
    return kkt_certificate(ref, w, ref.multipliers_from_oracle(nlp, y, zL, zU))


def _assert_kkt_point(cert, tol=1e-8, s_d=None):
    """tol applies to IPOPT's scaled optimality error: stationarity / s_d, s_d = max(100, mean |multiplier|) / 100 over the
    multipliers of the formulation the solver iterates on (for the goldens and the oracle s_d = 1 anyway)."""
    if s_d is None:
        assert cert["stationarity_scaled"] <= tol, cert
    else:
        assert cert["stationarity"] <= tol * s_d, (cert, s_d)
    assert cert["equality"] <= tol and cert["inequality"] <= tol and cert["bounds"] <= 1e-12, cert
    assert cert["sign"] <= tol, cert
    # interior point: the products sit at the final barrier parameter (~ tol / 10), and an inequality row evaluated WITHOUT its slack
    # differs from the slack by the row's feasibility error (<= tol), which enters multiplied by the row multiplier (O(100) here)
    assert cert["complementarity"] <= 100 * tol, cert


@pytest.mark.parametrize("name", GOLDEN)
def test_golden_solutions_are_kkt_points_of_the_unmodified_reference_nlp(name):
    """Every committed golden solution, with the oracle's multipliers, is a first-order KKT point of the reference problem as
    the reference states it (hard inequalities; nothing of the elastic / slack / clipping machinery is involved)."""
    from oracle.nlp import CollocationNLP

    prob, guess, gold = load_golden(name)
    nlp = CollocationNLP(prob)
    x = nlp.pack(type(guess)(gold["z"], gold["lam"], gold["mu"], gold["dt"], gold.get("pl"), gold.get("pm"), gold.get("ps")))
    cert = _certificate(prob, nlp, x, gold["y"], gold["zL"], gold["zU"])
    # 4-vehicle instance: multipliers reach 4e5 (nearly dependent collocation rows), two correct FP64 evaluations of grad f + J'y
    # (numpy sparse in the oracle: 2.7e-9, torch autograd here: 2.7e-8) differ by ~|y| eps sqrt(n): 1e-8 is below the rounding floor
    _assert_kkt_point(cert, tol=1e-7 if name == "joint_vehicle_0_1_2_3" else 1e-8)
    # the elastic variables (each ~ mu / rho at the final barrier parameter) contribute rho * sum(e) ~ 1e-6 to the penalised objective
    assert abs(cert["objective"] - gold["obj"]) <= 1e-7 * abs(gold["obj"])


def test_certificate_recovers_multipliers_from_nothing_on_a_small_instance(strategy_file):
    """No solver multipliers at all: bounded least squares on stationarity + complementarity of the reference NLP."""
    from conflict_rez_b200.problem import CollocationGuess
    from oracle import ipm
    from oracle.nlp import CollocationNLP
    from oracle.reference_nlp import ReferenceNLP, kkt_certificate

    tiny, tguess = make_case(strategy_file, ("vehicle_2",))
    tiny.n_sets = np.array([2])
    tiny.obs_A, tiny.obs_b = tiny.obs_A[:1], tiny.obs_b[:1]
    tiny.n_per_set = 2
    tiny.final_heading = np.array([np.nan])
    M = int(tiny.nodes[0])
    idx = np.linspace(0, 29, M).astype(int)
    tg = CollocationGuess(tguess.z[:, idx], tguess.lam[:, idx][:, :, :1], tguess.mu[:, idx][:, :, :1], np.float64(1.0))
    tn = CollocationNLP(tiny)
    r = ipm.solve(tn, tn.init_slacks(tn.pack(tg)), ipm.IpmOptions(tol=1e-9, constr_viol_tol=1e-9, compl_inf_tol=1e-9, max_iter=500))
    assert r.status == 0
    u = tn.unpack(r.x)
    ref = ReferenceNLP(tiny)
    w = ref.variables(u["z"], u["lam"], u["mu"], u["dt"], u["pair_lam"], u["pair_mu"], u["pair_s"])
    cert = kkt_certificate(ref, w, recover=True)
    _assert_kkt_point(cert)
    # a perturbed point is not a KKT point and the certificate says so
    u["z"][0, 5, 0] += 1e-3
    w2 = ref.variables(u["z"], u["lam"], u["mu"], u["dt"], u["pair_lam"], u["pair_mu"], u["pair_s"])
    bad = kkt_certificate(ref, w2, recover=True)
    assert max(bad["stationarity"], bad["equality"]) > 1e-5


@pytest.mark.parametrize("name", GOLDEN)
def test_solver_output_is_a_kkt_point_of_the_unmodified_reference_nlp(backend, name):
    """The solver's own returned point (tol 1e-8, status Solve_Succeeded) passes the same certificate, with the solver's own
    multipliers read back through the debug ABI."""
    from oracle.nlp import CollocationNLP

    lib, dev = backend
    prob, guess, gold = load_golden(name)
    nlp = CollocationNLP(prob)
    tol = 1e-7 if name == "joint_vehicle_0_1_2_3" else 1e-8  # multipliers of 4e5 on the 4-vehicle instance: see test_parity.py
    sv = ObcaSolver(prob, SolveOptions(tol=tol, constr_viol_tol=tol, max_iter=500), device=dev, lib=lib)
    res = sv.solve(guess)
    assert res.status[0] == 0, res.return_status(0)
    assert res.elastic[0] <= 1e-8
    ix, iy = build_maps(sv.layout(), nlp)
    xd, yd, zLd, zUd = sv.debug_get_iterate(0)
    cert = _certificate(prob, nlp, xd[ix], yd[iy], zLd[ix], zUd[ix])
    L = sv.layout()
    s_d = max(100.0, (np.abs(yd).sum() + zLd.sum() + zUd.sum()) / (L["m_active"] + L["nb"])) / 100.0  # the solver's own scaling (obca_ipm.h)
    _assert_kkt_point(cert, tol=tol, s_d=s_d)
    print(name, "certificate", {k: float("%.2e" % v) for k, v in cert.items()}, "s_d %.2f" % s_d)
    sv.close()
