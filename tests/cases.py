"""Shared helpers of the parity tests: golden fixtures, oracle-side linear algebra, independent geometry checks."""
import os

import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from conflict_rez_b200.problem import CollocationGuess, CollocationProblem

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# Collocation rows that [NULLSP] drops as dependent (rank test: remainder <= 1e-8 of the row's norm) are satisfied only up to
# that remainder, and a remainder above 1e-7 of the row's scale is kept as an implied row instead: 1e-7 relative to |rhs|
# bounds their residual.  Where the step solves the dependent rows exactly (the stop move) it measures at rounding level.
# The emulation's steps meet 6e-15 (unrefined) and 2e-14 (refined) there.
DROPPED_ROW_TOL = 1e-7


def load_golden(name):
    d = dict(np.load(os.path.join(GOLDEN, name + ".npz")))
    d.update(np.load(os.path.join(GOLDEN, name + "_multipliers.npz")))
    prob = CollocationProblem(
        n_sets=d["p_n_sets"], obs_A=d["p_obs_A"], obs_b=d["p_obs_b"], tube_A=d["p_tube_A"], tube_b=d["p_tube_b"], init_pose=d["p_init_pose"],
        final_heading=d["p_final_heading"], body_G=d["p_body_G"], body_g=d["p_body_g"], wb=float(d["p_wb"]), region=d["p_region"], limits=d["p_limits"],
        K=int(d["p_K"]), n_per_set=int(d["p_n_per_set"]), dmin=float(d["p_dmin"]), shrink_tube=float(d["p_shrink"]),
    )
    has_pairs = "g_pl" in d
    guess = CollocationGuess(d["g_z"], d["g_lam"], d["g_mu"], d["g_dt"], d["g_pl"] if has_pairs else None, d["g_pm"] if has_pairs else None, d["g_ps"] if has_pairs else None)
    sol = {k[2:]: v for k, v in d.items() if k.startswith("s_")}
    return prob, guess, sol


def kkt_system(nlp, x, y, zL, zU, mu, delta_w, kappa_d=1e-4, dc_local=1e-8):
    """The primal-dual Newton system K [dx; dy] = rhs of the solver (csrc/obca_kkt.h) assembled from the oracle's sparse
    derivatives: returns K (csc), rhs, c(x), grad f + J'y."""
    hasL, hasU = np.isfinite(nlp.xL), np.isfinite(nlp.xU)
    gL, gU = np.where(hasL, x - nlp.xL, 1.0), np.where(hasU, nlp.xU - x, 1.0)
    Sigma = np.where(hasL, zL / gL, 0.0) + np.where(hasU, zU / gU, 0.0)
    J = nlp.jac(x)
    gl = nlp.grad_f(x) + J.T @ y
    gphi = gl - np.where(hasL, mu / gL, 0.0) + np.where(hasU, mu / gU, 0.0) + kappa_d * mu * ((hasL & ~hasU).astype(float) - (hasU & ~hasL).astype(float))
    c = nlp.c(x)
    dc = np.zeros(nlp.m)
    for r in nlp.r_obs + nlp.r_pair:
        dc[np.ravel(r)] = dc_local
    K = sp.bmat([[nlp.hess(x, y) + sp.diags(Sigma + delta_w), J.T], [J, -sp.diags(dc)]], format="csc")
    return K, np.concatenate([-gphi, -c]), c, gl


def step_residual(K, rhs, n, d):
    """Relative residual of the step d = [dx; dy] in K d = rhs, row by row: |K d - rhs|_i / |rhs|_inf.
    Returns (rows, worst of the n primal rows (r1), worst of the constraint rows (r2)).  Not scaled by |K| |d|: the
    entries of K span twelve decades (Sigma of the bound multipliers), and |K| |d| would call almost anything small."""
    rows = np.abs(K @ d - rhs) / np.abs(rhs).max()
    return rows, rows[:n].max(), rows[n:].max()


def backward_error(K, rhs, n, d):
    """Backward error of d in K d = rhs, row by row: |K d - rhs|_i / ((|K| |d|)_i + |rhs|_inf).  Returns (rows, r1, r2) like
    ``step_residual``.  Where |K| |d| dwarfs |rhs| (large delta_w, multipliers of 1e8 mid-solve) rounding alone leaves a
    residual far above eps |rhs|; this measure charges each row for the magnitude of its own products."""
    rows = np.abs(K @ d - rhs) / (abs(K) @ np.abs(d) + np.abs(rhs).max())
    return rows, rows[:n].max(), rows[n:].max()


def kkt_residual(nlp, x, y, zL, zU, mu, dw, dx, dy, backward=False):
    """Relative residual (``step_residual``) or, with ``backward``, backward error (``backward_error``) of any step (dx, dy),
    in the oracle's numbering, in the oracle's assembled K: (rows, r1, r2).  Meaningful where K is singular too, where a
    forward comparison is not."""
    K, rhs, _, _ = kkt_system(nlp, x, y, zL, zU, mu, dw)
    return (backward_error if backward else step_residual)(K, rhs, nlp.n, np.concatenate([dx, dy]))


def oracle_newton_step(nlp, x, y, zL, zU, mu, delta_w, kappa_d=1e-4, dc_local=1e-8):
    """Reference Newton step: sparse LU of the full primal-dual system with iterative refinement.
    Returns dx, dy, c(x), grad f + J'y and the step's own residual (rows, r1, r2) as ``step_residual`` defines it: where
    K is numerically singular (vehicle_0's final approach over-collocates k = 0) the LU "solution" is no solution at all,
    and a forward comparison against it means nothing."""
    K, rhs, c, gl = kkt_system(nlp, x, y, zL, zU, mu, delta_w, kappa_d, dc_local)
    lu = spla.splu(K)
    sol = lu.solve(rhs)
    for _ in range(3):
        sol += lu.solve(rhs - K @ sol)
    return sol[: nlp.n], sol[nlp.n :], c, gl, step_residual(K, rhs, nlp.n, sol)


def _negative_pivots(K, n, delta_c):
    d2 = K.diagonal()[n:]
    Kc = (K - sp.diags(np.concatenate([np.zeros(n), np.where(d2 == 0.0, delta_c, 0.0)]))).tocsc()
    lu = spla.splu(Kc, permc_spec="MMD_AT_PLUS_A", diag_pivot_thresh=0.0, options=dict(SymmetricMode=True))
    assert np.array_equal(lu.perm_r, lu.perm_c), "the factorisation pivoted off the diagonal: the pivot count is not the inertia"
    d = lu.U.diagonal()
    assert np.isfinite(d).all() and (d != 0).all()
    return int((d < 0).sum())


def kkt_inertia_ok(nlp, x, y, zL, zU, mu, dw, delta_c=(1e-10, 1e-12)):
    """True iff K has exactly m negative eigenvalues (inertia (n, m, 0): IPOPT's acceptance test, the solver's ``ok``).

    Symmetric-mode SuperLU with diag_pivot_thresh = 0 takes every nonzero diagonal entry as its pivot, so it factorises
    P K P' = L U with U = D L', and by Sylvester's law of inertia the negative eigenvalues of K are the negative pivots of D.
    The rows of K without a -dc entry (collocation, initial, terminal, tube rows) get -delta_c on the diagonal, IPOPT's
    delta_c: with an exact zero there a pivot can vanish and SuperLU leaves the diagonal.  Where J loses rank (vehicle_0's
    final approach) the eigenvalues this adds are negative, as the dropped dependent rows of [NULLSP] are the solver's own
    analogue of delta_c.  The answer is taken at two values of delta_c and must not depend on it: 1e-8 is already too large
    where multipliers of 1e8 sit on nearly dependent rows (a few extra negative pivots mid-solve on the 4-vehicle instance)."""
    K, _, _, _ = kkt_system(nlp, x, y, zL, zU, mu, dw)
    counts = [_negative_pivots(K, nlp.n, dc) for dc in delta_c]
    assert len({c == nlp.m for c in counts}) == 1, ("the inertia test depends on delta_c: K does not determine it", counts, nlp.m)
    return counts[0] == nlp.m


# ---------------------------------------------------------------------------------------------------------------
# independent geometry (no duals involved): used for size-independent property checks of a solution
# ---------------------------------------------------------------------------------------------------------------
def body_corners(x, y, psi, G, g):
    lf, hw, lr = g[0], g[1], g[2]
    loc = np.array([[lf, hw], [-lr, hw], [-lr, -hw], [lf, -hw]])
    c, s = np.cos(psi), np.sin(psi)
    R = np.stack([np.stack([c, -s], -1), np.stack([s, c], -1)], -2)
    return np.einsum("...ij,kj->...ki", R, loc) + np.stack([x, y], -1)[..., None, :]


def _seg_dist(p, a, b):
    ab = b - a
    t = np.clip(np.sum((p - a) * ab, -1) / np.maximum(np.sum(ab * ab, -1), 1e-300), 0, 1)
    return np.linalg.norm(p - (a + t[..., None] * ab), axis=-1)


def _inside(p, poly):
    """p (...,2) strictly inside convex CCW-or-CW quad poly (...,4,2)?"""
    sign = None
    ok = np.ones(p.shape[:-1], dtype=bool)
    for i in range(4):
        a, b = poly[..., i, :], poly[..., (i + 1) % 4, :]
        cr = (b[..., 0] - a[..., 0]) * (p[..., 1] - a[..., 1]) - (b[..., 1] - a[..., 1]) * (p[..., 0] - a[..., 0])
        sign = np.sign(cr) if sign is None else sign
        ok &= np.sign(cr) == sign
    return ok


def quad_distance(P, Q):
    """Distance between convex quads (0 when they overlap)."""
    d = np.full(P.shape[:-2], np.inf)
    for i in range(4):
        for j in range(4):
            d = np.minimum(d, _seg_dist(P[..., i, :], Q[..., j, :], Q[..., (j + 1) % 4, :]))
            d = np.minimum(d, _seg_dist(Q[..., i, :], P[..., j, :], P[..., (j + 1) % 4, :]))
    over = np.zeros(P.shape[:-2], dtype=bool)
    for i in range(4):
        over |= _inside(P[..., i, :], Q) | _inside(Q[..., i, :], P)
    return np.where(over, 0.0, d)


def rect_vertices(A, b):
    V = np.zeros((4, 2))
    for i in range(4):
        j = (i + 1) % 4
        V[i] = np.linalg.solve(np.array([A[i], A[j]]), np.array([b[i], b[j]]))
    return V


def check_solution_properties(prob, z, dt, tol=1e-5):
    """Size-independent checks of a (B,V,M,7) trajectory batch against the problem statement itself."""
    from oracle.collocation import collocation_coefficients, f_ct

    A, _, _ = collocation_coefficients(prob.K)
    B = z.shape[0]
    init = prob.init_pose if prob.init_pose.ndim == 3 else np.broadcast_to(prob.init_pose, (B,) + prob.init_pose.shape)
    worst = {}
    for a in range(prob.V):
        M, N = int(prob.nodes[a]), int(prob.N[a])
        za = z[:, a, :M]
        worst["init"] = max(worst.get("init", 0), np.abs(za[:, 0, :3] - init[:, a]).max(), np.abs(za[:, 0, 3:]).max())
        zi = za.reshape(B, N, prob.K + 1, 7)
        poly = np.einsum("jk,bijc->bikc", A, zi[..., :5]) / np.reshape(dt, (B, 1, 1, 1))
        x, y, psi, v, de, ua, uw = [zi[..., c] for c in range(7)]
        f = np.stack([v * np.cos(psi), v * np.sin(psi), v / prob.wb * np.tan(de), ua, uw], -1)
        worst["collocation"] = max(worst.get("collocation", 0), np.abs(poly - f).max())
        worst["continuity"] = max(worst.get("continuity", 0), np.abs(zi[:, 1:, 0] - zi[:, :-1, -1]).max())
        end = za[:, -1]
        term = np.abs(end[:, 3:]).max()
        if np.isfinite(prob.final_heading[a]):
            term = max(term, np.abs(end[:, 2] - prob.final_heading[a]).max())
        worst["terminal"] = max(worst.get("terminal", 0), term)
        lo = np.array([prob.region[0], prob.region[2], -np.inf, prob.limits[0], prob.limits[2], prob.limits[4], prob.limits[6]])
        hi = np.array([prob.region[1], prob.region[3], np.inf, prob.limits[1], prob.limits[3], prob.limits[5], prob.limits[7]])
        worst["bounds"] = max(worst.get("bounds", 0), np.maximum(lo - za, za - hi).max())
        # tube sets at the set transitions and at the end
        S = int(prob.n_sets[a])
        for q in range(1, S):
            n = M - 1 if q == S - 1 else q * prob.n_per_set * (prob.K + 1)
            p = za[:, n]
            back = p[:, :2]
            front = back + prob.wb * np.stack([np.cos(p[:, 2]), np.sin(p[:, 2])], -1)
            vb = (back @ prob.tube_A[a, q, 0].T - (prob.tube_b[a, q, 0] - prob.shrink_tube)).max()
            vf = (front @ prob.tube_A[a, q, 1].T - (prob.tube_b[a, q, 1] - prob.shrink_tube)).max()
            worst["tube"] = max(worst.get("tube", 0), vb, vf)
        # obstacle clearance by plain geometry
        corners = body_corners(za[..., 0], za[..., 1], za[..., 2], prob.body_G, prob.body_g)
        for j in range(prob.O):
            Vo = np.broadcast_to(rect_vertices(prob.obs_A[j], prob.obs_b[j]), corners.shape)
            worst["obstacle_clearance"] = min(worst.get("obstacle_clearance", np.inf), quad_distance(corners, Vo).min())
    for (a, b) in prob.pairs:
        m = int(min(prob.nodes[a], prob.nodes[b]))
        ca = body_corners(z[:, a, :m, 0], z[:, a, :m, 1], z[:, a, :m, 2], prob.body_G, prob.body_g)
        cb = body_corners(z[:, b, :m, 0], z[:, b, :m, 1], z[:, b, :m, 2], prob.body_G, prob.body_g)
        worst["vehicle_clearance"] = min(worst.get("vehicle_clearance", np.inf), quad_distance(ca, cb).min())
    return worst
