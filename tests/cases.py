"""Shared helpers of the parity tests: golden fixtures, oracle-side linear algebra, independent geometry checks."""
import os

import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from conflict_rez_b200.problem import CollocationGuess, CollocationProblem

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


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


def oracle_newton_step(nlp, x, y, zL, zU, mu, delta_w, kappa_d=1e-4, dc_local=1e-8):
    """Reference Newton step: sparse LU of the full primal-dual system with iterative refinement."""
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
    lu = spla.splu(K)
    rhs = np.concatenate([-gphi, -c])
    sol = lu.solve(rhs)
    for _ in range(3):
        sol += lu.solve(rhs - K @ sol)
    return sol[: nlp.n], sol[nlp.n :], c, gl


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
