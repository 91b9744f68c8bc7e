"""Warm start of the oracle IPM (IPOPT ``warm_start_init_point = yes``), the CPU statement the warm-start tests compare the kernel
against.

A warm start differs from the cold start of ``oracle.ipm.solve`` in the initial point only:

1. x0 (its slacks already set by ``nlp.init_slacks``) is pushed into its bounds with ``bound_push`` as both k1 and k2;
2. y starts at y0;
3. zL / zU start at zL0 / zU0 raised to at least ``mult_bound_push`` where the bound exists, 0 where it does not;
4. mu starts at mu0 when given and > 0, else at ``mu_init``, and never below the smallest mu of the run.

The iteration itself is the oracle's.  ``solve_warm`` is therefore built from the source of ``oracle.ipm.solve`` with exactly these
initialisation lines replaced; every replaced line must occur exactly once, so a change of the oracle fails here at import instead
of letting the two statements drift apart.
"""
import inspect
from dataclasses import dataclass

from oracle import ipm


@dataclass
class WarmStart:
    bound_push: float = 1e-3       # warm_start_bound_push
    mult_bound_push: float = 1e-3  # warm_start_mult_bound_push
    mu_init: float = 1e-3          # warm_start_mu_init


_REPLACE = [
    ("def solve(nlp, x0, opts: IpmOptions = None, kkt_factory=KktSolver) -> IpmResult:\n",
     "def solve_warm(nlp, x0, y0, zL0, zU0, mu0=None, ws=None, opts: IpmOptions = None, kkt_factory=KktSolver) -> IpmResult:\n"
     "    ws = ws or WarmStart()\n"),
    ("    x = push_into_bounds(np.asarray(x0, dtype=float), xL, xU, o.bound_push, o.bound_frac)\n",
     "    x = push_into_bounds(np.asarray(x0, dtype=float), xL, xU, ws.bound_push, ws.bound_push)\n"),
    ("    y = np.zeros(m)\n",
     "    y = np.array(y0, dtype=float)\n"),
    ("    zL, zU = np.where(hasL, 1.0, 0.0), np.where(hasU, 1.0, 0.0)\n",
     "    zL = np.where(hasL, np.maximum(np.asarray(zL0, dtype=float), ws.mult_bound_push), 0.0)\n"
     "    zU = np.where(hasU, np.maximum(np.asarray(zU0, dtype=float), ws.mult_bound_push), 0.0)\n"),
    ("    mu = o.mu_init\n",
     "    mu = max(min(o.tol, o.compl_inf_tol) / (o.kappa_eps + 1.0), mu0 if mu0 is not None and mu0 > 0 else ws.mu_init)\n"),
]


def _build():
    src = inspect.getsource(ipm.solve)
    for old, new in _REPLACE:
        assert src.count(old) == 1, "oracle.ipm.solve changed: %r" % old
        src = src.replace(old, new)
    ns = dict(vars(ipm), WarmStart=WarmStart)
    exec(compile(src, ipm.__file__ + " (warm start)", "exec"), ns)
    return ns["solve_warm"]


solve_warm = _build()
