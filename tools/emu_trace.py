"""Developer script: iteration tables of selected bench instances under the host emulation, from the solver's iteration record.

    python tools/emu_trace.py 3 17      # instances 3 and 17 of the 512-instance 4-vehicle bench batch (seed 0)

OBCA_TRACE=1 in the environment adds the emulation's remaining diagnostics (the variable that limits each primal step, the
KKT solve's messages).
"""
import os, sys, tempfile
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from conflict_rez_b200.control.strategy import write_strategy
from conflict_rez_b200.control.batch_planner import prepare_joint_batch, random_init_offsets
from conflict_rez_b200.solver import SolveOptions, format_history

ids = [int(a) for a in sys.argv[1:]]
from conflict_rez_b200 import solver as _s
lib = _s.load_library(os.path.join(ROOT, "tools/host_emu/libobca_hostemu.so"))
fn = os.path.join(tempfile.mkdtemp(), "4v"); write_strategy(fn)
agents = ["vehicle_0", "vehicle_1", "vehicle_2", "vehicle_3"]
opts = SolveOptions(tol=1e-2, constr_viol_tol=1e-2, max_iter=600, history=601)
offs = random_init_offsets(512, 4, seed=0)[ids]
plan = prepare_joint_batch(fn, agents, offs, opts, device="cpu", lib=lib)
sv = plan.solver
res = sv.solve(plan.guess)
print("status", res.status, "iters", res.iters)
for b, i in enumerate(ids):
    print("\ninstance %d: %s after %d iterations" % (i, res.return_status(b), res.iters[b]))
    print(format_history(res, b))
for a, r in zip(agents, plan.singles):
    print(a, "single status", r.status, "iters", r.iters, "obj", r.obj, "dt", r.dt)
