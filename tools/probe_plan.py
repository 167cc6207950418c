"""ADMM kernel time and per-phase SM cycles (CTA 0) of one launch plan.
  python tools/probe_plan.py <plan: compact|multi|smem> [problem] [horizon] [batch]
Prints one JSON line.  (The plan is read from the environment when the handle is created.)"""
import json
import os
import sys
from pathlib import Path

import numpy as np

plan = sys.argv[1]
name = sys.argv[2] if len(sys.argv) > 2 else "quadrotor"
horizon = int(sys.argv[3]) if len(sys.argv) > 3 else 0
B = int(sys.argv[4]) if len(sys.argv) > 4 else 4096
os.environ["OCP_B200_PLAN"] = plan
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import optimal_control_problem_b200 as ocp  # noqa: E402

prob = ocp.Problem(name, horizon=horizon)
frames, refs = prob.sample_inputs(B, 1)
sol = prob.solver
x = np.zeros((B, prob.N)); st = np.zeros((B, ocp.NSTATS))
sol.solve_batch(frames, refs, prob.lbx, prob.ubx, prob.lbg, prob.ubg, x, None, st)
sol.set_profiling(True)
for _ in range(2):
    x[:] = 0
    sol.solve_batch(frames, refs, prob.lbx, prob.ubx, prob.lbg, prob.ubg, x, None, st)
prof = sol.get_profile()
out = {"plan": plan, "problem": name, "B": B, "wide": sol.launch_plan()["wide"],
       "admm_ms_per_launch": round(prof["admm"]["ms"] / prof["admm"]["launches"], 4)}
# phase cycles: one instance per CTA, every SM at its residency
per_sm = out["wide"]["ctas_per_sm"]
Bp = 148 * per_sm
if Bp > 148:
    frames, refs = prob.sample_inputs(Bp, 1)
    x = np.zeros((Bp, prob.N)); st = np.zeros((Bp, ocp.NSTATS))
    sol.solve_batch(frames, refs, prob.lbx, prob.ubx, prob.lbg, prob.ubg, x, None, st)
    sol.set_profiling(True, phases=True)
    x[:] = 0
    sol.solve_batch(frames, refs, prob.lbx, prob.ubx, prob.lbg, prob.ubg, x, None, st)
    ph = sol.get_phase_cycles()
    out["phase_kcycles_per_qp"] = {k: round(v / 10 / 1e3, 1) for k, v in ph.items() if v}
    out["total_kcycles_per_qp"] = round(sum(v for k, v in ph.items() if not k.startswith(("solve_", "factor_"))) / 1e4, 1)
print(json.dumps(out))
