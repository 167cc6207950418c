"""Small solves through every placement of the ADMM kernels, for compute-sanitizer (one tool per gpurun call):
  compute-sanitizer --tool memcheck  python tools/sanitize_cases.py
  compute-sanitizer --tool racecheck python tools/sanitize_cases.py
Placements: all-shared (deep), two-CTA multi, compact, big (two-chain bulk-copy ring), mixed (streamed
generic blocks), PCG fallback; plus the assembly, objective and shift kernels that every solve launches.  Each case is
checked against the oracle so that a "clean" run is also a correct one."""
import os
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "tests"))
import _oracle  # noqa: E402
import optimal_control_problem_b200 as ocp  # noqa: E402

CASES = [  # (label, problem, horizon, env)
    ("smem (deep plan)", "quadrotor", 5, {"OCP_B200_PLAN": "smem"}),
    ("multi 192x2", "quadrotor", 5, {"OCP_B200_PLAN": "multi"}),
    ("compact", "quadrotor", 5, {"OCP_B200_PLAN": "compact"}),
    ("big (twisted ring)", "cartpole", 16, {"OCP_B200_PLAN": "big", "OCP_B200_FORCE_STREAM": "1"}),
    ("mixed (streamed blocks)", "centroidal", 3, {"OCP_B200_PLAN": "mixed", "OCP_B200_FORCE_STREAM": "1"}),
]
KEYS = ("OCP_B200_PLAN", "OCP_B200_FORCE_STREAM")

ok = True
for label, name, H, env in CASES:
    for k in KEYS:
        os.environ.pop(k, None)
    os.environ.update(env)
    prob = ocp.Problem(name, horizon=H, alpha=0.5, step_num=2)
    s = prob.get_settings()
    s.eps_abs = s.eps_rel = 1e-6          # tight: exercises the rho-update refactorisation as well
    prob.solver.update_settings(s)
    B = 2
    frames, refs = prob.sample_inputs(B, 77)
    x0 = np.tile(frames, (1, H))
    x = x0.copy(); st = np.zeros((B, ocp.NSTATS))
    prob.solver.solve_batch(frames, refs, prob.lbx, prob.ubx, prob.lbg, prob.ubg, x, None, st)
    ora = _oracle.OracleProblem(name, horizon=H, alpha=0.5, step_num=2)
    ora.set_qp_settings(_oracle.settings_from_b200(s))
    ox, _, ost = ora.solve_batch(frames, refs, x0=x0)
    err = float(np.abs(x - ox).max() / max(1.0, np.abs(ox).max()))
    same = bool(np.array_equal(st[:, ocp.STAT["admm_iters"]], ost[:, 2]))
    plan = prob.solver.launch_plan()
    print(f"{label:26s} {name} H={H} place {plan['deep']['place']} threads {plan['deep']['threads']} "
          f"admm iters {st[:, ocp.STAT['admm_iters']].tolist()} rho updates {st[:, ocp.STAT['rho_updates']].tolist()} "
          f"rel err vs oracle {err:.2e} iterations equal {same}", flush=True)
    ok = ok and err < 1e-5 and same
# PCG fallback kernel (a pattern without stage structure)
rng = np.random.default_rng(5)
n, me = 70, 20
import scipy.sparse as sp  # noqa: E402
M = rng.standard_normal((n, n)) * (rng.random((n, n)) < 0.2)
P = sp.csc_matrix(M @ M.T + n * np.eye(n)); P.sort_indices()
A = sp.csc_matrix(np.vstack([np.eye(n), rng.standard_normal((me, n)) * (rng.random((me, n)) < 0.3)])); A.sort_indices()
xf = rng.standard_normal(n)
l = A @ xf - 1.0; u = A @ xf + 1.0
x, y, info = ocp.cucaqp_solve(n, n + me, P.indptr, P.indices, P.data, rng.standard_normal(n), A.indptr, A.indices, A.data, l, u,
                              eps_abs=1e-5, eps_rel=1e-5)
print("pcg fallback               status", info[0], "iters", info[1], flush=True)
# shift kernel
for k in KEYS:
    os.environ.pop(k, None)
print("ALL CASES MATCH THE ORACLE" if ok else "MISMATCH", flush=True)
sys.exit(0 if ok else 1)
