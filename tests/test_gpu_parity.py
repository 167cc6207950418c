"""GPU parity tests proper: the CUDA path, called through the C ABI (include/ocp_b200.h), against
the CPU oracle on the same seeded inputs.

Tolerances (FP64 on both sides; by default the GPU factorises the reduced KKT system P + sigma I +
A' diag(rho) A directly (bordered block-tridiagonal LDL', admm_direct_kernel.cuh / admm_compact_kernel.cuh;
PCG to a relative residual of pcg_tol = 1e-10 where that structure is absent) where the oracle uses
an exact LDL' solve of the full KKT system, so ADMM iterates agree to rounding amplified by the
conditioning of the scaled KKT system):
  * sparsity patterns / CSC index arrays: bit-exact;
  * local-system values (H, grad, J, l - c, u - c): 1e-12 relative;
  * QP primal / dual solutions, SQP iterates: 1e-6 relative to the vector's inf-norm
    (BASELINE.json north_star), with identical ADMM iteration counts, rho updates and statuses.
"""
import numpy as np
import pytest

import _oracle

pytestmark = pytest.mark.gpu

REL_VALUES = 1e-12
REL_SOLUTION = 1e-6


def rel_err(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return float(np.abs(a - b).max() / max(1.0, np.abs(b).max()))


def random_iterate(prob, B, seed):
    rng = np.random.default_rng(seed)
    frames, refs = prob.sample_inputs(B, seed)
    x = np.tile(frames, (1, prob.horizon)) + 0.05 * rng.standard_normal((B, prob.N))
    return frames, refs, x


@pytest.mark.parametrize("name", ["quadrotor", "cartpole", "centroidal"])
def test_patterns_bit_exact(problems, name):
    prob, ora = problems(name)
    assert prob.dims == dict(np=ora.np_, nf=ora.nf, horizon=ora.horizon, ng=ora.ng, n=ora.n, m=ora.m,
                             nnz_h=ora.nnz_h, nnz_a=ora.nnz_a)
    for a in ("h_colptr", "h_rowidx", "a_colptr", "a_rowidx"):
        assert np.array_equal(getattr(prob, a), getattr(ora, a)), a


@pytest.mark.parametrize("name,B", [("quadrotor", 5), ("cartpole", 3), ("centroidal", 3)])
def test_local_system_matches_oracle(problems, name, B):
    prob, ora = problems(name)
    frames, refs, x = random_iterate(prob, B, 0xB200 + 7)
    hv, q, av, l, u = prob.solver.export_qp(frames, refs, prob.lbx, prob.ubx, prob.lbg, prob.ubg, x)
    for b in range(B):
        ohv, oq, oav, ol, ou = ora.local_system(frames[b], refs[b], x[b])
        assert rel_err(hv[b], ohv) < REL_VALUES
        assert rel_err(q[b], oq) < REL_VALUES
        assert rel_err(av[b], oav) < REL_VALUES
        fin = np.isfinite(ol)
        assert np.array_equal(np.isfinite(l[b]), fin) and np.array_equal(l[b][~fin], ol[~fin])
        assert rel_err(l[b][fin], ol[fin]) < REL_VALUES
        fin = np.isfinite(ou)
        assert np.array_equal(np.isfinite(u[b]), fin) and np.array_equal(u[b][~fin], ou[~fin])
        assert rel_err(u[b][fin], ou[fin]) < REL_VALUES


def test_local_system_without_frame_pin(problems):
    prob, ora = problems("quadrotor")
    frames, refs, x = random_iterate(prob, 2, 11)
    hv, q, av, l, u = prob.solver.export_qp(None, refs, prob.lbx, prob.ubx, prob.lbg, prob.ubg, x)
    for b in range(2):
        ohv, oq, oav, ol, ou = ora.local_system(None, refs[b], x[b])
        assert np.array_equal(np.isfinite(l[b]), np.isfinite(ol))
        fin = np.isfinite(ol)
        assert rel_err(l[b][fin], ol[fin]) < REL_VALUES
        assert rel_err(av[b], oav) < REL_VALUES


def _qp_case(prob, ora, seed, B=3):
    frames, refs, x = random_iterate(prob, B, seed)
    sys_ = [ora.local_system(frames[b], refs[b], x[b]) for b in range(B)]
    return [np.stack([s[k] for s in sys_]) for k in range(5)]


@pytest.mark.parametrize("name", ["quadrotor", "cartpole"])
@pytest.mark.parametrize("eps", [1e-3, 1e-7])
def test_qp_solution_matches_oracle(problems, native, name, eps):
    prob, ora = problems(name)
    hv, q, av, l, u = _qp_case(prob, ora, 21)
    s = prob.get_settings()
    s.eps_abs = s.eps_rel = eps
    prob.solver.update_settings(s)
    x, y, info = prob.solver.qp_solve_batch(hv, q, av, l, u)
    sv = _oracle.settings_from_b200(s)
    for b in range(hv.shape[0]):
        ox, oy, oinfo, _ = _oracle.qp_solve(prob.n, prob.m, prob.h_colptr, prob.h_rowidx, hv[b], q[b], prob.a_colptr,
                                            prob.a_rowidx, av[b], l[b], u[b], settings=sv)
        assert info[b, native.INFO["status"]] == oinfo[0] == native.QP_SOLVED
        assert info[b, native.INFO["iters"]] == oinfo[1]
        assert info[b, native.INFO["rho_updates"]] == oinfo[6]
        assert rel_err(x[b], ox) < REL_SOLUTION
        assert rel_err(y[b], oy) < REL_SOLUTION
        assert abs(info[b, native.INFO["prim_res"]] - oinfo[3]) <= 1e-6 * max(1.0, abs(oinfo[3])) + 1e-9
        assert abs(info[b, native.INFO["dual_res"]] - oinfo[4]) <= 1e-6 * max(1.0, abs(oinfo[4])) + 1e-9


def test_admm_trace_matches_oracle(problems, native):
    prob, ora = problems("quadrotor")
    hv, q, av, l, u = _qp_case(prob, ora, 5, B=1)
    s = prob.get_settings()
    s.eps_abs = s.eps_rel = 1e-8
    prob.solver.update_settings(s)
    trace, x, y = prob.solver.admm_trace(hv[0], q[0], av[0], l[0], u[0])
    ox, oy, oinfo, otrace = _oracle.qp_solve(prob.n, prob.m, prob.h_colptr, prob.h_rowidx, hv[0], q[0], prob.a_colptr,
                                             prob.a_rowidx, av[0], l[0], u[0], settings=_oracle.settings_from_b200(s))
    assert len(trace) == len(otrace) > 1
    assert np.array_equal(trace[:, 0], otrace[:, 0])                      # iteration numbers of the checks
    assert np.allclose(trace[:, 3], otrace[:, 3], rtol=1e-6)              # rho schedule
    assert np.allclose(trace[:, 1], otrace[:, 1], rtol=1e-4, atol=1e-10)  # primal residual history
    assert np.allclose(trace[:, 2], otrace[:, 2], rtol=1e-4, atol=1e-10)  # dual residual history
    assert np.array_equal(trace[:, 5], otrace[:, 5])
    assert rel_err(x, ox) < REL_SOLUTION


@pytest.mark.parametrize("precond", [0, 1, 2])
def test_linear_system_solvers_agree(problems, native, precond):
    prob, ora = problems("quadrotor")
    hv, q, av, l, u = _qp_case(prob, ora, 9, B=2)
    s = prob.get_settings()
    s.eps_abs = s.eps_rel = 1e-6
    s.pcg_precond = precond
    s.pcg_max_iter = 2000
    prob.solver.update_settings(s)
    x, y, info = prob.solver.qp_solve_batch(hv, q, av, l, u)
    sv = _oracle.settings_from_b200(s)
    for b in range(2):
        ox, oy, oinfo, _ = _oracle.qp_solve(prob.n, prob.m, prob.h_colptr, prob.h_rowidx, hv[b], q[b], prob.a_colptr,
                                            prob.a_rowidx, av[b], l[b], u[b], settings=sv)
        assert info[b, 1] == oinfo[1]
        assert rel_err(x[b], ox) < REL_SOLUTION


@pytest.mark.parametrize("name,B,alpha,steps", [("quadrotor", 6, 0.1, 10), ("quadrotor", 4, 1.0, 5),
                                                ("cartpole", 2, 0.5, 3), ("centroidal", 2, 1.0, 2)])
def test_sqp_solve_matches_oracle(problems, native, name, B, alpha, steps):
    prob, ora = problems(name)
    frames, refs = prob.sample_inputs(B, 0xB200 + 2)
    s = prob.get_settings()
    s.sqp_alpha, s.sqp_step_num = alpha, steps
    prob.solver.update_settings(s)
    # start every instance from its initial state held over the horizon (x = 0 makes the first
    # cart-pole QP primal infeasible, which is covered by test_infeasible_step_propagates_nan)
    x0 = np.tile(frames, (1, prob.horizon))
    x = x0.copy(); f = np.zeros(B); st = np.zeros((B, native.NSTATS))
    prob.solver.solve_batch(frames, refs, prob.lbx, prob.ubx, prob.lbg, prob.ubg, x, f, st)
    ora.set_schedule(steps, alpha)
    ora.set_qp_settings(_oracle.settings_from_b200(s))
    ox, of, ost = ora.solve_batch(frames, refs, x0=x0)
    assert np.isfinite(ox).all()
    assert np.array_equal(st[:, native.STAT["sqp_steps"]], ost[:, 1])
    assert np.array_equal(st[:, native.STAT["admm_iters"]], ost[:, 2])
    assert np.array_equal(st[:, native.STAT["qp_status"]], ost[:, 0])
    assert rel_err(x, ox) < REL_SOLUTION
    assert np.allclose(f, of, rtol=1e-6, atol=1e-9)
    assert np.allclose(st[:, native.STAT["objective"]], of, rtol=1e-6, atol=1e-9)


def test_infeasible_step_propagates_nan(problems, native):
    """Cart-pole from x = 0 with the pole pinned near theta = pi: the first QP is primal infeasible;
    OSQP returns NaN and the reference adds it to the iterate unchecked (SQPOptimizationSolver.cpp:
    155-177).  Both sides must agree on that, status included."""
    prob, ora = problems("cartpole")
    frames, refs = prob.sample_inputs(2, 0xB200 + 2)
    s = prob.get_settings()
    s.sqp_alpha, s.sqp_step_num = 0.5, 2
    prob.solver.update_settings(s)
    x = np.zeros((2, prob.N)); st = np.zeros((2, native.NSTATS))
    prob.solver.solve_batch(frames, refs, prob.lbx, prob.ubx, prob.lbg, prob.ubg, x, None, st)
    ora.set_schedule(2, 0.5)
    ora.set_qp_settings(_oracle.settings_from_b200(s))
    ox, of, ost = ora.solve_batch(frames, refs)
    assert np.array_equal(np.isnan(x), np.isnan(ox))
    assert np.array_equal(st[:, native.STAT["qp_status"]], ost[:, 0])


def test_throughput_plan_matches_oracle_and_latency_plan(problems, native):
    """Batches larger than the SM count run the 2-CTA/SM plan (factor blocks in an L2 slab), small
    batches the all-shared-memory plan: same arithmetic, so the same bits -- and the oracle's answer."""
    prob, ora = problems("quadrotor")
    B = 400
    frames, refs = prob.sample_inputs(B, 0xB200 + 5)
    s = prob.get_settings()
    s.sqp_alpha, s.sqp_step_num = 0.1, 4
    prob.solver.update_settings(s)
    x = np.zeros((B, prob.N)); st = np.zeros((B, native.NSTATS))
    prob.solver.solve_batch(frames, refs, prob.lbx, prob.ubx, prob.lbg, prob.ubg, x, None, st)
    pick = [0, 147, 148, 295, 296, 399]
    for b in pick:
        xb = np.zeros((1, prob.N))
        prob.solver.solve_batch(frames[b:b + 1], refs[b:b + 1], prob.lbx, prob.ubx, prob.lbg, prob.ubg, xb)
        assert np.array_equal(xb[0], x[b])
    ora.set_schedule(4, 0.1)
    ora.set_qp_settings(_oracle.settings_from_b200(s))
    ox, of, ost = ora.solve_batch(frames[pick], refs[pick])
    assert rel_err(x[pick], ox) < REL_SOLUTION
    assert np.array_equal(st[pick][:, native.STAT["admm_iters"]], ost[:, 2])
    assert (st[:, native.STAT["qp_status"]] == native.QP_SOLVED).all()


def test_batch_equals_single_instance(problems, native):
    """Every instance of a batch gets the bits it gets when solved alone."""
    prob, _ = problems("quadrotor")
    frames, refs = prob.sample_inputs(5, 3)
    s = prob.get_settings()
    s.sqp_alpha, s.sqp_step_num = 0.5, 3
    prob.solver.update_settings(s)
    x = np.zeros((5, prob.N))
    prob.solver.solve_batch(frames, refs, prob.lbx, prob.ubx, prob.lbg, prob.ubg, x)
    for b in (0, 4):
        xb = np.zeros((1, prob.N))
        prob.solver.solve_batch(frames[b:b + 1], refs[b:b + 1], prob.lbx, prob.ubx, prob.lbg, prob.ubg, xb)
        assert np.array_equal(xb[0], x[b])


@pytest.mark.parametrize("case", [1, 2, 3, 4, 5, 6, 7])
def test_reference_kat_cases_on_gpu(native, case):
    """test/test.cpp:13-185 through SQPOptimizationSolver::getOptimalSolution (alpha=1, one step:
    the cases are QPs) -- analytic optimum within the OSQP tolerance the reference runs with, and
    the oracle's answer to 1e-6."""
    kat = native.KatProblem(case, step_num=1, alpha=1.0)
    x, f = kat.solve()
    expected = _oracle.kat_expected(case)
    assert np.abs(x - expected).max() < 5e-3
    ox, of, _ = _oracle.kat_solve(case, 1, 1.0)
    assert rel_err(x, ox) < REL_SOLUTION
    s = native.default_settings()
    s.eps_abs = s.eps_rel = 1e-9
    s.sqp_alpha, s.sqp_step_num = 1.0, 1
    kat2 = native.KatProblem(case, step_num=1, alpha=1.0)
    kat2.set_settings(s)
    x2, _ = kat2.solve()
    assert np.abs(x2 - expected).max() < 1e-6


def _check_certificates(native, settings):
    """Primal: x in [0,1] with the row x >= 2 -> status 3 and a NaN solution, which the reference adds to its
    iterate unchecked (SURVEY.md §3.3).  Dual: min -x with x >= 0 and no curvature (empty H) -> status 5."""
    hc, hr = [0, 1], [0]
    ac, ar = [0, 2], [0, 1]
    sol = native.Solver.create(1, 2, hc, hr, ac, ar, settings=settings)
    x, y, info = sol.qp_solve_batch(np.array([[1.0]]), np.array([[0.0]]), np.array([[1.0, 1.0]]),
                                    np.array([[0.0, 2.0]]), np.array([[1.0, 3.0]]))
    ox, oy, oinfo, _ = _oracle.qp_solve(1, 2, hc, hr, [1.0], [0.0], ac, ar, [1.0, 1.0], [0.0, 2.0], [1.0, 3.0])
    assert info[0, 0] == oinfo[0] == native.QP_PRIMAL_INFEASIBLE
    assert np.isnan(x).all() and np.isnan(ox).all()
    hc, hr = [0, 0], []
    ac, ar = [0, 1], [0]
    sol = native.Solver.create(1, 1, hc, hr, ac, ar, settings=settings)
    x, y, info = sol.qp_solve_batch(np.zeros((1, 0)), np.array([[-1.0]]), np.array([[1.0]]),
                                    np.array([[0.0]]), np.array([[np.inf]]))
    ox, oy, oinfo, _ = _oracle.qp_solve(1, 1, hc, hr, [], [-1.0], ac, ar, [1.0], [0.0], [np.inf])
    assert info[0, 0] == oinfo[0] == native.QP_DUAL_INFEASIBLE
    assert np.isnan(x).all() and np.isnan(ox).all()


def test_infeasible_qp_reports_certificate(native):
    """Both certificates on the direct kernel (the default preconditioner, BLOCK_TRIDIAG)."""
    _check_certificates(native, native.default_settings())


@pytest.mark.parametrize("precond", [0, 1])
def test_infeasible_qp_reports_certificate_on_pcg(native, precond):
    """Both certificates on the PCG kernel (DIAGONAL and BLOCK_JACOBI preconditioners)."""
    s = native.default_settings()
    s.pcg_precond = precond
    _check_certificates(native, s)


def test_class_api_single_instance(problems, native):
    """OptimalControlProblem::computeOptimalTrajectory: pins the first frame, warm-starts the next call."""
    prob = native.Problem("quadrotor", alpha=1.0, step_num=4)
    ora = _oracle.OracleProblem("quadrotor", alpha=1.0, step_num=4)
    frames, refs = prob.sample_inputs(1, 99)
    x1, f1 = prob.compute_optimal_trajectory(frames[0], refs[0])
    ox1, of1, _ = ora.solve_batch(frames, refs)
    assert rel_err(x1, ox1[0]) < REL_SOLUTION
    assert abs(x1[:prob.nf] - frames[0]).max() < 1e-3          # first frame pinned (to OSQP tolerance)
    x2, f2 = prob.compute_optimal_trajectory(frames[0], refs[0])  # continues from x1
    ox2, of2, _ = ora.solve_batch(frames, refs, x0=ox1)
    assert rel_err(x2, ox2[0]) < REL_SOLUTION
    assert f2 <= f1 + 1e-6


def test_full_size_batch_properties(problems, native):
    """BASELINE.json configs[2] at full size (4096 quadrotor instances), checked through properties
    that do not need the oracle at that size: every QP solved in the oracle's iteration count,
    the pinned first frame follows x_k = frame * (1 - 0.9^k) (alpha = 0.1 steps towards a
    pinned value), dynamics defects shrink, and a seeded sample equals the oracle."""
    prob, ora = problems("quadrotor")
    B = 4096
    frames, refs = prob.sample_inputs(B, 0xB200 + 2)
    s = prob.get_settings()
    s.sqp_alpha, s.sqp_step_num = 0.1, 10
    prob.solver.update_settings(s)
    x = np.zeros((B, prob.N)); f = np.zeros(B); st = np.zeros((B, native.NSTATS))
    prob.solver.solve_batch(frames, refs, prob.lbx, prob.ubx, prob.lbg, prob.ubg, x, f, st)
    assert np.isfinite(x).all() and np.isfinite(f).all()
    assert (st[:, native.STAT["qp_status"]] == native.QP_SOLVED).all()
    assert (st[:, native.STAT["sqp_steps"]] == 10).all()
    assert (st[:, native.STAT["admm_iters"]] == 250).all()          # 25 per QP, first termination check
    assert np.abs(x[:, :prob.nf] - frames * (1 - 0.9 ** 10)).max() < 5e-3
    pick = np.array([0, 1, 777, 2048, 4095])
    ora.set_schedule(10, 0.1)
    ora.set_qp_settings(_oracle.settings_from_b200(s))
    ox, of, ost = ora.solve_batch(frames[pick], refs[pick])
    assert rel_err(x[pick], ox) < REL_SOLUTION
    assert np.allclose(f[pick], of, rtol=1e-6)
    # a second tick warm-starts from the first: the objective keeps decreasing for every instance
    f2 = np.zeros(B)
    prob.solver.solve_batch(frames, refs, prob.lbx, prob.ubx, prob.lbg, prob.ubg, x, f2, st)
    assert np.isfinite(f2).all()


def test_empty_batch_and_bad_arguments(problems, native):
    prob, _ = problems("quadrotor")
    lib = native.cuda_lib()
    assert lib.ocp_b200_solve_batch(prob.solver.handle, 0, None, None, None, None, None, None, None, None, None) == 0
    assert lib.ocp_b200_solve_batch(prob.solver.handle, 2, None, None, None, None, None, None, None, None, None) == 1
    assert b"bad arguments" in lib.ocp_b200_last_error()
    assert lib.ocp_b200_solve_batch(None, 1, None, None, None, None, None, None, None, None, None) == 1


def _cartpole_yaml(verbose, gen_code, alpha=1.0, steps=6, horizon=8):
    return f"""
optimal_control_problem:
  discretization_settings:
    dt: 0.01
    horizon: {horizon}
  solver_settings:
    max_iter: 1000
    warm_start: true
    verbose: {str(verbose).lower()}
    gen_code: {str(gen_code).lower()}
    load_lib: false
    solve_method: CUDA_SQP
    SQP_settings:
      alpha: {alpha}
      step_num: {steps}
  OCP_variables:
    - name: state
      size: 4
      lower_bound: [-2.4, -.inf, -.inf, -.inf]
      upper_bound: [2.4, .inf, .inf, .inf]
    - name: force
      size: 1
      lower_bound: [-20.0]
      upper_bound: [20.0]
"""


def test_verbose_mode_and_gen_code(native, capfd):
    """verbose: true steps one SQP iteration at a time with the reference's verbose-only early exit
    (||dx||_2 < 1e-6, SQPOptimizationSolver.cpp:183-197); without convergence it must give the same
    iterate as the silent path.  gen_code: true serialises localSystemFunction (:403-425)."""
    from pathlib import Path
    quiet = native.Problem("cartpole", yaml_text=_cartpole_yaml(False, True))
    loud = native.Problem("cartpole", yaml_text=_cartpole_yaml(True, False))
    frame = np.array([0.05, 0.2, 0.0, 0.1, 0.0]); ref = np.zeros(4)
    xq, fq = quiet.compute_optimal_trajectory(frame, ref)
    xl, fl = loud.compute_optimal_trajectory(frame, ref)
    out = capfd.readouterr().out
    assert "SQP start" in out and "step 1/6" in out
    assert np.allclose(xq, xl, rtol=0, atol=1e-9)
    saved = Path(native.SHARE_DIR) / "code_gen" / "localSystemFunction.casadi"
    assert saved.exists() and saved.stat().st_size > 1000


def _random_qp(seed, n, m_extra, density=0.3):
    import scipy.sparse as sp
    rng = np.random.default_rng(seed)
    M = rng.standard_normal((n, n)) * (rng.random((n, n)) < density)
    P = M @ M.T + n * np.eye(n)
    G = rng.standard_normal((m_extra, n)) * (rng.random((m_extra, n)) < density)
    A = np.vstack([np.eye(n), G])
    xf = rng.standard_normal(n)
    l = np.concatenate([xf - rng.random(n), G @ xf - rng.random(m_extra)])
    u = np.concatenate([xf + rng.random(n), G @ xf + rng.random(m_extra)])
    l[n:n + 2] = u[n:n + 2] = (G @ xf)[:2]
    q = rng.standard_normal(n)

    def csc(Mat):
        S = sp.csc_matrix(Mat); S.sort_indices()
        return S.indptr.astype(np.int32), S.indices.astype(np.int32), S.data.astype(np.float64)
    return csc(P), q, csc(A), l, u


@pytest.mark.parametrize("n,m_extra", [(12, 9), (40, 25), (90, 40)])
def test_cucaqp_class_on_general_patterns(native, n, m_extra):
    """The CuCaQP life cycle (setDimension / setSystem / initSolver / solve / getSolution,
    CuCaQP.cpp:22-41, 271-288, 183-224) on QPs without stage structure: a single dense block up to
    64 columns (direct kernel), wider patterns through the PCG fallback kernel."""
    (hp, hi, hx), q, (ap, ai, ax), l, u = _random_qp(1000 + n, n, m_extra)
    m = n + m_extra
    x, y, info = native.cucaqp_solve(n, m, hp, hi, hx, q, ap, ai, ax, l, u, eps_abs=1e-6, eps_rel=1e-6)
    ox, oy, oinfo, _ = _oracle.qp_solve(n, m, hp, hi, hx, q, ap, ai, ax, l, u,
                                        settings=_oracle.settings_vector(eps_abs=1e-6, eps_rel=1e-6))
    assert info[native.INFO["status"]] == oinfo[0] == native.QP_SOLVED
    assert info[native.INFO["iters"]] == oinfo[1]
    assert rel_err(x, ox) < REL_SOLUTION
    assert rel_err(y, oy) < REL_SOLUTION


def test_cucaqp_fewer_constraints_than_variables(native):
    """The reference accepts any m > 0 (CuCaQP.cpp:22-41); a QP with m < n has no identity block at all."""
    import scipy.sparse as sp
    rng = np.random.default_rng(77)
    n, m = 14, 5
    M = rng.standard_normal((n, n)) * (rng.random((n, n)) < 0.4)
    S = sp.csc_matrix(M @ M.T + n * np.eye(n)); S.sort_indices()
    G = sp.csc_matrix(rng.standard_normal((m, n)) * (rng.random((m, n)) < 0.6)); G.sort_indices()
    xf = rng.standard_normal(n)
    l = G @ xf - rng.random(m); u = G @ xf + rng.random(m)
    l[0] = u[0]
    q = rng.standard_normal(n)
    args = (n, m, S.indptr.astype(np.int32), S.indices.astype(np.int32), S.data, q, G.indptr.astype(np.int32),
            G.indices.astype(np.int32), G.data, l, u)
    x, y, info = native.cucaqp_solve(*args, eps_abs=1e-7, eps_rel=1e-7)
    ox, oy, oinfo, _ = _oracle.qp_solve(*args, settings=_oracle.settings_vector(eps_abs=1e-7, eps_rel=1e-7))
    assert info[native.INFO["status"]] == oinfo[0] == native.QP_SOLVED
    assert info[native.INFO["iters"]] == oinfo[1]
    assert rel_err(x, ox) < REL_SOLUTION and rel_err(y, oy) < REL_SOLUTION


def test_inconsistent_bounds_give_a_zero_step(problems, native):
    """lbx > ubx on one variable: osqp_setup rejects the QP (validate_data); the reference ignores
    the failure (SQPOptimizationSolver.cpp:155-157) -- restated as a zero step on both sides."""
    prob, ora = problems("quadrotor")
    frames, refs = prob.sample_inputs(3, 17)
    lbx, ubx = prob.lbx.copy(), prob.ubx.copy()
    lbx[40], ubx[40] = 1.0, -1.0
    s = prob.get_settings()
    s.sqp_alpha, s.sqp_step_num = 0.5, 2
    prob.solver.update_settings(s)
    x0 = np.tile(frames, (1, prob.horizon))
    x = x0.copy(); st = np.zeros((3, native.NSTATS))
    prob.solver.solve_batch(frames, refs, lbx, ubx, prob.lbg, prob.ubg, x, None, st)
    assert np.array_equal(x, x0)
    assert (st[:, native.STAT["qp_status"]] == native.QP_UNSOLVED).all()
    assert (st[:, native.STAT["admm_iters"]] == 0).all()


def test_adaptive_rho_inside_a_batched_solve(problems, native):
    """Tight tolerances force rho updates (refactorisations on the device) inside the throughput plan."""
    prob, ora = problems("quadrotor")
    B = 160
    frames, refs = prob.sample_inputs(B, 23)
    s = prob.get_settings()
    s.sqp_alpha, s.sqp_step_num = 1.0, 2
    s.eps_abs = s.eps_rel = 1e-7
    prob.solver.update_settings(s)
    x = np.zeros((B, prob.N)); st = np.zeros((B, native.NSTATS))
    prob.solver.solve_batch(frames, refs, prob.lbx, prob.ubx, prob.lbg, prob.ubg, x, None, st)
    assert (st[:, native.STAT["rho_updates"]] >= 1).sum() > B // 4     # a good part of the batch adapts rho
    pick = [0, 79, 159] + [int(b) for b in np.flatnonzero(st[:, native.STAT["rho_updates"]] >= 1)[:3]]
    ora.set_schedule(2, 1.0)
    ora.set_qp_settings(_oracle.settings_from_b200(s))
    ox, of, ost = ora.solve_batch(frames[pick], refs[pick])
    assert np.array_equal(st[pick][:, native.STAT["admm_iters"]], ost[:, 2])
    assert np.array_equal(st[pick][:, native.STAT["rho_updates"]], ost[:, 7])
    assert rel_err(x[pick], ox) < REL_SOLUTION


@pytest.mark.parametrize("max_iter,eps", [(60, 1e-12), (40, 2e-5), (25, 1e-12)])
def test_iteration_limit_statuses(problems, native, max_iter, eps):
    """max_iter reached: OSQP re-tests with 10x tolerances (SOLVED_INACCURATE) before reporting
    MAX_ITER_REACHED; the last iterate is returned either way.  Also covers limits that are not a
    multiple of check_termination."""
    prob, ora = problems("quadrotor")
    hv, q, av, l, u = _qp_case(prob, ora, 31, B=2)
    s = prob.get_settings()
    s.eps_abs = s.eps_rel = eps
    s.admm_max_iter = max_iter
    prob.solver.update_settings(s)
    x, y, info = prob.solver.qp_solve_batch(hv, q, av, l, u)
    sv = _oracle.settings_from_b200(s)
    for b in range(2):
        ox, oy, oinfo, _ = _oracle.qp_solve(prob.n, prob.m, prob.h_colptr, prob.h_rowidx, hv[b], q[b], prob.a_colptr,
                                            prob.a_rowidx, av[b], l[b], u[b], settings=sv)
        assert info[b, native.INFO["status"]] == oinfo[0]
        assert oinfo[0] in (native.QP_MAX_ITER, native.QP_SOLVED_INACCURATE, native.QP_SOLVED)
        assert info[b, native.INFO["iters"]] == oinfo[1] <= max_iter
        assert rel_err(x[b], ox) < REL_SOLUTION


@pytest.mark.parametrize("name,horizon,plan", [
    ("cartpole", 9, "mixed"),      # blocks of 15 columns (odd size, generic code), border of 4: narrow-border path
    ("cartpole", 27, "mixed"),
    ("centroidal", 6, "mixed"),    # blocks of 36 (compile-time streamed code), border of 24: wide-border path
    ("cartpole", 40, "big"),       # blocks of 20, twisted sweeps through the two-chain ring
    ("quadrotor", 5, "multi"),     # two CTAs per SM, factor blocks in the slab
])
def test_streamed_factor_paths_match_oracle(native, monkeypatch, name, horizon, plan):
    """The slab-resident (streamed) factor code on problems small enough to compare quickly: the launch
    plan is forced and the factor kept out of shared memory (OCP_B200_PLAN / OCP_B200_FORCE_STREAM are
    read when the handle is created)."""
    monkeypatch.setenv("OCP_B200_PLAN", plan)
    monkeypatch.setenv("OCP_B200_FORCE_STREAM", "1")
    prob = native.Problem(name, horizon=horizon)
    ora = _oracle.OracleProblem(name, horizon=horizon)
    B, alpha, steps = 3, 0.5, 3
    frames, refs = prob.sample_inputs(B, 0xB200 + 11)
    s = prob.get_settings()
    s.sqp_alpha, s.sqp_step_num = alpha, steps
    prob.solver.update_settings(s)
    x0 = np.tile(frames, (1, prob.horizon))
    x = x0.copy(); f = np.zeros(B); st = np.zeros((B, native.NSTATS))
    prob.solver.solve_batch(frames, refs, prob.lbx, prob.ubx, prob.lbg, prob.ubg, x, f, st)
    assert prob.solver.device_dims()["resident"] & 2      # direct block-tridiagonal kernel, not PCG
    ora.set_schedule(steps, alpha)
    ora.set_qp_settings(_oracle.settings_from_b200(s))
    ox, of, ost = ora.solve_batch(frames, refs, x0=x0)
    assert np.isfinite(ox).all()
    assert np.array_equal(st[:, native.STAT["admm_iters"]], ost[:, 2])
    assert np.array_equal(st[:, native.STAT["qp_status"]], ost[:, 0])
    assert rel_err(x, ox) < REL_SOLUTION
    assert np.allclose(f, of, rtol=1e-6, atol=1e-9)


@pytest.mark.parametrize("name,horizon", [("quadrotor", 20), ("quadrotor", 5), ("cartpole", 20)])
def test_compact_plan_matches_oracle(native, monkeypatch, name, horizon):
    """The four-CTA/SM throughput kernel (admm_compact_kernel.cuh: stage-periodic index templates, slab-streamed
    q / l / u / D / E / P, phase-shared buffers) forced onto small batches: same iterates as the oracle, and --
    with tight tolerances -- through its rho-update refactorisation path (x, z, y parked in the slab)."""
    monkeypatch.setenv("OCP_B200_PLAN", "compact")
    prob = native.Problem(name, horizon=horizon)
    ora = _oracle.OracleProblem(name, horizon=horizon)
    assert prob.solver.launch_plan()["wide"]["place"] == 4 and prob.solver.launch_plan()["deep"]["place"] == 4
    B = 3
    frames, refs = prob.sample_inputs(B, 0xB200 + 17)
    for alpha, steps, eps in ((0.5, 3, 1e-3), (1.0, 2, 1e-7)):
        s = prob.get_settings()
        s.sqp_alpha, s.sqp_step_num = alpha, steps
        s.eps_abs = s.eps_rel = eps
        prob.solver.update_settings(s)
        x0 = np.tile(frames, (1, prob.horizon))
        x = x0.copy(); f = np.zeros(B); st = np.zeros((B, native.NSTATS))
        prob.solver.solve_batch(frames, refs, prob.lbx, prob.ubx, prob.lbg, prob.ubg, x, f, st)
        ora.set_schedule(steps, alpha)
        ora.set_qp_settings(_oracle.settings_from_b200(s))
        ox, of, ost = ora.solve_batch(frames, refs, x0=x0)
        assert np.isfinite(ox).all()
        assert np.array_equal(st[:, native.STAT["admm_iters"]], ost[:, 2])
        assert np.array_equal(st[:, native.STAT["rho_updates"]], ost[:, 7])
        assert np.array_equal(st[:, native.STAT["qp_status"]], ost[:, 0])
        assert rel_err(x, ox) < REL_SOLUTION
        assert np.allclose(f, of, rtol=1e-6, atol=1e-9)
    if name == "quadrotor" and horizon == 20:
        assert st[:, native.STAT["rho_updates"]].sum() >= 1      # the refactorisation path ran


def test_launch_plans_of_the_headline_shape(problems, native):
    """The H = 20 quadrotor runs its small batches on the all-shared-memory placement (it is within 2 KB of the limit:
    once it did not fit, the plan fell back to the streamed placement and every latency number was 40 % worse without
    any test noticing) and its large batches on the compact kernel at four CTAs per SM."""
    prob, _ = problems("quadrotor")
    plan = prob.solver.launch_plan()
    assert plan["deep"]["place"] == 1 and plan["deep"]["threads"] == 384
    assert plan["wide"]["place"] == 4 and plan["wide"]["ctas_per_sm"] == 4


def test_compact_plan_qp_level(native, monkeypatch):
    """QP-level entry points on the compact kernel: primal / dual solutions, residuals, the check trace, a primal
    and a dual infeasible QP (certificate -> NaN solution) and inconsistent bounds (zero step)."""
    monkeypatch.setenv("OCP_B200_PLAN", "compact")
    prob = native.Problem("quadrotor")
    ora = _oracle.OracleProblem("quadrotor")
    hv, q, av, l, u = _qp_case(prob, ora, 21)
    s = prob.get_settings()
    s.eps_abs = s.eps_rel = 1e-7
    prob.solver.update_settings(s)
    x, y, info = prob.solver.qp_solve_batch(hv, q, av, l, u)
    sv = _oracle.settings_from_b200(s)
    for b in range(hv.shape[0]):
        ox, oy, oinfo, otrace = _oracle.qp_solve(prob.n, prob.m, prob.h_colptr, prob.h_rowidx, hv[b], q[b], prob.a_colptr,
                                                 prob.a_rowidx, av[b], l[b], u[b], settings=sv)
        assert info[b, native.INFO["status"]] == oinfo[0] == native.QP_SOLVED
        assert info[b, native.INFO["iters"]] == oinfo[1]
        assert info[b, native.INFO["rho_updates"]] == oinfo[6]
        assert rel_err(x[b], ox) < REL_SOLUTION and rel_err(y[b], oy) < REL_SOLUTION
    trace, tx, ty = prob.solver.admm_trace(hv[0], q[0], av[0], l[0], u[0])
    ox, oy, oinfo, otrace = _oracle.qp_solve(prob.n, prob.m, prob.h_colptr, prob.h_rowidx, hv[0], q[0], prob.a_colptr,
                                             prob.a_rowidx, av[0], l[0], u[0], settings=sv)
    assert len(trace) == len(otrace) > 1 and np.array_equal(trace[:, 0], otrace[:, 0])
    assert np.allclose(trace[:, 3], otrace[:, 3], rtol=1e-6)
    assert np.allclose(trace[:, 1], otrace[:, 1], rtol=1e-4, atol=1e-10)
    # primal infeasible: the whole first frame is pinned and the first defect row fixes the roll angle of stage 1
    # (up to its residual), so a bound row that wants that angle in [5, 6] cannot hold
    l2, u2 = l.copy(), u.copy()
    row = prob.np_ + prob.nf + 3
    l2[:, row], u2[:, row] = 5.0, 6.0
    x2, y2, info2 = prob.solver.qp_solve_batch(hv, q, av, l2, u2)
    for b in range(hv.shape[0]):
        ox, oy, oinfo, _ = _oracle.qp_solve(prob.n, prob.m, prob.h_colptr, prob.h_rowidx, hv[b], q[b], prob.a_colptr,
                                            prob.a_rowidx, av[b], l2[b], u2[b], settings=sv)
        assert info2[b, native.INFO["status"]] == oinfo[0] == native.QP_PRIMAL_INFEASIBLE
        assert info2[b, native.INFO["iters"]] == oinfo[1]
        assert np.array_equal(np.isnan(x2[b]), np.isnan(ox))
    # dual infeasible: no curvature, and the first rotor input of the last stage (rows 0..n-1 of A bound the
    # variables) released, so the linear cost decreases without limit along it.  The iterates grow without bound
    # here, and so do the rounding differences between the two linear solves: the certificate is the same, the
    # check at which it fires need not be.
    h4, l4, u4 = np.zeros_like(hv), l.copy(), u.copy()
    row = prob.n - 4
    l4[:, row], u4[:, row] = -np.inf, np.inf
    x4, y4, info4 = prob.solver.qp_solve_batch(h4, q, av, l4, u4)
    for b in range(hv.shape[0]):
        ox, oy, oinfo, _ = _oracle.qp_solve(prob.n, prob.m, prob.h_colptr, prob.h_rowidx, h4[b], q[b], prob.a_colptr,
                                            prob.a_rowidx, av[b], l4[b], u4[b], settings=sv)
        assert info4[b, native.INFO["status"]] == oinfo[0] == native.QP_DUAL_INFEASIBLE
        assert np.isnan(x4[b]).all() and np.isnan(ox).all()
    # l > u: osqp_setup refuses, zero step
    l3 = l.copy(); l3[:, 5] = u[:, 5] + 1.0
    x3, y3, info3 = prob.solver.qp_solve_batch(hv, q, av, l3, u)
    assert (info3[:, native.INFO["status"]] == native.QP_UNSOLVED).all() and (x3 == 0).all()


def test_repeated_batches_are_bit_identical(problems, native):
    """compute-sanitizer's racecheck is closed on the GPU pool this is developed on; the next best evidence against
    races in the hand-numbered named barriers / phase-shared buffers: the same batch, solved three times with every SM
    at its full residency (CTAs meet in different phase combinations every time), gives the same bits, and so does
    every instance solved alone on the other launch plan."""
    prob, _ = problems("quadrotor")
    B = 1000
    frames, refs = prob.sample_inputs(B, 0xB200 + 77)
    s = prob.get_settings()
    s.sqp_alpha, s.sqp_step_num = 0.3, 3
    s.eps_abs = s.eps_rel = 1e-5
    prob.solver.update_settings(s)
    runs = []
    for _ in range(3):
        x = np.zeros((B, prob.N)); st = np.zeros((B, native.NSTATS))
        prob.solver.solve_batch(frames, refs, prob.lbx, prob.ubx, prob.lbg, prob.ubg, x, None, st)
        runs.append((x, st))
    for x, st in runs[1:]:
        assert np.array_equal(x, runs[0][0]) and np.array_equal(st, runs[0][1])
    for b in (0, 333, 999):
        xb = np.zeros((1, prob.N))
        prob.solver.solve_batch(frames[b:b + 1], refs[b:b + 1], prob.lbx, prob.ubx, prob.lbg, prob.ubg, xb)
        assert np.array_equal(xb[0], runs[0][0][b])
