"""The generated stage-assembly kernel (kernel 1, host/src/StageCodegen.cpp) against the 40-digit sympy reference of
tests/stage_reference.py, on models that each exist for one code path of the generator.

The tests call the stage library's C entry points directly (ctypes, torch CUDA tensors), so they choose the leading
dimensions and may pass frames = NULL.  Per array they require |gpu - ref| <= 1e-12 * max(1, |ref|_inf); entries that
are exact constants (the identity 1.0, linear coefficients, infinite bounds) must be equal."""
import ctypes as C

import numpy as np
import pytest

import stage_reference as sr

pytestmark = pytest.mark.gpu

REL_VALUES = 1e-12
SENTINEL = -7.25e77


def _torch():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("no CUDA device")
    return torch


class StageLib:
    """ocp_b200_model_assemble / ocp_b200_model_objective of one stage library on torch CUDA tensors."""

    def __init__(self, problem):
        self.pr = problem
        self.lib = C.CDLL(problem.model_library)
        vp = C.c_void_p
        self.lib.ocp_b200_model_assemble.argtypes = [C.c_int] + [vp] * 8 + [C.c_int, vp, C.c_int, vp, C.c_int, vp, vp,
                                                                            C.c_int, vp]
        self.lib.ocp_b200_model_objective.argtypes = [C.c_int, vp, vp, vp, vp]
        self.torch = _torch()

    def _t(self, a):
        return self.torch.from_numpy(np.ascontiguousarray(a, np.float64)).cuda()

    def assemble(self, p, x, frames=None, pad=0):
        """-> (hv, q, av, l, u) as numpy [B, ld] arrays, ld = nnz (or n, m) + pad, sentinel-filled beforehand."""
        torch, pr = self.torch, self.pr
        B = x.shape[0]
        ld = dict(h=pr.nnz_h + pad, n=pr.n + pad, a=pr.nnz_a + pad, m=pr.m + pad)
        out = {k: torch.full((B, v), SENTINEL, dtype=torch.float64, device="cuda") for k, v in
               (("hv", ld["h"]), ("q", ld["n"]), ("av", ld["a"]), ("l", ld["m"]), ("u", ld["m"]))}
        ins = [self._t(x), self._t(p) if pr.np_ else None, self._t(frames) if frames is not None else None,
               self._t(pr.lbx), self._t(pr.ubx), self._t(pr.lbg), self._t(pr.ubg)]
        ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        rc = self.lib.ocp_b200_model_assemble(B, *[ptr(t) for t in ins], ptr(out["hv"]), ld["h"], ptr(out["q"]), ld["n"],
                                              ptr(out["av"]), ld["a"], ptr(out["l"]), ptr(out["u"]), ld["m"], stream)
        assert rc == 0, rc
        torch.cuda.synchronize()
        res = tuple(out[k].cpu().numpy() for k in ("hv", "q", "av", "l", "u"))
        widths = (pr.nnz_h, pr.n, pr.nnz_a, pr.m, pr.m)
        for arr, w in zip(res, widths):    # nothing written outside [0, nnz) of a row
            assert (arr[:, w:] == SENTINEL).all()
        return tuple(arr[:, :w] for arr, w in zip(res, widths))

    def objective(self, p, x):
        torch = self.torch
        B = x.shape[0]
        f = torch.full((B,), SENTINEL, dtype=torch.float64, device="cuda")
        xt, pt = self._t(x), (self._t(p) if self.pr.np_ else None)
        rc = self.lib.ocp_b200_model_objective(B, C.c_void_p(xt.data_ptr()), None if pt is None else C.c_void_p(pt.data_ptr()),
                                               C.c_void_p(f.data_ptr()), C.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0, rc
        torch.cuda.synchronize()
        return f.cpu().numpy()


_refs, _libs = {}, {}


def _ref(name):
    if name not in _refs:
        _refs[name] = sr.Reference(sr.SPECS[name])
    return _refs[name]


def _lib(name, lanes=None):
    if (name, lanes) not in _libs:
        _libs[(name, lanes)] = StageLib(sr.build_product(name, lanes))
    return _libs[(name, lanes)]


def _close(name, what, got, ref, worst):
    err = np.abs(got - ref).max() if got.size else 0.0
    assert err <= REL_VALUES * max(1.0, np.abs(ref).max() if ref.size else 0.0), (name, what, err)
    worst[what] = max(worst.get(what, 0.0), float(err))


def _exact_positions(pr, spec):
    """CCS positions of A whose value is an exact constant: the identity block, and the linear coefficients of the
    `constants` model."""
    pos = [pr.a_colptr[j] for j in range(pr.n)]   # the identity row heads every column
    if spec.name == "constants":
        pos = list(range(pr.nnz_a))
    return np.array(pos)


@pytest.mark.parametrize("name", sorted(sr.SPECS))
@pytest.mark.parametrize("with_frames", [False, True])
def test_values_match_reference(native, name, with_frames):
    spec = sr.SPECS[name]
    lib, ref = _lib(name), _ref(name)
    frames, p, x = spec.sample(3, 0x5A + len(name))
    hv, q, av, l, u = lib.assemble(p, x, frames if with_frames else None)
    f = lib.objective(p, x)
    worst = {}
    pos = _exact_positions(lib.pr, spec)
    for b in range(3):
        rhv, rq, rav, rl, ru, rf = ref.local_system(lib.pr, p[b], x[b], frames[b] if with_frames else None)
        for what, got, want in (("H", hv[b], rhv), ("q", q[b], rq), ("J", av[b], rav)):
            _close(name, what, got, want, worst)
        for what, got, want in (("l", l[b], rl), ("u", u[b], ru)):
            fin = np.isfinite(want)
            assert np.array_equal(got[~fin], want[~fin]), (name, what)   # +-inf bounds exactly
            _close(name, what, got[fin], want[fin], worst)
        _close(name, "f", np.array([f[b]]), np.array([rf]), worst)
        assert np.array_equal(av[b][pos].view(np.int64), rav[pos].view(np.int64)), (name, "exact J entries")
    print(f"{name} frames={with_frames}: largest |gpu - ref| " + ", ".join(f"{k} {v:.2e}" for k, v in worst.items()))


@pytest.mark.parametrize("name", sorted(sr.SPECS))
def test_batch_shapes_and_leading_dimensions(native, name):
    """B in {1, UNITS_PER_WARP - 1, UNITS_PER_WARP + 1, 1000} (ragged last warps), ld = nnz and nnz + 1 (odd: the
    16-byte alignment of a row alternates between instances): every instance bit-identical to the same instance
    assembled alone with ld = nnz, and nothing written past nnz in any row."""
    spec = sr.SPECS[name]
    lib = _lib(name)
    upw = 32 // sr.generated_header(lib.pr)["UNIT_LANES"]
    frames, p, x = spec.sample(1000, 0xB5 + len(name))
    alone = {}
    for B in sorted({1, max(upw - 1, 1), upw + 1, 1000}):
        for pad in (0, 1):
            got = lib.assemble(p[:B], x[:B], frames[:B], pad=pad)
            check = range(B) if B < 1000 else list(range(0, 1000, 37)) + [998, 999]
            for b in check:
                if b not in alone:
                    alone[b] = lib.assemble(p[b:b + 1], x[b:b + 1], frames[b:b + 1])
                for g, a in zip(got, alone[b]):
                    assert np.array_equal(g[b].view(np.int64), a[0].view(np.int64)), (name, B, pad, b)
            if B == 1000:   # ... and every instance matches the reference of the batch, not only its neighbours
                for b in (0, 517, 999):
                    rhv, rq, rav, rl, ru, _ = _ref(name).local_system(lib.pr, p[b], x[b], frames[b])
                    _close(name, "H", got[0][b], rhv, {})
                    _close(name, "J", got[2][b], rav, {})
    f = lib.objective(p, x)
    for b in (0, 1, 999):
        assert np.array_equal(f[b:b + 1], lib.objective(p[b:b + 1], x[b:b + 1]))


@pytest.mark.parametrize("name,lanes", [("ops_all", 16), ("rate_cost", 32)])
def test_forced_lane_counts_are_bit_identical(native, name, lanes):
    """Each lane runs the same template text whatever the unit width: the results do not depend on UNIT_LANES."""
    spec = sr.SPECS[name]
    frames, p, x = spec.sample(37, 0x1A + lanes)
    a = _lib(name).assemble(p, x, frames, pad=1)
    b = _lib(name, lanes).assemble(p, x, frames, pad=1)
    for u, v in zip(a, b):
        assert np.array_equal(u.view(np.int64), v.view(np.int64))
    assert np.array_equal(_lib(name).objective(p, x), _lib(name, lanes).objective(p, x))


@pytest.fixture(scope="module")
def quad128(native):
    import _oracle
    return sr.build_named("quadrotor", 128), _oracle.OracleProblem("quadrotor", horizon=128)


def test_quadrotor_long_horizon_matches_oracle(native, quad128):
    """quadrotor H = 128 (the p group stores straight to global memory; the objective loop runs over 129 groups)
    against the oracle's local system and objective."""
    pr, ora = quad128
    lib = StageLib(pr)
    frames, refs = pr.sample_inputs(5, 0xC0DE)
    rng = np.random.default_rng(3)
    x = np.tile(frames, (1, 128)) + rng.uniform(-0.05, 0.05, (5, pr.N))
    for pad in (0, 1):
        for fr in (frames, None):
            got = lib.assemble(refs, x, fr, pad=pad)
            for b in range(5):
                want = ora.local_system(None if fr is None else fr[b], refs[b], x[b])
                for what, g, w in zip(("H", "q", "J", "l", "u"), got, want):
                    fin = np.isfinite(w)
                    assert np.array_equal(g[b][~fin], w[~fin]), what
                    _close("quadrotor128", what, g[b][fin], w[fin], {})
    f = lib.objective(refs, x)
    for b in range(5):
        assert abs(f[b] - ora.objective(refs[b], x[b])) <= REL_VALUES * max(1.0, abs(f[b]))


def test_sqp_solve_quadrotor_long_horizon(native, quad128):
    """One SQP solve at H = 128, B = 3: the long-horizon layout reaches the ADMM kernels intact."""
    import _oracle
    pr, ora = quad128
    frames, refs = pr.sample_inputs(3, 0xC0DF)
    s = pr.get_settings()
    ora.set_qp_settings(_oracle.settings_from_b200(s))
    ora.set_schedule(1, 1.0)
    x = np.tile(frames, (1, 128))
    f = np.zeros(3); st = np.zeros((3, native.NSTATS))
    pr.solver.update_settings(_settings_one_step(pr, s))
    pr.solver.solve_batch(frames, refs, pr.lbx, pr.ubx, pr.lbg, pr.ubg, x, f, st)
    ox, of, ost = ora.solve_batch(frames, refs, x0=np.tile(frames, (1, 128)))
    assert np.array_equal(st[:, native.STAT["qp_status"]], ost[:, 0])
    assert np.array_equal(st[:, native.STAT["admm_iters"]], ost[:, 2])
    assert np.abs(x - ox).max() <= 1e-6 * max(1.0, np.abs(ox).max())


def _settings_one_step(pr, s):
    s = s.copy()
    s.sqp_step_num, s.sqp_alpha = 1, 1.0
    return s


def test_sqp_solve_param_rows_matches_reference_qp(native):
    """One SQP step of `param_rows` (border rows built from p) at B = 3 against the oracle's OSQP on the reference
    local system: same status and iteration count, x within 1e-6."""
    import _oracle
    spec = sr.SPECS["param_rows"]
    pr, ref = sr.build_product("param_rows"), _ref("param_rows")
    frames, p, _ = spec.sample(3, 0x77)
    x0 = np.tile(frames, (1, spec.horizon))
    s = _settings_one_step(pr, pr.get_settings())
    s.eps_abs = s.eps_rel = 1e-7
    pr.solver.update_settings(s)
    x = x0.copy(); f = np.zeros(3); st = np.zeros((3, native.NSTATS))
    pr.solver.solve_batch(frames, p, pr.lbx, pr.ubx, pr.lbg, pr.ubg, x, f, st)
    sv = _oracle.settings_from_b200(s)
    for b in range(3):
        hv, q, av, l, u, _ = ref.local_system(pr, p[b], x0[b], frames[b])
        dx, _, info, _ = _oracle.qp_solve(pr.n, pr.m, pr.h_colptr, pr.h_rowidx, hv, q, pr.a_colptr, pr.a_rowidx, av, l, u,
                                          settings=sv)
        assert st[b, native.STAT["qp_status"]] == info[0]
        assert st[b, native.STAT["admm_iters"]] == info[1]
        want = x0[b] + dx[pr.np_:]
        assert np.abs(x[b] - want).max() <= 1e-6 * max(1.0, np.abs(want).max())
