"""High-precision reference of the generated stage-assembly kernel -- TEST INFRASTRUCTURE.

Each test model below is written once against a small math namespace and a registration object with the
front end's method names (``get_variable``, ``reference_``, ``add_vector_cost``, ``add_scalar_cost``,
``add_equation_constraint``, ``add_inequality_constraint``).  It runs twice:

* with ``optimal_control_problem_b200.symbolic`` (``SXMath`` / ``OptimalControlProblem``): genSolver() builds the
  product -- casadi-lite AD, StageCodegen, nvcc;
* with sympy symbols (``SymMath`` / ``SymOCP``): the reference.  It shares no code with casadi-lite.

The reference builds the local system exactly as the front end defines it: w = [p; x], c = [p; x; g]; g is
left - right for equations and the expression itself for inequalities, in registration order; a vector cost is
sum_i w_i v_i^2; l - c and u - c with l = [p; lbx; lbg], u = [p; ubx; ubg] and, when frames are given, the first
frame pinned.  Every float constant of an expression is replaced by the exact rational it stands for, the
derivatives are taken by sympy and the values evaluated by mpmath at 40 significant digits, then rounded to
float64.  Non-smooth functions (fabs, sign, fmin, fmax) are written as Piecewise, so their derivatives are the
one-sided ones of the branch taken; the test points keep every argument away from the kinks.
"""
from __future__ import annotations

import atexit
import math
import os
import shutil
import tempfile
from dataclasses import dataclass, field

import numpy as np

INF = math.inf


# ---------------------------------------------------------------------------------------------
# math namespaces
# ---------------------------------------------------------------------------------------------
class SXMath:
    """The product: optimal_control_problem_b200.symbolic."""

    def __init__(self):
        import optimal_control_problem_b200.symbolic as sym
        for name in ("sin", "cos", "tan", "asin", "acos", "atan", "exp", "log", "sqrt", "fabs", "sign", "tanh", "sinh",
                     "cosh", "sq", "pow", "atan2", "fmin", "fmax"):
            setattr(self, name, getattr(sym, name))
        self.vec = sym.vertcat


class SymMath:
    """The reference: sympy."""

    def __init__(self):
        import sympy as sp
        self.sp = sp
        for name in ("sin", "cos", "tan", "asin", "acos", "atan", "exp", "log", "sqrt", "tanh", "sinh", "cosh", "atan2"):
            setattr(self, name, getattr(sp, name))

    def vec(self, parts):
        return [self.sp.sympify(p) for p in parts]

    def sq(self, a): return a * a
    def pow(self, a, b): return self.sp.Pow(a, b)
    def fabs(self, a): return self.sp.Piecewise((a, a >= 0), (-a, True))
    def sign(self, a): return self.sp.Piecewise((1, a > 0), (-1, a < 0), (0, True))
    def fmin(self, a, b): return self.sp.Piecewise((a, self.sp.sympify(a) < b), (b, True))
    def fmax(self, a, b): return self.sp.Piecewise((a, self.sp.sympify(b) < a), (b, True))


# ---------------------------------------------------------------------------------------------
# model specifications
# ---------------------------------------------------------------------------------------------
@dataclass
class Spec:
    name: str
    fields: list                # [(name, size, lower bounds, upper bounds)] of one frame
    np_: int
    horizon: int
    deploy: object              # deploy(ocp, M)
    x_range: tuple = (0.2, 0.6)  # instance sampling: x and p uniform in these ranges
    p_range: tuple = (0.5, 1.5)
    dt: float = 0.1
    extra: dict = field(default_factory=dict)

    @property
    def nf(self):
        return sum(f[1] for f in self.fields)

    def yaml(self) -> str:
        def vec(v):
            return "[" + ", ".join(".inf" if b == INF else "-.inf" if b == -INF else repr(float(b)) for b in v) + "]"
        s = (f"  discretization_settings:\n    dt: {self.dt}\n    horizon: {self.horizon}\n"
             "  solver_settings:\n    max_iter: 1000\n    warm_start: true\n    verbose: false\n    gen_code: false\n"
             "    recompile: false\n    load_lib: false\n    solve_method: CUDA_SQP\n"
             "    SQP_settings:\n      alpha: 1.0\n      step_num: 1\n  OCP_variables:\n")
        for name, size, lb, ub in self.fields:
            s += f"    - name: {name}\n      size: {size}\n      lower_bound: {vec(lb)}\n      upper_bound: {vec(ub)}\n"
        return s

    def bounds(self):
        lb = np.concatenate([np.asarray(f[2], float) for f in self.fields])
        ub = np.concatenate([np.asarray(f[3], float) for f in self.fields])
        return np.tile(lb, self.horizon), np.tile(ub, self.horizon)

    def sample(self, B: int, seed: int):
        """(frames [B, nf], p [B, np], x [B, N]): x and p inside the domains the model was written for."""
        rng = np.random.default_rng(seed)
        x = rng.uniform(*self.x_range, size=(B, self.nf * self.horizon))
        p = rng.uniform(*self.p_range, size=(B, self.np_))
        frames = rng.uniform(*self.x_range, size=(B, self.nf))
        return frames, p, x


QUADRANTS = ((1.0, 1.0), (-1.0, 1.0), (-1.0, -1.0), (1.0, -1.0))


def _ops_all(o, M):
    """Every operator StageCodegen emits, in g rows (J) and in the cost (H).  x, u in [0.2, 0.6], p in [0.5, 1.5]:
    asin / acos arguments in [-0.3, 0.3], log / sqrt / pow bases positive, atan2 in all four quadrants, fmin / fmax /
    fabs / sign with both outcomes (the derivatives of fmin and fmax emit `<`), every argument at least 0.1 from a
    kink."""
    P = o.reference_
    H = o.horizon
    for k in range(H):
        x, u = o.get_variable(k, "x"), o.get_variable(k, "u")
        a, b, c, d, e, f = x[0], x[1], x[2], x[3], u[0], u[1]
        q1, q2 = QUADRANTS[(2 * k) % 4], QUADRANTS[(2 * k + 1) % 4]
        rows = [
            M.sin(a) * b + M.cos(c) - M.tan(0.5 * d),
            M.asin(1.5 * (a - 0.4)) + M.acos(1.5 * (b - 0.4)) * e,
            M.atan(c * d) + M.exp(0.5 * e) - M.log(a + P[1]),
            M.sqrt(b + P[2]) * M.pow(c + 0.5, P[0]) + M.fabs(d - 0.9) + M.fabs(e + 0.1) * f,
            M.atan2(q1[0] * a, q1[1] * b) + M.atan2(q2[0] * c, q2[1] * d),
            M.fmin(a, b + 0.5) * c + M.fmin(c, d - 0.5) + M.fmax(e, f + 0.5) * a + M.fmax(a, b - 0.5),
            M.tanh(a - b) + M.sinh(c) * M.cosh(d) + M.sign(e - 0.9) * a + M.sign(f + 0.1) * b,
            a / (b + 1.0) - M.sq(c) + (-d) * e,
        ]
        o.add_inequality_constraint("ops", [-INF, -1.0, -INF, 0.0, -5.0, -INF, -3.0, -INF], M.vec(rows),
                                    [INF, INF, 2.0, INF, 5.0, 4.0, INF, INF])
        o.add_vector_cost([1.0, 2.0, 0.5, 1.5], M.vec([a - 0.3 * P[0], b - 0.3 * P[1], c - 0.3 * P[2], d]))
        o.add_scalar_cost(
            M.exp(a * b) + M.log(c + P[0]) * M.sqrt(d + 0.1) + M.sinh(e) * M.cosh(f) + M.tanh(a * c) + M.atan(b * d)
            + M.sin(a) * M.cos(b) + M.asin(1.5 * (c - 0.4)) * M.acos(1.5 * (d - 0.4)) + M.pow(a + 0.5, P[1])
            + M.atan2(q2[0] * e, q2[1] * f) * a + M.fmin(a * b, c + 0.4) * d + M.fmin(a, b - 0.5) * e
            + M.fmax(d * e + 0.2, f - 0.5) * b + M.fmax(c - 0.6, d * e) * c + M.fabs(a - 0.9) * b + M.fabs(c + 0.1) * d
            + M.sign(d - 0.9) * e * e + M.sq(e - f) + M.tan(0.5 * a) * c / (d + 1.0))
        if k + 1 < H:
            xn = o.get_variable(k + 1, "x")
            o.add_equation_constraint("dynamics", xn, M.vec([a + 0.1 * M.sin(e), b + 0.1 * M.cos(f) * a,
                                                             0.9 * c + 0.1 * a * b, d + 0.05 * M.exp(-e)]))


def _param_rows(o, M):
    """p inside dynamics and inequality rows (border rows: the p group gets Jacobian tangents and owns rows beyond its
    identity block), a g row that reads p only, and a constant g row (owner: group 0)."""
    P = o.reference_
    H = o.horizon
    for k in range(H):
        x, u = o.get_variable(k, "x"), o.get_variable(k, "u")
        o.add_vector_cost([1.0, 2.0, 3.0], M.vec([x[0] - P[0], x[1] - P[1], x[2] - P[2]]))
        o.add_vector_cost([0.1, 0.2], M.vec([u[0], u[1]]))
        o.add_scalar_cost(0.05 * P[3] * x[0] * u[0])
        if k + 1 < H:
            o.add_equation_constraint("dynamics", o.get_variable(k + 1, "x"),
                                      M.vec([x[0] + 0.1 * x[1] * P[0], x[1] + 0.1 * (u[0] - P[1] * M.sin(x[0])),
                                             x[2] + 0.1 * u[1] * P[2]]))
        o.add_inequality_constraint("mixed", [-2.0, -INF], M.vec([x[0] + P[3] * u[0], x[1] * x[1] - P[0]]), [2.0, 1.0])
    o.add_inequality_constraint("p_only", [-INF], M.vec([P[0] * P[1] + M.sin(P[2])]), [5.0])
    o.add_inequality_constraint("constant", [0.0], M.vec([2.0]), [3.0])


def _rate_cost(o, M):
    """A cost that couples neighbouring stages, (u_k - u_{k-1})^2, and a cost term with no variable.  Every stage but
    the last owns 10 g rows, more than UNIT_LANES = 8: lane-select runs in 2 chunks."""
    P = o.reference_
    H = o.horizon
    o.add_scalar_cost(1.25)
    for k in range(H):
        x, u = o.get_variable(k, "x"), o.get_variable(k, "u")
        o.add_vector_cost([1.0, 1.0, 2.0, 0.5, 0.5], M.vec([x[0] - P[0], x[1] - P[1], x[2], x[3], x[4]]))
        if k > 0:
            up = o.get_variable(k - 1, "u")
            o.add_vector_cost([3.0, 2.0, 1.0], M.vec([u[0] - up[0], u[1] - up[1], u[2] - up[2]]))
        if k + 1 < H:
            o.add_equation_constraint("dynamics", o.get_variable(k + 1, "x"),
                                      M.vec([x[0] + 0.1 * x[1], x[1] + 0.1 * u[0] * M.cos(x[0]), x[2] + 0.1 * x[3] * u[1],
                                             x[3] + 0.1 * (u[2] - x[4]), x[4] + 0.1 * x[0] * x[2]]))
        o.add_inequality_constraint("path", [-INF] * 5,
                                    M.vec([x[0] * u[0], x[1] + u[1], x[2] * x[3] - u[2], M.sq(x[4]), x[0] + x[1] + x[2]]),
                                    [1.0, 2.0, 3.0, 4.0, 5.0])


def _no_param(o, M):
    """np = 0: no p group, no reference."""
    H = o.horizon
    for k in range(H):
        x, u = o.get_variable(k, "x"), o.get_variable(k, "u")
        o.add_vector_cost([1.0, 0.5, 0.25], M.vec([x[0] - 0.4, x[1], x[2]]))
        o.add_vector_cost([0.1], M.vec([u[0]]))
        if k + 1 < H:
            o.add_equation_constraint("dynamics", o.get_variable(k + 1, "x"),
                                      M.vec([x[0] + 0.1 * x[1], x[1] + 0.1 * (u[0] - M.sin(x[0])), x[2] + 0.1 * x[0] * u[0]]))


def _wide_param(o, M):
    """64 parameters, every one coupled to every stage by the cost: the p group's Hessian range holds 64 x 31
    entries, an image far over the shared-memory budget; the p group also runs 2 passes of 32 lanes."""
    P = o.reference_
    H = o.horizon
    for k in range(H):
        x, u = o.get_variable(k, "x"), o.get_variable(k, "u")
        o.add_vector_cost([1.0 + i / 64.0 for i in range(64)], M.vec([x[0] - P[i] for i in range(64)]))
        o.add_vector_cost([0.5, 0.1], M.vec([x[1] - P[63], u[0]]))
        if k + 1 < H:
            o.add_equation_constraint("dynamics", o.get_variable(k + 1, "x"),
                                      M.vec([x[0] + 0.1 * x[1], x[1] + 0.1 * (u[0] - M.sin(x[0]))]))


CONSTANTS = (0.1, 1.0 / 3.0, 1e-300, -2.5e300, 5e-324, -0.0)


def _constants(o, M):
    """Linear rows whose coefficients only print exactly with 17 significant digits (or need their exponent):
    their J entries are these literals and must arrive bit-exact."""
    P = o.reference_
    H = o.horizon
    c = CONSTANTS
    for k in range(H):
        x, u = o.get_variable(k, "x"), o.get_variable(k, "u")
        o.add_inequality_constraint("linear", [-INF] * 3,
                                    M.vec([c[0] * x[0] + c[1] * u[0], c[2] * x[0] + c[3] * u[0], c[4] * x[0] + c[5] * u[0]]),
                                    [1.0, 1.0, 1.0])
        o.add_vector_cost([1.0, 0.5], M.vec([x[0] - P[0], u[0]]))


SPECS = {
    "ops_all": Spec("ops_all", [("x", 4, [-INF, 0.0, -1.0, -INF], [INF, 1.0, INF, 2.0]), ("u", 2, [-1.0, -INF], [1.0, INF])],
                    3, 3, _ops_all),
    "param_rows": Spec("param_rows", [("x", 3, [-INF, -1.0, -INF], [INF, 1.0, 5.0]), ("u", 2, [-1.0, -1.0], [1.0, 1.0])],
                       4, 6, _param_rows),
    "rate_cost": Spec("rate_cost", [("x", 5, [-INF] * 5, [INF] * 5), ("u", 3, [-2.0, -2.0, -INF], [2.0, 2.0, INF])],
                      2, 5, _rate_cost),
    "no_param": Spec("no_param", [("x", 3, [-INF, -2.0, -INF], [INF, 2.0, INF]), ("u", 1, [-1.0], [1.0])], 0, 4, _no_param),
    "wide_param": Spec("wide_param", [("x", 2, [-INF, -INF], [INF, INF]), ("u", 1, [-1.0], [1.0])], 64, 30, _wide_param),
    "constants": Spec("constants", [("x", 1, [-INF], [INF]), ("u", 1, [-1.0], [1.0])], 1, 2, _constants),
}


# ---------------------------------------------------------------------------------------------
# the product: build a spec through the Python front end (memoised per process, private share directory)
# ---------------------------------------------------------------------------------------------
_built = {}
_share_root = None


def _share_dir(tag: str) -> str:
    global _share_root
    if _share_root is None:
        _share_root = tempfile.mkdtemp(prefix="ocp_stage_assembly_")
        atexit.register(shutil.rmtree, _share_root, True)
    path = os.path.join(_share_root, tag)
    os.makedirs(path, exist_ok=True)
    return path


def _with_share_dir(tag: str, env: dict, build):
    """Runs build() with genSolver()'s stage-library cache in a private directory and `env` set."""
    import optimal_control_problem_b200 as ocp
    lib = ocp.host_lib()
    keys = ["OCP_B200_SHARE_DIR", *env]
    saved = {k: os.environ.get(k) for k in keys}
    try:
        lib.ocp_host_set_share_dir(_share_dir(tag).encode())
        os.environ.update(env)
        return build()
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
        lib.ocp_host_set_share_dir(str(saved["OCP_B200_SHARE_DIR"] or ocp.SHARE_DIR).encode())


def build_product(name: str, lanes: int | None = None):
    """The generated problem of SPECS[name] (optimal_control_problem_b200.Problem); `lanes` forces
    OCP_B200_ASSEMBLE_LANES for its stage library."""
    key = (name, lanes)
    if key not in _built:
        spec = SPECS[name]
        tag = name if lanes is None else f"{name}_lanes{lanes}"

        def build():
            import optimal_control_problem_b200.symbolic as sym
            M = SXMath()

            class Model(sym.OptimalControlProblem):
                def deploy_constraints_and_add_cost(self):
                    spec.deploy(self, M)

            ocp = Model(spec.yaml(), name=f"stage_ref_{tag}")
            if spec.np_ > 0:
                ocp.set_reference(sym.SX.sym("ref", spec.np_))
            ocp.deploy_constraints_and_add_cost()
            ocp.gen_solver()
            return ocp

        env = {} if lanes is None else {"OCP_B200_ASSEMBLE_LANES": str(lanes)}
        _built[key] = _with_share_dir(tag, env, build)
    return _built[key].problem


def build_named(name: str, horizon: int):
    """A benchmark problem (problems/problems.cpp) at another horizon, in a private share directory."""
    import optimal_control_problem_b200 as ocp
    key = (name, horizon)
    if key not in _built:
        _built[key] = _with_share_dir(f"{name}_h{horizon}", {}, lambda: ocp.Problem(name, horizon=horizon))
    return _built[key]


def generated_header(problem) -> dict:
    """The generator's decisions, read from the generated .cu next to the stage library."""
    import re
    src = open(os.path.splitext(problem.model_library)[0] + ".cu").read()
    out = {}
    for key in ("NUM_GROUPS", "STAGE_A", "STAGE_H", "UNIT_LANES", "WARPS_PER_BLOCK"):
        out[key] = int(re.search(rf"\b{key} = (\d+)", src).group(1))
    m = re.search(r"// groups: (\d+), stage templates: (\d+)", src)
    out["templates"] = int(m.group(2))
    m = re.search(r"groups storing straight to global memory: (\d+), static shared memory of assemble_kernel: (\d+) bytes", src)
    out["direct_groups"], out["smem_bytes"] = int(m.group(1)), int(m.group(2))
    out["groups"] = [tuple(int(v) for v in g.split(",")) for g in re.findall(r"^  \{([-\d,]+)\},$", src, re.M)]
    out["source"] = src
    return out


# ---------------------------------------------------------------------------------------------
# the reference
# ---------------------------------------------------------------------------------------------
class SymOCP:
    """Registration object of the reference: the front end's method names on sympy expressions."""

    def __init__(self, spec: Spec):
        import sympy as sp
        self.spec, self.horizon = spec, spec.horizon
        nf, H = spec.nf, spec.horizon
        self.P = list(sp.symbols(f"p0:{spec.np_}", real=True)) if spec.np_ else []
        self.X = list(sp.symbols(f"x0:{nf * H}", real=True))
        self.reference_ = self.P if spec.np_ else None
        self.offsets, off = {}, 0
        for name, size, _, _ in spec.fields:
            self.offsets[name] = (off, size)
            off += size
        self.f_terms, self.g, self.lbg, self.ubg = [], [], [], []

    def get_variable(self, k, field):
        off, size = self.offsets[field]
        base = k * self.spec.nf + off
        return self.X[base:base + size]

    def add_scalar_cost(self, c):
        self.f_terms.append(c)

    def add_vector_cost(self, weights, v):
        assert len(weights) == len(v)
        self.f_terms.append(sum(w * e * e for w, e in zip(weights, v)))

    def add_equation_constraint(self, name, left, right=None):
        right = right if right is not None else [0] * len(left)
        assert len(left) == len(right)
        self.g += [a - b for a, b in zip(left, right)]
        self.lbg += [0.0] * len(left)
        self.ubg += [0.0] * len(left)

    def add_inequality_constraint(self, name, lower, expression, upper):
        assert len(lower) == len(expression) == len(upper)
        self.g += list(expression)
        self.lbg += [float(v) for v in lower]
        self.ubg += [float(v) for v in upper]


class Reference:
    """Exact local system of a model: sparse sympy derivatives, mpmath values at 40 digits, rounded to float64."""

    DPS = 40

    def __init__(self, spec: Spec, deploy=None):
        import sympy as sp
        self.spec = spec
        o = SymOCP(spec)
        (deploy or spec.deploy)(o, SymMath())
        exact = lambda e: sp.sympify(e).xreplace({a: sp.Rational(a) for a in sp.sympify(e).atoms(sp.Float)})
        terms = [exact(t) for t in o.f_terms]
        g = [exact(e) for e in o.g]
        w = o.P + o.X
        index = {s: i for i, s in enumerate(w)}
        self.np_, self.N, self.ng = len(o.P), len(o.X), len(g)
        self.n = self.np_ + self.N
        self.m = self.n + self.ng
        self.lbg, self.ubg = np.array(o.lbg, float), np.array(o.ubg, float)
        grad, hess = {}, {}
        for t in terms:
            for v in sorted(t.free_symbols, key=index.get):
                dv = sp.diff(t, v)
                if dv == 0:
                    continue
                grad[index[v]] = grad.get(index[v], 0) + dv
                for u_ in sorted(dv.free_symbols, key=index.get):
                    duv = sp.diff(dv, u_)
                    if duv != 0:
                        hess[(index[u_], index[v])] = hess.get((index[u_], index[v]), 0) + duv
        jac = {}
        for r, e in enumerate(g):
            for v in sorted(e.free_symbols, key=index.get):
                d = sp.diff(e, v)
                if d != 0:
                    jac[(self.n + r, index[v])] = d
        self.grad_keys, self.hess_keys, self.jac_keys = sorted(grad), sorted(hess), sorted(jac)
        exprs = [sum(terms) if terms else sp.Integer(0)] + [grad[k] for k in self.grad_keys] + \
                [hess[k] for k in self.hess_keys] + [jac[k] for k in self.jac_keys] + g
        self._fn = sp.lambdify(w, exprs, modules="mpmath", cse=True)

    def evaluate(self, p, x) -> dict:
        """f, grad [n], H (dense n x n), J (dense m x n) and g at one point, each entry rounded from 40 digits."""
        import mpmath
        with mpmath.workdps(self.DPS):
            vals = self._fn(*[mpmath.mpf(float(v)) for v in np.concatenate([np.asarray(p, float).ravel(), np.asarray(x, float).ravel()])])
            vals = [float(v) for v in vals]
        it = iter(vals)
        f = next(it)
        grad = np.zeros(self.n)
        for k in self.grad_keys:
            grad[k] = next(it)
        H = np.zeros((self.n, self.n))
        for k in self.hess_keys:
            H[k] = next(it)
        J = np.zeros((self.m, self.n))
        J[np.arange(self.n), np.arange(self.n)] = 1.0
        for k in self.jac_keys:
            J[k] = next(it)
        g = np.array([next(it) for _ in range(self.ng)])
        return dict(f=f, grad=grad, H=H, J=J, g=g)

    def local_system(self, problem, p, x, frame=None):
        """(hv, q, av, l, u, f) in the product's CCS value order; asserts that every nonzero of the exact H and J lies
        inside the product's pattern."""
        e = self.evaluate(p, x)
        lbx, ubx = self.spec.bounds()
        if frame is not None:
            lbx, ubx = lbx.copy(), ubx.copy()
            lbx[:self.spec.nf] = frame
            ubx[:self.spec.nf] = frame
        p = np.asarray(p, float).ravel()
        c = np.concatenate([p, np.asarray(x, float).ravel(), e["g"]])
        l = np.concatenate([p, lbx, self.lbg]) - c
        u = np.concatenate([p, ubx, self.ubg]) - c
        hv = _gather(e["H"], problem.h_colptr, problem.h_rowidx, "H")
        av = _gather(e["J"], problem.a_colptr, problem.a_rowidx, "J")
        return hv, e["grad"], av, l, u, e["f"]


def _gather(dense, colptr, rowidx, what):
    n = dense.shape[1]
    inside = np.zeros(dense.shape, bool)
    vals = np.empty(len(rowidx))
    for j in range(n):
        rows = rowidx[colptr[j]:colptr[j + 1]]
        inside[rows, j] = True
        vals[colptr[j]:colptr[j + 1]] = dense[rows, j]
    outside = np.argwhere((dense != 0) & ~inside)
    assert outside.size == 0, f"exact {what} has nonzeros outside the product's pattern: {outside[:8].tolist()}"
    return vals


# ---------------------------------------------------------------------------------------------
# the three benchmark models, for the check of the reference against tests/indep_models.py
# ---------------------------------------------------------------------------------------------
def indep_model_spec(name: str, horizon: int) -> Spec:
    """Spec of a benchmark model written with indep_models' model code (rk4 + ode on scalars)."""
    import indep_models as im
    model = im.MODELS[name]
    nx, nu = model.nx, model.nu

    def deploy(o, M):
        X, P = o.X, o.P
        g, _, _ = im.constraints(model, o.horizon, X, M)
        o.add_equation_constraint("model", g)
        o.lbg[:] = im.constraints(model, o.horizon, [0.0] * len(X), im.NumMath)[1]
        o.ubg[:] = im.constraints(model, o.horizon, [0.0] * len(X), im.NumMath)[2]
        o.add_scalar_cost(im.objective(model, o.horizon, X, P))

    return Spec(name, [("state", nx, model.lb[:nx], model.ub[:nx]), ("input", nu, model.lb[nx:], model.ub[nx:])],
                nx, horizon, deploy, dt=model.dt)
