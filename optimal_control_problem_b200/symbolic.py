"""Python front-end for defining optimal control problems (SURVEY.md 8f item 3).

The reference ships a pybind11 module that is commented out (src/pybind/python_bindings.cpp:380-445):
an ``OptimalControlProblem`` class to subclass in Python, with ``deploy_constraints_and_add_cost``
overridden and costs / constraints written as CasADi ``SX`` expressions.  This module is the working
counterpart with the same method names.  Expressions are opaque handles to the C++ ``casadi::SX``
objects of the host library (``host/casadi/casadi.hpp``); nothing symbolic happens in Python, and
``gen_solver()`` runs exactly the C++ ``OptimalControlProblem::genSolver()`` (symbolic AD, CUDA stage
code generation, nvcc).  Solving goes through the same classes and the same C ABI as a C++ caller.

    class CartPole(OptimalControlProblem):
        def deploy_constraints_and_add_cost(self):
            for k in range(self.horizon):
                x, u = self.get_variable(k, "state"), self.get_variable(k, "force")
                self.add_vector_cost([1.0, 10.0, 0.1, 0.1], x - self.reference_)
                if k + 1 < self.horizon:
                    self.add_equation_constraint("dynamics", self.get_variable(k + 1, "state"), step(x, u))
    ocp = CartPole(yaml_text, name="cartpole_py")
    ocp.set_reference(SX.sym("ref", 4))
    ocp.deploy_constraints_and_add_cost()
    ocp.gen_solver()
    x = ocp.compute_optimal_trajectory(frame, reference)
"""
from __future__ import annotations

import ctypes as C
from typing import Iterable, Sequence

import numpy as np

from . import Problem, _dp, _f64, _hcheck, host_lib

__all__ = ["SX", "OptimalControlProblem", "vertcat", "sin", "cos", "tan", "asin", "acos", "atan", "exp", "log", "sqrt",
           "fabs", "sign", "tanh", "sinh", "cosh", "sq", "pow", "atan2", "fmin", "fmax", "default_yaml"]


class SX:
    """A column vector of symbolic expressions (handle to a ``casadi::SX`` in the host library)."""

    __slots__ = ("_h",)
    __array_priority__ = 1000   # numpy scalars / arrays defer to the reflected operators below

    def __init__(self, handle):
        self._h = handle

    def __del__(self):
        try:
            if self._h:
                host_lib().ocp_host_sx_free(self._h)
                self._h = None
        except Exception:
            pass

    # ---- creation
    @staticmethod
    def sym(name: str, n: int = 1) -> "SX":
        out = C.c_void_p()
        _hcheck(host_lib().ocp_host_sx_sym(name.encode(), int(n), C.byref(out)))
        return SX(out)

    @staticmethod
    def const(values) -> "SX":
        v = np.ascontiguousarray(np.atleast_1d(np.asarray(values, dtype=np.float64)).ravel())
        out = C.c_void_p()
        _hcheck(host_lib().ocp_host_sx_const(_dp(v), v.size, C.byref(out)))
        return SX(out)

    @staticmethod
    def zeros(n: int = 1) -> "SX":
        return SX.const(np.zeros(n))

    @staticmethod
    def _wrap(x) -> "SX":
        return x if isinstance(x, SX) else SX.const(x)

    # ---- shape, indexing
    def size1(self) -> int:
        return host_lib().ocp_host_sx_size(self._h)

    def __len__(self) -> int:
        return self.size1()

    def __getitem__(self, idx) -> "SX":
        n = self.size1()
        if isinstance(idx, slice):
            start, stop, step = idx.indices(n)
            if step != 1:
                raise IndexError("SX slices must be contiguous")
        else:
            i = int(idx)
            if i < 0:
                i += n
            if not 0 <= i < n:
                raise IndexError("SX index out of range")
            start, stop = i, i + 1
        out = C.c_void_p()
        _hcheck(host_lib().ocp_host_sx_slice(self._h, start, stop, C.byref(out)))
        return SX(out)

    def __iter__(self):
        return (self[i] for i in range(self.size1()))

    # ---- arithmetic (element-wise, a 1-by-1 operand broadcasts -- as in CasADi)
    @staticmethod
    def _binary(op: str, a, b) -> "SX":
        a, b = SX._wrap(a), SX._wrap(b)
        out = C.c_void_p()
        _hcheck(host_lib().ocp_host_sx_binary(op.encode(), a._h, b._h, C.byref(out)))
        return SX(out)

    @staticmethod
    def _unary(op: str, a) -> "SX":
        a = SX._wrap(a)
        out = C.c_void_p()
        _hcheck(host_lib().ocp_host_sx_unary(op.encode(), a._h, C.byref(out)))
        return SX(out)

    def __add__(self, o): return SX._binary("add", self, o)
    def __radd__(self, o): return SX._binary("add", o, self)
    def __sub__(self, o): return SX._binary("sub", self, o)
    def __rsub__(self, o): return SX._binary("sub", o, self)
    def __mul__(self, o): return SX._binary("mul", self, o)
    def __rmul__(self, o): return SX._binary("mul", o, self)
    def __truediv__(self, o): return SX._binary("div", self, o)
    def __rtruediv__(self, o): return SX._binary("div", o, self)
    def __pow__(self, o): return SX._binary("pow", self, o)
    def __neg__(self): return SX._unary("neg", self)


def vertcat(parts: Iterable) -> SX:
    items = [SX._wrap(p) for p in parts]
    arr = (C.c_void_p * len(items))(*[p._h for p in items])
    out = C.c_void_p()
    _hcheck(host_lib().ocp_host_sx_vertcat(arr, len(items), C.byref(out)))
    return SX(out)


def _make_unary(op):
    def f(x) -> SX:
        return SX._unary(op, x)
    f.__name__ = op
    return f


def _make_binary(op):
    def f(a, b) -> SX:
        return SX._binary(op, a, b)
    f.__name__ = op
    return f


sin, cos, tan, asin, acos, atan = (_make_unary(o) for o in ("sin", "cos", "tan", "asin", "acos", "atan"))
exp, log, sqrt, fabs, sign, sq = (_make_unary(o) for o in ("exp", "log", "sqrt", "fabs", "sign", "sq"))
tanh, sinh, cosh = (_make_unary(o) for o in ("tanh", "sinh", "cosh"))
pow, atan2, fmin, fmax = (_make_binary(o) for o in ("pow", "atan2", "fmin", "fmax"))   # noqa: A001


def default_yaml(name: str, horizon: int = 0, alpha: float = 0.1, step_num: int = 10) -> str:
    """YAML text of a built-in benchmark problem (variables, bounds, discretisation, CUDA_SQP settings)."""
    buf = C.create_string_buffer(1 << 16)
    _hcheck(host_lib().ocp_host_default_yaml(name.encode(), horizon, alpha, step_num, buf, len(buf)))
    return buf.value.decode()


class OptimalControlProblem:
    """Subclass and override ``deploy_constraints_and_add_cost`` -- the reference's user model
    (include/optimal_control_problem/OptimalControlProblem.h:65-106), method names as in its pybind module.

    ``yaml_text``: the ``optimal_control_problem:`` node (or a document containing it) with
    ``solve_method: CUDA_SQP``; ``name`` names the generated stage library."""

    def __init__(self, yaml_text: str, name: str = "python_ocp"):
        out = C.c_void_p()
        _hcheck(host_lib().ocp_host_scripted_create(name.encode(), yaml_text.encode(), C.byref(out)))
        self._h = out
        self.name = name
        horizon, dt, nf = C.c_int(), C.c_double(), C.c_int()
        _hcheck(host_lib().ocp_host_scripted_info(self._h, C.byref(horizon), C.byref(dt), C.byref(nf)))
        self.horizon, self.dt, self.frame_size = horizon.value, dt.value, nf.value
        self.reference_: SX | None = None
        self._problem: Problem | None = None
        self._trajectory = None

    def __del__(self):
        try:
            if self._problem is None and self._h:   # after gen_solver() the Problem wrapper owns the handle
                host_lib().ocp_host_problem_destroy(self._h)
            self._h = None
        except Exception:
            pass

    # ---- OCPConfig
    def get_variable(self, k: int, field: str) -> SX:
        out = C.c_void_p()
        _hcheck(host_lib().ocp_host_scripted_variable(self._h, int(k), field.encode(), C.byref(out)))
        return SX(out)

    def get_horizon(self) -> int: return self.horizon
    def get_dt(self) -> float: return self.dt
    def get_frame_size(self) -> int: return self.frame_size

    # ---- registration
    def set_reference(self, reference: SX) -> None:
        _hcheck(host_lib().ocp_host_scripted_set_reference(self._h, reference._h))
        self.reference_ = reference

    def get_reference(self) -> SX | None:
        return self.reference_

    def add_scalar_cost(self, cost) -> None:
        cost = SX._wrap(cost)   # held until the call returns: a temporary's handle would be freed before it is read
        _hcheck(host_lib().ocp_host_scripted_add_scalar_cost(self._h, cost._h))

    def add_vector_cost(self, weights: Sequence[float], cost: SX) -> None:
        w = _f64(weights)
        # the C++ addVectorCost(std::vector<double>) keeps the reference's exit(-5) on a size mismatch
        # (OptimalControlProblem.cpp:591); from Python that would kill the interpreter: check here
        if w.size != cost.size1():
            raise ValueError(f"weight vector has {w.size} entries, cost vector {cost.size1()}")
        _hcheck(host_lib().ocp_host_scripted_add_vector_cost(self._h, _dp(w), w.size, cost._h))

    def add_inequality_constraint(self, name: str, lower, expression: SX, upper) -> None:
        lb, ub = _f64(np.atleast_1d(lower)), _f64(np.atleast_1d(upper))
        if lb.size != ub.size:
            raise ValueError("lower and upper bound sizes differ")
        _hcheck(host_lib().ocp_host_scripted_add_inequality(self._h, name.encode(), _dp(lb), expression._h, _dp(ub), lb.size))

    def add_equation_constraint(self, name: str, left: SX, right: SX | None = None) -> None:
        _hcheck(host_lib().ocp_host_scripted_add_equation(self._h, name.encode(), left._h,
                                                          right._h if right is not None else None))

    def deploy_constraints_and_add_cost(self) -> None:
        raise NotImplementedError("override deploy_constraints_and_add_cost() in a subclass")

    # ---- solver
    def gen_solver(self) -> None:
        """``OptimalControlProblem::genSolver()`` (CUDA_SQP branch): needs no GPU.  Idempotent: a second
        call returns without building a second owner of the host handle."""
        if self._problem is not None:
            return
        _hcheck(host_lib().ocp_host_scripted_gen_solver(self._h))
        self._problem = Problem._adopt(self.name, self._h)

    @property
    def problem(self) -> Problem:
        """The generated problem: dimensions, sparsity patterns, bounds, the device handle, batched solves."""
        if self._problem is None:
            raise RuntimeError("gen_solver() has not been called")
        return self._problem

    def get_constraint_lower_bounds(self) -> np.ndarray: return self.problem.lbg.copy()
    def get_constraint_upper_bounds(self) -> np.ndarray: return self.problem.ubg.copy()

    def compute_optimal_trajectory(self, frame, reference) -> np.ndarray:
        x, _ = self.problem.compute_optimal_trajectory(frame, reference)
        self._trajectory = x
        return x

    def compute_optimal_trajectory_batch(self, frames, references):
        return self.problem.compute_optimal_trajectory_batch(frames, references)

    def get_optimal_trajectory(self) -> np.ndarray | None:
        return self._trajectory

    def get_optimal_input_first_frame(self) -> np.ndarray | None:
        return None if self._trajectory is None else self._trajectory[: self.frame_size].copy()
