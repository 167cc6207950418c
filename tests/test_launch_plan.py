"""The whole launch plan of a handle, pinned: which kernel runs each batch size, with how many threads, how much
dynamic shared memory, how many CTAs per SM and how large a per-CTA slab (launch_plan()), and the dimensions and
kernel bits of device_dims().

The expected values (golden/launch_plans.json) hold for a B200 with 148 SMs and 227 KB of opt-in shared memory per
block; on another device the plans differ and the test skips.  Cases: every shape of test_gpu_block_shapes.SHAPES with
no override, under each placement it lists (with that test's environment), with OCP_B200_PLAN=none and with the
DIAGONAL preconditioner; the three models at their benchmark horizons and the quadrotor at H = 128; and a handle
re-planned by update_settings.
"""
import json
from pathlib import Path

import pytest

from test_gpu_block_shapes import SHAPES, _qp, _shape_id

pytestmark = pytest.mark.gpu

GOLDEN = Path(__file__).resolve().parent / "golden" / "launch_plans.json"
ENV_KEYS = ("OCP_B200_PLAN", "OCP_B200_FORCE_STREAM")


def _shape_cases():
    """(case id, shape, environment, pcg_precond or None)"""
    for shape in SHAPES:
        sid = _shape_id(shape)
        yield f"{sid}-default", shape, {}, None
        for place in shape[6]:
            if place == "pcg":
                continue   # no override: the default case above
            env = {"OCP_B200_PLAN": place}
            if place == "mixed":
                env["OCP_B200_FORCE_STREAM"] = "1"
            yield f"{sid}-{place}", shape, env, None
        yield f"{sid}-none", shape, {"OCP_B200_PLAN": "none"}, None
        yield f"{sid}-diagonal", shape, {}, "diagonal"


SHAPE_CASES = {c[0]: c[1:] for c in _shape_cases()}
MODEL_CASES = {f"{name}-H{h}": (name, h) for name, h in (("quadrotor", 20), ("cartpole", 200), ("centroidal", 50),
                                                          ("quadrotor", 128))}


@pytest.fixture(scope="module")
def golden():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    p = torch.cuda.get_device_properties(0)
    if p.multi_processor_count != 148 or p.shared_memory_per_block_optin != 227 * 1024:
        pytest.skip(f"plans are pinned for 148 SMs and 227 KB of opt-in shared memory, not {p.name}")
    return json.loads(GOLDEN.read_text())


def _set_env(monkeypatch, env):
    for k in ENV_KEYS:
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)


def record(sol):
    return dict(plan=sol.launch_plan(), dims=sol.device_dims())


@pytest.mark.parametrize("case", list(SHAPE_CASES))
def test_shape_plan(native, monkeypatch, golden, case):
    shape, env, precond = SHAPE_CASES[case]
    _set_env(monkeypatch, env)
    settings = None
    if precond == "diagonal":
        settings = native.default_settings()
        settings.pcg_precond = native.PRECOND_DIAGONAL
    d = _qp(shape, B=1)
    np_, nf, horizon = shape[:3]
    sol = native.Solver.create(d["n"], d["m"], d["hp"], d["hi"], d["ap"], d["ar"], settings=settings, np_=np_, nf=nf,
                               horizon=horizon)
    assert record(sol) == golden[case]


@pytest.mark.parametrize("case", list(MODEL_CASES))
def test_model_plan(native, monkeypatch, golden, case):
    _set_env(monkeypatch, {})
    name, horizon = MODEL_CASES[case]
    prob = native.Problem(name, horizon=horizon)   # owns the handle: kept alive while the handle is read
    assert record(prob.solver) == golden[case]


def test_replanning(native, monkeypatch, golden):
    """update_settings re-plans when the preconditioner changes: the PCG stage reports what a fresh PCG handle of the
    same pattern reports (no placement of the direct plan left behind in the kernel bits of device_dims), and switching
    back gives the first plan again."""
    _set_env(monkeypatch, {})
    prob = native.Problem("quadrotor", horizon=20)
    sol = prob.solver
    first = record(sol)
    assert first == golden["quadrotor-H20"]
    s = sol.get_settings()
    s.pcg_precond = native.PRECOND_DIAGONAL
    sol.update_settings(s)
    fresh = native.Solver.create(prob.n, prob.m, prob.h_colptr, prob.h_rowidx, prob.a_colptr, prob.a_rowidx, settings=s,
                                 np_=prob.np_, nf=prob.nf, horizon=prob.horizon)
    assert record(sol) == record(fresh)
    s.pcg_precond = native.PRECOND_BLOCK_TRIDIAG
    sol.update_settings(s)
    assert record(sol) == first
