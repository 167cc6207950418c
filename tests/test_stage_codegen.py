"""StageCodegen's decisions for the stage-assembly kernel (kernel 1), read from the generated .cu, and the sympy
reference of tests/stage_reference.py checked where an independent witness exists.  No GPU: nvcc cross-compiles."""
import numpy as np
import pytest

import stage_reference as sr

STATIC_SMEM_LIMIT = 48 * 1024   # static __shared__ of one kernel


def _check_budget(h):
    assert h["smem_bytes"] == h["WARPS_PER_BLOCK"] * (32 // h["UNIT_LANES"]) * (h["STAGE_A"] + h["STAGE_H"]) * 8
    assert h["smem_bytes"] <= 40 * 1024 < STATIC_SMEM_LIMIT
    # every staged group fits the image; the others store straight to global memory
    for g in h["groups"]:
        a_len, h_len = g[6], g[8]
        staged = g[12] if len(g) > 12 else 1
        assert staged == (a_len + h_len <= 640)
        if staged:
            assert a_len <= h["STAGE_A"] and h_len <= h["STAGE_H"]
    assert h["direct_groups"] == sum(1 for g in h["groups"] if len(g) > 12 and g[12] == 0)


def test_headline_quadrotor_keeps_its_layout(native):
    """quadrotor H = 20: every group stays staged (the p group's image is 12 + 252 doubles), two 16-lane units per
    warp, and the generated kernel has no direct-store path at all."""
    h = sr.generated_header(native.Problem("quadrotor", horizon=20))
    assert (h["UNIT_LANES"], h["STAGE_A"], h["STAGE_H"], h["NUM_GROUPS"], h["templates"]) == (16, 142, 252, 21, 4)
    assert h["direct_groups"] == 0 and all(len(g) == 12 for g in h["groups"])
    assert "gA" not in h["source"] and "staged" not in h["source"].split("struct GroupInfo")[1].split("};")[0]
    _check_budget(h)


@pytest.mark.parametrize("name,horizon,lanes,a,hh", [
    ("quadrotor", 128, 16, 142, 28),    # past the old limit of H = 115; back to two units per warp
    ("cartpole", 400, 8, 24, 9),        # past the old limit of H = 377
])
def test_long_horizons_build(native, name, horizon, lanes, a, hh):
    """The p group's Hessian range grows with H; it stores straight to global memory, so the kernel's shared memory
    and lane count are those of the stage groups."""
    h = sr.generated_header(sr.build_named(name, horizon))
    assert (h["UNIT_LANES"], h["STAGE_A"], h["STAGE_H"], h["NUM_GROUPS"]) == (lanes, a, hh, horizon + 1)
    assert h["direct_groups"] == 1 and h["groups"][0][12] == 0 and all(g[12] == 1 for g in h["groups"][1:])
    _check_budget(h)


@pytest.mark.parametrize("name", sorted(sr.SPECS))
def test_test_models_build(native, name):
    """Each test model generates, compiles, and takes the path it exists for."""
    pr = sr.build_product(name)
    h = sr.generated_header(pr)
    _check_budget(h)
    spec = sr.SPECS[name]
    assert (pr.np_, pr.nf, pr.horizon) == (spec.np_, spec.nf, spec.horizon)
    a_len = [g[6] for g in h["groups"]]
    if name == "wide_param":
        assert h["groups"][0][8] >= 64 * 31 and h["direct_groups"] == 1 and h["UNIT_LANES"] == 32
    else:
        assert h["direct_groups"] == 0
    if name in ("ops_all", "rate_cost", "param_rows", "no_param", "constants"):
        assert h["UNIT_LANES"] == 8
    if name == "no_param":
        assert h["NUM_GROUPS"] == spec.horizon
    else:
        assert h["NUM_GROUPS"] == spec.horizon + 1
    if name == "param_rows":
        assert h["groups"][0][6] > spec.np_           # the p group owns Jacobian entries beyond its identity block
    if name == "rate_cost":
        assert "lane == 7) cv" in h["source"] and "const int i = 8 + lane" in h["source"]   # two lane-select chunks
        assert any(v % 2 for v in a_len)              # odd value ranges: copy_out's head and tail paths


@pytest.mark.parametrize("name,lanes", [("ops_all", 16), ("rate_cost", 32)])
def test_forced_lane_counts_build(native, name, lanes):
    """OCP_B200_ASSEMBLE_LANES widens the units of a model whose default is 8 lanes."""
    h = sr.generated_header(sr.build_product(name, lanes))
    assert h["UNIT_LANES"] == lanes
    _check_budget(h)


def test_constant_bank_limit_is_refused_before_nvcc(native, monkeypatch):
    """c_groups holds 52 bytes per group in the 64 KB constant bank: a cart-pole of 1300 stages is within the 16-bit
    index limit but needs 1301 groups.  The generator refuses it by name, before nvcc would run."""
    monkeypatch.setenv("OCP_B200_NVCC", "/nonexistent/nvcc")
    with pytest.raises(RuntimeError, match=r"codegen: 1301 column groups .* 64 KB constant bank .* at most 1260 groups"):
        sr.build_named("cartpole", 1300)


@pytest.mark.parametrize("name,horizon", [("quadrotor", 3), ("cartpole", 4)])
def test_reference_matches_independent_witness(name, horizon):
    """The sympy / mpmath reference on indep_models' model code against indep_models.local_system_dense (complex-step
    derivatives, hand-written cost derivatives): the reference is right where an independent witness exists."""
    import indep_models as im
    spec = sr.indep_model_spec(name, horizon)
    ref = sr.Reference(spec)
    rng = np.random.default_rng(7)
    nf = spec.nf
    for _ in range(2):
        p = rng.uniform(-0.5, 0.5, spec.np_)
        x = rng.uniform(-0.3, 0.3, nf * horizon)
        frame = rng.uniform(-0.3, 0.3, nf)
        e = ref.evaluate(p, x)
        Hm, grad, J, l, u = im.local_system_dense(name, horizon, p, x, frame)
        assert np.abs(e["H"] - Hm).max() <= 1e-12 * max(1.0, np.abs(Hm).max())
        assert np.abs(e["grad"] - grad).max() <= 1e-12 * max(1.0, np.abs(grad).max())
        assert np.abs(e["J"] - J).max() <= 1e-12 * max(1.0, np.abs(J).max())
        assert np.isclose(e["f"], im.objective_value(name, horizon, p, x), rtol=1e-13)
        lbx, ubx = spec.bounds()
        lbx[:nf] = frame
        ubx[:nf] = frame
        c = np.concatenate([p, x, e["g"]])
        for mine, theirs in ((np.concatenate([p, lbx, ref.lbg]) - c, l), (np.concatenate([p, ubx, ref.ubg]) - c, u)):
            fin = np.isfinite(theirs)
            assert np.array_equal(np.isfinite(mine), fin)
            assert np.abs(mine[fin] - theirs[fin]).max() <= 1e-12 * max(1.0, np.abs(theirs[fin]).max())
