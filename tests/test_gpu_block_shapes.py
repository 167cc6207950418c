"""Every block-structure path of the direct and compact ADMM kernels, on synthetic stage-structured QPs.

The three model problems reach only a few of the code paths the kernels choose from the shape of the reduced KKT
matrix (border width np, block size bs = G * nf, block count nb, pitch, placement).  Here `stage_qp` builds
multiple-shooting-shaped QPs of any (np, nf, horizon), QP-only handles solve them under a forced launch plan, and the
CPU oracle (tests/_oracle.py, itself checked against scipy in test_oracle_qp.py) solves the same arrays.

Checks, for every shape and placement of SHAPES:
  * the launch plan: tri_ok / tri_np / tri_bs / tri_nb and the placement of both plans.  A forced placement that
    does not fit fails the test instead of running some other kernel unnoticed;
  * a few-iteration probe: 1 and 3 ADMM iterations from a cold start without rho adaptation, with and without Ruiz
    scaling.  Both sides have then done the same one or three solves of the same linear system, so x and y agree
    to rounding (PROBE_TOL).  A wrong factor block or border term is visible here even where ADMM would damp it;
  * full solves at eps 1e-3 and 1e-7 (the latter adapts rho, which refactorises): status, iteration count and rho
    updates identical, x, y and residuals within 1e-6.
test_persistent_instance_loop runs more instances than the grid holds CTAs (the persistent loop of next_instance).
"""
import numpy as np
import pytest

import _oracle
from test_gpu_parity import rel_err

REL_SOLUTION = 1e-6
# FP64 on both sides, same operations up to the order of the sums and the factorisation method: rounding amplified by
# the condition number of the reduced system (< 1e6 by construction) stays far below this.
PROBE_TOL = 1e-9

RHO, SIGMA, RHO_MIN, RHO_EQ = 0.1, 1e-6, 1e-6, 1e3   # OSQP defaults (rho, sigma), rho_i of free / equality rows
PLACE = {"mixed": 0, "smem": 1, "multi": 2, "big": 3, "compact": 4, "pcg": -1}


def _csc(rows, cols, ncol):
    """CSC pattern of the coordinate list and the permutation that puts values given in list order into it."""
    rows, cols = np.asarray(rows, np.int64), np.asarray(cols, np.int64)
    order = np.lexsort((rows, cols))
    colptr = np.zeros(ncol + 1, np.int64)
    np.add.at(colptr, cols + 1, 1)
    return np.cumsum(colptr).astype(np.int32), rows[order].astype(np.int32), order


def _mask(rng, r, c, density):
    return rng.random((r, c)) < density


def _pick(rng, r, c, count, upper=False):
    """r x c mask with `count` entries (strictly above the diagonal when `upper`)."""
    m = np.zeros((r, c), bool)
    cand = [(i, j) for i in range(r) for j in range(c) if not upper or j > i]
    if cand:
        for k in rng.choice(len(cand), size=min(count, len(cand)), replace=False):
            m[cand[k]] = True
    return m


def stage_qp(np_, nf, horizon, seed, variant=None, B=2):
    """A multiple-shooting-shaped QP: columns [border (np_) | stage 0 (nf) | ... | stage horizon-1].

    P: SPD block per stage, coupling of neighbouring stages, border-border and border-stage entries; full symmetric
    pattern (both triangles, as _random_qp in test_gpu_parity.py), strictly diagonally dominant, so P >= I.
    A: an identity row per variable (border pinned, stage variables free, one-sided, boxed or fixed), then per stage
    the dynamics rows to the next stage (optionally with a border entry) and inequality rows local to the stage.
    Every stage has the same pattern; the values differ between stages and instances.  No row and no entry of P spans
    more than two neighbouring stages, so the block-tridiagonal structure holds for any grouping of stages.

    variant: None; "long_rows": one more row over the whole border and two neighbouring stages (more than 64
    entries); "irregular": extra rows on stages 0, 1, 3 and the last (at horizon 6: 5 regions in the stage-periodic
    index of the CSR of A); "too_irregular": extra rows on stages 0, 3, 5, 8 and the last (at horizon 12: 8 regions,
    more than the 6 the compact kernel takes).

    Returns ((h_colptr, h_rowidx), (a_colptr, a_rowidx), hv [B, nnz_h], q [B, n], av [B, nnz_a], l [B, m], u [B, m]).
    """
    rng = np.random.default_rng([seed, np_, nf, horizon])
    n = np_ + nf * horizon
    col = lambda k, c: np_ + k * nf + c   # noqa: E731
    # ---- pattern of P (upper triangle, diagonal included)
    # few off-diagonal entries: the symmetrised P must fit the compact kernel's overlay of z | y (nnz <= 2 m)
    pbb = _pick(rng, np_, np_, np_ // 4, upper=True) | np.eye(np_, dtype=bool)
    pss = _pick(rng, nf, nf, nf // 2, upper=True) | np.eye(nf, dtype=bool)
    pcc = _pick(rng, nf, nf, max(1, nf // 4))
    pbs = _pick(rng, np_, nf, max(1, nf // 4))
    pi, pj = [], []
    for r, c in zip(*np.nonzero(pbb)):
        pi.append(r); pj.append(c)
    for k in range(horizon):
        for a, b in zip(*np.nonzero(pss)):
            pi.append(col(k, a)); pj.append(col(k, b))
        for r, c in zip(*np.nonzero(pbs)):
            pi.append(r); pj.append(col(k, c))
        if k + 1 < horizon:
            for a, b in zip(*np.nonzero(pcc)):
                pi.append(col(k, a)); pj.append(col(k + 1, b))
    pi, pj = np.array(pi), np.array(pj)
    off = pi != pj
    hrows = np.concatenate([pi, pj[off]]); hcols = np.concatenate([pj, pi[off]])
    hp, hi, horder = _csc(hrows, hcols, n)

    # ---- pattern of A: list of rows, each (columns, kind); kind picks the value distribution and the bound type
    nx, ni = max(1, nf // 2), max(1, nf // 4)
    dyn = _mask(rng, nx, nf, 0.3)
    dyn[np.arange(nx), np.arange(nx)] = True
    ineq = _mask(rng, ni, nf, 0.4)
    ineq[np.arange(ni), np.arange(ni) % nf] = True
    # identity rows of the stage variables: 0 free, 1 lower only, 2 upper only, 3 boxed, 4 fixed
    stage_kind = rng.choice(5, size=nf, p=[0.25, 0.15, 0.15, 0.35, 0.10])
    rows = [([j], "pin" if j < np_ else ("free", "lower", "upper", "box", "fix")[stage_kind[(j - np_) % nf]])
            for j in range(n)]

    def extra_rows(k, count):
        return [(sorted({col(k, (k + 3 * e) % nf), col(k, (2 * k + e + 1) % nf)}), "ineq") for e in range(count)]

    extra = {}   # stage -> number of extra rows
    if variant == "irregular":
        extra = {0: 1, 1: 2, 3: 3, horizon - 1: 1}
    elif variant == "too_irregular":
        extra = {0: 2, 3: 1, 5: 2, 8: 3, horizon - 1: 1}
    for k in range(horizon):
        if k + 1 < horizon:
            for i in range(nx):
                cols = [col(k, c) for c in np.flatnonzero(dyn[i])] + [col(k + 1, i)]
                if np_ > 0 and i < 2:
                    cols = [i % np_] + cols
                rows.append((cols, "dyn"))
        for i in range(ni):
            rows.append(([col(k, c) for c in np.flatnonzero(ineq[i])], "ineq"))
        rows += extra_rows(k, extra.get(k, 0))
    if variant == "long_rows":
        k = horizon // 2 - 1
        rows.append((list(range(np_)) + list(range(col(k, 0), col(k + 2, 0))), "ineq"))
    m = len(rows)
    ai = np.concatenate([np.full(len(c), i) for i, (c, _) in enumerate(rows)])
    aj = np.concatenate([np.asarray(c) for c, _ in rows])
    ap, ar, aorder = _csc(ai, aj, n)
    kinds = [kd for _, kd in rows]

    hv, qs, av, ls, us = [], [], [], [], []
    for b in range(B):
        r = np.random.default_rng([seed, np_, nf, horizon, b + 1])
        # P: off-diagonal entries, then a diagonal that dominates every row by 1..2
        vals = 0.3 * r.standard_normal(len(pi))
        vals[~off] = 0.0
        full = np.concatenate([vals, vals[off]])
        rowsum = np.zeros(n)
        np.add.at(rowsum, hrows, np.abs(full))
        vals[~off] = rowsum[pi[~off]] + 1.0 + r.random(int((~off).sum()))
        hv.append(np.concatenate([vals, vals[off]])[horder])
        # A: identity rows 1, dynamics rows x_{k+1}[i] = sum_j a_ij x_k[j] (+ border), inequality rows N(0, 1)
        a = []
        for cols, kd in rows:
            if kd == "dyn":
                v = 0.4 * r.standard_normal(len(cols)); v[-1] = -1.0
            elif kd == "ineq":
                v = r.standard_normal(len(cols))
            else:
                v = np.ones(1)
            a.append(v)
        a = np.concatenate(a)
        av.append(a[aorder])
        # bounds around a feasible point xf
        xf = r.standard_normal(n)
        Ax = np.zeros(m)
        np.add.at(Ax, ai, a * xf[aj])
        lo, up = Ax - 0.1 - r.random(m), Ax + 0.1 + r.random(m)
        for i, kd in enumerate(kinds):
            if kd in ("pin", "fix", "dyn"):
                lo[i] = up[i] = Ax[i]
            elif kd == "free":
                lo[i], up[i] = -np.inf, np.inf
            elif kd == "lower":
                up[i] = np.inf
            elif kd == "upper":
                lo[i] = -np.inf
        ls.append(lo); us.append(up)
        qs.append(r.standard_normal(n))
    return (hp, hi), (ap, ar), np.array(hv), np.array(qs), np.array(av), np.array(ls), np.array(us)


def reduced_matrix(n, hp, hi, hv, ap, ar, av, l, u, rho=RHO, sigma=SIGMA):
    """P + sigma I + A' diag(rho_i) A with OSQP's rho_i: RHO_MIN for free rows, 1e3 rho for equality rows."""
    import scipy.sparse as sp
    P = sp.csc_matrix((hv, hi, hp), shape=(n, n)).toarray()
    A = sp.csc_matrix((av, ar, ap), shape=(len(l), n)).toarray()
    rho_i = np.where(np.isinf(l) & np.isinf(u), RHO_MIN, np.where(u - l < 1e-4, RHO_EQ * rho, rho))
    return P + sigma * np.eye(n) + A.T @ (rho_i[:, None] * A)


# (np, nf, horizon, variant, bs, nb, placements): the block size bs = G * nf (G the largest divisor of the horizon with
# G * nf <= 20) and the block count nb the host must report, and the placements to force.  "mixed" also sets
# OCP_B200_FORCE_STREAM (factor in the global slab, streamed through the ring); "pcg" forces nothing: the shape must
# fall back to the PCG kernel.  Compact chains (sweep_chain, mid = nb / 2): mid, nb - 2 - mid, mid, nb - 1 - mid
# stages; the first kTmemBlocks = 8 come from Tensor Memory, then one prefetched slab stage, then plain slab loads.
SHAPES = [
    (0, 16, 6, None, 16, 6, ("smem", "multi", "compact")),       # no border, more than one block: twisted<16>
    (12, 16, 1, None, 16, 1, ("smem", "compact")),               # nb = 1: twisted split mid = 0, all chains empty
    (12, 16, 3, None, 16, 3, ("smem", "multi", "compact")),      # nb = 3: chains of 1, 0, 1, 1 stages
    (12, 8, 10, None, 16, 5, ("smem", "compact")),               # G = 2 stages per block; template period half a block
    (40, 16, 8, None, 16, 8, ("smem", "compact")),               # np > 32 on twisted<16>; compact border np != 12
    (64, 16, 4, None, 16, 4, ("smem", "compact")),               # the widest border the direct kernels take
    (12, 16, 16, None, 16, 16, ("compact",)),                    # longest chain 8: Tensor Memory only; border by warp
    (12, 16, 18, None, 16, 18, ("compact",)),                    # chain of 9 (one prefetched slab stage) next to 8
    (12, 16, 19, None, 16, 19, ("compact",)),                    # chains 9, 8, 9, 9; N = 304, border rows by warp
    (12, 16, 24, None, 16, 24, ("compact",)),                    # chains of 12: slab tail; N = 384, half-warp rows
    (4, 5, 12, None, 20, 3, ("smem", "big", "compact")),         # G = 4, bs = 20, nb = 3: BIG falls back (nb < 4)
    (33, 20, 8, None, 20, 8, ("big", "compact")),                # np > 32 on twisted<20> and stream_twisted<20>
    (8, 24, 5, None, 24, 5, ("mixed", "smem")),                  # tri_solve_stream<24>; generic tri_solve on smem
    (40, 36, 4, None, 36, 4, ("mixed",)),                        # parallel diagonal phase with np > 32
    (5, 7, 7, None, 7, 7, ("smem", "multi", "big", "mixed")),    # odd bs, pitch bs + 1: generic factor and sweeps
    (3, 1, 23, None, 1, 23, ("smem", "multi")),                  # bs = 1, 23 blocks
    (6, 64, 3, None, 64, 3, ("mixed",)),                         # bs = 64, the largest block: only the mixed placement fits
    (40, 16, 8, "long_rows", 16, 8, ("smem", "mixed", "compact")),   # rows_long; the compact kernel refuses
    (12, 16, 6, "irregular", 16, 6, ("compact",)),               # 5 regions in the periodic index
    (12, 16, 12, "too_irregular", 16, 12, ("compact",)),         # 8 regions: the compact kernel refuses
    (65, 8, 4, None, 16, 2, ("pcg",)),                           # border wider than 64: PCG
    (4, 65, 2, None, 65, 2, ("pcg",)),                           # block wider than 64: PCG
]
COMPACT_REFUSED = ("long_rows", "too_irregular")
SEED = 7


def _shape_id(shape):
    np_, nf, horizon, variant = shape[:4]
    return f"np{np_}-nf{nf}-H{horizon}" + (f"-{variant}" if variant else "")


CASES = [pytest.param(shape, place, id=f"{_shape_id(shape)}-{place}") for shape in SHAPES for place in shape[6]]


def _qp(shape, B=2):
    np_, nf, horizon, variant = shape[:4]
    (hp, hi), (ap, ar), hv, q, av, l, u = stage_qp(np_, nf, horizon, SEED, variant, B=B)
    return dict(n=np_ + nf * horizon, m=l.shape[1], hp=hp, hi=hi, ap=ap, ar=ar, hv=hv, q=q, av=av, l=l, u=u)


def _check_conditioning(d):
    for b in range(d["q"].shape[0]):
        K = reduced_matrix(d["n"], d["hp"], d["hi"], d["hv"][b], d["ap"], d["ar"], d["av"][b], d["l"][b], d["u"][b])
        assert np.linalg.cond(K) < 1e6


def _oracle_solve(d, b, settings):
    return _oracle.qp_solve(d["n"], d["m"], d["hp"], d["hi"], d["hv"][b], d["q"][b], d["ap"], d["ar"], d["av"][b],
                            d["l"][b], d["u"][b], settings=settings)


def _solver(native, monkeypatch, shape, place, d):
    """QP-only handle under the forced plan, with the plan fields this shape and placement claim checked."""
    np_, nf, horizon, variant, bs, nb = shape[:6]
    monkeypatch.delenv("OCP_B200_PLAN", raising=False)
    monkeypatch.delenv("OCP_B200_FORCE_STREAM", raising=False)
    if place != "pcg":
        monkeypatch.setenv("OCP_B200_PLAN", place)
    if place == "mixed":
        monkeypatch.setenv("OCP_B200_FORCE_STREAM", "1")
    sol = native.Solver.create(d["n"], d["m"], d["hp"], d["hi"], d["ap"], d["ar"], np_=np_, nf=nf, horizon=horizon)
    plan = sol.launch_plan()
    assert (plan["tri_np"], plan["tri_bs"], plan["tri_nb"]) == (np_, bs, nb)
    assert plan["tri_ok"] == (place != "pcg")
    if place == "compact" and variant in COMPACT_REFUSED:
        assert plan["wide"]["place"] != 4 and plan["deep"]["place"] != 4
    else:
        assert plan["wide"]["place"] == plan["deep"]["place"] == PLACE[place], plan
    return sol


def _settings(native, place):
    s = native.default_settings()
    if place == "pcg":
        # the PCG kernel solves each system to a relative residual; at the default 1e-10 the inexact solves change the
        # ADMM iterates by more than rounding (other iteration counts at eps 1e-7).  Ask for one that leaves only rounding.
        s.pcg_tol, s.pcg_max_iter = 1e-14, 2000
    return s


@pytest.mark.gpu
@pytest.mark.parametrize("shape,place", CASES)
def test_block_shape_matches_oracle(native, monkeypatch, shape, place):
    d = _qp(shape)
    _check_conditioning(d)
    sol = _solver(native, monkeypatch, shape, place, d)
    B = d["q"].shape[0]
    args = (d["hv"], d["q"], d["av"], d["l"], d["u"])
    # (a) one and three iterations from a cold start, rho fixed, with and without Ruiz scaling
    worst = 0.0
    for iters in (1, 3):
        for scaling in (0, 10):
            s = _settings(native, place)
            s.admm_max_iter, s.adaptive_rho, s.scaling_iters = iters, 0, scaling
            sol.update_settings(s)
            x, y, info = sol.qp_solve_batch(*args)
            sv = _oracle.settings_from_b200(s)
            for b in range(B):
                ox, oy, oinfo, _ = _oracle_solve(d, b, sv)
                assert info[b, native.INFO["status"]] == oinfo[0]
                assert info[b, native.INFO["iters"]] == oinfo[1] == iters
                err = max(rel_err(x[b], ox), rel_err(y[b], oy))
                assert err <= PROBE_TOL, (iters, scaling, b, err)
                worst = max(worst, err)
    print(f"probe: largest relative error {worst:.2e}")
    # (b) full solves; the tight tolerance adapts rho (refactorisations)
    for eps in (1e-3, 1e-7):
        s = _settings(native, place)
        s.eps_abs = s.eps_rel = eps
        sol.update_settings(s)
        x, y, info = sol.qp_solve_batch(*args)
        sv = _oracle.settings_from_b200(s)
        for b in range(B):
            ox, oy, oinfo, _ = _oracle_solve(d, b, sv)
            assert info[b, native.INFO["status"]] == oinfo[0] == native.QP_SOLVED
            assert info[b, native.INFO["iters"]] == oinfo[1]
            assert info[b, native.INFO["rho_updates"]] == oinfo[6]
            assert rel_err(x[b], ox) < REL_SOLUTION
            assert rel_err(y[b], oy) < REL_SOLUTION
            assert abs(info[b, native.INFO["prim_res"]] - oinfo[3]) <= 1e-6 * max(1.0, abs(oinfo[3])) + 1e-9
            assert abs(info[b, native.INFO["dual_res"]] - oinfo[4]) <= 1e-6 * max(1.0, abs(oinfo[4])) + 1e-9


def _shape(np_, nf, horizon):
    return next(sh for sh in SHAPES if sh[:4] == (np_, nf, horizon, None))


@pytest.mark.gpu
@pytest.mark.parametrize("shape,place", [
    pytest.param(_shape(0, 16, 6), "compact", id="np0-nf16-H6-compact"),   # no border, bs = 16
    pytest.param(_shape(4, 5, 12), "big", id="np4-nf5-H12-big"),           # bs = 20
    pytest.param(_shape(5, 7, 7), "multi", id="np5-nf7-H7-multi"),         # odd bs
])
def test_persistent_instance_loop(native, monkeypatch, shape, place):
    """More instances than the grid has CTAs: the CTAs of the first wave take the rest from the instance counter
    (next_instance).  Every instance gets the bits it gets when solved alone, and a sample matches the oracle."""
    d1 = _qp(shape, B=1)
    sol = _solver(native, monkeypatch, shape, place, d1)
    plan = sol.launch_plan()
    wave = plan["wide"]["ctas_per_sm"] * plan["num_sms"]
    B = wave + 3
    d = _qp(shape, B=B)
    x, y, info = sol.qp_solve_batch(d["hv"], d["q"], d["av"], d["l"], d["u"])
    for b in range(B):
        xb, yb, ib = sol.qp_solve_batch(*(d[k][b:b + 1] for k in ("hv", "q", "av", "l", "u")))
        assert np.array_equal(xb[0], x[b]) and np.array_equal(yb[0], y[b]) and np.array_equal(ib[0], info[b]), b
    sv = _oracle.settings_from_b200(sol.get_settings())
    for b in (0, wave - 1, wave, B - 1):
        ox, oy, oinfo, _ = _oracle_solve(d, b, sv)
        assert info[b, native.INFO["status"]] == oinfo[0] == native.QP_SOLVED
        assert info[b, native.INFO["iters"]] == oinfo[1]
        assert rel_err(x[b], ox) < REL_SOLUTION and rel_err(y[b], oy) < REL_SOLUTION


@pytest.mark.parametrize("shape", [pytest.param(sh, id=_shape_id(sh)) for sh in SHAPES])
def test_stage_qp_generator(shape):
    """The generator itself, without a GPU: well-conditioned reduced systems, QPs the oracle solves, and the block
    structure the shape matrix relies on (no row or P entry across more than two neighbouring stages; rows of more
    than 64 entries exactly in the long_rows variant)."""
    np_, nf, horizon, variant = shape[:4]
    d = _qp(shape)
    _check_conditioning(d)
    sv = _oracle.settings_vector()
    for b in range(d["q"].shape[0]):
        assert _oracle_solve(d, b, sv)[2][0] == 1   # QP_SOLVED
    stage = lambda j: np.where(j < np_, -1, (j - np_) // nf)   # noqa: E731
    hcol = np.repeat(np.arange(d["n"]), np.diff(d["hp"]))
    si, sj = stage(d["hi"]), stage(hcol)
    assert (np.abs(si - sj)[(si >= 0) & (sj >= 0)] <= 1).all()
    acol = np.repeat(np.arange(d["n"]), np.diff(d["ap"]))
    sa = stage(acol)
    for i in range(d["m"]):
        st = sa[(d["ar"] == i) & (sa >= 0)]
        assert st.size == 0 or st.max() - st.min() <= 1
    row_len = np.bincount(d["ar"], minlength=d["m"])
    assert (row_len.max() > 64) == (variant == "long_rows")
    # the compact kernel parks the symmetrised P on its z | y vectors (make_layout): nnz_p <= 2 m, both rounded up to
    # even counts, or it refuses the problem
    ev = lambda v: (v + 1) & ~1   # noqa: E731
    assert ev(d["hi"].size) <= 2 * ev(d["m"])
