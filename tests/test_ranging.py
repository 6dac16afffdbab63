"""Sensitivity ranging (yalps_b200/sensitivity.py) without a GPU: ranges_from_tableau against a literal per-id
statement of its definition, and the ranges of the oracle's final tableaus against re-solves of shifted models."""
import math

import numpy as np
import pytest

from test_sensitivity import LP_CASES, _non_degenerate, oracle_final, random_lp
from yalps_b200 import solver as S
from yalps_b200.sensitivity import model_ranges, ranges_from_tableau, reduced_from_tableau, row_pairs
from yalps_b200.tableau import constraint_rows, entries

INF = math.inf


# ------------------------------------------------------------------------------------------- the definition
def per_id_ranges(m, W, H, pos, prec, pairs=None, optimal=True):
    """One id at a time, one cell at a time, exactly as the definition reads."""
    M = np.asarray(m, np.float64).reshape(H, W)
    lo, hi = [-INF] * (W + H), [INF] * (W + H)

    def direction(u):
        p = int(pos[u])
        if 1 <= p < W:
            return [float(M[r, p]) for r in range(H)]
        return [1.0 if r == p - W else 0.0 for r in range(H)]

    for v in range(W + H):
        if v in (0, W) or not optimal:
            lo[v] = hi[v] = math.nan
            continue
        p = int(pos[v])
        if v < W:
            if 1 <= p < W:
                hi[v] = -min(float(M[0, p]), 0.0)
            elif 1 <= p - W < H:
                for c in range(1, W):
                    a = float(M[p - W, c])
                    if abs(a) > prec:
                        q = min(float(M[0, c]), 0.0) / a
                        if a > 0:
                            lo[v] = max(lo[v], q)
                        else:
                            hi[v] = min(hi[v], q)
        else:
            k = v - W
            d = direction(v)
            if pairs is not None and pairs[k] >= 0:
                e = direction(W + int(pairs[k]))
                d = [x - y for x, y in zip(d, e)]
            for r in range(1, H):
                if abs(d[r]) > prec:
                    q = -max(float(M[r, 0]), 0.0) / d[r]
                    if d[r] > 0:
                        lo[v] = max(lo[v], q)
                    else:
                        hi[v] = min(hi[v], q)
        lo[v], hi[v] = lo[v] + 0.0, hi[v] + 0.0
    return np.array(lo), np.array(hi)


def same_bits(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return a.shape == b.shape and np.array_equal(a.view(np.uint64), b.view(np.uint64))


def synthetic(rng, H, W, prec=1e-8, with_pairs=True):
    """A random 'final' tableau: +-0, cells at exactly +-precision, a random basis permutation and random pairs."""
    M = rng.normal(size=(H, W)) * (rng.random((H, W)) < 0.7)
    special = rng.integers(0, H * W, 6 + H * W // 10)
    vals = np.array([0.0, -0.0, prec, -prec, 2 * prec, -2 * prec])
    M.reshape(-1)[special] = vals[rng.integers(0, vals.size, special.size)]
    M[0, 0] = -abs(M[0, 0])
    ids = np.array([v for v in range(W + H) if v not in (0, W)])
    slots = np.array([s for s in range(W + H) if s not in (0, W)])
    pos = np.zeros(W + H, np.int32)
    pos[W] = W
    pos[ids] = rng.permutation(slots)
    pairs = None
    if with_pairs and H > 2:
        pairs = np.full(H, -1, np.int32)
        rows = rng.permutation(np.arange(1, H))
        for i in range(0, len(rows) - 1, 2):
            if rng.random() < 0.6:
                pairs[rows[i]], pairs[rows[i + 1]] = rows[i + 1], rows[i]
    return M.reshape(-1), pos, pairs


@pytest.mark.parametrize("seed", range(40))
def test_reference_equals_definition_bit_for_bit(seed):
    rng = np.random.default_rng(seed)
    H, W = int(rng.integers(2, 12)), int(rng.integers(2, 14))
    prec = [1e-8, 0.5, 0.0][seed % 3]
    m, pos, pairs = synthetic(rng, H, W, prec if prec else 1e-8)
    for pr in (None, pairs):
        got = ranges_from_tableau(m, W, H, pos, prec, pr)
        exp = per_id_ranges(m, W, H, pos, prec, pr)
        assert same_bits(got[0], exp[0]) and same_bits(got[1], exp[1])


def test_reference_rules():
    rng = np.random.default_rng(123)
    for _ in range(30):
        H, W = int(rng.integers(2, 30)), int(rng.integers(2, 30))
        m, pos, pairs = synthetic(rng, H, W)
        lo, hi = ranges_from_tableau(m, W, H, pos, 1e-8, pairs)
        keep = np.ones(W + H, bool)
        keep[[0, W]] = False
        assert np.isnan(lo[[0, W]]).all() and np.isnan(hi[[0, W]]).all()
        assert not np.isnan(lo[keep]).any() and not np.isnan(hi[keep]).any()
        assert (lo[keep] <= 0).all() and (hi[keep] >= 0).all()
        assert not np.signbit(lo[keep][lo[keep] == 0]).any() and not np.signbit(hi[keep][hi[keep] == 0]).any()
        lo, hi = ranges_from_tableau(m, W, H, pos, 1e-8, pairs, optimal=False)
        assert np.isnan(lo).all() and np.isnan(hi).all()


def test_row_pairs():
    rows = [("a", 1, -1), ("b", 2, 3), ("c", -1, 4), ("d", -1, -1), ("e", 5, 6)]
    assert row_pairs(rows, 7).tolist() == [-1, -1, 3, 2, -1, 6, 5]


# ------------------------------------------------------------------------------------ against re-solves
def _oracle_ranges(model, options=None):
    opt = {**S._DEFAULTS, **(options or {})}
    tm, st, val, m, pos, var = oracle_final(model, opt)
    t = tm.tableau
    rows = constraint_rows(list(entries(model["constraints"])))
    lo, hi = ranges_from_tableau(m, t.width, t.height, pos, opt["precision"], row_pairs(rows, t.height), st == 0)
    return tm, st, m, pos, rows, lo, hi


def _raw(model):
    tm, st, _, m, pos, _ = oracle_final(model)
    return st, -tm.sign * m[0], tm, m, pos


def _set_cost(model, name, delta):
    ob = model.get("objective")
    vs = []
    for k, cs in entries(model["variables"]):
        if k == name:
            cs = list(entries(cs))
            if any(ck == ob for ck, _ in cs):
                cs = [(ck, cv + delta) if ck == ob else (ck, cv) for ck, cv in cs]
            else:
                cs.append((ob, delta))
        vs.append((k, cs))
    return {**model, "variables": vs}


def _shift_bounds(model, key, t):
    cons = [(k, ({b: v + t for b, v in dict(entries(con)).items()} if k == key else con))
            for k, con in entries(model["constraints"])]
    return {**model, "constraints": cons}


def _x(tm, m, pos):
    W, H = tm.tableau.width, tm.tableau.height
    M = m.reshape(H, W)
    return np.array([M[pos[j] - W, 0] if pos[j] >= W else 0.0 for j in range(1, W)])


def _has_objective(model, tm):
    ob = model.get("objective")
    return ob is not None and any(ck == ob for _, cs in entries(model["variables"]) for ck, _ in entries(cs))


def _check_inside(model, strict):
    """Re-solves at the midpoint toward each finite end (+-1 toward an infinite one) stay on the line of the shadow
    price / the variable's value; with `strict`, 5 % past each finite end leaves it (or the LP turns infeasible)."""
    tm, st, m, pos, rows, lo, hi = _oracle_ranges(model)
    assert st == 0
    W, H = tm.tableau.width, tm.tableau.height
    base = -tm.sign * m[0]
    red = reduced_from_tableau(m, W, H, pos)
    cost, rhs = model_ranges(tm.variables, rows, lo, hi, W, tm.sign)
    checks = 0
    for (key, up, lw), (_, a, b) in zip(rows, rhs):
        y = (-tm.sign * red[W + up] if up >= 0 else 0.0) - (-tm.sign * red[W + lw] if lw >= 0 else 0.0)
        for t in (a * 0.5 if a > -INF else -1.0, b * 0.5 if b < INF else 1.0):
            st2, r2, *_ = _raw(_shift_bounds(model, key, t))
            lin = base + y * t
            assert st2 == 0 and abs(r2 - lin) <= 1e-6 * (1 + abs(lin)), (key, t, (a, b), st2, r2, lin)
            checks += 1
        if strict:
            for t in (a - 0.05 * (1 + abs(a)) if a > -INF else None, b + 0.05 * (1 + abs(b)) if b < INF else None):
                if t is None:
                    continue
                st2, r2, *_ = _raw(_shift_bounds(model, key, t))
                lin = base + y * t
                assert st2 != 0 or abs(r2 - lin) > 1e-7 * (1 + abs(lin)), (key, t, (a, b), r2, lin)
                checks += 1
    if not _has_objective(model, tm):
        return checks
    x0 = _x(tm, m, pos)
    for j, (name, a, b) in enumerate(cost):
        for d in (a * 0.5 if a > -INF else -1.0, b * 0.5 if b < INF else 1.0):
            st2, r2, *_ = _raw(_set_cost(model, name, d))
            lin = base + x0[j] * d
            assert st2 == 0 and abs(r2 - lin) <= 1e-6 * (1 + abs(lin)), (name, d, (a, b), st2, r2, lin)
            checks += 1
        if strict:
            for d in (a - 0.05 * (1 + abs(a)) if a > -INF else None, b + 0.05 * (1 + abs(b)) if b < INF else None):
                if d is None:
                    continue
                st2, r2, tm2, m2, pos2 = _raw(_set_cost(model, name, d))
                assert st2 != 0 or not np.allclose(_x(tm2, m2, pos2), x0, rtol=1e-9, atol=1e-9), (name, d, (a, b))
                checks += 1
    return checks


@pytest.mark.parametrize("seed", range(40))
def test_random_lp_ranges_against_resolves(seed):
    model = random_lp(seed)
    tm, st, *_ = oracle_final(model)
    if st != 0:
        pytest.skip("not optimal")
    strict = _non_degenerate(model) and not any("equal" in con for _, con in model["constraints"])
    assert _check_inside(model, strict) > 0


GOLDEN_LP = [c for c in LP_CASES if {**S._DEFAULTS, **c["options"]}["precision"] == 1e-8
             and not c["options"].get("checkCycles")]


@pytest.mark.parametrize("case", GOLDEN_LP, ids=[c["name"] for c in GOLDEN_LP])
def test_golden_lp_ranges_inside(case):
    tm, st, *_ = oracle_final(case["model"])
    if st != 0:
        pytest.skip("not optimal")
    _check_inside(case["model"], strict=False)


@pytest.mark.parametrize("seed", range(20))
def test_key_ranges_equal_explicit_direction(seed):
    model = random_lp(seed)
    tm, st, m, pos, rows, lo, hi = _oracle_ranges(model)
    if st != 0:
        pytest.skip("not optimal")
    W, H = tm.tableau.width, tm.tableau.height
    M = m.reshape(H, W)
    _, rhs = model_ranges(tm.variables, rows, lo, hi, W, tm.sign)

    def direction(k):
        p = pos[W + k]
        return M[:, p].copy() if p < W else np.eye(H)[p - W]

    for (key, up, lw), (_, a, b) in zip(rows, rhs):
        d = np.zeros(H)
        if up >= 0:
            d = direction(up)
        if lw >= 0:
            d = d - direction(lw)
        x = -np.maximum(M[1:, 0], 0.0) / np.where(np.abs(d[1:]) > 1e-8, d[1:], np.nan)
        ea = np.max(x[d[1:] > 1e-8], initial=-INF) + 0.0
        eb = np.min(x[d[1:] < -1e-8], initial=INF) + 0.0
        assert (a, b) == (ea, eb), (key, (a, b), (ea, eb))


# ------------------------------------------------------------------------------------------- model level
def _oracle_solution(model, options=None):
    """What solve(model, {..., ranging: True}) returns, computed from the oracle's final tableau."""
    opt = {**S._DEFAULTS, **(options or {}), "ranging": True}
    tm, st, val, m, pos, var = oracle_final(model, opt)
    _, _, _, _, rows, lo, hi = _oracle_ranges(model, opt)
    t = tm.tableau
    rhs = m.reshape(t.height, t.width)[:, 0].copy()
    sol = S._solution(tm, S.STATUS_NAMES[st], val, rhs, pos, var, opt)
    return S._with_sensitivity(sol, tm, model, reduced_from_tableau(m, t.width, t.height, pos), (lo, hi))


def test_worked_examples():
    sol = _oracle_solution({"direction": "maximize", "objective": "p", "constraints": {"c": {"max": 4}},
                            "variables": {"x": {"c": 1, "p": 3}}})
    assert sol["rhsRanges"] == [["c", -4.0, INF]] and sol["costRanges"] == [["x", -3.0, INF]]
    assert sol["shadowPrices"] == [["c", 3.0]]
    # minimise twin: the objective row holds -3, the sign flip maps (lo, hi) to (-hi, -lo)
    sol = _oracle_solution({"direction": "minimize", "objective": "p", "constraints": {"c": {"min": 4}},
                            "variables": {"x": {"c": 1, "p": 3}}})
    assert sol["result"] == 12.0 and sol["shadowPrices"] == [["c", 3.0]]
    assert sol["rhsRanges"] == [["c", -4.0, INF]] and sol["costRanges"] == [["x", -3.0, INF]]
    # a key with no finite bound
    sol = _oracle_solution({"direction": "maximize", "objective": "p", "constraints": {"c": {"max": 4}, "free": {}},
                            "variables": {"x": {"c": 1, "p": 3, "free": 1}}})
    assert sol["rhsRanges"][1] == ["free", -INF, INF]


def test_zeros_are_positive_and_non_optimal_is_empty():
    for seed in range(10):
        sol = _oracle_solution(random_lp(seed))
        for _, a, b in sol.get("costRanges", []) + sol.get("rhsRanges", []):
            assert a <= 0 <= b
            assert a != 0 or math.copysign(1.0, a) == 1.0
            assert b != 0 or math.copysign(1.0, b) == 1.0
    sol = _oracle_solution({"direction": "maximize", "objective": "p", "constraints": {"c": {"min": 4, "max": 3}},
                            "variables": {"x": {"c": 1, "p": 3}}})
    assert sol["status"] == "infeasible" and sol["costRanges"] == [] and sol["rhsRanges"] == []


def test_ranging_rejects_milp_before_any_engine():
    model = {"direction": "maximize", "objective": "p", "constraints": {"c": {"max": 4}},
             "variables": {"x": {"c": 1, "p": 3}}, "integers": ["x"]}
    created = []
    real = S.get_engine
    S.get_engine = lambda device=0: created.append(device)
    try:
        with pytest.raises(ValueError):
            S.solve(model, {"ranging": True})
        with pytest.raises(ValueError):
            S.solve_many([model], {"ranging": True})
    finally:
        S.get_engine = real
    assert created == []
