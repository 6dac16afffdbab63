"""Shadow prices and reduced costs (yalps_b200/sensitivity.py) on the oracle's final tableaus: the sign and row
conventions are settled here against scipy's HiGHS marginals, finite differences and LP duality, without a GPU."""
import math

import numpy as np
import pytest
from scipy.optimize import linprog

from conftest import GOLDEN, load_cases
from oracle import lib as O
from yalps_b200 import solver as S
from yalps_b200 import tableau as T
from yalps_b200.mps import netlib_model
from yalps_b200.sensitivity import model_sensitivity, reduced_from_tableau, split_reduced
from yalps_b200.tableau import constraint_rows, entries, tableau_model

LP_CASES = [c for c in load_cases() if not c["model"].get("integers") and not c["model"].get("binaries")]


def oracle_final(model: dict, options: dict = None):
    """Oracle simplex on the model's tableau: (tabmod, status, value, final matrix, pos, var)."""
    opt = {**S._DEFAULTS, **(options or {})}
    tm = tableau_model(model)
    t = tm.tableau
    m = t.matrix.copy()
    pos, var = t.position_of_variable.copy(), t.variable_at_position.copy()
    st, val, _ = O.simplex(m, t.width, t.height, pos, var, opt["precision"], opt["maxPivots"], opt["checkCycles"])
    return tm, st, val, m, pos, var


def oracle_sensitivity(model: dict, options: dict = None) -> dict:
    """What solve(model, {..., sensitivity: True}) returns, computed from the oracle's final tableau."""
    opt = {**S._DEFAULTS, **(options or {})}
    tm, st, val, m, pos, var = oracle_final(model, opt)
    t = tm.tableau
    rhs = m.reshape(t.height, t.width)[:, 0].copy()
    sol = S._solution(tm, S.STATUS_NAMES[st], val, rhs, pos, var, opt)
    return S._with_sensitivity(sol, tm, model, reduced_from_tableau(m, t.width, t.height, pos))


# ------------------------------------------------------------------------------------------------ random LPs
def random_lp(seed: int):
    """A feasible, bounded LP with every constraint kind; returns (model, x0)."""
    rng = np.random.default_rng(seed)
    n, m = int(rng.integers(3, 7)), int(rng.integers(3, 7))
    A = np.round(rng.uniform(0.5, 5.0, (m, n)) * (rng.random((m, n)) < 0.8), 3)
    x0 = np.round(rng.uniform(0.5, 3.0, n), 3)
    ax = A @ x0
    cons = []
    for i in range(m):
        kind = ["lessEq", "greaterEq", "equalTo", "inRange"][i % 4]
        if kind == "lessEq":
            cons.append((f"c{i}", {"max": float(np.round(ax[i] + rng.uniform(-1, 1), 3))}))
        elif kind == "greaterEq":
            cons.append((f"c{i}", {"min": float(np.round(ax[i] - rng.uniform(-1, 1), 3))}))
        elif kind == "equalTo":
            cons.append((f"c{i}", {"equal": float(np.round(ax[i], 3))}))
        else:
            cons.append((f"c{i}", {"min": float(np.round(ax[i] - rng.uniform(0, 2), 3)),
                                   "max": float(np.round(ax[i] + rng.uniform(0, 2), 3))}))
    cons.append(("cap", {"max": float(np.round(x0.sum() * 2, 3))}))  # keeps maximisation bounded
    cost = np.round(rng.uniform(-2, 4, n), 3)
    variables = [(f"x{j}", [(f"c{i}", float(A[i, j])) for i in range(m) if A[i, j] != 0.0] + [("cap", 1.0),
                                                                                                ("obj", float(cost[j]))])
                 for j in range(n)]
    direction = "maximize" if seed % 2 else "minimize"
    return {"direction": direction, "objective": "obj", "constraints": cons, "variables": variables}


def highs_marginals(model: dict):
    """(result, {key: d result / d shift of all the key's bounds}, {variable: d result / d x_j}) from HiGHS."""
    keys = [k for k, _ in model["constraints"]]
    names = [k for k, _ in model["variables"]]
    n = len(names)
    coef = {k: np.zeros(n) for k in keys}
    c = np.zeros(n)
    for j, (_, cs) in enumerate(model["variables"]):
        for ck, v in cs:
            if ck == "obj":
                c[j] = v
            else:
                coef[ck][j] = v
    dirn = -1.0 if model["direction"] == "maximize" else 1.0  # linprog minimises dirn * objective
    A_ub, b_ub, A_eq, b_eq, tags = [], [], [], [], []
    for k, con in model["constraints"]:
        if "equal" in con:
            A_eq.append(coef[k])
            b_eq.append(con["equal"])
            continue
        if "max" in con:
            A_ub.append(coef[k])
            b_ub.append(con["max"])
            tags.append((k, 1.0))
        if "min" in con:
            A_ub.append(-coef[k])
            b_ub.append(-con["min"])
            tags.append((k, -1.0))
    r = linprog(dirn * c, A_ub=np.array(A_ub) if A_ub else None, b_ub=b_ub or None,
                A_eq=np.array(A_eq) if A_eq else None, b_eq=b_eq or None, bounds=[(0, None)] * n, method="highs")
    assert r.status == 0
    shadow = {k: 0.0 for k in keys}
    for (k, s), mg in zip(tags, r.ineqlin.marginals):
        shadow[k] += s * mg * dirn
    if A_eq:
        eq_keys = [k for k, con in model["constraints"] if "equal" in con]
        for k, mg in zip(eq_keys, r.eqlin.marginals):
            shadow[k] += mg * dirn
    reduced = {names[j]: float(r.lower.marginals[j]) * dirn for j in range(n)}
    return dirn * r.fun, shadow, reduced


def _non_degenerate(model) -> bool:
    """Optimal with every basic value above 1e-9, except the slack of an equality's second row: its two rows are
    both tight, so one of their slacks is basic at 0 in every optimal basis."""
    tm, st, _, m, pos, var = oracle_final(model)
    t = tm.tableau
    offset = {k: u for k, u, _ in constraint_rows(model["constraints"])}
    eq_rows = {offset[k] + i for k, con in model["constraints"] if "equal" in con for i in (0, 1)}
    values = m.reshape(t.height, t.width)[:, 0]
    keep = [r for r in range(1, t.height) if not (var[t.width + r] - t.width in eq_rows)]
    return st == 0 and bool(np.all(values[keep] > 1e-9))


SEEDS = list(range(40))


@pytest.mark.parametrize("seed", SEEDS)
def test_random_lp_matches_highs_marginals(seed):
    model = random_lp(seed)
    if not _non_degenerate(model):
        pytest.skip("optimal basis is degenerate or the LP is not optimal: marginals are not unique")
    sol = oracle_sensitivity(model)
    result, shadow, reduced = highs_marginals(model)
    assert math.isclose(sol["result"], result, rel_tol=1e-9, abs_tol=1e-8)
    for k, v in sol["shadowPrices"]:
        assert math.isclose(v, shadow[k], rel_tol=1e-9, abs_tol=1e-9), (k, v, shadow[k])
    for k, v in sol["reducedCosts"]:
        assert math.isclose(v, reduced[k], rel_tol=1e-9, abs_tol=1e-9), (k, v, reduced[k])


def _shift(model, key, delta):
    cons = []
    for k, con in model["constraints"]:
        if k == key:
            con = {b: v + delta for b, v in con.items()}
        cons.append((k, con))
    return {**model, "constraints": cons}


@pytest.mark.parametrize("seed", SEEDS[:16])
def test_random_lp_finite_differences(seed):
    model = random_lp(seed)
    if not _non_degenerate(model):
        pytest.skip("degenerate optimal basis: one-sided derivatives may differ")
    sol = oracle_sensitivity(model)
    base = _raw_result(model)
    delta = 1e-6
    for k, v in sol["shadowPrices"]:
        fd = (_raw_result(_shift(model, k, delta)) - base) / delta  # (unrounded results: the reported ones are rounded)
        assert math.isclose(fd, v, rel_tol=1e-6, abs_tol=1e-6), (k, fd, v)


def _raw_result(model) -> float:
    tm, st, _, m, _, _ = oracle_final(model)
    assert st == 0
    return -tm.sign * m[0]


# --------------------------------------------------------------------------------------- reference cases
@pytest.mark.parametrize("case", LP_CASES, ids=[c["name"] for c in LP_CASES])
def test_golden_lp_duality(case):
    """Any optimal basis, degenerate ones included: dual feasibility, complementary slackness, strong duality."""
    opt = {**S._DEFAULTS, **case["options"]}
    tm, st, val, m, pos, var = oracle_final(case["model"], opt)
    if st != 0:
        pytest.skip("not optimal")
    t = tm.tableau
    W, H = t.width, t.height
    red = reduced_from_tableau(m, W, H, pos)
    # dual sign feasibility: optimal means no row-0 cell above precision (src/simplex.ts:71-79)
    assert np.all(red <= opt["precision"])
    # basic variables carry no reduced cost (+0.0 exactly)
    basic = pos >= W
    assert np.all(red[basic] == 0.0) and not np.any(np.signbit(red[basic]))
    y, d = split_reduced(red, W, tm.sign)
    # non-zero shadow price only on tight rows: activity recomputed from the primal solution
    M0 = t.matrix.reshape(H, W)
    final_rhs = m.reshape(H, W)[:, 0]
    x = np.zeros(W)
    for j in range(1, W):
        x[j] = final_rhs[pos[j] - W] if pos[j] >= W else 0.0
    b0 = M0[:, 0]
    slack = b0[1:] - M0[1:, 1:] @ x[1:]
    scale = 1.0 + np.abs(b0[1:]) + np.abs(M0[1:, 1:]) @ np.abs(x[1:])
    assert np.all(np.abs(slack[y[1:] != 0.0]) <= 1e-7 * scale[y[1:] != 0.0])
    # strong duality: result = sum_r y(r) * rhs_r of the initial tableau, within 1e-9 of the terms' magnitude (the
    # unrounded result: the reported one is rounded to `precision`)
    result = -tm.sign * m[0]
    terms = y[1:] * b0[1:]
    assert abs(result - terms.sum()) <= 1e-9 * (1.0 + np.abs(terms).sum()), (result, terms.sum())
    # the model-level lists: one entry per variable and per merged key
    rows = constraint_rows(list(entries(case["model"]["constraints"])))
    rc, sp = model_sensitivity(tm.variables, rows, red, W, tm.sign)
    assert [k for k, _ in rc] == [k for k, _ in tm.variables] and [k for k, _ in sp] == [k for k, *_ in rows]


def test_worked_examples():
    sol = oracle_sensitivity({"direction": "maximize", "objective": "p", "constraints": {"c": {"max": 4}},
                              "variables": {"x": {"c": 1, "p": 3}}})
    assert sol["result"] == 12.0 and sol["shadowPrices"] == [["c", 3.0]] and sol["reducedCosts"] == [["x", 0.0]]
    sol = oracle_sensitivity({"direction": "minimize", "objective": "p", "constraints": {"c": {"min": 4}},
                              "variables": {"x": {"c": 1, "p": 3}}})
    assert sol["result"] == 12.0 and sol["shadowPrices"] == [["c", 3.0]]


def test_non_optimal_gives_empty_lists():
    sol = oracle_sensitivity({"direction": "maximize", "objective": "p", "constraints": {"c": {"min": 4, "max": 3}},
                              "variables": {"x": {"c": 1, "p": 3}}})
    assert sol["status"] == "infeasible" and sol["reducedCosts"] == [] and sol["shadowPrices"] == []


# ------------------------------------------------------------------------------------------ row numbering
def _committed_mps_models():
    import gzip
    import json
    import os
    out = [netlib_model(open(os.path.join(GOLDEN, "afiro.mps")).read())]
    with gzip.open(os.path.join(GOLDEN, "netlib_bounded.json.gz"), "rt") as f:
        for c in json.load(f):
            try:
                out.append(netlib_model(c["mps"]))
            except ValueError:
                pass
    return out


def test_constraint_rows_match_both_builders():
    models = [c["model"] for c in load_cases()] + _committed_mps_models()
    assert len(models) >= 47
    for model in models:
        variables = list(entries(model["variables"]))
        constraints = list(entries(model["constraints"]))
        rows = constraint_rows(constraints)
        n_rows = 1 + sum((u >= 0) + (lo >= 0) for _, u, lo in rows)
        sign = -1.0 if model.get("direction") == "minimize" else 1.0
        width = len(variables) + 1
        _, _, py_rows = T._stores_python(variables, constraints, model.get("objective"), sign, width, [])
        assert py_rows == n_rows
        if T._NATIVE is not None:
            _, _, native_rows = T._NATIVE.build(variables, constraints, model.get("objective"), sign, width, [], entries)
            assert native_rows == n_rows
        tm = tableau_model(model)
        if not model.get("binaries"):
            assert tm.tableau.height == n_rows
        # numbering: distinct rows 1..n_rows-1, upper before lower
        nums = [r for _, u, lo in rows for r in (u, lo) if r >= 0]
        assert nums == list(range(1, n_rows))


def test_sensitivity_rejects_milp_before_any_engine():
    model = {"direction": "maximize", "objective": "p", "constraints": {"c": {"max": 4}},
             "variables": {"x": {"c": 1, "p": 3}}, "integers": ["x"]}
    created = []
    real = S.get_engine
    S.get_engine = lambda device=0: created.append(device)
    try:
        with pytest.raises(ValueError):
            S.solve(model, {"sensitivity": True})
        with pytest.raises(ValueError):
            S.solve_many([model], {"sensitivity": True})
    finally:
        S.get_engine = real
    assert created == []
