"""Certificates of infeasible and unbounded LPs (yalps_b200/sensitivity.py) without a GPU: certificate_from_tableau
against a literal per-id statement of its definition, and the certificates of the oracle's final tableaus against the
Farkas and ray identities of the original tableau and the model."""
import math

import numpy as np
import pytest
from scipy.optimize import linprog

from conftest import load_netlib
from oracle import lib as O
from test_sensitivity import LP_CASES, oracle_final
from yalps_b200 import solver as S
from yalps_b200.sensitivity import certificate_from_tableau, model_certificate
from yalps_b200.tableau import constraint_rows, entries

INF = math.inf


# ------------------------------------------------------------------------------------------- the definition
def per_id_certificate(m, W, H, pos, status, value, prec):
    """One id at a time, exactly as the definition reads (the row choice is the reference's strict-< scan)."""
    M = np.asarray(m, np.float64).reshape(H, W)
    out = [math.nan] * (W + H)
    if status == 1:
        r, best = -1, INF
        for k in range(1, H):
            v = float(M[k, 0])
            if v < -prec and v < best:
                r, best = k, v
        if r < 0:
            return np.array(out)
        for v in range(W + H):
            p = int(pos[v])
            if v == 0:
                out[v] = float(M[r, 0])
            elif v == W:
                out[v] = 0.0
            elif 1 <= p < W:
                out[v] = float(M[r, p])
            elif p == W + r:
                out[v] = 1.0
            else:
                out[v] = 0.0
    elif status == 2:
        if not (1.0 <= value < W):
            return np.array(out)
        c = int(value)
        for v in range(W + H):
            p = int(pos[v])
            if v == 0:
                out[v] = float(M[0, c])
            elif v == W:
                out[v] = 0.0
            elif p == c:
                out[v] = 1.0
            elif W + 1 <= p < W + H:
                out[v] = -float(M[p - W, c])
            else:
                out[v] = 0.0
    return np.array(out)


def same_bits(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return a.shape == b.shape and np.array_equal(a.view(np.uint64), b.view(np.uint64))


def synthetic(rng, H, W, prec=1e-8):
    """A random 'final' tableau with a random basis, and a (status, value) pair: ties, NaN and +-inf in column 0 and in
    the cells, signed zeros, cells at exactly -precision, and values outside the column range."""
    M = rng.normal(size=(H, W)) * (rng.random((H, W)) < 0.7)
    special = rng.integers(0, H * W, 6 + H * W // 8)
    vals = np.array([0.0, -0.0, prec, -prec, -2 * prec, np.nan, INF, -INF, -1.5, -1.5])
    M.reshape(-1)[special] = vals[rng.integers(0, vals.size, special.size)]
    if H > 3 and rng.random() < 0.5:  # a tie for the most negative RHS
        rows = rng.choice(np.arange(1, H), 2, replace=False)
        M[rows, 0] = -3.25
    ids = np.array([v for v in range(W + H) if v not in (0, W)])
    slots = np.array([s for s in range(W + H) if s not in (0, W)])
    pos = np.zeros(W + H, np.int32)
    pos[W] = W
    pos[ids] = rng.permutation(slots)
    status = int(rng.integers(0, 5))
    value = [float(rng.integers(0, W + 2)), rng.uniform(-1, W + 1), math.nan, -0.0, float(W - 1), 1.0][rng.integers(0, 6)]
    return M.reshape(-1), pos, status, value


@pytest.mark.parametrize("seed", range(60))
def test_reference_equals_definition_bit_for_bit(seed):
    rng = np.random.default_rng(seed)
    H, W = int(rng.integers(2, 12)), int(rng.integers(2, 14))
    prec = [1e-8, 0.5, 0.0][seed % 3]
    m, pos, status, value = synthetic(rng, H, W, prec if prec else 1e-8)
    for st in (status, 1, 2):
        got = certificate_from_tableau(m, W, H, pos, st, value, prec)
        exp = per_id_certificate(m, W, H, pos, st, value, prec)
        assert same_bits(got, exp), (st, value)


def test_reference_special_rules():
    nan = math.nan
    # rows: NaN never qualifies, -inf does; the first of two equal minima wins; -0.0 is copied as it is
    M = np.array([[0.0, 1.0, 2.0],
                  [nan, -1.0, 5.0],
                  [-INF, -0.0, 3.0],
                  [-INF, 4.0, -2.0]])
    pos = np.array([0, 1, 2, 3, 4, 5, 6], np.int32)  # identity: ids 1, 2 non-basic, slacks 4..6 basic at rows 1..3
    c = certificate_from_tableau(M, 3, 4, pos, 1, nan, 1e-8)
    assert same_bits(c, [-INF, -0.0, 3.0, 0.0, 0.0, 1.0, 0.0])
    # no qualifying row, an out-of-range column, and every other status: NaN
    M2 = M.copy()
    M2[1:, 0] = [nan, -1e-9, 0.0]
    assert np.isnan(certificate_from_tableau(M2, 3, 4, pos, 1, nan, 1e-8)).all()
    for value in (0.0, 3.0, -0.5, nan, INF):
        assert np.isnan(certificate_from_tableau(M, 3, 4, pos, 2, value, 1e-8)).all()
    for st in (0, 3, 4, -4):
        assert np.isnan(certificate_from_tableau(M, 3, 4, pos, st, 1.0, 1e-8)).all()
    # unbounded: a plain negation, signed zeros flip
    M3 = np.array([[0.0, 2.0, 1.0], [1.0, -0.0, 0.0], [1.0, -INF, 1.0], [1.0, nan, 1.0]])
    c = certificate_from_tableau(M3, 3, 4, pos, 2, 1.7, 1e-8)
    assert same_bits(c, [2.0, 1.0, 0.0, 0.0, 0.0, INF, -nan])


# ------------------------------------------------------------------------------------- oracle final tableaus
def _tableau_checks(M0, W, H, cert, status, prec):
    """Farkas identities (status 1) or ray identities (status 2) of cert against the original tableau M0."""
    A = np.asarray(M0, np.float64).reshape(H, W)
    y = cert[W + 1:W + H]
    if status == 1:
        assert (y >= -prec).all()
        assert cert[0] < -prec
        comb = y @ A[1:, 1:]
        mag = np.abs(y) @ np.abs(A[1:, 1:])
        assert np.all(np.abs(comb - cert[1:W]) <= prec * (1 + mag)), np.max(np.abs(comb - cert[1:W]) / (1 + mag))
        assert (cert[1:W] >= -prec * (1 + mag)).all()
        b = y @ A[1:, 0]
        assert abs(b - cert[0]) <= prec * (1 + np.abs(y) @ np.abs(A[1:, 0]))
    else:
        d = cert[1:W]
        assert (d >= -prec).all() and (y >= -prec).all() and cert[0] > prec
        slack = -(A[1:, 1:] @ d)
        mag = np.abs(A[1:, 1:]) @ np.abs(d)
        assert np.all(np.abs(slack - y) <= prec * (1 + mag))
        obj = A[0, 1:] @ d
        assert abs(obj - cert[0]) <= prec * (1 + np.abs(A[0, 1:]) @ np.abs(d))


def _model_coefs(model):
    """{key: {variable: coefficient}} and the merged (min, max) of each key."""
    coef = {}
    for name, cs in entries(model["variables"]):
        for k, v in entries(cs):
            coef.setdefault(k, {})[name] = coef.get(k, {}).get(name, 0.0) + float(v)
    bounds = {}
    for k, con in entries(model["constraints"]):
        eq = con.get("equal")
        lo = eq if eq is not None else con.get("min")
        hi = eq if eq is not None else con.get("max")
        lo = -INF if lo is None else float(lo)
        hi = INF if hi is None else float(hi)
        a, b = bounds.get(k, (-INF, INF))
        bounds[k] = (max(a, lo), min(b, hi))
    return coef, bounds


def _model_checks(model, sol, cert0, prec):
    coef, bounds = _model_coefs(model)
    names = [k for k, _ in entries(model["variables"])]
    if sol["status"] == "infeasible":
        farkas = sol["infeasibilityCertificate"]
        assert [k for k, _ in farkas] == list(bounds) and sol["unboundedRay"] == []
        terms = [m * (bounds[k][1] if m > 0 else bounds[k][0]) for k, m in farkas if m != 0]
        total = sum(terms)
        scale = 1 + sum(abs(t) for t in terms)
        if all(lo <= hi for lo, hi in bounds.values()):  # a key with min > max is infeasible on its own
            assert total <= cert0 + prec * scale and cert0 < 0
        for j in names:
            s = sum(m * coef.get(k, {}).get(j, 0.0) for k, m in farkas)
            mag = sum(abs(m * coef.get(k, {}).get(j, 0.0)) for k, m in farkas)
            assert s >= -prec * (1 + mag), (j, s)
    else:
        ray = dict(sol["unboundedRay"])
        assert list(ray) == names and sol["infeasibilityCertificate"] == []
        assert all(d >= -prec for d in ray.values())
        for k, (lo, hi) in bounds.items():
            ad = sum(v * ray[j] for j, v in coef.get(k, {}).items() if j in ray)
            mag = sum(abs(v * ray[j]) for j, v in coef.get(k, {}).items() if j in ray)
            if hi < INF:
                assert ad <= prec * (1 + mag), (k, ad)
            if lo > -INF:
                assert ad >= -prec * (1 + mag), (k, ad)


def oracle_certificate(model, options=None):
    """What solve(model, {..., certificate: True}) returns, computed from the oracle's final tableau, and cert."""
    opt = {**S._DEFAULTS, **(options or {}), "certificate": True}
    tm, st, val, m, pos, var = oracle_final(model, opt)
    t = tm.tableau
    cert = certificate_from_tableau(m, t.width, t.height, pos, st, val, opt["precision"])
    rhs = m.reshape(t.height, t.width)[:, 0].copy()
    sol = S._solution(tm, S.STATUS_NAMES[st], val, rhs, pos, var, opt)
    return S._with_certificate(sol, tm, model, cert), tm, st, cert


GOLDEN = [c for c in LP_CASES if oracle_final(c["model"], {**S._DEFAULTS, **c["options"]})[1] in (1, 2)]


def test_golden_has_the_cases():
    assert sorted(oracle_final(c["model"], {**S._DEFAULTS, **c["options"]})[1] for c in GOLDEN) == [1, 1, 1, 1, 1, 2]


@pytest.mark.parametrize("case", GOLDEN, ids=[c["name"] for c in GOLDEN])
def test_golden_certificates(case):
    sol, tm, st, cert = oracle_certificate(case["model"], case["options"])
    prec = {**S._DEFAULTS, **case["options"]}["precision"]
    _tableau_checks(tm.tableau.matrix, tm.tableau.width, tm.tableau.height, cert, st, prec)
    _model_checks(case["model"], sol, cert[0], prec)


def random_infeasible(seed):
    """Rows a.x >= lo with a in [0.5, 5] that a small cap on sum x cannot reach, mixed with ordinary rows."""
    rng = np.random.default_rng(1000 + seed)
    n, m = int(rng.integers(2, 7)), int(rng.integers(2, 6))
    cap = float(np.round(rng.uniform(0.5, 2.0), 3))
    cons = [("cap", {"max": cap})]
    variables = {f"x{j}": {"cap": 1.0, "obj": float(np.round(rng.uniform(-2, 3), 3))} for j in range(n)}
    for i in range(m):
        a = np.round(rng.uniform(0.5, 5.0, n), 3)
        kind = i % 3
        for j in range(n):
            variables[f"x{j}"][f"c{i}"] = float(a[j])
        if kind == 0:  # out of reach: a.x <= 5 * sum x <= 5 * cap
            cons.append((f"c{i}", {"min": float(np.round(5 * cap + rng.uniform(0.5, 3), 3))}))
        elif kind == 1:
            cons.append((f"c{i}", {"max": float(np.round(rng.uniform(1, 10), 3))}))
        else:
            cons.append((f"c{i}", {"min": 0.0, "max": float(np.round(rng.uniform(5, 20), 3))}))
    return {"direction": "maximize" if seed % 2 else "minimize", "objective": "obj", "constraints": cons,
            "variables": list(variables.items())}


def random_unbounded(seed):
    """A maximisation whose variables x_k only meet `min` rows (or none), so increasing it never ends."""
    rng = np.random.default_rng(2000 + seed)
    n, m = int(rng.integers(2, 7)), int(rng.integers(2, 6))
    free = int(rng.integers(0, n))
    variables = {f"x{j}": {"obj": float(np.round(rng.uniform(0.5, 3), 3) if j == free else rng.uniform(-2, 3))}
                 for j in range(n)}
    cons = []
    for i in range(m):
        a = np.round(rng.uniform(0.5, 5.0, n) * (rng.random(n) < 0.7), 3)
        if i % 2:  # a max row that leaves the free variable out
            a[free] = 0.0
            cons.append((f"c{i}", {"max": float(np.round(rng.uniform(1, 10), 3))}))
        else:  # a min row the free variable alone can meet
            a[free] = float(np.round(rng.uniform(0.5, 5.0), 3))
            cons.append((f"c{i}", {"min": float(np.round(rng.uniform(0, 3), 3))}))
        for j in range(n):
            if a[j]:
                variables[f"x{j}"][f"c{i}"] = float(a[j])
    sign = 1.0 if seed % 2 else -1.0  # minimise the negated objective half the time
    if sign < 0:
        for v in variables.values():
            v["obj"] = -v["obj"]
    return {"direction": "maximize" if sign > 0 else "minimize", "objective": "obj", "constraints": cons,
            "variables": list(variables.items())}


def highs_status(model):
    """scipy HiGHS status of the model: 2 infeasible, 3 unbounded."""
    names = [k for k, _ in entries(model["variables"])]
    coef, bounds = _model_coefs(model)
    c = np.array([coef.get(model["objective"], {}).get(j, 0.0) for j in names])
    A_ub, b_ub = [], []
    for k, (lo, hi) in bounds.items():
        if k == model["objective"]:
            continue
        row = np.array([coef.get(k, {}).get(j, 0.0) for j in names])
        if hi < INF:
            A_ub.append(row)
            b_ub.append(hi)
        if lo > -INF:
            A_ub.append(-row)
            b_ub.append(-lo)
    dirn = -1.0 if model["direction"] == "maximize" else 1.0
    r = linprog(dirn * c, A_ub=np.array(A_ub) if A_ub else None, b_ub=b_ub or None, bounds=[(0, None)] * len(names),
                method="highs")
    return r.status


@pytest.mark.parametrize("kind,seed", [("infeasible", s) for s in range(25)] + [("unbounded", s) for s in range(25)])
def test_random_certificates(kind, seed):
    model = random_infeasible(seed) if kind == "infeasible" else random_unbounded(seed)
    sol, tm, st, cert = oracle_certificate(model)
    assert highs_status(model) == (2 if kind == "infeasible" else 3)
    assert st == (1 if kind == "infeasible" else 2)
    _tableau_checks(tm.tableau.matrix, tm.tableau.width, tm.tableau.height, cert, st, 1e-8)
    _model_checks(model, sol, cert[0], 1e-8)


NL = load_netlib()


@pytest.mark.parametrize("name", ["ITEST2", "ITEST6", "BGPRTR", "KLEIN1"])
def test_netlib_infeasible(name):
    g = NL.get(name)
    H, W = g["height"], g["width"]
    work = np.ascontiguousarray(g["matrix"], np.float64).reshape(1, -1).copy()
    exp = O.simplex_batch(work, W, H, 1e-8, 8192, g["check_cycles"])
    st = int(exp["status"][0])
    assert st == 1
    cert = certificate_from_tableau(work[0], W, H, exp["pos"][0], st, float(exp["value"][0]), 1e-8)
    assert same_bits(cert, per_id_certificate(work[0], W, H, exp["pos"][0], st, float(exp["value"][0]), 1e-8))
    _tableau_checks(g["matrix"], W, H, cert, st, 1e-8)


# ------------------------------------------------------------------------------------------- model level
def test_worked_examples():
    sol, _, _, cert = oracle_certificate({"direction": "maximize", "objective": "p", "constraints": {"c": {"max": -1}},
                                          "variables": {"x": {"c": 1, "p": 1}}})
    assert sol["status"] == "infeasible" and same_bits(cert, [-1.0, 1.0, 0.0, 1.0])
    assert sol["infeasibilityCertificate"] == [["c", 1.0]] and sol["unboundedRay"] == []
    sol, _, _, cert = oracle_certificate({"direction": "maximize", "objective": "p",
                                          "constraints": {"c1": {"min": 3}, "c2": {"max": 1}},
                                          "variables": {"x": {"c1": 1, "c2": 1, "p": 1}, "y": {"c1": 1, "c2": 1, "p": 2}}})
    assert sol["status"] == "infeasible" and cert[0] == -2.0
    assert sol["infeasibilityCertificate"] == [["c1", -1.0], ["c2", 1.0]]
    sol, _, _, cert = oracle_certificate({"direction": "maximize", "objective": "p", "constraints": {"c": {"max": 1}},
                                          "variables": {"x": {"c": 1, "p": 1}, "y": {"c": -1, "p": 1}}})
    assert sol["status"] == "unbounded" and sol["variables"] == [["y", INF]] and cert[0] == 2.0
    assert sol["unboundedRay"] == [["x", 1.0], ["y", 1.0]] and sol["infeasibilityCertificate"] == []


def test_other_statuses_give_empty_lists():
    rows = constraint_rows([("c", {"max": 4})])
    nan = np.full(4, math.nan)
    for st in (0, 3, 4):
        assert model_certificate([("x", {})], rows, nan, 2, st) == ([], [])
    sol, *_ = oracle_certificate({"direction": "maximize", "objective": "p", "constraints": {"c": {"max": 4}},
                                  "variables": {"x": {"c": 1, "p": 3}}})
    assert sol["status"] == "optimal" and sol["infeasibilityCertificate"] == [] and sol["unboundedRay"] == []


def test_certificate_rejects_milp_before_any_engine():
    model = {"direction": "maximize", "objective": "p", "constraints": {"c": {"max": 4}},
             "variables": {"x": {"c": 1, "p": 3}}, "integers": ["x"]}
    created = []
    real = S.get_engine
    S.get_engine = lambda device=0: created.append(device)
    try:
        with pytest.raises(ValueError):
            S.solve(model, {"certificate": True})
        with pytest.raises(ValueError):
            S.solve_many([model], {"certificate": True})
    finally:
        S.get_engine = real
    assert created == []
