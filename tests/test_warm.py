"""Warm starts without a GPU (yalps_b200/warm.py): the start tableau of a variant pinned against cold solves of the
changed model on the oracle and against scipy HiGHS, the model-level mapping of solve_variants, and the input checks of
the Engine calls against a fake library."""
import math
import zlib

import numpy as np
import pytest
from scipy.optimize import linprog

import yalps_b200
from conftest import same_bits
from oracle import lib as O
from oracle.model import result_is_optimal
from test_certificate import _model_coefs, random_infeasible, random_unbounded
from test_sensitivity import LP_CASES, oracle_final, random_lp
from yalps_b200 import _ffi
from yalps_b200 import solver as S
from yalps_b200.engine import make_options
from yalps_b200.sensitivity import model_ranges, ranges_from_tableau, reduced_from_tableau, row_pairs
from yalps_b200.tableau import _merged_rows, entries, tableau_model
from yalps_b200.warm import variant_vectors, warm_tableau

INF = math.inf
OPT = dict(S._DEFAULTS)


# ------------------------------------------------------------------------------------------- helpers
def apply_variant(model, variant):
    """The changed model itself: each changed key's entries merged into one with the new bounds (same first-seen order,
    so the same rows), each changed objective coefficient replaced."""
    cons = list(entries(model["constraints"]))
    merged = {key: (hi, lo) for key, _, _, hi, lo in _merged_rows(cons)}
    change = dict(entries(variant.get("constraints") or {}))
    out, seen = [], set()
    for key, con in cons:
        if key not in change:
            out.append((key, con))
            continue
        if key in seen:
            continue
        seen.add(key)
        hi, lo = merged[key]
        for bound, v in change[key].items():
            if bound in ("max", "equal"):
                hi = float(v)
            if bound in ("min", "equal"):
                lo = float(v)
        out.append((key, {**({"max": hi} if math.isfinite(hi) else {}), **({"min": lo} if math.isfinite(lo) else {})}))
    obj = dict(entries(variant.get("objective") or {}))
    variables = []
    for name, cs in entries(model["variables"]):
        cs = dict(entries(cs))
        if name in obj:
            cs[model["objective"]] = float(obj[name])
        variables.append((name, list(cs.items())))
    return {**model, "constraints": out, "variables": variables}


def base_final(model, opt=OPT):
    """(tableau model, M0, status, F, pos, var) of the oracle's cold solve."""
    tm, st, val, F, pos, var = oracle_final(model, opt)
    return tm, tm.tableau.matrix.copy(), st, F, pos, var


def warm_solve(M0, F, pos, var, H, W, rhs, obj, opt=OPT):
    """Oracle run of the reference loop on the warm tableau: (status, value, pivots, T final, pos, var)."""
    T = warm_tableau(M0, F, pos, H, W, rhs, obj).copy()
    p, v = pos.copy(), var.copy()
    st, val, piv = O.simplex(T, W, H, p, v, opt["precision"], opt["maxPivots"], opt["checkCycles"])
    return st, val, piv, T, p, v


SAME_BASIS = [0]


def objective_coef(model, name):
    for n, cs in entries(model["variables"]):
        if n == name:
            return float(dict(entries(cs)).get(model["objective"], 0.0))
    raise KeyError(name)


def highs(model):
    """(scipy HiGHS status: 0 optimal, 2 infeasible, 3 unbounded; result in the model's direction)."""
    names = [k for k, _ in entries(model["variables"])]
    coef, bounds = _model_coefs(model)
    c = np.array([coef.get(model["objective"], {}).get(j, 0.0) for j in names])
    A, b = [], []
    for k, (lo, hi) in bounds.items():
        if k == model["objective"]:
            continue
        row = np.array([coef.get(k, {}).get(j, 0.0) for j in names])
        if hi < INF:
            A.append(row)
            b.append(hi)
        if lo > -INF:
            A.append(-row)
            b.append(-lo)
    dirn = -1.0 if model.get("direction") == "maximize" else 1.0
    r = linprog(dirn * c, A_ub=np.array(A) if A else None, b_ub=b or None, bounds=[(0, None)] * len(names),
                method="highs")
    return r.status, (dirn * r.fun if r.status == 0 else None)


def lp_models():
    cases = [(c["name"], c["model"]) for c in LP_CASES]
    return cases + [(f"random_lp{s}", random_lp(s)) for s in range(20)]


MODELS = lp_models()


# ------------------------------------------------------------------------------------------- the definition
@pytest.mark.parametrize("name,model", MODELS, ids=[m[0] for m in MODELS])
def test_no_change_gives_the_final_tableau(name, model):
    tm, M0, st, F, pos, var = base_final(model)
    H, W = tm.tableau.height, tm.tableau.width
    m0 = M0.reshape(H, W)
    assert same_bits(warm_tableau(M0, F, pos, H, W), F)
    assert same_bits(warm_tableau(M0, F, pos, H, W, m0[:, 0].copy(), m0[0].copy()), F)


def test_definition_by_hand():
    """max 3x + 2y s.t. x + y <= 4, x <= 3: the optimum x = 3, y = 1; the signs of both passes spelled out."""
    model = {"direction": "maximize", "objective": "p", "constraints": {"a": {"max": 4}, "b": {"max": 3}},
             "variables": {"x": {"p": 3, "a": 1, "b": 1}, "y": {"p": 2, "a": 1}}}
    tm, M0, st, F, pos, var = base_final(model)
    H, W = tm.tableau.height, tm.tableau.width
    assert st == 0 and -tm.sign * F[0] == 11.0
    # a: 4 -> 5 moves y up by one (and the objective by 2); b: 3 -> 2 moves x down and y up by one
    for new, value in (({"a": {"max": 5}}, 13.0), ({"b": {"max": 2}}, 10.0)):
        rhs, _ = variant_vectors(model, [{"constraints": new}], tm.tableau)
        T = warm_tableau(M0, F, pos, H, W, rhs[0], None).reshape(H, W)
        assert -tm.sign * T[0, 0] == value
    # y's coefficient 2 -> 2.5 (y basic): objective 3*3 + 2.5 = 11.5, still optimal
    _, obj = variant_vectors(model, [{"objective": {"y": 2.5}}], tm.tableau)
    st2, val, piv, T, *_ = warm_solve(M0, F, pos, var, H, W, None, obj[0])
    assert (st2, piv) == (0, (0, 0)) and -tm.sign * T[0] == 11.5


def in_range_variants(model, tm, F, pos, opt=OPT):
    """Variants that move one key's bounds or one objective coefficient halfway to each finite end of its range."""
    t = tm.tableau
    rows = [(k, u, l) for k, u, l, _, _ in _merged_rows(list(entries(model["constraints"])))]
    merged = {k: (hi, lo) for k, _, _, hi, lo in _merged_rows(list(entries(model["constraints"])))}
    lo, hi = ranges_from_tableau(F, t.width, t.height, pos, opt["precision"], row_pairs(rows, t.height))
    cost, rhs = model_ranges(tm.variables, rows, lo, hi, t.width, tm.sign)
    out = []
    for key, a, b in rhs:
        for end in (a, b):
            if math.isfinite(end) and end != 0.0:
                h, lw = merged[key]
                d = end / 2
                bounds = {**({"max": h + d} if math.isfinite(h) else {}), **({"min": lw + d} if math.isfinite(lw) else {})}
                if bounds:
                    out.append({"constraints": {key: bounds}})
    for name, a, b in cost:
        for end in (a, b):
            if math.isfinite(end) and end != 0.0:
                out.append({"objective": {name: objective_coef(model, name) + end / 2}})
    return out


OPTIMAL = [(n, m) for n, m in MODELS if oracle_final(m)[1] == 0]


@pytest.mark.parametrize("name,model", OPTIMAL, ids=[m[0] for m in OPTIMAL])
def test_variants_inside_the_ranges_take_no_pivot(name, model):
    """Inside rhsRanges / costRanges the base's basis stays optimal: the warm tableau is already final, and its column
    0 and row 0 are those of the cold solve of the changed model, compared per variable id where the cold solve ends
    in the same basis (else, at an alternative optimum, the objective value only)."""
    tm, M0, st, F, pos, var = base_final(model)
    H, W = tm.tableau.height, tm.tableau.width
    variants = in_range_variants(model, tm, F, pos)
    if not variants:
        pytest.skip("no finite range end")
    rhs, obj = variant_vectors(model, variants, tm.tableau)
    for i, v in enumerate(variants):
        st, val, piv, T, p, _ = warm_solve(M0, F, pos, var, H, W, None if rhs is None else rhs[i],
                                           None if obj is None else obj[i])
        assert (st, piv) == (0, (0, 0)), (v, st, piv)
        ctm, cst, _, CF, cpos, _ = oracle_final(apply_variant(model, v))
        assert cst == 0
        Tm, Cm = T.reshape(H, W), CF.reshape(H, W)
        x = lambda M, q: np.where(q[:W + H] >= W, M[:, 0][np.clip(q[:W + H] - W, 0, H - 1)], 0.0)
        np.testing.assert_allclose(Tm[0, 0], Cm[0, 0], rtol=1e-9, atol=1e-9)
        if set(np.flatnonzero(p >= W)) == set(np.flatnonzero(cpos >= W)):  # not an alternative optimum
            SAME_BASIS[0] += 1
            np.testing.assert_allclose(reduced_from_tableau(T, W, H, p), reduced_from_tableau(CF, W, H, cpos),
                                       rtol=1e-9, atol=1e-9)
            np.testing.assert_allclose(x(Tm, p), x(Cm, cpos), rtol=1e-9, atol=1e-9)


def random_variant(rng, model, kind):
    """A random RHS, objective or combined change of every key / variable, large enough to change the basis."""
    v = {}
    if kind in ("rhs", "both"):
        cons = {}
        for key, _, _, hi, lo in _merged_rows(list(entries(model["constraints"]))):
            if rng.random() < 0.6:
                f = float(rng.uniform(-0.5, 1.5))
                b = {}
                if math.isfinite(hi):
                    b["max"] = round(hi * (1 + f) + float(rng.uniform(-1, 1)), 3)
                if math.isfinite(lo):
                    b["min"] = min(round(lo * (1 + f) + float(rng.uniform(-1, 1)), 3), b.get("max", INF))
                cons[key] = b
        v["constraints"] = cons
    if kind in ("obj", "both"):
        v["objective"] = {name: round(float(rng.uniform(-3, 4)), 3) for name, _ in entries(model["variables"])
                          if rng.random() < 0.6}
    return v


BIG = ([(f"random_lp{s}", random_lp(s)) for s in range(20)] + [(f"infeasible{s}", random_infeasible(s)) for s in range(6)]
       + [(f"unbounded{s}", random_unbounded(s)) for s in range(6)])
TOTALS = {"warm": 0, "cold": 0, "lps": 0}


@pytest.mark.parametrize("kind", ["rhs", "obj", "both"])
@pytest.mark.parametrize("name,model", BIG, ids=[m[0] for m in BIG])
def test_larger_changes_agree_with_cold_solves(name, model, kind):
    """Statuses equal the cold solve's, optimal results agree within the validator's tolerance, HiGHS agrees on both."""
    rng = np.random.default_rng(zlib.crc32(f"{name}:{kind}".encode()))
    tm, M0, st0, F, pos, var = base_final(model)
    H, W = tm.tableau.height, tm.tableau.width
    variants = [random_variant(rng, model, kind) for _ in range(6)]
    rhs, obj = variant_vectors(model, variants, tm.tableau)
    for i, v in enumerate(variants):
        st, val, piv, T, p, q = warm_solve(M0, F, pos, var, H, W, None if rhs is None else rhs[i],
                                           None if obj is None else obj[i])
        changed = apply_variant(model, v)
        ctm, cst, cval, CF, _, _ = oracle_final(changed)
        _, _, cpiv = O.simplex(ctm.tableau.matrix.copy(), W, H, ctm.tableau.position_of_variable.copy(),
                               ctm.tableau.variable_at_position.copy())
        TOTALS["warm"] += sum(piv)
        TOTALS["cold"] += sum(cpiv)
        TOTALS["lps"] += 1
        assert st == cst, (v, st, cst)
        hs, hval = highs(changed)
        assert hs == {0: 0, 1: 2, 2: 3}[st], (v, st, hs)
        if st == 0:
            result = -tm.sign * T[0]
            assert result_is_optimal(result, -tm.sign * CF[0], OPT), (result, -tm.sign * CF[0])
            assert result_is_optimal(result, hval, OPT), (result, hval)


def test_report_pivot_totals():
    """Warm and cold pivots of test_larger_changes_agree_with_cold_solves (printed, not asserted)."""
    if TOTALS["lps"]:
        print(f"\nwarm starts: {TOTALS['lps']} variants, {TOTALS['warm']} pivots warm vs {TOTALS['cold']} cold; "
              f"{SAME_BASIS[0]} in-range variants ended in the cold solve's basis")


# ------------------------------------------------------------------------------------------- the model-level mapping
FURNITURE = {"direction": "maximize", "objective": "profit",
             "constraints": {"wood": {"max": 300}, "labor": {"max": 110}, "storage": {"max": 400}},
             "variables": {"table": {"wood": 30, "labor": 5, "profit": 1200, "storage": 30},
                           "dresser": {"wood": 20, "labor": 10, "profit": 1600, "storage": 50}}}


def test_mapping_max_min_equal_and_objective():
    model = {"direction": "minimize", "objective": "cost",
             "constraints": [("a", {"max": 10}), ("b", {"min": 1, "max": 8}), ("a", {"min": 2}), ("c", {"equal": 5})],
             "variables": {"x": {"cost": 2, "a": 1, "b": 1, "c": 1}, "y": {"cost": 3, "a": 1, "c": 2}}}
    t = tableau_model(model).tableau
    # rows: a max 1, a min 2 (merged key, first-seen order), b max 3, b min 4, c max 5, c min 6
    col0 = t.matrix.reshape(t.height, t.width)[:, 0]
    rhs, obj = variant_vectors(model, [{"constraints": {"a": {"max": 12}, "b": {"min": 3}}},
                                       {"constraints": {"c": {"equal": 7}, "a": {"min": 0.5, "max": 9}}},
                                       {"objective": {"y": 4}}], t)
    assert rhs.shape == (3, t.height) and obj.shape == (3, t.width)
    assert rhs[0].tolist() == [col0[0], 12, -2, 8, -3, 5, -5]
    assert rhs[1].tolist() == [col0[0], 9, -0.5, 8, -1, 7, -7]
    assert same_bits(rhs[2], col0)
    row0 = t.matrix[:t.width]
    assert same_bits(obj[0], row0) and same_bits(obj[1], row0)
    assert obj[2].tolist() == [row0[0], row0[1], -4.0]  # minimise: the tableau holds -c
    # no change at all: each variant is the base from its own final basis
    rhs, obj = variant_vectors(model, [{}, {"constraints": {}}], t)
    assert obj is None and same_bits(rhs, np.tile(col0, (2, 1)))


@pytest.mark.parametrize("variant,msg", [
    ({"constraints": {"nope": {"max": 1}}}, "no constraint"),
    ({"objective": {"nope": 1}}, "no variable"),
    ({"constraints": {"wood": {"min": 1}}}, "no finite 'min'"),
    ({"constraints": {"wood": {"equal": 1}}}, "no finite 'equal'"),
    ({"constraints": {"wood": {"max": INF}}}, "infinite"),
    ({"constraints": {"wood": {"most": 1}}}, "no bound kind"),
    ({"bounds": {}}, "unknown field"),
])
def test_mapping_errors(variant, msg):
    with pytest.raises(ValueError, match=msg):
        yalps_b200.solve_variants(FURNITURE, [variant], engine=object())


def test_milp_and_iis_are_refused():
    with pytest.raises(ValueError, match="LP models only"):
        yalps_b200.solve_variants({**FURNITURE, "integers": ["table"]}, [{}], engine=object())
    with pytest.raises(ValueError, match="iis"):
        yalps_b200.solve_variants(FURNITURE, [{}], {"iis": True}, engine=object())


class OracleWarmEngine:
    """solve_warm / solve_warm_sparse on the oracle: the reference loop on warm_tableau of the base's cold solve."""

    def __init__(self):
        self.calls = []

    def _run(self, M0, H, W, rhs, obj, options, want_duals, want_ranges, pairs, want_certificates, final=None):
        from yalps_b200.sensitivity import certificate_from_tableau
        F, pos, var = M0.copy(), np.arange(W + H, dtype=np.int32), np.arange(W + H, dtype=np.int32)
        O.simplex(F, W, H, pos, var, options.precision, options.max_pivots, bool(options.check_cycles))
        n = len(rhs if rhs is not None else obj)
        out = {k: [] for k in ("status", "value", "rhs", "pos", "var", "reduced", "range_lo", "range_hi",
                               "certificate")}
        for i in range(n):
            T = warm_tableau(M0, F, pos, H, W, None if rhs is None else rhs[i], None if obj is None else obj[i]).copy()
            p, v = pos.copy(), var.copy()
            st, val, _ = O.simplex(T, W, H, p, v, options.precision, options.max_pivots, bool(options.check_cycles))
            lo, hi = ranges_from_tableau(T, W, H, p, options.precision, pairs, optimal=st == 0)
            for k, x in (("status", st), ("value", val), ("rhs", T[::W].copy()), ("pos", p), ("var", v),
                         ("reduced", reduced_from_tableau(T, W, H, p)), ("range_lo", lo), ("range_hi", hi),
                         ("certificate", certificate_from_tableau(T, W, H, p, st, val, options.precision))):
                out[k].append(x)
        return {k: np.asarray(x) for k, x in out.items()}

    def solve_warm(self, base, H, W, rhs, obj, options, want_duals, want_ranges, pairs, want_certificates):
        self.calls.append("dense")
        return self._run(np.asarray(base, np.float64).copy(), H, W, rhs, obj, options, want_duals, want_ranges, pairs,
                         want_certificates)

    def solve_warm_sparse(self, cells, values, H, W, rhs, obj, options, want_duals, want_ranges, pairs,
                          want_certificates):
        self.calls.append("sparse")
        M0 = np.zeros(H * W)
        M0[cells] = values
        return self._run(M0, H, W, rhs, obj, options, want_duals, want_ranges, pairs, want_certificates)


def test_furniture_variants_on_the_oracle():
    """The README example: three wood budgets and a new dresser price, against solve() of each changed model."""
    variants = [{"constraints": {"wood": {"max": v}}} for v in (250, 300, 350)] + [{"objective": {"dresser": 2000}}]
    eng = OracleWarmEngine()
    got = yalps_b200.solve_variants(FURNITURE, variants, {"ranging": True, "certificate": True}, engine=eng)
    assert eng.calls == ["dense"]
    for v, sol in zip(variants, got):
        cold = apply_variant(FURNITURE, v)
        tm, st, val, F, pos, var = oracle_final(cold)
        assert sol["status"] == "optimal" and st == 0
        assert result_is_optimal(sol["result"], -tm.sign * F[0], OPT)
        assert set(sol) == {"status", "result", "variables", "reducedCosts", "shadowPrices", "costRanges", "rhsRanges",
                            "infeasibilityCertificate", "unboundedRay"}
        assert [k for k, _ in sol["shadowPrices"]] == ["wood", "labor", "storage"]
    print("\nfurniture variants:", [s["result"] for s in got])


def test_big_models_go_through_the_sparse_entry():
    n = 400
    model = {"direction": "maximize", "objective": "p",
             "constraints": [(f"c{i}", {"max": 1.0 + i}) for i in range(n)],
             "variables": [(f"x{j}", [("p", 1.0 + (j % 3))] + [(f"c{j}", 1.0)]) for j in range(n)]}
    eng = OracleWarmEngine()
    got = yalps_b200.solve_variants(model, [{"constraints": {"c0": {"max": 2.0}}}], engine=eng)
    assert eng.calls == ["sparse"] and got[0]["status"] == "optimal"


# ------------------------------------------------------------------------------------------- Engine input checks
class FakeLib:
    def __init__(self):
        self.calls = []

    def yalps_create(self, device, out):
        out._obj.value = 0x1000
        return 0

    def yalps_create_multi(self, devices, ndev, out):
        out._obj.value = 0x2000
        return 0

    def _warm(self, kind, args):
        self.calls.append((kind,) + tuple(a is None for a in args))
        return 0

    def yalps_solve_warm(self, *a):
        return self._warm("warm", a[4:10])

    def yalps_solve_warm_sparse(self, *a):
        return self._warm("sparse", a[7:12])

    def yalps_multi_solve_warm(self, *a):
        return self._warm("multi", a[4:10])

    def __getattr__(self, name):
        if name.startswith("yalps_destroy"):
            return lambda *a: None
        raise AttributeError(name)


@pytest.fixture
def fake(monkeypatch):
    lib = FakeLib()
    monkeypatch.setattr(_ffi, "load", lambda: lib)
    return lib


def test_engine_warm_calls(fake):
    eng = yalps_b200.Engine(0)
    base = np.zeros(12)
    out = eng.solve_warm(base, 3, 4, rhs=np.zeros((5, 3)), want_duals=True, want_ranges=True,
                         pairs=np.array([-1, -1, -1]), want_certificates=True)
    assert out["status"].shape == (5,) and out["reduced"].shape == (5, 7) and out["certificate"].shape == (5, 7)
    assert out["base"] == {"status": 0, "value": 0.0, "pivots": (0, 0)}
    ident = np.arange(7)
    out = eng.solve_warm(base, 3, 4, obj=np.zeros((2, 4)), final=(base, ident, ident))
    assert out["base"] is None and out["status"].shape == (2,)
    eng.solve_warm_sparse([1], [2.0], 3, 4, rhs=np.zeros(3), obj=np.zeros(4))
    yalps_b200.MultiEngine([0, 0]).solve_warm(base, 3, 4, rhs=np.zeros((1, 3)))
    # is None: (base, final, pos, var, rhs, obj), sparse: (final, pos, var, rhs, obj)
    assert fake.calls == [("warm", False, True, True, True, False, True), ("warm", False, False, False, False, True, False),
                          ("sparse", True, True, True, False, False), ("multi", False, True, True, True, False, True)]


@pytest.mark.parametrize("call", [
    dict(rhs=None, obj=None),                                        # nothing changes
    dict(rhs=np.zeros(4)),                                           # not whole columns
    dict(obj=np.zeros(5)),                                           # not whole rows
    dict(rhs=np.zeros((2, 3)), obj=np.zeros((3, 4))),                # different counts
    dict(rhs=np.zeros(3), final=(np.zeros(12), np.arange(6), np.arange(7))),  # short basis
    dict(rhs=np.zeros(3), final=(np.zeros(11), np.arange(7), np.arange(7))),  # short final tableau
    dict(rhs=np.zeros(3), options=make_options(precision=-1e-8)),
    dict(rhs=np.zeros(3), options=make_options(precision=math.nan)),
])
def test_bad_warm_arguments_are_refused(fake, call):
    with pytest.raises(ValueError):
        yalps_b200.Engine(0).solve_warm(np.zeros(12), 3, 4, **call)
    with pytest.raises(ValueError):
        yalps_b200.MultiEngine([0]).solve_warm(np.zeros(12), 3, 4, **call)
    with pytest.raises(ValueError):
        yalps_b200.Engine(0).solve_warm(np.zeros(11), 3, 4, rhs=np.zeros(3))  # base of the wrong size
    assert fake.calls == []
