"""Warm starts that add constraints and variables, without a GPU (yalps_b200/warm.py steps 2, 4 and 5): the extended
start tableau pinned against today's warm tableau, against cold oracle solves of the changed model and scipy HiGHS,
against the applyCuts row of branch and cut, and against tableau_model of the changed model; the padding of a mixed
batch, the model-level refusals, and the Engine input checks against a fake library."""
import math
import zlib

import numpy as np
import pytest
from scipy.optimize import linprog

import yalps_b200
from conftest import load_netlib, same_bits
from oracle import lib as O
from oracle.model import result_is_optimal
from test_certificate import random_infeasible, random_unbounded
from test_sensitivity import oracle_final, random_lp
from test_warm import FURNITURE, OPT, OracleWarmEngine, apply_variant, base_final, highs
from yalps_b200 import _ffi
from yalps_b200.sensitivity import certificate_from_tableau, ranges_from_tableau, reduced_from_tableau
from yalps_b200.tableau import _merged_rows, entries, tableau_model
from yalps_b200.warm import extended_basis, variant_additions, variant_vectors, warm_tableau

INF = math.inf


# ------------------------------------------------------------------------------------------- helpers
def cold_tableau(M0, H, W, rows, cols):
    """The changed model's initial tableau at tableau level: M0 with the columns appended on the right and the rows at
    the bottom."""
    K, M = len(rows), len(cols)
    C = np.zeros((H + K, W + M))
    C[:H, :W] = np.asarray(M0).reshape(H, W)
    for j in range(M):
        C[:H, W + j] = cols[j]
    for i in range(K):
        C[H + i] = rows[i]
    return C.reshape(-1)


def solve_ext(M0, F, pos, var, H, W, rhs=None, obj=None, rows=None, cols=None, opt=OPT):
    """The reference loop on the extended start tableau: (status, value, pivots, T final, pos, var)."""
    K = 0 if rows is None else len(rows)
    M = 0 if cols is None else len(cols)
    T = warm_tableau(M0, F, pos, H, W, rhs, obj, rows, cols).copy()
    p, v = extended_basis(pos, var, H, W, K, M)
    st, val, piv = O.simplex(T, W + M, H + K, p, v, opt["precision"], opt["maxPivots"], opt["checkCycles"])
    return st, val, piv, T, p, v


def solve_cold(C, H, W, opt=OPT):
    ident = np.arange(H + W, dtype=np.int32)
    return O.simplex(C.copy(), W, H, ident.copy(), ident.copy(), opt["precision"], opt["maxPivots"],
                     opt["checkCycles"])


def highs_tableau(C, H, W):
    """scipy HiGHS on a tableau: maximise row 0 . x over rows a.x <= b, x >= 0; (status 0/2/3, final M[0,0])."""
    m = C.reshape(H, W)
    r = linprog(-m[0, 1:], A_ub=m[1:, 1:], b_ub=m[1:, 0], bounds=[(0, None)] * (W - 1), method="highs")
    return r.status, (r.fun if r.status == 0 else None)


def vertex(F, pos, H, W):
    """The structural values of the final basis."""
    p = np.asarray(pos)[1:W]
    return np.where(p >= W, F.reshape(H, W)[:, 0][np.clip(p - W, 0, H - 1)], 0.0)


def random_additions(rng, M0, F, pos, H, W, K, M):
    """K rows that cut off the base vertex (a.x <= a.x* scaled down) and M columns, each a copy of a base column with a
    more attractive cost, plus random added-column coefficients in the added rows."""
    x = vertex(F, pos, H, W)
    m0 = M0.reshape(H, W)
    cols = []
    for _ in range(M):
        j = int(rng.integers(1, W))
        g = m0[:, j].copy()
        g[0] = g[0] + abs(g[0]) * 0.25 + 0.5
        cols.append(g)
    rows = []
    for _ in range(K):
        a = np.zeros(W + M)
        support = rng.random(W - 1) < max(0.3, 3.0 / W)
        a[1:W] = np.round(rng.uniform(0.5, 3.0, W - 1), 3) * support
        a[W:] = np.round(rng.uniform(0.0, 2.0, M), 3) * (rng.random(M) < 0.5)
        ax = float(a[1:W] @ x)
        a[0] = round(ax * float(rng.uniform(0.5, 0.95)), 3) if ax > 0 else float(rng.uniform(0.5, 2.0))
        if rng.random() < 0.3:  # a lower row: -a.x <= -min
            a = -a
            a[0] = -round(ax * float(rng.uniform(0.2, 0.8)), 3)
        rows.append(a)
    return (np.array(rows).reshape(K, W + M) if K else None), (np.array(cols).reshape(M, H) if M else None)


def agree(M0, F, pos, var, H, W, rhs, obj, rows, cols, tally):
    """Warm on the extended tableau vs cold oracle solve of the changed tableau vs HiGHS: status and value."""
    K = 0 if rows is None else len(rows)
    M = 0 if cols is None else len(cols)
    st, val, piv, T, _, _ = solve_ext(M0, F, pos, var, H, W, rhs, obj, rows, cols)
    base = M0.reshape(H, W).copy()
    if rhs is not None:
        base[:, 0] = rhs
    if obj is not None:
        base[0, 1:] = obj[1:]
    C = cold_tableau(base, H, W, [] if rows is None else rows, [] if cols is None else cols)
    cst, cval, cpiv = solve_cold(C, H + K, W + M)
    tally["warm"] += sum(piv)
    tally["cold"] += sum(cpiv)
    assert st == cst, (st, cst)
    hs, hval = highs_tableau(C, H + K, W + M)
    assert hs == {0: 0, 1: 2, 2: 3}[st], (st, hs)
    if st == 0:
        assert abs(T[0] - cval) <= 1e-6 * max(1.0, abs(cval)), (T[0], cval)
        assert abs(T[0] - hval) <= 1e-6 * max(1.0, abs(hval)), (T[0], hval)


TALLY = {"warm": 0, "cold": 0}
KINDS = ["rows", "cols", "both", "rows+rhs", "cols+obj", "both+rhs+obj"]


def variant_inputs(rng, M0, F, pos, H, W, kind):
    K = int(rng.integers(1, 5)) if "rows" in kind or "both" in kind else 0
    M = int(rng.integers(1, 3)) if "cols" in kind or "both" in kind else 0
    rows, cols = random_additions(rng, M0, F, pos, H, W, K, M)
    m0 = M0.reshape(H, W)
    rhs = obj = None
    if "rhs" in kind:
        rhs = m0[:, 0] * (1 + 0.3 * rng.uniform(-1, 1, H) * (rng.random(H) < 0.5))
    if "obj" in kind:
        obj = m0[0] * (1 + 0.3 * rng.uniform(-1, 1, W) * (rng.random(W) < 0.5))
    return rhs, obj, rows, cols


# ------------------------------------------------------------------------------------------- the definition
RANDOM = ([(f"random_lp{s}", random_lp(s)) for s in range(16)] + [(f"infeasible{s}", random_infeasible(s))
                                                                   for s in range(4)]
          + [(f"unbounded{s}", random_unbounded(s)) for s in range(4)])


@pytest.mark.parametrize("name,model", RANDOM, ids=[m[0] for m in RANDOM])
def test_no_addition_is_todays_warm_tableau(name, model):
    tm, M0, st, F, pos, var = base_final(model)
    H, W = tm.tableau.height, tm.tableau.width
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    rhs = M0.reshape(H, W)[:, 0] + rng.uniform(-1, 1, H)
    obj = M0.reshape(H, W)[0] + rng.uniform(-1, 1, W)
    for r, o in ((None, None), (rhs, None), (None, obj), (rhs, obj)):
        assert same_bits(warm_tableau(M0, F, pos, H, W, r, o, np.zeros((0, W)), np.zeros((0, H))),
                         warm_tableau(M0, F, pos, H, W, r, o))
    p, v = extended_basis(pos, var, H, W, 0, 0)
    assert np.array_equal(p, pos) and np.array_equal(v, var)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("name,model", RANDOM, ids=[m[0] for m in RANDOM])
def test_random_lps_agree_with_cold_solves(name, model, kind):
    tm, M0, st, F, pos, var = base_final(model)
    H, W = tm.tableau.height, tm.tableau.width
    rng = np.random.default_rng(zlib.crc32(f"{name}:{kind}".encode()))
    for _ in range(4):
        agree(M0, F, pos, var, H, W, *variant_inputs(rng, M0, F, pos, H, W, kind), TALLY)


NL = load_netlib()


def _netlib_optimal():
    from oracle import model as OM
    out = []
    for n in NL.names:
        g = NL.get(n)
        if float(NL.z[f"{n}/oracle_seconds"][0]) > 0.3 or g["list"] not in (0, 1) or g["status"] != 0:
            continue
        if OM.result_is_optimal(g["value"], g["index_value"], {**OM.DEFAULT_OPTIONS, "checkCycles": g["check_cycles"]}):
            out.append(n)
    return out[:6]


NETLIB = _netlib_optimal()


@pytest.mark.parametrize("kind", ["rows", "cols", "both+rhs+obj"])
@pytest.mark.parametrize("name", NETLIB)
def test_netlib_agrees_with_cold_solves(name, kind):
    g = NL.get(name)
    H, W = g["height"], g["width"]
    M0 = g["matrix"].copy()
    F = M0.copy()
    pos, var = np.arange(H + W, dtype=np.int32), np.arange(H + W, dtype=np.int32)
    O.simplex(F, W, H, pos, var, 1e-8, 8192, g["check_cycles"])
    rng = np.random.default_rng(zlib.crc32(f"{name}:{kind}".encode()))
    rhs, obj, rows, cols = variant_inputs(rng, M0, F, pos, H, W, kind)
    if rhs is not None:  # Netlib bounds are tight: small moves only
        rhs = M0.reshape(H, W)[:, 0] * (1 + 0.01 * (rhs / np.where(M0.reshape(H, W)[:, 0] == 0, 1, M0.reshape(H, W)[:, 0]) - 1))
    agree(M0, F, pos, var, H, W, rhs, obj, rows, cols, TALLY)


def test_report_pivot_totals():
    """Warm and cold pivots of the agreement tests (printed, not asserted)."""
    print(f"\nadded rows / columns: {TALLY['warm']} pivots warm vs {TALLY['cold']} cold")


@pytest.mark.parametrize("name,model", RANDOM[:16], ids=[m[0] for m in RANDOM[:16]])
def test_one_variable_cut_is_the_apply_cuts_row(name, model):
    tm, M0, st, F, pos, var = base_final(model)
    H, W = tm.tableau.height, tm.tableau.width
    for j in range(1, W):
        for sign, value in ((1.0, 0.75), (-1.0, 1.25)):
            a = np.zeros(W)
            a[0], a[j] = sign * value, sign
            T = warm_tableau(M0, F, pos, H, W, rows=a[None, :]).reshape(H + 1, W)
            ref, rpos, rvar = O.apply_cuts(F.copy(), W, H, pos.copy(), var.copy(), [sign], [j], [value])
            assert np.array_equal(T[H], ref.reshape(H + 1, W)[H]), (j, sign)  # == : zeros may differ in sign
            assert same_bits(T[:H], ref.reshape(H + 1, W)[:H])
            p, v = extended_basis(pos, var, H, W, 1, 0)
            assert np.array_equal(p, rpos) and np.array_equal(v, rvar)


def test_added_column_by_hand():
    """max 3x + 2y s.t. x + y <= 4, x <= 3 (x = 3, y = 1): a chair z of profit 4 using 1 of a is worth 4 - 2 = 2 more
    per unit than y (its reduced cost) and beats x too, so z = 4 (16); a budget row x + y + z <= 3 then cuts it to 12."""
    model = {"direction": "maximize", "objective": "p", "constraints": {"a": {"max": 4}, "b": {"max": 3}},
             "variables": {"x": {"p": 3, "a": 1, "b": 1}, "y": {"p": 2, "a": 1}}}
    tm, M0, st, F, pos, var = base_final(model)
    H, W = tm.tableau.height, tm.tableau.width
    g = np.array([[4.0, 1.0, 0.0]])
    T = warm_tableau(M0, F, pos, H, W, cols=g).reshape(H, W + 1)
    assert T[0, W] == 2.0
    st, val, piv, T, *_ = solve_ext(M0, F, pos, var, H, W, cols=g)
    assert st == 0 and -T[0] == 16.0
    st, val, piv, T, *_ = solve_ext(M0, F, pos, var, H, W, rows=np.array([[3.0, 1.0, 1.0, 1.0]]), cols=g)
    assert st == 0 and -T[0] == 12.0


# ------------------------------------------------------------------------------------------- the model level
def apply_additions(model, variant):
    """The changed model itself: apply_variant's changes, the added keys appended after the model's (an existing key's
    new bound as one more entry of that key, which tableau.ts merges), the added variables after the model's."""
    m = apply_variant(model, variant)
    add_c = list(entries(variant.get("addConstraints") or {}))
    cons = list(m["constraints"]) + [(k, {b: v for b, v in spec.items() if b != "coefficients"}) for k, spec in add_c]
    new = {k: dict(entries(spec["coefficients"])) for k, spec in add_c if "coefficients" in spec}
    variables = []
    for name, cs in m["variables"]:
        cs = [(k, c) for k, c in cs if k not in new] + [(k, co[name]) for k, co in new.items() if name in co]
        variables.append((name, cs))
    variables += [(name, list(entries(cs))) for name, cs in entries(variant.get("addVariables") or {})]
    return {**m, "constraints": cons, "variables": variables}


CHAIR = {"addVariables": {"chair": {"profit": 500, "wood": 8, "labor": 4, "budget": 60}},
         "addConstraints": {"budget": {"max": 900, "coefficients": {"table": 100, "dresser": 150}},
                            "wood": {"min": 100}}}
MODEL_VARIANTS = [
    CHAIR,
    {"addConstraints": {"budget": {"max": 900, "coefficients": {"table": 100, "dresser": 150}}}},
    {"addVariables": {"chair": {"profit": 500, "wood": 8, "labor": 4}}, "objective": {"table": 1000}},
    {"addConstraints": {"mix": {"equal": 5, "coefficients": {"table": 1, "dresser": 1}}},
     "constraints": {"labor": {"max": 120}}},
    {"addConstraints": {"storage": {"min": 390}, "floor": {"min": 1, "max": 4, "coefficients": {"dresser": 1}}},
     "addVariables": {"shelf": {"floor": 0, "storage": 20, "profit": 300}}},
    {"addConstraints": {"wood": {"min": 350}}},  # infeasible: wood <= 300 and >= 350
    {"addVariables": {"free": {"profit": 1}}},  # unbounded: a profitable column in no constraint
    {},
]


def test_built_rows_and_columns_are_tableau_model_cells():
    """Every added row and column equals the cells of tableau_model of the changed model, rows matched by (key, side),
    columns by name, bit for bit (negative zeros included)."""
    t = tableau_model(FURNITURE).tableau
    H, W = t.height, t.width
    add = variant_additions(FURNITURE, MODEL_VARIANTS, t)
    for i, v in enumerate(MODEL_VARIANTS):
        ct = tableau_model(apply_additions(FURNITURE, v)).tableau
        C = ct.matrix.reshape(ct.height, ct.width)
        crow = {(k, s): r for k, u, l, _, _ in _merged_rows(list(entries(apply_additions(FURNITURE, v)["constraints"])))
                for s, r in (("max", u), ("min", l)) if r >= 0}
        mine = {(k, s): r for k, u, l in add.keys[i] for s, r in (("max", u), ("min", l)) if r >= 0}
        assert set(mine) == set(crow)
        names = [n for n, _ in add.variables[i]]
        assert names == [n for n, _ in entries(apply_additions(FURNITURE, v)["variables"])]
        nv = len(names)
        for (key, side), r in mine.items():
            c = crow[(key, side)]
            if r >= H:  # an added row over the base and the variant's own columns
                assert same_bits(add.rows[i, r - H, :nv + 1], C[c, :nv + 1]), (key, side)
                assert not add.rows[i, r - H, nv + 1:].any()
            for j in range(nv - (W - 1)):  # the added columns in the base rows
                if r < H:
                    assert same_bits(add.cols[i, j, r], C[c, W + j]), (key, side, j)
        for j in range(nv - (W - 1)):
            assert same_bits(add.cols[i, j, 0], C[0, W + j])
        assert not add.rows[i, len([1 for r in mine.values() if r >= H]):].any()  # padding rows are zero
        assert not add.cols[i, nv - (W - 1):].any()  # padding columns are zero


def test_no_addition_takes_todays_path():
    eng = OracleWarmEngine()
    got = yalps_b200.solve_variants(FURNITURE, [{"constraints": {"wood": {"max": 250}}}], engine=eng)
    assert eng.calls == ["dense"] and got[0]["status"] == "optimal"
    assert variant_additions(FURNITURE, [{}, {"addVariables": {}}], tableau_model(FURNITURE).tableau) is None


class OracleExtendEngine(OracleWarmEngine):
    """solve_warm with add_rows / add_cols on the oracle: the reference loop on the extended warm tableau."""

    def solve_warm(self, base, H, W, rhs, obj, options, want_duals, want_ranges, pairs, want_certificates,
                   add_rows=None, add_cols=None):
        if add_rows is None:
            return super().solve_warm(base, H, W, rhs, obj, options, want_duals, want_ranges, pairs, want_certificates)
        self.calls.append("extend")
        M0 = np.asarray(base, np.float64).copy()
        F, pos, var = M0.copy(), np.arange(W + H, dtype=np.int32), np.arange(W + H, dtype=np.int32)
        O.simplex(F, W, H, pos, var, options.precision, options.max_pivots, bool(options.check_cycles))
        n, K, M = add_rows.shape[0], add_rows.shape[1], add_cols.shape[1]
        Hx, Wx = H + K, W + M
        out = {k: [] for k in ("status", "value", "pivots", "rhs", "pos", "var", "reduced", "range_lo", "range_hi",
                               "certificate", "matrices")}
        for i in range(n):
            T = warm_tableau(M0, F, pos, H, W, None if rhs is None else rhs[i], None if obj is None else obj[i],
                             add_rows[i], add_cols[i]).copy()
            p, v = extended_basis(pos, var, H, W, K, M)
            st, val, piv = O.simplex(T, Wx, Hx, p, v, options.precision, options.max_pivots,
                                     bool(options.check_cycles))
            pr = None if pairs is None else np.asarray(pairs).reshape(n, Hx)[i]
            lo, hi = ranges_from_tableau(T, Wx, Hx, p, options.precision, pr, optimal=st == 0)
            for k, x in (("status", st), ("value", val), ("pivots", piv), ("rhs", T[::Wx].copy()), ("pos", p),
                         ("var", v), ("reduced", reduced_from_tableau(T, Wx, Hx, p)), ("range_lo", lo),
                         ("range_hi", hi), ("matrices", T),
                         ("certificate", certificate_from_tableau(T, Wx, Hx, p, st, val, options.precision))):
                out[k].append(x)
        return {k: np.asarray(x) for k, x in out.items()}


def test_solve_variants_matches_cold_solves():
    """Status and result of every model variant against the oracle's cold solve of the changed model and HiGHS, and
    the ranging and certificate fields name the added keys and variables."""
    eng = OracleExtendEngine()
    got = yalps_b200.solve_variants(FURNITURE, MODEL_VARIANTS, {"ranging": True, "certificate": True}, engine=eng)
    assert eng.calls == ["extend"]
    for v, sol in zip(MODEL_VARIANTS, got):
        changed = apply_additions(FURNITURE, v)
        tm, st, val, F, pos, var = oracle_final(changed)
        assert sol["status"] == ("optimal", "infeasible", "unbounded")[st], (v, sol["status"], st)
        hs, hval = highs(changed)
        assert hs == {0: 0, 1: 2, 2: 3}[st]
        names = [n for n, _ in entries(changed["variables"])]
        keys = list(dict.fromkeys(k for k, _ in changed["constraints"]))
        if st == 0:
            assert result_is_optimal(sol["result"], -tm.sign * F[0], OPT) and result_is_optimal(sol["result"], hval, OPT)
            assert [k for k, *_ in sol["rhsRanges"]] == keys and [k for k, _ in sol["shadowPrices"]] == keys
            assert [k for k, *_ in sol["costRanges"]] == names
            assert {k for k, _ in sol["variables"]} <= set(names)
        elif st == 1:
            assert [k for k, _ in sol["infeasibilityCertificate"]] == keys
        else:
            assert [k for k, _ in sol["unboundedRay"]] == names
    chair = got[0]
    print("\nchair / budget variant:", chair["result"], chair["variables"])


def test_padding_is_invisible():
    """A mixed-K/M batch gives every variant what it gets alone, after relabelling the ids of the padding."""
    t = tableau_model(FURNITURE).tableau
    H, W = t.height, t.width
    eng = OracleExtendEngine()
    batch = yalps_b200.solve_variants(FURNITURE, MODEL_VARIANTS, {"sensitivity": True, "certificate": True}, engine=eng)
    for i, v in enumerate(MODEL_VARIANTS):  # alone: no padding, and today's path for the variant that adds nothing
        alone = yalps_b200.solve_variants(FURNITURE, [v], {"sensitivity": True, "certificate": True},
                                          engine=OracleExtendEngine())[0]
        assert batch[i] == alone, (v, batch[i], alone)
    # and at tableau level: the padded variant's real cells and pivots equal the unpadded one's
    add = variant_additions(FURNITURE, MODEL_VARIANTS, t)
    tm, M0, st, F, pos, var = base_final(FURNITURE)
    K, M = add.rows.shape[1], add.cols.shape[1]
    for i in range(len(MODEL_VARIANTS)):
        ki = sum(1 for _, u, l in add.keys[i] for r in (u, l) if r >= H)
        mi = len(add.variables[i]) - (W - 1)
        pst, pval, ppiv, PT, pp, pv = solve_ext(M0, F, pos, var, H, W, rows=add.rows[i], cols=add.cols[i])
        ast, aval, apiv, AT, ap, av = solve_ext(M0, F, pos, var, H, W, rows=add.rows[i, :ki, :W + mi] if ki else None,
                                                cols=add.cols[i, :mi] if mi else None)
        assert (pst, ppiv) == (ast, apiv) and same_bits(pval, aval)
        PT, AT = PT.reshape(H + K, W + M), AT.reshape(H + ki, W + mi)
        assert same_bits(PT[:H + ki, 0], AT[:, 0]) and same_bits(PT[0, :W + mi], AT[0])


@pytest.mark.parametrize("variant,msg", [
    ({"addConstraints": {"budget": {"max": 1, "coefficients": {"chair": 1}}}}, "no variable 'chair'"),
    ({"addConstraints": {"budget": {"max": 1, "coefficients": {"nope": 1}}}}, "no variable 'nope'"),
    ({"addVariables": {"table": {"profit": 1}}}, "clashes"),
    ({"addConstraints": {"wood": {"max": 200}}}, "already has a finite 'max'"),
    ({"addConstraints": {"wood": {"equal": 200}}}, "already has a finite 'max'"),
    ({"addConstraints": {"wood": {"min": 1, "coefficients": {"table": 1}}}}, "'coefficients' is refused"),
    ({"addConstraints": {"budget": {"max": 1}}}, "needs 'coefficients'"),
    ({"addConstraints": {"budget": {"coefficients": {"table": 1}}}}, "no bound"),
    ({"addConstraints": {"budget": {"most": 1, "coefficients": {"table": 1}}}}, "no bound kind"),
    ({"addConstraints": {"budget": {"max": INF, "coefficients": {"table": 1}}}}, "not finite"),
    ({"addConstraints": {"budget": {"max": 1, "coefficients": {"table": math.nan}}}}, "not finite"),
    ({"addConstraints": {"wood": {"min": -INF}}}, "not finite"),
    ({"addVariables": {"chair": {"profit": INF}}}, "not finite"),
    ({"addVariables": {"chair": {"nope": 1}}}, "no constraint 'nope'"),
    ({"addConstraints": {"profit": {"max": 1, "coefficients": {"table": 1}}}}, "objective"),
    ({"addVariables": {"chair": {"profit": 1}}, "integers": ["chair"]}, "integer"),
    ({"addVariables": {"chair": {"profit": 1}}, "binaries": ["chair"]}, "integer"),
    ({"addConstraints": [("budget", {"max": 1, "coefficients": {"table": 1}}),
                         ("budget", {"min": 0, "coefficients": {"table": 1}})]}, "added twice"),
])
def test_addition_errors(variant, msg):
    with pytest.raises(ValueError, match=msg):
        yalps_b200.solve_variants(FURNITURE, [variant], engine=object())


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

    def _call(self, kind, a):
        self.calls.append((kind,) + tuple(a))
        return 0

    def yalps_solve_warm(self, *a):
        return self._call("warm", a[1:4])

    def yalps_solve_warm_extend(self, *a):
        return self._call("extend", a[1:6] + tuple(x is None for x in a[12:14]))

    def yalps_solve_warm_extend_sparse(self, *a):
        return self._call("sparse", a[1:6] + tuple(x is None for x in a[14:16]))

    def yalps_multi_solve_warm_extend(self, *a):
        return self._call("multi", a[1:6] + tuple(x is None for x in a[12:14]))

    def __getattr__(self, name):
        if name.startswith("yalps_destroy"):
            return lambda *a: None
        raise AttributeError(name)


@pytest.fixture
def fake(monkeypatch):
    lib = FakeLib()
    monkeypatch.setattr(_ffi, "load", lambda: lib)
    return lib


def test_engine_extend_calls(fake):
    eng = yalps_b200.Engine(0)
    base = np.zeros(12)  # 3 x 4
    out = eng.solve_warm(base, 3, 4, add_rows=np.zeros((5, 2, 6)), add_cols=np.zeros((5, 2, 3)), want_duals=True,
                         want_ranges=True, pairs=np.full(5, -1), want_matrices=True)
    assert out["status"].shape == (5,) and out["rhs"].shape == (5, 5) and out["reduced"].shape == (5, 11)
    assert out["matrices"].shape == (5, 30)
    eng.solve_warm(base, 3, 4, rhs=np.zeros((2, 3)), add_rows=np.zeros((2, 1, 4)))
    eng.solve_warm(base, 3, 4, add_cols=np.zeros((2, 1, 3)))
    eng.solve_warm(base, 3, 4, rhs=np.zeros(3))
    eng.solve_warm_sparse([1], [2.0], 3, 4, add_cols=np.zeros((1, 1, 3)))
    yalps_b200.MultiEngine([0, 0]).solve_warm(base, 3, 4, add_rows=np.zeros((3, 0, 4)))
    assert fake.calls == [("extend", 5, 3, 4, 2, 2, False, False), ("extend", 2, 3, 4, 1, 0, False, True),
                          ("extend", 2, 3, 4, 0, 1, True, False), ("warm", 1, 3, 4),
                          ("sparse", 1, 3, 4, 0, 1, True, False), ("multi", 3, 3, 4, 0, 0, True, True)]


@pytest.mark.parametrize("call", [
    dict(add_rows=np.zeros((2, 1, 5))),                                   # row width W + M with M = 0
    dict(add_rows=np.zeros((2, 1, 4)), add_cols=np.zeros((2, 1, 3))),     # rows miss the added column
    dict(add_cols=np.zeros((2, 1, 4))),                                   # columns over the base rows
    dict(add_cols=np.zeros((2, 3))),                                      # not (n, M, H)
    dict(rhs=np.zeros((3, 3)), add_cols=np.zeros((2, 1, 3))),             # different counts
    dict(add_rows=np.zeros((2, 1, 5)), add_cols=np.zeros((3, 1, 3))),     # different counts
    dict(add_rows=np.zeros((2, 1, 4)), pairs=np.full(3, -1), want_ranges=True),  # pairs cover H + K rows
])
def test_bad_extend_arguments_are_refused(fake, call):
    with pytest.raises(ValueError):
        yalps_b200.Engine(0).solve_warm(np.zeros(12), 3, 4, **call)
    with pytest.raises(ValueError):
        yalps_b200.MultiEngine([0]).solve_warm(np.zeros(12), 3, 4, **call)
    assert fake.calls == []
