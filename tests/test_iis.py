"""Irreducible infeasible subsets without a GPU (yalps_b200/iis.py): the zero-row fact on the oracle, a host
restatement of the search (iis_reference, which tests/test_gpu_iis.py holds the GPU to) checked against scipy HiGHS, the
model-level mapping, solve() with `iis` on an oracle-backed engine, and the input checks of the Engine calls."""
import ctypes as C
import math

import numpy as np
import pytest
from scipy.optimize import linprog

import yalps_b200
from conftest import load_netlib
from oracle import lib as O
from test_certificate import GOLDEN as GOLDEN_CERT, random_infeasible, random_unbounded
from test_sensitivity import LP_CASES, oracle_final
from yalps_b200 import _ffi
from yalps_b200 import solver as S
from yalps_b200.engine import make_options
from yalps_b200.iis import model_iis
from yalps_b200.sensitivity import certificate_from_tableau
from yalps_b200.tableau import constraint_rows, entries, tableau_model

INF = math.inf
NL = load_netlib()
NETLIB_INFEASIBLE = ["ITEST2", "ITEST6", "BGPRTR", "KLEIN1"]
GOLDEN_INFEASIBLE = [c for c in GOLDEN_CERT if oracle_final(c["model"], {**S._DEFAULTS, **c["options"]})[1] == 1]


# ------------------------------------------------------------------------------------------- the reference
def subset_tableaus(M, H, W, sets) -> np.ndarray:
    """T_S for every S of `sets`: the rows outside S (row 0 excepted) set to +0.0."""
    T = np.asarray(M, np.float64).reshape(H, W)
    out = np.empty((len(sets), H * W))
    for i, s in enumerate(sets):
        keep = np.zeros(H, bool)
        keep[0] = True
        keep[list(s)] = True
        out[i] = np.where(keep[:, None], T, 0.0).reshape(-1)
    return out


def subset_batch(M, H, W, sets, precision=1e-8, max_pivots=8192, check_cycles=False):
    """Oracle solve of T_S for every S of `sets`, with each LP's certificate support (sorted rows, infeasible only)."""
    work = subset_tableaus(M, H, W, sets)
    exp = O.simplex_batch(work, W, H, precision, max_pivots, check_cycles)
    exp["matrices"] = work
    exp["support"] = []
    for i in range(len(sets)):
        st = int(exp["status"][i])
        if st != 1:
            exp["support"].append([])
            continue
        cert = certificate_from_tableau(work[i], W, H, exp["pos"][i], st, float(exp["value"][i]), precision)
        exp["support"].append([k for k in range(1, H) if cert[W + k] > 0.0])
    return exp


def iis_reference(M, H, W, precision=1e-8, max_pivots=8192, check_cycles=False, max_rounds=None):
    """The deletion search of yalps_iis (yalps_b200/iis.py), one oracle batch per round.  max_rounds stands in for the
    timeout: the rounds after round 0 that may run."""
    kw = dict(precision=precision, max_pivots=max_pivots, check_cycles=check_cycles)
    allrows = list(range(1, H))
    e = subset_batch(M, H, W, [allrows], **kw)
    rounds, lps, phases = 1, 1, e["pivots"].sum(axis=0)
    status = int(e["status"][0])
    res = {"status": status, "rows": [], "undecided": 0, "timed_out": False}
    if status == 1:
        S_, fallback = e["support"][0], allrows
        while True:
            if max_rounds is not None and rounds - 1 >= max_rounds:
                res.update(rows=fallback, timed_out=True)
                break
            sets = [S_] + [[r for r in S_ if r != u] for u in S_]
            e = subset_batch(M, H, W, sets, **kw)
            rounds, lps, phases = rounds + 1, lps + len(sets), phases + e["pivots"].sum(axis=0)
            if e["status"][0] != 1:
                S_ = fallback
                continue
            cand = [i for i in range(1, len(sets)) if e["status"][i] == 1]
            if not cand:
                res.update(rows=S_, undecided=sum(int(e["status"][i] == 4) for i in range(1, len(sets))))
                break
            best = min(cand, key=lambda i: (len(e["support"][i]), i))
            fallback = sets[best]
            S_ = e["support"][best]
    res.update(rounds=rounds, lps=lps, pivots=int(phases.sum()), phase_pivots=(int(phases[0]), int(phases[1])),
               irreducible=status == 1 and res["undecided"] == 0 and not res["timed_out"])
    return res


# ------------------------------------------------------------------------------------------- models
def random_feasible(seed):
    """max c.x over positive rows a.x <= b: optimal."""
    rng = np.random.default_rng(3000 + seed)
    n, m = int(rng.integers(2, 7)), int(rng.integers(2, 7))
    variables = {f"x{j}": {"obj": float(np.round(rng.uniform(0.5, 3), 3))} for j in range(n)}
    cons = []
    for i in range(m):
        a = np.round(rng.uniform(0.5, 5.0, n), 3)
        for j in range(n):
            variables[f"x{j}"][f"c{i}"] = float(a[j])
        cons.append((f"c{i}", {"max": float(np.round(rng.uniform(1, 10), 3))} if i % 3 else
                     {"min": 0.5, "max": float(np.round(rng.uniform(5, 20), 3))}))
    return {"direction": "maximize", "objective": "obj", "constraints": cons, "variables": list(variables.items())}


def objective_cut(seed):
    """random_feasible plus a key that asks for an objective 1 better than its optimum z*."""
    model = random_feasible(seed)
    tm, st, val, *_ = oracle_final(model)
    assert st == 0
    zstar = -tm.sign * val
    for _, coefs in model["variables"]:
        coefs["cut"] = coefs["obj"]
    model["constraints"] = model["constraints"] + [("cut", {"min": zstar + 1.0})]
    return model


def tableau_of(model):
    t = tableau_model(model).tableau
    return t.matrix, t.height, t.width


def iis_models():
    """(name, matrix, height, width) of every model the search is checked on."""
    out = [(c["name"], *tableau_of(c["model"])) for c in GOLDEN_INFEASIBLE]
    out += [(f"random_infeasible{s}", *tableau_of(random_infeasible(s))) for s in range(25)]
    for name in NETLIB_INFEASIBLE:
        g = NL.get(name)
        out.append((name, g["matrix"], g["height"], g["width"]))
    out += [(f"objective_cut{s}", *tableau_of(objective_cut(s))) for s in range(5)]
    return out


MODELS = iis_models()


def highs_feasible(M, H, W, rows) -> bool:
    """Does some x >= 0 satisfy M[k,1:].x <= M[k,0] for every k in rows? (scipy HiGHS)"""
    T = np.asarray(M, np.float64).reshape(H, W)
    rows = list(rows)
    if not rows:
        return True
    r = linprog(np.zeros(W - 1), A_ub=T[rows, 1:], b_ub=T[rows, 0], bounds=[(0, None)] * (W - 1), method="highs")
    assert r.status in (0, 2), r.message
    return r.status == 0


# ------------------------------------------------------------------------------------------- the zero-row fact
def restricted_model(model, rows, keep):
    """The model with the bounds of the rows outside `keep` removed (their keys keep their other bound)."""
    cons = []
    for key, up, lo in rows:
        c = {}
        bounds = dict(_merged_bounds(model)[key])
        if up >= 0 and up in keep:
            c["max"] = bounds["max"]
        if lo >= 0 and lo in keep:
            c["min"] = bounds["min"]
        cons.append((key, c))
    return {**model, "constraints": cons}


def _merged_bounds(model):
    out = {}
    for key, con in entries(model["constraints"]):
        eq = con.get("equal")
        lo = eq if eq is not None else con.get("min")
        hi = eq if eq is not None else con.get("max")
        a, b = out.get(key, {"min": -INF, "max": INF}).values()
        out[key] = {"min": max(a, -INF if lo is None else float(lo)), "max": min(b, INF if hi is None else float(hi))}
    return out


FACT_MODELS = ([(c["name"], c["model"]) for c in GOLDEN_INFEASIBLE]
               + [(f"random_infeasible{s}", random_infeasible(s)) for s in range(10)]
               + [(f"random_feasible{s}", random_feasible(s)) for s in range(10)]
               + [(f"random_unbounded{s}", random_unbounded(s)) for s in range(5)]
               + [(c["name"], c["model"]) for c in LP_CASES[:10]])


@pytest.mark.parametrize("name,model", FACT_MODELS, ids=[m[0] for m in FACT_MODELS])
def test_zero_rows_are_removed_rows(name, model):
    tm = tableau_model(model)
    t = tm.tableau
    H, W = t.height, t.width
    rows = constraint_rows(list(entries(model["constraints"])))
    rng = np.random.default_rng(abs(hash(name)) % 2 ** 32)
    for trial in range(4):
        keep = sorted(int(r) for r in np.flatnonzero(rng.random(H - 1) < [0.9, 0.6, 0.3, 1.0][trial]) + 1)
        got = subset_batch(t.matrix, H, W, [keep])
        red = tableau_model(restricted_model(model, rows, set(keep))).tableau
        assert red.height == len(keep) + 1 and red.width == W
        m = red.matrix.copy()
        pos, var = red.position_of_variable.copy(), red.variable_at_position.copy()
        st, val, piv = O.simplex(m, W, red.height, pos, var)
        assert int(got["status"][0]) == st and tuple(got["pivots"][0]) == piv
        assert np.float64(got["value"][0]).tobytes() == np.float64(val).tobytes() or (math.isnan(val) and
                                                                                      math.isnan(got["value"][0]))
        # row-index map: full row keep[j] <-> restricted row j + 1; ids W + r move with their rows
        rmap = {0: 0, **{k: j + 1 for j, k in enumerate(keep)}}
        f = lambda v: v if v < W else W + rmap[v - W]
        full = got["matrices"][0].reshape(H, W)
        assert np.array_equal(full[[0] + keep].view(np.uint64), m.reshape(-1, W).view(np.uint64))
        gone = [r for r in range(1, H) if r not in rmap]
        assert np.array_equal(full[gone].view(np.uint64), np.zeros((len(gone), W), np.uint64))
        assert np.array_equal(got["rhs"][0][[0] + keep].view(np.uint64), m.reshape(-1, W)[:, 0].view(np.uint64))
        gp = got["pos"][0]
        for v in range(W + H):
            if v >= W and v - W in gone:
                assert gp[v] == v  # a removed row's slack stays basic in its own row
            else:
                assert f(int(gp[v])) == pos[f(v)]
                assert got["var"][0][int(gp[v])] == v


# ------------------------------------------------------------------------------------------- the search
@pytest.mark.parametrize("name,M,H,W", MODELS, ids=[m[0] for m in MODELS])
def test_reference_finds_an_iis_highs_agrees(name, M, H, W):
    res = iis_reference(M, H, W)
    # KLEIN1 is degenerate: five of the last round's deletion tests cycle under the reference's pivot rule, so those
    # rows stay undecided for the solver (HiGHS below shows the set is irreducible all the same)
    assert res["status"] == 1 and res["irreducible"] == (name != "KLEIN1"), res
    assert res["undecided"] == (5 if name == "KLEIN1" else 0)
    rows = res["rows"]
    assert rows == sorted(rows) and len(rows) >= 1
    assert not highs_feasible(M, H, W, rows)
    for r in rows:
        assert highs_feasible(M, H, W, [k for k in rows if k != r]), (r, rows)
    assert res["rounds"] <= H + 1


def test_reference_on_feasible_and_unbounded_models():
    for model in (random_feasible(0), random_unbounded(0)):
        M, H, W = tableau_of(model)
        res = iis_reference(M, H, W)
        assert res["status"] in (0, 2) and res["rows"] == [] and not res["irreducible"]
        assert (res["rounds"], res["lps"]) == (1, 1)


def test_reference_timeout_returns_the_last_infeasible_set():
    M, H, W = tableau_of(random_infeasible(3))
    res = iis_reference(M, H, W, max_rounds=0)
    assert res["timed_out"] and not res["irreducible"] and res["rows"] == list(range(1, H)) and res["rounds"] == 1
    res1 = iis_reference(M, H, W, max_rounds=1)
    assert res1["timed_out"] and res1["rounds"] == 2 and len(res1["rows"]) < H - 1
    assert not highs_feasible(M, H, W, res1["rows"])


# ------------------------------------------------------------------------------------------- model level
WORKED = {"direction": "maximize", "objective": "p",
          "constraints": {"c1": {"min": 3}, "c2": {"max": 1}, "c3": {"max": 10}},
          "variables": {"x": {"c1": 1, "c2": 1, "c3": 1, "p": 1}, "y": {"c1": 1, "c2": 1, "p": 2}}}
WORKED_IIS = [["c1", "min"], ["c2", "max"]]


def test_model_iis_mapping():
    rows = constraint_rows([("a", {"max": 1}), ("b", {"min": 2, "max": 5}), ("c", {"equal": 3}), ("d", {}),
                            ("e", {"min": 4, "max": 1})])
    assert [r[1:] for r in rows] == [(1, -1), (2, 3), (4, 5), (-1, -1), (6, 7)]
    assert model_iis(rows, []) == []
    assert model_iis(rows, np.array([3, 1], np.int32)) == [["a", "max"], ["b", "min"]]
    assert model_iis(rows, [5, 4, 7, 6]) == [["c", "max"], ["c", "min"], ["e", "max"], ["e", "min"]]


class OracleEngine:
    """The Engine calls solve() and solve_many() make for an LP with `iis`, served by the oracle and iis_reference."""

    def __init__(self):
        self.iis_calls = 0

    def solve_tableau(self, matrix, height, width, integers, sign, options):
        m = np.array(matrix, np.float64)
        pos = np.arange(width + height, dtype=np.int32)
        var = pos.copy()
        st, val, piv = O.simplex(m, width, height, pos, var, options.precision, options.max_pivots,
                                 options.check_cycles)
        return {"status": st, "result": val, "rhs": m.reshape(height, width)[:, 0].copy(), "pos": pos, "var": var,
                "stats": {}, "root_status": st, "root_value": val, "root_pivots": piv}

    def solve_ragged(self, tableaus, shapes, options, **kw):
        out = []
        for t, (h, w) in zip(tableaus, shapes):
            r = self.solve_tableau(t, h, w, [], 1.0, options)
            out.append({**r, "value": r["result"]})
        return out

    def iis(self, matrix, height, width, options):
        self.iis_calls += 1
        return iis_reference(matrix, height, width, options.precision, options.max_pivots, bool(options.check_cycles))


def test_worked_example_end_to_end_on_the_oracle():
    eng = OracleEngine()
    sol = S.solve(WORKED, {"iis": True}, engine=eng)
    assert sol["status"] == "infeasible" and sol["irreducibleInfeasibleSet"] == WORKED_IIS
    assert eng.iis_calls == 1
    feasible, unbounded = random_feasible(1), random_unbounded(1)
    for model, status in ((feasible, "optimal"), (unbounded, "unbounded")):
        sol = S.solve(model, {"iis": True}, engine=eng)
        assert sol["status"] == status and sol["irreducibleInfeasibleSet"] == []
        assert {k: v for k, v in sol.items() if k != "irreducibleInfeasibleSet"} == S.solve(model, engine=eng)
    assert eng.iis_calls == 1  # the search runs for infeasible models only
    many = S.solve_many([WORKED, feasible, unbounded], {"iis": True}, engine=eng)
    assert [s["irreducibleInfeasibleSet"] for s in many] == [WORKED_IIS, [], []]
    assert eng.iis_calls == 2


def test_iis_rejects_milp_before_any_engine():
    model = {**WORKED, "integers": ["x"]}
    created = []
    real = S.get_engine
    S.get_engine = lambda device=0: created.append(device)
    try:
        with pytest.raises(ValueError):
            S.solve(model, {"iis": True})
        with pytest.raises(ValueError):
            S.solve_many([model], {"iis": True})
    finally:
        S.get_engine = real
    assert created == []


# ------------------------------------------------------------------------------------------- input checks
class FakeLib:
    """Records the IIS entries' calls; writes status 1 and two rows."""

    def __init__(self):
        self.calls = []

    def yalps_create(self, device, out):
        out._obj.value = 0x1000
        return 0

    def yalps_multi_ctx(self, m, rank):
        return 0x1000

    def yalps_create_multi(self, devices, ndev, out):
        out._obj.value = 0x2000
        return 0

    def yalps_solve_row_subsets(self, ctx, n, h, w, base, keep, opt, status, value, pivots, cert, support):
        self.calls.append(("subsets", n, h, w, cert is None))
        return 0

    def yalps_iis(self, ctx, h, w, matrix, opt, status, rows, count, stats):
        self.calls.append(("iis", ctx.value, h, w))
        status._obj.value, count._obj.value = 1, 2
        C.memmove(rows.value, np.array([2, 5], np.int32).ctypes.data, 8)
        C.memmove(stats.value, np.array([3, 9, 40, 0, 0], np.int64).ctypes.data, 40)
        return 0

    def yalps_iis_sparse(self, ctx, h, w, nnz, cells, values, opt, status, rows, count, stats):
        self.calls.append(("iis_sparse", ctx.value, h, w, nnz))
        status._obj.value, count._obj.value = 1, 0
        C.memmove(stats.value, np.array([1, 1, 2, 1, 0], np.int64).ctypes.data, 40)
        return 0

    def __getattr__(self, name):
        if name.startswith("yalps_destroy"):
            return lambda *a: None
        raise AttributeError(name)


@pytest.fixture
def fake(monkeypatch):
    lib = FakeLib()
    monkeypatch.setattr(_ffi, "load", lambda: lib)
    return lib


def test_engine_iis_calls(fake):
    eng = yalps_b200.Engine(0)
    base = np.zeros(33 * 4)
    keep = np.full((3, 2), 0xffffffff, np.uint32)
    keep[:, 1] = 1  # row 32 is the last one
    out = eng.solve_row_subsets(base, keep, 33, 4, want_certificates=True)
    assert out["support"].shape == (3, 2) and out["certificate"].shape == (3, 37)
    eng.solve_row_subsets(base, keep, 33, 4)
    assert fake.calls == [("subsets", 3, 33, 4, False), ("subsets", 3, 33, 4, True)]
    r = eng.iis(np.zeros(24), 6, 4)
    assert r["rows"].tolist() == [2, 5] and (r["rounds"], r["lps"], r["pivots"], r["irreducible"]) == (3, 9, 40, True)
    r = yalps_b200.MultiEngine([0, 0]).iis_sparse([1, 2], [1.0, 2.0], 6, 4)
    assert r["rows"].tolist() == [] and r["irreducible"] is False  # an undecided row
    assert fake.calls[2:] == [("iis", 0x1000, 6, 4), ("iis_sparse", 0x1000, 6, 4, 2)]


@pytest.mark.parametrize("precision", [-1e-8, math.nan, -0.5])
def test_negative_or_nan_precision_is_refused(fake, precision):
    eng = yalps_b200.Engine(0)
    opt = make_options(precision=precision)
    with pytest.raises(ValueError):
        eng.solve_row_subsets(np.zeros(12), np.zeros((1, 1), np.uint32), 3, 4, opt)
    with pytest.raises(ValueError):
        eng.iis(np.zeros(12), 3, 4, opt)
    with pytest.raises(ValueError):
        eng.iis_sparse([], [], 3, 4, opt)
    with pytest.raises(ValueError):
        yalps_b200.MultiEngine([0]).iis(np.zeros(12), 3, 4, opt)
    assert fake.calls == []
    eng.iis(np.zeros(12), 3, 4, make_options(precision=0.0))
    assert len(fake.calls) == 1


def test_stray_mask_bits_are_refused(fake):
    eng = yalps_b200.Engine(0)
    with pytest.raises(ValueError):
        eng.solve_row_subsets(np.zeros(12), np.array([[0b1000]], np.uint32), 3, 4)  # row 3 of a 3-row tableau
    with pytest.raises(ValueError):
        eng.solve_row_subsets(np.zeros(33 * 4), np.array([[1, 2]], np.uint32), 33, 4)  # row 33
    with pytest.raises(ValueError):
        eng.solve_row_subsets(np.zeros(33 * 4), np.zeros(3, np.uint32), 33, 4)  # not whole masks
    assert fake.calls == []
    eng.solve_row_subsets(np.zeros(32 * 4), np.full((2, 1), 0xffffffff, np.uint32), 32, 4)  # 32 rows: no stray bits
    assert fake.calls == [("subsets", 2, 32, 4, True)]
