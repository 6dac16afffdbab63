"""Row subsets and the IIS search on the GPU (include/yalps_b200.h "irreducible infeasible subsets"): the subset entry bit
for bit against the oracle on T_S on every kernel path, a call of several pipeline chunks, Engine.iis / iis_sparse equal
to tests/test_iis.py's iis_reference round for round, and solve() / solve_many() with `iis`."""
import os

import numpy as np
import pytest

import yalps_b200
from conftest import same_bits
from oracle import lib as O
from test_gpu_sensitivity import PATHS
from test_iis import MODELS, WORKED, WORKED_IIS, iis_reference, random_feasible, subset_batch, subset_tableaus
from test_certificate import random_unbounded
from yalps_b200 import engine as E
from yalps_b200.sensitivity import certificate_from_tableau
from yalps_b200.tableau import SPARSE_OVER_BYTES, tableau_model

pytestmark = pytest.mark.gpu


@pytest.fixture
def tuned(engine):
    yield engine
    engine.set_tuning(E.PATH_AUTO, 0, 0)


def random_masks(rng, n, H, density):
    """n keep masks (uint32 (n, words)) and the row sets they keep; the first keeps every row."""
    words = (H + 31) // 32
    keep = np.zeros((n, words), np.uint32)
    sets = []
    for i in range(n):
        rows = list(range(1, H)) if i == 0 else [r for r in range(1, H) if rng.random() < density]
        for r in rows:
            keep[i, r >> 5] |= np.uint32(1 << (r & 31))
        if rng.random() < 0.5:
            keep[i, 0] |= np.uint32(1)  # bit 0 is ignored: row 0 always stays
        sets.append(rows)
    return keep, sets


def support_masks(supports, n, H):
    words = (H + 31) // 32
    out = np.zeros((n, words), np.uint32)
    for i, s in enumerate(supports):
        for r in s:
            out[i, r >> 5] |= np.uint32(1 << (r & 31))
    return out


def check_subsets(eng, base, H, W, keep, sets, opt=None, **kw):
    got = eng.solve_row_subsets(base, keep, H, W, opt, want_certificates=True)
    exp = subset_batch(base, H, W, sets, **kw)
    n = len(sets)
    assert np.array_equal(got["status"], exp["status"])
    assert np.array_equal(got["pivots"], exp["pivots"])
    assert same_bits(got["value"], exp["value"])
    cert = np.stack([certificate_from_tableau(exp["matrices"][i], W, H, exp["pos"][i], int(exp["status"][i]),
                                              float(exp["value"][i]), kw.get("precision", 1e-8)) for i in range(n)])
    assert same_bits(got["certificate"], cert)
    assert np.array_equal(got["support"], support_masks(exp["support"], n, H))
    return got


def infeasible_base(seed, m, nv):
    """A synthetic tableau whose first rows ask a.x >= nv^2 (a in [0, 1]): out of reach together with enough of the
    rows a.x <= b, so some subsets are infeasible and some are not."""
    neg = max(2, m // 8)
    M = O.generate_synthetic(seed, 1, m, nv, neg)[0].reshape(m + 1, nv + 1)
    M[1:neg + 1, 0] = -float(nv * nv)
    return M.reshape(-1)


@pytest.mark.parametrize("name,path,threads,rows", PATHS, ids=[p[0] for p in PATHS])
def test_subsets_bit_exact_on_every_path(tuned, name, path, threads, rows):
    m, nv = 16, 32
    n = 3 if path in (E.PATH_GRID, E.PATH_GRID_RESIDENT, E.PATH_CLUSTER) else 40
    base = infeasible_base(1, m, nv)
    keep, sets = random_masks(np.random.default_rng(7), n, m + 1, 0.6)
    tuned.set_tuning(path, threads, rows)
    got = check_subsets(tuned, base, m + 1, nv + 1, keep, sets)
    if n > 3:
        assert (got["status"] == 1).any() and (got["status"] != 1).any()


@pytest.mark.parametrize("m,nv,n", [(32, 64, 300), (150, 99, 60), (400, 299, 8)], ids=["33x65", "151x100", "401x300"])
def test_subsets_bit_exact_automatic(engine, m, nv, n):
    base = infeasible_base(2, m, nv)
    keep, sets = random_masks(np.random.default_rng(m), n, m + 1, 0.7)
    check_subsets(engine, base, m + 1, nv + 1, keep, sets)
    # checkCycles and an exhausted budget apply to every subset LP
    check_subsets(engine, base, m + 1, nv + 1, keep[:8], sets[:8], E.make_options(check_cycles=True, max_pivots=3),
                  check_cycles=True, max_pivots=3)


def test_subsets_spanning_several_chunks(engine):
    m, nv, n = 32, 64, 10000  # the replica rule cuts this into 8 pipeline chunks
    base = infeasible_base(3, m, nv)
    keep, sets = random_masks(np.random.default_rng(3), n, m + 1, 0.8)
    got = engine.solve_row_subsets(base, keep, m + 1, nv + 1)
    work = subset_tableaus(base, m + 1, nv + 1, sets)
    exp = O.simplex_batch(work, nv + 1, m + 1, nthreads=os.cpu_count() or 1)
    assert np.array_equal(got["status"], exp["status"]) and np.array_equal(got["pivots"], exp["pivots"])
    assert same_bits(got["value"], exp["value"])
    assert ((got["support"] != 0).any(axis=1) == (got["status"] == 1)).all()


def big_infeasible():
    """A model whose tableau (401 x 300) is above the 768 KB line, so solve() builds it as cell stores."""
    rng = np.random.default_rng(11)
    n = 299
    variables = {f"x{j}": {"cap": 1.0, "obj": float(rng.uniform(-1, 2))} for j in range(n)}
    cons = [("cap", {"max": 2.0})]
    for i in range(398):
        cols = rng.choice(n, 5, replace=False)
        for j in cols:
            variables[f"x{j}"][f"c{i}"] = float(np.round(rng.uniform(0.5, 5.0), 3))
        cons.append((f"c{i}", {"max": float(np.round(rng.uniform(5, 50), 3))}))
    for j in range(n):
        variables[f"x{j}"]["far"] = float(np.round(rng.uniform(0.5, 2.0), 3))
    cons.append(("far", {"min": 10.0}))
    return {"direction": "maximize", "objective": "obj", "constraints": cons, "variables": list(variables.items())}


def check_iis(got, exp):
    assert got["status"] == exp["status"] and got["rows"].tolist() == list(exp["rows"])
    assert (got["rounds"], got["lps"], got["pivots"], got["irreducible"]) == \
        (exp["rounds"], exp["lps"], exp["pivots"], exp["irreducible"])


@pytest.mark.parametrize("name,M,H,W", MODELS, ids=[m[0] for m in MODELS])
def test_iis_equals_reference(engine, name, M, H, W):
    exp = iis_reference(M, H, W)
    check_iis(engine.iis(M, H, W), exp)
    cells = np.flatnonzero(np.asarray(M).view(np.uint64)).astype(np.int32)  # -0.0 included
    check_iis(engine.iis_sparse(cells, np.asarray(M)[cells], H, W), exp)


def test_iis_above_the_sparse_line(engine):
    t = tableau_model(big_infeasible(), SPARSE_OVER_BYTES).tableau
    assert t.matrix is None and t.height * t.width * 8 > SPARSE_OVER_BYTES
    exp = iis_reference(t.dense(), t.height, t.width)
    assert exp["status"] == 1 and exp["irreducible"]
    check_iis(engine.iis_sparse(t.cells, t.values, t.height, t.width), exp)
    check_iis(engine.iis(t.matrix, t.height, t.width), exp)


def test_iis_feasible_unbounded_and_timeout(engine):
    for model, st in ((random_feasible(2), 0), (random_unbounded(2), 2)):
        t = tableau_model(model).tableau
        r = engine.iis(t.matrix, t.height, t.width)
        assert r["status"] == st and r["rows"].size == 0 and (r["rounds"], r["lps"]) == (1, 1) and not r["irreducible"]
    M, H, W = next(m[1:] for m in MODELS if m[0] == "KLEIN1")
    r = engine.iis(M, H, W, E.make_options(timeout_ms=0.0))
    assert r["status"] == 1 and r["rows"].tolist() == list(range(1, H)) and not r["irreducible"] and r["rounds"] == 1
    with pytest.raises(yalps_b200._ffi.YalpsError):  # the C entry checks precision too
        engine._check(engine._lib.yalps_iis(engine._ctx, H, W, M.ctypes.data_as(E.C.c_void_p),
                                            E.C.byref(E.make_options(precision=-1.0)), E.C.byref(E.C.c_int32()),
                                            np.empty(H, np.int32).ctypes.data_as(E.C.c_void_p),
                                            E.C.byref(E.C.c_int32()), None))


def test_solve_with_iis(engine):
    sol = yalps_b200.solve(WORKED, {"iis": True}, engine=engine)
    assert sol["status"] == "infeasible" and sol["irreducibleInfeasibleSet"] == WORKED_IIS
    both = yalps_b200.solve(WORKED, {"iis": True, "certificate": True, "ranging": True}, engine=engine)
    alone = yalps_b200.solve(WORKED, {"certificate": True, "ranging": True}, engine=engine)
    assert both == {**alone, "irreducibleInfeasibleSet": WORKED_IIS}
    big = big_infeasible()
    models = [WORKED, random_feasible(3), random_unbounded(3), big]
    many = yalps_b200.solve_many(models, {"iis": True}, engine=engine)
    singles = [yalps_b200.solve(m, {"iis": True}, engine=engine) for m in models]
    assert many == singles
    assert [s["status"] for s in many] == ["infeasible", "optimal", "unbounded", "infeasible"]
    assert [len(s["irreducibleInfeasibleSet"]) > 0 for s in many] == [True, False, False, True]
    with yalps_b200.MultiEngine([0, 0]) as multi:
        assert yalps_b200.solve(WORKED, {"iis": True}, engine=multi) == sol
        assert yalps_b200.solve(big, {"iis": True}, engine=multi) == singles[3]
        assert yalps_b200.solve_many(models, {"iis": True, "certificate": True}, engine=multi) == \
            yalps_b200.solve_many(models, {"iis": True, "certificate": True}, engine=engine)
