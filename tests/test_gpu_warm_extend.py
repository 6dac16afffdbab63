"""Warm starts that add constraints and variables, on the GPU (include/yalps_b200.h, yalps_solve_warm_extend):
k_expand_warm's extended start tableau bit for bit against warm_tableau (also where the added shape crosses a kernel's
shape class), the solve bit for bit against the oracle's loop on that tableau on every kernel path, the sparse entry
against the dense one, a call of several pipeline chunks on one GPU and on two ranks, solve_variants against solve() of
each changed model, and the C entry's refusals."""
import ctypes as C

import numpy as np
import pytest

import yalps_b200
from conftest import load_netlib, same_bits
from oracle import lib as O
from oracle.model import result_is_optimal
from test_gpu_sensitivity import PATHS
from test_gpu_warm import INTS, WANT, assert_same, synthetic_base, variants
from test_sensitivity import random_lp
from test_warm import OPT
from test_warm_extend import FURNITURE, MODEL_VARIANTS, OracleExtendEngine, apply_additions, random_additions
from yalps_b200 import engine as E
from yalps_b200.sensitivity import certificate_from_tableau, ranges_from_tableau, reduced_from_tableau
from yalps_b200.tableau import SPARSE_OVER_BYTES
from yalps_b200.warm import extended_basis, warm_tableau

pytestmark = pytest.mark.gpu


@pytest.fixture
def tuned(engine):
    yield engine
    engine.set_tuning(E.PATH_AUTO, 0, 0)


def additions(M0, F, pos, H, W, n, K, M, seed):
    """(n, K, W+M) rows and (n, M, H) columns: per variant random cuts of the base vertex and attractive columns, with
    every third variant adding fewer (zero rows and columns, as solve_variants pads a batch)."""
    rng = np.random.default_rng(seed)
    rows, cols = np.zeros((n, K, W + M)), np.zeros((n, M, H))
    for i in range(n):
        k, m = (K, M) if i % 3 else (K // 2, M // 2)
        r, c = random_additions(rng, M0, F, pos, H, W, k, m)
        if k:
            rows[i, :k, :W + m] = r
        if m:
            cols[i, :m] = c
    return rows, cols


def oracle_ext(M0, F, pos, var, H, W, rhs, obj, rows, cols, precision=1e-8, max_pivots=8192, check_cycles=False):
    """The reference loop on every extended start tableau, with the reduced costs, ranges and certificates."""
    n, K, M = rows.shape[0], rows.shape[1], cols.shape[1]
    Hx, Wx = H + K, W + M
    mats = np.stack([warm_tableau(M0, F, pos, H, W, None if rhs is None else rhs[i], None if obj is None else obj[i],
                                  rows[i], cols[i]) for i in range(n)])
    start = mats.copy()
    p0, v0 = extended_basis(pos, var, H, W, K, M)
    res = {k: [] for k in ("status", "value", "pivots", "pos", "var", "reduced", "range_lo", "range_hi",
                           "certificate")}
    for i in range(n):
        p, v = p0.copy(), v0.copy()
        st, val, piv = O.simplex(mats[i], Wx, Hx, p, v, precision, max_pivots, check_cycles)
        lo, hi = ranges_from_tableau(mats[i], Wx, Hx, p, precision, optimal=st == 0)
        for k, x in (("status", st), ("value", val), ("pivots", piv), ("pos", p), ("var", v),
                     ("reduced", reduced_from_tableau(mats[i], Wx, Hx, p)), ("range_lo", lo), ("range_hi", hi),
                     ("certificate", certificate_from_tableau(mats[i], Wx, Hx, p, st, val, precision))):
            res[k].append(x)
    out = {k: np.asarray(x) for k, x in res.items()}
    out["matrices"] = mats
    out["rhs"] = mats.reshape(n, Hx, Wx)[:, :, 0].copy()
    out["start"], out["var0"] = start, v0
    return out


# base (m, nv, neg) + (K, M): K1t's 33x65 reached from below, 33x64 + 2 columns (leaves K1t), a row-split shape, and
# one base without a change of column 0 or row 0
EXPAND = [(30, 62, 5, 2, 2), (32, 63, 6, 0, 2), (31, 64, 6, 3, 0), (80, 110, 15, 10, 10), (8, 16, 2, 1, 1)]


@pytest.mark.parametrize("kind", ["none", "both"])
@pytest.mark.parametrize("m,nv,neg,K,M", EXPAND, ids=[f"{s[0] + 1}x{s[1] + 1}+{s[3]}x{s[4]}" for s in EXPAND])
def test_expand_kernel_is_bit_exact(engine, m, nv, neg, K, M, kind):
    """maxPivots 0: the returned tableaus and var are the extended start tableaus and basis, bit for bit."""
    H, W = m + 1, nv + 1
    M0, F, pos, var, *_ = synthetic_base(m, nv, neg, 7100 + m)
    n = 10
    rhs, obj = variants(M0, H, W, n, "both", m) if kind == "both" else (None, None)
    rows, cols = additions(M0, F, pos, H, W, n, K, M, m)
    got = engine.solve_warm(M0, H, W, rhs, obj, E.make_options(max_pivots=0), final=(F, pos, var), want_matrices=True,
                            add_rows=rows, add_cols=cols)
    exp = oracle_ext(M0, F, pos, var, H, W, rhs, obj, rows, cols, max_pivots=0)
    assert same_bits(got["matrices"], exp["start"])
    assert np.array_equal(got["var"], np.tile(exp["var0"], (n, 1)))


# base shapes whose extended shape (K = 2 rows, M = 2 columns added) is test_gpu_warm's shape for the path
PATH_SHAPES = {"TMEM": (30, 62, 6, 64), "SMEM": (30, 62, 6, 48), "GMEM": (58, 78, 9, 24),
               "SPLIT_SMEM": (88, 118, 20, 12), "SPLIT_GMEM": (88, 118, 20, 12), "CLUSTER": (198, 258, 30, 3),
               "GRID_RESIDENT": (68, 298, 10, 2), "GRID": (68, 298, 10, 2), "AUTO": (30, 62, 8, 500)}


@pytest.mark.parametrize("check_cycles", [False, True])
@pytest.mark.parametrize("name,path,threads,rows", PATHS, ids=[p[0] for p in PATHS])
def test_extend_solve_is_bit_exact_on_every_path(tuned, name, path, threads, rows, check_cycles):
    m, nv, neg, n = PATH_SHAPES[name]
    H, W = m + 1, nv + 1
    kw = dict(check_cycles=check_cycles)
    M0, F, pos, var, *_ = synthetic_base(m, nv, neg, 8100 + m, **kw)
    rhs, obj = variants(M0, H, W, n, "both", n + m, eps=0.05)
    add_r, add_c = additions(M0, F, pos, H, W, n, 2, 2, n + m)
    exp = oracle_ext(M0, F, pos, var, H, W, rhs, obj, add_r, add_c, **kw)
    tuned.set_tuning(path, threads, rows)
    got = tuned.solve_warm(M0, H, W, rhs, obj, E.make_options(**kw), final=(F, pos, var), add_rows=add_r,
                           add_cols=add_c, **WANT)
    assert_same(got, exp, where=name)
    # the base solved inside the call gives the same bits
    if name == "AUTO":
        inside = tuned.solve_warm(M0, H, W, rhs, obj, E.make_options(**kw), add_rows=add_r, add_cols=add_c, **WANT)
        assert_same(inside, exp)


def test_sparse_entry_equals_dense():
    m, nv = 300, 400
    assert (m + 1) * (nv + 1) * 8 > SPARSE_OVER_BYTES
    H, W = m + 1, nv + 1
    M0, F, pos, var, *_ = synthetic_base(m, nv, 30, 9101)
    rhs, obj = variants(M0, H, W, 6, "both", 3)
    add_r, add_c = additions(M0, F, pos, H, W, 6, 3, 2, 5)
    cells = np.flatnonzero(M0).astype(np.int32)
    with yalps_b200.Engine(0) as eng:
        dense = eng.solve_warm(M0, H, W, rhs, obj, add_rows=add_r, add_cols=add_c, **WANT)
        sparse = eng.solve_warm_sparse(cells, M0[cells], H, W, rhs, obj, add_rows=add_r, add_cols=add_c, **WANT)
        given = eng.solve_warm_sparse(cells, M0[cells], H, W, rhs, obj, final=(F, pos, var), add_rows=add_r,
                                      add_cols=add_c, **WANT)
    assert_same(sparse, dense)
    assert_same(given, dense)
    assert sparse["base"] == dense["base"]


def test_extend_across_pipeline_chunks(engine):
    """10,000 AFIRO variants with 2 added rows and 1 added column run in 8 pipeline chunks: the LPs on each side of
    every chunk boundary equal the oracle (slice offsets of rhs, obj, rows and columns), and two ranks give the same
    bits."""
    g = load_netlib().get("AFIRO")
    H, W = g["height"], g["width"]
    M0 = np.ascontiguousarray(g["matrix"], np.float64)
    F, pos, var = M0.copy(), np.arange(W + H, dtype=np.int32), np.arange(W + H, dtype=np.int32)
    O.simplex(F, W, H, pos, var)
    n, per_chunk = 10000, (10000 + 7) // 8
    rhs, obj = variants(M0, H, W, n, "both", 19, eps=0.05)
    add_r, add_c = additions(M0, F, pos, H, W, n, 2, 1, 23)
    want = dict(want_duals=True, want_certificates=True, want_ranges=True,
                pairs=np.tile(np.full(H + 2, -1, np.int32), (n, 1)))
    got = engine.solve_warm(M0, H, W, rhs, obj, add_rows=add_r, add_cols=add_c, **want)
    edges = np.array([b + d for b in range(per_chunk, n, per_chunk) for d in (-1, 0)] + [0, n - 1])
    exp = oracle_ext(M0, F, pos, var, H, W, rhs[edges], obj[edges], add_r[edges], add_c[edges])
    keys_f = ("value", "rhs", "reduced", "certificate", "range_lo", "range_hi")
    assert_same({k: got[k][edges] for k in INTS + keys_f}, exp, keys_f=keys_f)
    with yalps_b200.MultiEngine([0, 0]) as me:
        many = me.solve_warm(M0, H, W, rhs, obj, add_rows=add_r, add_cols=add_c, **want)
    assert_same(many, got, keys_f=keys_f)
    assert many["base"] == got["base"]
    print(f"\nAFIRO extended variants: {got['pivots'].sum(axis=0).tolist()} pivots (phase 1, phase 2) for {n} LPs")


def test_solve_variants(engine):
    """solve_variants with addConstraints / addVariables equals the oracle's loop on the extended warm tableau exactly,
    and solve() of each changed model in status and (within the validator's tolerance) result; the ranging and
    certificate fields name the added keys and variables."""
    opts = {"ranging": True, "certificate": True}
    cases = [(FURNITURE, MODEL_VARIANTS)]
    rng = np.random.default_rng(11)
    for s in range(6):
        model = random_lp(s)
        names = [n for n, _ in model["variables"]] if not isinstance(model["variables"], dict) else list(model["variables"])
        vs = []
        for i in range(6):
            a, b = (int(t) for t in rng.choice(len(names), 2, replace=False))
            v = {}
            if i % 3 != 2:
                v["addConstraints"] = {"cut": {"max": round(float(rng.uniform(0.5, 3.0)), 3),
                                               "coefficients": {names[a]: 1, names[b]: 1}}}
            if i % 3 != 1:
                cs = dict(dict(model["variables"])[names[a]])
                cs[model["objective"]] = float(cs.get(model["objective"], 0.0)) + 1.0
                if "addConstraints" in v:
                    cs["cut"] = 1.0
                v["addVariables"] = {"extra": cs}
            vs.append(v)
        cases.append((model, vs))
    for model, vs in cases:
        got = yalps_b200.solve_variants(model, vs, opts, engine=engine)
        assert got == yalps_b200.solve_variants(model, vs, opts, engine=OracleExtendEngine())
        for v, sol in zip(vs, got):
            cold = yalps_b200.solve(apply_additions(model, v), opts, engine=engine)
            assert sol["status"] == cold["status"] and set(sol) == set(cold), v
            if sol["status"] == "optimal":
                assert result_is_optimal(sol["result"], cold["result"], OPT), (v, sol["result"], cold["result"])
                assert [k for k, *_ in sol["rhsRanges"]] == [k for k, *_ in cold["rhsRanges"]]
                assert [k for k, *_ in sol["costRanges"]] == [k for k, *_ in cold["costRanges"]]
            elif sol["status"] == "infeasible":
                assert [k for k, _ in sol["infeasibilityCertificate"]] == [k for k, _ in cold["infeasibilityCertificate"]]


def test_bad_additions_reach_the_caller(engine):
    M0, F, pos, var, *_ = synthetic_base(4, 5, 1, 1)
    H, W = 5, 6
    with pytest.raises(ValueError):
        engine.solve_warm(M0, H, W, add_rows=np.zeros((2, 1, W + 1)))
    lib, opt = engine._lib, E.make_options()
    st = np.zeros(2, np.int32)
    rows = np.zeros(2 * (W + 1))
    base = M0.ctypes.data_as(C.c_void_p)

    def call(K, M, rows_in, cols_in):
        return lib.yalps_solve_warm_extend(engine._ctx, 2, H, W, K, M, base, None, None, None, None, None, rows_in,
                                           cols_in, C.byref(opt), None, None, None, st.ctypes.data_as(C.c_void_p),
                                           None, None, None, None, None, None, None, None, None, None, None)

    r = rows.ctypes.data_as(C.c_void_p)
    assert call(-1, 0, r, None) == -2
    assert call(0, -1, None, r) == -2
    assert call(1, 0, None, None) == -2
    assert call(0, 1, None, None) == -2
    assert call(1 << 20, 1 << 12, r, r) == -3
