"""Warm starts on the GPU (include/yalps_b200.h "warm starts"): k_expand_warm bit for bit against warm_tableau, the warm
solve bit for bit against the oracle's loop on the warm tableau on every kernel path, the base solved inside the call
against a caller-supplied one, the sparse entry against the dense one, a call of several pipeline chunks (one GPU and two
ranks), and solve_variants against solve() and the CPU mapping."""
import numpy as np
import pytest

import yalps_b200
from conftest import load_netlib, same_bits, same_value
from oracle import lib as O
from oracle.model import result_is_optimal
from test_gpu_sensitivity import PATHS
from test_sensitivity import random_lp
from test_warm import FURNITURE, OPT, OracleWarmEngine, apply_variant
from yalps_b200 import engine as E
from yalps_b200.sensitivity import certificate_from_tableau, ranges_from_tableau, reduced_from_tableau
from yalps_b200.tableau import SPARSE_OVER_BYTES
from yalps_b200.warm import warm_tableau

pytestmark = pytest.mark.gpu


@pytest.fixture
def tuned(engine):
    yield engine
    engine.set_tuning(E.PATH_AUTO, 0, 0)


def synthetic_base(m, nv, neg, first, **kw):
    """(M0, F, pos, var, status, value, pivots) of one synthetic LP and the oracle's cold solve of it."""
    M0 = O.generate_synthetic(first, 1, m, nv, neg)[0].copy()
    H, W = m + 1, nv + 1
    F = M0.copy()
    pos, var = np.arange(W + H, dtype=np.int32), np.arange(W + H, dtype=np.int32)
    st, val, piv = O.simplex(F, W, H, pos, var, **kw)
    return M0, F, pos, var, st, val, piv


def variants(M0, H, W, n, kind, seed, eps=0.2):
    """n variants: rhs (n, H) and/or obj (n, W), a random share of each changed by up to +-eps relative (the first
    variant of each kind unchanged)."""
    rng = np.random.default_rng(seed)
    m0 = M0.reshape(H, W)
    rhs = obj = None
    if kind in ("rhs", "both"):
        rhs = np.tile(m0[:, 0], (n, 1))
        f = 1 + eps * rng.uniform(-1, 1, (n, H)) * (rng.random((n, H)) < 0.5)
        f[0] = 1.0
        rhs = np.where(f != 1.0, rhs * f + (rng.random((n, H)) < 0.05) * rng.uniform(-1, 1, (n, H)), rhs)
    if kind in ("obj", "both"):
        obj = np.tile(m0[0], (n, 1))
        f = 1 + eps * rng.uniform(-1, 1, (n, W)) * (rng.random((n, W)) < 0.5)
        f[0] = 1.0
        obj = np.where(f != 1.0, obj * f + (rng.random((n, W)) < 0.1) * rng.uniform(-1, 1, (n, W)), obj)
    return rhs, obj


def oracle_warm(M0, F, pos, var, H, W, rhs, obj, precision=1e-8, max_pivots=8192, check_cycles=False):
    """The reference loop on every warm tableau, with the reduced costs, ranges and certificates of its finals."""
    n = len(rhs if rhs is not None else obj)
    mats = np.stack([warm_tableau(M0, F, pos, H, W, None if rhs is None else rhs[i], None if obj is None else obj[i])
                     for i in range(n)])
    start = mats.copy()
    res = {k: [] for k in ("status", "value", "pivots", "pos", "var", "reduced", "range_lo", "range_hi",
                           "certificate")}
    for i in range(n):
        p, v = pos.copy(), var.copy()
        st, val, piv = O.simplex(mats[i], W, H, p, v, precision, max_pivots, check_cycles)
        lo, hi = ranges_from_tableau(mats[i], W, H, p, precision, optimal=st == 0)
        for k, x in (("status", st), ("value", val), ("pivots", piv), ("pos", p), ("var", v),
                     ("reduced", reduced_from_tableau(mats[i], W, H, p)), ("range_lo", lo), ("range_hi", hi),
                     ("certificate", certificate_from_tableau(mats[i], W, H, p, st, val, precision))):
            res[k].append(x)
    out = {k: np.asarray(x) for k, x in res.items()}
    out["matrices"] = mats
    out["rhs"] = mats.reshape(n, H, W)[:, :, 0].copy()
    out["start"] = start
    return out


INTS = ("status", "pivots", "pos", "var")
FLOATS = ("value", "rhs", "matrices", "reduced", "range_lo", "range_hi", "certificate")


def assert_same(got, exp, keys_i=INTS, keys_f=FLOATS, where=""):
    for k in keys_i:
        assert np.array_equal(got[k], exp[k]), (where, k)
    for k in keys_f:
        assert same_bits(got[k], exp[k]), (where, k)


WANT = dict(want_matrices=True, want_duals=True, want_ranges=True, want_certificates=True)

# (m, nv, neg): K1t small and at its edge, K1/K1s, K2/K2s and a KC-size base
SHAPES = [(8, 16, 2), (32, 64, 6), (50, 40, 10), (90, 120, 20), (200, 260, 30), (600, 800, 60)]


@pytest.mark.parametrize("kind", ["rhs", "obj", "both"])
@pytest.mark.parametrize("m,nv,neg", SHAPES, ids=[f"{s[0] + 1}x{s[1] + 1}" for s in SHAPES])
def test_expand_kernel_is_bit_exact(engine, m, nv, neg, kind):
    """maxPivots 0: the returned tableaus are the start tableaus k_expand_warm built."""
    H, W = m + 1, nv + 1
    M0, F, pos, var, *_ = synthetic_base(m, nv, neg, 7000 + m)
    rhs, obj = variants(M0, H, W, 12 if m < 500 else 4, kind, m)
    got = engine.solve_warm(M0, H, W, rhs, obj, E.make_options(max_pivots=0), final=(F, pos, var), want_matrices=True)
    exp = np.stack([warm_tableau(M0, F, pos, H, W, None if rhs is None else rhs[i], None if obj is None else obj[i])
                    for i in range(len(got["status"]))])
    assert same_bits(got["matrices"], exp)
    assert np.array_equal(got["var"], np.tile(var, (len(exp), 1)))


PATH_SHAPES = {"TMEM": (32, 64, 6, 64), "SMEM": (32, 64, 6, 48), "GMEM": (60, 80, 9, 24), "SPLIT_SMEM": (90, 120, 20, 12),
               "SPLIT_GMEM": (90, 120, 20, 12), "CLUSTER": (200, 260, 30, 3), "GRID_RESIDENT": (70, 300, 10, 2),
               "GRID": (70, 300, 10, 2), "AUTO": (32, 64, 8, 500)}


@pytest.mark.parametrize("precision", [1e-8, 1e-6])
@pytest.mark.parametrize("check_cycles", [False, True])
@pytest.mark.parametrize("name,path,threads,rows", PATHS, ids=[p[0] for p in PATHS])
def test_warm_solve_is_bit_exact_on_every_path(tuned, name, path, threads, rows, check_cycles, precision):
    m, nv, neg, n = PATH_SHAPES[name]
    H, W = m + 1, nv + 1
    kw = dict(precision=precision, check_cycles=check_cycles)
    M0, F, pos, var, *_ = synthetic_base(m, nv, neg, 8000 + m, **kw)
    rhs, obj = variants(M0, H, W, n, "both", n + m)
    rhs[: n // 3] = M0.reshape(H, W)[:, 0]   # a third objective-only,
    obj[n // 3: 2 * n // 3] = M0[:W]         # a third RHS-only
    exp = oracle_warm(M0, F, pos, var, H, W, rhs, obj, **kw)
    tuned.set_tuning(path, threads, rows)
    got = tuned.solve_warm(M0, H, W, rhs, obj, E.make_options(**kw), final=(F, pos, var), **WANT)
    assert_same(got, exp, where=name)


@pytest.mark.parametrize("m,nv,neg,n", [(20, 30, 5, 7), (32, 64, 8, 300), (90, 120, 20, 40)])
def test_automatic_shapes_and_the_base_solved_inside(engine, m, nv, neg, n):
    """At automatic shapes: the base solved inside the call gives the same bits as the oracle's final given as
    `final`, and out["base"] reports the oracle's cold solve."""
    H, W = m + 1, nv + 1
    M0, F, pos, var, st, val, piv = synthetic_base(m, nv, neg, 8500 + m)
    rhs, obj = variants(M0, H, W, n, "both", m)
    exp = oracle_warm(M0, F, pos, var, H, W, rhs, obj)
    inside = engine.solve_warm(M0, H, W, rhs, obj, **WANT)
    given = engine.solve_warm(M0, H, W, rhs, obj, final=(F, pos, var), **WANT)
    assert inside["base"]["status"] == st and inside["base"]["pivots"] == piv
    assert same_value(inside["base"]["value"], val) and given["base"] is None
    assert_same(inside, exp)
    assert_same(given, exp)


def test_sparse_entry_equals_dense():
    """A base above SPARSE_OVER_BYTES given as (cell, value) stores gives the dense entry's bits."""
    m, nv = 300, 400
    assert (m + 1) * (nv + 1) * 8 > SPARSE_OVER_BYTES
    H, W = m + 1, nv + 1
    M0, F, pos, var, *_ = synthetic_base(m, nv, 30, 9001)
    rhs, obj = variants(M0, H, W, 6, "both", 3)
    cells = np.flatnonzero(M0).astype(np.int32)
    with yalps_b200.Engine(0) as eng:
        dense = eng.solve_warm(M0, H, W, rhs, obj, **WANT)
        sparse = eng.solve_warm_sparse(cells, M0[cells], H, W, rhs, obj, **WANT)
        given = eng.solve_warm_sparse(cells, M0[cells], H, W, rhs, obj, final=(F, pos, var), **WANT)
    assert_same(sparse, dense)
    assert_same(given, dense)
    assert sparse["base"] == dense["base"]


def test_warm_across_pipeline_chunks(engine):
    """10,000 variants of AFIRO run in 8 pipeline chunks: the LPs on each side of every chunk boundary equal the oracle,
    and two ranks on one GPU give the same bits."""
    g = load_netlib().get("AFIRO")
    H, W = g["height"], g["width"]
    M0 = np.ascontiguousarray(g["matrix"], np.float64)
    F, pos, var = M0.copy(), np.arange(W + H, dtype=np.int32), np.arange(W + H, dtype=np.int32)
    O.simplex(F, W, H, pos, var)
    n, per_chunk = 10000, (10000 + 7) // 8
    rhs, obj = variants(M0, H, W, n, "both", 17, eps=0.05)
    got = engine.solve_warm(M0, H, W, rhs, obj, want_duals=True, want_certificates=True)
    edges = np.array([b + d for b in range(per_chunk, n, per_chunk) for d in (-1, 0)] + [0, n - 1])
    exp = oracle_warm(M0, F, pos, var, H, W, rhs[edges], obj[edges])
    keys_f = ("value", "rhs", "reduced", "certificate")
    assert_same({k: got[k][edges] for k in INTS + keys_f}, exp, keys_f=keys_f)
    with yalps_b200.MultiEngine([0, 0]) as me:
        many = me.solve_warm(M0, H, W, rhs, obj, want_duals=True, want_certificates=True)
    assert_same(many, got, keys_f=keys_f)
    assert many["base"] == got["base"]
    print(f"\nAFIRO warm variants: {got['pivots'].sum(axis=0).tolist()} pivots (phase 1, phase 2) for {n} LPs")


def model_variants(model, rng, k):
    keys = [key for key, _ in (model["constraints"].items() if isinstance(model["constraints"], dict)
                               else model["constraints"])]
    out = []
    for i in range(k):
        v = {}
        key = keys[int(rng.integers(len(keys)))]
        con = dict(model["constraints"])[key] if not isinstance(model["constraints"], dict) else model["constraints"][key]
        if i % 3 != 1:
            v["constraints"] = {key: {b: round(float(x) * float(rng.uniform(0.7, 1.3)), 3) for b, x in con.items()}}
        if i % 3 != 0:
            names = [n for n, _ in (model["variables"].items() if isinstance(model["variables"], dict)
                                    else model["variables"])]
            v["objective"] = {names[int(rng.integers(len(names)))]: round(float(rng.uniform(-2, 4)), 3)}
        out.append(v)
    return out


@pytest.mark.parametrize("opts", [{}, {"sensitivity": True}, {"ranging": True, "certificate": True}])
def test_solve_variants(engine, opts):
    """solve_variants equals the CPU mapping of the oracle's loop on the warm tableau exactly, and solve() of each
    changed model in status and (within the validator's tolerance) result."""
    rng = np.random.default_rng(5)
    cases = [(FURNITURE, [{"constraints": {"wood": {"max": v}}} for v in (250, 300, 350)]
              + [{"objective": {"dresser": 2000}}])]
    cases += [(random_lp(s), None) for s in range(6)]
    for model, vs in cases:
        vs = vs or model_variants(model, rng, 6)
        got = yalps_b200.solve_variants(model, vs, opts, engine=engine)
        assert got == yalps_b200.solve_variants(model, vs, opts, engine=OracleWarmEngine())
        for v, sol in zip(vs, got):
            cold = yalps_b200.solve(apply_variant(model, v), opts, engine=engine)
            assert sol["status"] == cold["status"] and set(sol) == set(cold), v
            if sol["status"] == "optimal":
                assert result_is_optimal(sol["result"], cold["result"], OPT), (v, sol["result"], cold["result"])


def test_errors_reach_the_caller(engine):
    M0, F, pos, var, *_ = synthetic_base(4, 5, 1, 1)
    bad = var.copy()
    bad[0], bad[1] = bad[1], bad[0]
    with pytest.raises(E.YalpsError, match="inverse"):
        engine.solve_warm(M0, 5, 6, M0.reshape(5, 6)[:, 0][None], final=(F, pos, bad))
