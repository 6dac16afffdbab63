"""Certificates on the GPU (k_certificate, include/yalps_b200.h "certificates"): bit for bit
yalps_b200.sensitivity.certificate_from_tableau of the oracle's final tableau on every kernel path and entry point,
and solve() / solve_many() with `certificate` equal to the CPU mapping of tests/test_certificate.py."""
import numpy as np
import pytest

import yalps_b200
from conftest import load_netlib, same_bits
from oracle import lib as O
from test_certificate import GOLDEN, oracle_certificate, synthetic
from test_gpu_sensitivity import PATHS, oracle_batch, special_batch
from yalps_b200 import engine as E
from yalps_b200.sensitivity import certificate_from_tableau

pytestmark = pytest.mark.gpu

NL = load_netlib()


def expected(mats, status, value, pos, H, W, precision=1e-8):
    mats = np.asarray(mats).reshape(-1, H * W)
    pos = np.asarray(pos).reshape(-1, W + H)
    return np.stack([certificate_from_tableau(mats[i], W, H, pos[i], int(status[i]), float(value[i]), precision)
                     for i in range(mats.shape[0])])


def mixed_batch(n, m, nv, seed=0):
    """special_batch with a real share of infeasible and unbounded LPs: every fourth LP gets a row that no x >= 0 can
    meet (and the most negative RHS), every fourth a column that raises the objective and that no row bounds."""
    mats = special_batch(n, m, nv, seed)
    rng = np.random.default_rng(100 + seed)
    H, W = m + 1, nv + 1
    M = mats.reshape(n, H, W)
    for i in range(n):
        if i % 4 == 1:
            r = int(rng.integers(1, H))
            M[i, r, 1:] = np.abs(M[i, r, 1:])
            M[i, r, 0] = -abs(M[i, r, 0]) - rng.uniform(1, 100)
        elif i % 4 == 2:
            c = int(rng.integers(1, W))
            M[i, 1:, c] = -np.abs(M[i, 1:, c])
            M[i, 0, c] = abs(M[i, 0, c]) + rng.uniform(1, 10)
    return mats


@pytest.fixture
def tuned(engine):
    yield engine
    engine.set_tuning(E.PATH_AUTO, 0, 0)


# ------------------------------------------------------------------------------------------- device entry
@pytest.mark.parametrize("H,W,n", [(2, 2, 5), (5, 9, 40), (33, 65, 300), (200, 120, 20), (257, 129, 6), (600, 300, 3),
                                   (1000, 1500, 2), (4097, 8193, 1)])
def test_device_entry_synthetic(engine, H, W, n):
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(H * 7 + W)
    mats, poss, status, value = [], [], [], []
    for i in range(n):
        m, p, st, v = synthetic(rng, H, W)
        mats.append(m)
        poss.append(p)
        status.append([1, 2, st][i % 3])
        value.append(v)
    mats, poss = np.stack(mats), np.stack(poss)
    status, value = np.asarray(status, np.int32), np.asarray(value, np.float64)
    dev = torch.device("cuda:0")
    d_m, d_pos = torch.from_numpy(mats).to(dev), torch.from_numpy(poss).to(dev)
    d_st, d_val = torch.from_numpy(status).to(dev), torch.from_numpy(value).to(dev)
    d_cert = torch.full((n, W + H), 7.0, dtype=torch.float64, device=dev)
    engine.certificate_device(n, H, W, d_m.data_ptr(), d_pos.data_ptr(), d_st.data_ptr(), d_val.data_ptr(),
                              d_cert.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert same_bits(d_cert.cpu().numpy(), expected(mats, status, value, poss, H, W))


# ------------------------------------------------------------------------------------------- host entries
@pytest.mark.parametrize("name,path,threads,rows", PATHS, ids=[p[0] for p in PATHS])
@pytest.mark.parametrize("gen", ["special", "mixed"])
def test_paths_bit_exact(tuned, name, path, threads, rows, gen):
    n = 4 if path in (E.PATH_GRID, E.PATH_GRID_RESIDENT, E.PATH_CLUSTER) else 40
    m, nv = 16, 32
    H, W = m + 1, nv + 1
    mats = special_batch(n, m, nv) if gen == "special" else mixed_batch(n, m, nv)
    tuned.set_tuning(path, threads, rows)
    opt = E.make_options()
    exp = oracle_batch(mats, H, W)
    cert = expected(exp["matrices"], exp["status"], exp["value"], exp["pos"], H, W)
    for extra in ({}, {"want_duals": True, "want_ranges": True}):
        got = tuned.solve_batch(mats, H, W, opt, want_matrices=True, want_certificates=True, **extra)
        plain = tuned.solve_batch(mats, H, W, opt, want_matrices=True, **extra)
        assert same_bits(got["certificate"], cert)
        # requesting certificates changes no other output bit
        for k in ("status", "pivots", "pos", "var"):
            assert np.array_equal(got[k], plain[k]), k
        for k in ("value", "rhs", "matrices") + (("reduced", "range_lo", "range_hi") if extra else ()):
            assert same_bits(got[k], plain[k]), k


def test_statuses_covered(engine):
    mats = mixed_batch(40, 16, 32)
    got = engine.solve_batch(mats, 17, 33, want_certificates=True)
    st = got["status"]
    assert {0, 1, 2} <= set(st.tolist())
    assert np.isnan(got["certificate"][(st != 1) & (st != 2)]).all()
    assert not np.isnan(got["certificate"][(st == 1) | (st == 2)]).any()


def test_pipelined_chunks(engine):
    m, nv, n = 32, 64, 4500  # 78 MB of tableaus: more than one 64 MiB pipeline chunk
    H, W = m + 1, nv + 1
    mats = mixed_batch(n, m, nv, seed=11)
    exp = oracle_batch(mats, H, W)
    cert = expected(exp["matrices"], exp["status"], exp["value"], exp["pos"], H, W)
    for path in (E.PATH_GMEM, E.PATH_AUTO):
        engine.set_tuning(path, 64 if path == E.PATH_GMEM else 0, 0)
        try:
            got = engine.solve_batch(mats, H, W, want_certificates=True)
        finally:
            engine.set_tuning(E.PATH_AUTO, 0, 0)
        assert same_bits(got["certificate"], cert)


def test_zero_copy_single_lp(engine):
    mats = mixed_batch(4, 16, 32, seed=3)
    for i in range(4):
        got = engine.solve_batch(mats[i], 17, 33, want_certificates=True)
        exp = oracle_batch(mats[i], 17, 33)
        assert same_bits(got["certificate"], expected(exp["matrices"], exp["status"], exp["value"], exp["pos"], 17, 33))


@pytest.mark.parametrize("small", [True, False], ids=["zero_copy", "chunked"])
def test_ragged_mixed_routes(engine, small):
    shapes = [(9, 17), (33, 65), (5, 9)] * 3 if small else [(9, 17), (33, 65), (17, 33), (61, 121), (129, 257),
                                                                (300, 500), (5, 9)] * 3
    tabs = [mixed_batch(4, h - 1, w - 1, seed=i)[i % 4] for i, (h, w) in enumerate(shapes)]
    got = engine.solve_ragged(tabs, shapes, want_certificates=True, want_duals=True)
    plain = engine.solve_ragged(tabs, shapes, want_duals=True)
    seen = set()
    for i, (h, w) in enumerate(shapes):
        exp = oracle_batch(tabs[i], h, w)
        seen.add(int(exp["status"][0]))
        assert same_bits(got[i]["certificate"], expected(exp["matrices"], exp["status"], exp["value"], exp["pos"], h, w)[0])
        assert np.array_equal(got[i]["pos"], plain[i]["pos"]) and same_bits(got[i]["reduced"], plain[i]["reduced"])
    assert {1, 2} <= seen


def test_sparse_entry_above_zero_copy(engine):
    m, nv = 300, 400  # 965 KB of tableau: above the 768 KB zero-copy limit
    H, W = m + 1, nv + 1
    seen = set()
    for seed in range(4):
        dense = mixed_batch(4, m, nv, seed=20 + seed)[1 + seed % 2].copy()
        M = dense.reshape(H, W)
        rng = np.random.default_rng(seed)
        M[1:, 1:] *= rng.random((m, nv)) < 0.1  # sparse
        nz = np.flatnonzero(dense.view(np.uint64) != 0)
        sp = engine.solve_lp_sparse(nz.astype(np.int32), dense[nz], H, W, want_certificates=True)
        exp = oracle_batch(dense, H, W)
        assert sp["status"] == exp["status"][0]
        seen.add(sp["status"])
        assert same_bits(sp["certificate"], expected(exp["matrices"], exp["status"], exp["value"], exp["pos"], H, W)[0])
    assert {1, 2} <= seen


def test_multi_equals_single(engine):
    multi = yalps_b200.MultiEngine([0, 0])
    try:
        mats = mixed_batch(50, 16, 32, seed=7)
        a = multi.solve_batch(mats, 17, 33, want_certificates=True)
        b = engine.solve_batch(mats, 17, 33, want_certificates=True)
        assert same_bits(a["certificate"], b["certificate"])
        shapes = [(9, 17), (33, 65), (17, 33)] * 4
        tabs = [mixed_batch(4, h - 1, w - 1, seed=i)[i % 4] for i, (h, w) in enumerate(shapes)]
        ra = multi.solve_ragged(tabs, shapes, want_certificates=True)
        rb = engine.solve_ragged(tabs, shapes, want_certificates=True)
        assert all(same_bits(x["certificate"], y["certificate"]) for x, y in zip(ra, rb))
    finally:
        multi.close()


# ------------------------------------------------------------------------------------------------- Netlib
# These models end `infeasible` because of the reference's tolerance-free rule, so only the bits are asserted.
@pytest.mark.parametrize("name", ["ITEST2", "ITEST6", "BGPRTR", "KLEIN1", "KLEIN2"])
def test_netlib_against_oracle(engine, name):
    g = NL.get(name)
    H, W = g["height"], g["width"]
    got = engine.solve_batch(g["matrix"], H, W, E.make_options(check_cycles=g["check_cycles"]), want_certificates=True)
    exp = oracle_batch(g["matrix"], H, W, check_cycles=g["check_cycles"])
    assert exp["status"][0] == 1
    assert same_bits(got["certificate"], expected(exp["matrices"], exp["status"], exp["value"], exp["pos"], H, W))


@pytest.mark.parametrize("name", ["AGG", "25FV47"])
def test_netlib_against_own_tableau(engine, name):
    g = NL.get(name)
    H, W = g["height"], g["width"]
    got = engine.solve_batch(g["matrix"], H, W, E.make_options(check_cycles=g["check_cycles"]), want_matrices=True,
                             want_certificates=True)
    assert got["status"][0] == 1
    exp = expected(got["matrices"], got["status"], got["value"], got["pos"], H, W)
    assert same_bits(got["certificate"], exp)


# ------------------------------------------------------------------------------------------------- model level
WORKED = [
    {"direction": "maximize", "objective": "p", "constraints": {"c": {"max": -1}}, "variables": {"x": {"c": 1, "p": 1}}},
    {"direction": "maximize", "objective": "p", "constraints": {"c1": {"min": 3}, "c2": {"max": 1}},
     "variables": {"x": {"c1": 1, "c2": 1, "p": 1}, "y": {"c1": 1, "c2": 1, "p": 2}}},
    {"direction": "maximize", "objective": "p", "constraints": {"c": {"max": 1}},
     "variables": {"x": {"c": 1, "p": 1}, "y": {"c": -1, "p": 1}}},
]


def test_solve_with_certificate_equals_cpu_mapping(engine):
    cases = [(c["model"], c["options"]) for c in GOLDEN] + [(m, {}) for m in WORKED]
    for model, options in cases:
        got = yalps_b200.solve(model, {**options, "certificate": True}, engine=engine)
        assert repr(got) == repr(oracle_certificate(model, options)[0])
        plain = yalps_b200.solve(model, options, engine=engine)
        assert repr({k: got[k] for k in plain}) == repr(plain)
        both = yalps_b200.solve(model, {**options, "certificate": True, "ranging": True}, engine=engine)
        assert repr({k: both[k] for k in got}) == repr(got)
    plain_cases = [m for m, o in cases if not o]
    many = yalps_b200.solve_many(plain_cases, {"certificate": True}, engine=engine)
    assert repr(many) == repr([oracle_certificate(m)[0] for m in plain_cases])
    assert repr([{k: s[k] for k in p} for s, p in zip(many, yalps_b200.solve_many(plain_cases, engine=engine))]) == \
        repr(yalps_b200.solve_many(plain_cases, engine=engine))
