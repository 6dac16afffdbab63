"""Reduced-cost output (`reduced`, include/yalps_b200.h "dual values") on the GPU: bit for bit row 0 of the oracle's
final tableau re-indexed by variable, on every kernel path and entry point; solve() / solve_many() with
`sensitivity` equal the CPU mapping of tests/test_sensitivity.py applied to the oracle's tableau."""
import gzip
import json
import os

import numpy as np
import pytest

import yalps_b200
from conftest import GOLDEN, load_cases, load_netlib, same_bits
from oracle import lib as O
from test_sensitivity import LP_CASES, oracle_sensitivity
from yalps_b200 import engine as E
from yalps_b200.mps import netlib_model
from yalps_b200.sensitivity import reduced_from_tableau
from yalps_b200.tableau import tableau_model

pytestmark = pytest.mark.gpu

NL = load_netlib()
NETLIB_QUICK = [n for n in NL.names if float(NL.z[f"{n}/oracle_seconds"][0]) < 1.0]

# (name, path, threads per LP, row groups)
PATHS = [("TMEM", E.PATH_TMEM, 0, 0), ("SMEM", E.PATH_SMEM, 32, 0), ("GMEM", E.PATH_GMEM, 64, 0),
         ("SPLIT_SMEM", E.PATH_SMEM, 128, 4), ("SPLIT_GMEM", E.PATH_GMEM, 128, 2), ("CLUSTER", E.PATH_CLUSTER, 0, 0),
         ("GRID_RESIDENT", E.PATH_GRID_RESIDENT, 0, 0), ("GRID", E.PATH_GRID, 0, 0), ("AUTO", E.PATH_AUTO, 0, 0)]


def oracle_batch(mats, height, width, precision=1e-8, max_pivots=8192, check_cycles=False):
    """Oracle outputs plus the expected reduced vectors."""
    work = np.ascontiguousarray(mats, np.float64).reshape(-1, height * width).copy()
    exp = O.simplex_batch(work, width, height, precision, max_pivots, check_cycles, nthreads=os.cpu_count() or 1)
    exp["reduced"] = np.stack([reduced_from_tableau(work[i], width, height, exp["pos"][i]) for i in range(work.shape[0])])
    exp["matrices"] = work
    return exp


def special_batch(n, m, nv, seed=0):
    """Synthetic LPs with signed zeros, tiny and huge cells, and infeasible rows."""
    mats = O.generate_synthetic(seed, n, m, nv, 3)
    rng = np.random.default_rng(seed)
    for i in range(0, n, 3):
        cells = rng.integers(0, (m + 1) * (nv + 1), 6)
        mats[i, cells[:2]] = -0.0
        mats[i, cells[2:4]] = 1e-300
        mats[i, cells[4]] = 1e300
    return mats


@pytest.fixture
def tuned(engine):
    yield engine
    engine.set_tuning(E.PATH_AUTO, 0, 0)


@pytest.mark.parametrize("name,path,threads,rows", PATHS, ids=[p[0] for p in PATHS])
@pytest.mark.parametrize("opts", [{}, {"check_cycles": True}, {"max_pivots": 3}], ids=["plain", "cycles", "budget"])
def test_paths_bit_exact(tuned, name, path, threads, rows, opts):
    n = 3 if path in (E.PATH_GRID, E.PATH_GRID_RESIDENT, E.PATH_CLUSTER) else 40
    m, nv = 16, 32
    mats = special_batch(n, m, nv)
    tuned.set_tuning(path, threads, rows)
    opt = E.make_options(**opts)
    got = tuned.solve_batch(mats, m + 1, nv + 1, opt, want_matrices=True, want_duals=True)
    plain = tuned.solve_batch(mats, m + 1, nv + 1, opt, want_matrices=True)
    exp = oracle_batch(mats, m + 1, nv + 1, max_pivots=opts.get("max_pivots", 8192),
                       check_cycles=opts.get("check_cycles", False))
    assert np.array_equal(got["status"], exp["status"]) and np.array_equal(got["pos"], exp["pos"])
    assert same_bits(got["reduced"], exp["reduced"])
    # requesting duals changes no other output bit; reduced is row 0 of the final tableau
    for k in ("status", "pivots", "pos", "var"):
        assert np.array_equal(got[k], plain[k]), k
    for k in ("value", "rhs", "matrices"):
        assert same_bits(got[k], plain[k]), k
    for i in range(n):
        assert same_bits(got["reduced"][i], reduced_from_tableau(got["matrices"][i], nv + 1, m + 1, got["pos"][i]))
    if opts.get("max_pivots") == 3:
        assert (got["status"] == 4).any()  # exhausted budgets: cycled


def test_statuses_covered(engine):
    m, nv = 16, 32
    mats = special_batch(60, m, nv)
    infeasible = mats[1].reshape(m + 1, nv + 1)
    infeasible[1, :] = 0.0
    infeasible[1, 0] = -1.0  # 0 <= -1: phase 1 finds no entering column
    unbounded = mats[2].reshape(m + 1, nv + 1)
    unbounded[:, :] = O.generate_synthetic(99, 1, m, nv, 0)[0].reshape(m + 1, nv + 1)
    unbounded[0, 1] = 5.0
    unbounded[1:, 1] = -1.0  # column 1 improves the objective and no row limits it
    got = engine.solve_batch(mats, m + 1, nv + 1, E.make_options(max_pivots=6), want_duals=True)
    exp = oracle_batch(mats, m + 1, nv + 1, max_pivots=6)
    assert np.array_equal(got["status"], exp["status"])
    assert set(got["status"].tolist()) == {0, 1, 2, 4}
    assert same_bits(got["reduced"], exp["reduced"])


def test_ragged_mixed_sizes(engine):
    shapes = [(9, 17), (33, 65), (17, 33), (61, 121), (129, 257), (5, 9)] * 5
    tabs = [O.generate_synthetic(i, 1, h - 1, w - 1, 2)[0] for i, (h, w) in enumerate(shapes)]
    got = engine.solve_ragged(tabs, shapes, want_duals=True, want_matrices=True)
    plain = engine.solve_ragged(tabs, shapes)
    for i, (h, w) in enumerate(shapes):
        exp = oracle_batch(tabs[i], h, w)
        assert got[i]["status"] == exp["status"][0]
        assert same_bits(got[i]["reduced"], exp["reduced"][0])
        assert np.array_equal(got[i]["pos"], plain[i]["pos"]) and same_bits(got[i]["rhs"], plain[i]["rhs"])


def test_pipelined_chunks(engine):
    m, nv, n = 32, 64, 4500  # 78 MB of tableaus: more than one 64 MiB pipeline chunk
    mats = O.generate_synthetic(11, n, m, nv, 2)
    engine.set_tuning(E.PATH_GMEM, 64, 0)  # the HBM-resident kernel keeps the pipelined route (no zero-copy call)
    try:
        got = engine.solve_batch(mats, m + 1, nv + 1, want_duals=True)
    finally:
        engine.set_tuning(E.PATH_AUTO, 0, 0)
    got_auto = engine.solve_batch(mats, m + 1, nv + 1, want_duals=True)
    exp = oracle_batch(mats, m + 1, nv + 1)
    assert same_bits(got["reduced"], exp["reduced"]) and same_bits(got_auto["reduced"], exp["reduced"])


def test_device_entry(engine):
    torch = pytest.importorskip("torch")
    m, nv, n = 16, 32, 300
    mats = O.generate_synthetic(3, n, m, nv, 2)
    H, W = m + 1, nv + 1
    dev = torch.device("cuda:0")
    d_m = torch.from_numpy(mats).to(dev)
    d_work = torch.empty_like(d_m)
    d_status = torch.empty(n, dtype=torch.int32, device=dev)
    d_pos = torch.empty((n, W + H), dtype=torch.int32, device=dev)
    d_red = torch.full((n, W + H), float("nan"), dtype=torch.float64, device=dev)
    engine.solve_batch_device(n, H, W, d_m.data_ptr(), d_work=d_work.data_ptr(), d_status=d_status.data_ptr(),
                              d_pos=d_pos.data_ptr(), d_reduced=d_red.data_ptr(),
                              stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    exp = oracle_batch(mats, H, W)
    assert np.array_equal(d_pos.cpu().numpy(), exp["pos"])
    assert same_bits(d_red.cpu().numpy(), exp["reduced"])


@pytest.mark.parametrize("name", NETLIB_QUICK)
def test_netlib(engine, name):
    g = NL.get(name)
    H, W = g["height"], g["width"]
    got = engine.solve_batch(g["matrix"], H, W, E.make_options(check_cycles=g["check_cycles"]), want_duals=True)
    exp = oracle_batch(g["matrix"], H, W, check_cycles=g["check_cycles"])
    assert got["status"][0] == g["status"] and np.array_equal(got["pos"][0], g["final_pos"])
    assert same_bits(got["reduced"], exp["reduced"])


# ------------------------------------------------------------------------------------------------------ replicas
def _replica_case(eps, n=200, seed=5):
    m, nv = 24, 48
    base = O.generate_synthetic(seed, 1, m, nv, 0)[0]
    H, W = m + 1, nv + 1
    rng = np.random.default_rng(seed)
    b0 = base.reshape(H, W)[:, 0]
    rhs = np.repeat(b0[None, :], n, 0) * (1.0 + eps * rng.uniform(-1, 1, (n, H)))
    mats = np.repeat(base[None, :], n, 0).reshape(n, H, W).copy()
    mats[:, :, 0] = rhs
    return base, rhs, H, W, mats.reshape(n, -1)


@pytest.mark.parametrize("eps", [0.0, 0.5], ids=["on_path", "forks"])
@pytest.mark.parametrize("sharing", [True, False], ids=["shared", "solo"])
def test_replicas(engine, eps, sharing):
    base, rhs, H, W, mats = _replica_case(eps)
    engine.set_replica_sharing(sharing)
    try:
        got = engine.solve_replicas(base, rhs, H, W, want_duals=True)
        forks = engine.replica_forks
        plain = engine.solve_replicas(base, rhs, H, W)
    finally:
        engine.set_replica_sharing(True)
    exp = oracle_batch(mats, H, W)
    assert np.array_equal(got["status"], exp["status"]) and np.array_equal(got["pos"], exp["pos"])
    assert same_bits(got["reduced"], exp["reduced"])
    assert same_bits(got["rhs"], plain["rhs"]) and np.array_equal(got["pivots"], plain["pivots"])
    if sharing:
        assert forks == 0 if eps == 0.0 else forks > 0
    else:
        assert forks == -1


# --------------------------------------------------------------------------------------------- sparse, multi
def test_sparse_entry_equals_dense(engine):
    big = [n for n in NETLIB_QUICK if NL.get(n)["height"] * NL.get(n)["width"] * 8 > (768 << 10)]
    names = ["AFIRO"] + big[:2]  # one densified small call, and the device-side cell scatter
    for name in names:
        g = NL.get(name)
        if g["check_cycles"]:
            continue
        H, W = g["height"], g["width"]
        nz = np.flatnonzero(g["matrix"].view(np.uint64) != 0)  # -0.0 is a store too
        sp = engine.solve_lp_sparse(nz.astype(np.int32), g["matrix"][nz], H, W)
        dn = engine.solve_batch(g["matrix"], H, W, want_duals=True)
        assert sp["status"] == dn["status"][0] and np.array_equal(sp["pos"], dn["pos"][0])
        assert same_bits(sp["reduced"], dn["reduced"][0]) and same_bits(sp["rhs"], dn["rhs"][0])


def test_multi_equals_single(engine):
    multi = yalps_b200.MultiEngine([0, 0])
    try:
        mats = special_batch(50, 16, 32, seed=7)
        a = multi.solve_batch(mats, 17, 33, want_duals=True)
        b = engine.solve_batch(mats, 17, 33, want_duals=True)
        assert same_bits(a["reduced"], b["reduced"]) and np.array_equal(a["pos"], b["pos"])
        shapes = [(9, 17), (33, 65), (17, 33)] * 4
        tabs = [O.generate_synthetic(i, 1, h - 1, w - 1, 1)[0] for i, (h, w) in enumerate(shapes)]
        ra, rb = multi.solve_ragged(tabs, shapes, want_duals=True), engine.solve_ragged(tabs, shapes, want_duals=True)
        assert all(same_bits(x["reduced"], y["reduced"]) for x, y in zip(ra, rb))
        base, rhs, H, W, _ = _replica_case(0.5, n=64)
        a = multi.solve_replicas(base, rhs, H, W, want_duals=True)
        b = engine.solve_replicas(base, rhs, H, W, want_duals=True)
        assert same_bits(a["reduced"], b["reduced"])
    finally:
        multi.close()


# ------------------------------------------------------------------------------------------------- model level
def test_without_option_nothing_changes(engine):
    for case in LP_CASES[:10]:
        a = yalps_b200.solve(case["model"], case["options"], engine=engine)
        b = yalps_b200.solve(case["model"], {**case["options"], "sensitivity": False}, engine=engine)
        assert set(a) == {"status", "result", "variables"} and repr(a) == repr(b)
    models = [c["model"] for c in LP_CASES]
    for s in yalps_b200.solve_many(models, engine=engine):
        assert set(s) == {"status", "result", "variables"}


def _bounded_netlib_models():
    with gzip.open(os.path.join(GOLDEN, "netlib_bounded.json.gz"), "rt") as f:
        cases = json.load(f)
    out = []
    for c in cases:
        try:
            model = netlib_model(c["mps"])
        except ValueError:
            continue
        if not model.get("integers") and not model.get("binaries"):
            out.append((c["name"], model))
    return out


def test_solve_with_sensitivity_equals_cpu_mapping(engine):
    for case in LP_CASES:
        opts = {**case["options"], "sensitivity": True}
        got = yalps_b200.solve(case["model"], opts, engine=engine)
        assert repr(got) == repr(oracle_sensitivity(case["model"], opts)), case["name"]
    many = yalps_b200.solve_many([c["model"] for c in LP_CASES if not c["options"]], {"sensitivity": True},
                                 engine=engine)
    exp = [oracle_sensitivity(c["model"], {"sensitivity": True}) for c in LP_CASES if not c["options"]]
    assert repr(many) == repr(exp)


def test_solve_with_sensitivity_bounded_netlib(engine):
    models = _bounded_netlib_models()
    assert models
    for name, model in models:
        got = yalps_b200.solve(model, {"sensitivity": True}, engine=engine)  # big ones take the cell-pair entry
        assert repr(got) == repr(oracle_sensitivity(model, {"sensitivity": True})), name
