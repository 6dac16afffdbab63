"""Sensitivity ranges on the GPU (k_ranging, include/yalps_b200.h "sensitivity ranging"): bit for bit
yalps_b200.sensitivity.ranges_from_tableau of the oracle's final tableau on every kernel path and entry point, and
solve() / solve_many() with `ranging` equal to the CPU mapping of tests/test_ranging.py."""
import numpy as np
import pytest

import yalps_b200
from conftest import load_netlib, same_bits
from oracle import lib as O
from test_gpu_sensitivity import NETLIB_QUICK, PATHS, _bounded_netlib_models, oracle_batch, special_batch
from test_ranging import _oracle_solution, random_lp, synthetic
from test_sensitivity import LP_CASES
from yalps_b200 import engine as E
from yalps_b200.sensitivity import ranges_from_tableau, row_pairs
from yalps_b200.tableau import constraint_rows, entries, tableau_model

pytestmark = pytest.mark.gpu

NL = load_netlib()


def expected(mats, status, pos, H, W, pairs=None, precision=1e-8):
    mats = np.asarray(mats).reshape(-1, H * W)
    pos = np.asarray(pos).reshape(-1, W + H)
    pr = None if pairs is None else np.asarray(pairs).reshape(-1, H)
    out = [ranges_from_tableau(mats[i], W, H, pos[i], precision, None if pr is None else pr[i], status[i] == 0)
           for i in range(mats.shape[0])]
    return np.stack([o[0] for o in out]), np.stack([o[1] for o in out])


def random_pairs(rng, n, H):
    out = np.full((n, H), -1, np.int32)
    for i in range(n):
        rows = rng.permutation(np.arange(1, H))
        for j in range(0, len(rows) - 1, 2):
            if rng.random() < 0.5:
                out[i, rows[j]], out[i, rows[j + 1]] = rows[j + 1], rows[j]
    return out


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
    mats, poss, prs = [], [], []
    for _ in range(n):
        m, p, pr = synthetic(rng, H, W, with_pairs=False)
        mats.append(m)
        poss.append(p)
    mats, poss = np.stack(mats), np.stack(poss)
    pairs = random_pairs(rng, n, H)
    status = np.where(rng.random(n) < 0.8, 0, rng.integers(1, 5, n)).astype(np.int32)
    status[0] = 0
    dev = torch.device("cuda:0")
    d_m, d_pos = torch.from_numpy(mats).to(dev), torch.from_numpy(poss).to(dev)
    d_st, d_pr = torch.from_numpy(status).to(dev), torch.from_numpy(pairs).to(dev)
    for with_pairs, with_status in ((False, False), (True, True)):
        d_lo = torch.full((n, W + H), 7.0, dtype=torch.float64, device=dev)
        d_hi = torch.full((n, W + H), 7.0, dtype=torch.float64, device=dev)
        engine.ranging_device(n, H, W, d_m.data_ptr(), d_pos.data_ptr(), d_lo.data_ptr(), d_hi.data_ptr(),
                              d_status=d_st.data_ptr() if with_status else 0,
                              d_pairs=d_pr.data_ptr() if with_pairs else 0,
                              stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        st = status if with_status else np.zeros(n, np.int32)
        lo, hi = expected(mats, st, poss, H, W, pairs if with_pairs else None)
        assert same_bits(d_lo.cpu().numpy(), lo) and same_bits(d_hi.cpu().numpy(), hi)


# ------------------------------------------------------------------------------------------- host entries
@pytest.mark.parametrize("name,path,threads,rows", PATHS, ids=[p[0] for p in PATHS])
def test_paths_bit_exact(tuned, name, path, threads, rows):
    n = 3 if path in (E.PATH_GRID, E.PATH_GRID_RESIDENT, E.PATH_CLUSTER) else 40
    m, nv = 16, 32
    H, W = m + 1, nv + 1
    mats = special_batch(n, m, nv)
    pairs = random_pairs(np.random.default_rng(1), n, H)
    tuned.set_tuning(path, threads, rows)
    opt = E.make_options()
    got = tuned.solve_batch(mats, H, W, opt, want_matrices=True, want_duals=True, want_ranges=True, pairs=pairs)
    plain = tuned.solve_batch(mats, H, W, opt, want_matrices=True, want_duals=True)
    exp = oracle_batch(mats, H, W)
    lo, hi = expected(exp["matrices"], exp["status"], exp["pos"], H, W, pairs)
    assert same_bits(got["range_lo"], lo) and same_bits(got["range_hi"], hi)
    # requesting ranges changes no other output bit
    for k in ("status", "pivots", "pos", "var"):
        assert np.array_equal(got[k], plain[k]), k
    for k in ("value", "rhs", "matrices", "reduced"):
        assert same_bits(got[k], plain[k]), k


def test_random_and_golden_lps(engine):
    models = [random_lp(s) for s in range(30)] + [c["model"] for c in LP_CASES if not c["options"]]
    for model in models:
        tm = tableau_model(model)
        t = tm.tableau
        pairs = row_pairs(constraint_rows(list(entries(model["constraints"]))), t.height)
        got = engine.solve_batch(t.matrix, t.height, t.width, want_ranges=True, pairs=pairs)
        exp = oracle_batch(t.matrix, t.height, t.width)
        lo, hi = expected(exp["matrices"], exp["status"], exp["pos"], t.height, t.width, pairs)
        assert same_bits(got["range_lo"], lo) and same_bits(got["range_hi"], hi)


@pytest.mark.parametrize("name", NETLIB_QUICK)
def test_netlib(engine, name):
    g = NL.get(name)
    H, W = g["height"], g["width"]
    got = engine.solve_batch(g["matrix"], H, W, E.make_options(check_cycles=g["check_cycles"]), want_ranges=True)
    exp = oracle_batch(g["matrix"], H, W, check_cycles=g["check_cycles"])
    lo, hi = expected(exp["matrices"], exp["status"], exp["pos"], H, W)
    assert same_bits(got["range_lo"], lo) and same_bits(got["range_hi"], hi)


def test_pipelined_chunks(engine):
    m, nv, n = 32, 64, 4500  # 78 MB of tableaus: more than one 64 MiB pipeline chunk
    H, W = m + 1, nv + 1
    mats = O.generate_synthetic(11, n, m, nv, 2)
    pairs = random_pairs(np.random.default_rng(2), n, H)
    exp = oracle_batch(mats, H, W)
    lo, hi = expected(exp["matrices"], exp["status"], exp["pos"], H, W, pairs)
    for path in (E.PATH_GMEM, E.PATH_AUTO):
        engine.set_tuning(path, 64 if path == E.PATH_GMEM else 0, 0)
        try:
            got = engine.solve_batch(mats, H, W, want_ranges=True, pairs=pairs)
        finally:
            engine.set_tuning(E.PATH_AUTO, 0, 0)
        assert same_bits(got["range_lo"], lo) and same_bits(got["range_hi"], hi)


@pytest.mark.parametrize("small", [True, False], ids=["zero_copy", "chunked"])
def test_ragged_mixed_routes(engine, small):
    shapes = [(9, 17), (33, 65), (5, 9)] * 3 if small else [(9, 17), (33, 65), (17, 33), (61, 121), (129, 257),
                                                                (300, 500), (5, 9)] * 3
    tabs = [O.generate_synthetic(i, 1, h - 1, w - 1, 2)[0] for i, (h, w) in enumerate(shapes)]
    rng = np.random.default_rng(3)
    pairs = [random_pairs(rng, 1, h)[0] for h, _ in shapes]
    got = engine.solve_ragged(tabs, shapes, want_ranges=True, pairs=pairs, want_duals=True)
    plain = engine.solve_ragged(tabs, shapes, want_duals=True)
    for i, (h, w) in enumerate(shapes):
        exp = oracle_batch(tabs[i], h, w)
        lo, hi = expected(exp["matrices"], exp["status"], exp["pos"], h, w, pairs[i])
        assert same_bits(got[i]["range_lo"], lo[0]) and same_bits(got[i]["range_hi"], hi[0])
        assert np.array_equal(got[i]["pos"], plain[i]["pos"]) and same_bits(got[i]["reduced"], plain[i]["reduced"])


def test_bad_pairs_are_refused(engine):
    mats = O.generate_synthetic(1, 2, 4, 6, 0)
    bad = np.full((2, 5), -1, np.int32)
    bad[1, 1] = 2  # not symmetric
    with pytest.raises(yalps_b200.engine.YalpsError):
        engine.solve_batch(mats, 5, 7, want_ranges=True, pairs=bad)
    bad[1, 2] = 1
    bad[0, 0] = 3  # row 0 has no pair
    with pytest.raises(yalps_b200.engine.YalpsError):
        engine.solve_batch(mats, 5, 7, want_ranges=True, pairs=bad)


def test_sparse_entry_equals_dense(engine):
    big = [n for n in NETLIB_QUICK if NL.get(n)["height"] * NL.get(n)["width"] * 8 > (768 << 10)]
    for name in ["AFIRO"] + big[:2]:
        g = NL.get(name)
        if g["check_cycles"]:
            continue
        H, W = g["height"], g["width"]
        nz = np.flatnonzero(g["matrix"].view(np.uint64) != 0)
        sp = engine.solve_lp_sparse(nz.astype(np.int32), g["matrix"][nz], H, W, want_ranges=True)
        dn = engine.solve_batch(g["matrix"], H, W, want_ranges=True)
        assert sp["status"] == dn["status"][0] and np.array_equal(sp["pos"], dn["pos"][0])
        assert same_bits(sp["range_lo"], dn["range_lo"][0]) and same_bits(sp["range_hi"], dn["range_hi"][0])


def test_multi_equals_single(engine):
    multi = yalps_b200.MultiEngine([0, 0])
    try:
        mats = special_batch(50, 16, 32, seed=7)
        pairs = random_pairs(np.random.default_rng(4), 50, 17)
        a = multi.solve_batch(mats, 17, 33, want_ranges=True, pairs=pairs)
        b = engine.solve_batch(mats, 17, 33, want_ranges=True, pairs=pairs)
        assert same_bits(a["range_lo"], b["range_lo"]) and same_bits(a["range_hi"], b["range_hi"])
        shapes = [(9, 17), (33, 65), (17, 33)] * 4
        tabs = [O.generate_synthetic(i, 1, h - 1, w - 1, 1)[0] for i, (h, w) in enumerate(shapes)]
        ra, rb = multi.solve_ragged(tabs, shapes, want_ranges=True), engine.solve_ragged(tabs, shapes, want_ranges=True)
        assert all(same_bits(x["range_lo"], y["range_lo"]) and same_bits(x["range_hi"], y["range_hi"])
                   for x, y in zip(ra, rb))
    finally:
        multi.close()


# ------------------------------------------------------------------------------------------------- model level
def test_solve_with_ranging_equals_cpu_mapping(engine):
    for case in LP_CASES:
        opts = {**case["options"], "ranging": True}
        got = yalps_b200.solve(case["model"], opts, engine=engine)
        assert repr(got) == repr(_oracle_solution(case["model"], opts)), case["name"]
    many = yalps_b200.solve_many([c["model"] for c in LP_CASES if not c["options"]], {"ranging": True}, engine=engine)
    exp = [_oracle_solution(c["model"]) for c in LP_CASES if not c["options"]]
    assert repr(many) == repr(exp)


def test_solve_with_ranging_bounded_netlib(engine):
    for name, model in _bounded_netlib_models():
        got = yalps_b200.solve(model, {"ranging": True}, engine=engine)  # big ones take the cell-pair entry
        assert repr(got) == repr(_oracle_solution(model)), name
