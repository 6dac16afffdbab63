"""The drop-in boundary (SURVEY 8b), exercised through the C ABI on a device:

* `simplex(tableau, options)` with the tableau's own basis bookkeeping (yalps_solve_batch_basis): a branch and cut
  driven ONLY through that call, one node at a time, exactly as src/branchAndCut.ts:122-164 would drive a replaced
  `simplex` import -- node for node against the oracle;
* replicas (yalps_solve_replicas) against the plain batch entry;
* one process, several GPUs (yalps_multi_*): same bits as one GPU, incumbent min-allreduce, sharded frontier,
  many MILPs.  On a 1-GPU box the multi tests run with two logical ranks on GPU 0.
"""
import heapq
import math

import numpy as np
import pytest

from conftest import load_cases, load_netlib, same_bits, same_value
from oracle import lib as O, model as M
import yalps_b200
from yalps_b200 import engine as E
from yalps_b200.sensitivity import reduced_from_tableau
from yalps_b200.tableau import Tableau, tableau_model

pytestmark = pytest.mark.gpu
CASES = load_cases()


def js_round(x):
    r = math.floor(x)
    return r + 1.0 if x - r >= 0.5 else float(r)


def most_fractional(t, ints):
    """src/branchAndCut.ts:64-85"""
    best, var, val = 0.0, 0, 0.0
    for iv in ints:
        row = int(t.position_of_variable[iv]) - t.width
        if row < 0:
            continue
        v = float(t.matrix[row * t.width])
        frac = abs(v - js_round(v))
        if frac > best:
            best, var, val = frac, iv, v
    return var, val, best


class _Br:
    __slots__ = ("ev", "cuts")

    def __init__(self, ev, cuts):
        self.ev, self.cuts = ev, cuts

    def __lt__(self, o):
        return self.ev - o.ev < 0


def branch_and_cut_through_simplex(engine, tm, opt, copt):
    """src/branchAndCut.ts:89-176 with `simplex` replaced by Engine.simplex (one C-ABI call per node)."""
    t = tm.tableau
    status, result = engine.simplex(t, copt)
    stats = {"nodes": 0, "root": (status, result)}
    if not tm.integers or status != "optimal":
        return status, result, t, stats
    var, val, frac = most_fractional(t, tm.integers)
    if frac <= opt["precision"]:
        return status, result, t, stats
    heap = []
    heapq.heappush(heap, _Br(result, [(-1.0, var, float(math.ceil(val)))]))
    heapq.heappush(heap, _Br(result, [(1.0, var, float(math.floor(val)))]))
    threshold = result * (1.0 - tm.sign * opt["tolerance"])
    best_eval, best, it = math.inf, None, 0
    root_m, root_pos, root_var = t.matrix.copy(), t.position_of_variable.copy(), t.variable_at_position.copy()
    while it < opt["maxIterations"] and heap and best_eval >= threshold:
        br = heapq.heappop(heap)
        if br.ev > best_eval:
            break
        m, p, v = O.apply_cuts(root_m, t.width, t.height, root_pos, root_var, [c[0] for c in br.cuts],
                               [c[1] for c in br.cuts], [c[2] for c in br.cuts])
        node = Tableau(m, t.width, t.height + len(br.cuts), p, v)
        st, res = engine.simplex(node, copt)
        stats["nodes"] += 1
        if st == "optimal" and res < best_eval:
            var, val, frac = most_fractional(node, tm.integers)
            if frac <= opt["precision"]:
                best_eval, best = res, node
            else:
                upper, lower = [], []
                for cut in br.cuts:
                    if cut[1] == var:
                        (lower if cut[0] < 0 else upper).append(cut)
                    else:
                        upper.append(cut)
                        lower.append(cut)
                lower.append((1.0, var, float(math.floor(val))))
                upper.append((-1.0, var, float(math.ceil(val))))
                heapq.heappush(heap, _Br(res, upper))
                heapq.heappush(heap, _Br(res, lower))
        it += 1
    if best is None:
        return "infeasible", math.nan, t, stats
    return "optimal", best_eval, best, stats


@pytest.mark.parametrize("name", ["Knapsack 1", "Fancy Stock Cutting Problem", "Integer Wood Shop Problem",
                                  "Cutting Stock", "Taco Party", "Integer Sports Complex Problem"])
def test_branch_and_cut_driven_through_the_simplex_shaped_entry(engine, name):
    case = next(c for c in CASES if c["name"] == name)
    o = case["oracle"]
    opt = {**M.DEFAULT_OPTIONS, **case["options"]}
    copt = E.make_options(opt["precision"], opt["maxPivots"], opt["checkCycles"])
    tm = tableau_model(case["model"])
    status, result, final, stats = branch_and_cut_through_simplex(engine, tm, opt, copt)
    assert status == o["status"] and same_value(-tm.sign * result, o["result"])
    assert stats["nodes"] == o["nodes"]
    assert stats["root"][0] == o["root_status"] and same_value(stats["root"][1], o["root_result"])
    h = final.height
    assert np.array_equal(final.position_of_variable, o["final_pos"])
    assert same_bits(final.matrix.reshape(h, final.width)[:, 0], o["final_rhs"])


def mid_trajectory_states(n, m, nv, neg, first, k):
    """Tableaus with a non-identity basis: the oracle stopped after at most k pivots per phase."""
    mats = O.generate_synthetic(first, n, m, nv, neg)
    H, W = m + 1, nv + 1
    pos = np.tile(np.arange(W + H, dtype=np.int32), (n, 1))
    var = pos.copy()
    for i in range(n):
        O.simplex(mats[i], W, H, pos[i], var[i], max_pivots=k)
    return mats, pos, var


@pytest.mark.parametrize("path,m,nv,neg,n", [(E.PATH_TMEM, 32, 64, 6, 200), (E.PATH_TMEM, 50, 40, 10, 64),
                                             (E.PATH_SMEM, 32, 64, 6, 96), (E.PATH_SMEM, 90, 120, 20, 24),
                                             (E.PATH_GMEM, 60, 80, 9, 40), (E.PATH_CLUSTER, 200, 260, 30, 3),
                                             (E.PATH_GRID, 70, 300, 10, 2), (E.PATH_GRID_RESIDENT, 70, 300, 10, 2), (E.PATH_AUTO, 20, 30, 5, 5),
                                             (E.PATH_AUTO, 32, 64, 8, 1000)])
def test_caller_supplied_basis_on_every_kernel_path(engine, path, m, nv, neg, n):
    H, W = m + 1, nv + 1
    mats, pos, var = mid_trajectory_states(n, m, nv, neg, 9100 + m, 3)
    assert not np.array_equal(pos[0], np.arange(W + H))
    exp_m, exp_pos, exp_var = mats.copy(), pos.copy(), var.copy()
    exp = [O.simplex(exp_m[i], W, H, exp_pos[i], exp_var[i]) for i in range(n)]
    engine.set_tuning(path, 0)
    try:
        got = engine.solve_batch(mats, H, W, want_matrices=True, pos_in=pos, var_in=var)
    finally:
        engine.set_tuning(E.PATH_AUTO, 0)
    assert got["status"].tolist() == [e[0] for e in exp]
    assert same_bits(got["value"], np.array([e[1] for e in exp]))
    assert got["pivots"].tolist() == [list(e[2]) for e in exp]
    assert np.array_equal(got["pos"], exp_pos) and np.array_equal(got["var"], exp_var)
    assert same_bits(got["matrices"], exp_m)


def test_basis_arguments_are_validated(engine):
    mats, pos, var = mid_trajectory_states(2, 4, 5, 1, 1, 2)
    bad = var.copy()
    bad[1, 0], bad[1, 1] = bad[1, 1], bad[1, 0]  # no longer the inverse of pos
    with pytest.raises(E.YalpsError) as e:
        engine.solve_batch(mats, 5, 6, pos_in=pos, var_in=bad)
    assert e.value.code == -2 and "inverse" in str(e.value)
    with pytest.raises(E.YalpsError):
        engine.solve_batch(mats, 5, 6, pos_in=pos, var_in=None)


def test_in_place_contract_outputs_may_alias_inputs(engine):
    """simplex() mutates the tableau it is given (src/simplex.ts:5-39): the same arrays as input and output."""
    tm = tableau_model(next(c for c in CASES if c["name"] == "Knapsack 1")["model"])
    t = tm.tableau
    ref = M.tableau_model(next(c for c in CASES if c["name"] == "Knapsack 1")["model"]).tableau
    st, val, _ = O.simplex(ref.matrix, ref.width, ref.height, ref.pos, ref.var)
    status, value = engine.simplex(t)
    assert E.STATUS_NAMES.index(status) == st and same_value(value, val)
    assert same_bits(t.matrix, ref.matrix) and np.array_equal(t.position_of_variable, ref.pos)
    assert np.array_equal(t.variable_at_position, ref.var)


# ------------------------------------------------------------------------------------------------ replicas
@pytest.mark.parametrize("name,n", [("ADLITTLE", 300), ("SC105", 600), ("AFIRO", 1000)])
def test_replicas_equal_the_expanded_batch_and_the_oracle(engine, name, n):
    g = load_netlib().get(name)
    H, W = g["height"], g["width"]
    base = g["matrix"]
    rng = np.random.default_rng(5)
    rhs = np.tile(base.reshape(H, W)[:, 0], (n, 1)) * (1.0 + 1e-2 * (2.0 * rng.random((n, H)) - 1.0))
    mats = np.tile(base, (n, 1))
    mats.reshape(n, H, W)[:, :, 0] = rhs
    got = engine.solve_replicas(base, rhs, H, W)
    ref = engine.solve_batch(mats, H, W)
    for k in ("status", "pivots", "pos", "var"):
        assert np.array_equal(got[k], ref[k]), k
    assert same_bits(got["value"], ref["value"]) and same_bits(got["rhs"], ref["rhs"])
    sample = mats[:48].copy()
    exp = O.simplex_batch(sample, W, H)
    assert np.array_equal(got["status"][:48], exp["status"]) and np.array_equal(got["pivots"][:48], exp["pivots"])
    assert same_bits(got["rhs"][:48], exp["rhs"]) and np.array_equal(got["pos"][:48], exp["pos"])


def _replica_case(base, H, W, n, eps, seed):
    rng = np.random.default_rng(seed)
    rhs = np.tile(base.reshape(H, W)[:, 0], (n, 1)) * (1.0 + eps * (2.0 * rng.random((n, H)) - 1.0))
    mats = np.tile(base, (n, 1))
    mats.reshape(n, H, W)[:, :, 0] = rhs
    return rhs, mats


@pytest.mark.parametrize("name,n,eps,kw", [
    ("SC105", 700, 1e-2, {}), ("ADLITTLE", 500, 1e-2, {}), ("AFIRO", 400, 1e-2, {}),
    ("SC105", 300, 0.0, {}),                      # every replica IS the leader: nobody leaves the path
    ("SC105", 300, 0.9, {}),                      # wild right-hand sides: forks from the first steps on
    ("ADLITTLE", 300, 1e-2, {"max_pivots": 20}),  # the leader ends "cycled" on its budget, in phase 1 or 2
    ("ADLITTLE", 300, 1e-2, {"max_pivots": 61}),
    ("SC105", 300, 1e-3, {"precision": 1e-6}),
    ("KLEIN1", 200, 1e-2, {}),                    # an infeasible leader
])
def test_replica_path_sharing_is_bit_exact(engine, name, n, eps, kw):
    """yalps_solve_replicas with path sharing (the replicas follow the recorded trace of the base tableau with their RHS
    column only and continue alone from the leader's snapshot where they would choose differently) against the oracle's
    solve of every replica on its own: every output, bit for bit -- and against the same call with sharing off."""
    g = load_netlib().get(name)
    H, W = g["height"], g["width"]
    base = g["matrix"]
    rhs, mats = _replica_case(base, H, W, n, eps, 11)
    opt = E.make_options(**kw)
    got = engine.solve_replicas(base, rhs, H, W, opt)
    forks = engine.replica_forks
    assert forks >= 0, "path sharing was not used"
    if eps == 0.0:
        assert forks == 0
    work = mats.copy()
    exp = O.simplex_batch(work, W, H, **kw)
    for k in ("status", "pivots", "pos", "var"):
        assert np.array_equal(got[k], exp[k]), (name, k, forks)
    assert same_bits(got["rhs"], exp["rhs"]), (name, forks)
    nan = np.isnan(exp["value"])
    assert np.array_equal(np.isnan(got["value"]), nan) and same_bits(got["value"][~nan], exp["value"][~nan])
    engine.set_replica_sharing(False)
    try:
        off = engine.solve_replicas(base, rhs, H, W, opt)
        assert engine.replica_forks == -1
    finally:
        engine.set_replica_sharing(True)
    for k in ("status", "pivots", "pos", "var"):
        assert np.array_equal(got[k], off[k]), k
    assert same_bits(got["rhs"], off["rhs"])


def test_replica_path_sharing_synthetic_phase2_and_statuses(engine):
    """A dense synthetic base (phase 2 only; perturbed replicas fork in the ratio test), an unbounded one, and a base whose
    trace does not fit the snapshot memory (KB-size trace capacity is exercised through a huge pivot budget)."""
    for (m_, nv, neg, n, eps) in ((20, 30, 0, 400, 1e-2), (40, 60, 8, 300, 5e-2), (12, 9, 3, 300, 0.3)):
        H, W = m_ + 1, nv + 1
        base = O.generate_synthetic(900 + m_, 1, m_, nv, neg)[0]
        rhs, mats = _replica_case(base, H, W, n, eps, 3)
        got = engine.solve_replicas(base, rhs, H, W)
        assert engine.replica_forks >= 0
        exp = O.simplex_batch(mats.copy(), W, H)
        for k in ("status", "pivots", "pos", "var"):
            assert np.array_equal(got[k], exp[k]), (m_, k)
        assert same_bits(got["rhs"], exp["rhs"])
    base = np.array([[0.0, 1.0, 1.0], [4.0, -1.0, 1.0], [2.0, -2.0, 1.0]]).reshape(-1)  # unbounded along column 1
    rhs = np.array([[0.0, 4.0, 2.0], [0.0, 1.0, 7.0], [0.0, -3.0, 2.0], [0.0, 4.0, -2.0]])
    mats = np.tile(base, (4, 1))
    mats.reshape(4, 3, 3)[:, :, 0] = rhs
    got = engine.solve_replicas(base, rhs, 3, 3)
    exp = O.simplex_batch(mats.copy(), 3, 3)
    assert np.array_equal(got["status"], exp["status"]) and np.array_equal(got["pivots"], exp["pivots"])
    assert same_bits(got["rhs"], exp["rhs"]) and np.array_equal(got["pos"], exp["pos"])


def test_replicas_across_pipeline_chunks(engine):
    """10,000 replicas are solved in 8 pipeline chunks of 1,250 (a call of more than 8,192 LPs is cut in eighths), with
    path sharing on and off: every output equals the batch entry on the expanded tableaus bit for bit, the LPs on each
    side of every chunk boundary equal the oracle, and two ranks on one GPU give the same bits."""
    g = load_netlib().get("AFIRO")
    H, W = g["height"], g["width"]
    base = g["matrix"]
    n, per_chunk = 10000, (10000 + 7) // 8
    rhs, mats = _replica_case(base, H, W, n, 1e-2, 17)
    ref = engine.solve_batch(mats, H, W, want_duals=True)
    edges = np.array([b + d for b in range(per_chunk, n, per_chunk) for d in (-1, 0)])
    work = mats[edges].copy()
    exp = O.simplex_batch(work, W, H)
    exp["reduced"] = np.stack([reduced_from_tableau(work[i], W, H, exp["pos"][i]) for i in range(edges.size)])
    ints, floats = ("status", "pivots", "pos", "var"), ("value", "rhs", "reduced")
    for sharing in (True, False):
        engine.set_replica_sharing(sharing)
        try:
            got = engine.solve_replicas(base, rhs, H, W, want_duals=True)
            forks = engine.replica_forks
        finally:
            engine.set_replica_sharing(True)
        assert forks >= 0 if sharing else forks == -1
        for k in ints:
            assert np.array_equal(got[k], ref[k]) and np.array_equal(got[k][edges], exp[k]), (sharing, k)
        for k in floats:
            assert same_bits(got[k], ref[k]), (sharing, k)
        assert same_bits(got["rhs"][edges], exp["rhs"]) and same_bits(got["reduced"][edges], exp["reduced"]), sharing
        assert all(same_value(a, b) for a, b in zip(got["value"][edges], exp["value"])), sharing
    with yalps_b200.MultiEngine([0, 0]) as me:
        many = me.solve_replicas(base, rhs, H, W, want_duals=True)
    for k in ints:
        assert np.array_equal(many[k], got[k]), k
    for k in floats:
        assert same_bits(many[k], got[k]), k


# ------------------------------------------------------------------------------------------------ several GPUs, one process
def rank_devices():
    import torch
    n = torch.cuda.device_count()
    return list(range(n)) if n >= 2 else [0, 0]  # one GPU: two logical ranks on it


@pytest.fixture(scope="module")
def multi():
    m = yalps_b200.MultiEngine(rank_devices())
    yield m
    m.close()


def test_multi_batch_equals_one_gpu_bit_for_bit(engine, multi):
    for (m_, nv, neg, n) in ((32, 64, 4, 2001), (12, 20, 3, 7), (80, 100, 10, 150)):
        mats = O.generate_synthetic(31000, n, m_, nv, neg)
        one = engine.solve_batch(mats, m_ + 1, nv + 1, want_matrices=True)
        many = multi.solve_batch(mats, m_ + 1, nv + 1, want_matrices=True)
        for k in ("status", "pivots", "pos", "var"):
            assert np.array_equal(one[k], many[k]), k
        for k in ("value", "rhs", "matrices"):
            assert same_bits(one[k], many[k]), k
    exp = O.simplex_batch(mats[:32].copy(), nv + 1, m_ + 1)
    assert np.array_equal(many["status"][:32], exp["status"]) and same_bits(many["rhs"][:32], exp["rhs"])


def test_multi_fewer_lps_than_ranks_and_empty(multi):
    mats = O.generate_synthetic(1, 1, 6, 9, 2)
    out = multi.solve_batch(mats, 7, 10)
    exp = O.simplex_batch(mats.copy(), 10, 7)
    assert np.array_equal(out["status"], exp["status"]) and same_bits(out["rhs"], exp["rhs"])
    assert multi.solve_batch(np.zeros(0), 3, 4)["status"].shape == (0,)


def test_multi_basis_in_and_replicas(engine, multi):
    mats, pos, var = mid_trajectory_states(301, 32, 64, 6, 777, 3)
    one = engine.solve_batch(mats, 33, 65, pos_in=pos, var_in=var)
    many = multi.solve_batch(mats, 33, 65, pos_in=pos, var_in=var)
    assert np.array_equal(one["pos"], many["pos"]) and same_bits(one["rhs"], many["rhs"])
    g = load_netlib().get("ADLITTLE")
    H, W = g["height"], g["width"]
    rng = np.random.default_rng(9)
    rhs = np.tile(g["matrix"].reshape(H, W)[:, 0], (257, 1)) * (1.0 + 1e-2 * (2.0 * rng.random((257, H)) - 1.0))
    a, b = engine.solve_replicas(g["matrix"], rhs, H, W), multi.solve_replicas(g["matrix"], rhs, H, W)
    assert np.array_equal(a["pivots"], b["pivots"]) and same_bits(a["rhs"], b["rhs"]) and np.array_equal(a["pos"], b["pos"])


def test_multi_ragged_equals_one_gpu(engine, multi):
    rng = np.random.default_rng(3)
    shapes, tabs = [], []
    for i in range(40):
        m_, nv = int(rng.integers(2, 40)), int(rng.integers(2, 70))
        tabs.append(O.generate_synthetic(500 + i, 1, m_, nv, int(rng.integers(0, m_ // 2 + 1)))[0])
        shapes.append((m_ + 1, nv + 1))
    one = engine.solve_ragged(tabs, shapes, want_matrices=True)
    many = multi.solve_ragged(tabs, shapes, want_matrices=True)
    for a, b in zip(one, many):
        assert a["status"] == b["status"] and a["pivots"] == b["pivots"] and same_value(a["value"], b["value"])
        assert np.array_equal(a["pos"], b["pos"]) and same_bits(a["rhs"], b["rhs"]) and same_bits(a["matrix"], b["matrix"])


def test_incumbent_allreduce_is_a_min_over_ranks(multi):
    w = multi.size
    vals = [7.5 - r for r in range(w)]
    assert multi.incumbent_allreduce(vals).tolist() == [min(vals)] * w
    vals = [math.inf] * w
    assert multi.incumbent_allreduce(vals).tolist() == vals
    vals = [math.nan] + [3.25] * (w - 1)  # NaN = "no incumbent on this rank"
    assert multi.incumbent_allreduce(vals).tolist() == [3.25] * w
    assert multi.launch_count >= 6


@pytest.mark.parametrize("name", ["Knapsack 1", "Fancy Stock Cutting Problem", "Large Farm MIP", "Monster 2",
                                  "Vendor Selection"])
def test_sharded_frontier_reproduces_the_single_gpu_search(multi, name):
    case = next(c for c in CASES if c["name"] == name)
    o = case["oracle"]
    info = {}
    sol = yalps_b200.solve(case["model"], case["options"], engine=multi, info=info)
    assert sol["status"] == o["status"] and same_value(sol["result"], o["result"])
    assert [list(v) for v in sol["variables"]] == [list(v) for v in o["variables"]]
    assert info["nodes"] == o["nodes"] and info["node_pivots"] == o["node_pivots"]
    assert np.array_equal(info["final_pos"], o["final_pos"]) and same_bits(info["final_rhs"], o["final_rhs"])
    if name in ("Monster 2", "Vendor Selection"):  # nodes beyond one SM's shared memory: every multi-node wave is dealt
        assert info["sharded_waves"] >= 1
    if info["waves"] >= 4:
        assert info["allreduces"] >= 1


def test_solve_many_on_several_gpus_equals_solve(multi):
    default = [c for c in CASES if not c["options"] and c["name"] not in ("Monster 2", "Vendor Selection")]
    sols = yalps_b200.solve_many([c["model"] for c in default], engine=multi)
    for c, s in zip(default, sols):
        assert s["status"] == c["oracle"]["status"] and same_value(s["result"], c["oracle"]["result"]), c["name"]
        assert [list(v) for v in s["variables"]] == [list(v) for v in c["oracle"]["variables"]], c["name"]


# ------------------------------------------------------------------------------- one large LP over the ranks (8f-3)
def _large_equal(got, exp, what):
    assert got["status"] == int(exp["status"][0]), what
    assert same_value(got["value"], exp["value"][0]), what
    assert got["pivots"] == tuple(int(x) for x in exp["pivots"][0]), what
    assert np.array_equal(got["pos"], exp["pos"][0]) and np.array_equal(got["var"], exp["var"][0]), what
    assert same_bits(got["rhs"], exp["rhs"][0]), what


def _oracle_one(mats, H, W, **kw):
    work = mats.copy()
    exp = O.simplex_batch(work, W, H, **kw)
    exp["matrices"] = work
    return exp


@pytest.mark.parametrize("m_,nv,neg", [(32, 64, 6), (5, 3, 2), (100, 300, 40), (300, 90, 100), (1, 1, 0), (0, 4, 0)])
def test_large_lp_over_the_ranks_is_bit_exact(multi, m_, nv, neg):
    """yalps_multi_solve_large: rows dealt round robin over the ranks, pivot row / column exchanged through peer memory
    from inside one persistent kernel per rank -- every output bit against the oracle, final tableau included."""
    H, W = m_ + 1, nv + 1
    mats = O.generate_synthetic(4100, 1, m_, nv, neg) if m_ else np.array([[0.0, 1.0, -2.0, 0.0, 3.0]])
    exp = _oracle_one(mats, H, W)
    got = multi.solve_large(mats, H, W, want_matrix=True)
    _large_equal(got, exp, f"large {H}x{W}")
    assert same_bits(got["matrix"], exp["matrices"].reshape(-1)), "final tableau"
    assert got["kernel_ms"] > 0.0


def test_large_lp_statuses_budgets_and_check_cycles(multi):
    t = np.array([[0, 10, -57, -9, -24], [0, 0.5, -5.5, -2.5, 9], [0, 0.5, -1.5, -0.5, 1], [1, 1, 0, 0, 0]], float)
    for kw in ({"check_cycles": True}, {"check_cycles": False, "max_pivots": 9}, {"max_pivots": 0}, {"max_pivots": 2.5}):
        m = t.reshape(1, -1).copy()
        exp = _oracle_one(m, 4, 5, **kw)
        got = multi.solve_large(m, 4, 5, E.make_options(**kw), want_matrix=True)
        _large_equal(got, exp, f"large {kw}")
        assert same_bits(got["matrix"], exp["matrices"].reshape(-1))
    # infeasible and unbounded
    for mat, H, W in ((np.array([[0.0, 1.0], [-1.0, 1.0]]), 2, 2), (np.array([[0.0, 1.0, 1.0], [4.0, -1.0, 1.0]]), 2, 3)):
        exp = _oracle_one(mat.reshape(1, -1), H, W)
        got = multi.solve_large(mat, H, W)
        _large_equal(got, exp, f"large status {int(exp['status'][0])}")


def test_large_lp_netlib_and_more_ranks(engine):
    """Sparse Netlib models (row skip, long phase 1) over 2, 3 and 4 ranks: the rank count must not change a bit."""
    import torch
    ndev = torch.cuda.device_count()
    nl = load_netlib()
    for world in (2, 3, 4):
        devs = [i % ndev for i in range(world)]
        with yalps_b200.MultiEngine(devs) as me:
            for name in ("AFIRO", "SC105", "ADLITTLE"):
                g = nl.get(name)
                got = me.solve_large(g["matrix"], g["height"], g["width"], E.make_options(check_cycles=g["check_cycles"]))
                assert got["status"] == g["status"] and got["pivots"] == g["pivots"], (name, world)
                assert same_value(got["value"], g["value"]) and np.array_equal(got["pos"], g["final_pos"])
                assert same_bits(got["rhs"], g["final_rhs"]), (name, world)
            mats = O.generate_synthetic(77, 1, 200, 500, 30)
            exp = _oracle_one(mats, 201, 501)
            _large_equal(me.solve_large(mats, 201, 501), exp, f"200x500 on {world} ranks")


def test_large_lp_equals_the_grid_kernel_at_size(engine, multi):
    """1025 x 2049 (16.8 MB), 40 pivots: the multi-rank kernel against the single-GPU grid kernel and the oracle."""
    import torch
    m_, nv, cap = 1024, 2048, 40
    H, W = m_ + 1, nv + 1
    d = torch.empty(H * W, dtype=torch.float64, device="cuda")
    engine.generate_synthetic_device(0, 1, m_, nv, d.data_ptr())
    torch.cuda.synchronize()
    mats = d.cpu().numpy().reshape(1, -1)
    opt = E.make_options(max_pivots=cap)
    exp = _oracle_one(mats, H, W, max_pivots=cap)
    got = multi.solve_large(mats, H, W, opt, want_matrix=True)
    _large_equal(got, exp, "1025x2049")
    assert same_bits(got["matrix"], exp["matrices"].reshape(-1))
    one = engine.solve_batch(mats, H, W, opt, want_matrices=True)
    assert same_bits(one["matrices"][0], got["matrix"])
