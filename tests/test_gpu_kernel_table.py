"""Every instantiation of the kernel tables, forced on the device and named: each `k_simplex` entry in both layouts,
each cluster entry as KC and as KG, each `k_bnb` config.  A call runs under torch.profiler (CUDA activities) and the
test asserts by kernel name that exactly the intended instantiation ran -- a forced path that quietly took another
kernel (a row-split entry at its capacity falls back to one row group) would otherwise still pass the parity checks.
The outputs are compared with the oracle bit for bit at the edges of each entry's shape class: both ends of its width
window, heights around its update-block height RU, and the tallest tableau its carve-up takes (tests/test_kernel_table.py
derives all of them from the tables).  The last test is the ledger: every parsed instantiation must have been seen."""
import json
import math
import tempfile

import numpy as np
import pytest

import test_kernel_table as T
import yalps_b200
from conftest import same_bits, same_value
from oracle import lib as O, model as M
from yalps_b200 import engine as E
from yalps_b200.sensitivity import reduced_from_tableau

pytestmark = pytest.mark.gpu

SEEN = set()  # canonical names of every table kernel the profiler saw in this module (the ledger)


@pytest.fixture
def tuned(engine):
    yield engine
    engine.set_tuning(E.PATH_AUTO, 0, 0)
    engine.set_bnb_mode(0)


class Launches:
    """Profiles the block: .names = canonical names of the table kernels launched in it (any other simplex-family
    kernel -- K1t, K4 -- under its raw name, so that an exact comparison fails), .grids = {name: set of grid sizes}."""

    def __enter__(self):
        import torch
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.synchronize()
        self.prof = profile(activities=[ProfilerActivity.CUDA])
        self.prof.__enter__()
        return self

    def __exit__(self, *exc):
        import torch
        torch.cuda.synchronize()
        self.prof.__exit__(*exc)
        with tempfile.NamedTemporaryFile(suffix=".json") as f:
            self.prof.export_chrome_trace(f.name)
            with open(f.name) as g:
                events = json.load(g)["traceEvents"]
        self.names, self.grids = set(), {}
        for ev in events:
            if ev.get("cat") != "kernel":
                continue
            raw = ev.get("name", "")
            name = T.canonical_kernel_name(raw) or (raw if ("k_simplex" in raw or "k_bnb" in raw) else None)
            if name:
                self.names.add(name)
                g = ev.get("args", {}).get("grid")
                self.grids.setdefault(name, set()).add(g[0] if isinstance(g, list) else g)
        SEEN.update(n for n in self.names if n in set(T.all_instantiations()))
        return False


def assert_same(got, exp, what):
    assert np.array_equal(got["status"], exp["status"]), f"{what}: status {got['status']} != {exp['status']}"
    assert np.array_equal(np.asarray(got["pivots"]).reshape(-1, 2), np.asarray(exp["pivots"]).reshape(-1, 2)), f"{what}: pivots"
    gv, ev = np.asarray(got["value"]), np.asarray(exp["value"])
    assert np.array_equal(np.isnan(gv), np.isnan(ev)) and same_bits(gv[~np.isnan(gv)], ev[~np.isnan(ev)]), f"{what}: value"
    assert np.array_equal(got["pos"].reshape(-1), exp["pos"].reshape(-1)), f"{what}: pos"
    assert np.array_equal(got["var"].reshape(-1), exp["var"].reshape(-1)), f"{what}: var"
    assert same_bits(got["rhs"].reshape(-1), exp["rhs"].reshape(-1)), f"{what}: rhs"
    g, x = got["matrices"].reshape(-1), exp["matrices"].reshape(-1)
    if not same_bits(g, x):
        k = int(np.flatnonzero(g.view(np.uint64) != x.view(np.uint64))[0])
        raise AssertionError(f"{what}: final tableau, first differing cell {k}: {g[k]!r} != {x[k]!r}")
    assert same_bits(got["reduced"].reshape(-1), exp["reduced"].reshape(-1)), f"{what}: reduced"


def solve(eng, mats, H, W, opt=None, **kw):
    return eng.solve_batch(mats, H, W, opt, want_matrices=True, want_duals=True, **kw)


def oracle_from_basis(mats, pos, var, H, W):
    """O.simplex on every LP from its own basis (the node LPs of src/branchAndCut.ts:127)."""
    m, p, v = mats.copy(), pos.copy(), var.copy()
    res = [O.simplex(m[i], W, H, p[i], v[i]) for i in range(m.shape[0])]
    return {"status": np.array([r[0] for r in res], np.int32), "value": np.array([r[1] for r in res]),
            "pivots": np.array([r[2] for r in res], np.int64), "rhs": m.reshape(-1, H, W)[:, :, 0].copy(), "pos": p,
            "var": v, "matrices": m,
            "reduced": np.stack([reduced_from_tableau(m[i], W, H, p[i]) for i in range(m.shape[0])])}


def mid_trajectory(H, W, seed, n=6, k=2):
    """edge_batch LPs the oracle stopped after at most k pivots per phase: a non-identity basis to resume from."""
    mats = T.edge_batch(H, W, seed, n)
    pos = np.tile(np.arange(W + H, dtype=np.int32), (n, 1))
    var = pos.copy()
    for i in range(n):
        O.simplex(mats[i], W, H, pos[i], var[i], max_pivots=k)
    return mats, pos, var


# ------------------------------------------------------------------------------------------------ k_simplex
@pytest.mark.parametrize("p", T.SIMPLEX_ENTRIES, ids=T.entry_id)
def test_simplex_entry(tuned, monkeypatch, p):
    """One entry of the k_simplex table in one layout, forced with set_tuning(path, NWC*NWR*32, NWR): every edge shape,
    a maxPivots budget, checkCycles with the Chvatal LP, a caller-supplied mid-trajectory basis, the atomic LP queue,
    and the tallest tableau -- all on exactly this instantiation; one row more runs what the host rules say."""
    e, resident = p
    eng = tuned
    info = eng.device_info()
    optin, sms = info["smem_per_block_optin"], info["sm_count"]
    c = T.simplex_cases(e, resident, optin)
    want = T.simplex_name(e, resident)
    path, threads, rows = T.forcing(e, resident)
    eng.set_tuning(path, threads, rows)

    with Launches() as L:
        for H, W in c["shapes"]:
            mats = T.edge_batch(H, W, 17 * W + H)
            assert_same(solve(eng, mats, H, W), T.oracle_batch(mats, H, W), f"{want} {H}x{W}")
        H, W = T.budget_shape(c)
        mats = T.edge_batch(H, W, 5)
        assert_same(solve(eng, mats, H, W, E.make_options(max_pivots=2)), T.oracle_batch(mats, H, W, max_pivots=2),
                    f"{want} {H}x{W} maxPivots=2")
        H, W = T.cycle_shape(e, resident)
        mats = T.chvatal_batch(H, W, 3)
        assert_same(solve(eng, mats, H, W, E.make_options(check_cycles=True)),
                    T.oracle_batch(mats, H, W, check_cycles=True), f"{want} {H}x{W} checkCycles")
        H, W = c["shapes"][0]
        mats, pos, var = mid_trajectory(H, W, 7 * W + H)
        assert_same(solve(eng, mats, H, W, pos_in=pos, var_in=var), oracle_from_basis(mats, pos, var, H, W),
                    f"{want} {H}x{W} basis in")
    assert L.names == {want}, L.names

    # more LPs than CTAs: the persistent CTAs pull LPs from the atomic queue
    monkeypatch.setenv("YALPS_CTAS_PER_SM", "1")
    H, W = T.queue_shape(c)
    mats = T.edge_batch(H, W, 11, sms + 7)
    with Launches() as L:
        got = solve(eng, mats, H, W)
    assert L.names == {want} and L.grids[want] == {sms}, (L.names, L.grids)
    assert_same(got, T.oracle_batch(mats, H, W), f"{want} {H}x{W} queue")
    monkeypatch.delenv("YALPS_CTAS_PER_SM")

    # the tallest tableau the forced path takes, and one row more
    tall, W = c["tall"]
    for H in (tall, tall + 1):
        mats = T.tall_tableau(H, W, H)
        route = T.forced_route(path, threads, rows, H, W, optin)
        with Launches() as L:
            try:
                got = solve(eng, mats, H, W)
            except E.YalpsError as err:
                got = err
        if route == T.TOO_LARGE:
            assert H == tall + 1 and isinstance(got, E.YalpsError) and got.code == T.TOO_LARGE, got
            assert not L.names
            continue
        assert not isinstance(got, Exception), got
        assert L.names == {route[0]}, (H, W, L.names, route)
        assert (route[0] == want) == (H == tall)
        assert_same(got, T.oracle_batch(mats, H, W), f"{route[0]} {H}x{W} tall")
        del got, mats


# ------------------------------------------------------------------------------------------------ KC and KG
@pytest.mark.parametrize("case", T.cluster_cases(), ids=lambda c: f"{T.cluster_name(c[0], False)}-{c[2]}x{c[1]}-C{c[3]}")
def test_cluster_entry(tuned, case):
    """KC (PATH_CLUSTER) at both edges of each cluster entry's width window, with every cluster size 2, 4, 8, 16."""
    e, W, H, C = case
    eng = tuned
    n = 5
    mats = T.edge_batch(H, W, 31 * W + H, n)
    eng.set_tuning(E.PATH_CLUSTER, 0)
    with Launches() as L:
        got = solve(eng, mats, H, W)
    want = T.cluster_name(e, False)
    assert L.names == {want}, L.names
    (grid,) = L.grids[want]
    assert grid % C == 0 and (C == 16 or grid == n * C), (grid, C)
    assert_same(got, T.oracle_batch(mats, H, W), f"{want} {H}x{W}")


KG_CASES = [(e, W) for i, e in enumerate(T.cluster_table())
            for W in (T.first_covering_window(T.cluster_table(), i)[0] + 2, T.first_covering_window(T.cluster_table(), i)[1] + 1)]


@pytest.mark.parametrize("case", KG_CASES, ids=lambda c: f"{T.cluster_name(c[0], True)}-W{c[1]}")
def test_grid_resident_entry(tuned, case):
    """KG (PATH_GRID_RESIDENT) at both edges of each entry's width window: one LP over min(SMs, H-1) CTAs."""
    e, W = case
    eng = tuned
    H = 40
    sms = eng.device_info()["sm_count"]
    plan = T.plan_gridres(H, W, eng.device_info()["smem_per_block_optin"], sms)
    assert plan is not None and plan[0] == e
    mats = T.edge_batch(H, W, 13 * W, 2)
    eng.set_tuning(E.PATH_GRID_RESIDENT, 0)
    with Launches() as L:
        got = solve(eng, mats, H, W)
    want = T.cluster_name(e, True)
    assert L.names == {want} and L.grids[want] == {plan[1]}, (L.names, L.grids)
    assert_same(got, T.oracle_batch(mats, H, W), f"{want} {H}x{W}")


# ------------------------------------------------------------------------------------------------ k_bnb
def _oracle_search(model, options):
    info = {}
    sol = M.solve(model, {**M.DEFAULT_OPTIONS, **options}, info)
    return sol, info


def _assert_same_search(sol, info, ref, rinfo, what):
    assert sol["status"] == ref["status"] and same_value(sol["result"], ref["result"]), what
    assert [list(v) for v in sol["variables"]] == [list(v) for v in ref["variables"]], what
    assert info["nodes"] == rinfo["nodes"] and info["node_pivots"] == rinfo["node_pivots"], what
    assert np.array_equal(info["final_pos"], rinfo["final_pos"]), what
    assert same_bits(info["final_rhs"], rinfo["final_rhs"]), what


@pytest.mark.parametrize("name,nv,nc,seed,iters", [c for c in T.BNB_CASES if c[0] != "deep"], ids=lambda x: str(x))
def test_bnb_config(tuned, name, nv, nc, seed, iters):
    """The wider device-resident search configs: the whole search in one launch of k_bnb<4,1,4> (W <= 257) or
    k_bnb<4,2,4> (W <= 513), and the host wave driver, node for node against the oracle."""
    eng = tuned
    model, options = T.knapsack_milp(nv, nc, seed, iters)
    ref, rinfo = _oracle_search(model, options)
    want = name.replace("bnb", "k_bnb")
    for mode in (2, 1):
        eng.set_bnb_mode(mode)
        info = {}
        with Launches() as L:
            sol = yalps_b200.solve(model, options, engine=eng, info=info)
        _assert_same_search(sol, info, ref, rinfo, f"{name} mode {mode}")
        if mode == 2:
            assert info["waves"] == 1 and want in L.names, (info["waves"], L.names)
        else:
            assert not any(n.startswith("k_bnb") for n in L.names), L.names


def test_bnb_cut_depth_beyond_the_device_capacity(tuned):
    """A search whose cut depth passes the cut rows the device kernel can hold at its width (bnb.inl:464-467): in the
    default mode the device search gives up and the wave driver repeats it -- still the oracle's search."""
    eng = tuned
    name, nv, nc, seed, iters = next(c for c in T.BNB_CASES if c[0] == "deep")
    model, options = T.knapsack_milp(nv, nc, seed, iters)
    ref, rinfo = _oracle_search(model, options)
    tm = M.tableau_model(model)
    capacity = T.bnb_cut_capacity(tm.tableau.height, tm.tableau.width, len(tm.integers),
                                  eng.device_info()["smem_per_block_optin"])
    assert capacity is not None and rinfo["max_cuts"] > capacity
    eng.set_bnb_mode(0)
    info = {}
    with Launches() as L:
        sol = yalps_b200.solve(model, options, engine=eng, info=info)
    _assert_same_search(sol, info, ref, rinfo, "deep")
    assert T.bnb_name(T.bnb_config_for(tm.tableau.width)) in L.names and info["waves"] > 1, (L.names, info["waves"])


def test_bnb_narrowest_config(tuned):
    """k_bnb<2,1,4> (W <= 129) on a golden MILP, so that the ledger covers the whole B&B table."""
    from conftest import load_cases
    case = next(c for c in load_cases() if c["name"] == "Large Farm MIP")
    ref, rinfo = _oracle_search(case["model"], case["options"])
    tuned.set_bnb_mode(2)
    info = {}
    with Launches() as L:
        sol = yalps_b200.solve(case["model"], case["options"], engine=tuned, info=info)
    _assert_same_search(sol, info, ref, rinfo, "Large Farm MIP")
    assert "k_bnb<2,1,4>" in L.names and info["waves"] == 1


# ------------------------------------------------------------------------------------------------ ledger
def test_ledger_every_instantiation_ran():
    """Runs last in this module: every instantiation parsed from the tables was seen by the profiler above."""
    missing = [n for n in T.all_instantiations() if n not in SEEN]
    assert not missing, f"{len(missing)} of {len(T.all_instantiations())} instantiations never ran: {missing}"
