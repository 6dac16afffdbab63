"""The kernels' exact-division fallbacks on the GPU: every kernel path, every k_simplex and cluster instantiation, the
multi-GPU row split, the replica follower and the ranging / certificate passes run the batches of
tests/test_division_sites.py, whose trajectories reach every division site's fallback, and are compared with the oracle
bit for bit.  Each forced path is checked by kernel name under torch.profiler, so that a path that quietly took
another kernel cannot pass.

Floating-point outputs compare bit for bit, except that any NaN equals any NaN: the reference's arithmetic has one
NaN, and the payload of a NaN that inf - inf leaves need not be the same on the CPU and the GPU."""
import json
import math
import os
import re
import tempfile

import numpy as np
import pytest

import test_kernel_table as T
import yalps_b200
from oracle import lib as O
from test_division_sites import PRECISIONS, SHAPES, division_edge_batch
from test_gpu_boundary import rank_devices
from test_gpu_sensitivity import PATHS
from yalps_b200 import engine as E
from yalps_b200.sensitivity import certificate_from_tableau, ranges_from_tableau, reduced_from_tableau

pytestmark = pytest.mark.gpu

# the kernel family each forced path must launch (AUTO: whatever the rules choose)
FAMILY = {E.PATH_TMEM: "k_simplex_tmem", E.PATH_SMEM: "k_simplex", E.PATH_GMEM: "k_simplex",
          E.PATH_CLUSTER: "k_simplex_cluster", E.PATH_GRID_RESIDENT: "k_simplex_cluster", E.PATH_GRID: "k_simplex_grid"}
_KERNEL = re.compile(r"\b(k_\w+)(<[^>]*>)?")


class Kernels:
    """The kernels launched inside the block, by name: .families ("k_simplex_tmem", ...) and .names (with template
    arguments, "k_simplex<2,1,1,true>" as test_kernel_table.canonical_kernel_name writes the table kernels)."""

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
        self.families, self.names = set(), set()
        for ev in events:
            if ev.get("cat") != "kernel":
                continue
            raw = ev.get("name", "")
            m = _KERNEL.search(raw)
            if m:
                self.families.add(m.group(1))
                self.names.add(T.canonical_kernel_name(raw) or m.group(1))
        return False


def _bits_or_nan(a, b):
    a = np.ascontiguousarray(a, np.float64).reshape(-1)
    b = np.ascontiguousarray(b, np.float64).reshape(-1)
    if a.shape != b.shape:
        return -2
    bad = (a.view(np.uint64) != b.view(np.uint64)) & ~(np.isnan(a) & np.isnan(b))
    return int(np.flatnonzero(bad)[0]) if bad.any() else -1


def assert_same(got, exp, what, keys=("rhs", "matrices", "reduced")):
    assert np.array_equal(got["status"], exp["status"]), f"{what}: status {got['status']} != {exp['status']}"
    assert np.array_equal(np.asarray(got["pivots"]).reshape(-1, 2), np.asarray(exp["pivots"]).reshape(-1, 2)), \
        f"{what}: pivots"
    for k in ("pos", "var"):
        assert np.array_equal(np.asarray(got[k]).reshape(-1), np.asarray(exp[k]).reshape(-1)), f"{what}: {k}"
    for k in ("value",) + tuple(keys):
        i = _bits_or_nan(got[k], exp[k])
        if i != -1:
            g, x = np.asarray(got[k]).reshape(-1), np.asarray(exp[k]).reshape(-1)
            raise AssertionError(f"{what}: {k} differs" + (f" first at {i}: {g[i]!r} != {x[i]!r}" if i >= 0 else ""))


def oracle(mats, H, W, precision):
    work = np.ascontiguousarray(mats, np.float64).reshape(-1, H * W).copy()
    exp = O.simplex_batch(work, W, H, precision, nthreads=os.cpu_count() or 1)
    exp["matrices"] = work
    exp["reduced"] = np.stack([reduced_from_tableau(work[i], W, H, exp["pos"][i]) for i in range(work.shape[0])])
    return exp


_BATCHES = {}


def batch(H, W, precision):
    """The division_edge_batch of (H, W) (the seed of tests/test_division_sites.py) and its oracle outputs."""
    if (H, W, precision) not in _BATCHES:
        mats = division_edge_batch(H, W, 17 * W + H)
        _BATCHES[(H, W, precision)] = (mats, oracle(mats, H, W, precision))
    return _BATCHES[(H, W, precision)]


def solve(eng, mats, H, W, precision, **kw):
    return eng.solve_batch(mats, H, W, E.make_options(precision=precision), want_matrices=True, want_duals=True, **kw)


@pytest.fixture
def tuned(engine):
    yield engine
    engine.set_tuning(E.PATH_AUTO, 0, 0)


# ------------------------------------------------------------------------------------------------- every path
@pytest.mark.parametrize("precision", PRECISIONS, ids=["p1e-8", "p0"])
@pytest.mark.parametrize("name,path,threads,rows", PATHS, ids=[p[0] for p in PATHS])
def test_paths(tuned, name, path, threads, rows, precision):
    """Every kernel path of test_gpu_sensitivity at every shape it takes (a forced path that cannot take a shape
    fails with YALPS_ERR_TOO_LARGE; each path takes at least one)."""
    tuned.set_tuning(path, threads, rows)
    ran = 0
    for H, W in SHAPES:
        mats, exp = batch(H, W, precision)
        with Kernels() as K:
            try:
                got = solve(tuned, mats, H, W, precision)
            except E.YalpsError as err:
                assert err.code == T.TOO_LARGE and path != E.PATH_AUTO, (H, W, err)
                continue
        if path in FAMILY:
            assert FAMILY[path] in K.families, (H, W, K.families)
        assert_same(got, exp, f"{name} {H}x{W} precision {precision}")
        ran += 1
    assert ran, f"{name} took none of the shapes"


# ------------------------------------------------------------------------------------------- every instantiation
@pytest.mark.parametrize("p", T.SIMPLEX_ENTRIES, ids=T.entry_id)
def test_simplex_entry(tuned, p):
    """Each k_simplex entry in its layout at the widest width of its window: the fallback loops are unrolled per
    KC x VW, so every instantiation has its own copy."""
    e, resident = p
    prev, cap = T.simplex_window(e, 2 if resident else 1)
    optin = tuned.device_info()["smem_per_block_optin"]
    W = cap + 1
    H = min(40, T.tallest_height(e, resident, W, optin))
    if H < 2:  # only the objective row fits at the widest width: the widest width at which constraint rows do
        W = prev + 2
        H = min(40, T.tallest_height(e, resident, W, optin))
    tuned.set_tuning(*T.forcing(e, resident))
    want = T.simplex_name(e, resident)
    for precision in PRECISIONS:
        mats = division_edge_batch(H, W, 3 * W + H)
        with Kernels() as K:
            got = solve(tuned, mats, H, W, precision)
        assert {n for n in K.names if n.startswith("k_simplex")} == {want}, K.names
        assert_same(got, oracle(mats, H, W, precision), f"{want} {H}x{W} precision {precision}")


@pytest.mark.parametrize("case", T.cluster_cases(), ids=lambda c: f"{T.cluster_name(c[0], False)}-{c[2]}x{c[1]}-C{c[3]}")
def test_cluster_entry(tuned, case):
    """Each KC entry at each of its test_kernel_table shapes, once."""
    e, W, H, C = case
    tuned.set_tuning(E.PATH_CLUSTER, 0)
    want = T.cluster_name(e, False)
    mats = division_edge_batch(H, W, 5 * W + H)
    for precision in PRECISIONS:
        with Kernels() as K:
            got = solve(tuned, mats, H, W, precision)
        assert want in K.names, K.names
        assert_same(got, oracle(mats, H, W, precision), f"{want} {H}x{W} precision {precision}")


# ------------------------------------------------------------------------------------------------ K4m, replicas
def test_solve_large_two_ranks():
    """K4m: one LP with its rows dealt over two ranks (two GPUs, or two logical ranks on one), final matrix too."""
    multi = yalps_b200.MultiEngine(rank_devices())
    try:
        for H, W in ((65, 65), (201, 261)):
            for precision in PRECISIONS:
                mats, exp = batch(H, W, precision)
                for i in range(mats.shape[0]):
                    got = multi.solve_large(mats[i], H, W, E.make_options(precision=precision), want_matrix=True)
                    one = {"status": np.array([got["status"]]), "value": np.array([got["value"]]),
                           "pivots": np.array(got["pivots"]), "pos": got["pos"], "var": got["var"], "rhs": got["rhs"],
                           "matrices": got["matrix"]}
                    ref = {k: np.atleast_1d(exp[k][i]) for k in exp}
                    assert_same(one, ref, f"solve_large {H}x{W} LP {i} precision {precision}", keys=("rhs", "matrices"))
    finally:
        multi.close()


REPLICA_RHS = (0.0, -0.0, 1e-320, -1e-320, 1e-300, 1e-15, math.inf, -math.inf, math.nan, -1e307)


@pytest.mark.parametrize("sharing", [True, False], ids=["shared", "solo"])
def test_replicas(engine, sharing):
    """Replicas of bases whose own trajectories pass through fallback divisions, with right-hand sides perturbed to
    tiny, denormal, infinite and NaN values: the follower's ratio tests and RHS pivots, and the forks."""
    H, W = 33, 65
    mats, _ = batch(H, W, 1e-8)
    rng = np.random.default_rng(3)
    engine.set_replica_sharing(sharing)
    try:
        for i in range(0, mats.shape[0], 3):
            base = mats[i]
            b0 = base.reshape(H, W)[:, 0]
            n = 24
            rhs = np.repeat(b0[None, :], n, 0)
            for j in range(1, n):  # replica 0 is the base itself: the leader's path
                rows = rng.integers(0, H, 1 + j % 3)
                rhs[j, rows] = rng.choice(REPLICA_RHS, rows.size)
            full = np.repeat(base[None, :], n, 0).reshape(n, H, W).copy()
            full[:, :, 0] = rhs
            got = engine.solve_replicas(base, rhs, H, W, want_duals=True)
            exp = oracle(full.reshape(n, -1), H, W, 1e-8)
            assert_same(got, exp, f"replicas of LP {i} sharing={sharing}", keys=("rhs", "reduced"))
    finally:
        engine.set_replica_sharing(True)


# ------------------------------------------------------------------------------------------- ranging, certificates
@pytest.mark.parametrize("H,W", [(33, 65), (65, 65), (91, 131), (201, 261)], ids=lambda x: str(x))
def test_ranging_and_certificates(engine, H, W):
    """k_ranging (warp mode up to 256 x 128, tile mode beyond) and k_certificate on the final tableaus that are
    finite: through solve_batch, and ranging_device on the oracle's own final tableaus."""
    torch = pytest.importorskip("torch")
    for precision in PRECISIONS:
        mats, exp = batch(H, W, precision)
        fin = np.flatnonzero(np.isfinite(exp["matrices"]).all(axis=1))
        assert fin.size >= 10, fin.size
        got = engine.solve_batch(mats[fin], H, W, E.make_options(precision=precision), want_ranges=True,
                                 want_certificates=True)
        lo, hi, cert = [], [], []
        for i in fin:
            m, pos = exp["matrices"][i], exp["pos"][i]
            a, b = ranges_from_tableau(m, W, H, pos, precision, None, exp["status"][i] == 0)
            lo.append(a)
            hi.append(b)
            cert.append(certificate_from_tableau(m, W, H, pos, int(exp["status"][i]), float(exp["value"][i]), precision))
        lo, hi, cert = np.stack(lo), np.stack(hi), np.stack(cert)
        for k, x in (("range_lo", lo), ("range_hi", hi), ("certificate", cert)):
            assert _bits_or_nan(got[k], x) == -1, (H, W, precision, k)

        dev = torch.device("cuda:0")
        d_m = torch.from_numpy(np.ascontiguousarray(exp["matrices"][fin])).to(dev)
        d_pos = torch.from_numpy(np.ascontiguousarray(exp["pos"][fin])).to(dev)
        d_st = torch.from_numpy(np.ascontiguousarray(exp["status"][fin])).to(dev)
        d_lo = torch.full((fin.size, W + H), 7.0, dtype=torch.float64, device=dev)
        d_hi = torch.full((fin.size, W + H), 7.0, dtype=torch.float64, device=dev)
        engine.ranging_device(fin.size, H, W, d_m.data_ptr(), d_pos.data_ptr(), d_lo.data_ptr(), d_hi.data_ptr(),
                              precision=precision, d_status=d_st.data_ptr(),
                              stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert _bits_or_nan(d_lo.cpu().numpy(), lo) == -1 and _bits_or_nan(d_hi.cpu().numpy(), hi) == -1
