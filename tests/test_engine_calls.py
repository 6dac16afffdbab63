"""Engine and MultiEngine batch calls against a fake libyalps_b200 (no GPU): which C entry each call reaches, with which
arguments and NULLs, and how the outputs the entry writes come back to the caller."""
import ctypes as C
import itertools

import numpy as np
import pytest

import yalps_b200
from yalps_b200 import _ffi

CTX, MULTI = 0x1000, 0x2000

# Output arguments of the widest batch entries (include/yalps_b200.h), with the input `pairs` in its place.
WIDE = ["status", "value", "pivots", "rhs", "pos", "var", "matrices", "reduced", "pairs", "range_lo", "range_hi",
        "certificate"]
# argument name -> (dtype, what one value is counted per): outputs and array inputs of the entries below
ARRAYS = {
    "status": (np.int32, "lp"), "value": (np.float64, "lp"), "pivots": (np.int64, "lp2"), "rhs": (np.float64, "row"),
    "pos": (np.int32, "var"), "var": (np.int32, "var"), "matrices": (np.float64, "cell"),
    "reduced": (np.float64, "var"), "range_lo": (np.float64, "var"), "range_hi": (np.float64, "var"),
    "certificate": (np.float64, "var"),
    "matrices_in": (np.float64, "cell"), "pos_in": (np.int32, "var"), "var_in": (np.int32, "var"),
    "pairs": (np.int32, "row"), "heights": (np.int32, "lp"), "widths": (np.int32, "lp"),
    "mat_offsets": (np.int64, "lp"), "base": (np.float64, "one"), "rhs_in": (np.float64, "row"),
    "cells": (np.int32, "nnz"), "values": (np.float64, "nnz"),
}
OUTPUTS = [k for k in ARRAYS if k in WIDE and k != "pairs"]
LAYOUTS = {
    "yalps_solve_batch_certificate": ["n", "h", "w", "matrices_in", "pos_in", "var_in", "opt"] + WIDE,
    "yalps_multi_solve_batch_certificate": ["n", "h", "w", "matrices_in", "pos_in", "var_in", "opt"] + WIDE,
    "yalps_solve_ragged_certificate": ["n", "heights", "widths", "mat_offsets", "matrices_in", "pos_in", "var_in",
                                       "opt"] + WIDE,
    "yalps_multi_solve_ragged_certificate": ["n", "heights", "widths", "mat_offsets", "matrices_in", "opt"] + WIDE,
    "yalps_solve_replicas_duals": ["n", "h", "w", "base", "rhs_in", "opt", "status", "value", "pivots", "rhs", "pos",
                                   "var", "reduced"],
    "yalps_multi_solve_replicas_duals": ["n", "h", "w", "base", "rhs_in", "opt", "status", "value", "pivots", "rhs",
                                         "pos", "var", "reduced"],
    "yalps_solve_sparse_certificate": ["h", "w", "nnz", "cells", "values", "opt", "status", "value", "pivots", "rhs",
                                       "pos", "var", "reduced", "pairs", "range_lo", "range_hi", "certificate"],
}


def pattern(name: str, count: int) -> np.ndarray:
    """What the fake writes to output `name`: distinct values per output and per element."""
    return (np.arange(count) + 1000 * (OUTPUTS.index(name) + 1)).astype(ARRAYS[name][0])


def addr(arg) -> int:
    return C.addressof(arg._obj) if type(arg).__name__ == "CArgObject" else arg.value


class FakeLib:
    """Records every batch call (entry, handle, scalars, input bytes, and which outputs are NULL) and fills each output
    with pattern(), sized from the call's own scalars and shape arrays."""

    def __init__(self):
        self.calls = []
        self.pinned = []

    def yalps_create(self, device, out):
        out._obj.value = CTX
        return 0

    def yalps_create_multi(self, devices, ndev, out):
        out._obj.value = MULTI
        return 0

    def yalps_host_alloc(self, ctx, n, out):
        self.pinned.append(C.create_string_buffer(max(n, 1)))
        out._obj.value = C.addressof(self.pinned[-1])
        return 0

    def __getattr__(self, name):
        if name in LAYOUTS:
            return lambda handle, *args: self._batch(name, handle, args)
        if name.startswith("yalps_destroy"):
            return lambda *a: None
        if name.endswith("last_error"):
            return lambda *a: b"fake"
        raise AttributeError(name)

    def _batch(self, name, handle, args):
        a = dict(zip(LAYOUTS[name], args))
        assert len(args) == len(LAYOUTS[name])
        n = a.get("n", 1)
        if "heights" in a:
            hs = np.frombuffer(C.string_at(addr(a["heights"]), 4 * n), np.int32).astype(np.int64)
            ws = np.frombuffer(C.string_at(addr(a["widths"]), 4 * n), np.int32).astype(np.int64)
        else:
            hs, ws = np.full(n, a["h"]), np.full(n, a["w"])
        count = {"lp": n, "lp2": 2 * n, "row": int(hs.sum()), "var": int((hs + ws).sum()),
                 "cell": int((hs * ws).sum()), "one": int(hs[0] * ws[0]) if n else 0, "nnz": a.get("nnz", 0)}
        rec = {"fn": name, "handle": {CTX: "ctx", MULTI: "multi"}[handle.value], "args": []}
        for role, v in a.items():
            if role not in ARRAYS:
                rec["args"].append((role, bytes(v._obj) if role == "opt" else v))
            elif v is None:
                rec["args"].append((role, None))
            else:
                dtype, per = ARRAYS[role]
                nbytes = count[per] * np.dtype(dtype).itemsize
                if role in OUTPUTS:
                    C.memmove(addr(v), pattern(role, count[per]).ctypes.data, nbytes)
                    rec["args"].append((role, ("out", nbytes)))
                else:
                    rec["args"].append((role, C.string_at(addr(v), nbytes)))
        self.calls.append(rec)
        return 0


@pytest.fixture
def fake(monkeypatch):
    lib = FakeLib()
    monkeypatch.setattr(_ffi, "load", lambda: lib)
    return lib


@pytest.fixture
def eng(fake):
    return yalps_b200.Engine(0)


@pytest.fixture
def multi(fake):
    return yalps_b200.MultiEngine([0, 0])


H, W, N = 3, 4, 5
PV = H + W
MATS = np.arange(N * H * W, dtype=np.float64)
PAIRS = np.array([-1, 2, 1], np.int32)
SHAPES = [(2, 3), (4, 2), (1, 5)]
TABS = [np.arange(h * w, dtype=np.float64) + 100 * i for i, (h, w) in enumerate(SHAPES)]
RAGGED_PAIRS = [np.array([-1, -1], np.int32), np.array([-1, 2, 1, -1], np.int32), np.array([-1], np.int32)]
RANGES = ("off", "on", "on+pairs")  # want_ranges without / with pairs


def nulls(rec) -> dict:
    return {role: v is None for role, v in rec["args"]}


@pytest.mark.parametrize("want_matrices,want_basis,want_duals,ranges,want_certificates",
                         list(itertools.product([False, True], [False, True], [False, True], RANGES, [False, True])))
def test_solve_batch_arguments(fake, eng, want_matrices, want_basis, want_duals, ranges, want_certificates):
    out = eng.solve_batch(MATS, H, W, want_matrices=want_matrices, want_basis=want_basis, want_duals=want_duals,
                          want_ranges=ranges != "off", pairs=PAIRS if ranges == "on+pairs" else None,
                          want_certificates=want_certificates)
    (rec,) = fake.calls
    assert rec["fn"] == "yalps_solve_batch_certificate" and rec["handle"] == "ctx"
    args = dict(rec["args"])
    assert (args["n"], args["h"], args["w"]) == (N, H, W)
    assert args["matrices_in"] == MATS.tobytes()
    assert args["pairs"] == (np.tile(PAIRS, N).tobytes() if ranges == "on+pairs" else None)
    assert nulls(rec) == {
        "n": False, "h": False, "w": False, "matrices_in": False, "pos_in": True, "var_in": True, "opt": False,
        "status": False, "value": False, "pivots": False, "rhs": False, "pos": not want_basis, "var": not want_basis,
        "matrices": not want_matrices, "reduced": not want_duals, "pairs": ranges != "on+pairs",
        "range_lo": ranges == "off", "range_hi": ranges == "off", "certificate": not want_certificates}
    # keys: the batch_outputs() set always (None when off); ranges and certificates only when asked for
    keys = ["status", "value", "pivots", "rhs", "pos", "var", "matrices", "reduced"]
    keys += ["range_lo", "range_hi"] if ranges != "off" else []
    keys += ["certificate"] if want_certificates else []
    assert list(out) == keys
    wanted = {"pos": want_basis, "var": want_basis, "matrices": want_matrices, "reduced": want_duals}
    size = {"lp": (N,), "lp2": (N, 2), "row": (N, H), "var": (N, PV), "cell": (N, H * W)}
    for k in keys:
        if not wanted.get(k, True):
            assert out[k] is None, k
            continue
        dtype, per = ARRAYS[k]
        assert out[k].dtype == dtype and out[k].shape == size[per], k
        assert np.array_equal(out[k].reshape(-1), pattern(k, out[k].size)), k


@pytest.mark.parametrize("want_matrices,want_duals,ranges,want_certificates",
                         list(itertools.product([False, True], [False, True], RANGES, [False, True])))
def test_engine_and_multi_pass_the_same_arguments(fake, eng, multi, want_matrices, want_duals, ranges,
                                                  want_certificates):
    kw = dict(want_matrices=want_matrices, want_duals=want_duals, want_ranges=ranges != "off",
              want_certificates=want_certificates)
    pos_in = np.tile(np.arange(PV, dtype=np.int32), N)
    eng.solve_batch(MATS, H, W, pos_in=pos_in, var_in=pos_in, pairs=PAIRS if ranges == "on+pairs" else None, **kw)
    multi.solve_batch(MATS, H, W, pos_in=pos_in, var_in=pos_in, pairs=PAIRS if ranges == "on+pairs" else None, **kw)
    eng.solve_ragged(TABS, SHAPES, pairs=RAGGED_PAIRS if ranges == "on+pairs" else None, **kw)
    multi.solve_ragged(TABS, SHAPES, pairs=RAGGED_PAIRS if ranges == "on+pairs" else None, **kw)
    eng.solve_replicas(MATS[:H * W], MATS[:N * H], H, W, want_duals=want_duals)
    multi.solve_replicas(MATS[:H * W], MATS[:N * H], H, W, want_duals=want_duals)
    e_batch, m_batch, e_rag, m_rag, e_rep, m_rep = fake.calls
    assert [c["fn"] for c in fake.calls] == [
        "yalps_solve_batch_certificate", "yalps_multi_solve_batch_certificate", "yalps_solve_ragged_certificate",
        "yalps_multi_solve_ragged_certificate", "yalps_solve_replicas_duals", "yalps_multi_solve_replicas_duals"]
    assert [c["handle"] for c in fake.calls] == ["ctx", "multi"] * 3
    assert e_batch["args"] == m_batch["args"]
    assert e_rep["args"] == m_rep["args"]
    # the single-GPU ragged entry also takes a basis, passed as NULL
    assert ("pos_in", None) in e_rag["args"] and ("var_in", None) in e_rag["args"]
    assert [a for a in e_rag["args"] if a[0] not in ("pos_in", "var_in")] == m_rag["args"]


@pytest.mark.parametrize("multi_engine", [False, True])
@pytest.mark.parametrize("want_matrices,want_duals,ranges,want_certificates",
                         list(itertools.product([False, True], [False, True], RANGES, [False, True])))
def test_solve_ragged_slices(fake, eng, multi, multi_engine, want_matrices, want_duals, ranges, want_certificates):
    e = multi if multi_engine else eng
    res = e.solve_ragged(TABS, SHAPES, want_matrices=want_matrices, want_duals=want_duals,
                         want_ranges=ranges != "off", pairs=RAGGED_PAIRS if ranges == "on+pairs" else None,
                         want_certificates=want_certificates)
    (rec,) = fake.calls
    args = dict(rec["args"])
    assert args["heights"] == np.array([h for h, _ in SHAPES], np.int32).tobytes()
    assert args["widths"] == np.array([w for _, w in SHAPES], np.int32).tobytes()
    assert args["mat_offsets"] == np.array([0, 6, 14], np.int64).tobytes()
    assert args["matrices_in"] == np.concatenate(TABS).tobytes()
    assert args["pairs"] == (np.concatenate(RAGGED_PAIRS).tobytes() if ranges == "on+pairs" else None)
    for role in ("range_lo", "range_hi"):
        assert (args[role] is None) == (ranges == "off")
    assert (args["certificate"] is None) == (not want_certificates)
    assert (args["reduced"] is None) == (not want_duals)
    assert (args["matrices"] is None) == (not want_matrices)
    keys = ["status", "value", "pivots", "rhs", "pos", "var", "matrix"]
    keys += ["reduced"] if want_duals else []
    keys += ["range_lo", "range_hi"] if ranges != "off" else []
    keys += ["certificate"] if want_certificates else []
    row = cell = pv = 0
    for i, ((h, w), r) in enumerate(zip(SHAPES, res)):
        assert list(r) == keys
        assert r["status"] == pattern("status", 3)[i] and type(r["status"]) is int
        assert r["value"] == pattern("value", 3)[i] and type(r["value"]) is float
        piv = pattern("pivots", 6)
        assert r["pivots"] == (piv[2 * i], piv[2 * i + 1]) and all(type(p) is int for p in r["pivots"])
        assert np.array_equal(r["rhs"], pattern("rhs", 7)[row:row + h]) and r["rhs"].dtype == np.float64
        for k in ("pos", "var", "reduced", "range_lo", "range_hi", "certificate"):
            if k in r:
                assert np.array_equal(r[k], pattern(k, 17)[pv:pv + h + w]) and r[k].dtype == ARRAYS[k][0], k
        if want_matrices:
            assert np.array_equal(r["matrix"], pattern("matrices", 19)[cell:cell + h * w])
        else:
            assert r["matrix"] is None
        row, cell, pv = row + h, cell + h * w, pv + h + w
    assert e.solve_ragged([], []) == [] and len(fake.calls) == 1


@pytest.mark.parametrize("multi_engine", [False, True])
def test_pinned_out_is_reused(fake, eng, multi, multi_engine):
    out = eng.batch_outputs(N, H, W, pinned=True)
    assert list(out) == ["status", "value", "pivots", "rhs", "pos", "var", "matrices", "reduced"]
    assert out["matrices"] is None and out["reduced"] is None and len(fake.pinned) == 6
    arrays = {k: v for k, v in out.items() if v is not None}
    e = multi if multi_engine else eng
    for _ in range(2):
        got = e.solve_batch(MATS, H, W, out=out)
        assert got is out and all(got[k] is a for k, a in arrays.items())
    # a reused out gains the extras a later call asks for, and keeps them
    got = e.solve_batch(MATS, H, W, out=out, want_duals=True, want_ranges=True, want_certificates=True)
    extras = [got[k] for k in ("reduced", "range_lo", "range_hi", "certificate")]
    assert all(a.shape == (N, PV) and a.dtype == np.float64 for a in extras)
    e.solve_batch(MATS, H, W, out=out, want_duals=True, want_ranges=True, want_certificates=True)
    assert all(got[k] is a for k, a in zip(("reduced", "range_lo", "range_hi", "certificate"), extras))
    pinned = {C.addressof(b) for b in fake.pinned}
    for rec in fake.calls:
        passed = dict(rec["args"])
        assert passed["matrices"] is None
    assert {out[k].ctypes.data for k in arrays} <= pinned


@pytest.mark.parametrize("multi_engine", [False, True])
@pytest.mark.parametrize("want_duals", [False, True])
def test_solve_replicas(fake, eng, multi, multi_engine, want_duals):
    e = multi if multi_engine else eng
    out = e.solve_replicas(MATS[:H * W], MATS[:N * H], H, W, want_duals=want_duals)
    (rec,) = fake.calls
    args = dict(rec["args"])
    assert (args["n"], args["base"], args["rhs_in"]) == (N, MATS[:H * W].tobytes(), MATS[:N * H].tobytes())
    assert (args["reduced"] is None) == (not want_duals)
    assert list(out) == ["status", "value", "pivots", "rhs", "pos", "var", "matrices", "reduced"]
    assert out["matrices"] is None and (out["reduced"] is None) == (not want_duals)
    assert out["rhs"].shape == (N, H) and np.array_equal(out["rhs"].reshape(-1), pattern("rhs", N * H))
    with pytest.raises(ValueError, match="base must hold"):
        e.solve_replicas(MATS[:H * W - 1], MATS[:N * H], H, W)


@pytest.mark.parametrize("want_ranges,want_certificates", list(itertools.product([False, True], [False, True])))
def test_solve_lp_sparse(fake, eng, want_ranges, want_certificates):
    cells = np.array([1, 5, 6], np.int32)
    vals = np.array([1.0, -2.0, 3.0])
    r = eng.solve_lp_sparse(cells, vals, H, W, want_ranges=want_ranges, pairs=PAIRS if want_ranges else None,
                            want_certificates=want_certificates)
    (rec,) = fake.calls
    args = dict(rec["args"])
    assert rec["fn"] == "yalps_solve_sparse_certificate"
    assert (args["h"], args["w"], args["nnz"], args["cells"], args["values"]) == (H, W, 3, cells.tobytes(),
                                                                                  vals.tobytes())
    assert args["pairs"] == (PAIRS.tobytes() if want_ranges else None)
    assert [k for k, v in rec["args"] if v is None] == ([] if want_ranges else ["pairs", "range_lo", "range_hi"]) + (
        [] if want_certificates else ["certificate"])
    keys = ["status", "value", "pivots", "rhs", "pos", "var", "reduced"]
    keys += ["range_lo", "range_hi"] if want_ranges else []
    keys += ["certificate"] if want_certificates else []
    assert list(r) == keys
    assert (r["status"], r["value"], r["pivots"]) == (1000, 2000.0, (3000, 3001))
    assert type(r["status"]) is int and type(r["value"]) is float
    for k in keys[3:]:
        assert r[k].shape == ((H,) if k == "rhs" else (PV,)) and r[k].dtype == ARRAYS[k][0]
        assert np.array_equal(r[k], pattern(k, r[k].size)), k


def test_multi_rejects_what_engine_rejects(fake, eng, multi):
    for e in (eng, multi):
        with pytest.raises(ValueError, match="not a multiple"):
            e.solve_batch(MATS[:-1], H, W)
        with pytest.raises(ValueError, match="not a multiple"):
            e.solve_batch(MATS, 0, W)
        with pytest.raises(ValueError, match="different batch size"):
            e.solve_batch(MATS, H, W, out=eng.batch_outputs(N + 1, H, W))
        with pytest.raises(ValueError, match="pos_in / var_in"):
            e.solve_batch(MATS, H, W, pos_in=np.zeros(N * PV - 1, np.int32), var_in=np.zeros(N * PV, np.int32))
        with pytest.raises(ValueError, match="pairs needs"):
            e.solve_batch(MATS, H, W, want_ranges=True, pairs=np.zeros(H + 1, np.int32))
    assert fake.calls == []
