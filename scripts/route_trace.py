#!/usr/bin/env python
"""Kernel-path trace: for a fixed grid of cases (entry point x batch size x shape x density x tuning path), what every
call launches and returns.  Per case one JSON line: the kernels (name, grid, block, dynamic shared memory) and the
copies / memsets seen by torch.profiler with CUDA activities, the launch-count delta of the engine, the error of a
call that fails, and a hash of every output.  The kernels and copies are listed sorted: the K4 lanes of a node wave and
the two pipeline streams of a host batch overlap, so their order in time is not reproducible.

Two builds route alike when their traces are identical:
    python scripts/route_trace.py OUT.jsonl [--quick]
It uses only the Python API.  When the profiler sees no kernel of the library the script fails: launch counts and
hashes alone would not show which kernels ran."""
import argparse, hashlib, json, os, sys, tempfile
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch
from torch.profiler import ProfilerActivity, profile
import yalps_b200
from yalps_b200 import engine as E
from yalps_b200._ffi import YalpsError
from oracle import lib as O
from conftest import load_cases
from oracle import model as M

PATHS = {"AUTO": E.PATH_AUTO, "SMEM": E.PATH_SMEM, "GMEM": E.PATH_GMEM, "GRID": E.PATH_GRID, "CLUSTER": E.PATH_CLUSTER,
         "TMEM": E.PATH_TMEM, "GRID_RES": E.PATH_GRID_RESIDENT}
# both sides of the size thresholds of the policy: K1t short (<= 33 rows) / tall (<= 65x65) / beyond, a tableau in one
# SM's shared memory or not, the 40,000-cell row-split-vs-K4 line, one cluster's shared memory, the grid's, K4 only
SHAPES = [(9, 17), (33, 65), (34, 65), (65, 65), (66, 66), (120, 200), (150, 260), (160, 260), (200, 260), (600, 1200),
          (300, 3000)]
MAX_CELLS = 8_000_000  # per case: n * H * W


def tableaus(n, H, W, sparse, seed):
    m = O.generate_synthetic(seed, n, H - 1, W - 1, 2).reshape(n, H, W)
    if sparse:  # 85 % zeros below the objective row, the right-hand sides kept
        rng = np.random.default_rng(seed)
        keep = rng.random((n, H - 1, W - 1)) < 0.15
        m[:, 1:, 1:] *= keep
    return np.ascontiguousarray(m)


def random_pairs(n, H, seed):
    """Row pairs of n LPs of H rows (sensitivity ranging): random disjoint pairs of rows 1..H-1, -1 elsewhere."""
    rng = np.random.default_rng(seed)
    out = np.full((n, H), -1, np.int32)
    for i in range(n):
        rows = rng.permutation(np.arange(1, H))
        for j in range(0, len(rows) - 1, 2):
            if rng.random() < 0.5:
                out[i, rows[j]], out[i, rows[j + 1]] = rows[j + 1], rows[j]
    return out


def duplicated_stores(cells, values):
    """The stores with every tenth one preceded by a store of another value to the same cell (the last store wins)."""
    dc, dv = [], []
    for k, (c, v) in enumerate(zip(cells.tolist(), values.tolist())):
        if k % 10 == 0:
            dc.append(c)
            dv.append(v + 1.5)
        dc.append(c)
        dv.append(v)
    return np.asarray(dc, np.int32), np.asarray(dv, np.float64)


def tableau_outputs(r):
    """solve_tableau's result without its timings"""
    return {k: np.asarray(v) for k, v in r.items() if k != "stats"} | {
        "nodes": np.array([r["stats"]["nodes"], r["stats"]["node_pivots"], r["stats"]["max_cuts"]])}


def node_outputs(r, nodes, H, W):
    """bnb_solve_nodes' result without the rows past each node's own height, which it leaves as they were"""
    out = {k: r[k] for k in ("status", "value", "pivots")}
    for j, cuts in enumerate(nodes):
        h = H + len(cuts)
        out |= {f"{j}:rhs": r["rhs"][j, :h], f"{j}:pos": r["pos"][j, :W + h], f"{j}:var": r["var"][j, :W + h],
                f"{j}:matrix": r["matrices"][j, :h * W]}
    return out


def digest(outs):
    h = hashlib.sha256()
    for k in sorted(outs):
        v = outs[k]
        if v is not None:
            h.update(k.encode()); h.update(np.ascontiguousarray(v).tobytes())
    return h.hexdigest()[:24]


def trace(eng, fn):
    """Run fn under the profiler: (kernels, copies, launch-count delta, error, hash of fn's outputs)."""
    torch.cuda.synchronize()
    c0 = eng.launch_count
    err, outs = None, {}
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        try:
            outs = fn()
        except YalpsError as e:
            err = [e.code, str(e)]
        torch.cuda.synchronize()
    dc = eng.launch_count - c0
    with tempfile.NamedTemporaryFile(suffix=".json") as f:
        prof.export_chrome_trace(f.name)
        events = json.load(open(f.name))["traceEvents"]
    kernels, copies = [], []
    for ev in events:
        cat, a = ev.get("cat", ""), ev.get("args", {})
        if cat == "kernel":
            kernels.append([ev["name"], a.get("grid"), a.get("block"), a.get("shared memory")])
        elif cat in ("gpu_memcpy", "gpu_memset"):
            copies.append([ev["name"], a.get("bytes")])
    return sorted(kernels, key=str), sorted(copies, key=str), dc, err, digest(outs)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--quick", action="store_true", help="a few cases only (rehearsal)")
    args = ap.parse_args()
    eng = yalps_b200.Engine(0)
    sms = eng.device_info()["sm_count"]
    ns = [1, 16, 17, 2 * sms + 1, 8 * sms + 1]
    shapes, paths = (SHAPES[:2], ["AUTO", "GRID"]) if args.quick else (SHAPES, list(PATHS))
    stream = torch.cuda.current_stream().cuda_stream
    seen_library_kernel = False
    out = open(args.out, "w")

    def emit(case, fn, who=None):
        nonlocal seen_library_kernel
        k, c, dc, err, hsh = trace(who or eng, fn)
        seen_library_kernel |= any("k_simplex" in x[0] for x in k)
        out.write(json.dumps({**case, "kernels": k, "copies": c, "launches": dc, "error": err, "hash": hsh}) + "\n")
        out.flush()

    for (H, W) in shapes:
        for n in ns:
            if n * H * W > MAX_CELLS:
                continue
            for sparse in (False, True):
                m = tableaus(n, H, W, sparse, seed=H * 7919 + W)
                dens = "sparse" if sparse else "dense"
                rag_shapes = [[(H, W), (9, 17), (H // 2 + 1, W // 2 + 1)][i % 3] for i in range(n)]
                rag = [tableaus(1, h, w, sparse, seed=i)[0].reshape(-1) for i, (h, w) in enumerate(rag_shapes)]
                rhs = m[:, :, 0].copy()
                d_in = torch.from_numpy(m.reshape(-1)).cuda()
                for pname in paths:
                    if pname != "AUTO" and (n == 16 or sparse):  # the K4 line and the density rules are automatic ones
                        continue
                    eng.set_tuning(PATHS[pname], 0)
                    case = {"shape": [H, W], "n": n, "density": dens, "path": pname}
                    emit({"entry": "batch", **case}, lambda: eng.solve_batch(m, H, W, want_matrices=True, want_duals=sparse))
                    emit({"entry": "ragged", **case}, lambda: {
                        f"{i}:{k}": np.asarray(v) for i, r in enumerate(
                            eng.solve_ragged(rag, rag_shapes, want_matrices=True, want_duals=sparse))
                        for k, v in r.items() if v is not None})

                    def device():
                        pv = H + W
                        t = {"work": torch.empty_like(d_in), "mout": torch.zeros_like(d_in),
                             "status": torch.zeros(n, dtype=torch.int32, device="cuda"),
                             "value": torch.zeros(n, dtype=torch.float64, device="cuda"),
                             "pivots": torch.zeros(n, 2, dtype=torch.int64, device="cuda"),
                             "rhs": torch.zeros(n * H, dtype=torch.float64, device="cuda"),
                             "pos": torch.zeros(n * pv, dtype=torch.int32, device="cuda"),
                             "var": torch.zeros(n * pv, dtype=torch.int32, device="cuda"),
                             "red": torch.zeros(n * pv, dtype=torch.float64, device="cuda")}
                        eng.solve_batch_device(n, H, W, d_in.data_ptr(), d_work=t["work"].data_ptr(),
                                               d_status=t["status"].data_ptr(), d_value=t["value"].data_ptr(),
                                               d_pivots=t["pivots"].data_ptr(), d_rhs=t["rhs"].data_ptr(),
                                               d_pos=t["pos"].data_ptr(), d_var=t["var"].data_ptr(),
                                               d_matrices_out=t["mout"].data_ptr(), stream=stream,
                                               d_reduced=t["red"].data_ptr() if sparse else 0)
                        torch.cuda.synchronize()
                        return {k: v.cpu().numpy() for k, v in t.items() if k != "work"}
                    emit({"entry": "device", **case}, device)
                    for share in (True, False):
                        eng.set_replica_sharing(share)
                        emit({"entry": "replicas", "sharing": share, **case},
                             lambda: {k: v for k, v in eng.solve_replicas(m[0], rhs, H, W, want_duals=sparse).items()}
                             | {"forks": np.array([eng.replica_forks])})
                    eng.set_replica_sharing(True)
                del d_in
    eng.set_tuning(E.PATH_AUTO, 0)
    # ranges with paired rows, one engine and two ranks on one GPU; the zero-copy small call and the chunk pipeline
    multi = yalps_b200.MultiEngine([0, 0])
    for (H, W) in [(9, 17), (33, 65), (120, 200)]:
        for n in (1, 17, 2 * sms + 1):
            m = tableaus(n, H, W, True, seed=H + n)
            pairs = random_pairs(n, H, seed=n)
            rag_shapes = [[(H, W), (9, 17)][i % 2] for i in range(n)]
            rag = [tableaus(1, h, w, True, seed=i)[0].reshape(-1) for i, (h, w) in enumerate(rag_shapes)]
            rag_pairs = [random_pairs(1, h, seed=i)[0] for i, (h, _) in enumerate(rag_shapes)]
            rhs = m[:, :, 0].copy()
            case = {"shape": [H, W], "n": n}
            for who, x in (("engine", eng), ("multi", multi)):
                emit({"entry": "batch_ranges", "on": who, **case}, lambda: x.solve_batch(
                    m, H, W, want_matrices=True, want_duals=True, want_ranges=True, pairs=pairs), x)
                emit({"entry": "ragged_ranges", "on": who, **case}, lambda: {
                    f"{i}:{k}": np.asarray(v) for i, r in enumerate(x.solve_ragged(
                        rag, rag_shapes, want_matrices=True, want_duals=True, want_ranges=True, pairs=rag_pairs))
                    for k, v in r.items() if v is not None}, x)
            emit({"entry": "replicas", "on": "multi", **case},
                 lambda: multi.solve_replicas(m[0], rhs, H, W, want_duals=True), multi)
    multi.close()
    # tableaus given as (cell, value) stores, below and above the 768 KB zero-copy limit, with and without duplicate
    # cells; a MILP whose root (above 256 KB) stays on the device for branch and cut
    cases = {c["name"]: c for c in load_cases()}
    for name in ["Monster Problem", "Monster 2"]:
        tm = yalps_b200.tableau_model(cases[name]["model"], 0)
        t = tm.tableau
        stores = {"plain": (t.cells, t.values), "duplicates": duplicated_stores(t.cells, t.values)}
        dense = np.zeros(t.height * t.width)
        for c, v in zip(t.cells.tolist(), t.values.tolist()):
            dense[c] = v
        emit({"entry": "tableau", "model": name}, lambda: tableau_outputs(
            eng.solve_tableau(dense, t.height, t.width, tm.integers, tm.sign)))
        for kind, (c, v) in stores.items():
            for limit in ("below", "above") if not tm.integers else ("above",):
                h, w = (t.height, t.width) if limit == "above" else (t.height // 4, t.width // 4)  # a corner
                keep = ((c // t.width) < h) & ((c % t.width) < w)
                cs, vs = ((c // t.width) * w + c % t.width)[keep].astype(np.int32), v[keep]
                case = {"model": name, "stores": kind, "limit": limit}
                emit({"entry": "tableau_sparse", **case}, lambda: tableau_outputs(
                    eng.solve_tableau_sparse(cs, vs, h, w, tm.integers, tm.sign)))
                if not tm.integers:
                    emit({"entry": "lp_sparse", **case}, lambda: eng.solve_lp_sparse(
                        cs, vs, h, w, want_ranges=True, pairs=random_pairs(1, h, seed=h)[0]))
                    emit({"entry": "lp_sparse", "ranges": False, **case}, lambda: eng.solve_lp_sparse(cs, vs, h, w))
    # node waves: synthetic roots (solved by the oracle) and the big sparse Monster 2 root
    roots = []
    for (H, W) in shapes[:8]:
        t = tableaus(1, H, W, False, seed=H + W)[0].reshape(-1).copy()
        pos = np.arange(W + H, dtype=np.int32); var = pos.copy()
        st, _, _ = O.simplex(t, W, H, pos, var)
        roots.append((f"{H}x{W}", t, H, W, pos, var, list(range(1, W))))
    if not args.quick:
        c = next(x for x in load_cases() if x["name"] == "Monster 2")
        tm = M.tableau_model(c["model"]); tt = tm.tableau
        O.simplex(tt.matrix, tt.width, tt.height, tt.pos, tt.var)
        roots.append(("Monster 2", tt.matrix, tt.height, tt.width, tt.pos, tt.var, list(tm.integers)))
    for name, t, H, W, pos, var, ints in roots:
        eng.bnb_set_root(t, H, W, pos, var, 8)
        rng = np.random.default_rng(11)
        for n in (1, 6, 17, 2 * sms + 1):
            nodes = [[(float(rng.choice([1.0, -1.0])), int(rng.choice(ints)), float(rng.integers(0, 3)))
                      for _ in range(int(rng.integers(1, 5)))] for _ in range(n)]
            for pname in paths:
                eng.set_tuning(PATHS[pname], 0)
                emit({"entry": "nodes", "root": name, "n": n, "path": pname},
                     lambda: node_outputs(eng.bnb_solve_nodes(nodes, want_matrices=True), nodes, H, W))
    eng.set_tuning(E.PATH_AUTO, 0)
    out.close()
    eng.close()
    if not seen_library_kernel:
        sys.exit("route_trace: the profiler saw no kernel of the library; kernel names, grids and blocks are not traced")


if __name__ == "__main__":
    main()
