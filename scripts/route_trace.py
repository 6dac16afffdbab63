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

    def emit(case, fn):
        nonlocal seen_library_kernel
        k, c, dc, err, hsh = trace(eng, fn)
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
                     lambda: {k: v for k, v in eng.bnb_solve_nodes(nodes, want_matrices=True).items() if k != "stride_h"})
    eng.set_tuning(E.PATH_AUTO, 0)
    out.close()
    eng.close()
    if not seen_library_kernel:
        sys.exit("route_trace: the profiler saw no kernel of the library; kernel names, grids and blocks are not traced")


if __name__ == "__main__":
    main()
