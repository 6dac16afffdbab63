"""Cost of warm starts that add constraints and variables (yalps_solve_warm_extend) against cold solves of the rebuilt
tableaus.  Prints the card name and power limit with the numbers.

For SC105 and ADLITTLE, 10,000 variants each, in three cases: 1-4 added rows that cut off the base's optimal vertex
(a random non-negative a with a.x <= (0.5..0.95) a.x*), 1-2 added columns that copy a basic column at a better cost
(so their reduced cost is attractive), and both.  A batch is padded to its largest K and M with zero rows and columns,
as solve_variants pads it.  Per case:
  - warm: phase-1 / phase-2 pivots per LP (mean, max) and end-to-end ms of Engine.solve_warm (base solved inside the
    call; host clock around calls that end in a synchronise, after a warm-up);
  - cold: the same for solve_batch of every variant's rebuilt (padded) tableau, and how many statuses differ;
  - the k_expand_warm kernel of the warm call (torch.profiler, its own run).
Also k_expand_warm for the K = M = 0 call of scripts/warm_cost.py (config-3 RHS variants), to set against that script.

    python scripts/warm_extend_cost.py [--n 10000] [--reps 3]
"""
import argparse
import json
import os
import sys
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import yalps_b200  # noqa: E402
from bench_workloads import netlib_base  # noqa: E402
from warm_cost import card, kernel_ms, pivots, timed  # noqa: E402


def additions(rng, M0, F, pos, H, W, n, case):
    """(rows (n, K, W+M) or None, cols (n, M, H) or None, cold tableaus (n, (H+K)*(W+M)))."""
    m0, f = M0.reshape(H, W), F.reshape(H, W)
    p = pos[1:W]
    x = np.where(p >= W, f[:, 0][np.clip(p - W, 0, H - 1)], 0.0)
    basic = np.flatnonzero(p >= W) + 1
    ks = rng.integers(1, 5, n) if case in ("rows", "both") else np.zeros(n, int)
    ms = rng.integers(1, 3, n) if case in ("cols", "both") else np.zeros(n, int)
    K, M = int(ks.max()), int(ms.max())
    rows, cols = np.zeros((n, K, W + M)), np.zeros((n, M, H))
    for i in range(n):
        for j in range(ms[i]):
            g = m0[:, int(rng.choice(basic))].copy()
            g[0] = g[0] + 0.05 * abs(g[0]) + 0.01
            cols[i, j] = g
        for h in range(ks[i]):
            a = np.round(rng.uniform(0.5, 3.0, W - 1), 3) * (rng.random(W - 1) < 0.1)
            rows[i, h, 1:W] = a
            rows[i, h, W:W + ms[i]] = np.round(rng.uniform(0.0, 2.0, ms[i]), 3)
            ax = float(a @ x)
            rows[i, h, 0] = ax * float(rng.uniform(0.5, 0.95)) if ax > 0 else 1.0
    cold = np.zeros((n, H + K, W + M))
    cold[:, :H, :W] = m0
    cold[:, :H, W:] = cols.transpose(0, 2, 1)
    cold[:, H:] = rows
    return (rows if K else None), (cols if M else None), cold.reshape(n, -1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=10000)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    print("card:", card())
    eng = yalps_b200.Engine(0)
    opt = yalps_b200.make_options()
    n = args.n
    for name in ("SC105", "ADLITTLE"):
        g = netlib_base(name)
        H, W, M0 = g["height"], g["width"], np.ascontiguousarray(g["matrix"], np.float64)
        base = eng.solve_batch(M0, H, W, opt, want_matrices=True)
        F, pos = base["matrices"][0], base["pos"][0]
        # K = M = 0: the RHS variants of scripts/warm_cost.py
        d = torch.empty(n * H * W, dtype=torch.float64, device="cuda")
        eng.generate_replicas_device(0, n, M0, H, W, g["row_groups"], d.data_ptr())
        torch.cuda.synchronize()
        rhs = d.view(n, H, W)[:, :, 0].cpu().numpy().copy()
        del d
        kms, launches = kernel_ms(lambda: eng.solve_warm(M0, H, W, rhs=rhs, options=opt), "k_expand_warm")
        print(json.dumps({"model": name, "case": "K=M=0 (warm_cost.py RHS variants)", "n": n,
                          "k_expand_warm": {"ms": kms, "launches": launches}}))
        for case in ("rows", "cols", "both"):
            rng = np.random.default_rng(zlib.crc32(f"{name}:{case}".encode()))
            rows, cols, cold = additions(rng, M0, F, pos, H, W, n, case)
            K = 0 if rows is None else rows.shape[1]
            M = 0 if cols is None else cols.shape[1]
            row = {"model": name, "shape": [H, W], "case": case, "K": K, "M": M, "n": n}
            call = lambda: eng.solve_warm(M0, H, W, options=opt, add_rows=rows, add_cols=cols)  # noqa: E731
            ms, w = timed(call, args.reps)
            row["warm"] = {"ms": ms, **pivots(w)}
            ms, c = timed(lambda: eng.solve_batch(cold, H + K, W + M, opt), args.reps)
            row["cold_batch"] = {"ms": ms, **pivots(c)}
            row["status_mismatches"] = int((c["status"] != w["status"]).sum())
            ok = (c["status"] == 0) & (w["status"] == 0)
            row["statuses"] = np.bincount(w["status"], minlength=5).tolist()
            row["max_rel_value_diff"] = float(np.max(np.abs(c["value"] - w["value"])[ok] /
                                                     np.maximum(1.0, np.abs(c["value"][ok])), initial=0.0))
            kms, launches = kernel_ms(call, "k_expand_warm")
            row["k_expand_warm"] = {"ms": kms, "launches": launches}
            print(json.dumps(row))
    eng.close()


if __name__ == "__main__":
    main()
