"""Cost of the IIS search (yalps_iis) and of its subset machinery.  Prints the card name and power limit with the
numbers.

  1. per model: rounds, LPs, pivots per phase (from the host restatement of the search), and the wall time of
     Engine.iis (it ends in a synchronise) against tests/test_iis.py's iis_reference on the host cores, with the bytes
     that cross PCIe per round: row masks in and per-LP results out, against shipping the dense subset tableaus.
  2. k_expand_subsets against k_expand_replicas at the same n x H x W (one pipeline chunk of 33x65 LPs, larger than
     L2), kernel time from torch.profiler with L2 flushed before each call, as bytes written per second against the
     card's HBM figure.

    python scripts/iis_cost.py [--reps 5] [--n 8000] [--hbm-gbs 7700]
"""
import argparse
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import yalps_b200  # noqa: E402
from oracle import lib as O  # noqa: E402
from test_gpu_iis import big_infeasible  # noqa: E402
from test_iis import MODELS, iis_reference  # noqa: E402
from yalps_b200.tableau import tableau_model  # noqa: E402


def card() -> str:
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                       text=True).strip().splitlines()[0]
    except (OSError, subprocess.CalledProcessError):
        return torch.cuda.get_device_name(0) + ", power limit unknown"


def median_ms(f, reps):
    f()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        f()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts))


def per_model(eng, reps):
    t = tableau_model(big_infeasible()).tableau
    models = [m for m in MODELS if m[0] in ("ITEST2", "ITEST6", "BGPRTR", "KLEIN1", "objective_cut0", "random_infeasible0")]
    models.append(("big_infeasible", t.matrix, t.height, t.width))
    print("model HxW | rounds | LPs | pivots phase 1 / 2 | irreducible | yalps_iis ms | iis_reference ms (host) | "
          "PCIe bytes per round, masks + results / dense tableaus")
    for name, M, H, W in models:
        ref = iis_reference(M, H, W)
        got = eng.iis(M, H, W)
        assert got["rows"].tolist() == list(ref["rows"]) and got["pivots"] == ref["pivots"], name
        g = median_ms(lambda: eng.iis(M, H, W), reps)
        r = median_ms(lambda: iis_reference(M, H, W), max(1, reps // 2))
        words = (H + 31) // 32
        per_lp_small = words * 4 + 4 + 8 + 16 + words * 4 + 4  # mask in; status, value, pivots, support, count out
        lps_round = ref["lps"] / ref["rounds"]
        print(f"{name} {H}x{W} | {ref['rounds']} | {ref['lps']} | {ref['phase_pivots'][0]} / {ref['phase_pivots'][1]} | "
              f"{ref['irreducible']} | {g:.3f} | {r:.3f} | {lps_round * per_lp_small:.0f} / "
              f"{lps_round * H * W * 8:.0f} (mean {lps_round:.1f} LPs per round)")


def kernel_times(eng, n, hbm_gbs):
    H, W = 33, 65
    base = O.generate_synthetic(5, 1, H - 1, W - 1, 2)[0]
    words = (H + 31) // 32
    rng = np.random.default_rng(0)
    keep = rng.integers(0, 2 ** 32, (n, words), dtype=np.uint64).astype(np.uint32)
    keep[:, -1] &= np.uint32((1 << (H % 32)) - 1)
    rhs = np.tile(base.reshape(H, W)[:, 0], (n, 1))
    eng.set_replica_sharing(False)  # k_expand_replicas runs only without path sharing
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    calls = {"k_expand_subsets": lambda: eng.solve_row_subsets(base, keep, H, W),
             "k_expand_replicas": lambda: eng.solve_replicas(base, rhs, H, W)}
    for f in calls.values():
        f()
    torch.cuda.synchronize()
    written = n * H * W * 8
    for name, f in calls.items():
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                flush.zero_()
                torch.cuda.synchronize()
                f()
            torch.cuda.synchronize()
        us = [getattr(e, "device_time", None) or e.cuda_time for e in prof.events() if name in e.name]
        t = float(np.median(us)) * 1e-6
        gbs = written / t / 1e9
        print(f"{name}: {n} x {H}x{W} ({written / 1e6:.1f} MB written, L2 flushed before each call): kernel us median "
              f"{t * 1e6:.1f} over {len(us)} launches -> {gbs:.0f} GB/s written = {100 * gbs / hbm_gbs:.1f} % of "
              f"{hbm_gbs:.0f} GB/s")
    eng.set_replica_sharing(True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--n", type=int, default=8000)  # one pipeline chunk (the rule splits n > 8191)
    ap.add_argument("--hbm-gbs", type=float, default=7700.0)
    a = ap.parse_args()
    print("card:", card())
    eng = yalps_b200.Engine(0)
    per_model(eng, a.reps)
    kernel_times(eng, a.n, a.hbm_gbs)
    print("card:", card())


if __name__ == "__main__":
    main()
