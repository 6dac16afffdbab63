"""Cost of warm starts (yalps_solve_warm) against cold solves.  Prints the card name and power limit with the numbers.

  1. Config-3-style RHS-perturbed variants (eps 1e-2, the replica generator) of SC105 and ADLITTLE: yalps_solve_warm
     (base solved inside the call) against yalps_solve_replicas with path sharing on and off.  Phase-1 / phase-2 pivots
     per LP (mean, max) and end-to-end ms (host clock around calls that end in a synchronise).
  2. The k_expand_warm kernel of the same call (torch.profiler, its own run): time, bytes written (the working copies
     and var_in) plus the per-LP column read, and GB/s.
  3. Objective-perturbed variants (every coefficient * (1 + 1e-2 u)): yalps_solve_warm against solve_batch of the
     rebuilt tableaus.

    python scripts/warm_cost.py [--n 10000] [--reps 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import yalps_b200  # noqa: E402
from bench_workloads import netlib_base  # noqa: E402


def card() -> str:
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                       text=True).strip().splitlines()[0]
    except (OSError, subprocess.CalledProcessError):
        return torch.cuda.get_device_name(0) + ", power limit unknown"


def timed(fn, reps):
    fn()  # warm-up: allocates the device pools
    t0 = time.perf_counter()
    for _ in range(reps):
        out = fn()
    return (time.perf_counter() - t0) / reps * 1e3, out


def pivots(out):
    p = out["pivots"]
    return {"p1_mean": float(p[:, 0].mean()), "p1_max": int(p[:, 0].max()), "p2_mean": float(p[:, 1].mean()),
            "p2_max": int(p[:, 1].max())}


def kernel_ms(fn, name):
    from torch.profiler import ProfilerActivity, profile
    fn()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    ev = [e for e in prof.events() if name in e.name and e.device_type.name == "CUDA"]
    return sum(e.device_time for e in ev) / 1e3, len(ev)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=10000)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    print("card:", card())
    eng = yalps_b200.Engine(0)
    opt = yalps_b200.make_options()
    for name in ("SC105", "ADLITTLE"):
        g = netlib_base(name)
        H, W, M0 = g["height"], g["width"], g["matrix"]
        n = args.n
        d = torch.empty(n * H * W, dtype=torch.float64, device="cuda")
        eng.generate_replicas_device(0, n, M0, H, W, g["row_groups"], d.data_ptr())
        torch.cuda.synchronize()
        rhs = d.view(n, H, W)[:, :, 0].cpu().numpy().copy()
        del d
        row = {"model": name, "shape": [H, W], "n": n}
        ms, w = timed(lambda: eng.solve_warm(M0, H, W, rhs=rhs, options=opt), args.reps)
        row["warm"] = {"ms": ms, **pivots(w), "base_pivots": w["base"]["pivots"]}
        for sharing in (True, False):
            eng.set_replica_sharing(sharing)
            ms, r = timed(lambda: eng.solve_replicas(M0, rhs, H, W, opt), args.reps)
            row["replicas_sharing_" + ("on" if sharing else "off")] = {"ms": ms, **pivots(r)}
            assert np.array_equal(r["status"], w["status"]), "warm and cold statuses differ"
            row["max_abs_value_diff"] = float(np.max(np.abs(r["value"] - w["value"])[r["status"] == 0], initial=0.0))
        eng.set_replica_sharing(True)
        kms, launches = kernel_ms(lambda: eng.solve_warm(M0, H, W, rhs=rhs, options=opt), "k_expand_warm")
        nbytes = n * (H * W * 8 + (H + W) * 4 + H * 8)
        row["k_expand_warm"] = {"ms": kms, "launches": launches, "bytes": nbytes, "gbs": nbytes / (kms * 1e-3) / 1e9}
        # objective-perturbed variants against cold solves of the rebuilt tableaus
        rng = np.random.default_rng(1)
        obj = np.tile(M0[:W], (n, 1)) * (1 + 1e-2 * rng.uniform(-1, 1, (n, W)))
        mats = np.tile(M0, (n, 1))
        mats[:, :W] = obj
        ms, wo = timed(lambda: eng.solve_warm(M0, H, W, obj=obj, options=opt), args.reps)
        row["obj_warm"] = {"ms": ms, **pivots(wo)}
        ms, co = timed(lambda: eng.solve_batch(mats, H, W, opt), args.reps)
        row["obj_cold_batch"] = {"ms": ms, **pivots(co)}
        assert np.array_equal(co["status"], wo["status"]), "warm and cold statuses differ (objective)"
        print(json.dumps(row))
    eng.close()


if __name__ == "__main__":
    main()
