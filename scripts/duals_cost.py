"""Cost of the reduced-cost output (reduced_out / d_reduced): config 2 through the device entry (kernel time) and
config 3 through the replica entry (end to end, pinned host buffers), each with and without the output, alternating in
one process.  Prints the card name and power limit with the numbers.

    python scripts/duals_cost.py [--n2 65536] [--n3 65536] [--model SC105] [--reps 5]
"""
import argparse
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench_workloads as BW  # noqa: E402
import yalps_b200  # noqa: E402
from yalps_b200.engine import make_options  # noqa: E402


def card() -> str:
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                       text=True).strip().splitlines()[0]
    except (OSError, subprocess.CalledProcessError):
        return torch.cuda.get_device_name(0) + ", power limit unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n2", type=int, default=65536)
    ap.add_argument("--n3", type=int, default=65536)
    ap.add_argument("--model", default="SC105")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    eng = yalps_b200.Engine(0)
    opt = make_options()
    stream = torch.cuda.current_stream().cuda_stream
    print(f"card: {card()}")

    # config 2: 33x65 synthetic LPs in device memory, kernel time by CUDA events
    n, m, nv = args.n2, 32, 64
    H, W = m + 1, nv + 1
    d = torch.empty(n * H * W, dtype=torch.float64, device="cuda")
    eng.generate_synthetic_device(0, n, m, nv, d.data_ptr(), stream=stream)
    outs = {k: torch.empty(n * s, dtype=t, device="cuda") for k, s, t in
            (("st", 1, torch.int32), ("val", 1, torch.float64), ("piv", 2, torch.int64), ("rhs", H, torch.float64),
             ("pos", W + H, torch.int32), ("var", W + H, torch.int32))}
    red = torch.empty(n * (W + H), dtype=torch.float64, device="cuda")

    def step2(duals):
        eng.solve_batch_device(n, H, W, d.data_ptr(), opt, d_status=outs["st"].data_ptr(), d_value=outs["val"].data_ptr(),
                               d_pivots=outs["piv"].data_ptr(), d_rhs=outs["rhs"].data_ptr(),
                               d_pos=outs["pos"].data_ptr(), d_var=outs["var"].data_ptr(),
                               d_reduced=red.data_ptr() if duals else 0, stream=stream)

    times = {False: [], True: []}
    for duals in (False, True):
        step2(duals)
    torch.cuda.synchronize()
    for _ in range(args.reps):
        for duals in (False, True):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            step2(duals)
            e1.record()
            torch.cuda.synchronize()
            times[duals].append(e0.elapsed_time(e1))
    print(f"config2 device entry {n} x {H}x{W}: kernel ms without {np.median(times[False]):.3f} "
          f"(min {min(times[False]):.3f}), with reduced {np.median(times[True]):.3f} (min {min(times[True]):.3f})")

    # config 3: RHS-perturbed replicas of a Netlib model through yalps_solve_replicas(_duals), end to end
    g = BW.netlib_base(args.model)
    H, W = g["height"], g["width"]
    n = args.n3
    dr = torch.empty(n * H * W, dtype=torch.float64, device="cuda")
    eng.generate_replicas_device(0, n, g["matrix"], H, W, g["row_groups"], dr.data_ptr(), stream=stream)
    torch.cuda.synchronize()
    h_rhs = eng.pinned_empty((n, H), np.float64)
    h_rhs[:] = dr.view(n, H, W)[:, :, 0].cpu().numpy()
    del dr
    out = eng.batch_outputs(n, H, W, pinned=True, want_duals=True)
    base = g["matrix"]
    times = {False: [], True: []}
    for duals in (False, True):
        eng.solve_replicas(base, h_rhs, H, W, opt, out=out, want_duals=duals)
    for _ in range(args.reps):
        for duals in (False, True):
            t0 = time.perf_counter()
            eng.solve_replicas(base, h_rhs, H, W, opt, out=out, want_duals=duals)
            times[duals].append((time.perf_counter() - t0) * 1e3)
    print(f"config3 replicas {args.model} {n} x {H}x{W}: end-to-end ms without {np.median(times[False]):.2f} "
          f"(min {min(times[False]):.2f}), with reduced {np.median(times[True]):.2f} (min {min(times[True]):.2f}); "
          f"extra D2H {8 * (W + H) * n / 1e6:.1f} MB; forks {eng.replica_forks}")
    eng.close()


if __name__ == "__main__":
    main()
