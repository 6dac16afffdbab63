"""Cost of sensitivity ranging (k_ranging).  Prints the card name and power limit with the numbers.

  1. config 2 through the device entry: k_ranging kernel time by CUDA events over the final tableaus of 65,536 33x65
     LPs (yalps_ranging_device), with the bytes it reads, GB/s and share of the card's HBM figure.
  2. end to end, host buffers in and out: yalps_solve_batch_ranging against yalps_solve_batch_duals + matrices_out +
     numpy ranging on the host, for config 2 and for a batch of a Netlib model (default SC105), alternating in one
     process.

    python scripts/ranging_cost.py [--n2 65536] [--n3 4096] [--model SC105] [--reps 5] [--hbm-gbs 7700]
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
from yalps_b200.sensitivity import ranges_from_tableau  # noqa: E402


def card() -> str:
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                       text=True).strip().splitlines()[0]
    except (OSError, subprocess.CalledProcessError):
        return torch.cuda.get_device_name(0) + ", power limit unknown"


def host_ranging(out, n, H, W, precision):
    for i in range(n):
        ranges_from_tableau(out["matrices"][i], W, H, out["pos"][i], precision, None, out["status"][i] == 0)


def end_to_end(eng, mats, n, H, W, opt, reps, label):
    """yalps_solve_batch_ranging vs yalps_solve_batch_duals + matrices_out + numpy ranging, pinned host buffers."""
    o_dev = eng.batch_outputs(n, H, W, pinned=True, want_duals=True)
    o_dev["range_lo"], o_dev["range_hi"] = eng.pinned_empty((n, W + H), np.float64), eng.pinned_empty((n, W + H), np.float64)
    o_host = eng.batch_outputs(n, H, W, want_matrices=True, pinned=True, want_duals=True)
    times = {"device": [], "host": []}

    def run(kind):
        t0 = time.perf_counter()
        if kind == "device":
            eng.solve_batch(mats, H, W, opt, out=o_dev, want_duals=True, want_ranges=True)
        else:
            eng.solve_batch(mats, H, W, opt, out=o_host, want_matrices=True, want_duals=True)
            host_ranging(o_host, n, H, W, opt.precision)
        return (time.perf_counter() - t0) * 1e3

    for kind in times:
        run(kind)
    for _ in range(reps):
        for kind in times:
            times[kind].append(run(kind))
    d2h_dev = 16 * (W + H) * n
    d2h_host = 8 * H * W * n
    print(f"{label} {n} x {H}x{W}: end-to-end ms  yalps_solve_batch_ranging {np.median(times['device']):.2f} "
          f"(min {min(times['device']):.2f}) | duals + matrices_out + numpy ranging {np.median(times['host']):.2f} "
          f"(min {min(times['host']):.2f}); D2H of ranges {d2h_dev / 1e6:.1f} MB vs final tableaus {d2h_host / 1e6:.1f} MB")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n2", type=int, default=65536)
    ap.add_argument("--n3", type=int, default=4096)
    ap.add_argument("--model", default="SC105")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--hbm-gbs", type=float, default=7700.0, help="the card's HBM bandwidth figure (GB/s)")
    args = ap.parse_args()
    eng = yalps_b200.Engine(0)
    opt = make_options()
    stream = torch.cuda.current_stream().cuda_stream
    print(f"card: {card()}")

    # 1. config 2: k_ranging over final tableaus in device memory
    n, m, nv = args.n2, 32, 64
    H, W = m + 1, nv + 1
    d = torch.empty(n * H * W, dtype=torch.float64, device="cuda")
    eng.generate_synthetic_device(0, n, m, nv, d.data_ptr(), stream=stream)
    fin = torch.empty_like(d)
    work = torch.empty_like(d)
    st = torch.empty(n, dtype=torch.int32, device="cuda")
    pos = torch.empty(n * (W + H), dtype=torch.int32, device="cuda")
    lo = torch.empty(n * (W + H), dtype=torch.float64, device="cuda")
    hi = torch.empty_like(lo)
    eng.solve_batch_device(n, H, W, d.data_ptr(), opt, d_work=work.data_ptr(), d_status=st.data_ptr(),
                           d_pos=pos.data_ptr(), d_matrices_out=fin.data_ptr(), stream=stream)
    torch.cuda.synchronize()
    print(f"config2 statuses: {np.bincount(st.cpu().numpy(), minlength=5).tolist()} (optimal, infeasible, unbounded, "
          f"timedout, cycled)")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # larger than L2: every pass reads from HBM

    def ranging():
        eng.ranging_device(n, H, W, fin.data_ptr(), pos.data_ptr(), lo.data_ptr(), hi.data_ptr(),
                           precision=opt.precision, d_status=st.data_ptr(), stream=stream)

    ranging()
    torch.cuda.synchronize()
    ms = []
    for _ in range(max(args.reps, 10)):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ranging()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    t = float(np.median(ms))
    read = n * (H * W * 8 + (W + H) * 4 + 4)  # final tableaus, pos, status
    written = n * (W + H) * 16
    gbs = (read + written) / (t * 1e-3) / 1e9
    print(f"config2 k_ranging {n} x {H}x{W} (L2 flushed before each pass): kernel ms median {t:.3f} (min {min(ms):.3f}); "
          f"{read / 1e9:.3f} GB read + {written / 1e9:.3f} GB written -> {gbs:.0f} GB/s = "
          f"{100 * gbs / args.hbm_gbs:.0f} % of {args.hbm_gbs:.0f} GB/s")
    del flush, work

    # 2. end to end through the host entries
    mats = d.view(n, H * W).cpu().numpy()
    del d, fin
    end_to_end(eng, mats, n, H, W, opt, args.reps, "config2")
    g = BW.netlib_base(args.model)
    H, W = g["height"], g["width"]
    n = args.n3
    dr = torch.empty(n * H * W, dtype=torch.float64, device="cuda")
    eng.generate_replicas_device(0, n, g["matrix"], H, W, g["row_groups"], dr.data_ptr(), stream=stream)
    torch.cuda.synchronize()
    mats = dr.view(n, H * W).cpu().numpy()
    del dr
    end_to_end(eng, mats, n, H, W, opt, args.reps, f"{args.model} batch")
    eng.close()


if __name__ == "__main__":
    main()
