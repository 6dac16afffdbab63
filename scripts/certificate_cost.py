"""Cost of certificates (k_certificate).  Prints the card name and power limit with the numbers.

  1. k_certificate kernel time by CUDA events over the final tableaus of 65,536 33x65 LPs in device memory
     (yalps_certificate_device), once with almost every LP infeasible (column 0, pos and one row read per LP) and once
     with config 2's own, almost all optimal, finals (the NaN fill), with the bytes each pass moves and their share of
     the card's HBM figure.
  2. config 2 end to end through solve_batch (host buffers in and out), with and without want_certificates,
     alternating in one process.  The difference includes keeping the final tableaus on the device.
  3. one 25FV47-size LP (the Netlib tableau, as a model) through solve(), with and without the option `certificate`.

    python scripts/certificate_cost.py [--n 65536] [--reps 5] [--hbm-gbs 7700]
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
from yalps_b200.tableau import tableau_model  # noqa: E402


def card() -> str:
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                       text=True).strip().splitlines()[0]
    except (OSError, subprocess.CalledProcessError):
        return torch.cuda.get_device_name(0) + ", power limit unknown"


def kernel_time(eng, n, H, W, fin, pos, st, val, cert, opt, stream, reps, hbm_gbs, label):
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # larger than L2: every pass reads from HBM

    def run():
        eng.certificate_device(n, H, W, fin.data_ptr(), pos.data_ptr(), st.data_ptr(), val.data_ptr(), cert.data_ptr(),
                               precision=opt.precision, stream=stream)

    run()
    torch.cuda.synchronize()
    ms = []
    for _ in range(max(reps, 20)):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    t = float(np.median(ms))
    s = st.cpu().numpy()
    hit = int(((s == 1) | (s == 2)).sum())
    # per LP: status and value; per LP with a certificate: column 0, pos and one row of W cells (or a column of H)
    read = n * 12 + hit * (H * 8 + (W + H) * 4 + max(W, H) * 8)
    written = n * (W + H) * 8
    gbs = (read + written) / (t * 1e-3) / 1e9
    print(f"{label}: statuses {np.bincount(s, minlength=5).tolist()}; k_certificate {n} x {H}x{W} (L2 flushed before "
          f"each pass): kernel ms median {t:.4f} (min {min(ms):.4f}); {read / 1e6:.1f} MB read + {written / 1e6:.1f} MB "
          f"written -> {gbs:.0f} GB/s = {100 * gbs / hbm_gbs:.1f} % of {hbm_gbs:.0f} GB/s")


def alternate(reps, runs):
    """Median ms of each callable in `runs`, run alternately after one warm-up each."""
    times = {k: [] for k in runs}
    for f in runs.values():
        f()
    for _ in range(reps):
        for k, f in runs.items():
            t0 = time.perf_counter()
            f()
            times[k].append((time.perf_counter() - t0) * 1e3)
    return {k: (float(np.median(v)), min(v)) for k, v in times.items()}


def model_of(g) -> dict:
    """A maximisation whose tableau is the Netlib tableau g (row r: a.x <= M[r,0]; row 0: the objective)."""
    H, W = g["height"], g["width"]
    M = g["matrix"].reshape(H, W)
    cons = [(f"r{r}", {"max": float(M[r, 0])}) for r in range(1, H)]
    variables = []
    for j in range(1, W):
        nz = np.flatnonzero(M[:, j])
        variables.append((f"x{j}", [("obj" if r == 0 else f"r{r}", float(M[r, j])) for r in nz]))
    return {"direction": "maximize", "objective": "obj", "constraints": cons, "variables": variables}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=65536)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--hbm-gbs", type=float, default=7700.0, help="the card's HBM bandwidth figure (GB/s)")
    args = ap.parse_args()
    eng = yalps_b200.Engine(0)
    opt = make_options()
    stream = torch.cuda.current_stream().cuda_stream
    print(f"card: {card()}")

    # 1. kernel time over final tableaus in device memory
    n, m, nv = args.n, 32, 64
    H, W = m + 1, nv + 1
    d = torch.empty(n * H * W, dtype=torch.float64, device="cuda")
    eng.generate_synthetic_device(0, n, m, nv, d.data_ptr(), stream=stream)
    torch.cuda.synchronize()
    mats = d.view(n, H * W).cpu().numpy()
    bad = d.clone().view(n, H, W)  # row 1 made unreachable: every LP ends infeasible in phase 1
    bad[:, 1, 1:].abs_()
    bad[:, 1, 0] = -100.0
    fin, work = torch.empty_like(d), torch.empty_like(d)
    st = torch.empty(n, dtype=torch.int32, device="cuda")
    val = torch.empty(n, dtype=torch.float64, device="cuda")
    pos = torch.empty(n * (W + H), dtype=torch.int32, device="cuda")
    cert = torch.empty(n * (W + H), dtype=torch.float64, device="cuda")
    for src, label in ((bad, "infeasible"), (d, "config2 finals")):
        eng.solve_batch_device(n, H, W, src.data_ptr(), opt, d_work=work.data_ptr(), d_status=st.data_ptr(),
                               d_value=val.data_ptr(), d_pos=pos.data_ptr(), d_matrices_out=fin.data_ptr(),
                               stream=stream)
        torch.cuda.synchronize()
        kernel_time(eng, n, H, W, fin, pos, st, val, cert, opt, stream, args.reps, args.hbm_gbs, label)
    del d, bad, fin, work

    # 2. config 2 end to end, pinned host buffers
    o_plain = eng.batch_outputs(n, H, W, pinned=True)
    o_cert = eng.batch_outputs(n, H, W, pinned=True)
    o_cert["certificate"] = eng.pinned_empty((n, W + H), np.float64)
    r = alternate(args.reps, {
        "plain": lambda: eng.solve_batch(mats, H, W, opt, out=o_plain),
        "cert": lambda: eng.solve_batch(mats, H, W, opt, out=o_cert, want_certificates=True)})
    print(f"config2 {n} x {H}x{W} end to end ms: solve_batch {r['plain'][0]:.2f} (min {r['plain'][1]:.2f}) | "
          f"with want_certificates {r['cert'][0]:.2f} (min {r['cert'][1]:.2f}); +{r['cert'][0] - r['plain'][0]:.2f} ms, "
          f"D2H of certificates {8 * (W + H) * n / 1e6:.1f} MB")

    # 3. one 25FV47-size LP through solve()
    g = BW.netlib_base("25FV47")
    model = model_of(g)
    t = tableau_model(model).tableau
    same = np.array_equal(t.dense().view(np.uint64) & ~np.uint64(1 << 63), g["matrix"].view(np.uint64) & ~np.uint64(1 << 63))
    r = alternate(args.reps, {"plain": lambda: yalps_b200.solve(model, engine=eng),
                              "cert": lambda: yalps_b200.solve(model, {"certificate": True}, engine=eng)})
    sol = yalps_b200.solve(model, {"certificate": True}, engine=eng)
    nz = sum(1 for _, v in sol["infeasibilityCertificate"] if v != 0)
    print(f"25FV47-size LP ({g['height']}x{g['width']}, tableau equal up to zero signs: {same}) through solve(): "
          f"status {sol['status']}, {nz} keys with a non-zero multiplier; ms {r['plain'][0]:.2f} (min {r['plain'][1]:.2f}) "
          f"| with certificate {r['cert'][0]:.2f} (min {r['cert'][1]:.2f})")
    eng.close()


if __name__ == "__main__":
    main()
