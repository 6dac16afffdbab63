#!/usr/bin/env python
"""bench.py -- headline benchmark of the batched simplex hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--workload config2|...]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path (the batched simplex kernel) over one batch of synthetic LPs.
N=1 workload = BASELINE.json configs[1]: 65,536 synthetic feasible dense LPs 32x64 (tableau 33x65 fp64),
generated on the device with the integer-hash PRNG of the reference's test helpers (SURVEY 8d).
For N>1 (torchrun, one rank per GPU) every rank solves its own 65,536 LPs (weak scaling, no data-path
collective: LPs are independent); the time is the max over ranks, the value the sum of all ranks' pivots.

`value`     pivots/s with the tableaus already resident in HBM (device entry point of the C ABI)
`e2e`       pivots/s through the host C-ABI call (yalps_solve_batch) from pinned host buffers, H2D of the
            tableaus and D2H of status/value/pivots/RHS/basis inside the timed region
`roofline`  SURVEY 8(d): algorithmic bytes = 16*W*(1+R) + 8*(2(H-1)+2(W-1)) per pivot with R, the rows a pivot
            rewrites, COUNTED ON THE DEVICE in a measuring pass, against the shared-memory stream bandwidth
            measured live (north_star's denominator; K1 keeps the tableau in shared memory).  The automatic
            path for this workload is K1t, which keeps the tableau in TENSOR memory: its own stream bandwidth
            (tcgen05.ld/st, measured live too) and the HBM view are reported alongside
`secondary` (N=1 only) BASELINE.json configs 3, 4, 5 and 1 (AFIRO, last) with the same fields per workload (bench_workloads.py)
`cpu_baseline` the CPU restatement of the reference loop (oracle/, C -O2 -ffp-contract=off; Node is not
            available) on the box's host cores, bounded sample of the same workload

--impl reference times that CPU restatement alone (all host threads) and prints the same JSON shape.

--dump-outputs DIR writes what the last timed step returned for rank 0's LPs (status, value, pivots, RHS, basis) as
DIR/<name>.npy, so that two builds can be compared output for output on the same generated inputs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (n LPs per GPU, m rows, n vars, neg rows)
    "config2": (65536, 32, 64, 0),
    "config2_phase1": (65536, 32, 64, 8),
    "small": (4096, 32, 64, 0),
}
METRIC = "batched_simplex_pivots_per_s"


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "20"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def bind_to_gpu_numa_node(index):
    """Pin this rank to the CPUs of the NUMA node its GPU hangs off, BEFORE any pinned allocation (first-touch puts
    the staging buffers next to the GPU's PCIe root): with 8 ranks streaming 1.1 GB per step each, host tableaus that
    cross the socket interconnect halve the end-to-end rate.  Best effort; returns a description for the JSON line."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(index)],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if not out:
            return None
        bus = out[-12:] if len(out) >= 12 else out  # 00000000:1B:00.0 -> 0000:1b:00.0
        base = f"/sys/bus/pci/devices/{bus}"
        node = int(open(base + "/numa_node").read().strip())
        if node < 0:
            return None
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.extend(range(int(a), int(b or a) + 1))
        allowed = sorted(set(cpus) & os.sched_getaffinity(0))
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return {"numa_node": node, "cpus": len(allowed)}
    except Exception:
        return None


def cpu_baseline(n_lp, m, nv, neg, first, threads, salt=0x5BD1E995):
    """Times the oracle (CPU restatement of the reference loop) on n_lp LPs of the workload."""
    import numpy as np
    from oracle import lib as O
    mats = O.generate_synthetic(first, n_lp, m, nv, neg, salt)
    t0 = time.perf_counter()
    res = O.simplex_batch(mats, nv + 1, m + 1, nthreads=threads, want_pos=False)
    dt = time.perf_counter() - t0
    piv = int(res["pivots"].sum())
    assert (res["status"] == 0).all() or neg > 0
    return piv / dt, n_lp / dt, piv, dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    n, m, nv, neg = WORKLOADS[args.workload]
    cores = host_cores()
    sample = n  # every step is the whole batch of the native arm's step (same config, same sample as its cpu_baseline)
    for _ in range(args.warmup):
        cpu_baseline(min(sample, 2048), m, nv, neg, 0, cores)
    tot_piv, tot_t, tot_lp = 0, 0.0, 0
    rates = []  # per-step samples, as benchmarks/benchmark.ts:64-79 reports mean and standard deviation
    for s in range(args.steps):
        _, _, piv, dt = cpu_baseline(sample, m, nv, neg, (s * sample) % n, cores)
        tot_piv += piv
        tot_t += dt
        tot_lp += sample
        rates.append(piv / dt)
    value = tot_piv / tot_t
    mean = sum(rates) / len(rates)
    sigma = (sum((r - mean) ** 2 for r in rates) / max(1, len(rates) - 1)) ** 0.5
    one_thread = cpu_baseline(2048, m, nv, neg, 0, 1)[0]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "pivots/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args.workload, n, m, nv, neg), "l2": "inputs larger than L2"},
        "lps_per_s": tot_lp / tot_t,
        "samples": {"n": len(rates), "mean": mean, "stddev": sigma, "unit": "pivots/s"},
        "cpu_baseline": {"value": value, "unit": "pivots/s", "cores": cores, "kind": "port",
                         "sample": f"all {sample} LPs of one step per step, {cores} threads; single thread: "
                                   f"{one_thread:.4g} pivots/s",
                         "note": "C restatement of src/simplex.ts (oracle/), not Node/V8: no JS engine in this image"},
        "e2e": {"value": value, "unit": "pivots/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit_line(line)
    return 0


def workload_name(name, n, m, nv, neg):
    return (f"{name}: {n} synthetic dense LPs {m}x{nv} fp64 per GPU (tableau {m + 1}x{nv + 1}, "
            f"{'feasible start' if not neg else str(neg) + ' infeasible rows'}), BASELINE.json configs[1]; tableaus stay on chip "
            f"for the whole solve (automatic kernel: one LP per warp in tensor memory, K1t; --path 1: one LP per CTA in "
            f"shared memory, K1)")


def run_native(args):
    import numpy as np
    import torch
    import yalps_b200
    from yalps_b200.engine import make_options

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    all_cpus = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa_node(local) if world > 1 else None
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)

    n, m, nv, neg = WORKLOADS[args.workload]
    H, W = m + 1, nv + 1
    cells = H * W
    eng = yalps_b200.Engine(local)
    if args.threads or args.path:
        eng.set_tuning(args.path, args.threads)
    opt = make_options()
    stream = torch.cuda.current_stream().cuda_stream

    # ---- inputs resident in HBM (LP ids are disjoint per rank)
    d_in = torch.empty(n * cells, dtype=torch.float64, device=dev)
    eng.generate_synthetic_device(rank * n, n, m, nv, d_in.data_ptr(), neg_rows=neg, stream=stream)
    d_status = torch.empty(n, dtype=torch.int32, device=dev)
    d_value = torch.empty(n, dtype=torch.float64, device=dev)
    d_piv = torch.empty(n, 2, dtype=torch.int64, device=dev)
    d_rhs = torch.empty(n, H, dtype=torch.float64, device=dev)
    d_pos = torch.empty(n, W + H, dtype=torch.int32, device=dev)
    d_var = torch.empty(n, W + H, dtype=torch.int32, device=dev)

    def step():
        eng.solve_batch_device(n, H, W, d_in.data_ptr(), opt, d_status=d_status.data_ptr(),
                               d_value=d_value.data_ptr(), d_pivots=d_piv.data_ptr(), d_rhs=d_rhs.data_ptr(),
                               d_pos=d_pos.data_ptr(), d_var=d_var.data_ptr(), stream=stream)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    pivots_per_step = int(d_piv.sum().item())
    statuses = torch.bincount(d_status.to(torch.int64), minlength=5).tolist()
    # measuring pass: rows rewritten by the rank-1 updates (R of SURVEY 8d), counted by the kernel itself
    d_rows = torch.zeros(1, dtype=torch.int64, device=dev)
    eng.set_row_counter(d_rows.data_ptr(), per_lp=False)
    step()
    torch.cuda.synchronize()
    eng.set_row_counter(0)
    rows_per_step = int(d_rows.item())

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = eng.launch_count
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    t_begin = torch.cuda.Event(enable_timing=True)
    t_end = torch.cuda.Event(enable_timing=True)
    t_begin.record()
    for e0, e1 in evs:
        e0.record()
        step()
        e1.record()
    t_end.record()
    barrier()
    launches = eng.launch_count - launches0
    elapsed_ms = t_begin.elapsed_time(t_end)
    kernel_ms = sum(e0.elapsed_time(e1) for e0, e1 in evs) / args.steps

    # ---- e2e: host buffers through the reference-facing C-ABI call
    h_in = eng.pinned_empty((n * cells,), np.float64)
    torch.cuda.synchronize()
    h_in[:] = d_in.cpu().numpy()
    e2e_steps = max(1, min(args.steps, 5))
    h_out = eng.batch_outputs(n, H, W, pinned=True)
    out = eng.solve_batch(h_in, H, W, opt, out=h_out)  # warm-up (allocates the device staging pool)
    assert int(out["pivots"].sum()) == pivots_per_step
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        out = eng.solve_batch(h_in, H, W, opt, out=h_out)
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    # the bare copy of the same bytes on every rank at once: what the box's PCIe / host-memory fabric allows
    barrier()
    h2d_s = eng.measure_h2d_seconds(h_in, reps=3, nstreams=2)
    clocks = sampler.stop() if rank == 0 else None  # sampled over the device-timed and the end-to-end regions
    if args.dump_outputs and rank == 0:  # the timed step's outputs: the end-to-end calls use their own buffers
        dump_outputs(args.dump_outputs, {"status": d_status, "value": d_value, "pivots": d_piv, "rhs": d_rhs,
                                         "pos": d_pos, "var": d_var})
    h2d = n * cells * 8
    d2h = n * (4 + 8 + 16 + H * 8 + 2 * (W + H) * 4)

    # ---- max over ranks, sum of work
    t = torch.tensor([elapsed_ms, e2e_s * 1e3, kernel_ms, h2d_s * 1e3], dtype=torch.float64, device=dev)
    work = torch.tensor([float(pivots_per_step)], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(work, op=dist.ReduceOp.SUM)
    elapsed_ms, e2e_ms, kernel_ms_max, h2d_ms = (float(x) for x in t.tolist())
    total_pivots_step = float(work.item())

    if rank == 0:
        value = total_pivots_step * args.steps / (elapsed_ms * 1e-3)
        import bench_workloads as BW
        alg_bytes = BW.pivot_bytes(H, W, pivots_per_step, rows_per_step)  # SURVEY 8(d) with the counted R
        bytes_per_pivot = alg_bytes / pivots_per_step
        achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
        smem_gbs, _ = eng.measure_smem_bandwidth()
        tmem_gbs, _ = eng.measure_tmem_bandwidth()
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        hbm_alg = n * (cells * 8 + 4 + 8 + 16 + H * 8 + 2 * (W + H) * 4) / (kernel_ms * 1e-3) / 1e9
        traffic = None
        try:  # dram bytes per launch of this kernel from the committed ncu --set full capture (profiles/)
            ncu = json.load(open(os.path.join(ROOT, "profiles", "r01k_k1t_ncu_summary.json")))
            if args.workload == "config2":
                traffic = ncu["dram_bytes_per_launch"]
        except (OSError, KeyError, ValueError):
            pass
        os.sched_setaffinity(0, all_cpus)  # the CPU baseline uses every host core again
        cores = host_cores()
        cpu_n = n  # the whole batch of one step, several times over: a few seconds of CPU work in total
        cpu_baseline(min(n, 4096), m, nv, neg, 0, cores)  # warm-up (thread pool, page faults)
        reps = [cpu_baseline(cpu_n, m, nv, neg, 0, cores) for _ in range(5)]
        cpu_v = sum(r[2] for r in reps) / sum(r[3] for r in reps)
        cpu_lps = cpu_n * len(reps) / sum(r[3] for r in reps)
        cpu_dt = sum(r[3] for r in reps)
        cpu_1, _, _, _ = cpu_baseline(min(n, 4096), m, nv, neg, 0, 1)
        line = {
            "metric": METRIC, "value": value, "unit": "pivots/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(args.workload, n, m, nv, neg),
                       "l2": f"inputs larger than L2 ({n * cells * 8 / 1e6:.0f} MB per GPU read every step)",
                       "parallelism": f"{world} x independent LP shards, no collective on the data path",
                       "pivots_per_step_per_gpu": pivots_per_step, "status_counts": statuses},
            "lps_per_s": n * world * args.steps / (elapsed_ms * 1e-3),
            "e2e": {"value": total_pivots_step / (e2e_ms * 1e-3), "unit": "pivots/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms, "lps_per_s": n * world / (e2e_ms * 1e-3),
                    "api": "yalps_solve_batch (host pointers; pinned input and output buffers; chunked H2D/kernel/D2H pipeline)",
                    "pcie_gbs": (h2d + d2h) * world / (e2e_ms * 1e-3) / 1e9, "numa_binding": numa,
                    "h2d_ceiling_gbs": h2d * world / (h2d_ms * 1e-3) / 1e9,
                    "h2d_ceiling_note": "bare cudaMemcpyAsync of the same pinned tableaus on all ranks at once (two streams per "
                                        "GPU, max over ranks): the end-to-end step cannot beat h2d_bytes / this rate",
                    "ms_floor_from_ceiling": h2d_ms},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": {"bound": "smem", "achieved": achieved, "peak": smem_gbs, "unit": "GB/s",
                         "frac": achieved / smem_gbs, "traffic": traffic,
                         "traffic_note": "dram__bytes_read+write per launch (ncu --set full, profiles/r01k_k1t_ncu_summary.json); "
                                         "the tableau is read from HBM once, every pivot runs out of tensor memory",
                         "peak_source": "measured live: ld/st.shared.f64 stream on all SMs (yalps_measure_smem_bandwidth)",
                         "bytes_per_unit": bytes_per_pivot, "units_per_launch": pivots_per_step,
                         "bytes_formula": "16*W*(pivots + rows_rewritten) + pivots*8*(2(H-1)+2(W-1)), SURVEY 8(d)",
                         "rows_rewritten": rows_per_step, "mean_rows_per_pivot": rows_per_step / pivots_per_step,
                         "rows_dense": H - 1,
                         "kernel_ms": kernel_ms,
                         "kernel": "k_simplex_tmem (K1t)" if args.path in (0, 6) and args.threads == 0 else "k_simplex<NW,KC,resident>",
                         "tmem": {"achieved": achieved, "peak": tmem_gbs, "frac": achieved / tmem_gbs,
                                  "peak_source": "measured live: tcgen05.ld/st.32x32b.x32 read-modify-write stream, 16 warps/SM "
                                                 "(yalps_measure_tmem_bandwidth)",
                                  "note": "K1t keeps the tableau rows in tensor memory; the shared-memory stream stays the "
                                          "headline denominator because BASELINE.json's target is quoted on it"},
                         "hbm": {"achieved": hbm_alg, "peak": hbm_peak, "frac": hbm_alg / hbm_peak,
                                 "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback",
                                 "note": "tableau read once + results written once per LP"}},
            "cpu_baseline": {"value": cpu_v, "unit": "pivots/s", "cores": cores, "kind": "port",
                             "sample": f"all {cpu_n} LPs of one step, 5 passes, {cores} threads, {cpu_dt:.2f} s in total; "
                                       f"single thread {cpu_1:.4g} pivots/s",
                             "lps_per_s": cpu_lps,
                             "note": "C restatement of src/simplex.ts (oracle/), not Node/V8"},
        }
        if world == 1 and args.workload == "config2" and not args.no_secondary:
            line["secondary"] = BW.run_all(torch, eng, hbm_peak, cores)
        if world > 1 and args.workload == "config2" and not args.no_secondary:
            # strong scaling of ONE large LP over the N GPUs, driven by this process alone (the other ranks wait on the
            # host, their GPUs idle: a NCCL barrier kernel would sit on the SMs the cooperative kernels need)
            try:
                del d_in, d_rhs, d_pos, d_var
                torch.cuda.empty_cache()
                line["multi_gpu_large_lp"] = BW.config5_multi(torch, eng, list(range(world)))
            except Exception as e:  # the headline must survive a failure of the extra measurement
                line["multi_gpu_large_lp"] = {"error": f"{type(e).__name__}: {e}"}
        emit_line(line)
    if world > 1 and args.workload == "config2" and not args.no_secondary:
        from datetime import timedelta
        store = dist.distributed_c10d._get_default_store()
        if rank == 0:
            store.set("yalps_large_lp_done", "1")
        else:
            try:
                store.wait(["yalps_large_lp_done"], timedelta(seconds=300))
            except Exception:
                pass
    eng.close()
    if dist is not None:
        dist.destroy_process_group()
    return 0


DUMP_BYTES = 64 * 10**6


def dump_outputs(out_dir, arrays, seed=0):
    """Per-LP device outputs -> out_dir/<name>.npy: int32 fields as float32 (exact: they are far below 2**24), the
    rest as float64.  When the batch's outputs exceed DUMP_BYTES, every file holds the same fixed seeded sample of LPs
    (identical from run to run); lp_index.npy lists the LPs written, in order."""
    import numpy as np
    host = {k: v.cpu().numpy() for k, v in arrays.items()}
    host = {k: a.astype(np.float32 if a.dtype == np.int32 else np.float64) for k, a in host.items()}
    n = len(host["status"])
    per_lp = 8 + sum(a[:1].nbytes for a in host.values())  # lp_index included
    keep = min(n, (DUMP_BYTES - 4096) // per_lp)  # 4096: room for the .npy headers
    idx = np.arange(n) if keep == n else np.sort(np.random.default_rng(seed).choice(n, keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "lp_index.npy"), idx.astype(np.float64))
    for k, a in host.items():
        np.save(os.path.join(out_dir, k + ".npy"), np.ascontiguousarray(a[idx]))


def emit_line(line):
    """The JSON line goes to the REAL stdout; everything else a library prints there (NCCL's version banner) was
    sent to stderr by quiet_stdout()."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


def quiet_stdout():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["native", "reference"], default="native")
    ap.add_argument("--workload", choices=sorted(WORKLOADS), default="config2")
    ap.add_argument("--threads", type=int, default=0, help="threads per LP (0 = auto)")
    ap.add_argument("--path", type=int, default=0, help="0 auto, 1 smem (K1), 2 gmem (K2), 6 tmem (K1t)")
    ap.add_argument("--no-secondary", action="store_true", help="skip the configs 3/4/5 block of the N=1 line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32/float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs applies to --impl native")
    quiet_stdout()
    if args.impl == "reference":
        return run_reference(args)
    return run_native(args)


if __name__ == "__main__":
    sys.exit(main())
