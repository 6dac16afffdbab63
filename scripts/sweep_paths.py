#!/usr/bin/env python
"""K1 (shared-memory resident) vs K2 (HBM/L2 resident) across tableau sizes and CTA widths, dense synthetic LPs
and sparse Netlib replicas: the data behind the automatic path / width policy (choose_route in yalps_b200.cu)."""
import json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch
import yalps_b200
from yalps_b200 import engine as E
from conftest import load_netlib
eng = yalps_b200.Engine(0)
stream = torch.cuda.current_stream().cuda_stream

def timeit(n, H, W, d, work, path, threads):
    st = torch.empty(n, dtype=torch.int32, device="cuda"); piv = torch.empty(n, 2, dtype=torch.int64, device="cuda")
    eng.set_tuning(path, threads)
    def run():
        if path == E.PATH_GMEM: work.copy_(d)
        eng.solve_batch_device(n, H, W, d.data_ptr(), d_work=work.data_ptr(), d_status=st.data_ptr(), d_pivots=piv.data_ptr(), stream=stream)
    try:
        run(); torch.cuda.synchronize()
    except Exception as e:
        return None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); run(); run(); e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 2
    if path == E.PATH_GMEM:
        e0.record(); work.copy_(d); work.copy_(d); e1.record(); torch.cuda.synchronize(); ms -= e0.elapsed_time(e1) / 2
    return ms, int(piv.sum().item())

cases = []
for (m, nv, n) in [(8, 16, 65536), (16, 32, 65536), (32, 64, 65536), (48, 96, 32768), (64, 128, 16384), (96, 192, 8192), (128, 256, 4096)]:
    H, W = m + 1, nv + 1
    d = torch.empty(n * H * W, dtype=torch.float64, device="cuda")
    eng.generate_synthetic_device(0, n, m, nv, d.data_ptr())
    cases.append((f"dense {m}x{nv}", n, H, W, d))
NL = load_netlib()
for name, n in (("AFIRO", 65536), ("SC50A", 65536), ("ADLITTLE", 32768), ("BLEND", 16384), ("SC105", 16384)):
    g = NL.get(name); H, W = g["height"], g["width"]
    d = torch.empty(n * H * W, dtype=torch.float64, device="cuda")
    eng.generate_replicas_device(0, n, g["matrix"], H, W, g["row_groups"], d.data_ptr())
    cases.append((f"netlib {name}", n, H, W, d))
for label, n, H, W, d in cases:
    work = torch.empty_like(d)
    for path, pn in ((E.PATH_SMEM, "K1"), (E.PATH_GMEM, "K2")):
        for threads in (32, 64, 128, 256, 512):
            r = timeit(n, H, W, d, work, path, threads)
            if r is None: continue
            ms, p = r
            print(json.dumps({"case": label, "shape": [H, W], "n": n, "kernel": pn, "threads": threads, "ms": round(ms, 3),
                              "Mpivots_per_s": round(p / ms / 1e3, 2), "kLPs_per_s": round(n / ms, 1)}), flush=True)
    del work
eng.close()
