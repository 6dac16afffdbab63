"""bench.py --dump-outputs: what the timed step returned, written as float32 / float64 .npy files within a size budget,
on a fixed sample of LPs when the batch's outputs are larger."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, same_bits

import bench


def _fake_outputs(n, H=5, W=4):
    rng = np.random.default_rng(1)
    return {"status": rng.integers(0, 5, n, dtype=np.int32), "value": rng.standard_normal(n),
            "pivots": rng.integers(0, 1000, (n, 2), dtype=np.int64), "rhs": rng.standard_normal((n, H)),
            "pos": rng.integers(0, W + H, (n, W + H), dtype=np.int32), "var": rng.integers(0, W + H, (n, W + H), dtype=np.int32)}


def _read(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def _check(got, ref):
    idx = got.pop("lp_index").astype(np.int64)
    assert sorted(got) == sorted(ref)
    for k, a in got.items():
        assert a.dtype == (np.float32 if ref[k].dtype == np.int32 else np.float64), k
        assert np.array_equal(a.view(np.uint8), ref[k][idx].astype(a.dtype).view(np.uint8)), k
    return idx


def test_small_batch_is_written_whole(tmp_path):
    ref = _fake_outputs(300)
    bench.dump_outputs(str(tmp_path), {k: torch.from_numpy(v) for k, v in ref.items()})
    assert np.array_equal(_check(_read(tmp_path), ref), np.arange(300))


def test_large_batch_is_a_fixed_sample_within_the_budget(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 200_000)
    ref = _fake_outputs(3000)
    idx = []
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), {k: torch.from_numpy(v) for k, v in ref.items()})
        assert sum(os.path.getsize(tmp_path / run / f) for f in os.listdir(tmp_path / run)) <= bench.DUMP_BYTES
        idx.append(_check(_read(tmp_path / run), ref))
    assert 0 < len(idx[0]) < 3000 and np.all(np.diff(idx[0]) > 0)
    assert np.array_equal(idx[0], idx[1])


@pytest.mark.gpu
def test_bench_dump_matches_the_oracle(tmp_path):
    from oracle import lib as O
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
           "--workload", "small", "--dump-outputs", str(tmp_path)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    n, m, nv, neg = bench.WORKLOADS["small"]
    r = O.simplex_batch(O.generate_synthetic(0, n, m, nv, neg), nv + 1, m + 1, nthreads=os.cpu_count() or 1)
    got = _read(tmp_path)
    assert np.array_equal(got["lp_index"], np.arange(n))
    for k in ("status", "pivots", "pos", "var"):
        assert np.array_equal(got[k], r[k]), k
    assert same_bits(got["value"], r["value"]) and same_bits(got["rhs"], r["rhs"])
