"""Every narrower batch entry point of include/yalps_b200.h is its widest sibling called with NULL for the extras, bit
for bit.  The Python layer only calls the widest entries, so each narrower one is called here once, through _ffi, on
a batch with infeasible rows and tiny, huge and signed-zero cells -- below and above the 768 KB zero-copy limit, so
that both the small call and the chunk pipeline run."""
import ctypes as C

import numpy as np
import pytest

import yalps_b200
from conftest import same_bits
from test_gpu_sensitivity import special_batch
from yalps_b200 import engine as E

pytestmark = pytest.mark.gpu

SIZES = {"small": (40, 16, 32), "chunked": (300, 32, 64)}  # n, m, nvars: 0.18 MB and 5.1 MB of tableaus


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _outputs(n, rows, pvs, cells):
    """Output arrays filled with a pattern, so that an output one call writes and the other does not shows."""
    return {"status": np.full(n, -7, np.int32), "value": np.full(n, 7.5), "pivots": np.full(2 * n, -7, np.int64),
            "rhs": np.full(rows, 7.5), "pos": np.full(pvs, -7, np.int32), "var": np.full(pvs, -7, np.int32),
            "matrices": None if cells is None else np.full(cells, 7.5)}


def _check_same(call, n, rows, pvs, cells=None):
    """call(out, widest) -> return code; the narrow and the widest call agree in every output bit."""
    narrow, wide = _outputs(n, rows, pvs, cells), _outputs(n, rows, pvs, cells)
    assert call(narrow, False) == 0 and call(wide, True) == 0
    for k, v in narrow.items():
        if v is not None:
            assert same_bits(v, wide[k]) if v.dtype == np.float64 else np.array_equal(v, wide[k]), k


def _batch(size):
    n, m, nv = SIZES[size]
    return special_batch(n, m, nv, seed=n), n, m + 1, nv + 1


def _ragged(size):
    n, m, nv = SIZES[size]
    shapes = [[(m + 1, nv + 1), (9, 17), (m // 2 + 1, nv // 2 + 1)][i % 3] for i in range(n)]
    mats = [special_batch(1, h - 1, w - 1, seed=i)[0] for i, (h, w) in enumerate(shapes)]
    heights = np.asarray([s[0] for s in shapes], np.int32)
    widths = np.asarray([s[1] for s in shapes], np.int32)
    offs = np.zeros(n + 1, np.int64)
    np.cumsum(heights.astype(np.int64) * widths, out=offs[1:])
    return np.concatenate(mats), heights, widths, offs, n


def _outs(o):
    return _p(o["status"]), _p(o["value"]), _p(o["pivots"]), _p(o["rhs"]), _p(o["pos"]), _p(o["var"])


@pytest.mark.parametrize("size", SIZES)
def test_batch_entries(engine, size):
    lib, ctx, opt = engine._lib, engine._ctx, E.make_options()
    mats, n, H, W = _batch(size)
    m = _p(mats)
    for narrow in ("yalps_solve_batch", "yalps_solve_batch_basis", "yalps_solve_batch_duals"):
        def call(o, widest, narrow=narrow):
            if widest:
                return lib.yalps_solve_batch_ranging(ctx, n, H, W, m, None, None, C.byref(opt), *_outs(o),
                                                     _p(o["matrices"]), None, None, None, None)
            if narrow == "yalps_solve_batch":
                return lib.yalps_solve_batch(ctx, n, H, W, m, C.byref(opt), *_outs(o), _p(o["matrices"]))
            if narrow == "yalps_solve_batch_basis":
                return lib.yalps_solve_batch_basis(ctx, n, H, W, m, None, None, C.byref(opt), *_outs(o),
                                                   _p(o["matrices"]))
            return lib.yalps_solve_batch_duals(ctx, n, H, W, m, None, None, C.byref(opt), *_outs(o), _p(o["matrices"]),
                                               None)
        _check_same(call, n, n * H, n * (H + W), n * H * W)


@pytest.mark.parametrize("size", SIZES)
def test_ragged_entries(engine, size):
    lib, ctx, opt = engine._lib, engine._ctx, E.make_options()
    packed, heights, widths, offs, n = _ragged(size)
    hw, mo = (_p(heights), _p(widths)), _p(offs[:-1].copy())
    rows, pvs = int(heights.sum()), int(heights.sum() + widths.sum())
    for narrow in ("yalps_solve_ragged", "yalps_solve_ragged_basis", "yalps_solve_ragged_duals"):
        def call(o, widest, narrow=narrow):
            mat = _p(o["matrices"])
            if widest:
                return lib.yalps_solve_ragged_ranging(ctx, n, *hw, mo, _p(packed), None, None, C.byref(opt), *_outs(o),
                                                      mat, None, None, None, None)
            if narrow == "yalps_solve_ragged":
                return lib.yalps_solve_ragged(ctx, n, *hw, mo, _p(packed), C.byref(opt), *_outs(o), mat)
            if narrow == "yalps_solve_ragged_basis":
                return lib.yalps_solve_ragged_basis(ctx, n, *hw, mo, _p(packed), None, None, C.byref(opt), *_outs(o), mat)
            return lib.yalps_solve_ragged_duals(ctx, n, *hw, mo, _p(packed), None, None, C.byref(opt), *_outs(o), mat,
                                                None)
        _check_same(call, n, rows, pvs, packed.size)


@pytest.mark.parametrize("size", SIZES)
def test_replica_entries(engine, size):
    lib, ctx, opt = engine._lib, engine._ctx, E.make_options()
    mats, n, H, W = _batch(size)
    base = np.ascontiguousarray(mats[0])
    rhs = np.ascontiguousarray(mats.reshape(n, H, W)[:, :, 0])

    def call(o, widest):
        if widest:
            return lib.yalps_solve_replicas_duals(ctx, n, H, W, _p(base), _p(rhs), C.byref(opt), *_outs(o), None)
        return lib.yalps_solve_replicas(ctx, n, H, W, _p(base), _p(rhs), C.byref(opt), *_outs(o))
    _check_same(call, n, n * H, n * (H + W))


@pytest.mark.parametrize("size", SIZES)
def test_device_entries(engine, size):
    import torch
    lib, ctx, opt = engine._lib, engine._ctx, E.make_options()
    mats, n, H, W = _batch(size)
    d_in = torch.from_numpy(mats.reshape(-1)).cuda()
    stream = torch.cuda.current_stream().cuda_stream
    z = lambda t: C.c_void_p(t.data_ptr())

    def call(o, widest):
        d = {k: torch.from_numpy(v).cuda() for k, v in o.items() if v is not None}
        work, mout = torch.empty_like(d_in), torch.full_like(d_in, 7.5)
        args = (ctx, n, H, W, z(d_in), z(work), C.byref(opt), z(d["status"]), z(d["value"]), z(d["pivots"]),
                z(d["rhs"]), z(d["pos"]), z(d["var"]), z(mout), C.c_void_p(stream))
        rc = lib.yalps_solve_batch_device_duals(*args, None) if widest else lib.yalps_solve_batch_device(*args)
        torch.cuda.synchronize()
        for k, t in d.items():
            o[k][:] = t.cpu().numpy()
        o["matrices"][:] = mout.cpu().numpy()
        return rc
    _check_same(call, n, n * H, n * (H + W), n * H * W)


@pytest.mark.parametrize("size", SIZES)
def test_multi_rank_entries(size):
    opt = E.make_options()
    mats, n, H, W = _batch(size)
    packed, heights, widths, offs, rn = _ragged(size)
    hw, mo = (_p(heights), _p(widths)), _p(offs[:-1].copy())
    rows, pvs = int(heights.sum()), int(heights.sum() + widths.sum())
    base = np.ascontiguousarray(mats[0])
    rhs = np.ascontiguousarray(mats.reshape(n, H, W)[:, :, 0])
    with yalps_b200.MultiEngine([0, 0]) as multi:
        lib, mh = multi._lib, multi._m
        for narrow in ("yalps_multi_solve_batch", "yalps_multi_solve_batch_duals"):
            def call(o, widest, narrow=narrow):
                args = (mh, n, H, W, _p(mats), None, None, C.byref(opt), *_outs(o), _p(o["matrices"]))
                if widest:
                    return lib.yalps_multi_solve_batch_ranging(*args, None, None, None, None)
                return getattr(lib, narrow)(*args, *((None,) if narrow.endswith("_duals") else ()))
            _check_same(call, n, n * H, n * (H + W), n * H * W)
        for narrow in ("yalps_multi_solve_ragged", "yalps_multi_solve_ragged_duals"):
            def call(o, widest, narrow=narrow):
                args = (mh, rn, *hw, mo, _p(packed), C.byref(opt), *_outs(o), _p(o["matrices"]))
                if widest:
                    return lib.yalps_multi_solve_ragged_ranging(*args, None, None, None, None)
                return getattr(lib, narrow)(*args, *((None,) if narrow.endswith("_duals") else ()))
            _check_same(call, rn, rows, pvs, packed.size)

        def call(o, widest):
            args = (mh, n, H, W, _p(base), _p(rhs), C.byref(opt), *_outs(o))
            return lib.yalps_multi_solve_replicas_duals(*args, None) if widest else lib.yalps_multi_solve_replicas(*args)
        _check_same(call, n, n * H, n * (H + W))
