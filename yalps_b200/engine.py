"""Engine: one context of libyalps_b200.so on one GPU (numpy in, numpy out).

This is the thin host layer north_star describes: it packs tableaus (RHS column 0, objective row 0,
src/tableau.ts:9-21) into host buffers and calls the C ABI; all arithmetic happens in the sm_100a
kernels.  Device-resident entry points take raw device pointers (e.g. `torch.Tensor.data_ptr()`).
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Optional, Sequence

import numpy as np

from . import _ffi
from ._ffi import Options, YalpsError

STATUS_NAMES = ("optimal", "infeasible", "unbounded", "timedout", "cycled")  # enum yalps_status

PATH_AUTO, PATH_SMEM, PATH_GMEM, PATH_GRID, PATH_CLUSTER, PATH_TMEM, PATH_GRID_RESIDENT = 0, 1, 2, 3, 5, 6, 7


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _basis_in(pos_in, var_in, size: int) -> tuple:
    p = None if pos_in is None else np.ascontiguousarray(pos_in, np.int32).reshape(-1)
    v = None if var_in is None else np.ascontiguousarray(var_in, np.int32).reshape(-1)
    for arr in (p, v):
        if arr is not None and arr.size != size:
            raise ValueError("pos_in / var_in need n*(width+height) entries")
    return p, v


def _pairs_in(pairs, n: int, rows: int):
    """pairs as int32 (n*rows for n uniform LPs of `rows` rows, or the packed rows of a ragged batch); a single LP's
    (rows,) array applies to every LP of a uniform batch."""
    if pairs is None:
        return None
    p = np.ascontiguousarray(pairs, np.int32).reshape(-1)
    if p.size == rows and n > 1:
        p = np.tile(p, n)
    if p.size != n * rows:
        raise ValueError("pairs needs one entry per tableau row (packed like rhs)")
    return p


# The per-LP outputs of a batch call, as the C Outputs table (csrc/yalps_b200.cu) describes them, in the order the
# widest entries take them: key, dtype, packing and the want_* flag that turns the output on (None: always on).
# Packing: a tuple is the shape of one LP's values; "row" is one value per tableau row (like rhs), "var" one per
# variable id (like pos) and "cell" one per cell of the final tableau.
_OUTPUTS = (
    ("status", np.int32, (), None),
    ("value", np.float64, (), None),
    ("pivots", np.int64, (2,), None),
    ("rhs", np.float64, "row", None),
    ("pos", np.int32, "var", "want_basis"),
    ("var", np.int32, "var", "want_basis"),
    ("matrices", np.float64, "cell", "want_matrices"),
    ("reduced", np.float64, "var", "want_duals"),
    ("range_lo", np.float64, "var", "want_ranges"),
    ("range_hi", np.float64, "var", "want_ranges"),
    ("certificate", np.float64, "var", "want_certificates"),
)
# Outputs a call passes only when it asks for them (else NULL), and adds to a reused `out` that lacks them.  The other
# outputs are passed as `out` holds them.
_EXTRAS = ("want_duals", "want_ranges", "want_certificates")


def _shape(n: int, pack, height: int, width: int) -> tuple:
    """The shape of one output of n uniform LPs."""
    if isinstance(pack, tuple):
        return (n,) + pack
    return (n, {"row": height, "var": height + width, "cell": height * width}[pack])


def _batch_outputs(n: int, height: int, width: int, want: dict, mk=np.empty) -> dict:
    """Fresh buffers of n uniform LPs: a key for every output up to the reduced costs, None where its flag is off (the
    ranges and certificates are keys only when asked for, see _add_outputs)."""
    return {key: mk(_shape(n, pack, height, width), dtype) if flag is None or want.get(flag) else None
            for key, dtype, pack, flag in _OUTPUTS if flag not in ("want_ranges", "want_certificates")}


def _add_outputs(out: dict, n: int, height: int, width: int, want: dict):
    """The extras a call wants, added to `out` where it lacks them."""
    for key, dtype, pack, flag in _OUTPUTS:
        if flag in _EXTRAS and want.get(flag) and out.get(key) is None:
            out[key] = np.empty(_shape(n, pack, height, width), dtype)


def _out_args(out: dict, want: dict, pairs=None, omit: tuple = ()) -> list:
    """The output arguments of a widest entry in table order, with the input `pairs` before range_lo; `omit`: the flags
    of outputs a narrower entry does not take."""
    args = []
    for key, _, _, flag in _OUTPUTS:
        if flag in omit:
            continue
        if key == "range_lo":
            args.append(_ptr(pairs))
        args.append(_ptr(out[key]) if flag not in _EXTRAS or want[flag] else None)
    return args


def _offsets(counts) -> np.ndarray:
    """n + 1 int64 prefix sums of per-LP counts."""
    offs = np.zeros(len(counts) + 1, np.int64)
    np.cumsum(counts, out=offs[1:])
    return offs


def _pack_ragged(tableaus: Sequence, heights: np.ndarray, widths: np.ndarray) -> tuple:
    """(cell offsets, n + 1 int64; the float64 tableaus back to back) of LPs of the given shapes."""
    offs = _offsets(heights.astype(np.int64) * widths)
    packed = np.empty(int(offs[-1]), np.float64)
    for i, t in enumerate(tableaus):
        packed[offs[i]:offs[i + 1]] = np.asarray(t, np.float64).reshape(-1)
    return offs, packed


def _solve_uniform(check, fn, handle, matrices, height: int, width: int, options, out, pos_in, var_in, pairs,
                   want: dict) -> dict:
    """Engine/MultiEngine.solve_batch through fn, a yalps_*solve_batch_certificate entry, on handle (ctx or multi)."""
    opt = options or make_options()
    m = np.ascontiguousarray(matrices, dtype=np.float64).reshape(-1)
    cells = height * width
    if cells <= 0 or m.size % cells:
        raise ValueError(f"matrices has {m.size} values, not a multiple of {height}x{width}")
    n = m.size // cells
    if out is None:
        out = _batch_outputs(n, height, width, want)
    elif out["status"].shape[0] != n:
        raise ValueError("out was allocated for a different batch size")
    _add_outputs(out, n, height, width, want)
    p, v = _basis_in(pos_in, var_in, n * (width + height))
    pr = _pairs_in(pairs, n, height) if want["want_ranges"] else None
    check(fn(handle, n, height, width, _ptr(m), _ptr(p), _ptr(v), C.byref(opt), *_out_args(out, want, pr)))
    return out


def _solve_replicas(check, fn, handle, base, rhs, height: int, width: int, options, out, want: dict) -> dict:
    """Engine/MultiEngine.solve_replicas through fn, a yalps_*solve_replicas_duals entry, on handle."""
    opt = options or make_options()
    b = np.ascontiguousarray(base, np.float64).reshape(-1)
    r = np.ascontiguousarray(rhs, np.float64).reshape(-1)
    if b.size != height * width or r.size % height:
        raise ValueError("base must hold height*width values and rhs n*height")
    n = r.size // height
    if out is None:
        out = _batch_outputs(n, height, width, want)
    _add_outputs(out, n, height, width, want)
    check(fn(handle, n, height, width, _ptr(b), _ptr(r), C.byref(opt),
             *_out_args(out, want, omit=("want_matrices", "want_ranges", "want_certificates"))))
    return out


def _solve_ragged(check, fn, handle, tableaus, shapes, options, pairs, want: dict, basis_in: bool) -> list:
    """Engine/MultiEngine.solve_ragged through fn, a yalps_*solve_ragged_certificate entry, on handle; basis_in: fn
    takes pos_in / var_in (passed as NULL)."""
    opt = options or make_options()
    n = len(tableaus)
    if n == 0:
        return []
    heights = np.asarray([s[0] for s in shapes], np.int32)
    widths = np.asarray([s[1] for s in shapes], np.int32)
    offs, packed = _pack_ragged(tableaus, heights, widths)
    at = {"row": _offsets(heights), "var": _offsets(heights.astype(np.int64) + widths), "cell": offs}
    out = {key: np.empty((n,) + pack if isinstance(pack, tuple) else int(at[pack][-1]), dtype)
           if flag is None or want[flag] else None for key, dtype, pack, flag in _OUTPUTS}
    pr = None if not want["want_ranges"] or pairs is None else _pairs_in(
        np.concatenate([np.asarray(p, np.int32).reshape(-1) for p in pairs]), 1, int(at["row"][-1]))
    check(fn(handle, n, _ptr(heights), _ptr(widths), _ptr(offs[:-1].copy()), _ptr(packed),
             *((None, None) if basis_in else ()), C.byref(opt), *_out_args(out, want, pr)))
    res = []
    for i in range(n):
        r = {"status": int(out["status"][i]), "value": float(out["value"][i]),
             "pivots": (int(out["pivots"][i, 0]), int(out["pivots"][i, 1]))}
        for key, _, pack, flag in _OUTPUTS:
            if isinstance(pack, str) and (flag not in _EXTRAS or want[flag]):
                a, o = out[key], at[pack]
                r["matrix" if key == "matrices" else key] = None if a is None else a[o[i]:o[i + 1]]
        res.append(r)
    return res


def _solve_warm(check, fn, handle, base, height: int, width: int, rhs, obj, options, final, pairs, want: dict,
                cells=None, add_rows=None, add_cols=None) -> dict:
    """Engine/MultiEngine.solve_warm (base: the dense initial tableau) and Engine.solve_warm_sparse (cells given, base:
    their values) through fn, a yalps_*solve_warm* entry, on handle; a yalps_*solve_warm_extend* entry when add_rows or
    add_cols is given."""
    opt = options or make_options()
    if not opt.precision >= 0.0:  # NaN fails too
        raise ValueError(f"precision must be >= 0, got {opt.precision}")
    H, W = int(height), int(width)
    if H < 1 or W < 1:
        raise ValueError(f"bad shape {H}x{W}")
    b = np.ascontiguousarray(base, np.float64).reshape(-1)
    if cells is None:
        if b.size != H * W:
            raise ValueError("base must hold height*width values")
        base_args = (_ptr(b),)
    else:
        cells = np.ascontiguousarray(cells, np.int32).reshape(-1)
        if cells.size != b.size:
            raise ValueError("cells and values must have the same length")
        base_args = (int(cells.size), _ptr(cells) if cells.size else None, _ptr(b) if b.size else None)
    r = None if rhs is None else np.ascontiguousarray(rhs, np.float64).reshape(-1)
    o = None if obj is None else np.ascontiguousarray(obj, np.float64).reshape(-1)
    extend = add_rows is not None or add_cols is not None
    if r is None and o is None and not extend:
        raise ValueError("rhs and obj may not both be None")
    if (r is not None and r.size % H) or (o is not None and o.size % W):
        raise ValueError("rhs must hold n*height values and obj n*width")
    counts = [] if r is None else [r.size // H]
    counts += [] if o is None else [o.size // W]
    K = M = 0
    ext_args = ()
    if extend:
        g = None if add_cols is None else np.ascontiguousarray(add_cols, np.float64)
        if g is not None and (g.ndim != 3 or g.shape[2] != H):
            raise ValueError("add_cols must be (n, M, height): M added columns per variant over the base rows")
        M = 0 if g is None else g.shape[1]
        a = None if add_rows is None else np.ascontiguousarray(add_rows, np.float64)
        if a is not None and (a.ndim != 3 or a.shape[2] != W + M):
            raise ValueError("add_rows must be (n, K, width + M): K added rows per variant over the base and added "
                             "columns")
        K = 0 if a is None else a.shape[1]
        counts += [x.shape[0] for x in (a, g) if x is not None]
        ext_args = (_ptr(a) if K else None, _ptr(g) if M else None)
    n = counts[0]
    if any(c != n for c in counts):
        raise ValueError("rhs, obj, add_rows and add_cols must describe the same number of variants")
    f = fp = fv = None
    if final is not None:
        f = np.ascontiguousarray(final[0], np.float64).reshape(-1)
        fp, fv = _basis_in(final[1], final[2], H + W)
        if f.size != H * W or fp is None or fv is None:
            raise ValueError("final is (matrix of height*width values, pos, var)")
    out = _batch_outputs(n, H + K, W + M, want)
    _add_outputs(out, n, H + K, W + M, want)
    pr = _pairs_in(pairs, n, H + K) if want["want_ranges"] else None
    bs, bv, bp = C.c_int32(), C.c_double(), np.zeros(2, np.int64)
    shape = (H, W, K, M) if extend else (H, W)
    check(fn(handle, n, *shape, *base_args, _ptr(f), _ptr(fp), _ptr(fv), _ptr(r), _ptr(o), *ext_args, C.byref(opt),
             C.byref(bs), C.byref(bv), _ptr(bp), *_out_args(out, want, pr)))
    out["base"] = None if final is not None else {"status": bs.value, "value": bv.value,
                                                   "pivots": (int(bp[0]), int(bp[1]))}
    return out


def _check_precision(opt: Options):
    if not opt.precision >= 0.0:  # NaN fails too
        raise ValueError(f"precision must be >= 0 for row subsets (a zeroed row is a removed row only then), "
                         f"got {opt.precision}")


def _iis(check, lib, ctx, height: int, width: int, options, matrix=None, cells=None, values=None) -> dict:
    """Engine/MultiEngine.iis (matrix given) and iis_sparse (cells, values given) on ctx."""
    opt = options or make_options()
    _check_precision(opt)
    rows = np.empty(max(int(height), 1), np.int32)
    status, count = C.c_int32(), C.c_int32()
    stats = np.zeros(5, np.int64)
    if matrix is not None:
        m = np.ascontiguousarray(matrix, np.float64).reshape(-1)
        if m.size != height * width:
            raise ValueError("matrix must hold height * width cells")
        check(lib.yalps_iis(ctx, height, width, _ptr(m), C.byref(opt), C.byref(status), _ptr(rows), C.byref(count),
                            _ptr(stats)))
    else:
        cells = np.ascontiguousarray(cells, np.int32).reshape(-1)
        values = np.ascontiguousarray(values, np.float64).reshape(-1)
        if cells.size != values.size:
            raise ValueError("cells and values must have the same length")
        check(lib.yalps_iis_sparse(ctx, height, width, int(cells.size), _ptr(cells) if cells.size else None,
                                   _ptr(values) if values.size else None, C.byref(opt), C.byref(status), _ptr(rows),
                                   C.byref(count), _ptr(stats)))
    return {"status": status.value, "rows": rows[:count.value].copy(), "rounds": int(stats[0]), "lps": int(stats[1]),
            "pivots": int(stats[2]), "irreducible": bool(status.value == 1 and stats[3] == 0 and stats[4] == 0)}


_STATS = ("nodes", "node_pivots", "max_cuts", "max_heap", "waves", "device_nodes", "wave_us", "bnb_us",
          "sharded_waves", "allreduces")


def _search_result(width: int, status, result, out_h, rhs, pos, var, stats, root: Optional[tuple] = None) -> dict:
    """The dict of a branch-and-cut call from its C outputs; root: (status, value, pivots) of the root LP, if reported.
    stats names its first len(stats) counters."""
    h = out_h.value
    res = {"status": status.value, "result": result.value, "height": h, "rhs": rhs[:h], "pos": pos[:width + h],
           "var": var[:width + h]}
    if root is not None:
        res.update(root_status=root[0].value, root_value=root[1].value,
                   root_pivots=(int(root[2][0]), int(root[2][1])))
    res["stats"] = {k: int(v) for k, v in zip(_STATS, stats)}
    return res


def make_options(precision=1e-8, max_pivots=8192, check_cycles=False, tolerance=0.0, timeout_ms=math.inf,
                 max_iterations=32768) -> Options:
    o = Options()
    o.precision = float(precision)
    o.max_pivots = float(max_pivots)
    o.tolerance = float(tolerance)
    o.timeout_ms = float(timeout_ms)
    o.max_iterations = float(max_iterations)
    o.check_cycles = 1 if check_cycles else 0
    o.reserved = 0
    return o


class Engine:
    def __init__(self, device: int = 0):
        self._lib = _ffi.load()
        self._ctx = C.c_void_p()
        rc = self._lib.yalps_create(int(device), C.byref(self._ctx))
        if rc != 0:
            msg = self._lib.yalps_last_error(None)
            raise YalpsError(rc, msg.decode() if msg else "yalps_create failed")
        self.device = int(device)

    # ------------------------------------------------------------------ plumbing
    def close(self):
        if getattr(self, "_ctx", None) and self._ctx.value:
            self._lib.yalps_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _check(self, rc: int):
        if rc != 0:
            msg = self._lib.yalps_last_error(self._ctx)
            raise YalpsError(rc, msg.decode() if msg else "")

    def device_info(self) -> dict:
        v = [C.c_int32() for _ in range(4)]
        self._check(self._lib.yalps_device_info(self._ctx, *[C.byref(x) for x in v]))
        return {"sm_count": v[0].value, "smem_per_block_optin": v[1].value, "cc": (v[2].value, v[3].value)}

    def set_tuning(self, path: int = PATH_AUTO, threads_per_lp: int = 0, row_groups: int = 0):
        self._check(self._lib.yalps_set_tuning(self._ctx, path, threads_per_lp))
        self._check(self._lib.yalps_set_row_groups(self._ctx, row_groups))

    def set_bnb_mode(self, mode: int):
        """0 = device-resident search when it fits (default), 1 = host wave driver only, 2 = device kernel only."""
        self._check(self._lib.yalps_bnb_set_mode(self._ctx, int(mode)))

    def set_wave(self, wave: int):
        self._check(self._lib.yalps_bnb_set_wave(self._ctx, int(wave)))

    @property
    def launch_count(self) -> int:
        return int(self._lib.yalps_launch_count(self._ctx))

    def set_row_counter(self, d_rows: int = 0, per_lp: bool = False):
        """Device uint64 counter(s) the kernels add the rewritten rows of every pivot to (0 = off)."""
        self._check(self._lib.yalps_set_row_counter(self._ctx, C.c_void_p(d_rows) if d_rows else None, int(per_lp)))

    def pinned_empty(self, shape, dtype) -> np.ndarray:
        """numpy array over page-locked memory (freed with the engine's process)."""
        dtype = np.dtype(dtype)
        n = int(np.prod(shape)) * dtype.itemsize
        p = C.c_void_p()
        self._check(self._lib.yalps_host_alloc(self._ctx, n, C.byref(p)))
        buf = (C.c_char * max(n, 1)).from_address(p.value)
        return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    # ------------------------------------------------------------------ simplex batches
    def batch_outputs(self, n: int, height: int, width: int, want_matrices: bool = False, want_basis: bool = True,
                      pinned: bool = False, want_duals: bool = False) -> dict:
        """Output buffers for solve_batch; pinned=True allocates them page-locked (reusable across calls)."""
        return _batch_outputs(n, height, width, {"want_matrices": want_matrices, "want_basis": want_basis,
                                                 "want_duals": want_duals}, self.pinned_empty if pinned else np.empty)

    def solve_batch(self, matrices: np.ndarray, height: int, width: int, options: Optional[Options] = None,
                    want_matrices: bool = False, want_basis: bool = True, out: Optional[dict] = None,
                    pos_in: Optional[np.ndarray] = None, var_in: Optional[np.ndarray] = None,
                    want_duals: bool = False, want_ranges: bool = False, pairs: Optional[np.ndarray] = None,
                    want_certificates: bool = False) -> dict:
        """n same-shape tableaus, `matrices` float64 of n*height*width values (not modified).
        `out` may be a dict from batch_outputs() to reuse (pinned) result buffers.
        pos_in / var_in (int32, n*(width+height)): the basis bookkeeping the tableaus arrive with (the node LPs of
        src/branchAndCut.ts:127); None = the identity of a fresh tableau (src/tableau.ts:95-98).
        want_duals: also out["reduced"] (n, width+height), row 0 of the final tableau per variable id
        (yalps_solve_batch_duals; yalps_b200.sensitivity turns it into shadow prices and reduced costs).
        want_ranges: also out["range_lo"], out["range_hi"] (n, width+height), the sensitivity ranges computed on the
        device from the final tableaus (yalps_solve_batch_ranging); `pairs` (int32 per row, -1 = none; one LP's
        (height,) array or n*height values) pairs the two rows of a key (yalps_b200.sensitivity.row_pairs).
        want_certificates: also out["certificate"] (n, width+height), the Farkas certificate of an infeasible LP or the
        ray of an unbounded one, computed on the device from the final tableaus (yalps_solve_batch_certificate; NaN
        for every other status)."""
        return _solve_uniform(self._check, self._lib.yalps_solve_batch_certificate, self._ctx, matrices, height, width,
                              options, out, pos_in, var_in, pairs,
                              {"want_matrices": want_matrices, "want_basis": want_basis, "want_duals": want_duals,
                               "want_ranges": want_ranges, "want_certificates": want_certificates})

    def simplex(self, tableau, options: Optional[Options] = None) -> tuple:
        """simplex(tableau, options) -> (status, number), src/simplex.ts:144, with the reference's in-place contract:
        `tableau` is a yalps_b200.Tableau (.matrix float64 height*width, .width, .height, .position_of_variable,
        .variable_at_position) and all three arrays are overwritten with the final state."""
        opt = options or make_options()
        m = tableau.matrix
        if not (isinstance(m, np.ndarray) and m.dtype == np.float64 and m.flags.c_contiguous):
            raise ValueError("tableau.matrix must be a contiguous float64 array (it is modified in place)")
        h, w = int(tableau.height), int(tableau.width)
        pos = np.ascontiguousarray(tableau.position_of_variable, np.int32)
        var = np.ascontiguousarray(tableau.variable_at_position, np.int32)
        status, value = np.empty(1, np.int32), np.empty(1, np.float64)
        self._check(self._lib.yalps_solve_batch_basis(self._ctx, 1, h, w, _ptr(m), _ptr(pos), _ptr(var), C.byref(opt),
                                                      _ptr(status), _ptr(value), None, None, _ptr(pos), _ptr(var),
                                                      _ptr(m)))
        tableau.position_of_variable[:] = pos
        tableau.variable_at_position[:] = var
        return STATUS_NAMES[int(status[0])], float(value[0])

    def solve_replicas(self, base: np.ndarray, rhs: np.ndarray, height: int, width: int,
                       options: Optional[Options] = None, want_basis: bool = True, out: Optional[dict] = None,
                       want_duals: bool = False) -> dict:
        """n replicas of `base` (height*width) that differ only in column 0: rhs is float64 (n, height).
        want_duals: also out["reduced"] (n, width+height), as solve_batch."""
        return _solve_replicas(self._check, self._lib.yalps_solve_replicas_duals, self._ctx, base, rhs, height, width,
                               options, out, {"want_basis": want_basis, "want_duals": want_duals})

    def solve_warm(self, base: np.ndarray, height: int, width: int, rhs: Optional[np.ndarray] = None,
                   obj: Optional[np.ndarray] = None, options: Optional[Options] = None, final: Optional[tuple] = None,
                   want_basis: bool = True, want_matrices: bool = False, want_duals: bool = False,
                   want_ranges: bool = False, pairs: Optional[np.ndarray] = None,
                   want_certificates: bool = False, add_rows: Optional[np.ndarray] = None,
                   add_cols: Optional[np.ndarray] = None) -> dict:
        """n variants of the LP whose initial tableau is `base` (height*width), each solved from the base's final
        basis (yalps_solve_warm; yalps_b200.warm states the start tableau): rhs float64 (n, height) gives each its own
        column 0, obj (n, width) its own row 0 (obj[:, 0] ignored); either may be None, not both.  final = (matrix, pos,
        var) of the base's final tableau, or None: the library solves the base first and keeps that tableau on the
        device.  Returns the outputs of solve_batch (same flags) plus out["base"]: {"status", "value", "pivots"} of the
        base when the library solved it, else None.  Bit-exact against the reference loop on the warm tableau, not
        against a cold solve of the changed model (the pivot path differs).
        add_rows float64 (n, K, width + M) and add_cols (n, M, height), either or both (yalps_solve_warm_extend): each
        variant also adds K constraint rows and M variable columns in initial-tableau form; rhs and obj may then both
        be None, and the outputs and pairs have the (height + K) x (width + M) shape."""
        extend = add_rows is not None or add_cols is not None
        return _solve_warm(self._check, self._lib.yalps_solve_warm_extend if extend else self._lib.yalps_solve_warm,
                           self._ctx, base, height, width, rhs, obj, options, final, pairs,
                           {"want_basis": want_basis, "want_matrices": want_matrices, "want_duals": want_duals,
                            "want_ranges": want_ranges, "want_certificates": want_certificates},
                           add_rows=add_rows, add_cols=add_cols)

    def solve_warm_sparse(self, cells: np.ndarray, values: np.ndarray, height: int, width: int,
                          rhs: Optional[np.ndarray] = None, obj: Optional[np.ndarray] = None,
                          options: Optional[Options] = None, final: Optional[tuple] = None, want_basis: bool = True,
                          want_matrices: bool = False, want_duals: bool = False, want_ranges: bool = False,
                          pairs: Optional[np.ndarray] = None, want_certificates: bool = False,
                          add_rows: Optional[np.ndarray] = None, add_cols: Optional[np.ndarray] = None) -> dict:
        """solve_warm with the base's initial tableau given as ordered (cell, value) stores into a zero matrix
        (yalps_solve_warm_sparse, yalps_solve_warm_extend_sparse): it is built on the device and never exists densely
        on the host."""
        extend = add_rows is not None or add_cols is not None
        fn = self._lib.yalps_solve_warm_extend_sparse if extend else self._lib.yalps_solve_warm_sparse
        return _solve_warm(self._check, fn, self._ctx, values, height, width, rhs, obj, options, final, pairs,
                           {"want_basis": want_basis, "want_matrices": want_matrices, "want_duals": want_duals,
                            "want_ranges": want_ranges, "want_certificates": want_certificates}, cells=cells,
                           add_rows=add_rows, add_cols=add_cols)

    def set_replica_sharing(self, on: bool = True):
        """solve_replicas: follow the base tableau's pivot path while a replica makes the same choices (default on)."""
        self._check(self._lib.yalps_set_replica_sharing(self._ctx, int(bool(on))))

    @property
    def replica_forks(self) -> int:
        """Replicas of the last solve_replicas call that left the shared path (-1: sharing was not used)."""
        return int(self._lib.yalps_replica_forks(self._ctx))

    def solve_ragged(self, tableaus: Sequence[np.ndarray], shapes: Sequence[tuple], options: Optional[Options] = None,
                     want_matrices: bool = False, want_duals: bool = False, want_ranges: bool = False,
                     pairs: Optional[Sequence] = None, want_certificates: bool = False) -> list:
        """LPs of different shapes in one call.  tableaus[i] is float64 of height_i*width_i values.
        want_duals: every result also has "reduced" (width_i+height_i values, as solve_batch).
        want_ranges: every result also has "range_lo", "range_hi" (as solve_batch); pairs[i] (height_i int32) or None.
        want_certificates: every result also has "certificate" (width_i+height_i values, as solve_batch)."""
        return _solve_ragged(self._check, self._lib.yalps_solve_ragged_certificate, self._ctx, tableaus, shapes,
                             options, pairs, {"want_basis": True, "want_matrices": want_matrices,
                                              "want_duals": want_duals, "want_ranges": want_ranges,
                                              "want_certificates": want_certificates}, basis_in=True)

    def solve_batch_device(self, n: int, height: int, width: int, d_matrices: int, options: Optional[Options] = None,
                           d_work: int = 0, d_status: int = 0, d_value: int = 0, d_pivots: int = 0, d_rhs: int = 0,
                           d_pos: int = 0, d_var: int = 0, d_matrices_out: int = 0, stream: int = 0,
                           d_reduced: int = 0):
        """Everything already in device memory (raw pointers); enqueues on `stream` and returns.
        d_reduced (float64, n*(width+height)): reduced costs per variable id, as solve_batch's out["reduced"]."""
        opt = options or make_options()
        z = lambda p: C.c_void_p(p) if p else None
        self._check(self._lib.yalps_solve_batch_device_duals(self._ctx, n, height, width, z(d_matrices), z(d_work),
                                                             C.byref(opt), z(d_status), z(d_value), z(d_pivots),
                                                             z(d_rhs), z(d_pos), z(d_var), z(d_matrices_out),
                                                             z(stream), z(d_reduced)))

    def ranging_device(self, n: int, height: int, width: int, d_matrices: int, d_pos: int, d_range_lo: int,
                       d_range_hi: int, precision: float = 1e-8, d_status: int = 0, d_pairs: int = 0, stream: int = 0):
        """Sensitivity ranges of n final tableaus already in device memory (yalps_ranging_device, raw pointers):
        d_pos int32 n*(width+height), d_status int32 n (0: all optimal), d_pairs int32 n*height (0: none); writes
        float64 n*(width+height) to d_range_lo / d_range_hi.  Enqueues on `stream` and returns."""
        z = lambda p: C.c_void_p(p) if p else None
        self._check(self._lib.yalps_ranging_device(self._ctx, n, height, width, z(d_matrices), z(d_pos), z(d_status),
                                                   z(d_pairs), float(precision), z(d_range_lo), z(d_range_hi),
                                                   z(stream)))

    def certificate_device(self, n: int, height: int, width: int, d_matrices: int, d_pos: int, d_status: int,
                           d_value: int, d_cert: int, precision: float = 1e-8, stream: int = 0):
        """Certificates of n final tableaus already in device memory (yalps_certificate_device, raw pointers): d_pos
        int32 n*(width+height), d_status int32 n, d_value float64 n, as a solve reported them; writes float64
        n*(width+height) to d_cert.  Enqueues on `stream` and returns."""
        z = lambda p: C.c_void_p(p) if p else None
        self._check(self._lib.yalps_certificate_device(self._ctx, n, height, width, z(d_matrices), z(d_pos),
                                                       z(d_status), z(d_value), float(precision), z(d_cert),
                                                       z(stream)))

    # ------------------------------------------------------------------ row subsets and irreducible infeasible subsets
    def solve_row_subsets(self, base: np.ndarray, keep: np.ndarray, height: int, width: int,
                          options: Optional[Options] = None, want_certificates: bool = False) -> dict:
        """n LPs of `base` (height*width) restricted to row subsets, expanded on the device (yalps_solve_row_subsets).
        keep: uint32 (n, words), words = (height + 31) // 32, bit r of word r // 32 keeps row r (row 0 always stays,
        bits of rows >= height must be clear); every other row is zeroed, which the simplex treats as removed.
        Returns status, value, pivots (as solve_batch) and support (uint32 (n, words): the rows whose Farkas multiplier
        is > +0.0, zero words unless infeasible); want_certificates adds certificate (n, width+height)."""
        opt = options or make_options()
        _check_precision(opt)
        words = (height + 31) // 32
        b = np.ascontiguousarray(base, np.float64).reshape(-1)
        k = np.ascontiguousarray(keep, np.uint32).reshape(-1)
        if b.size != height * width or k.size % words:
            raise ValueError("base must hold height*width values and keep n*((height+31)//32) words")
        n = k.size // words
        if height % 32 and n and (k.reshape(n, words)[:, -1] >> np.uint32(height % 32)).any():
            raise ValueError(f"keep has bits set for rows >= height {height}")
        out = {"status": np.empty(n, np.int32), "value": np.empty(n, np.float64), "pivots": np.empty((n, 2), np.int64),
               "support": np.empty((n, words), np.uint32)}
        if want_certificates:
            out["certificate"] = np.empty((n, width + height), np.float64)
        self._check(self._lib.yalps_solve_row_subsets(self._ctx, n, height, width, _ptr(b), _ptr(k), C.byref(opt),
                                                      _ptr(out["status"]), _ptr(out["value"]), _ptr(out["pivots"]),
                                                      _ptr(out.get("certificate")), _ptr(out["support"])))
        return out

    def iis(self, matrix: np.ndarray, height: int, width: int, options: Optional[Options] = None) -> dict:
        """An irreducible infeasible subset of the tableau's rows (yalps_iis): status (the model's own), rows (int32,
        ascending tableau rows; empty unless infeasible), rounds, lps and pivots (the work of the search, round 0
        included) and irreducible (False when a deletion test ended `cycled`, the timeout expired or the model is not
        infeasible)."""
        return _iis(self._check, self._lib, self._ctx, height, width, options, matrix=matrix)

    def iis_sparse(self, cells: np.ndarray, values: np.ndarray, height: int, width: int,
                   options: Optional[Options] = None) -> dict:
        """iis on a tableau given as ordered (cell, value) stores into a zero matrix (yalps_iis_sparse)."""
        return _iis(self._check, self._lib, self._ctx, height, width, options, cells=cells, values=values)

    def generate_synthetic_device(self, first: int, n: int, m: int, nvars: int, d_out: int, neg_rows: int = 0,
                                  salt: int = 0x5BD1E995, stream: int = 0):
        self._check(self._lib.yalps_generate_synthetic_device(self._ctx, first, n, m, nvars, neg_rows, salt,
                                                              C.c_void_p(d_out), C.c_void_p(stream) if stream else None))

    def generate_replicas_device(self, first: int, n: int, base: np.ndarray, height: int, width: int,
                                 group: np.ndarray, d_out: int, eps: float = 1e-2, salt: int = 0x2545F491,
                                 stream: int = 0):
        base = np.ascontiguousarray(base, np.float64).reshape(-1)
        group = np.ascontiguousarray(group, np.int32)
        ngroups = int(group.max()) + 1 if group.size else 0
        self._check(self._lib.yalps_generate_replicas_device(self._ctx, first, n, height, width, _ptr(base), _ptr(group),
                                                             ngroups, eps, salt, C.c_void_p(d_out),
                                                             C.c_void_p(stream) if stream else None))

    # ------------------------------------------------------------------ branch and cut
    def bnb_set_root(self, matrix: np.ndarray, height: int, width: int, pos: np.ndarray, var: np.ndarray,
                     max_extra_rows: int):
        m = np.ascontiguousarray(matrix, np.float64).reshape(-1)
        p = np.ascontiguousarray(pos, np.int32)
        v = np.ascontiguousarray(var, np.int32)
        self._check(self._lib.yalps_bnb_set_root(self._ctx, height, width, _ptr(m), _ptr(p), _ptr(v), max_extra_rows))
        self._root_shape = (height, width)

    def bnb_solve_nodes(self, cuts_per_node: Sequence[Sequence[tuple]], options: Optional[Options] = None,
                        want_matrices: bool = False) -> dict:
        """cuts_per_node[j] = [(sign, variable, value), ...] (Cut, src/branchAndCut.ts:18)."""
        opt = options or make_options()
        H, W = self._root_shape
        n = len(cuts_per_node)
        offs = np.zeros(n + 1, np.int32)
        np.cumsum([len(c) for c in cuts_per_node], out=offs[1:])
        flat = [c for cuts in cuts_per_node for c in cuts]
        sign = np.asarray([c[0] for c in flat], np.float64)
        var = np.asarray([c[1] for c in flat], np.int32)
        val = np.asarray([c[2] for c in flat], np.float64)
        hcap = H + (max((len(c) for c in cuts_per_node), default=0))
        out = {
            "status": np.empty(n, np.int32), "value": np.empty(n, np.float64), "pivots": np.empty((n, 2), np.int64),
            "rhs": np.empty((n, hcap), np.float64), "pos": np.empty((n, W + hcap), np.int32),
            "var": np.empty((n, W + hcap), np.int32),
            "matrices": np.empty((n, hcap * W), np.float64) if want_matrices else None, "stride_h": hcap,
        }
        self._check(self._lib.yalps_bnb_solve_nodes(self._ctx, n, _ptr(offs), _ptr(sign), _ptr(var), _ptr(val),
                                                    C.byref(opt), _ptr(out["status"]), _ptr(out["value"]),
                                                    _ptr(out["pivots"]), _ptr(out["rhs"]), _ptr(out["pos"]),
                                                    _ptr(out["var"]), _ptr(out["matrices"])))
        return out

    def solve_tableau_sparse(self, cells: np.ndarray, values: np.ndarray, height: int, width: int,
                             integers: Sequence[int], sign: float, options: Optional[Options] = None) -> dict:
        """solve_tableau on a tableau given as the ordered stores (cell = row*width + col, value) into a zero matrix
        (yalps_solve_sparse): the zeros are neither built on the host nor shipped over PCIe."""
        cells = np.ascontiguousarray(cells, np.int32).reshape(-1)
        values = np.ascontiguousarray(values, np.float64).reshape(-1)
        if cells.size != values.size:
            raise ValueError("cells and values must have the same length")
        return self.solve_tableau(values, height, width, integers, sign, options, cells=cells)

    def solve_lp_sparse(self, cells: np.ndarray, values: np.ndarray, height: int, width: int,
                        options: Optional[Options] = None, want_ranges: bool = False,
                        pairs: Optional[np.ndarray] = None, want_certificates: bool = False) -> dict:
        """One LP given as ordered (cell, value) stores into a zero matrix (yalps_solve_sparse_duals): status, value,
        pivots, rhs, pos, var and reduced, as solve_batch with n = 1 and want_duals; want_ranges adds range_lo and
        range_hi (`pairs` as solve_batch), want_certificates adds certificate (yalps_solve_sparse_certificate)."""
        opt = options or make_options()
        cells = np.ascontiguousarray(cells, np.int32).reshape(-1)
        values = np.ascontiguousarray(values, np.float64).reshape(-1)
        if cells.size != values.size:
            raise ValueError("cells and values must have the same length")
        want = {"want_basis": True, "want_duals": True, "want_ranges": want_ranges,
                "want_certificates": want_certificates}
        out = _batch_outputs(1, height, width, want)
        _add_outputs(out, 1, height, width, want)
        pr = _pairs_in(pairs, 1, height) if want_ranges else None
        self._check(self._lib.yalps_solve_sparse_certificate(self._ctx, height, width, int(cells.size),
                                                             _ptr(cells) if cells.size else None,
                                                             _ptr(values) if values.size else None, C.byref(opt),
                                                             *_out_args(out, want, pr, omit=("want_matrices",))))
        return {"status": int(out.pop("status")[0]), "value": float(out.pop("value")[0]),
                "pivots": tuple(int(p) for p in out.pop("pivots")[0]),
                **{k: a[0] for k, a in out.items() if a is not None}}

    def solve_tableau(self, matrix: np.ndarray, height: int, width: int, integers: Sequence[int], sign: float,
                      options: Optional[Options] = None, cells: Optional[np.ndarray] = None) -> dict:
        """Numeric part of solve() (src/YALPS.ts:77-91): root simplex + branch and cut when needed.
        (`cells` given: `matrix` holds the values of the sparse form, see solve_tableau_sparse.)"""
        opt = options or make_options()
        m = np.ascontiguousarray(matrix, np.float64).reshape(-1)
        ints = np.ascontiguousarray(integers, np.int32)
        cap = height + 2 * ints.size
        rhs = np.empty(cap, np.float64)
        pos = np.empty(width + cap, np.int32)
        var = np.empty(width + cap, np.int32)
        status, out_h, root_status = C.c_int32(), C.c_int32(), C.c_int32()
        result, root_value = C.c_double(), C.c_double()
        root_piv = np.zeros(2, np.int64)
        stats = np.zeros(8, np.int64)
        if cells is None:
            self._check(self._lib.yalps_solve(self._ctx, height, width, _ptr(m), _ptr(ints) if ints.size else None,
                                              int(ints.size), float(sign), C.byref(opt), C.byref(status), C.byref(result),
                                              C.byref(out_h), _ptr(rhs), _ptr(pos), _ptr(var), C.byref(root_status),
                                              C.byref(root_value), _ptr(root_piv), _ptr(stats)))
        else:
            self._check(self._lib.yalps_solve_sparse(self._ctx, height, width, int(cells.size),
                                                     _ptr(cells) if cells.size else None, _ptr(m) if m.size else None,
                                                     _ptr(ints) if ints.size else None, int(ints.size), float(sign),
                                                     C.byref(opt), C.byref(status), C.byref(result), C.byref(out_h),
                                                     _ptr(rhs), _ptr(pos), _ptr(var), C.byref(root_status),
                                                     C.byref(root_value), _ptr(root_piv), _ptr(stats)))
        return _search_result(width, status, result, out_h, rhs, pos, var, stats, (root_status, root_value, root_piv))

    def branch_and_cut(self, integers: Sequence[int], sign: float, init_result: float,
                       options: Optional[Options] = None) -> dict:
        """branchAndCut on the root previously given to bnb_set_root (src/branchAndCut.ts:89-176)."""
        opt = options or make_options()
        H, W = self._root_shape
        ints = np.ascontiguousarray(integers, np.int32)
        cap = H + 2 * ints.size
        rhs = np.empty(cap, np.float64)
        pos = np.empty(W + cap, np.int32)
        var = np.empty(W + cap, np.int32)
        status, out_h = C.c_int32(), C.c_int32()
        result = C.c_double()
        stats = np.zeros(8, np.int64)
        self._check(self._lib.yalps_branch_and_cut(self._ctx, _ptr(ints), int(ints.size), float(sign),
                                                   float(init_result), C.byref(opt), C.byref(status), C.byref(result),
                                                   C.byref(out_h), _ptr(rhs), _ptr(pos), _ptr(var), _ptr(stats)))
        return _search_result(W, status, result, out_h, rhs, pos, var, stats)

    # ------------------------------------------------------------------ probes
    def round_to_precision(self, x: np.ndarray, precision: float) -> np.ndarray:
        x = np.ascontiguousarray(x, np.float64).reshape(-1)
        out = np.empty_like(x)
        self._check(self._lib.yalps_round_to_precision(self._ctx, x.size, _ptr(x), float(precision), _ptr(out)))
        return out

    def probe_division(self, n: int, seed: int, mode: int) -> tuple:
        """(mismatches, (numerator bits, divisor bits) of the first one) of fastdiv.cuh vs __ddiv_rn."""
        bad = C.c_uint64()
        first = (C.c_uint64 * 2)()
        self._check(self._lib.yalps_probe_division(self._ctx, n, seed, mode, C.byref(bad), first))
        return int(bad.value), (int(first[0]), int(first[1]))

    def measure_tmem_bandwidth(self) -> tuple:
        g, c = C.c_double(), C.c_double()
        self._check(self._lib.yalps_measure_tmem_bandwidth(self._ctx, C.byref(g), C.byref(c)))
        return g.value, c.value

    def measure_l2_bandwidth(self, nbytes: int = 48 << 20) -> float:
        """GB/s (read + write) of an update-like stream over an L2-resident buffer."""
        g = C.c_double()
        self._check(self._lib.yalps_measure_l2_bandwidth(self._ctx, int(nbytes), C.byref(g)))
        return g.value

    def measure_h2d_seconds(self, pinned: np.ndarray, reps: int = 3, nstreams: int = 2) -> float:
        """Seconds per bare host-to-device copy of the whole (pinned) array."""
        sec = C.c_double()
        self._check(self._lib.yalps_measure_h2d_bandwidth(self._ctx, _ptr(pinned), pinned.nbytes, reps, nstreams,
                                                          C.byref(sec)))
        return sec.value

    def measure_smem_bandwidth(self) -> tuple:
        g, c = C.c_double(), C.c_double()
        self._check(self._lib.yalps_measure_smem_bandwidth(self._ctx, C.byref(g), C.byref(c)))
        return g.value, c.value


class MultiEngine:
    """yalps_multi: one process driving several GPUs (include/yalps_b200.h, csrc/multi.inl).  `devices` may repeat a
    GPU (several logical ranks on one device)."""

    def __init__(self, devices: Sequence[int]):
        self._lib = _ffi.load()
        self._m = C.c_void_p()
        dev = np.ascontiguousarray(devices, np.int32)
        rc = self._lib.yalps_create_multi(dev.ctypes.data_as(C.POINTER(C.c_int32)), int(dev.size), C.byref(self._m))
        if rc != 0:
            msg = self._lib.yalps_multi_last_error(None)
            raise YalpsError(rc, msg.decode() if msg else "yalps_create_multi failed")
        self.devices = [int(d) for d in dev]

    def close(self):
        if getattr(self, "_m", None) and self._m.value:
            self._lib.yalps_destroy_multi(self._m)
            self._m = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _check(self, rc: int):
        if rc != 0:
            msg = self._lib.yalps_multi_last_error(self._m)
            raise YalpsError(rc, msg.decode() if msg else "")

    @property
    def size(self) -> int:
        return int(self._lib.yalps_multi_size(self._m))

    @property
    def launch_count(self) -> int:
        return int(self._lib.yalps_multi_launch_count(self._m))

    def set_tuning(self, path: int = PATH_AUTO, threads_per_lp: int = 0, row_groups: int = 0):
        for r in range(self.size):
            ctx = C.c_void_p(self._lib.yalps_multi_ctx(self._m, r))
            if self._lib.yalps_set_tuning(ctx, path, threads_per_lp) or self._lib.yalps_set_row_groups(ctx, row_groups):
                raise YalpsError(-2, (self._lib.yalps_last_error(ctx) or b"").decode())

    def solve_batch(self, matrices: np.ndarray, height: int, width: int, options: Optional[Options] = None,
                    want_matrices: bool = False, pos_in=None, var_in=None, out: Optional[dict] = None,
                    want_duals: bool = False, want_ranges: bool = False, pairs=None,
                    want_certificates: bool = False) -> dict:
        return _solve_uniform(self._check, self._lib.yalps_multi_solve_batch_certificate, self._m, matrices, height,
                              width, options, out, pos_in, var_in, pairs,
                              {"want_matrices": want_matrices, "want_basis": True, "want_duals": want_duals,
                               "want_ranges": want_ranges, "want_certificates": want_certificates})

    def solve_replicas(self, base: np.ndarray, rhs: np.ndarray, height: int, width: int,
                       options: Optional[Options] = None, out: Optional[dict] = None, want_duals: bool = False) -> dict:
        return _solve_replicas(self._check, self._lib.yalps_multi_solve_replicas_duals, self._m, base, rhs, height,
                               width, options, out, {"want_basis": True, "want_duals": want_duals})

    def solve_warm(self, base: np.ndarray, height: int, width: int, rhs: Optional[np.ndarray] = None,
                   obj: Optional[np.ndarray] = None, options: Optional[Options] = None, final: Optional[tuple] = None,
                   want_basis: bool = True, want_matrices: bool = False, want_duals: bool = False,
                   want_ranges: bool = False, pairs: Optional[np.ndarray] = None,
                   want_certificates: bool = False, add_rows: Optional[np.ndarray] = None,
                   add_cols: Optional[np.ndarray] = None) -> dict:
        """Engine.solve_warm with the variants sharded over the ranks; every rank solves (or uploads) the base."""
        extend = add_rows is not None or add_cols is not None
        fn = self._lib.yalps_multi_solve_warm_extend if extend else self._lib.yalps_multi_solve_warm
        return _solve_warm(self._check, fn, self._m, base, height, width, rhs, obj, options, final, pairs,
                           {"want_basis": want_basis, "want_matrices": want_matrices, "want_duals": want_duals,
                            "want_ranges": want_ranges, "want_certificates": want_certificates},
                           add_rows=add_rows, add_cols=add_cols)

    def solve_ragged(self, tableaus: Sequence[np.ndarray], shapes: Sequence[tuple], options: Optional[Options] = None,
                     want_matrices: bool = False, want_duals: bool = False, want_ranges: bool = False,
                     pairs: Optional[Sequence] = None, want_certificates: bool = False) -> list:
        return _solve_ragged(self._check, self._lib.yalps_multi_solve_ragged_certificate, self._m, tableaus, shapes,
                             options, pairs, {"want_basis": True, "want_matrices": want_matrices,
                                              "want_duals": want_duals, "want_ranges": want_ranges,
                                              "want_certificates": want_certificates}, basis_in=False)

    def _rank0(self):
        """rank 0's ctx and a check that reads its error message"""
        ctx = C.c_void_p(self._lib.yalps_multi_ctx(self._m, 0))

        def check(rc: int):
            if rc != 0:
                msg = self._lib.yalps_last_error(ctx)
                raise YalpsError(rc, msg.decode() if msg else "")
        return ctx, check

    def iis(self, matrix: np.ndarray, height: int, width: int, options: Optional[Options] = None) -> dict:
        """Engine.iis on rank 0's context (the rounds of one search depend on each other)."""
        ctx, check = self._rank0()
        return _iis(check, self._lib, ctx, height, width, options, matrix=matrix)

    def iis_sparse(self, cells: np.ndarray, values: np.ndarray, height: int, width: int,
                   options: Optional[Options] = None) -> dict:
        """Engine.iis_sparse on rank 0's context."""
        ctx, check = self._rank0()
        return _iis(check, self._lib, ctx, height, width, options, cells=cells, values=values)

    def solve_large(self, matrix: np.ndarray, height: int, width: int, options: Optional[Options] = None,
                    want_matrix: bool = False) -> dict:
        """ONE LP with its rows dealt round robin over the ranks (yalps_multi_solve_large): peer-memory exchange of the
        pivot row and column from inside one persistent kernel per GPU.  Outputs as solve_batch for n = 1."""
        opt = options or make_options()
        m = np.ascontiguousarray(matrix, np.float64).reshape(-1)
        if m.size != height * width:
            raise ValueError("matrix must hold height * width cells")
        status, value, ms = C.c_int32(), C.c_double(), C.c_double()
        piv = np.zeros(2, np.int64)
        rhs, pos, var = np.empty(height), np.empty(width + height, np.int32), np.empty(width + height, np.int32)
        mat = np.empty(height * width, np.float64) if want_matrix else None
        self._check(self._lib.yalps_multi_solve_large(self._m, height, width, _ptr(m), C.byref(opt), C.byref(status),
                                                      C.byref(value), _ptr(piv), _ptr(rhs), _ptr(pos), _ptr(var),
                                                      _ptr(mat), C.byref(ms)))
        return {"status": status.value, "value": value.value, "pivots": (int(piv[0]), int(piv[1])), "rhs": rhs,
                "pos": pos, "var": var, "matrix": mat, "kernel_ms": ms.value}

    def incumbent_allreduce(self, local: Sequence[float]) -> np.ndarray:
        """Min-allreduce of one fp64 per rank (NCCL across the distinct GPUs)."""
        loc = np.ascontiguousarray(local, np.float64)
        if loc.size != self.size:
            raise ValueError("one value per rank")
        out = np.empty_like(loc)
        self._check(self._lib.yalps_incumbent_allreduce(self._m, loc.ctypes.data_as(C.POINTER(C.c_double)),
                                                        out.ctypes.data_as(C.POINTER(C.c_double))))
        return out

    def solve_tableau(self, matrix: np.ndarray, height: int, width: int, integers: Sequence[int], sign: float,
                      options: Optional[Options] = None, allreduce_every: int = 4) -> dict:
        """Engine.solve_tableau with the branch-and-bound frontier sharded over the ranks."""
        opt = options or make_options()
        m = np.ascontiguousarray(matrix, np.float64).reshape(-1)
        ints = np.ascontiguousarray(integers, np.int32)
        cap = height + 2 * ints.size
        rhs, pos, var = np.empty(cap, np.float64), np.empty(width + cap, np.int32), np.empty(width + cap, np.int32)
        status, out_h, root_status = C.c_int32(), C.c_int32(), C.c_int32()
        result, root_value = C.c_double(), C.c_double()
        root_piv, stats = np.zeros(2, np.int64), np.zeros(10, np.int64)
        self._check(self._lib.yalps_multi_solve(self._m, height, width, _ptr(m), _ptr(ints) if ints.size else None,
                                                int(ints.size), float(sign), C.byref(opt), int(allreduce_every),
                                                C.byref(status), C.byref(result), C.byref(out_h), _ptr(rhs), _ptr(pos),
                                                _ptr(var), C.byref(root_status), C.byref(root_value), _ptr(root_piv),
                                                _ptr(stats)))
        return _search_result(width, status, result, out_h, rhs, pos, var, stats, (root_status, root_value, root_piv))

    def solve_many_tableaus(self, tabmods: Sequence, options: Optional[Options] = None,
                            searches_per_device: int = 4) -> list:
        """yalps_multi_solve_many over TableauModel-like objects (.tableau.matrix/.height/.width, .integers, .sign)."""
        opt = options or make_options()
        n = len(tabmods)
        if n == 0:
            return []
        heights = np.asarray([tm.tableau.height for tm in tabmods], np.int32)
        widths = np.asarray([tm.tableau.width for tm in tabmods], np.int32)
        nints = np.asarray([len(tm.integers) for tm in tabmods], np.int64)
        offs, packed = _pack_ragged([tm.tableau.matrix for tm in tabmods], heights, widths)
        ioffs = _offsets(nints)
        ints = np.asarray([v for tm in tabmods for v in tm.integers], np.int32) if ioffs[-1] else np.zeros(1, np.int32)
        signs = np.asarray([tm.sign for tm in tabmods], np.float64)
        roffs = _offsets(heights + 2 * nints)
        poffs = _offsets(heights.astype(np.int64) + widths + 2 * nints)
        status, result, out_h = np.empty(n, np.int32), np.empty(n, np.float64), np.empty(n, np.int32)
        rhs, pos, var = np.empty(int(roffs[-1])), np.empty(int(poffs[-1]), np.int32), np.empty(int(poffs[-1]), np.int32)
        self._check(self._lib.yalps_multi_solve_many(self._m, n, _ptr(heights), _ptr(widths), _ptr(offs[:-1].copy()),
                                                     _ptr(packed), _ptr(ioffs), _ptr(ints), _ptr(signs), C.byref(opt),
                                                     int(searches_per_device), _ptr(status), _ptr(result), _ptr(out_h),
                                                     _ptr(rhs), _ptr(pos), _ptr(var)))
        res = []
        for i in range(n):
            h, w = int(out_h[i]), int(widths[i])
            res.append({"status": int(status[i]), "result": float(result[i]), "height": h,
                        "rhs": rhs[roffs[i]:roffs[i] + h], "pos": pos[poffs[i]:poffs[i] + w + h],
                        "var": var[poffs[i]:poffs[i] + w + h]})
        return res
