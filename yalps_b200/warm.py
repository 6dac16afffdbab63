"""Warm starts: the start tableau of a variant of an LP, derived from the base LP's final tableau.

A variant keeps the base's constraint coefficients and changes its right-hand sides (a new column 0 `b'`, H values,
b'[0] the new M0[0,0]) and/or its objective coefficients (a new row 0 `c'`, W values, c'[0] ignored).  Its start
tableau T keeps the base's final basis (pos / var) and is built from the base's initial tableau M0 and final tableau F
(any status: the reference's loop gives valid verdicts from any basis).  This module is the one place that states it;
k_expand_warm (csrc/aux_kernels.cuh) computes the same bits on the GPU.

dir(v) is the direction ranges_from_tableau uses: for a non-basic id (1 <= pos[v] < W) the column F[:, pos[v]], row 0
included; for a basic id the unit vector of row pos[v] - W; for id W + 0 the unit vector of row 0.

1. Column pass.  T = F.  delta_k = b'[k] - M0[k,0], rounded once and skipped when it is 0.0 (NaN is not skipped).  For
   every row r in 0..H-1 and every changed k in ascending order: T[r,0] = T[r,0] + delta_k * dir(W+k)[r], the product
   rounded, then the sum (no FMA).
2. Row pass, on the result of step 1.  delta_j = c'[j] - M0[0,j] for j = 1..W-1, skipped when 0.0.  For every column c
   in 0..W-1 and every changed j in ascending order: if x_j is non-basic, T[0,c] = T[0,c] + delta_j when c == pos[j];
   if x_j is basic at row q = pos[j] - W, T[0,c] = T[0,c] - delta_j * T[q,c].

With no change at all T is F bit for bit.

Why (exact arithmetic).  Row r of F reads basic_r = F[r,0] - sum_c F[r,c] * nonbasic_c.  Raising row k's RHS by delta
is the old system with slack s_k = -delta, so every basic value moves by +delta * dir(W+k): F[r,pos] * delta when s_k is
non-basic at column pos, and +delta on its own row when s_k is basic (the direction whose sign ranging already uses).
Row 0 is M0's row 0 minus a combination of the constraint rows fixed by the basis, so column 0 becomes B^-1 b' and the
objective value moves with it.  Raising the initial objective cell M0[0,j] = sign * c_j by delta adds delta to x_j's
reduced cost F[0,pos[j]] when x_j is non-basic; when x_j is basic at row q its cost enters row 0 through the pivots on
row q, which subtracts delta times row q, column 0 (the objective value) included.  So row 0 holds the reduced costs and
objective value of the same basis under the new costs.

The variant's solve is the reference loop run on T: phase 1 from a dual-feasible T (after RHS changes) is the dual
simplex, and after objective changes T stays primal feasible and phase 2 continues from the old vertex.  Its results
are bit-exact against that loop on T, not against a cold solve of the changed model: the pivot path differs, so
statuses agree and optimal values agree within the precision, but with alternative optima the vertex can differ.
"""
from __future__ import annotations

import math
from typing import Optional

import numpy as np

from .tableau import _merged_rows, entries


def direction(F: np.ndarray, pos: np.ndarray, height: int, width: int, v: int) -> np.ndarray:
    """dir(v) of the final tableau F (H x W) with positionOfVariable pos (module docstring)."""
    p = int(pos[v])
    if 1 <= p < width:
        return F[:, p].copy()
    d = np.zeros(height)
    d[p - width] = 1.0
    return d


def warm_tableau(M0: np.ndarray, F: np.ndarray, pos: np.ndarray, height: int, width: int,
                 rhs: Optional[np.ndarray] = None, obj: Optional[np.ndarray] = None) -> np.ndarray:
    """The start tableau T (flat, H*W float64) of the variant with column 0 `rhs` (H values, or None: unchanged) and
    row 0 `obj` (W values, obj[0] ignored, or None: unchanged) of the base with initial tableau M0 and final tableau F
    and positionOfVariable pos.  Its pos / var are the base's final ones."""
    H, W = int(height), int(width)
    m0 = np.asarray(M0, np.float64).reshape(H, W)
    f = np.asarray(F, np.float64).reshape(H, W)
    p = np.asarray(pos, np.int64).reshape(-1)
    T = f.copy()
    if rhs is not None:
        delta = np.asarray(rhs, np.float64).reshape(-1)[:H] - m0[:, 0]
        col = T[:, 0].copy()
        for k in np.flatnonzero(delta != 0.0):
            col = col + delta[k] * direction(f, p, H, W, W + int(k))
        T[:, 0] = col
    if obj is not None:
        delta = np.asarray(obj, np.float64).reshape(-1)[:W] - m0[0]
        row = T[0].copy()
        for j in np.flatnonzero(delta[1:] != 0.0) + 1:
            q = int(p[j])
            if q < W:
                row[q] = row[q] + delta[j]
            else:
                row = row - delta[j] * T[q - W]
        T[0] = row
    return T.reshape(-1)


def variant_vectors(model: dict, variants: list, tableau) -> tuple:
    """Model level: (rhs (n, H), obj (n, W)) of `variants` on the base `model` whose tableau (yalps_b200.tableau) is
    given; either is None when no variant changes it (rhs is the base's column 0 for every variant when no variant
    changes anything: each is then the base LP from its own final basis).  A variant is {"constraints": {key: {"min"|"max"|"equal": v}},
    "objective": {variable: coefficient}}, both optional.  A key's `max` sets its upper row's RHS, `min` sets its lower
    row's RHS to -min, `equal` both.  ValueError for an unknown key, bound or variable, and for a bound the base model
    does not have: an infinite bound has no tableau row."""
    rows = {key: (up, lo) for key, up, lo, _, _ in _merged_rows(list(entries(model["constraints"])))}
    cols = {key: j + 1 for j, (key, _) in enumerate(entries(model["variables"]))}
    col0, row0 = _base_col0_row0(tableau)
    n = len(variants)
    rhs = obj = None
    sign = -1.0 if model.get("direction") == "minimize" else 1.0
    for i, v in enumerate(variants):
        unknown = set(v) - {"constraints", "objective"}
        if unknown:
            raise ValueError(f"variant {i}: unknown field(s) {sorted(unknown)}")
        for key, bounds in entries(v.get("constraints") or {}):
            if key not in rows:
                raise ValueError(f"variant {i}: the base model has no constraint {key!r}")
            up, lo = rows[key]
            for bound, value in bounds.items():
                if bound not in ("min", "max", "equal"):
                    raise ValueError(f"variant {i}: constraint {key!r} has no bound kind {bound!r}")
                value = float(value)
                if not math.isfinite(value):
                    raise ValueError(f"variant {i}: constraint {key!r} {bound} = {value}: an infinite bound has no "
                                     f"tableau row")
                targets = {"max": [(up, value)], "min": [(lo, -value)], "equal": [(up, value), (lo, -value)]}[bound]
                for row, b in targets:
                    if row < 0:
                        raise ValueError(f"variant {i}: constraint {key!r} has no finite {bound!r} bound in the base "
                                         f"model, so no tableau row to change")
                    if rhs is None:
                        rhs = np.tile(col0, (n, 1))
                    rhs[i, row] = b
        for var, coef in entries(v.get("objective") or {}):
            if var not in cols:
                raise ValueError(f"variant {i}: the base model has no variable {var!r}")
            if obj is None:
                obj = np.tile(row0, (n, 1))
            obj[i, cols[var]] = sign * float(coef)
    if rhs is None and obj is None:
        rhs = np.tile(col0, (n, 1))
    return rhs, obj


def _base_col0_row0(tableau) -> tuple:
    """Column 0 and row 0 of a tableau in either form (the sparse form's later stores win)."""
    H, W = int(tableau.height), int(tableau.width)
    if tableau.matrix is not None:
        m = np.asarray(tableau.matrix, np.float64).reshape(H, W)
        return m[:, 0].copy(), m[0].copy()
    col0, row0 = np.zeros(H), np.zeros(W)
    cells, values = tableau.cells, tableau.values
    in_col = cells % W == 0
    col0[cells[in_col] // W] = values[in_col]
    in_row = cells < W
    row0[cells[in_row]] = values[in_row]
    return col0, row0

