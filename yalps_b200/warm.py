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

A variant may also add K rows and M columns (`rows`, `cols`; the start tableau is then (H+K) x (W+M)).  An added row
is in initial-tableau form over the W+M columns: a[0] the RHS, a[1..W-1] the base structurals, a[W..W+M-1] the added
ones (an upper row `a.x <= max`, a lower row `-a.x <= -min`, as tableau.ts builds them).  An added column g_j is in
initial-tableau form over the H base rows: g_j[0] = sign * cost, then its coefficient in each base row.  In base ids
and positions the steps are, with steps 1 and 3 the two passes above:

1. Column pass (column 0), as above.
2. Added columns: T[r, W+j] = sum_k g_j[k] * dir(W+k)[r] for every row r, from +0.0, k ascending, skipping
   g_j[k] == 0.0, product and sum rounded apart (dir read from F, row 0 included; dir(W+0) is e_0).
3. Row pass, as above, over all W+M columns: a cost change on a basic x_j reaches the added columns' row 0 too.
4. Added rows, on the result of 3.  Row i starts as t = (a[0], +0.0, ..., +0.0); for every structural v with
   a[v] != 0.0, base ids then added ids ascending: v non-basic: t[pos(v)] = t[pos(v)] + a[v]; v basic at row q:
   t[c] = t[c] - a[v] * T[q,c] for every c, column 0 included.  Added variables are non-basic at column W+j.
5. Basis (extended_basis): base structural v < W keeps id v; added structural j is W+j, non-basic at column W+j; base
   slack W+k becomes W+M+k; added row i's slack is W+M+H+i, basic at row H+i.

With K = M = 0 this is the tableau above bit for bit.

Why (exact arithmetic).  Row r of F reads basic_r = F[r,0] - sum_c F[r,c] * nonbasic_c.  Raising row k's RHS by delta
is the old system with slack s_k = -delta, so every basic value moves by +delta * dir(W+k): F[r,pos] * delta when s_k is
non-basic at column pos, and +delta on its own row when s_k is basic (the direction whose sign ranging already uses).
Row 0 is M0's row 0 minus a combination of the constraint rows fixed by the basis, so column 0 becomes B^-1 b' and the
objective value moves with it.  Raising the initial objective cell M0[0,j] = sign * c_j by delta adds delta to x_j's
reduced cost F[0,pos[j]] when x_j is non-basic; when x_j is basic at row q its cost enters row 0 through the pivots on
row q, which subtracts delta times row q, column 0 (the objective value) included.  So row 0 holds the reduced costs and
objective value of the same basis under the new costs.

An added column a_j (cost c_j) enters the old system as a non-basic variable at 0, so the basis is unchanged and its
column in the final tableau is B^-1 a_j: the combination of the base rows the pivots applied, which maps the initial
unit column of row k to dir(W+k) (the final column of slack k, or its unit row when it stayed basic).  Row 0 is the same
map applied to the cost cell, so T[0, W+j] is c_j's reduced cost under the costs of step 3's input, and step 3 then
moves it to the new costs as for every other column.  An added row reads sum_v a_v x_v + s = a[0] with a new slack s
basic: writing every basic x_v as its final row (x_v = T[q,0] - sum_c T[q,c] * nonbasic_c) substitutes the basic
variables out and leaves a row in the non-basic variables, with RHS a[0] - sum a_v T[q,0] = the slack's value at the
old vertex.  So the extended basis is the old one plus the new slacks: row 0 is untouched, the basis stays dual
feasible, and the added rows start primal infeasible exactly when the old vertex violates them -- phase 1 is then the
dual simplex, as for branch-and-cut nodes.  For a one-variable cut x_j <= v (or -x_j <= -v) step 4 is the applyCuts
row of k_assemble_nodes cell for cell (==; only the sign of a zero can differ: 0.0 - x against -x).

The variant's solve is the reference loop run on T: phase 1 from a dual-feasible T (after RHS changes) is the dual
simplex, and after objective changes T stays primal feasible and phase 2 continues from the old vertex.  Its results
are bit-exact against that loop on T, not against a cold solve of the changed model: the pivot path differs, so
statuses agree and optimal values agree within the precision, but with alternative optima the vertex can differ.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Optional

import numpy as np

from .sensitivity import row_pairs
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
                 rhs: Optional[np.ndarray] = None, obj: Optional[np.ndarray] = None,
                 rows: Optional[np.ndarray] = None, cols: Optional[np.ndarray] = None) -> np.ndarray:
    """The start tableau T (flat, (H+K)*(W+M) float64) of the variant with column 0 `rhs` (H values, or None:
    unchanged), row 0 `obj` (W values, obj[0] ignored, or None: unchanged), added rows `rows` (K x (W+M), or None) and
    added columns `cols` (M x H, or None) of the base with initial tableau M0 and final tableau F and
    positionOfVariable pos.  Its pos / var are extended_basis of the base's final ones."""
    H, W = int(height), int(width)
    g = np.zeros((0, H)) if cols is None else np.asarray(cols, np.float64).reshape(-1, H)
    M = g.shape[0]
    a = np.zeros((0, W + M)) if rows is None else np.asarray(rows, np.float64).reshape(-1, W + M)
    K = a.shape[0]
    m0 = np.asarray(M0, np.float64).reshape(H, W)
    f = np.asarray(F, np.float64).reshape(H, W)
    p = np.asarray(pos, np.int64).reshape(-1)
    T = np.zeros((H + K, W + M))
    T[:H, :W] = f
    if rhs is not None:
        delta = np.asarray(rhs, np.float64).reshape(-1)[:H] - m0[:, 0]
        col = T[:H, 0].copy()
        for k in np.flatnonzero(delta != 0.0):
            col = col + delta[k] * direction(f, p, H, W, W + int(k))
        T[:H, 0] = col
    for j in range(M):
        col = np.zeros(H)
        for k in np.flatnonzero(g[j] != 0.0):
            col = col + g[j, k] * direction(f, p, H, W, W + int(k))
        T[:H, W + j] = col
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
    for i in range(K):
        t = np.zeros(W + M)
        t[0] = a[i, 0]
        for v in np.flatnonzero(a[i, 1:] != 0.0) + 1:
            q = int(p[v]) if v < W else int(v)
            if q < W or v >= W:
                t[q] = t[q] + a[i, v]
            else:
                t = t - a[i, v] * T[q - W]
        T[H + i] = t
    return T.reshape(-1)


def extended_basis(pos: np.ndarray, var: np.ndarray, height: int, width: int, add_rows: int, add_cols: int) -> tuple:
    """(pos, var) of warm_tableau's start tableau with add_rows rows and add_cols columns from the base's final ones
    (step 5 of the module docstring); int32, (H+K) + (W+M) entries each."""
    H, W, K, M = int(height), int(width), int(add_rows), int(add_cols)
    v0 = np.asarray(var, np.int64).reshape(-1)[:H + W]
    ids = np.where(v0 < W, v0, v0 + M)  # base ids relabelled, in base position order
    var_x = np.arange(H + K + W + M, dtype=np.int64)
    var_x[:W] = ids[:W]
    var_x[W + M:W + M + H] = ids[W:]
    pos_x = np.empty_like(var_x)
    pos_x[var_x] = np.arange(var_x.size)
    return pos_x.astype(np.int32), var_x.astype(np.int32)


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
        marked = set(v) & {"integers", "binaries"}
        if marked:
            raise ValueError(f"variant {i}: {sorted(marked)}: variants are LPs, an added variable cannot be marked "
                             f"integer or binary")
        unknown = set(v) - {"constraints", "objective", "addConstraints", "addVariables"}
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



@dataclass
class Additions:
    """The added rows and columns of a batch of variants (variant_additions), padded to the batch's largest K and M
    with zero rows and columns, and what maps each variant's results back to its own names."""

    rows: np.ndarray  # (n, K, W + M): added rows in initial-tableau form over the padded columns
    cols: np.ndarray  # (n, M, H): added columns in initial-tableau form over the base rows
    variables: list  # per variant: the (name, coefficients) pairs of its columns 1.., base then added
    keys: list  # per variant: (key, upper row | -1, lower row | -1) over its rows, base keys then added keys
    pairs: np.ndarray  # (n, H + K): row_pairs of each variant's keys, -1 on padding rows


def variant_additions(model: dict, variants: list, tableau) -> Optional[Additions]:
    """Model level: the rows and columns `variants` add to the base `model` whose tableau is given, or None when none
    adds anything.  A variant may carry
      "addConstraints": {key: {"min" | "max" | "equal": value, "coefficients": {base variable: a}}}
      "addVariables": {name: {key or objective: coefficient}}  (the shape of model["variables"])
    A new key needs `coefficients` (over base variables; an added variable's coefficients come from addVariables only).
    An existing key takes the model's coefficients and may only add a bound it lacks.  Rows follow tableau.ts: a key's
    upper row `a.x <= max` before its lower row `-a.x <= -min` (an `equal` gives both, paired for ranging), in the order
    of addConstraints; added variables are columns in the order of addVariables.  An added variable may name base keys,
    the objective and the variant's added keys.  ValueError for an unknown key or variable, an added name that clashes
    with a base variable, a bound the model already has, a non-finite bound or coefficient, and a new key that has no
    bound, no coefficients, or the objective's name."""
    if not any(v.get("addConstraints") or v.get("addVariables") for v in variants):
        return None
    H, W = int(tableau.height), int(tableau.width)
    sign = -1.0 if model.get("direction") == "minimize" else 1.0
    objective = model.get("objective")
    merged = _merged_rows(list(entries(model["constraints"])))
    base_rows = {key: (up, lo) for key, up, lo, _, _ in merged}
    base_vars = [(name, dict(entries(cs))) for name, cs in entries(model["variables"])]
    col_of = {name: j + 1 for j, (name, _) in enumerate(base_vars)}

    def finite(i, what, value):
        value = float(value)
        if not math.isfinite(value):
            raise ValueError(f"variant {i}: {what} = {value} is not finite")
        return value

    built = []  # per variant: (added rows [(key, upper, value, {column: a})], added variables [(name, {key: c})])
    for i, v in enumerate(variants):
        added_vars, seen = [], set()
        for name, cs in entries(v.get("addVariables") or {}):
            if name in col_of or name in seen:
                raise ValueError(f"variant {i}: added variable {name!r} clashes with a variable of the model or "
                                 f"another added one")
            seen.add(name)
            added_vars.append((name, {key: finite(i, f"{name!r} coefficient of {key!r}", c)
                                      for key, c in entries(cs)}))
        added_rows, added_keys = [], set()
        for key, spec in entries(v.get("addConstraints") or {}):
            spec = dict(spec)
            for kind in set(spec) - {"min", "max", "equal", "coefficients"}:
                raise ValueError(f"variant {i}: added constraint {key!r} has no bound kind {kind!r}")
            if key in added_keys:
                raise ValueError(f"variant {i}: constraint {key!r} is added twice")
            added_keys.add(key)
            bound = {b: finite(i, f"constraint {key!r} {b}", spec[b]) for b in ("min", "max", "equal") if b in spec}
            hi = bound.get("equal", bound.get("max"))
            lo = bound.get("equal", bound.get("min"))
            if hi is None and lo is None:
                raise ValueError(f"variant {i}: added constraint {key!r} has no bound")
            if key in base_rows:
                if "coefficients" in spec:
                    raise ValueError(f"variant {i}: constraint {key!r} exists: it takes the model's coefficients, "
                                     f"'coefficients' is refused")
                up, lw = base_rows[key]
                for kind, value, row in (("max", hi, up), ("min", lo, lw)):
                    if value is not None and row >= 0:
                        raise ValueError(f"variant {i}: constraint {key!r} already has a finite {kind!r} bound; change "
                                         f"it through 'constraints'")
                coefs = {col_of[name]: float(cs[key]) for name, cs in base_vars if key in cs}
            else:
                if key == objective:
                    raise ValueError(f"variant {i}: an added constraint cannot be the objective {key!r}")
                if "coefficients" not in spec:
                    raise ValueError(f"variant {i}: the new constraint {key!r} needs 'coefficients'")
                coefs = {}
                for name, a in entries(spec["coefficients"]):
                    if name not in col_of:
                        raise ValueError(f"variant {i}: constraint {key!r}: the base model has no variable {name!r}")
                    coefs[col_of[name]] = finite(i, f"constraint {key!r} coefficient of {name!r}", a)
            if hi is not None:
                added_rows.append((key, True, hi, coefs))
            if lo is not None:
                added_rows.append((key, False, lo, coefs))
        for name, cs in added_vars:
            for key in cs:
                if key != objective and key not in base_rows and key not in added_keys:
                    raise ValueError(f"variant {i}: added variable {name!r}: no constraint {key!r} in the model or "
                                     f"the variant")
        built.append((added_rows, added_vars))

    n = len(variants)
    K = max(len(r) for r, _ in built)
    M = max(len(c) for _, c in built)
    rows = np.zeros((n, K, W + M))
    cols = np.zeros((n, M, H))
    out = Additions(rows, cols, [], [], np.full((n, H + K), -1, np.int32))
    base_keys = [(key, up, lo) for key, up, lo, _, _ in merged]
    for i, (added_rows, added_vars) in enumerate(built):
        where = {key: [up, lo] for key, up, lo in base_keys}  # key -> [upper row, lower row] over the extended rows
        order = [key for key, _, _ in base_keys]
        for h, (key, upper, value, coefs) in enumerate(added_rows):
            if key not in where:
                where[key] = [-1, -1]
                order.append(key)
            where[key][0 if upper else 1] = H + h
            rows[i, h, 0] = value if upper else -value
            for c, a in coefs.items():
                rows[i, h, c] = a if upper else -a
        for j, (name, cs) in enumerate(added_vars):
            for key, c in cs.items():
                if key == objective:
                    cols[i, j, 0] = sign * c
                up, lo = where.get(key, (-1, -1))
                for row, s in ((up, 1.0), (lo, -1.0)):
                    if row < 0:
                        continue
                    if row < H:
                        cols[i, j, row] = c if s > 0 else -c
                    else:
                        rows[i, row - H, W + j] = c if s > 0 else -c
        keys = [(key, where[key][0], where[key][1]) for key in order]
        out.variables.append([(name, cs) for name, cs in base_vars] + added_vars)
        out.keys.append(keys)
        out.pairs[i, :H + len(added_rows)] = row_pairs(keys, H + len(added_rows))
    return out
