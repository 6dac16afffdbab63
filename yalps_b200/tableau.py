"""Model -> tableau, host side (the producer at the drop-in boundary).

Same contract as `tableauModel` in the reference (src/tableau.ts:47-137): flat row-major float64
matrix, row 0 = objective row holding sign*coef, column 0 = RHS, one row per finite bound of each
merged constraint key (upper row first), one `x <= 1` row per binary after all constraints, identity
positionOfVariable / variableAtPosition.  tests/tableau.ts pins this layout bit for bit, including
negative zeros, and tests/test_tableau.py re-expresses those properties.

Unlike the reference this builder is array-oriented: constraint keys are resolved to row numbers
once, then every (variable, coefficient) pair becomes at most three scattered stores.
"""
from __future__ import annotations

import math
import re
from dataclasses import dataclass
from typing import Any, Iterable, Optional

import numpy as np

try:  # native core of the builder (csrc/tabfast.c, built by `make -C yalps_b200/csrc`); the loops below are the fallback
    from . import _tabfast as _NATIVE
except ImportError:  # pragma: no cover - the extension is part of the normal build
    _NATIVE = None

_INDEX_KEY = re.compile(r"0|[1-9][0-9]*")


def entries(obj) -> Iterable:
    """Pairs of a mapping-like argument in the order the reference would iterate it.

    dict plays the role of a JS object: canonical array-index keys first in ascending numeric order,
    then the remaining keys in insertion order (what Object.entries yields, src/tableau.ts:37).
    Any other iterable is taken as an iterable of (key, value) pairs (Array / Map, src/tableau.ts:36).
    """
    if isinstance(obj, dict):
        # (cheap pre-test: a canonical array index starts with a digit)
        numeric = [k for k in obj if isinstance(k, str) and k[:1].isdigit() and _INDEX_KEY.fullmatch(k) and int(k) < 4294967295]
        if not numeric:
            return obj.items()
        numeric.sort(key=int)
        seen = set(numeric)
        return [(k, obj[k]) for k in numeric] + [(k, v) for k, v in obj.items() if k not in seen]
    return obj


def _as_set(spec):
    """src/tableau.ts:41-45: True stays True, False/None -> empty set, iterables -> set."""
    if spec is True:
        return True
    if spec is None or spec is False:
        return frozenset()
    return spec if isinstance(spec, (set, frozenset)) else set(spec)


def _field(constraint, name):
    if isinstance(constraint, dict):
        return constraint.get(name)
    return getattr(constraint, name, None)


@dataclass
class Tableau:
    """src/tableau.ts:9-15"""

    matrix: Optional[np.ndarray]  # float64[height*width], row-major; None while only the sparse form below exists
    width: int
    height: int
    position_of_variable: np.ndarray  # int32[width+height]
    variable_at_position: np.ndarray  # int32[width+height]
    # the stores tableauModel makes into its zero-filled matrix, in order (cell = row*width + col; a later store to
    # the same cell wins): what yalps_solve_sparse takes, so that big sparse models never exist densely on the host
    cells: Optional[np.ndarray] = None  # int32[nnz]
    values: Optional[np.ndarray] = None  # float64[nnz]

    def dense(self) -> np.ndarray:
        """The flat row-major matrix (built from the sparse form on first use)."""
        if self.matrix is None:
            m = np.zeros(self.height * self.width, dtype=np.float64)
            if self.cells.size:
                m[self.cells] = self.values  # repeated indices are applied in order: the last one wins
            self.matrix = m
        return self.matrix


@dataclass
class TableauModel:
    """src/tableau.ts:26-31"""

    tableau: Tableau
    sign: float
    variables: list  # [(key, coefficients)]
    integers: list  # variable ids (1-based columns) that must be integral


def constraint_rows(constraints: list) -> list:
    """Merged constraint keys in first-seen order with their tableau rows (src/tableau.ts:73-86):
    [(key, upper row or -1, lower row or -1)].  A key's bounds are intersected over its entries; the upper row
    (`a.x <= max`) comes before the lower row (`-a.x <= -min`), rows count from 1, and an infinite bound has no row."""
    return [(key, up, lo) for key, up, lo, _, _ in _merged_rows(constraints)]


def _merged_rows(constraints: list) -> list:
    """constraint_rows plus each key's merged (upper, lower) bounds."""
    lower: dict[Any, float] = {}
    upper: dict[Any, float] = {}
    for key, con in constraints:
        eq = _field(con, "equal")
        lo = eq if eq is not None else _field(con, "min")
        hi = eq if eq is not None else _field(con, "max")
        lo = -math.inf if lo is None else float(lo)
        hi = math.inf if hi is None else float(hi)
        if key in lower:
            lower[key] = max(lower[key], lo)
            upper[key] = min(upper[key], hi)
        else:
            lower[key] = max(-math.inf, lo)
            upper[key] = min(math.inf, hi)
    out = []
    rows = 1
    for key in lower:
        up = lo = -1
        if math.isfinite(upper[key]):
            up = rows
            rows += 1
        if math.isfinite(lower[key]):
            lo = rows
            rows += 1
        out.append((key, up, lo, upper[key], lower[key]))
    return out


def _stores_python(variables: list, constraints: list, objective, sign: float, width: int, binary_cols: list):
    """The ordered stores of src/tableau.ts:73-134 as (cells, values, rows); specification of csrc/tabfast.c."""
    # merge constraints per key, first-seen order, and number their rows (src/tableau.ts:73-86)
    merged = _merged_rows(constraints)
    rows = 1 + sum((u >= 0) + (l >= 0) for _, u, l, _, _ in merged)
    rhs_rows: list[int] = []
    rhs_vals: list[float] = []
    for _, u, l, hi, lo in merged:
        if u >= 0:
            rhs_rows.append(u)
            rhs_vals.append(hi)
        if l >= 0:
            rhs_rows.append(l)
            rhs_vals.append(-lo)

    # coefficients: later duplicates of a key overwrite earlier ones (src/tableau.ts:100-117)
    # one lookup per coefficient: key -> (row offset of the upper row or -1, row offset of the lower row or -1, is objective)
    where: dict[Any, tuple] = {}
    for key, u, l, _, _ in merged:
        if u >= 0 or l >= 0:
            where[key] = (-1 if u < 0 else u * width, -1 if l < 0 else l * width, False)
    if objective is not None:
        u, l, _ = where.get(objective, (-1, -1, False))
        where[objective] = (u, l, True)
    idx: list[int] = []
    val: list[float] = []
    add_idx, add_val, find = idx.append, val.append, where.get
    for col, (_, coefs) in enumerate(variables, start=1):
        for ckey, coef in entries(coefs):
            hit = find(ckey)
            if hit is None:
                continue
            coef = float(coef)
            u, l, is_obj = hit
            if is_obj:
                add_idx(col)
                add_val(sign * coef)
            if u >= 0:
                add_idx(u + col)
                add_val(coef)
            if l >= 0:
                add_idx(l + col)
                add_val(-coef)
    for r, v in zip(rhs_rows, rhs_vals):  # RHS cells (src/tableau.ts:119-127)
        add_idx(r * width)
        add_val(v)
    for k, col in enumerate(binary_cols):  # src/tableau.ts:130-134
        r = rows + k
        idx += (r * width, r * width + col)
        val += (1.0, 1.0)

    return np.asarray(idx, dtype=np.int32), np.asarray(val, dtype=np.float64), rows


# solve() keeps tableaus above this size (the library's zero-copy small-call limit) in the sparse form only
SPARSE_OVER_BYTES = 768 << 10


def tableau_model(model: dict, sparse_over_bytes: Optional[int] = None) -> TableauModel:
    """`sparse_over_bytes`: tableaus larger than this are returned with `matrix=None` and only the (cells, values)
    form filled in (`Tableau.dense()` materialises them); None = always dense, as the reference."""
    sign = -1.0 if model.get("direction") == "minimize" else 1.0
    objective = model.get("objective")
    variables = list(entries(model["variables"]))
    nvars = len(variables)

    # integer / binary marking (src/tableau.ts:57-71); binary wins over integer
    ints: list[int] = []
    binary_cols: list[int] = []
    integers, binaries = model.get("integers"), model.get("binaries")
    if integers is not None or binaries is not None:
        bin_set = _as_set(binaries)
        int_set = True if bin_set is True else _as_set(integers)
        for col, (key, _) in enumerate(variables, start=1):
            if bin_set is True or key in bin_set:
                binary_cols.append(col)
                ints.append(col)
            elif int_set is True or key in int_set:
                ints.append(col)

    width = nvars + 1
    constraints = list(entries(model["constraints"]))
    if _NATIVE is not None:
        cells_b, values_b, rows = _NATIVE.build(variables, constraints, objective, sign, width, binary_cols, entries)
        cells, values = np.frombuffer(cells_b, dtype=np.int32), np.frombuffer(values_b, dtype=np.float64)
    else:
        cells, values, rows = _stores_python(variables, constraints, objective, sign, width, binary_cols)
    height = rows + len(binary_cols)
    if height * width >= 2 ** 31:
        raise OverflowError("height*width must be < 2^31 (src/tableau.ts:17)")

    ident = np.arange(width + height, dtype=np.int32)
    tableau = Tableau(None, width, height, ident.copy(), ident.copy(), cells, values)
    if sparse_over_bytes is None or height * width * 8 <= sparse_over_bytes:
        tableau.dense()
    return TableauModel(tableau, sign, variables, ints)
