"""Dual values of optimal LPs: shadow prices of constraints and reduced costs of variables.

The kernels report `reduced` (one float64 per variable id, packed like positionOfVariable, width + height per LP):
row 0 of the final tableau re-indexed by variable, reduced[v] = M[0, pos[v]] for a non-basic variable (1 <= pos[v] <
width) and +0.0 otherwise.  Ids 1..width-1 are the model's variables (columns), id width + r is the slack of tableau
row r.  This module is the one place that turns it into derivatives of the reported result (result = -sign * M[0,0],
the entering column is a positive row-0 cell, src/simplex.ts:71-79):

    d result / d x_j   =  sign * reduced[j]
    d result / d rhs_r = -sign * reduced[width + r] = y(r)

A constraint key owns at most two rows (tableau.constraint_rows): an upper row `a.x <= max` and a lower row
`-a.x <= -min`.  Shifting every finite bound of the key by t moves rhs(upper) by +t and rhs(lower) by -t, so the key's
shadow price is y(upper) - y(lower): d result / d max for a lessEq, d / d min for a greaterEq, d / d value for an
equalTo (one of its two slacks is basic, so the sum is valid in both directions).
"""
from __future__ import annotations

import numpy as np


def reduced_from_tableau(matrix: np.ndarray, width: int, height: int, pos: np.ndarray) -> np.ndarray:
    """What the kernels write into `reduced`, computed from a final tableau and its positionOfVariable (reference
    definition; the values are row-0 cells, bits as they are)."""
    row0 = np.asarray(matrix, np.float64).reshape(-1)[:width]
    p = np.asarray(pos, np.int64).reshape(-1)[:width + height]
    nonbasic = (p >= 1) & (p < width)
    return np.where(nonbasic, row0[np.where(nonbasic, p, 0)], 0.0)


def split_reduced(reduced: np.ndarray, width: int, sign: float) -> tuple:
    """Tableau level, vectorised over LPs: reduced (n, width + height) -> (y (n, height): d result / d rhs_r per row,
    d (n, width - 1): d result / d x_j per structural column j = 1..width-1)."""
    red = np.asarray(reduced, np.float64)
    red2 = red.reshape(-1, red.shape[-1])
    y = -sign * red2[:, width:]
    d = sign * red2[:, 1:width]
    if red.ndim == 1:
        return y[0], d[0]
    return y, d


def model_sensitivity(variables: list, rows: list, reduced: np.ndarray, width: int, sign: float) -> tuple:
    """Model level: (reducedCosts, shadowPrices) of one optimal LP.  `variables` are the model's (key, coefficients)
    pairs in column order, `rows` the (key, upper row | -1, lower row | -1) list of tableau.constraint_rows."""
    y, d = split_reduced(np.asarray(reduced, np.float64).reshape(-1), width, sign)
    reduced_costs = [[key, float(d[j])] for j, (key, _) in enumerate(variables)]
    shadow = []
    for key, up, lo in rows:
        v = 0.0
        if up >= 0:
            v = float(y[up])
        if lo >= 0:
            v = v - float(y[lo])
        shadow.append([key, v])
    return reduced_costs, shadow
