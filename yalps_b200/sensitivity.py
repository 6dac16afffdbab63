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

Ranging (how far the optimal basis holds) is one interval [lo, hi] per variable id, packed like `reduced`, with
b+_r = max(M[r,0], +0.0), g_c = min(M[0,c], +0.0), and a cell counting when |cell| > precision (ranges_from_tableau):

    structural j, non-basic at column c:  (-inf, -g_c)
    structural j, basic at row r:         (max g_c / M[r,c] over counting M[r,c] > 0, min over M[r,c] < 0), c = 1..W-1
    slack of row k:                       (max -b+_r / d[r] over counting d[r] > 0, min over d[r] < 0), r = 1..H-1

where [lo, hi] bounds the shift of the initial objective cell M0[0,j] = sign * c_j (structural) or of row k's initial
RHS (slack) that keeps the final basis optimal, resp. primal feasible.  d is the column of the final tableau that
shifting row k's RHS moves column 0 along (-d per unit), dir(W+k): the non-basic column M[:, pos], or the unit vector
of the basic row.  With a pair (the other row of the same constraint key, whose RHS moves by -t when row k's moves by
+t) d = dir(W+k) - dir(W+pair): a key with two finite bounds must be ranged as one, its two slacks always sum to a
constant.  An empty max is -inf, an empty min +inf, a zero is +0.0, and lo <= 0 <= hi.  Ids 0 and W and every id of a
non-optimal LP are NaN.

Certificates explain the other two outcomes, one float64 per variable id packed like `reduced`
(certificate_from_tableau):

    infeasible (status 1): r = the row phase 1 chose, the lowest r in 1..H-1 whose M[r,0] is the minimum over the rows
        with M[r,0] < -precision (the reference's strict-< scan: NaN never qualifies, -inf does).  Phase 1 returns
        `infeasible` on that row without pivoting (src/simplex.ts:106-142), so the final tableau is that tableau.
        cert[0] = M[r,0], cert[W] = +0.0, and for every other id v: M[r, pos[v]] if 1 <= pos[v] < W (bits as they
        are), 1.0 if pos[v] == W + r, +0.0 otherwise.
    unbounded (status 2): c = int(value), the entering column.  cert[0] = M[0,c], cert[W] = +0.0, and for every other
        id v: 1.0 if pos[v] == c, -M[pos[v] - W, c] if W < pos[v] < W + H (the sign bit flipped), +0.0 otherwise.
    every other status, an infeasible LP without a qualifying row, an unbounded LP with c outside 1..W-1: NaN.

Row r of the final tableau is sum_k y_k (original row k), where original row k reads a_k.x + s_k = b_k: the slack
entries cert[W + k] are the multipliers y_k (>= -precision, or the row would have had an entering column), the
structural entries equal sum_k y_k a_kj (>= -precision) and cert[0] = sum_k y_k b_k < 0.  So no x >= 0 satisfies every
row: a Farkas certificate.  A column c with no leaving row is a direction d >= 0 (cert[1..]) that keeps every row
feasible while the objective moves at rate d result / dt = sign * cert[0], the convention of reducedCosts.  Candidates
whose ratio was NaN or +-inf were rejected by the reference too, and the certificate is still its row or column; the
values are raw cells, nothing below precision is cleaned.  At model level (model_certificate) a key's multiplier is
cert[W + upper] - cert[W + lower], the sign convention of shadowPrices: m > 0 means its `max` takes part, m < 0 its
`min`.
"""
from __future__ import annotations

import numpy as np

_CHUNK = 256  # slack ids per vectorised step of ranges_from_tableau (bounds its H x _CHUNK temporaries)


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


def _z(x):
    """+0.0 for either zero (x + 0.0 rounds -0.0 to +0.0 and leaves everything else as it is)."""
    return x + 0.0


def ranges_from_tableau(matrix: np.ndarray, width: int, height: int, pos: np.ndarray, precision: float,
                        pairs: np.ndarray = None, optimal: bool = True) -> tuple:
    """What the kernels write into `range_lo` / `range_hi` (one value per variable id, packed like `reduced`),
    computed from a final tableau, its positionOfVariable and the row pairs (int per row, -1 = none; row_pairs).
    Reference definition: every value is one IEEE division followed by a max or min (module docstring)."""
    W, H = int(width), int(height)
    lo = np.full(W + H, -np.inf)
    hi = np.full(W + H, np.inf)
    if not optimal:
        lo[:] = hi[:] = np.nan
        return lo, hi
    M = np.asarray(matrix, np.float64).reshape(-1)[:H * W].reshape(H, W)
    p = np.asarray(pos, np.int64).reshape(-1)[:W + H]
    prec = float(precision)
    g = np.minimum(M[0], 0.0)
    bplus = np.maximum(M[:, 0], 0.0)
    nonbasic = (p >= 1) & (p < W)
    rows = np.arange(H)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        # structural variables
        js = np.arange(1, W)
        nb = nonbasic[js]
        hi[js[nb]] = -g[p[js[nb]]]
        bj = js[~nb]
        r = p[bj] - W
        ok = (r >= 1) & (r < H)
        bj, r = bj[ok], r[ok]
        if bj.size:
            A = M[r][:, 1:]
            Q = g[None, 1:] / A
            cnt = np.abs(A) > prec
            lo[bj] = np.where(cnt & (A > 0), Q, -np.inf).max(axis=1)
            hi[bj] = np.where(cnt & (A < 0), Q, np.inf).min(axis=1)

        # slacks: d = dir(W+k) [- dir(W+pair)]
        def direction(ids):
            q = p[ids]
            nbq = (q >= 1) & (q < W)
            D = M[:, np.where(nbq, q, 0)]
            return np.where(nbq[None, :], D, (rows[:, None] == (q - W)[None, :]).astype(np.float64))

        pr = None if pairs is None else np.asarray(pairs, np.int64).reshape(-1)[:H]
        for k0 in range(1, H, _CHUNK):
            ks = np.arange(k0, min(H, k0 + _CHUNK))
            d = direction(W + ks)
            if pr is not None:
                has = pr[ks] >= 0
                if has.any():
                    dq = direction(W + np.where(has, pr[ks], ks))
                    d = np.where(has[None, :], d - dq, d)
            d = d[1:]
            Q = -bplus[1:, None] / d
            cnt = np.abs(d) > prec
            lo[W + ks] = np.where(cnt & (d > 0), Q, -np.inf).max(axis=0)
            hi[W + ks] = np.where(cnt & (d < 0), Q, np.inf).min(axis=0)
    lo, hi = _z(lo), _z(hi)
    lo[[0, W]] = np.nan
    hi[[0, W]] = np.nan
    return lo, hi


def row_pairs(rows: list, height: int) -> np.ndarray:
    """pairs for ranges_from_tableau / the `_ranging` entries: upper <-> lower row of every key that has both, from
    the (key, upper row | -1, lower row | -1) list of tableau.constraint_rows; -1 elsewhere (int32, one per row)."""
    out = np.full(int(height), -1, np.int32)
    for _, up, lo in rows:
        if up >= 0 and lo >= 0:
            out[up], out[lo] = lo, up
    return out


def model_ranges(variables: list, rows: list, range_lo: np.ndarray, range_hi: np.ndarray, width: int,
                 sign: float) -> tuple:
    """Model level: (costRanges, rhsRanges) of one optimal LP from ranges computed with row_pairs(rows).
    costRanges [[variable, lo, hi]]: allowable shifts of the variable's objective coefficient.  rhsRanges
    [[key, lo, hi]]: allowable shift of all the key's finite bounds together (the shift its shadow price is the
    derivative for): the upper row's range, else the lower row's negated and swapped (its RHS is -min)."""
    lo = np.asarray(range_lo, np.float64).reshape(-1)
    hi = np.asarray(range_hi, np.float64).reshape(-1)
    W = int(width)
    cost = []
    for j, (key, _) in enumerate(variables):
        a, b = float(lo[j + 1]), float(hi[j + 1])
        cost.append([key, _z(a), _z(b)] if sign > 0 else [key, _z(-b), _z(-a)])
    rhs = []
    for key, up, lw in rows:
        if up >= 0:
            rhs.append([key, _z(float(lo[W + up])), _z(float(hi[W + up]))])
        elif lw >= 0:
            rhs.append([key, _z(-float(hi[W + lw])), _z(-float(lo[W + lw]))])
        else:
            rhs.append([key, -np.inf, np.inf])
    return cost, rhs


_SIGN = np.uint64(0x8000000000000000)


def certificate_from_tableau(matrix: np.ndarray, width: int, height: int, pos: np.ndarray, status: int, value: float,
                             precision: float) -> np.ndarray:
    """What the kernels write into `cert` (one value per variable id, packed like `reduced`), computed from a final
    tableau, its positionOfVariable and the status and value the solve reported (module docstring)."""
    W, H = int(width), int(height)
    out = np.full(W + H, np.nan)
    M = np.asarray(matrix, np.float64).reshape(-1)[:H * W].reshape(H, W)
    p = np.asarray(pos, np.int64).reshape(-1)[:W + H]
    prec = float(precision)
    if status == 1:
        b = M[1:, 0]
        ok = b < -prec  # NaN never qualifies
        if not ok.any():
            return out
        r = 1 + int(np.flatnonzero(ok & (b == b[ok].min()))[0])
        nonbasic = (p >= 1) & (p < W)
        out[:] = np.where(nonbasic, M[r][np.where(nonbasic, p, 0)], np.where(p == W + r, 1.0, 0.0))
        out[0] = M[r, 0]
    elif status == 2:
        x = float(value)
        if not (1.0 <= x < W):
            return out
        c = int(x)
        basic = (p > W) & (p < W + H)
        col = M[:, c].copy()
        col.view(np.uint64)[:] ^= _SIGN
        out[:] = np.where(p == c, 1.0, np.where(basic, col[np.where(basic, p - W, 0)], 0.0))
        out[0] = M[0, c]
    else:
        return out
    out[W] = 0.0
    return out


def model_certificate(variables: list, rows: list, cert: np.ndarray, width: int, status: int) -> tuple:
    """Model level: (infeasibilityCertificate, unboundedRay) of one LP from its certificate_from_tableau values, both
    empty unless the status matches.  infeasibilityCertificate [[key, m]] in first-seen order, m = cert[W + upper] -
    cert[W + lower] (a missing row counts as 0; m > 0: the key's max takes part, m < 0: its min).  unboundedRay
    [[variable, d]] in model order, d = cert[j + 1]."""
    c = np.asarray(cert, np.float64).reshape(-1)
    W = int(width)
    farkas, ray = [], []
    if status == 1 and not np.isnan(c[0]):
        for key, up, lw in rows:
            m = 0.0
            if up >= 0:
                m = float(c[W + up])
            if lw >= 0:
                m = m - float(c[W + lw])
            farkas.append([key, m])
    elif status == 2 and not np.isnan(c[0]):
        ray = [[key, float(c[j + 1])] for j, (key, _) in enumerate(variables)]
    return farkas, ray
