"""Irreducible infeasible subsets: which constraints of an infeasible LP conflict.

An IIS is a set of constraints that has no solution while dropping any one of them leaves a set that has one.  A
Farkas certificate (sensitivity.certificate_from_tableau) proves infeasibility, but it puts a multiplier on every key and
its support is often far from minimal; an IIS names the conflict.

Row subsets.  For a row set S of 1..H-1, T_S is the model tableau with every row outside S zeroed (+0.0 in every cell,
column 0 included).  Row 0, the objective, always stays, so "T_S is infeasible" means exactly "solve() of the model
restricted to S returns infeasible".  A zeroed row is a removed row for any precision >= 0: phase 1 only picks a row
with M[r,0] < -precision, the ratio test skips cells <= precision, and a pivot leaves every row whose pivot-column cell
is within 1e-16 untouched -- so status, value, pivot counts and every other row are bit-identical to solving the model
without that row.  All subset LPs of a model therefore have its height x width.  Variables keep their implicit x >= 0
in every subset; those bounds are never part of an IIS (bounds that mps.apply_bounds turns into rows are ordinary rows
and can be).

supp(cert) of an infeasible LP is the set of rows k with cert[W + k] > +0.0, the raw value: NaN and both zeros do not
count, noise of +1e-17 does (which only keeps a set larger).

The search (Engine.iis, yalps_iis; deterministic, so the GPU and a host restatement agree exactly):

    round 0: solve T.  Not infeasible -> its status, empty IIS.
    S <- supp(cert(T)); fallback <- all rows
    repeat:
        u_1 < ... < u_m = S;  one batch: LP_0 = T_S, LP_i = T_{S \\ {u_i}}
        LP_0 not infeasible:  S <- fallback; continue
        I = {i >= 1: LP_i infeasible};  I empty: return S
        i* = argmin over I of |supp(cert(LP_i))| (lowest i on ties)
        fallback <- S \\ {u_i*};  S <- supp(cert(LP_i*))

The result S was solved infeasible and every S \\ {r} was solved optimal or unbounded in the same batch: irreducible by
the solver's own judgement, unless some LP_i of the last round ended `cycled` (that row stays, undecided) or the
timeout expired between rounds (the last set solved infeasible is returned).
"""
from __future__ import annotations


def model_iis(rows: list, iis_rows) -> list:
    """Model level: the IIS tableau rows as [[constraint key, "max" | "min"], ...], keys in first-seen order, a key's
    upper row ("max", a.x <= max) before its lower row ("min", -a.x <= -min).  `rows` is the (key, upper row | -1,
    lower row | -1) list of tableau.constraint_rows; an `equal` key, or a key with min > max, can contribute both."""
    s = {int(r) for r in iis_rows}
    out = []
    for key, up, lo in rows:
        if up >= 0 and up in s:
            out.append([key, "max"])
        if lo >= 0 and lo in s:
            out.append([key, "min"])
    return out
