"""solve(model, options) / solve_many(models, options): the public API of the reference (src/index.ts:1-3,
src/YALPS.ts:73-92) in front of the B200 engine.

Model, Options and Solution keep the reference's shapes and spellings (src/types.ts):
  model   = {"direction", "objective", "constraints", "variables", "integers", "binaries"}
  options = {"precision", "checkCycles", "maxPivots", "tolerance", "timeout", "maxIterations",
             "includeZeroVariables"}
  solution = {"status": "optimal"|"infeasible"|"unbounded"|"timedout"|"cycled", "result", "variables"}
One option goes beyond the reference: `sensitivity` (default False).  When it is true (LP models only), every
Solution also has "reducedCosts" ([[variable, d result / d variable], ...], model order) and "shadowPrices"
([[constraint key, d result / d bound], ...], first-seen order): raw doubles for an optimal LP, empty lists
otherwise (yalps_b200.sensitivity has the conventions).
A second one, `ranging` (default False), implies `sensitivity` and adds "costRanges" ([[variable, lo, hi], ...]: the
allowable shifts of the variable's objective coefficient that keep the optimal basis) and "rhsRanges" ([[constraint
key, lo, hi], ...]: the allowable shifts of all of the key's finite bounds together over which its shadow price holds),
computed on the GPU from the final tableau; empty lists unless optimal.
A third one, `certificate` (default False), adds "infeasibilityCertificate" ([[constraint key, multiplier], ...],
first-seen order: non-negative combinations of the keys' max rows and min rows that read 0 <= negative, the Farkas
proof that no solution exists) and "unboundedRay" ([[variable, direction], ...], model order: a direction that keeps
every constraint satisfied while the result moves toward the reported +-inf), computed on the GPU from the final
tableau; each is an empty list unless the status is infeasible, resp. unbounded.
A fourth one, `iis` (default False), adds "irreducibleInfeasibleSet" ([[constraint key, "max" | "min"], ...], first-seen
order, a key's max before its min): a set of bounds that cannot hold together while any one fewer can, found by batched
deletion rounds on the GPU (yalps_b200.iis); an empty list unless the status is infeasible.  Variables keep x >= 0
throughout, and those bounds are never listed.
solve_variants(model, variants, options) re-optimises variants of one LP model (changed bounds and objective
coefficients, added constraints and variables) from the model's own final basis on the GPU (yalps_b200.warm), returning
one Solution per variant.
The tableau is built on the host (tableau.py), the simplex and branch-and-cut numerics run on the GPU
through the C ABI; there is no CPU solve path.
"""
from __future__ import annotations

import math
from typing import Optional, Sequence

import numpy as np

from .engine import Engine, MultiEngine, STATUS_NAMES, make_options
from .iis import model_iis
from .sensitivity import model_certificate, model_ranges, model_sensitivity, row_pairs
from .tableau import SPARSE_OVER_BYTES, Tableau, TableauModel, constraint_rows, entries, tableau_model
from .warm import variant_additions, variant_vectors

# src/YALPS.ts:52-60
_DEFAULTS = {
    "precision": 1e-8,
    "checkCycles": False,
    "maxPivots": 8192,
    "tolerance": 0,
    "timeout": math.inf,
    "maxIterations": 32768,
    "includeZeroVariables": False,
}

#: exported mutable copy, like `defaultOptions` (src/YALPS.ts:65); editing it does not change solve()
default_options = dict(_DEFAULTS)
defaultOptions = default_options

_engines: dict = {}


def get_engine(device: int = 0) -> Engine:
    """Process-wide engine per device (created on first use; raises if there is no CUDA device)."""
    eng = _engines.get(device)
    if eng is None:
        eng = _engines[device] = Engine(device)
    return eng


def _js_round(x: float) -> float:
    if math.isnan(x) or math.isinf(x) or abs(x) >= 2.0 ** 52:
        return x
    r = float(math.floor(x))
    if x - r >= 0.5:
        r += 1.0
    return -0.0 if r == 0.0 and math.copysign(1.0, x) < 0 else r


def round_to_precision(num: float, precision: float) -> float:
    """src/util.ts:1-4 (host copy, used only to format reported variable values)."""
    rounding = _js_round(1.0 / precision)
    return _js_round((num + 2.0 ** -52) * rounding) / rounding


def _c_options(opt: dict):
    return make_options(opt["precision"], opt["maxPivots"], opt["checkCycles"], opt["tolerance"], opt["timeout"],
                        opt["maxIterations"])


def _solution(tabmod: TableauModel, status: str, result: float, rhs, pos, var, opt: dict) -> dict:
    """src/YALPS.ts:8-50: needs only column 0 and the basis arrays of the final tableau."""
    width = tabmod.tableau.width
    precision = opt["precision"]
    names = tabmod.variables
    if status == "optimal" or (status == "timedout" and not math.isnan(result)):
        out = []
        for i, (key, _) in enumerate(names):
            row = int(pos[i + 1]) - width
            value = float(rhs[row]) if row >= 0 else 0.0
            if value > precision:
                out.append([key, round_to_precision(value, precision)])
            elif opt["includeZeroVariables"]:
                out.append([key, 0.0])
        return {"status": status, "result": -tabmod.sign * result, "variables": out}
    if status == "unbounded":
        v = int(var[int(result)]) - 1
        return {"status": "unbounded", "result": tabmod.sign * math.inf,
                "variables": [[names[v][0], math.inf]] if 0 <= v < len(names) else []}
    return {"status": status, "result": math.nan, "variables": []}


def _check_lp(tabmod: TableauModel):
    if tabmod.integers:
        raise ValueError("sensitivity, ranging, certificate and iis are defined for LP models only (this model has "
                         "integer or binary variables)")


def _wants(opt: dict) -> tuple:
    """(duals, ranges, certificate): what the options ask of the root LP."""
    rng = bool(opt.get("ranging"))
    return bool(opt.get("sensitivity")) or rng, rng, bool(opt.get("certificate"))


def _with_certificate(sol: dict, tabmod: TableauModel, model: dict, cert, rows: Optional[list] = None) -> dict:
    """Solution + infeasibilityCertificate / unboundedRay (both empty unless the status matches); rows: the model's
    constraint_rows unless given."""
    status = {"infeasible": 1, "unbounded": 2}.get(sol["status"], 0)
    rows = (rows if rows is not None else _rows(model)) if status == 1 else []
    farkas, ray = model_certificate(tabmod.variables, rows, cert, tabmod.tableau.width, status)
    return {**sol, "infeasibilityCertificate": farkas, "unboundedRay": ray}


def _with_iis(sol: dict, tabmod: TableauModel, model: dict, eng, copt) -> dict:
    """Solution + irreducibleInfeasibleSet: the search runs (on the tableau form solve built) only when infeasible."""
    out = []
    if sol["status"] == "infeasible":
        t = tabmod.tableau
        r = (eng.iis(t.matrix, t.height, t.width, copt) if t.matrix is not None
             else eng.iis_sparse(t.cells, t.values, t.height, t.width, copt))
        out = model_iis(_rows(model), r["rows"])
    return {**sol, "irreducibleInfeasibleSet": out}


def _rows(model: dict) -> list:
    return constraint_rows(list(entries(model["constraints"])))


def _with_sensitivity(sol: dict, tabmod: TableauModel, model: dict, reduced, ranges: Optional[tuple] = None,
                      rows: Optional[list] = None) -> dict:
    """Solution + reducedCosts / shadowPrices, and costRanges / rhsRanges when `ranges` = (range_lo, range_hi) is
    given (all empty unless optimal); rows: the model's constraint_rows unless given."""
    if sol["status"] != "optimal":
        out = {**sol, "reducedCosts": [], "shadowPrices": []}
        return out if ranges is None else {**out, "costRanges": [], "rhsRanges": []}
    rows = rows if rows is not None else _rows(model)
    rc, sp = model_sensitivity(tabmod.variables, rows, reduced, tabmod.tableau.width, tabmod.sign)
    out = {**sol, "reducedCosts": rc, "shadowPrices": sp}
    if ranges is None:
        return out
    cr, rr = model_ranges(tabmod.variables, rows, ranges[0], ranges[1], tabmod.tableau.width, tabmod.sign)
    return {**out, "costRanges": cr, "rhsRanges": rr}


def solve(model: dict, options: Optional[dict] = None, *, engine: Optional[Engine] = None,
          info: Optional[dict] = None) -> dict:
    """Runs the solver on `model` (src/YALPS.ts:73-92).  `info`, if given, receives engine statistics."""
    opt = {**_DEFAULTS, **(options or {})}
    # big model tableaus are almost all zeros: they go to the device as (cell, value) pairs (yalps_solve_sparse) and
    # never exist densely on the host; small ones take the library's zero-copy path as a dense image
    sparse_ok = hasattr(engine, "solve_tableau_sparse") if engine is not None else True
    tabmod = tableau_model(model, SPARSE_OVER_BYTES if sparse_ok else None)
    t = tabmod.tableau
    duals, rng, cert = _wants(opt)
    want_iis = bool(opt.get("iis"))
    if duals or cert or want_iis:
        _check_lp(tabmod)
    eng = engine or get_engine()
    if want_iis:
        sol = solve(model, {**opt, "iis": False}, engine=eng, info=info)
        return _with_iis(sol, tabmod, model, eng, _c_options(opt))
    if duals or cert:
        # the root LP is the whole solve: one LP with its reduced-cost row (dense batch of one, or the cell pairs), and
        # its ranges and certificate when asked for
        pairs = row_pairs(_rows(model), t.height) if rng else None
        if t.matrix is None:
            r = eng.solve_lp_sparse(t.cells, t.values, t.height, t.width, _c_options(opt), want_ranges=rng, pairs=pairs,
                                    want_certificates=cert)
            status, value, rhs, pos, var, red = (r["status"], r["value"], r["rhs"], r["pos"], r["var"], r["reduced"])
            piv = r["pivots"]
            ranges = (r["range_lo"], r["range_hi"]) if rng else None
            c = r["certificate"] if cert else None
        else:
            r = eng.solve_batch(t.matrix, t.height, t.width, _c_options(opt), want_duals=duals, want_ranges=rng,
                                pairs=pairs, want_certificates=cert)
            status, value = int(r["status"][0]), float(r["value"][0])
            rhs, pos, var = r["rhs"][0], r["pos"][0], r["var"][0]
            red = r["reduced"][0] if duals else None
            piv = (int(r["pivots"][0, 0]), int(r["pivots"][0, 1]))
            ranges = (r["range_lo"][0], r["range_hi"][0]) if rng else None
            c = r["certificate"][0] if cert else None
        if info is not None:
            info.update(nodes=0, node_pivots=0, max_cuts=0, max_heap=0, waves=0, device_nodes=0, wave_us=0, bnb_us=0,
                        root_status=STATUS_NAMES[status], root_value=value, root_pivots=piv, height=t.height,
                        width=t.width, final_rhs=rhs, final_pos=pos, final_var=var)
        sol = _solution(tabmod, STATUS_NAMES[status], value, rhs, pos, var, opt)
        if duals:
            sol = _with_sensitivity(sol, tabmod, model, red, ranges)
        return _with_certificate(sol, tabmod, model, c) if cert else sol
    if t.matrix is None:
        r = eng.solve_tableau_sparse(t.cells, t.values, t.height, t.width, tabmod.integers, tabmod.sign, _c_options(opt))
    else:
        # a MultiEngine shards the branch-and-bound frontier over its GPUs (same search, same result)
        r = eng.solve_tableau(t.matrix, t.height, t.width, tabmod.integers, tabmod.sign, _c_options(opt))
    if info is not None:
        info.update(r["stats"], root_status=STATUS_NAMES[r["root_status"]], root_value=r["root_value"],
                    root_pivots=r["root_pivots"], height=t.height, width=t.width, final_rhs=r["rhs"],
                    final_pos=r["pos"], final_var=r["var"])
    return _solution(tabmod, STATUS_NAMES[r["status"]], r["result"], r["rhs"], r["pos"], r["var"], opt)


def solve_variants(model: dict, variants: Sequence[dict], options: Optional[dict] = None, *,
                   engine: Optional[Engine] = None) -> list:
    """Solutions of variants of one LP model, each re-optimised from the model's final basis on the GPU
    (Engine.solve_warm; yalps_b200.warm states the start tableau).  A variant is {"constraints": {key: {"min" | "max" |
    "equal": value}}, "objective": {variable: coefficient}}, both parts optional: a key's `max` sets its upper row's
    right-hand side, `min` its lower row's (to -min), `equal` both; a coefficient replaces the variable's objective
    coefficient.  A variant may also add constraints and variables ("addConstraints", "addVariables";
    yalps_b200.warm.variant_additions has their form): each is solved at its batch's largest added shape, padded with
    zero rows and columns that no pivot chooses or changes, and mapped back with its own names.  Returns one Solution
    per variant in order, the shape solve() returns; the options `sensitivity`, `ranging` and `certificate` add their
    fields as in solve_many, added variables and keys included.  The results equal the reference's loop run from the
    warm tableau: statuses agree with a cold solve of the changed model and optimal results agree within the precision,
    but with alternative optima the reported vertex can differ.  ValueError for MILP models, the `iis` option, unknown
    keys or variables, a bound the base model does not have (an infinite bound has no tableau row), and the refusals of
    variant_additions."""
    opt = {**_DEFAULTS, **(options or {})}
    if opt.get("iis"):
        raise ValueError("solve_variants does not take the iis option (a search per variant)")
    sparse_ok = hasattr(engine, "solve_warm_sparse") if engine is not None else True
    tabmod = tableau_model(model, SPARSE_OVER_BYTES if sparse_ok else None)
    if tabmod.integers:
        raise ValueError("solve_variants is defined for LP models only (this model has integer or binary variables)")
    t = tabmod.tableau
    rhs, obj = variant_vectors(model, list(variants), t)
    add = variant_additions(model, list(variants), t)
    if not variants:
        return []
    duals, rng, cert = _wants(opt)
    pairs = (row_pairs(_rows(model), t.height) if add is None else add.pairs) if rng else None
    eng = engine or get_engine()
    want = dict(options=_c_options(opt), want_duals=duals, want_ranges=rng, pairs=pairs, want_certificates=cert)
    if add is not None:  # only then: an engine without the extend entries still serves every other variant batch
        want.update(add_rows=add.rows, add_cols=add.cols)
    if t.matrix is None:
        r = eng.solve_warm_sparse(t.cells, t.values, t.height, t.width, rhs, obj, **want)
    else:
        r = eng.solve_warm(t.matrix, t.height, t.width, rhs, obj, **want)
    out = []
    for i in range(len(variants)):
        tm, keys = tabmod, None
        if add is not None:  # the variant's own names over the padded shape
            H, W = t.height + add.rows.shape[1], t.width + add.cols.shape[1]
            tm = TableauModel(Tableau(None, W, H, None, None), tabmod.sign, add.variables[i], [])
            keys = add.keys[i]
        sol = _solution(tm, STATUS_NAMES[int(r["status"][i])], float(r["value"][i]), r["rhs"][i], r["pos"][i],
                        r["var"][i], opt)
        if duals:
            sol = _with_sensitivity(sol, tm, model, r["reduced"][i],
                                    (r["range_lo"][i], r["range_hi"][i]) if rng else None, rows=keys)
        out.append(_with_certificate(sol, tm, model, r["certificate"][i], rows=keys) if cert else sol)
    return out


def _worker_engines(device: int, count: int) -> list:
    """Extra engines (one ctx each, same GPU) for concurrent branch-and-cut searches; a ctx is single-threaded."""
    out = []
    for k in range(count):
        key = (device, "milp", k)
        eng = _engines.get(key)
        if eng is None:
            eng = _engines[key] = Engine(device)
        out.append(eng)
    return out


def solve_many(models: Sequence[dict], options: Optional[dict] = None, *, engine: Optional[Engine] = None,
               milp_workers: int = 4) -> list:
    """solveMany(models, options): all root LPs go to the device as ONE ragged batch (LPs of different sizes are
    grouped per kernel configuration by the library).  Models with integer variables whose root is optimal then
    run branch and cut; their searches are latency-bound node waves, so up to `milp_workers` of them run
    concurrently, each on its own context / streams of the same GPU (the C ABI releases the GIL for a whole search).
    Results are identical to calling solve() per model."""
    opt = {**_DEFAULTS, **(options or {})}
    copt = _c_options(opt)
    tabmods = [tableau_model(m) for m in models]
    duals, rng, cert = _wants(opt)
    want_iis = bool(opt.get("iis"))
    if duals or cert or want_iis:
        for tm in tabmods:
            _check_lp(tm)
    eng = engine or get_engine()
    if not tabmods:
        return []
    if want_iis:  # per infeasible model, one search after the other
        sols = solve_many(models, {**opt, "iis": False}, engine=eng, milp_workers=milp_workers)
        return [_with_iis(s, tm, m, eng, copt) for s, tm, m in zip(sols, tabmods, models)]
    if duals or cert:  # LP models only: the ragged root batch is the whole solve (one GPU or sharded)
        pairs = [row_pairs(_rows(m), tm.tableau.height) for tm, m in zip(tabmods, models)] if rng else None
        roots = eng.solve_ragged([tm.tableau.matrix for tm in tabmods],
                                 [(tm.tableau.height, tm.tableau.width) for tm in tabmods], copt, want_duals=duals,
                                 want_ranges=rng, pairs=pairs, want_certificates=cert)
        out = []
        for tm, m, r in zip(tabmods, models, roots):
            sol = _solution(tm, STATUS_NAMES[r["status"]], r["value"], r["rhs"], r["pos"], r["var"], opt)
            if duals:
                sol = _with_sensitivity(sol, tm, m, r["reduced"], (r["range_lo"], r["range_hi"]) if rng else None)
            out.append(_with_certificate(sol, tm, m, r["certificate"]) if cert else sol)
        return out
    if isinstance(eng, MultiEngine):  # one C-ABI call: roots sharded over the GPUs, searches dealt to worker contexts
        res = eng.solve_many_tableaus(tabmods, copt, searches_per_device=milp_workers)
        return [_solution(tm, STATUS_NAMES[r["status"]], r["result"], r["rhs"], r["pos"], r["var"], opt)
                for tm, r in zip(tabmods, res)]
    roots = eng.solve_ragged([tm.tableau.matrix for tm in tabmods],
                             [(tm.tableau.height, tm.tableau.width) for tm in tabmods], copt,
                             want_matrices=any(tm.integers for tm in tabmods))
    out: list = [None] * len(tabmods)
    milp = []
    for i, (tm, r) in enumerate(zip(tabmods, roots)):
        status = STATUS_NAMES[r["status"]]
        if not tm.integers or status != "optimal":
            out[i] = _solution(tm, status, r["value"], r["rhs"], r["pos"], r["var"], opt)
        else:
            milp.append(i)

    def search(e: Engine, i: int):
        tm, r = tabmods[i], roots[i]
        t = tm.tableau
        e.bnb_set_root(r["matrix"], t.height, t.width, r["pos"], r["var"], 2 * len(tm.integers))
        b = e.branch_and_cut(tm.integers, tm.sign, r["value"], copt)
        out[i] = _solution(tm, STATUS_NAMES[b["status"]], b["result"], b["rhs"], b["pos"], b["var"], opt)

    workers = max(1, min(int(milp_workers), len(milp)))
    if workers <= 1:
        for i in milp:
            search(eng, i)
    else:
        import queue
        import threading
        todo: "queue.SimpleQueue[int]" = queue.SimpleQueue()
        for i in milp:
            todo.put(i)
        errors: list = []

        def run(e: Engine):
            while True:
                try:
                    i = todo.get_nowait()
                except queue.Empty:
                    return
                try:
                    search(e, i)
                except Exception as exc:  # surfaced after the join
                    errors.append(exc)
                    return

        threads = [threading.Thread(target=run, args=(e,)) for e in _worker_engines(eng.device, workers)]
        for th in threads:
            th.start()
        for th in threads:
            th.join()
        if errors:
            raise errors[0]
    return out


solveMany = solve_many
