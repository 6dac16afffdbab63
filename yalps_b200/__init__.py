"""yalps_b200: B200-native batched simplex engine behind the YALPS solve() API.

Public surface mirrors src/index.ts:1-3 of the reference: `solve`, `default_options` and the constraint
helpers, plus the new `solve_many`.  Everything numeric runs in libyalps_b200.so (hand-written sm_100a
kernels, C ABI in include/yalps_b200.h); importing this package without the built library, or calling
it without a CUDA device, raises.
"""
from .constraint import equal_to, equalTo, greater_eq, greaterEq, in_range, inRange, less_eq, lessEq
from .engine import Engine, MultiEngine, STATUS_NAMES, make_options
from .iis import model_iis
from .solver import default_options, defaultOptions, get_engine, solve, solve_many, solveMany, solve_variants
from .mps import apply_bounds, model_from_mps, netlib_model
from .sensitivity import (certificate_from_tableau, model_certificate, model_ranges, model_sensitivity,
                          ranges_from_tableau, reduced_from_tableau, row_pairs, split_reduced)
from .tableau import Tableau, TableauModel, constraint_rows, tableau_model
from .warm import warm_tableau

__all__ = [
    "solve", "solve_many", "solveMany", "default_options", "defaultOptions", "less_eq", "greater_eq", "equal_to",
    "in_range", "lessEq", "greaterEq", "equalTo", "inRange", "Engine", "MultiEngine", "make_options", "STATUS_NAMES",
    "tableau_model", "Tableau", "TableauModel", "get_engine", "model_from_mps", "netlib_model", "apply_bounds",
    "constraint_rows", "split_reduced", "model_sensitivity", "reduced_from_tableau", "ranges_from_tableau", "row_pairs",
    "model_ranges", "certificate_from_tableau", "model_certificate", "model_iis", "solve_variants", "warm_tableau",
]
