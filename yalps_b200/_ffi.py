"""ctypes binding of libyalps_b200.so (C ABI in include/yalps_b200.h).

The library is the product: if it is missing, was not built, or no CUDA device is present, importing
callers get an exception -- there is no CPU fallback anywhere in this package.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
# YALPS_B200_LIB: alternative build of the same library (A/B experiments, instrumented builds)
LIB_PATH = os.environ.get("YALPS_B200_LIB") or os.path.join(_HERE, "libyalps_b200.so")

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)
_lp = C.POINTER(C.c_int64)
_vp = C.c_void_p


class Options(C.Structure):
    """struct yalps_options (include/yalps_b200.h) == Required<Options>, src/types.ts:203-265."""

    _fields_ = [
        ("precision", C.c_double),
        ("max_pivots", C.c_double),
        ("tolerance", C.c_double),
        ("timeout_ms", C.c_double),
        ("max_iterations", C.c_double),
        ("check_cycles", C.c_int32),
        ("reserved", C.c_int32),
    ]


class YalpsError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"yalps_b200 error {code}: {message}")
        self.code = code


# name -> (restype, argtypes); every symbol include/yalps_b200.h declares
SIGNATURES = {
    "yalps_default_options": (None, [C.POINTER(Options)]),
    "yalps_create": (C.c_int, [C.c_int, C.POINTER(_vp)]),
    "yalps_destroy": (None, [_vp]),
    "yalps_last_error": (C.c_char_p, [_vp]),
    "yalps_device_info": (C.c_int, [_vp, _ip, _ip, _ip, _ip]),
    "yalps_set_tuning": (C.c_int, [_vp, C.c_int32, C.c_int32]),
    "yalps_set_row_groups": (C.c_int, [_vp, C.c_int32]),
    "yalps_probe_division": (C.c_int, [_vp, C.c_int64, C.c_uint64, C.c_int32, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "yalps_launch_count": (C.c_int64, [_vp]),
    "yalps_set_row_counter": (C.c_int, [_vp, _vp, C.c_int32]),
    "yalps_host_alloc": (C.c_int, [_vp, C.c_uint64, C.POINTER(_vp)]),
    "yalps_host_free": (C.c_int, [_vp, _vp]),
    "yalps_solve_batch": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int32, _vp, C.POINTER(Options), _vp, _vp, _vp, _vp,
                                    _vp, _vp, _vp]),
    "yalps_solve_ragged": (C.c_int, [_vp, C.c_int64, _vp, _vp, _vp, _vp, C.POINTER(Options), _vp, _vp, _vp, _vp, _vp,
                                     _vp, _vp]),
    "yalps_solve_batch_basis": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int32, _vp, _vp, _vp, C.POINTER(Options), _vp, _vp,
                                          _vp, _vp, _vp, _vp, _vp]),
    "yalps_solve_ragged_basis": (C.c_int, [_vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(Options), _vp, _vp, _vp,
                                           _vp, _vp, _vp, _vp]),
    "yalps_solve_replicas": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int32, _vp, _vp, C.POINTER(Options), _vp, _vp, _vp,
                                       _vp, _vp, _vp]),
    "yalps_set_replica_sharing": (C.c_int, [_vp, C.c_int32]),
    "yalps_replica_forks": (C.c_int64, [_vp]),
    "yalps_create_multi": (C.c_int, [_ip, C.c_int32, C.POINTER(_vp)]),
    "yalps_destroy_multi": (None, [_vp]),
    "yalps_multi_last_error": (C.c_char_p, [_vp]),
    "yalps_multi_size": (C.c_int32, [_vp]),
    "yalps_multi_ctx": (_vp, [_vp, C.c_int32]),
    "yalps_multi_launch_count": (C.c_int64, [_vp]),
    "yalps_multi_solve_batch": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int32, _vp, _vp, _vp, C.POINTER(Options), _vp, _vp,
                                          _vp, _vp, _vp, _vp, _vp]),
    "yalps_multi_solve_ragged": (C.c_int, [_vp, C.c_int64, _vp, _vp, _vp, _vp, C.POINTER(Options), _vp, _vp, _vp, _vp, _vp,
                                           _vp, _vp]),
    "yalps_multi_solve_replicas": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int32, _vp, _vp, C.POINTER(Options), _vp, _vp,
                                             _vp, _vp, _vp, _vp]),
    "yalps_incumbent_allreduce": (C.c_int, [_vp, _dp, _dp]),
    "yalps_multi_solve": (C.c_int, [_vp, C.c_int32, C.c_int32, _vp, _vp, C.c_int32, C.c_double, C.POINTER(Options),
                                    C.c_int32, _ip, _dp, _ip, _vp, _vp, _vp, _ip, _dp, _vp, _vp]),
    "yalps_multi_solve_many": (C.c_int, [_vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(Options), C.c_int32,
                                         _vp, _vp, _vp, _vp, _vp, _vp]),
    "yalps_multi_solve_large": (C.c_int, [_vp, C.c_int32, C.c_int32, _vp, C.POINTER(Options), _ip, _dp, _vp, _vp, _vp, _vp,
                                          _vp, _dp]),
    "yalps_solve_batch_device": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int32, _vp, _vp, C.POINTER(Options), _vp,
                                           _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "yalps_generate_synthetic_device": (C.c_int, [_vp, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32,
                                                  C.c_uint32, _vp, _vp]),
    "yalps_generate_replicas_device": (C.c_int, [_vp, C.c_int64, C.c_int64, C.c_int32, C.c_int32, _vp, _vp, C.c_int32,
                                                 C.c_double, C.c_uint32, _vp, _vp]),
    "yalps_bnb_set_root": (C.c_int, [_vp, C.c_int32, C.c_int32, _vp, _vp, _vp, C.c_int32]),
    "yalps_bnb_solve_nodes": (C.c_int, [_vp, C.c_int64, _vp, _vp, _vp, _vp, C.POINTER(Options), _vp, _vp, _vp, _vp,
                                        _vp, _vp, _vp]),
    "yalps_branch_and_cut": (C.c_int, [_vp, _vp, C.c_int32, C.c_double, C.c_double, C.POINTER(Options), _ip, _dp, _ip,
                                       _vp, _vp, _vp, _vp]),
    "yalps_bnb_set_wave": (C.c_int, [_vp, C.c_int32]),
    "yalps_bnb_set_mode": (C.c_int, [_vp, C.c_int32]),
    "yalps_solve": (C.c_int, [_vp, C.c_int32, C.c_int32, _vp, _vp, C.c_int32, C.c_double, C.POINTER(Options), _ip, _dp,
                              _ip, _vp, _vp, _vp, _ip, _dp, _vp, _vp]),
    "yalps_solve_sparse": (C.c_int, [_vp, C.c_int32, C.c_int32, C.c_int64, _vp, _vp, _vp, C.c_int32, C.c_double,
                                     C.POINTER(Options), _ip, _dp, _ip, _vp, _vp, _vp, _ip, _dp, _vp, _vp]),
    "yalps_solve_batch_duals": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int32, _vp, _vp, _vp, C.POINTER(Options), _vp, _vp,
                                          _vp, _vp, _vp, _vp, _vp, _vp]),
    "yalps_solve_ragged_duals": (C.c_int, [_vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(Options), _vp, _vp, _vp,
                                           _vp, _vp, _vp, _vp, _vp]),
    "yalps_solve_replicas_duals": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int32, _vp, _vp, C.POINTER(Options), _vp, _vp,
                                             _vp, _vp, _vp, _vp, _vp]),
    "yalps_solve_batch_device_duals": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int32, _vp, _vp, C.POINTER(Options), _vp,
                                                 _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "yalps_solve_sparse_duals": (C.c_int, [_vp, C.c_int32, C.c_int32, C.c_int64, _vp, _vp, C.POINTER(Options), _vp, _vp,
                                           _vp, _vp, _vp, _vp, _vp]),
    "yalps_multi_solve_batch_duals": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int32, _vp, _vp, _vp, C.POINTER(Options),
                                                _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "yalps_multi_solve_ragged_duals": (C.c_int, [_vp, C.c_int64, _vp, _vp, _vp, _vp, C.POINTER(Options), _vp, _vp, _vp,
                                                 _vp, _vp, _vp, _vp, _vp]),
    "yalps_multi_solve_replicas_duals": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int32, _vp, _vp, C.POINTER(Options),
                                                   _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "yalps_solve_batch_ranging": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int32, _vp, _vp, _vp, C.POINTER(Options), _vp,
                                            _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "yalps_solve_ragged_ranging": (C.c_int, [_vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(Options), _vp, _vp,
                                             _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "yalps_solve_sparse_ranging": (C.c_int, [_vp, C.c_int32, C.c_int32, C.c_int64, _vp, _vp, C.POINTER(Options), _vp, _vp,
                                             _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "yalps_ranging_device": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int32, _vp, _vp, _vp, _vp, C.c_double, _vp, _vp,
                                       _vp]),
    "yalps_multi_solve_batch_ranging": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int32, _vp, _vp, _vp, C.POINTER(Options),
                                                  _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "yalps_multi_solve_ragged_ranging": (C.c_int, [_vp, C.c_int64, _vp, _vp, _vp, _vp, C.POINTER(Options), _vp, _vp, _vp,
                                                   _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "yalps_solve_batch_certificate": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int32, _vp, _vp, _vp, C.POINTER(Options),
                                                _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "yalps_solve_ragged_certificate": (C.c_int, [_vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(Options), _vp,
                                                 _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "yalps_solve_sparse_certificate": (C.c_int, [_vp, C.c_int32, C.c_int32, C.c_int64, _vp, _vp, C.POINTER(Options), _vp,
                                                 _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "yalps_certificate_device": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int32, _vp, _vp, _vp, _vp, C.c_double, _vp,
                                           _vp]),
    "yalps_multi_solve_batch_certificate": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int32, _vp, _vp, _vp,
                                                      C.POINTER(Options), _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                                      _vp, _vp, _vp]),
    "yalps_multi_solve_ragged_certificate": (C.c_int, [_vp, C.c_int64, _vp, _vp, _vp, _vp, C.POINTER(Options), _vp, _vp,
                                                       _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "yalps_solve_row_subsets": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int32, _vp, _vp, C.POINTER(Options), _vp, _vp,
                                          _vp, _vp, _vp]),
    "yalps_iis": (C.c_int, [_vp, C.c_int32, C.c_int32, _vp, C.POINTER(Options), _ip, _vp, _ip, _vp]),
    "yalps_iis_sparse": (C.c_int, [_vp, C.c_int32, C.c_int32, C.c_int64, _vp, _vp, C.POINTER(Options), _ip, _vp, _ip,
                                   _vp]),
    "yalps_solve_warm": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int32, _vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(Options),
                                   _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "yalps_solve_warm_sparse": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int32, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp,
                                          _vp, C.POINTER(Options), _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                          _vp, _vp, _vp, _vp, _vp]),
    "yalps_multi_solve_warm": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int32, _vp, _vp, _vp, _vp, _vp, _vp,
                                         C.POINTER(Options), _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                         _vp, _vp, _vp]),
    "yalps_solve_warm_extend": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _vp, _vp, _vp,
                                          _vp, _vp, _vp, _vp, _vp, C.POINTER(Options), _vp, _vp, _vp, _vp, _vp, _vp,
                                          _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "yalps_solve_warm_extend_sparse": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                                 C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                                 C.POINTER(Options), _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                                 _vp, _vp, _vp, _vp, _vp]),
    "yalps_multi_solve_warm_extend": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _vp, _vp,
                                                _vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(Options), _vp, _vp, _vp, _vp,
                                                _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "yalps_round_to_precision": (C.c_int, [_vp, C.c_int64, _vp, C.c_double, _vp]),
    "yalps_measure_smem_bandwidth": (C.c_int, [_vp, _dp, _dp]),
    "yalps_measure_tmem_bandwidth": (C.c_int, [_vp, _dp, _dp]),
    "yalps_measure_l2_bandwidth": (C.c_int, [_vp, C.c_uint64, _dp]),
    "yalps_measure_h2d_bandwidth": (C.c_int, [_vp, _vp, C.c_uint64, C.c_int32, C.c_int32, _dp]),
}

_lib = None


def build(verbose: bool = False) -> str:
    """Compile csrc/ for sm_100a with nvcc (cross-compiles without a GPU)."""
    subprocess.check_call(["make", "-C", os.path.join(_HERE, "csrc"), "-s"] + ([] if not verbose else ["V=1"]))
    return LIB_PATH


def load() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(yalps_b200 has no CPU fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib
