"""ctypes binding of ``libhrag_b200.so`` (C ABI declared in ``include/hrag_b200.h``).

There is no CPU fallback and no alternative backend: if the shared library is missing (not
built) this module raises, and ``hrag_create`` fails when no B200 is visible.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhrag_b200.so")

PPR_POWER, PPR_CHEBYSHEV = 0, 1
SIM_FP32, SIM_BF16X3, SIM_BF16 = 0, 1, 2
PPR_FP32, PPR_MIXED = 0, 1


class HragError(RuntimeError):
    pass


class Stats(C.Structure):
    _fields_ = [
        ("ms_sim_fact", C.c_double), ("ms_select_fact", C.c_double), ("ms_sim_passage", C.c_double),
        ("ms_seed", C.c_double), ("ms_ppr", C.c_double), ("ms_topk", C.c_double), ("ms_comm", C.c_double),
        ("ppr_sweeps", C.c_int64), ("ppr_columns", C.c_int64), ("kernel_launches", C.c_int64),
        ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64),
        ("ppr_residual", C.c_double), ("ppr_error_bound", C.c_double),
    ]

    def as_dict(self):
        return {name: getattr(self, name) for name, _ in self._fields_}


_p = C.c_void_p
_i32, _i64, _f32 = C.c_int32, C.c_int64, C.c_float

# name -> (restype, argtypes); exactly the declarations of include/hrag_b200.h
SIGNATURES = {
    "hrag_last_error": (C.c_char_p, []),
    "hrag_version": (C.c_char_p, []),
    "hrag_create": (C.c_int, [_p, C.c_int, C.c_int, C.POINTER(_p)]),
    "hrag_destroy": (None, [_p]),
    "hrag_comm_unique_id": (C.c_int, [_p]),
    "hrag_comm_init": (C.c_int, [_p, _p, C.c_int, C.c_int]),
    "hrag_comm_set_row_bounds": (C.c_int, [_p, _p, C.c_int]),
    "hrag_p2p_export": (C.c_int, [_p, _p]),
    "hrag_p2p_import": (C.c_int, [_p, _p, C.c_int]),
    "hrag_load_graph_csr": (C.c_int, [_p, _i64, _i64, _i64, _i64, _p, _p, _p]),
    "hrag_load_graph_coo": (C.c_int, [_p, _i64, _i64, _p, _p, _p]),
    "hrag_load_tables": (C.c_int, [_p, _i64, _p, _i64, _p, _p, _p]),
    "hrag_load_embeddings": (C.c_int, [_p, C.c_int, _i64, _i32, _p, C.c_int]),
    "hrag_load_embeddings_begin": (C.c_int, [_p, C.c_int, _i64, _i32]),
    "hrag_load_embeddings_chunk": (C.c_int, [_p, C.c_int, _i64, _i64, _p, C.c_int]),
    "hrag_set_options": (C.c_int, [_p, C.c_int, C.c_int, C.c_int, C.c_int]),
    "hrag_set_ppr_precision": (C.c_int, [_p, C.c_int, C.c_int, C.c_int]),
    "hrag_stage_a": (C.c_int, [_p, _i32, _p, _i32, _p, _p, _p]),
    "hrag_stage_b": (C.c_int, [_p, _i32, _p, _p, _p, _i32, _p, _f32, _f32, _i32, _i32, _i32, _f32, _p, _p]),
    "hrag_plan_sweeps": (C.c_int, [_f32, _f32, _i32, _i32, _p, _p, _p, _p, _p]),
    "hrag_retrieve_resident": (C.c_int, [_p, _i32, _p, _p, _f32, _f32, _i32, _i32, _i32, _f32, _p, _p]),
    "hrag_ppr": (C.c_int, [_p, _i32, _p, _f32, _i32, _f32, _p]),
    "hrag_similarity": (C.c_int, [_p, C.c_int, _i32, _p, _p]),
    "hrag_topk_similarity": (C.c_int, [_p, C.c_int, _i32, _p, _i32, _p, _p]),
    "hrag_knn_threshold": (C.c_int, [_p, C.c_int, _i32, _p, _f32, _i32, _p, _p, _p]),
    "hrag_bench_sweep": (C.c_int, [_p, _i32, _i32, _i32, C.POINTER(_f32)]),
    "hrag_set_tuning": (C.c_int, [_p, C.c_int]),
    "hrag_stream": (_p, [_p]),
    "hrag_get_stats": (C.c_int, [_p, C.POINTER(Stats)]),
    "hrag_reset_stats": (C.c_int, [_p]),
    "hrag_debug_keep_scores": (C.c_int, [_p, C.c_int]),
    "hrag_debug_copy": (C.c_int, [_p, C.c_int, _p, _i64, C.POINTER(_i64)]),
}

_lib = None


def load():
    """Load the shared library once; raises HragError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise HragError(
            f"{LIB_PATH} is missing: build it with `make -C hipporag_b200/csrc` (or "
            "`python -c 'import __graft_entry__ as g; g.build()'`). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here = header/library out of sync
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int):
    if rc != 0:
        raise HragError(load().hrag_last_error().decode("utf-8", "replace"))
