"""ctypes loader for libfvdb_b200.so (the C ABI of include/fvdb.h).

Fails loudly when the CUDA library is missing: there is no Python or CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# FVDB_LIB selects an experiment build of the same library (fabstir_vectordb_b200/build.py variants)
SO_PATH = os.environ.get("FVDB_LIB") or os.path.join(_HERE, "libfvdb_b200.so")

# fvdb_status (include/fvdb.h)
OK = 0
ERR_NOT_TRAINED = -1
ERR_DUPLICATE = -2
ERR_DIM_MISMATCH = -3
ERR_INSUFFICIENT_TRAINING = -4
ERR_INCONSISTENT_DIM = -5
ERR_INVALID_CONFIG = -6
ERR_CHUNK_LOAD = -7
ERR_NOT_FOUND = -8
ERR_NAN = -9
ERR_CUDA = -10
ERR_NO_DEVICE = -11
ERR_INVALID_ARG = -12
ERR_K_TOO_LARGE = -13
ERR_OOM = -14

METRIC_L2 = 0
METRIC_COS = 1
METRIC_DOT = 2
TIER_RECENT = 1
TIER_HISTORICAL = 2
TIER_BOTH = 3
SCAN_EXACT = 0
SCAN_TC = 1
OPT_SCAN_MODE = 1
OPT_SHORTLIST = 2
OPT_KMEANS_TC = 3
OPT_COALESCE = 4
OPT_PROOF_XMAX = 5
OPT_PIPELINE = 6
OPT_SCAN_SMS = 7


class TrainResult(C.Structure):
    """fvdb_train_result == TrainResult, src/ivf/core.rs:103-109."""
    _fields_ = [("iterations", C.c_uint32), ("converged", C.c_uint32),
                ("initial_error", C.c_float), ("final_error", C.c_float)]


class Stats(C.Structure):
    _fields_ = [("dim", C.c_uint32), ("nlist", C.c_uint32), ("trained", C.c_uint32),
                ("ivf_rows", C.c_uint64), ("flat_rows", C.c_uint64), ("deleted_rows", C.c_uint64),
                ("device_bytes", C.c_uint64), ("last_nq", C.c_uint32),
                ("last_fallback_queries", C.c_uint32), ("last_scanned_rows", C.c_uint64),
                ("last_algorithmic_bytes", C.c_uint64), ("last_device_ms", C.c_float),
                ("last_scan_ms", C.c_float), ("last_launches", C.c_uint32),
                ("last_batch_calls", C.c_uint32)]


_f32p = C.POINTER(C.c_float)
_u32p = C.POINTER(C.c_uint32)
_u64p = C.POINTER(C.c_uint64)
_vp = C.c_void_p

class ChunkInfo(C.Structure):
    """fvdb_chunk_info (include/fvdb_chunk.h)."""
    _fields_ = [("chunk_id", C.c_char * 128), ("start_idx", C.c_uint64), ("end_idx", C.c_uint64),
                ("n_vectors", C.c_uint64), ("dim", C.c_uint32)]


# symbol -> (restype, argtypes); every symbol include/fvdb.h, fvdb_synth.h and fvdb_chunk.h declare
SIGNATURES = {
    "fvdb_abi_version": (C.c_int, []),
    "fvdb_create": (C.c_int, [C.c_int, C.c_uint32, C.c_int, C.c_uint32, C.POINTER(_vp)]),
    "fvdb_destroy": (None, [_vp]),
    "fvdb_last_error": (C.c_char_p, [_vp]),
    "fvdb_set_option": (C.c_int, [_vp, C.c_int, C.c_uint64]),
    "fvdb_get_stats": (C.c_int, [_vp, C.POINTER(Stats)]),
    "fvdb_ivf_set_centroids": (C.c_int, [_vp, _f32p, C.c_uint32]),
    "fvdb_ivf_get_centroids": (C.c_int, [_vp, _f32p, _u32p]),
    "fvdb_ivf_train": (C.c_int, [_vp, _f32p, C.c_uint64, C.c_uint32, C.c_uint32, _f32p, C.c_uint64,
                                 C.POINTER(TrainResult)]),
    "fvdb_ivf_retrain": (C.c_int, [_vp, C.c_uint32, C.c_uint32, _f32p, C.c_uint64, C.POINTER(TrainResult)]),
    "fvdb_ivf_dump_lists": (C.c_int, [_vp, _u32p, _u32p, C.c_uint64, _u64p]),
    "fvdb_assign": (C.c_int, [_vp, _f32p, C.c_uint64, _u32p]),
    "fvdb_ivf_add": (C.c_int, [_vp, _f32p, _u32p, C.c_uint64, _u32p]),
    "fvdb_flat_add": (C.c_int, [_vp, _f32p, _u32p, C.c_uint64]),
    "fvdb_move_flat_to_ivf": (C.c_int, [_vp, _u32p, C.c_uint64, _u64p]),
    "fvdb_set_deleted": (C.c_int, [_vp, _u32p, C.c_uint64, C.c_int]),
    "fvdb_vacuum": (C.c_int, [_vp, _u64p]),
    "fvdb_search": (C.c_int, [_vp, _f32p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, _u64p,
                              C.c_uint64, _u32p, _f32p, _u32p]),
    "fvdb_search_postfilter": (C.c_int, [_vp, _f32p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, _u64p,
                                         C.c_uint64, _u32p, _f32p, _u32p]),
    "fvdb_host_alloc": (C.c_int, [C.c_size_t, C.POINTER(_vp)]),
    "fvdb_host_free": (None, [_vp]),
    "fvdb_search_device": (C.c_int, [_vp, _vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, _vp,
                                     C.c_uint64, _vp, _vp, _vp, _vp]),
    "fvdb_search_device_submit": (C.c_int, [_vp, _vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, _vp,
                                     C.c_uint64, _vp, _vp, _vp, _vp]),
    "fvdb_search_device_finish": (C.c_int, [_vp, _vp]),
    "fvdb_search_submit": (C.c_int, [_vp, _f32p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, _u32p, _f32p, _u32p]),
    "fvdb_search_finish": (C.c_int, [_vp]),
    "fvdb_coarse_device": (C.c_int, [_vp, _vp, C.c_uint32, C.c_uint32, _vp, _vp]),
    "fvdb_search_device_coarse": (C.c_int, [_vp, _vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, _vp,
                                            C.c_uint64, _vp, _vp, _vp, _vp, _vp]),
    "fvdb_coarse_device_submit": (C.c_int, [_vp, _vp, C.c_uint32, C.c_uint32, _vp, _vp]),
    "fvdb_search_device_coarse_submit": (C.c_int, [_vp, _vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, _vp,
                                                   C.c_uint64, _vp, _vp, _vp, _vp, _vp]),
    "fvdb_search_device_wait": (C.c_int, [_vp, C.c_uint32, _vp]),
    "fvdb_search_device_tiers": (C.c_int, [_vp, _vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, _vp,
                                           C.c_uint64, _vp, _vp, _vp]),
    "fvdb_search_device_tiers_submit": (C.c_int, [_vp, _vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, _vp,
                                                  C.c_uint64, _vp, _vp, _vp]),
    "fvdb_merge_topk_tiers_packed_device": (C.c_int, [_vp, _vp, C.c_uint32, C.c_uint32, C.c_uint32, _vp, _vp, _vp,
                                                      _vp]),
    "fvdb_merge_topk_device": (C.c_int, [_vp, _vp, _vp, _vp, C.c_uint32, C.c_uint32, C.c_uint32,
                                         _vp, _vp, _vp, _vp]),
    "fvdb_ivf_max_sqnorm": (C.c_int, [_vp, _f32p]),
    "fvdb_bounds_export": (C.c_int, [_vp, C.c_uint32, _vp]),
    "fvdb_bounds_import": (C.c_int, [_vp, _vp, C.c_uint32, C.c_uint32]),
    "fvdb_bounds_begin_batch": (C.c_int, [_vp, C.c_uint32, _vp]),
    "fvdb_merge_topk_packed_device": (C.c_int, [_vp, _vp, C.c_uint32, C.c_uint32, C.c_uint32, _vp, _vp, _vp, _vp]),
    "fvdb_ivf_add_device": (C.c_int, [_vp, _vp, _vp, C.c_uint64, C.c_uint32, C.c_uint32, _u64p]),
    "fvdb_flat_add_device": (C.c_int, [_vp, _vp, _vp, C.c_uint64]),
    "fvdb_ivf_add_device_owned": (C.c_int, [_vp, _vp, _vp, C.c_uint64, _vp, C.c_uint32, _u64p]),
    "fvdb_assign_device": (C.c_int, [_vp, _vp, C.c_uint64, _vp, _vp]),
    "fvdb_ivf_train_device": (C.c_int, [_vp, _vp, C.c_uint64, C.c_uint32, C.c_uint32, _vp,
                                        C.c_uint64, C.POINTER(TrainResult)]),
    "fvdb_kmeans_accumulate_device": (C.c_int, [_vp, _vp, C.c_uint64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "fvdb_kmeans_apply_device": (C.c_int, [_vp, _vp, _vp, _vp]),
    "fvdb_chunk_decode": (C.c_int, [_vp, C.c_size_t, C.POINTER(ChunkInfo), _vp, _vp, C.c_uint64]),
    "fvdb_chunk_encode": (C.c_int, [C.c_char_p, C.c_uint64, C.c_uint64, _vp, _vp, C.c_uint64, C.c_uint32,
                                    _vp, C.c_size_t, C.POINTER(C.c_size_t)]),
    "fvdb_chunk_last_error": (C.c_char_p, []),
    "fvdb_synth_rows_device": (C.c_int, [_vp, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32,
                                         C.c_float, C.c_uint64, _vp]),
    "fvdb_synth_rows_strided_device": (C.c_int, [_vp, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32,
                                                 C.c_float, C.c_uint64, C.c_uint32, C.c_uint64, _vp]),
    "fvdb_synth_queries_device": (C.c_int, [_vp, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint64,
                                            C.c_uint32, C.c_float, C.c_uint64, C.c_float, C.c_uint64,
                                            _vp]),
    "fvdb_synth_filter_device": (C.c_int, [_vp, C.c_uint64, C.c_uint32, C.c_uint64, _vp]),
}

_lib = None


def load():
    """dlopen libfvdb_b200.so and declare every entry point.  Raises if the library is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise RuntimeError(
            f"{SO_PATH} is missing: build it with `python -m fabstir_vectordb_b200.build` "
            "(there is no CPU fallback)")
    lib = C.CDLL(SO_PATH)
    for name, (res, args) in SIGNATURES.items():
        if os.environ.get("FVDB_LIB") and not hasattr(lib, name):
            continue  # an experiment build of an older source tree may lack newer entry points
        fn = getattr(lib, name)  # AttributeError if the .so does not export it
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
