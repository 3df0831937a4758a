"""
ctypes binding of liboctreelib_b200.so (C ABI declared in include/octreelib_b200.h).

The shared library is built in-tree by `__graft_entry__.build()` (nvcc, sm_100a only).  There is
no CPU fallback: if the library is missing, or no CUDA device is present when a kernel is needed,
the calls raise.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liboctreelib_b200.so")

OL_OK = 0
OL_ERR_INVALID, OL_ERR_CUDA, OL_ERR_ALLOC, OL_ERR_RANGE = 1, 2, 3, 4
OL_ERR_OUT_OF_NODE, OL_ERR_DEPTH_CAP, OL_ERR_NONFINITE, OL_ERR_STATE, OL_ERR_POSE = 5, 6, 7, 8, 9
OL_MAX_DEPTH = 21
RANSAC_FLAG_NO_TMA, RANSAC_FLAG_EXACT_ONLY, RANSAC_FLAG_VERIFY, RANSAC_FLAG_STATS = 1, 2, 4, 8
OL_ERR_INTERNAL = 10
OL_ERR_CAPACITY = 11
OL_ERR_UNSUPPORTED = 12
OL_MAP_CENTROID, OL_MAP_SHRINK, OL_MAP_FIRST = 0, 1, 2

ALLOC_FN = C.CFUNCTYPE(C.c_void_p, C.c_void_p, C.c_size_t)
FREE_FN = C.CFUNCTYPE(None, C.c_void_p, C.c_void_p)


class ForestConfig(C.Structure):
    _fields_ = [
        ("voxel_edge_length", C.c_double),
        ("corner", C.c_double * 3),
        ("single_cell", C.c_int32),
        ("max_depth", C.c_int32),
        ("device", C.c_int32),
        ("reserved", C.c_int32),
        ("stream", C.c_void_p),
        ("alloc", ALLOC_FN),
        ("free", FREE_FN),
        ("alloc_user", C.c_void_p),
    ]


class ForestStats(C.Structure):
    _fields_ = [(n, C.c_int64) for n in (
        "n_points_inserted", "n_points_alive", "n_poses", "n_cells", "n_cell_poses", "n_leaves", "n_internal",
        "n_blocks", "max_block_size", "max_depth_reached", "key_bits", "device_bytes_peak", "sample_oob_seen")]


OL_GEOM_EXTENT, OL_GEOM_THICKNESS = 0, 1
OL_GEOM_GT, OL_GEOM_LE = 0, 1
OL_GEOM_MAX_TERMS = 8


class GeomTerm(C.Structure):
    _fields_ = [("stat", C.c_int32), ("op", C.c_int32), ("min_points", C.c_int64), ("value", C.c_double)]


class NativeLibraryMissing(ImportError):
    pass


class ExchangeCapacityError(RuntimeError):
    """a rank would receive more rows than its exchange buffers hold (parallel.py grows them and retries)"""


_p = C.c_void_p
_i32, _i64, _u32, _u64, _f64 = C.c_int32, C.c_int64, C.c_uint32, C.c_uint64, C.c_double

# name -> (restype, argtypes); every symbol include/octreelib_b200.h declares
SIGNATURES = {
    "ol_abi_version": (C.c_int, []),
    "ol_last_error": (C.c_char_p, []),
    "ol_forest_create": (C.c_int, [C.POINTER(ForestConfig), C.POINTER(_p)]),
    "ol_forest_destroy": (C.c_int, [_p]),
    "ol_forest_insert": (C.c_int, [_p, _p, _i64, _i32, C.POINTER(_i32)]),
    "ol_forest_insert_batch": (C.c_int, [_p, _p, _p, _i32, C.POINTER(_i32)]),
    "ol_forest_insert_segments": (C.c_int, [_p, _p, _i64, _i32, _p, _p, _p, _i32, _i32]),
    "ol_forest_subdivide": (C.c_int, [_p, _i64, _p, _i32]),
    "ol_forest_subdivide_table": (C.c_int, [_p, _p, _i64, _i32, _p, _i32]),
    "ol_forest_subdivide_levels": (C.c_int, [_p, _p, _i32, _p, _p, _i64, _p, _p, _i32]),
    "ol_forest_subdivide_geometric": (C.c_int, [_p, _p, _i32, _p, _p, _i64, _p, _p, _p, _p, _i32]),
    "ol_forest_filter_geometric": (C.c_int, [_p, _p, _i64, _p, _i32, _p, _i32]),
    "ol_forest_export_block_stats": (C.c_int, [_p, _p, _i32, _p, _p, _p, _p, _p, C.POINTER(_i64)]),
    "ol_forest_export_shape": (C.c_int, [_p, _p, _p, _p, C.POINTER(_i64)]),
    "ol_forest_impose_shape": (C.c_int, [_p, _p, _p, _p, _i64]),
    "ol_forest_filter": (C.c_int, [_p, _p, _i64, _p, _i32]),
    "ol_forest_ransac": (C.c_int, [_p, _p, _i32, _i32, _f64, _p, _i32, _i32, _u32, _p]),
    "ol_forest_pose_point_counts": (C.c_int, [_p, _p]),
    "ol_forest_apply_mask": (C.c_int, [_p]),
    "ol_forest_apply_pose_mask": (C.c_int, [_p, _p, _i32, _p, _i64]),
    "ol_forest_map_leaves": (C.c_int, [_p, _i32, _f64, _p, _i32, _p]),
    "ol_forest_locate": (C.c_int, [_p, _p, _i64, _i32, _p, _p]),
    "ol_forest_profile": (C.c_int, [_p, _i32]),
    "ol_forest_profile_read": (C.c_int, [_p, C.c_char_p, _i64, C.POINTER(_i64)]),
    "ol_launch_count": (_u64, []),
    "ol_release_cached_memory": (_u64, []),
    "ol_forest_stats_get": (C.c_int, [_p, C.POINTER(ForestStats)]),
    "ol_forest_stats_light": (C.c_int, [_p, C.POINTER(ForestStats)]),
    "ol_forest_pose_counts": (C.c_int, [_p, _p]),
    "ol_forest_export_cells": (C.c_int, [_p, _p, _p, _p, _p, _p]),
    "ol_forest_export_cell_poses": (C.c_int, [_p, _p, _p]),
    "ol_forest_export_leaves": (C.c_int, [_p, _p, _p, _p, _p, _p]),
    "ol_forest_export_blocks": (C.c_int, [_p, _p, _p, _p, _p]),
    "ol_forest_export_ransac": (C.c_int, [_p, _i32, _p, _p, _p, _p, _p, _p, C.POINTER(_i64)]),
    "ol_forest_export_points": (C.c_int, [_p, _p, _i32, _i32, _p, _p, _p, _p, C.POINTER(_i64)]),
    "ol_ransac_evaluate": (C.c_int, [_p, _p, _i64, _p, _i64, _p, _i32, _i32, _f64, _p, _p, _p, _p, _u32, ALLOC_FN,
                                     FREE_FN, _p]),
    "ol_ransac_stats_read": (C.c_int, [C.POINTER(_u64 * 16), _i32]),
    "ol_measure_fma_peak": (C.c_int, [_p, C.POINTER(_f64), C.POINTER(_f64)]),
    "ol_host_cell_owner": (_u32, [_i64, _i64, _i64, _u32]),
    "ol_slab_histogram": (C.c_int, [_p, _p, _i64, _f64, _f64, _i32, _p]),
    "ol_partition_by_owner": (C.c_int, [_p, _p, _i64, _p, _i32, _f64, C.POINTER(_f64 * 3), _i32, _p, _p, _p, ALLOC_FN, FREE_FN,
                                        _p]),
    "ol_exchange_ctrl_bytes": (_i64, [_i32, _i32]),
    "ol_exchange_create": (C.c_int, [_i32, _i32, _i32, _i64, _i32, _p, _p, _i32, C.POINTER(_p)]),
    "ol_exchange_destroy": (C.c_int, [_p]),
    "ol_exchange_run": (C.c_int, [_p, _p, _p, _p, _p, _i32, _i32, _i32, _p, _p, _p]),
    "ol_forest_disown_points": (C.c_int, [_p]),
    "ol_sort_pairs_u64": (C.c_int, [_p, _p, _p, _i64, _i32, _i32, ALLOC_FN, FREE_FN, _p]),
    "ol_sort_pairs_u32": (C.c_int, [_p, _p, _p, _i64, _i32, _i32, ALLOC_FN, FREE_FN, _p]),
    "ol_debug_force_legacy_sort": (C.c_int, [_i32]),
    "ol_exclusive_scan_u32": (C.c_int, [_p, _p, _p, _i64, C.POINTER(_u64), ALLOC_FN, FREE_FN, _p]),
    "ol_host_floor_divide": (_f64, [_f64, _f64]),
    "ol_host_point_key": (C.c_int, [_f64, C.POINTER(_f64 * 3), _i32, _i32, C.POINTER(_f64 * 3),
                                    C.POINTER(_i64 * 3), C.POINTER(_u64), C.POINTER(_i32)]),
}

_lib = None


def lib():
    """Load the shared library (once).  Raises NativeLibraryMissing if it was not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeLibraryMissing(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). octreelib_b200 has no CPU fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        if handle.ol_abi_version() != 2:
            raise ImportError("liboctreelib_b200.so ABI version mismatch; rebuild it")
        _lib = handle
    return _lib


_EXC = {
    OL_ERR_INVALID: ValueError,
    OL_ERR_CUDA: RuntimeError,
    OL_ERR_ALLOC: MemoryError,
    OL_ERR_RANGE: ValueError,
    OL_ERR_OUT_OF_NODE: IndexError,
    OL_ERR_DEPTH_CAP: RecursionError,
    OL_ERR_NONFINITE: ValueError,
    OL_ERR_STATE: RuntimeError,
    OL_ERR_POSE: KeyError,
    OL_ERR_INTERNAL: AssertionError,
    OL_ERR_CAPACITY: ExchangeCapacityError,
    OL_ERR_UNSUPPORTED: NotImplementedError,
}


def check(status: int):
    """Map an ol_status to the exception class the reference would have raised."""
    if status != OL_OK:
        msg = lib().ol_last_error().decode("utf-8", "replace")
        # strip the "[ol_status n] " prefix for user-facing messages that tests compare verbatim
        if msg.startswith("[ol_status"):
            msg = msg.split("] ", 1)[-1]
        raise _EXC.get(status, RuntimeError)(msg)
