"""ctypes binding of libgxalign.so (include/gxalign.h).  The library is the product; this file is glue.

There is deliberately no fallback: if the shared library is missing or no sm_100 GPU is usable,
every call raises.  Nothing here imports or calls oracle/.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GX_LIB_PATH") or os.path.join(_HERE, "libgxalign.so")   # GX_LIB_PATH: A/B builds of the library

GX_OK = 0
GX_FLAG_TRACEBACK = 1
GX_FLAG_LCS_AT_MAX = 2
GX_FLAG_START_CELL = 4

EXPORTS = [
    "gx_init", "gx_shutdown", "gx_device_count", "gx_strerror", "gx_last_error", "gx_version", "gx_check_scores",
    "gx_align_pair", "gx_align_batch", "gx_score_batch", "gx_score_batch_cells", "gx_align_reads", "gx_plan_create", "gx_plan_upload", "gx_plan_execute",
    "gx_plan_fetch", "gx_plan_fetch_scores", "gx_plan_destroy", "gx_plan_stat", "gx_replay_ops", "gx_k0_measure",
    "gx_band_range", "gx_band_create", "gx_band_export", "gx_band_connect", "gx_band_upload", "gx_band_execute",
    "gx_band_score", "gx_band_stat", "gx_band_destroy", "gx_nw_score_banded", "gx_debug_planes", "gx_debug_tile_order",
]


class GxScores(C.Structure):
    _fields_ = [("s_match", C.c_int32), ("s_mismatch", C.c_int32), ("g", C.c_int32), ("h", C.c_int32)]


class GxResult(C.Structure):
    _fields_ = [
        ("score", C.c_int64),
        ("start_i", C.c_uint64), ("start_j", C.c_uint64), ("end_i", C.c_uint64), ("end_j", C.c_uint64),
        ("n_ops", C.c_uint64), ("matches", C.c_uint64), ("mismatches", C.c_uint64),
        ("gap_extensions", C.c_uint64), ("opening_gaps", C.c_uint64), ("lcs_at_first_max", C.c_uint64),
        ("fill_ms", C.c_double), ("walk_ms", C.c_double),
    ]


class GxError(RuntimeError):
    def __init__(self, status: int, detail: str = ""):
        self.status = status
        super().__init__(f"libgxalign status {status}: {detail}")


_lib = None
_lock = threading.Lock()
_inited_device = None


def load() -> C.CDLL:
    """dlopen the in-tree library and declare every prototype of include/gxalign.h."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -m genomics_rs_b200.build` "
                "(nvcc, sm_100a).  genomics_rs_b200 has no CPU or PyTorch fallback.")
        lib = C.CDLL(LIB_PATH)
        vp, u64, i32 = C.c_void_p, C.c_uint64, C.c_int
        lib.gx_init.argtypes = [i32]; lib.gx_init.restype = i32
        lib.gx_shutdown.argtypes = []; lib.gx_shutdown.restype = None
        lib.gx_device_count.argtypes = []; lib.gx_device_count.restype = i32
        lib.gx_strerror.argtypes = [i32]; lib.gx_strerror.restype = C.c_char_p
        lib.gx_last_error.argtypes = []; lib.gx_last_error.restype = C.c_char_p
        lib.gx_version.argtypes = []; lib.gx_version.restype = C.c_char_p
        lib.gx_check_scores.argtypes = [GxScores, u64, u64]; lib.gx_check_scores.restype = i32
        lib.gx_align_pair.argtypes = [vp, u64, vp, u64, GxScores, i32, i32, C.POINTER(GxResult), vp, u64]
        lib.gx_align_pair.restype = i32
        lib.gx_align_batch.argtypes = [vp, u64, vp, vp, vp, vp, u64, GxScores, i32, i32, vp, vp, vp]
        lib.gx_align_batch.restype = i32
        lib.gx_score_batch.argtypes = [vp, u64, vp, vp, vp, vp, u64, GxScores, i32, vp]
        lib.gx_score_batch.restype = i32
        lib.gx_score_batch_cells.argtypes = [vp, u64, vp, vp, vp, vp, u64, GxScores, i32, vp, vp, vp]
        lib.gx_score_batch_cells.restype = i32
        lib.gx_align_reads.argtypes = [vp, u64, vp, vp, vp, vp, u64, GxScores, i32, vp, vp, vp]
        lib.gx_align_reads.restype = i32
        lib.gx_plan_create.argtypes = [vp, vp, u64, GxScores, i32, i32, C.POINTER(vp)]; lib.gx_plan_create.restype = i32
        lib.gx_plan_upload.argtypes = [vp, vp, u64, vp, vp]; lib.gx_plan_upload.restype = i32
        lib.gx_plan_execute.argtypes = [vp]; lib.gx_plan_execute.restype = i32
        lib.gx_plan_fetch.argtypes = [vp, vp, vp, vp]; lib.gx_plan_fetch.restype = i32
        lib.gx_plan_fetch_scores.argtypes = [vp, vp]; lib.gx_plan_fetch_scores.restype = i32
        lib.gx_plan_destroy.argtypes = [vp]; lib.gx_plan_destroy.restype = None
        lib.gx_plan_stat.argtypes = [vp, i32]; lib.gx_plan_stat.restype = C.c_double
        lib.gx_replay_ops.argtypes = [vp, u64, u64, u64, vp, vp]; lib.gx_replay_ops.restype = i32
        lib.gx_k0_measure.argtypes = [vp, i32]; lib.gx_k0_measure.restype = i32
        lib.gx_band_range.argtypes = [u64, i32, i32, C.POINTER(u64), C.POINTER(u64)]; lib.gx_band_range.restype = i32
        lib.gx_band_create.argtypes = [u64, u64, i32, i32, i32, GxScores, C.POINTER(vp)]; lib.gx_band_create.restype = i32
        lib.gx_band_export.argtypes = [vp, vp, u64]; lib.gx_band_export.restype = i32
        lib.gx_band_connect.argtypes = [vp, vp, vp]; lib.gx_band_connect.restype = i32
        lib.gx_band_upload.argtypes = [vp, vp, vp]; lib.gx_band_upload.restype = i32
        lib.gx_band_execute.argtypes = [vp]; lib.gx_band_execute.restype = i32
        lib.gx_band_score.argtypes = [vp, C.POINTER(C.c_int64), C.POINTER(i32)]; lib.gx_band_score.restype = i32
        lib.gx_band_stat.argtypes = [vp, i32]; lib.gx_band_stat.restype = C.c_double
        lib.gx_band_destroy.argtypes = [vp]; lib.gx_band_destroy.restype = None
        lib.gx_nw_score_banded.argtypes = [vp, u64, vp, u64, GxScores, i32, C.POINTER(C.c_int64)]
        lib.gx_nw_score_banded.restype = i32
        lib.gx_debug_tile_order.argtypes = [vp, vp, u64, i32, i32, vp, u64, C.POINTER(u64)]; lib.gx_debug_tile_order.restype = i32
        lib.gx_debug_planes.argtypes = [vp, u64, vp, u64, GxScores, i32, vp, vp, vp]; lib.gx_debug_planes.restype = i32
        _lib = lib
    return _lib


def check(status: int) -> None:
    if status != GX_OK:
        lib = load()
        detail = lib.gx_strerror(status).decode()
        extra = lib.gx_last_error().decode()
        raise GxError(status, f"{detail}{' -- ' + extra if extra else ''}")


def ensure_init(device: int | None = None) -> C.CDLL:
    """gx_init on first use.  device defaults to $LOCAL_RANK (one process per GPU) or 0."""
    global _inited_device
    lib = load()
    if _inited_device is None:
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", "0"))
        check(lib.gx_init(device))
        _inited_device = device
    return lib


def shutdown() -> None:
    global _inited_device
    if _lib is not None and _inited_device is not None:
        _lib.gx_shutdown()
        _inited_device = None
