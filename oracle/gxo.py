"""ctypes front-end of the CPU oracle (oracle/gx_oracle.c).

TEST INFRASTRUCTURE ONLY.  Importable from tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs; never from genomics_rs_b200/ (the product path has no
CPU fallback).  See gx_oracle.c for the reference file:line each function restates.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from dataclasses import dataclass, field
from typing import List, Optional, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libgxoracle.so")

CHOICE_NAMES = ["Match", "Mismatch", "Insert", "Delete", "OpenInsert", "OpenDelete"]


class _Result(C.Structure):
    _fields_ = [
        ("score", C.c_int64),
        ("start_i", C.c_uint64), ("start_j", C.c_uint64), ("end_i", C.c_uint64), ("end_j", C.c_uint64),
        ("n_ops", C.c_uint64), ("matches", C.c_uint64), ("mismatches", C.c_uint64),
        ("gap_extensions", C.c_uint64), ("opening_gaps", C.c_uint64),
        ("lcs_at_first_max", C.c_uint64), ("first_max_i", C.c_uint64), ("first_max_j", C.c_uint64),
        ("fill_ms", C.c_double), ("walk_ms", C.c_double),
        ("status", C.c_int32), ("pad", C.c_int32),
    ]


@dataclass
class OracleAlignment:
    score: int
    start: Tuple[int, int]
    end: Tuple[int, int]
    matches: int
    mismatches: int
    gap_extensions: int
    opening_gaps: int
    ops: np.ndarray                      # uint8 AlignmentChoice discriminants, walk order
    ops_i: Optional[np.ndarray] = None
    ops_j: Optional[np.ndarray] = None
    lcs_at_first_max: int = 0
    first_max: Tuple[int, int] = (0, 0)
    fill_ms: float = 0.0
    walk_ms: float = 0.0
    status: int = 0

    @property
    def alignment(self) -> List[Tuple[str, int, int]]:
        return [(CHOICE_NAMES[c], int(i), int(j)) for c, i, j in zip(self.ops, self.ops_i, self.ops_j)]


def build(march: Optional[str] = None, force: bool = False, out_dir: Optional[str] = None) -> str:
    """Compile the oracle with gcc.  `march="native"` builds a host-tuned copy (bench cpu_baseline) into `out_dir`
    (default oracle/_build)."""
    if march is None:
        if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(os.path.join(_HERE, "gx_oracle.c")):
            subprocess.check_call(["make", "-C", _HERE, "-s"] + (["-B"] if force else []))
        return _SO
    out = os.path.join(out_dir or os.path.join(_HERE, "_build"), f"libgxoracle_{march}.so")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    subprocess.check_call([cc, "-O3", f"-march={march}", "-fPIC", "-std=c11", "-shared", "-o", out,
                           os.path.join(_HERE, "gx_oracle.c"), "-lpthread"])
    return out


_lib = None


def _bind(lib):
    u8p, u32p, u64p, i64p = (C.POINTER(C.c_uint8), C.POINTER(C.c_uint32), C.POINTER(C.c_uint64), C.POINTER(C.c_int64))
    lib.gxo_align_faithful.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                                       C.c_int, C.POINTER(_Result), C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
    lib.gxo_align_faithful.restype = C.c_int
    lib.gxo_align_linear.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                                     C.c_int, C.c_int, C.POINTER(_Result), C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
    lib.gxo_align_linear.restype = C.c_int
    lib.gxo_score_linear.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                                     C.c_int, i64p, u64p, u64p]
    lib.gxo_score_linear.restype = C.c_int
    lib.gxo_score_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64,
                                    C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_void_p]
    lib.gxo_score_batch.restype = C.c_int
    lib.gxo_nw_score_blocked.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                                         C.c_int, C.c_uint64, i64p]
    lib.gxo_nw_score_blocked.restype = C.c_int
    lib.gxo_nw_band.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_uint64, C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, i64p]
    lib.gxo_nw_band.restype = C.c_int
    lib.gxo_planes.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int,
                               C.c_void_p, C.c_void_p, C.c_void_p]
    lib.gxo_planes.restype = C.c_int
    lib.gxo_hash_ops.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64]
    lib.gxo_hash_ops.restype = C.c_uint64
    lib.gxo_sizeof_result.restype = C.c_uint64
    assert lib.gxo_sizeof_result() == C.sizeof(_Result)
    return lib


def lib(path: Optional[str] = None):
    global _lib
    if path is not None:
        return _bind(C.CDLL(path))
    if _lib is None:
        try:
            if not os.path.exists(_SO):
                build()
            _lib = _bind(C.CDLL(_SO))
        except OSError:
            build(force=True)
            _lib = _bind(C.CDLL(_SO))
    return _lib


def _bytes(s) -> np.ndarray:
    if isinstance(s, str):
        s = s.encode()
    if isinstance(s, (bytes, bytearray)):
        return np.frombuffer(bytes(s), dtype=np.uint8)
    return np.ascontiguousarray(s, dtype=np.uint8)


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p) if a.size else None


def _wrap(res: _Result, ops, oi, oj) -> OracleAlignment:
    k = int(res.n_ops)
    return OracleAlignment(
        score=int(res.score), start=(int(res.start_i), int(res.start_j)), end=(int(res.end_i), int(res.end_j)),
        matches=int(res.matches), mismatches=int(res.mismatches), gap_extensions=int(res.gap_extensions),
        opening_gaps=int(res.opening_gaps), ops=ops[:k].copy(), ops_i=oi[:k].copy(), ops_j=oj[:k].copy(),
        lcs_at_first_max=int(res.lcs_at_first_max), first_max=(int(res.first_max_i), int(res.first_max_j)),
        fill_ms=float(res.fill_ms), walk_ms=float(res.walk_ms), status=int(res.status))


def align_faithful(s1, s2, scores, is_local: bool, so: Optional[str] = None) -> OracleAlignment:
    """alignment_table + retrace exactly as written (48 B cells).  scores = (s_match, s_mismatch, g, h)."""
    a1, a2 = _bytes(s1), _bytes(s2)
    cap = a1.size + a2.size + 2
    ops = np.zeros(cap, np.uint8); oi = np.zeros(cap, np.uint32); oj = np.zeros(cap, np.uint32)
    res = _Result()
    lib(so).gxo_align_faithful(_ptr(a1), a1.size, _ptr(a2), a2.size, *[int(x) for x in scores], int(is_local),
                               C.byref(res), _ptr(ops), _ptr(oi), _ptr(oj), cap)
    if res.status not in (0,):
        raise RuntimeError(f"oracle faithful status {res.status}")
    return _wrap(res, ops, oi, oj)


def align_linear(s1, s2, scores, is_local: bool, traceback: bool = True) -> OracleAlignment:
    a1, a2 = _bytes(s1), _bytes(s2)
    cap = a1.size + a2.size + 2
    ops = np.zeros(cap, np.uint8); oi = np.zeros(cap, np.uint32); oj = np.zeros(cap, np.uint32)
    res = _Result()
    lib().gxo_align_linear(_ptr(a1), a1.size, _ptr(a2), a2.size, *[int(x) for x in scores], int(is_local), int(traceback),
                           C.byref(res), _ptr(ops), _ptr(oi), _ptr(oj), cap)
    if res.status != 0:
        raise RuntimeError(f"oracle linear status {res.status}")
    return _wrap(res, ops, oi, oj)


def score_linear(s1, s2, scores, is_local: bool) -> Tuple[int, int, int]:
    a1, a2 = _bytes(s1), _bytes(s2)
    sc = C.c_int64(); si = C.c_uint64(); sj = C.c_uint64()
    rc = lib().gxo_score_linear(_ptr(a1), a1.size, _ptr(a2), a2.size, *[int(x) for x in scores], int(is_local),
                                C.byref(sc), C.byref(si), C.byref(sj))
    if rc:
        raise RuntimeError(f"oracle score status {rc}")
    return int(sc.value), int(si.value), int(sj.value)


def score_batch(blob: np.ndarray, off1, len1, off2, len2, scores, is_local: bool, n_threads: int = 1,
                so: Optional[str] = None) -> np.ndarray:
    blob = np.ascontiguousarray(blob, np.uint8)
    off1, len1, off2, len2 = [np.ascontiguousarray(x, np.uint64) for x in (off1, len1, off2, len2)]
    out = np.zeros(len(off1), np.int64)
    rc = lib(so).gxo_score_batch(_ptr(blob), _ptr(off1), _ptr(len1), _ptr(off2), _ptr(len2), len(off1),
                                 *[int(x) for x in scores], int(is_local), int(n_threads), _ptr(out))
    if rc:
        raise RuntimeError(f"oracle batch status {rc}")
    return out


def nw_score_blocked(s1, s2, scores, n_threads: int = 8, blk: int = 4096) -> int:
    a1, a2 = _bytes(s1), _bytes(s2)
    sc = C.c_int64()
    rc = lib().gxo_nw_score_blocked(_ptr(a1), a1.size, _ptr(a2), a2.size, *[int(x) for x in scores], n_threads, blk, C.byref(sc))
    if rc:
        raise RuntimeError(f"oracle blocked status {rc}")
    return int(sc.value)


def nw_band(s1, s2_band, col0: int, scores, left=None):
    """One column band (columns col0+1 .. col0+len(s2_band)) of the global table.
    left = (V, I) int64 arrays of column col0 (rows 1..m), or None for col0 == 0.
    -> (score at the band's bottom-right cell, (V, I) of the band's last column)"""
    a1, a2 = _bytes(s1), _bytes(s2_band)
    m = a1.size
    out_v, out_i = np.zeros(m, np.int64), np.zeros(m, np.int64)
    if left is not None:
        in_v, in_i = np.ascontiguousarray(left[0], np.int64), np.ascontiguousarray(left[1], np.int64)
        assert in_v.size == m and in_i.size == m
    sc = C.c_int64()
    rc = lib().gxo_nw_band(_ptr(a1), m, _ptr(a2), a2.size, int(col0), *[int(x) for x in scores],
                           _ptr(in_v) if left is not None else None, _ptr(in_i) if left is not None else None,
                           _ptr(out_v), _ptr(out_i), C.byref(sc))
    if rc:
        raise RuntimeError(f"oracle band status {rc}")
    return int(sc.value), (out_v, out_i)


def planes(s1, s2, scores, is_local: bool):
    """(insert, delete, sub) score planes of the reference's table, (m+1) x (n+1) int64 each"""
    a1, a2 = _bytes(s1), _bytes(s2)
    out = [np.zeros((a1.size + 1, a2.size + 1), np.int64) for _ in range(3)]
    rc = lib().gxo_planes(_ptr(a1), a1.size, _ptr(a2), a2.size, *[int(x) for x in scores], int(is_local), *[_ptr(o) for o in out])
    if rc:
        raise RuntimeError(f"oracle planes status {rc}")
    return tuple(out)


def hash_ops(ops: np.ndarray, start: Tuple[int, int]) -> int:
    ops = np.ascontiguousarray(ops, np.uint8)
    return int(lib().gxo_hash_ops(_ptr(ops), ops.size, int(start[0]), int(start[1])))
