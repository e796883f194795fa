"""Host-side mirror of the reference's alignment interface over the libgxalign C ABI.

    alignment_table(&SequenceContainer, &Scores, is_local, reverse) -> (table, matches_at_max)   algo.rs:151-156
    retrace(&SequenceContainer, table, is_local) -> AlignedSequences                             algo.rs:287-291

The 48-byte-per-cell table of the reference never exists here: `alignment_table` returns a handle to a
finished device plan (codes in HBM, walk done), `retrace` fetches the result.  Same names, same
argument meaning, same result fields; errors that panic/exit in the reference raise here.
"""
from __future__ import annotations

import ctypes as C
import enum
import logging
from dataclasses import dataclass, field
from typing import List, Optional, Sequence as Seq, Tuple

import numpy as np

from . import _lib
from .config import Scores
from .sequence import Sequence, SequenceContainer

log = logging.getLogger("genomics_rs_b200")


class AlignmentChoice(enum.IntEnum):
    """algo.rs:124-133 (#[repr(u8)])"""
    Match = 0
    Mismatch = 1
    Insert = 2
    Delete = 3
    OpenInsert = 4
    OpenDelete = 5


@dataclass
class AlignedSequences:
    """algo.rs:135-146.  `alignment` is in walk order (start cell first), like the reference's Vec."""
    s1: Sequence
    s2: Sequence
    score: int
    matches: int
    mismatches: int
    gap_extensions: int
    opening_gaps: int
    ops: np.ndarray = field(repr=False)            # uint8 AlignmentChoice discriminants
    start: Tuple[int, int] = (0, 0)
    end: Tuple[int, int] = (0, 0)
    fill_ms: float = 0.0
    walk_ms: float = 0.0
    matches_at_max: Optional[int] = None           # alignment_table's 2nd return value (algo.rs:279-281), on request
    _ij: Optional[Tuple[np.ndarray, np.ndarray]] = field(default=None, repr=False)

    def coords(self) -> Tuple[np.ndarray, np.ndarray]:
        """(i, j) of every entry, replayed with the checked_sub rules of algo.rs:412-417."""
        if self._ij is None:
            n = int(self.ops.size)
            oi = np.zeros(n, np.uint32)
            oj = np.zeros(n, np.uint32)
            if n:
                lib = _lib.load()
                _lib.check(lib.gx_replay_ops(self.ops.ctypes.data, n, self.start[0], self.start[1],
                                             oi.ctypes.data, oj.ctypes.data))
            self._ij = (oi, oj)
        return self._ij

    @property
    def alignment(self) -> List[Tuple[AlignmentChoice, int, int]]:
        oi, oj = self.coords()
        return [(AlignmentChoice(int(c)), int(i), int(j)) for c, i, j in zip(self.ops, oi, oj)]

    def __str__(self) -> str:
        from .display import format_alignment
        return format_alignment(self)


def _scores_struct(scores) -> _lib.GxScores:
    if isinstance(scores, Scores):
        t = scores.as_tuple()
    else:
        t = tuple(int(x) for x in scores)
    for v in t:
        if not (-2**31 <= v < 2**31):
            raise _lib.GxError(3, "score does not fit int32")
    return _lib.GxScores(*t)


def _as_u8(s) -> np.ndarray:
    if isinstance(s, str):
        s = s.encode("utf-8")
    if isinstance(s, (bytes, bytearray, memoryview)):
        return np.frombuffer(bytes(s), dtype=np.uint8)
    return np.ascontiguousarray(s, dtype=np.uint8)


class Plan:
    """gx_plan wrapper: geometry fixed at creation, sequences uploaded once, executed any number of times."""

    def __init__(self, len1, len2, scores, is_local: bool, traceback: bool = True, start_cell: bool = False,
                 device: Optional[int] = None, lcs_at_max: bool = False):
        self.lib = _lib.ensure_init(device)
        self.len1 = np.ascontiguousarray(len1, np.uint64)
        self.len2 = np.ascontiguousarray(len2, np.uint64)
        assert self.len1.shape == self.len2.shape and self.len1.ndim == 1
        self.n_pairs = int(self.len1.size)
        self.traceback = bool(traceback)
        self.is_local = bool(is_local)
        flags = ((_lib.GX_FLAG_TRACEBACK if traceback else 0) | (_lib.GX_FLAG_START_CELL if start_cell else 0) |
                 (_lib.GX_FLAG_LCS_AT_MAX if lcs_at_max else 0))
        self._h = C.c_void_p()
        _lib.check(self.lib.gx_plan_create(self.len1.ctypes.data, self.len2.ctypes.data, self.n_pairs,
                                           _scores_struct(scores), int(self.is_local), flags, C.byref(self._h)))
        caps = (self.len1 + self.len2 + np.uint64(1)).astype(np.uint64)
        self.ops_off = np.zeros(self.n_pairs + 1, np.uint64)
        np.cumsum(caps, out=self.ops_off[1:])

    def upload(self, blob: np.ndarray, off1, off2) -> None:
        """blob may be any uint8 host buffer (pinned memory makes the copy a single DMA)."""
        off1 = np.ascontiguousarray(off1, np.uint64)
        off2 = np.ascontiguousarray(off2, np.uint64)
        ptr = blob.ctypes.data if isinstance(blob, np.ndarray) else int(blob[0])
        size = blob.size if isinstance(blob, np.ndarray) else int(blob[1])
        _lib.check(self.lib.gx_plan_upload(self._h, ptr, size, off1.ctypes.data, off2.ctypes.data))

    def execute(self) -> None:
        _lib.check(self.lib.gx_plan_execute(self._h))

    def fetch(self, out: Optional[np.ndarray] = None, ops: Optional[np.ndarray] = None):
        """-> (structured results array, ops blob, ops_off)"""
        if out is None:
            out = np.zeros(self.n_pairs, dtype=RESULT_DTYPE)
        if self.traceback and ops is None:
            ops = np.zeros(int(self.ops_off[-1]), np.uint8)
        _lib.check(self.lib.gx_plan_fetch(self._h, out.ctypes.data, ops.ctypes.data if ops is not None else None,
                                          self.ops_off.ctypes.data))
        return out, ops, self.ops_off

    def fetch_scores(self, out: Optional[np.ndarray] = None) -> np.ndarray:
        if out is None:
            out = np.zeros(self.n_pairs, np.int64)
        _lib.check(self.lib.gx_plan_fetch_scores(self._h, out.ctypes.data))
        return out

    def stat(self, what: int) -> float:
        return float(self.lib.gx_plan_stat(self._h, what))

    @property
    def fill_ms(self) -> float:
        return self.stat(0)

    @property
    def walk_ms(self) -> float:
        return self.stat(1)

    @property
    def launches(self) -> int:
        return int(self.stat(2))

    @property
    def cells(self) -> int:
        return int(self.stat(3))

    def close(self) -> None:
        if self._h:
            self.lib.gx_plan_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


RESULT_DTYPE = np.dtype([
    ("score", np.int64), ("start_i", np.uint64), ("start_j", np.uint64), ("end_i", np.uint64), ("end_j", np.uint64),
    ("n_ops", np.uint64), ("matches", np.uint64), ("mismatches", np.uint64), ("gap_extensions", np.uint64),
    ("opening_gaps", np.uint64), ("lcs_at_first_max", np.uint64), ("fill_ms", np.float64), ("walk_ms", np.float64)])
assert RESULT_DTYPE.itemsize == C.sizeof(_lib.GxResult)


class DeviceTable:
    """What `alignment_table` hands to `retrace`: an executed plan for one pair (codes stay in HBM)."""

    def __init__(self, plan: Plan, s1: Sequence, s2: Sequence, is_local: bool, scores=None):
        self.plan, self.s1, self.s2, self.is_local, self.scores = plan, s1, s2, is_local, scores

    @property
    def shape(self) -> Tuple[int, int]:
        return (len(self.s1.bytes()) + 1, len(self.s2.bytes()) + 1)   # Array2 shape, algo.rs:172


def alignment_table(sequence_container: SequenceContainer, scores, is_local: bool,
                    reverse_sequences: bool = False, matches_at_max: bool = False) -> Tuple[DeviceTable, Optional[int]]:
    """algo.rs:151-282.  Fills S/D/I on the GPU (and the direction codes retrace needs).
    The second return value (max_matches at the first max cell, algo.rs:279-281) is discarded by every caller of
    the reference; it costs a second fill pass, so it is computed only with matches_at_max=True (else None)."""
    if reverse_sequences:
        raise NotImplementedError("reverse_sequences is never passed by the reference (dead code, sequence.rs:103-112)")
    if len(sequence_container.sequences) > 2:                     # algo.rs:161-163
        log.warning("More than two sequences found. Only the first two will be used.")
    s1 = sequence_container.sequences[0]                           # IndexError <-> index panic, algo.rs:168-169
    s2 = sequence_container.sequences[1]
    b1, b2 = _as_u8(s1.sequence), _as_u8(s2.sequence)
    plan = Plan([b1.size], [b2.size], scores, is_local, traceback=True, lcs_at_max=matches_at_max)
    blob = np.concatenate([b1, b2]) if (b1.size + b2.size) else np.zeros(0, np.uint8)
    plan.upload(blob, [0], [b1.size])
    plan.execute()
    log.info("Sequence table shape: [%d, %d]", b1.size + 1, b2.size + 1)
    log.info("Table initialization complete, time taken: %dus", int(plan.fill_ms * 1000))
    second = None
    if matches_at_max:
        res, _, _ = plan.fetch()
        second = int(res[0]["lcs_at_first_max"])
    return DeviceTable(plan, s1, s2, is_local, scores), second


def retrace(sequence_container: SequenceContainer, alignment_table_: DeviceTable, is_local: bool,
            print_table: bool = False) -> AlignedSequences:
    """algo.rs:287-441.  The walk already ran on the device; this fetches ops, counters and score.
    print_table=True reproduces the reference's side effect at algo.rs:438: for small inputs (s1 < 200, s2 < 2000
    characters) the path grid and the three score planes go to stdout (display.rs:131-220)."""
    t = alignment_table_
    if bool(is_local) != bool(t.is_local):
        raise ValueError("retrace called with a different is_local than alignment_table")
    res, ops, ops_off = t.plan.fetch()
    r = res[0]
    n = int(r["n_ops"])
    out = AlignedSequences(
        s1=Sequence(t.s1.name, t.s1.sequence), s2=Sequence(t.s2.name, t.s2.sequence),
        score=int(r["score"]), matches=int(r["matches"]), mismatches=int(r["mismatches"]),
        gap_extensions=int(r["gap_extensions"]), opening_gaps=int(r["opening_gaps"]),
        ops=ops[:n].copy(), start=(int(r["start_i"]), int(r["start_j"])), end=(int(r["end_i"]), int(r["end_j"])),
        fill_ms=float(r["fill_ms"]), walk_ms=float(r["walk_ms"]))
    log.info("Starting at (%d, %d)", *out.start)
    log.info("Retrace complete, time taken: %dus", int(out.walk_ms * 1000))
    log.info("Retrace alignment size: %d", n)
    t.plan.close()
    if print_table:
        from .display import DISP_MAX_WIDTH, format_alignment_table
        b1, b2 = _as_u8(t.s1.sequence), _as_u8(t.s2.sequence)
        if b1.size < DISP_MAX_WIDTH and b2.size < DISP_MAX_WIDTH * 10 and t.scores is not None:
            print(format_alignment_table(out, score_planes(b1, b2, t.scores, is_local)), end="")
        else:
            log.warning("Sequence table too large to visualize")
    return out


def align(sequence_container: SequenceContainer, scores, is_local: bool) -> AlignedSequences:
    """alignment_table + retrace, the sequence main.rs:143-150 runs."""
    table, _ = alignment_table(sequence_container, scores, is_local, False)
    return retrace(sequence_container, table, is_local)


def pack_pairs(pairs: Seq[Tuple[object, object]]):
    """-> (blob, off1, len1, off2, len2) for gx_align_batch / Plan."""
    arrs = []
    off1, len1, off2, len2 = [], [], [], []
    pos = 0
    for a, b in pairs:
        a, b = _as_u8(a), _as_u8(b)
        off1.append(pos); len1.append(a.size); pos += a.size
        off2.append(pos); len2.append(b.size); pos += b.size
        arrs += [a, b]
    blob = np.concatenate(arrs) if arrs and pos else np.zeros(0, np.uint8)
    return blob, np.array(off1, np.uint64), np.array(len1, np.uint64), np.array(off2, np.uint64), np.array(len2, np.uint64)


def align_batch(pairs: Seq[Tuple[object, object]], scores, is_local: bool, traceback: bool = True,
                start_cell: bool = False, names: Optional[Seq[Tuple[str, str]]] = None,
                lcs_at_max: bool = False) -> List[AlignedSequences]:
    """Many independent pairs in one gx_align_batch call (one GPU; shard over ranks with parallel.scatter)."""
    lib = _lib.ensure_init()
    blob, off1, len1, off2, len2 = pack_pairs(pairs)
    n = len(pairs)
    res = np.zeros(n, dtype=RESULT_DTYPE)
    ops_off = np.zeros(n + 1, np.uint64)
    np.cumsum(len1 + len2 + np.uint64(1), out=ops_off[1:])
    ops = np.zeros(int(ops_off[-1]) if traceback else 0, np.uint8)
    flags = ((_lib.GX_FLAG_TRACEBACK if traceback else 0) | (_lib.GX_FLAG_START_CELL if start_cell else 0) |
             (_lib.GX_FLAG_LCS_AT_MAX if lcs_at_max else 0))
    _lib.check(lib.gx_align_batch(blob.ctypes.data if blob.size else None, blob.size, off1.ctypes.data, len1.ctypes.data,
                                  off2.ctypes.data, len2.ctypes.data, n, _scores_struct(scores), int(bool(is_local)), flags,
                                  res.ctypes.data, ops.ctypes.data if traceback else None, ops_off.ctypes.data))
    out = []
    for q in range(n):
        r = res[q]
        k = int(r["n_ops"])
        a, b = pairs[q]
        sa = a if isinstance(a, str) else bytes(_as_u8(a)).decode("latin-1")
        sb = b if isinstance(b, str) else bytes(_as_u8(b)).decode("latin-1")
        nm = names[q] if names else (f"s1_{q}", f"s2_{q}")
        o = int(ops_off[q])
        out.append(AlignedSequences(
            s1=Sequence(nm[0], sa), s2=Sequence(nm[1], sb), score=int(r["score"]), matches=int(r["matches"]),
            mismatches=int(r["mismatches"]), gap_extensions=int(r["gap_extensions"]), opening_gaps=int(r["opening_gaps"]),
            ops=ops[o:o + k].copy() if traceback else np.zeros(0, np.uint8),
            start=(int(r["start_i"]), int(r["start_j"])), end=(int(r["end_i"]), int(r["end_j"])),
            fill_ms=float(r["fill_ms"]), walk_ms=float(r["walk_ms"]),
            matches_at_max=int(r["lcs_at_first_max"]) if lcs_at_max else None))
    return out


def align_all(sequence_container: SequenceContainer, scores, is_local: bool, traceback: bool = True):
    """All-vs-all over a container (SURVEY 8f N3; BASELINE config 3 as a product feature): every pair (a, b), a < b,
    s1 = sequences[a], in one gx_align_batch call.  -> [((a, b), AlignedSequences)]"""
    seqs = sequence_container.sequences
    jobs = [(a, b) for a in range(len(seqs)) for b in range(a + 1, len(seqs))]
    out = align_batch([(seqs[a].sequence, seqs[b].sequence) for a, b in jobs], scores, is_local, traceback=traceback,
                      names=[(seqs[a].name, seqs[b].name) for a, b in jobs])
    return list(zip(jobs, out))


def score_planes(s1, s2, scores, is_local: bool):
    """(insert, delete, sub) score planes of the table, (m+1) x (n+1) int64 each, as the reference's small-table
    visualiser prints them (display.rs:190-220).  gx_debug_planes: m < 200 and n < 2000 like the reference."""
    lib = _lib.ensure_init()
    a, b = _as_u8(s1), _as_u8(s2)
    out = [np.zeros((a.size + 1, b.size + 1), np.int64) for _ in range(3)]
    _lib.check(lib.gx_debug_planes(a.ctypes.data if a.size else None, a.size, b.ctypes.data if b.size else None, b.size,
                                   _scores_struct(scores), int(bool(is_local)), *[o.ctypes.data for o in out]))
    return tuple(out)


def score_batch(blob: np.ndarray, off1, len1, off2, len2, scores, is_local: bool, out: Optional[np.ndarray] = None,
                start_cells: bool = False):
    """gx_score_batch: scores only (int64), the short-read workload's entry point.
    `out` (int64, one entry per pair) may be supplied to keep the result buffer across calls.
    start_cells=True (gx_score_batch_cells) -> (scores, start_i, start_j): each pair's start cell as uint64 arrays, the
    last cell that attains the maximum for local batches ((m, n) when that maximum is 0), (m, n) for global ones."""
    lib = _lib.ensure_init()
    blob = np.ascontiguousarray(blob, np.uint8)
    off1, len1, off2, len2 = [np.ascontiguousarray(x, np.uint64) for x in (off1, len1, off2, len2)]
    if out is None:
        out = np.empty(off1.size, np.int64)
    assert out.dtype == np.int64 and out.size == off1.size and out.flags.c_contiguous
    if start_cells:
        si, sj = np.empty(off1.size, np.uint64), np.empty(off1.size, np.uint64)
        _lib.check(lib.gx_score_batch_cells(blob.ctypes.data if blob.size else None, blob.size, off1.ctypes.data,
                                            len1.ctypes.data, off2.ctypes.data, len2.ctypes.data, off1.size,
                                            _scores_struct(scores), int(bool(is_local)), out.ctypes.data, si.ctypes.data,
                                            sj.ctypes.data))
        return out, si, sj
    _lib.check(lib.gx_score_batch(blob.ctypes.data if blob.size else None, blob.size, off1.ctypes.data, len1.ctypes.data,
                                  off2.ctypes.data, len2.ctypes.data, off1.size, _scores_struct(scores), int(bool(is_local)),
                                  out.ctypes.data))
    return out


def k0_measure() -> dict:
    """INT32/DPX issue rates measured on this GPU, CUDA-event timed (warp-instructions per clock per SM):
    the ALU pipe (VIADDMNMX, VIMNMX3), the FMA pipe (IMAD, IDP.4A), both together, and the dependency-free instruction
    mix of one score-only cell (5 instructions) and one traceback cell (9 instructions)."""
    lib = _lib.ensure_init()
    buf = (C.c_double * 9)()
    n = lib.gx_k0_measure(buf, 9)
    if n < 0:
        _lib.check(-n)
    keys = ["viaddmnmx", "vimnmx3", "imad", "idp4a", "alu_fma_pair", "score_cell", "traceback_cell", "sm_ghz", "sm_count"]
    return dict(zip(keys, [float(x) for x in buf]))
