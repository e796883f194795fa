"""Local start cells from the short-read kernels: read plans with GX_FLAG_START_CELL and gx_score_batch_cells.

The start cell is the last cell in row-major order that attains the table maximum (algo.rs:306-323), (m, n) when that
maximum is 0; global batches report (m, n).  Each GPU case compares with the oracle's score_linear, which keeps that
cell, and where noted also the whole gx_result with the same pairs through the wavefront path (plans of < 1024 pairs).
The read kernels rely on one argument (DESIGN.md 4, K4): no cell outside a pair's table can tie a positive maximum.
The tie cases below are built so that the cells that decide it lie in padded rows, padded columns, other lanes and the
other half of an s16x2 register."""
import ctypes as C
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from conftest import CONFIG_TOML, TEST_CONFIG, random_pair
from test_score_range import READS_MAX_LEN, _read_set, _reads16_edges, _stream_set, max_local_a

gpu = pytest.mark.gpu
_ACGT = np.frombuffer(b"ACGT", np.uint8)


# ---- the oracle's start cells for a packed batch: gxo_score_linear per pair, spread over threads (ctypes calls drop
# the GIL); the oracle's own batch call keeps only the scores
def oracle_cells(oracle, blob, off1, len1, off2, len2, scores, is_local):
    lib = oracle.lib()
    blob = np.ascontiguousarray(blob, np.uint8)
    base = blob.ctypes.data
    n = len(off1)
    sc, si, sj = np.zeros(n, np.int64), np.zeros(n, np.uint64), np.zeros(n, np.uint64)
    a, b, g, h = (int(x) for x in scores)

    def run(lo, hi):
        v, i, j = C.c_int64(), C.c_uint64(), C.c_uint64()
        for q in range(lo, hi):
            rc = lib.gxo_score_linear(base + int(off1[q]), int(len1[q]), base + int(off2[q]), int(len2[q]), a, b, g, h,
                                      int(is_local), C.byref(v), C.byref(i), C.byref(j))
            assert rc == 0, rc
            sc[q], si[q], sj[q] = v.value, i.value, j.value

    step = 4096
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 1) as ex:
        list(ex.map(lambda lo: run(lo, min(n, lo + step)), range(0, n, step)))
    return sc, si, sj


@pytest.fixture(scope="module")
def gx():
    import genomics_rs_b200 as gx
    from genomics_rs_b200 import _lib
    _lib.ensure_init()
    return gx


def _status(fn):
    from genomics_rs_b200 import _lib
    try:
        fn()
    except _lib.GxError as e:
        return e.status
    return 0


def _plan(gx, packed, scores, is_local=True, start_cell=True):
    """one plan -> (gx_result array, stat 9, stat 26)"""
    blob, off1, len1, off2, len2 = packed
    plan = gx.Plan(len1, len2, scores, is_local, traceback=False, start_cell=start_cell)
    try:
        plan.upload(blob, off1, off2)
        plan.execute()
        res, _, _ = plan.fetch()
        return res, plan.stat(9), plan.stat(26)
    finally:
        plan.close()


def _wavefront(gx, packed, scores, is_local=True):
    """the same pairs through the wavefront start-cell path: plans of 1023 pairs stay below the read-plan threshold"""
    blob, off1, len1, off2, len2 = packed
    parts = []
    for lo in range(0, len(off1), 1023):
        sl = slice(lo, lo + 1023)
        res, kind, _ = _plan(gx, (blob, off1[sl], len1[sl], off2[sl], len2[sl]), scores, is_local)
        assert kind == 0
        parts.append(res)
    return np.concatenate(parts)


_FIELDS = ("score", "start_i", "start_j", "end_i", "end_j", "n_ops", "matches", "mismatches", "gap_extensions",
           "opening_gaps", "lcs_at_first_max")


def _same_results(got, wave, what):
    for f in _FIELDS:
        bad = np.nonzero(got[f] != wave[f])[0]
        assert bad.size == 0, (what, f, bad[:5], got[f][bad[:5]], wave[f][bad[:5]])


def _same_oracle(score, si, sj, exp, what):
    es, ei, ej = exp
    for name, g, e in (("score", score, es), ("start_i", si, ei), ("start_j", sj, ej)):
        g = np.asarray(g).astype(np.int64)
        bad = np.nonzero(g != e.astype(np.int64))[0]
        assert bad.size == 0, (what, name, bad[:5], g[bad[:5]], e[bad[:5]])


def _both_kernels(monkeypatch):
    """runs the loop body with the default read kernel (yields False), then with GX_READS32 set (yields True)"""
    for force32 in (False, True):
        if force32:
            monkeypatch.setenv("GX_READS32", "1")
        else:
            monkeypatch.delenv("GX_READS32", raising=False)
        yield force32
    monkeypatch.delenv("GX_READS32", raising=False)


# ================================================================================================ every G x K class
@gpu
@pytest.mark.parametrize("max_len", [152, 153, 320, 321, 640])
def test_read_plan_start_cells_every_class(gx, oracle, max_len, monkeypatch):
    """1024-pair local start-cell plans in every G x K class, both kernels, at CONFIG_TOML, TEST_CONFIG and on both
    sides of each s16x2 limit: the read kernel runs (stat 9), in the expected lane width (stat 26), and matches the
    oracle and the wavefront path's whole gx_result"""
    packed = gx.pack_pairs(_read_set(max_len + 17, 1024, max_len))
    cases = [(CONFIG_TOML, 16), (TEST_CONFIG, 16)] + _reads16_edges(max_len)
    for scores, bits in cases:
        exp = oracle_cells(oracle, *packed, scores, True)
        wave = None
        for force32 in _both_kernels(monkeypatch):
            res, kind, used = _plan(gx, packed, scores)
            assert (kind, used) == (1, 32 if force32 else bits), (max_len, scores, force32)
            what = (max_len, scores, force32)
            _same_oracle(res["score"], res["start_i"], res["start_j"], exp, what)
            assert np.array_equal(res["end_i"], res["start_i"]) and np.array_equal(res["end_j"], res["start_j"])
            if wave is None:
                wave = _wavefront(gx, packed, scores)
            _same_results(res, wave, what)


# ================================================================================================ ties by construction
def _junk(rng, n, alphabet):
    return rng.choice(np.frombuffer(alphabet, np.uint8), size=n)


def _tie_pairs(rng, max_len):
    """[(name, s1, s2)] whose maxima tie in the places the kernels must tell apart, none longer than max_len.  Junk
    uses letters the other sequence never has, so that the only positive cells come from the planted copies."""
    x10, x5, y30 = (_junk(rng, k, b"ACGT") for k in (10, 5, 30))
    x = _junk(rng, max_len // 3, b"ACGT")
    s = []
    # two rows of one lane: s2 = X fits lane 0 (K >= 19), s1 = X junk X
    s.append(("rows_one_lane", np.concatenate([x10, _junk(rng, 7, b"W"), x10]), x10))
    # two columns of one lane's row: s2 = X junk X, 14 columns
    s.append(("cols_one_lane", x5, np.concatenate([x5, _junk(rng, 4, b"W"), x5])))
    # neighbouring lanes of one group: the second copy ends in lane 1
    s.append(("cols_two_lanes", x10, np.concatenate([x10, _junk(rng, 6, b"W"), x10])))
    # x vs x junk x, and transposed, as long as the batch allows
    xjx = np.concatenate([x, _junk(rng, x.size, b"W"), x])
    s.append(("x_vs_xjx", x, xjx))
    s.append(("xjx_vs_x", xjx, x))
    # maximum in the last row and the last column: n at, and one past, lane and group boundaries (K = 19, 20;
    # G * K = 152, 320)
    for n in (19, 20, 21, 41, 152, 153, 320, 321, 640):
        if n <= max_len:
            y = y30[:min(30, n - 1)]
            s.append((f"last_cell_n{n}", np.concatenate([_junk(rng, min(100, max_len - y.size), b"W"), y]),
                      np.concatenate([_junk(rng, n - y.size, b"S"), y])))
    # all-zero tables -> (m, n)
    s.append(("all_zero", np.full(max_len, ord("A"), np.uint8), np.full(max_len - 3, ord("C"), np.uint8)))
    s.append(("all_zero_short", np.full(1, ord("A"), np.uint8), np.full(7, ord("C"), np.uint8)))
    # empty and single-base pairs
    e = np.zeros(0, np.uint8)
    for name, a, b in (("m0", e, x10), ("n0", x10, e), ("m0n0", e, e), ("1x1_match", x5[:1], x5[:1]),
                       ("1x1_mismatch", np.array([ord("A")], np.uint8), np.array([ord("C")], np.uint8)),
                       ("1xn", x5[:1], x), ("mx1", x, x5[:1])):
        s.append((name, a, b))
    return s


def _dual_pairs(rng, max_len):
    """pairs for the two halves of one s16x2 register (indices 2d, 2d+1): the short one (m = 20) takes its maximum
    early, the long one in rows the short one only sees as padding; both ways round"""
    z = _junk(rng, 40, b"ACGT")
    short = (z[:20].copy(), z.copy())
    lng = (np.concatenate([_junk(rng, max_len - 40, b"W"), z]), z.copy())
    return [("dual_short_first", *short), ("dual_long_second", *lng), ("dual_long_first", *lng),
            ("dual_short_second", *short)]


def _tie_batch(seed, max_len):
    rng = np.random.default_rng(seed)
    named = _dual_pairs(rng, max_len) + _tie_pairs(rng, max_len)   # the dual pairs first: they start at even indices
    pairs = [(a, b) for _, a, b in named]
    assert max(max(len(a), len(b)) for a, b in pairs) == max_len
    while len(pairs) < 1024:
        m, n = (int(v) for v in rng.integers(0, max_len + 1, size=2))
        pairs.append(random_pair(rng, m, n, similar=bool(len(pairs) % 2), sub=0.06, indel=0.01))
    return [n for n, _, _ in named], pairs


@gpu
@pytest.mark.parametrize("max_len", [152, 153, 320, 321, 640])
def test_read_plan_start_cell_ties(gx, oracle, max_len, monkeypatch):
    """ties placed by construction -- rows and columns of one lane, neighbouring lanes, x vs x.junk.x both ways, the
    last row and column, the two halves of one s16x2 register with different m, all-zero, empty and single-base
    tables -- in every G x K class, through both kernels, against the oracle and the wavefront path"""
    names, pairs = _tie_batch(11 + max_len, max_len)
    packed = gx.pack_pairs(pairs)
    for scores in (CONFIG_TOML, TEST_CONFIG):
        exp = oracle_cells(oracle, *packed, scores, True)
        # the constructions do what they claim: the later copy wins, the all-zero and empty tables take (m, n)
        for q, name in enumerate(names):
            m, n = len(pairs[q][0]), len(pairs[q][1])
            cell = (int(exp[1][q]), int(exp[2][q]))
            if name in ("rows_one_lane", "xjx_vs_x") or name.startswith(("last_cell", "dual_long")):
                assert cell[0] == m, (name, cell)
            if name in ("cols_one_lane", "cols_two_lanes", "x_vs_xjx") or name.startswith("last_cell"):
                assert cell[1] == n, (name, cell)
            if name.startswith(("all_zero", "m0", "n0")) or name == "1x1_mismatch":
                assert exp[0][q] == 0 and cell == (m, n), (name, cell)
        wave = _wavefront(gx, packed, scores)
        for force32 in _both_kernels(monkeypatch):
            res, kind, used = _plan(gx, packed, scores)
            assert (kind, used) == (1, 32 if force32 else 16)
            _same_oracle(res["score"], res["start_i"], res["start_j"], exp, (scores, force32))
            _same_results(res, wave, (scores, force32))
            got, si, sj = gx.score_batch(*packed, scores, True, start_cells=True)
            _same_oracle(got, si, sj, exp, ("score_batch", scores, force32))


# ================================================================================================ key range
@gpu
def test_read_plan_start_cell_key_range(gx, oracle):
    """V just under 2^26, so the 32-bit kernel's key (V << 5) | k sits just under 2^31: 1024 identical 150 bp pairs at
    the largest local match score the contract accepts; the next one is refused by every start-cell entry point"""
    rng = np.random.default_rng(3)
    x = _ACGT[rng.integers(0, 4, size=150)]
    pairs = [(x, x)] * 1024
    packed = gx.pack_pairs(pairs)
    a = max_local_a(150, 150)
    scores = (a, -1, -1, -1)
    assert (150 * a) << 5 | 31 < 1 << 31 and (150 * a) >= (1 << 26) - 150
    res, kind, used = _plan(gx, packed, scores)
    assert (kind, used) == (1, 32)
    exp = oracle_cells(oracle, *packed, scores, True)
    assert int(exp[0][0]) == 150 * a and (int(exp[1][0]), int(exp[2][0])) == (150, 150)
    _same_oracle(res["score"], res["start_i"], res["start_j"], exp, "key range")
    got, si, sj = gx.score_batch(*packed, scores, True, start_cells=True)
    _same_oracle(got, si, sj, exp, "key range, score_batch")
    past = (a + 1, -1, -1, -1)
    assert _status(lambda: gx.Plan(packed[2], packed[4], past, True, traceback=False, start_cell=True).close()) == 3
    assert _status(lambda: gx.score_batch(*packed, past, True, start_cells=True)) == 3
    assert _status(lambda: gx.align_batch(pairs, past, True, traceback=False, start_cell=True)) == 3


# ================================================================================================ streamed path
@gpu
def test_score_batch_cells_streamed(gx, oracle, monkeypatch):
    """>= 2^18 + an odd number of ragged pairs (chunk-boundary layout): local at CONFIG_TOML and at the s16x2 vmax
    limit with both kernels; global -> (m, n) with gx_score_batch's scores"""
    blob, off1, len1, off2, len2 = packed = _stream_set()
    a = 8000 // 61 + 1
    for scores in (CONFIG_TOML, (a, -1, -1, -(15999 - 61 * a - 1))):
        exp = oracle_cells(oracle, *packed, scores, True)
        for force32 in _both_kernels(monkeypatch):
            got, si, sj = gx.score_batch(*packed, scores, True, start_cells=True)
            _same_oracle(got, si, sj, exp, (scores, force32))
            assert np.array_equal(got, gx.score_batch(*packed, scores, True)), (scores, force32)
    for scores in (CONFIG_TOML, TEST_CONFIG):
        got, si, sj = gx.score_batch(*packed, scores, False, start_cells=True)
        assert np.array_equal(got, gx.score_batch(*packed, scores, False)), scores
        assert np.array_equal(si, len1) and np.array_equal(sj, len2), scores
        assert np.array_equal(got, oracle.score_batch(*packed, scores, False, n_threads=os.cpu_count() or 1)), scores


def _with_long_pair(packed, m=700, n=650):
    blob, off1, len1, off2, len2 = packed
    rng = np.random.default_rng(9)
    a, b = random_pair(rng, m, n)
    blob2 = np.concatenate([blob, a, b])
    return (blob2, np.append(off1, np.uint64(blob.size)), np.append(len1, np.uint64(m)),
            np.append(off2, np.uint64(blob.size + m)), np.append(len2, np.uint64(n)))


@gpu
def test_score_batch_cells_fallbacks(gx, oracle):
    """what the streamed path declines goes through a start-cell plan, in the same call: < 1024 pairs (wavefront),
    2^18 pairs with one pair > 640 bp, and a local s_mismatch >= 0 batch"""
    stream = _stream_set()
    small = tuple(x[:1000] if i else x for i, x in enumerate(stream))
    for packed, scores, what in ((small, CONFIG_TOML, "< 1024 pairs"), (_with_long_pair(stream), CONFIG_TOML, "> 640 bp"),
                                 (stream, (1, 0, -1, -5), "s_mismatch >= 0")):
        exp = oracle_cells(oracle, *packed, scores, True)
        got, si, sj = gx.score_batch(*packed, scores, True, start_cells=True)
        _same_oracle(got, si, sj, exp, what)
        got, si, sj = gx.score_batch(*packed, scores, False, start_cells=True)
        assert np.array_equal(si, packed[2]) and np.array_equal(sj, packed[4]), what
        assert np.array_equal(got, oracle.score_batch(*packed, scores, False, n_threads=os.cpu_count() or 1)), what


# ================================================================================================ config 4
@gpu
def test_score_batch_cells_config4_parity(gx, oracle):
    """the first 100 000 pairs of the config-4 parity set: scores equal the frozen fixture, start cells the oracle"""
    from genomics_rs_b200 import workloads as wl
    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "config4_scores.npz"))
    packed = wl.reads150(0, wl.CONFIG4_PARITY_PAIRS, parity_set=True)
    got, si, sj = gx.score_batch(*packed, CONFIG_TOML, True, start_cells=True)
    assert np.array_equal(got, gold["parity"].astype(np.int64))
    exp = oracle_cells(oracle, *packed, CONFIG_TOML, True)
    _same_oracle(got, si, sj, exp, "config4 parity")


# ================================================================================================ refusals
@gpu
def test_score_batch_cells_refusals(gx):
    """the same status as gx_score_batch for bad scores, out-of-range lengths and bad offsets, on both routes; null
    start-cell outputs are GX_ERR_ARG"""
    from genomics_rs_b200 import _lib
    plan_set = gx.pack_pairs(_read_set(7, 1024, 150))
    for packed in (plan_set, _stream_set()):
        blob, off1, len1, off2, len2 = packed
        bad_off = off1.copy()
        bad_off[-1] = blob.size
        la = max_local_a(READS_MAX_LEN, READS_MAX_LEN) if len(off1) >= 1 << 18 else max_local_a(150, 150)
        cases = [(packed, (1, -1, -1, 1), True), (packed, (1, -1, 0, 0), False), (packed, (la + 1, -1, -1, -1), True),
                 ((blob, bad_off, len1, off2, len2), CONFIG_TOML, True)]
        for args, scores, is_local in cases:
            want = _status(lambda: gx.score_batch(*args, scores, is_local))
            assert want != 0, scores
            assert _status(lambda: gx.score_batch(*args, scores, is_local, start_cells=True)) == want, (scores, is_local)
    lib = _lib.load()
    blob, off1, len1, off2, len2 = plan_set
    out = np.zeros(len(off1), np.int64)
    cells = np.zeros(len(off1), np.uint64)
    for si, sj in ((None, cells.ctypes.data), (cells.ctypes.data, None)):
        rc = lib.gx_score_batch_cells(blob.ctypes.data, blob.size, off1.ctypes.data, len1.ctypes.data, off2.ctypes.data,
                                      len2.ctypes.data, len(off1), _lib.GxScores(*CONFIG_TOML), 1, out.ctypes.data, si, sj)
        assert rc == 1
    rc = lib.gx_score_batch_cells(None, 0, None, None, None, None, 0, _lib.GxScores(*CONFIG_TOML), 1, None, None, None)
    assert rc == 0


# ================================================================================================ CPU: the reference
def test_oracle_cells_match_faithful(oracle):
    """the start-cell reference of these tests (score_linear per pair, over threads) against the faithful restatement
    of alignment_table + retrace, on small random pairs with ties and empty tables"""
    rng = np.random.default_rng(21)
    pairs = []
    for q in range(300):
        m, n = int(rng.integers(0, 40)), int(rng.integers(0, 40))
        alphabet = b"AC" if q % 3 == 0 else b"ACGT"
        pairs.append(random_pair(rng, m, n, alphabet=alphabet, similar=bool(q % 2)))
    pairs += [(np.full(9, ord("A"), np.uint8), np.full(4, ord("C"), np.uint8))]
    from genomics_rs_b200.alignment import pack_pairs
    packed = pack_pairs(pairs)
    for scores in (CONFIG_TOML, TEST_CONFIG, (2, -1, -1, -3)):
        sc, si, sj = oracle_cells(oracle, *packed, scores, True)
        for q, (a, b) in enumerate(pairs):
            f = oracle.align_faithful(a, b, scores, True)
            assert (int(sc[q]), int(si[q]), int(sj[q])) == (f.score, *f.start), (q, scores)
        assert (int(si[-1]), int(sj[-1])) == (9, 4)
