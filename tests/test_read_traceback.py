"""Traceback for short-read sets: gx_align_reads (genomics_rs_b200.align_reads).

Every GPU case compares the whole gx_result (without the timing fields) and the op bytes with gx_align_batch and
GX_FLAG_TRACEBACK on the same pairs (the wavefront path), and with the oracle (align_linear; align_faithful on the small
cases).  The read kernel's classes are (G, K) = (8, 19), (16, 20), (32, 20): pairs up to 152, 320 and 640 bp."""
import os

import numpy as np
import pytest

from conftest import CONFIG_TOML, TEST_CONFIG, random_pair
from test_read_start_cells import _tie_batch
from test_score_range import READS_MAX_LEN, _stream_set, max_h, max_local_a, max_mx

gpu = pytest.mark.gpu
LARGE_GAPS = (2, -3, -40, -300)
GLOBAL_NONNEG = (3, 1, -2, -4)          # s_mismatch >= 0: global only
_FIELDS = ("score", "start_i", "start_j", "end_i", "end_j", "n_ops", "matches", "mismatches", "gap_extensions",
           "opening_gaps", "lcs_at_first_max")


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


def _packed_ops_off(len1, len2, slack=None):
    caps = np.asarray(len1, np.uint64) + np.asarray(len2, np.uint64) + np.uint64(1)
    if slack is not None:
        caps = caps + np.asarray(slack, np.uint64)
    ops_off = np.zeros(caps.size + 1, np.uint64)
    np.cumsum(caps, out=ops_off[1:])
    return ops_off


def _wavefront(packed, scores, is_local, ops_off):
    """gx_align_batch with GX_FLAG_TRACEBACK on the same pairs and the same ops_off -> (results, ops)"""
    from genomics_rs_b200 import _lib
    from genomics_rs_b200.alignment import RESULT_DTYPE, _scores_struct
    blob, off1, len1, off2, len2 = [np.ascontiguousarray(x) for x in packed]
    n = len(off1)
    res = np.zeros(n, RESULT_DTYPE)
    ops = np.zeros(max(int(ops_off[-1]), 1), np.uint8)
    lib = _lib.load()
    _lib.check(lib.gx_align_batch(blob.ctypes.data if blob.size else None, blob.size, off1.ctypes.data, len1.ctypes.data,
                                  off2.ctypes.data, len2.ctypes.data, n, _scores_struct(scores), int(is_local),
                                  _lib.GX_FLAG_TRACEBACK, res.ctypes.data, ops.ctypes.data, ops_off.ctypes.data))
    return res, ops


def _same_results(got, gops, exp, eops, ops_off, what, idx=None):
    idx = np.arange(len(got)) if idx is None else idx
    for f in _FIELDS:
        bad = np.nonzero(got[f][idx] != exp[f][idx])[0]
        assert bad.size == 0, (what, f, idx[bad[:5]], got[f][idx[bad[:5]]], exp[f][idx[bad[:5]]])
    for q in idx:
        o, k = int(ops_off[q]), int(got["n_ops"][q])
        assert np.array_equal(gops[o:o + k], eops[o:o + k]), (what, "ops", int(q))


def _same_oracle(oracle, got, gops, ops_off, pairs, scores, is_local, what, faithful=False):
    for q, (a, b) in enumerate(pairs):
        e = (oracle.align_faithful if faithful else oracle.align_linear)(a, b, scores, is_local)
        r = got[q]
        o, k = int(ops_off[q]), int(r["n_ops"])
        have = (int(r["score"]), (int(r["start_i"]), int(r["start_j"])), (int(r["end_i"]), int(r["end_j"])),
                int(r["matches"]), int(r["mismatches"]), int(r["gap_extensions"]), int(r["opening_gaps"]))
        want = (e.score, tuple(e.start), tuple(e.end), e.matches, e.mismatches, e.gap_extensions, e.opening_gaps)
        assert have == want, (what, q, len(a), len(b), have, want)
        assert k == e.ops.size and np.array_equal(gops[o:o + k], e.ops), (what, q)


def _check(gx, oracle, pairs, scores, is_local, what, faithful=False, ops_off=None):
    packed = gx.pack_pairs(pairs)
    if ops_off is None:
        ops_off = _packed_ops_off(packed[2], packed[4])
    got, gops, _ = gx.align_reads(*packed, scores, is_local, ops_off=ops_off)
    assert np.all(got["walk_ms"] == 0.0) and np.all(got["fill_ms"] == got["fill_ms"][0]) and got["fill_ms"][0] > 0.0
    exp, eops = _wavefront(packed, scores, is_local, ops_off)
    _same_results(got, gops, exp, eops, ops_off, what)
    _same_oracle(oracle, got, gops, ops_off, pairs, scores, is_local, what, faithful)
    return got


# ================================================================================================ every (G, K) class
def _class_pairs(rng, max_len, n_pairs):
    """lengths at and one past K, at G * K and at the class limit, m != n both ways, then random similar and dissimilar
    pairs up to max_len"""
    marks = sorted({v for v in (1, 18, 19, 20, 21, 40, 41, 151, 152, 153, 319, 320, 321, 639, 640) if v <= max_len})
    dims = [(max_len, max_len), (max_len, max_len - 1), (max_len - 1, max_len)]
    dims += [(v, w) for v in marks for w in (v, v + 1, v - 1) if 0 <= w <= max_len]
    pairs = [random_pair(rng, m, n, similar=bool(k % 2), sub=0.08, indel=0.03) for k, (m, n) in enumerate(dims)]
    while len(pairs) < n_pairs:
        m, n = (int(v) for v in rng.integers(0, max_len + 1, size=2))
        pairs.append(random_pair(rng, m, n, similar=bool(len(pairs) % 2), sub=0.08, indel=0.03))
    return pairs


@gpu
@pytest.mark.parametrize("max_len", [19, 20, 152, 153, 320, 321, 640])
def test_every_class(gx, oracle, max_len):
    """each class and its edges, global and local, at CONFIG_TOML, TEST_CONFIG and a large-gap scoring, plus a global
    scoring with s_mismatch >= 0"""
    pairs = _class_pairs(np.random.default_rng(100 + max_len), max_len, 192 if max_len > 320 else 256)
    assert max(max(len(a), len(b)) for a, b in pairs) == max_len
    cases = [(s, loc) for s in (CONFIG_TOML, TEST_CONFIG, LARGE_GAPS) for loc in (False, True)] + [(GLOBAL_NONNEG, False)]
    for scores, is_local in cases:
        _check(gx, oracle, pairs, scores, is_local, (max_len, scores, is_local))


# ================================================================================================ local ties and walk paths
def _walk_pairs(rng):
    """run-on local tails through zero cells that end on column 0 and on row 0, labels at i = m / j = n, byte values 0
    and 255, empty and single-base pairs"""
    x = rng.choice(np.frombuffer(b"ACGT", np.uint8), size=40)
    w, s = np.full(30, ord("W"), np.uint8), np.full(10, ord("S"), np.uint8)
    e = np.zeros(0, np.uint8)
    b01 = np.frombuffer(bytes([0, 255]), np.uint8)
    return [
        ("tail_col0", np.concatenate([w, x]), np.concatenate([s, x])),   # zero cells along row 30 to column 0
        ("tail_row0", x, np.concatenate([s, x])),                        # the diagonal reaches row 0
        ("tail_mid", np.concatenate([w, x, w]), np.concatenate([s, x, s])),
        ("last_differs", np.frombuffer(b"ACGTA", np.uint8), np.frombuffer(b"ACGTC", np.uint8)),
        ("bytes_0_255", rng.choice(b01, size=50), rng.choice(b01, size=47)),
        ("bytes_0_255_same", np.tile(b01, 20), np.tile(b01, 20)),
        ("m0", e, x[:7]), ("n0", x[:7], e), ("m0n0", e, e),
        ("1x1_match", x[:1], x[:1]), ("1x1_mismatch", np.array([0], np.uint8), np.array([255], np.uint8)),
        ("1xn", x[:1], x), ("mx1", x, x[:1]), ("0x1", e, x[:1]), ("1x0", x[:1], e),
    ]


@gpu
@pytest.mark.parametrize("max_len", [152, 153, 320, 321, 640])
def test_local_ties_and_walk_paths(gx, oracle, max_len):
    """the start-cell tie constructions (lanes, groups, padded cells, x vs x.junk.x, all-zero tables that walk along
    row m) and the walk constructions above, through the whole walk, local and global"""
    names, pairs = _tie_batch(11 + max_len, max_len)
    extra = _walk_pairs(np.random.default_rng(max_len))
    pairs = [(a, b) for _, a, b in extra] + pairs
    for scores in (CONFIG_TOML, TEST_CONFIG):
        for is_local in (True, False):
            got = _check(gx, oracle, pairs, scores, is_local, (max_len, scores, is_local))
            # the small constructions against the faithful restatement too
            _check(gx, oracle, pairs[:len(extra)], scores, is_local, ("faithful", max_len, scores, is_local), faithful=True)
            if is_local:
                # the constructions do what they claim: an all-zero table walks row m from (m, n) to column 0; the
                # tails end on column 0 (after zero cells of row 30) and on row 0 (the diagonal from (1, 11))
                q = len(extra) + names.index("all_zero")
                m, n = len(pairs[q][0]), len(pairs[q][1])
                r = got[q]
                assert (int(r["start_i"]), int(r["start_j"]), int(r["end_i"]), int(r["end_j"])) == (m, n, m, 1)
                assert int(r["n_ops"]) == n and int(r["opening_gaps"]) == 1
                extra_names = [nm for nm, _, _ in extra]
                r = got[extra_names.index("tail_col0")]
                assert (int(r["end_i"]), int(r["end_j"])) == (30, 1) and int(r["score"]) > 0
                r = got[extra_names.index("tail_row0")]
                assert (int(r["end_i"]), int(r["end_j"])) == (1, 11) and int(r["score"]) > 0


# ================================================================================================ int32 score contract
@gpu
def test_score_contract_edges(gx, oracle):
    """640 bp pairs at the edges of the contract the streamed read path checks (640 x 640): the last scorings inside
    agree with the wavefront path and the oracle, the first ones past are refused"""
    rng = np.random.default_rng(640)
    pairs = [random_pair(rng, 640, 640, similar=bool(q % 2), sub=0.05, indel=0.01) for q in range(48)]
    pairs += [random_pair(rng, 640, int(n), sub=0.05, indel=0.01) for n in rng.integers(600, 641, size=16)]
    mx = max_mx(READS_MAX_LEN, READS_MAX_LEN, -1)
    hm = max_h(READS_MAX_LEN, READS_MAX_LEN, 1)
    la = max_local_a(READS_MAX_LEN, READS_MAX_LEN)
    inside = [((mx, -mx, -mx, -1), False), ((1, -1, -1, -hm), False), ((la, -1, -1, -1), True)]
    past = [((mx + 1, -mx, -mx, -1), False), ((1, -1, -1, -hm - 1), False), ((la + 1, -1, -1, -1), True)]
    for scores, is_local in inside:
        _check(gx, oracle, pairs, scores, is_local, ("inside", scores, is_local))
    packed = gx.pack_pairs(pairs)
    for scores, is_local in past:
        assert _status(lambda: gx.align_reads(*packed, scores, is_local)) == 3, scores
    # the streamed read path checks every batch as if its pairs were 640 bp long: short pairs are refused alike
    short = gx.pack_pairs([(a[:60], b[:60]) for a, b in pairs[:4]])
    assert _status(lambda: gx.align_reads(*short, (la + 1, -1, -1, -1), True)) == 3


# ================================================================================================ streaming
@gpu
def test_streamed_chunks(gx):
    """2^18 + 4099 pairs: two chunks on different lanes, a ragged last one, and an ops_off with slack between pairs.
    Every score and start cell equals gx_score_batch_cells, a seeded sample of full results gx_align_batch's; the slack
    bytes stay untouched"""
    packed = _stream_set()
    blob, off1, len1, off2, len2 = packed
    n = len(off1)
    slack = (np.arange(n) % 5).astype(np.uint64)
    ops_off = _packed_ops_off(len1, len2, slack)
    for scores, is_local in ((CONFIG_TOML, True), (CONFIG_TOML, False), (TEST_CONFIG, True)):
        ops = np.full(int(ops_off[-1]), 0xEE, np.uint8)
        got, gops, _ = gx.align_reads(*packed, scores, is_local, ops=ops, ops_off=ops_off)
        sc, si, sj = gx.score_batch(*packed, scores, is_local, start_cells=True)
        assert np.array_equal(got["score"], sc), (scores, is_local)
        assert np.array_equal(got["start_i"], si) and np.array_equal(got["start_j"], sj), (scores, is_local)
        nops = got["n_ops"]
        assert np.all(nops <= len1 + len2 + np.uint64(1))
        assert np.array_equal(nops, got["matches"] + got["mismatches"] + got["gap_extensions"] + got["opening_gaps"])
        # bytes past each pair's ops are the sentinel
        used = np.zeros(gops.size, bool)
        starts = ops_off[:-1].astype(np.int64)
        cnt = nops.astype(np.int64)
        used[np.repeat(starts, cnt) + (np.arange(int(cnt.sum())) - np.repeat(np.cumsum(cnt) - cnt, cnt))] = True
        assert np.all(gops[~used] == 0xEE), (scores, is_local)
        assert np.all(gops[used] <= 5), (scores, is_local)
        rng = np.random.default_rng(7)
        idx = np.unique(np.concatenate([rng.choice(n, size=3000, replace=False),
                                        np.arange((1 << 18) - 8, (1 << 18) + 8), np.arange(n - 8, n)]))
        sub = tuple(x[idx] if i else x for i, x in enumerate(packed))
        sub_off = _packed_ops_off(sub[2], sub[4])
        exp, eops = _wavefront(sub, scores, is_local, sub_off)
        for f in _FIELDS:
            assert np.array_equal(got[f][idx], exp[f]), (scores, is_local, f)
        for k, q in enumerate(idx):
            o, c = int(ops_off[q]), int(nops[q])
            assert np.array_equal(gops[o:o + c], eops[int(sub_off[k]):int(sub_off[k]) + c]), (scores, is_local, int(q))


# ================================================================================================ config 4
@gpu
def test_config4_parity(gx):
    """the frozen config-4 parity set (100 000 local 150 bp pairs): every score equals the frozen one, and every n_ops
    matches its counters"""
    from genomics_rs_b200 import workloads as wl
    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "config4_scores.npz"))
    packed = wl.reads150(0, wl.CONFIG4_PARITY_PAIRS, parity_set=True)
    got, gops, ops_off = gx.align_reads(*packed, CONFIG_TOML, True)
    assert np.array_equal(got["score"], gold["parity"].astype(np.int64))
    assert np.array_equal(got["n_ops"], got["matches"] + got["mismatches"] + got["gap_extensions"] + got["opening_gaps"])
    idx = np.arange(0, len(got), 97)
    sub = tuple(x[idx] if i else x for i, x in enumerate(packed))
    sub_off = _packed_ops_off(sub[2], sub[4])
    exp, eops = _wavefront(sub, CONFIG_TOML, True, sub_off)
    for f in _FIELDS:
        assert np.array_equal(got[f][idx], exp[f]), f


# ================================================================================================ status codes
@gpu
def test_status_codes(gx):
    """each status of gx_align_reads for its case; an empty batch is GX_OK"""
    from genomics_rs_b200 import _lib
    from genomics_rs_b200.alignment import RESULT_DTYPE
    rng = np.random.default_rng(4)
    pairs = [random_pair(rng, 150, 150) for _ in range(64)]
    blob, off1, len1, off2, len2 = packed = gx.pack_pairs(pairs)
    assert _status(lambda: gx.align_reads(*packed, CONFIG_TOML, True)) == 0
    # GX_ERR_UNSUPPORTED: a pair longer than 640 bp, local with s_mismatch >= 0, a scattered chunk
    long = gx.pack_pairs(pairs[:3] + [random_pair(rng, 641, 20)])
    assert _status(lambda: gx.align_reads(*long, CONFIG_TOML, False)) == 9
    assert _status(lambda: gx.align_reads(*packed, (1, 0, -1, -5), True)) == 9
    assert _status(lambda: gx.align_reads(*packed, (1, 0, -1, -5), False)) == 0
    far = np.zeros(1 << 22, np.uint8)
    far[:150], far[-150:] = pairs[0][0], pairs[0][1]
    scattered = (far, np.array([0], np.uint64), np.array([150], np.uint64), np.array([far.size - 150], np.uint64),
                 np.array([150], np.uint64))
    assert _status(lambda: gx.align_reads(*scattered, CONFIG_TOML, True)) == 9
    # GX_ERR_OPS_CAP: one gap one byte short; a decreasing ops_off
    short_off = _packed_ops_off(len1, len2)
    short_off[5:] -= np.uint64(1)
    assert _status(lambda: gx.align_reads(*packed, CONFIG_TOML, True, ops_off=short_off)) == 4
    down = _packed_ops_off(len1, len2)
    down[10] = down[12]
    assert _status(lambda: gx.align_reads(*packed, CONFIG_TOML, True, ops_off=down)) == 4
    # GX_ERR_ARG: a sequence past the blob's end, null pointers
    bad = off2.copy()
    bad[-1] = blob.size
    assert _status(lambda: gx.align_reads(blob, off1, len1, bad, len2, CONFIG_TOML, True)) == 1
    lib = _lib.load()
    res = np.zeros(len(off1), RESULT_DTYPE)
    ops_off = _packed_ops_off(len1, len2)
    ops = np.zeros(int(ops_off[-1]), np.uint8)
    args = [blob.ctypes.data, blob.size, off1.ctypes.data, len1.ctypes.data, off2.ctypes.data, len2.ctypes.data, len(off1),
            _lib.GxScores(*CONFIG_TOML), 1, res.ctypes.data, ops.ctypes.data, ops_off.ctypes.data]
    assert lib.gx_align_reads(*args) == 0
    for k in (0, 2, 9, 10, 11):
        a = list(args)
        a[k] = None
        assert lib.gx_align_reads(*a) == 1, k
    # GX_ERR_SCORES / GX_ERR_RANGE
    assert _status(lambda: gx.align_reads(*packed, (1, -1, -1, 1), True)) == 2
    assert _status(lambda: gx.align_reads(*packed, (1, -1, 0, 0), False)) == 2
    la = max_local_a(READS_MAX_LEN, READS_MAX_LEN)
    assert _status(lambda: gx.align_reads(*packed, (la + 1, -1, -1, -1), True)) == 3
    # empty batch
    e = np.zeros(0, np.uint64)
    assert lib.gx_align_reads(None, 0, None, None, None, None, 0, _lib.GxScores(*CONFIG_TOML), 1, None, None, None) == 0
    res0, ops0, off0 = gx.align_reads(np.zeros(0, np.uint8), e, e, e, e, CONFIG_TOML, True)
    assert res0.size == 0 and off0.tolist() == [0]


# ================================================================================================ CPU
def test_default_ops_off_layout():
    """the wrapper's default ops_off is gx_align_batch's: prefix sums of len1 + len2 + 1"""
    off = _packed_ops_off([3, 0, 5], [2, 0, 0])
    assert off.tolist() == [0, 6, 7, 13]
    assert _packed_ops_off([1], [1], [4]).tolist() == [0, 7]
