"""Every kernel at the edges of the int32 score contract (gx_check_scores, include/gxalign.h):

    h <= 0, g < 0, h+g < 0;   (m+n+2)·max(|a|,|b|,|g|) + |h| < 2^29;   local: min(m,n)·max(a,0) < 2^26

Inside those bounds results must be bit-identical to the int64 oracle; the int32 layouts of the kernels (colbuf words,
the NEG32 sentinel, start-cell and first-maximum keys, the IDP.4A byte profile, the s16x2 read kernel) are all sized
against them.  The extreme scorings are derived from the contract's formulas below, so the tests follow the contract if
it changes.  Plan statistics (gx_plan_stat) say which path ran, so that each edge scoring is checked to land on the side
it claims.  The boundary arithmetic itself is checked without a GPU."""
import functools

import numpy as np
import pytest

from conftest import KR_COMBOS, force_kr, random_pair

gpu = pytest.mark.gpu

# ---- the contract, restated (check_scores_impl and the LCS-pass check in csrc/gx_api.cu)
CELL_LIM = 1 << 29     # (m+n+2)·max(|a|,|b|,|g|) + |h| < CELL_LIM
LOCAL_LIM = 1 << 26    # local: min(m,n)·max(a,0) < LOCAL_LIM
LCS_LIM = 1 << 26      # GX_FLAG_LCS_AT_MAX: (2·max_len+2)·max(|a|,|b|,|g|) + |h| < LCS_LIM
READS_MAX_LEN = 640    # the streamed read path checks every batch as if its pairs were this long


def max_mx(m, n, h):
    """largest max(|a|,|b|,|g|) the contract accepts for an m x n table and gap open h"""
    return (CELL_LIM - 1 - abs(h)) // (m + n + 2)


def max_h(m, n, mx):
    """largest |h| the contract accepts for an m x n table and max(|a|,|b|,|g|) = mx"""
    return CELL_LIM - 1 - (m + n + 2) * mx


def max_local_a(m, n):
    """largest match score the local bound accepts"""
    return (LOCAL_LIM - 1) // min(m, n)


def max_lcs_mx(max_len, h):
    """largest max(|a|,|b|,|g|) the first-maximum pass of GX_FLAG_LCS_AT_MAX accepts"""
    return (LCS_LIM - 1 - abs(h)) // (2 * max_len + 2)


def widest(pairs):
    """the (m, n) of the pair with the largest m+n: it binds the cell bound of a batch"""
    return max(((len(a), len(b)) for a, b in pairs), key=sum)


def chain1_keys_fit(k, scores):
    """CHAIN1 keys a local start cell as ((V + h+g) << log2 K) | k: with V = 0 that stays above INT32_MIN only while
    -(h+g) < 2^(31 - log2 K)"""
    a, b, g, h = scores
    return -(h + g) < (1 << (31 - (k.bit_length() - 1)))


# ---- comparisons
def _same(gpu, ora, what=""):
    assert gpu.score == ora.score, what
    assert tuple(gpu.start) == tuple(ora.start), what
    assert tuple(gpu.end) == tuple(ora.end), what
    assert (gpu.matches, gpu.mismatches, gpu.gap_extensions, gpu.opening_gaps) == (
        ora.matches, ora.mismatches, ora.gap_extensions, ora.opening_gaps), what
    assert np.array_equal(gpu.ops, ora.ops), what
    oi, oj = gpu.coords()
    assert np.array_equal(oi, ora.ops_i) and np.array_equal(oj, ora.ops_j), what


_ORACLE = {}


def _expect(oracle, a, b, scores, is_local):
    """the oracle's alignment of one pair, once per (pair, scoring, mode) across parametrizations"""
    key = (bytes(np.asarray(a, np.uint8)), bytes(np.asarray(b, np.uint8)), tuple(scores), bool(is_local))
    if key not in _ORACLE:
        small = len(a) * len(b) <= 100 * 100
        _ORACLE[key] = (oracle.align_faithful if small else oracle.align_linear)(a, b, scores, is_local)
    return _ORACLE[key]


def _check(res, pairs, oracle, scores, is_local, traceback, start_cell, what):
    for x, ((a, b), r) in enumerate(zip(pairs, res)):
        o = _expect(oracle, a, b, scores, is_local)
        tag = f"{what} pair {x} m={len(a)} n={len(b)} {scores} local={is_local} tb={traceback} start={start_cell}"
        if traceback:
            _same(r, o, tag)
        else:
            assert r.score == o.score, tag
            if start_cell:
                assert tuple(r.start) == tuple(o.start), tag


@pytest.fixture(scope="module")
def gx():
    import genomics_rs_b200 as gx
    from genomics_rs_b200 import _lib
    _lib.ensure_init()
    return gx


def _run(gx, pairs, scores, is_local, traceback=True, start_cell=False, lcs_at_max=False):
    """one plan through create / upload / execute / fetch -> (results, {stat: value} after the execute)"""
    blob, off1, len1, off2, len2 = gx.pack_pairs(pairs)
    plan = gx.Plan(len1, len2, scores, is_local, traceback=traceback, start_cell=start_cell, lcs_at_max=lcs_at_max)
    try:
        plan.upload(blob, off1, off2)
        plan.execute()
        res, ops, ops_off = plan.fetch()
        stats = {w: plan.stat(w) for w in (9, 15, 17, 21, 23, 24, 25, 26)}
    finally:
        plan.close()
    out = []
    for q, r in enumerate(res):
        k, o = int(r["n_ops"]), int(ops_off[q])
        out.append(gx.AlignedSequences(
            s1=gx.Sequence("s1", ""), s2=gx.Sequence("s2", ""), score=int(r["score"]), matches=int(r["matches"]),
            mismatches=int(r["mismatches"]), gap_extensions=int(r["gap_extensions"]), opening_gaps=int(r["opening_gaps"]),
            ops=ops[o:o + k].copy() if traceback else np.zeros(0, np.uint8),
            start=(int(r["start_i"]), int(r["start_j"])), end=(int(r["end_i"]), int(r["end_j"])),
            matches_at_max=int(r["lcs_at_first_max"]) if lcs_at_max else None))
    return out, stats


def _check_scores(scores, m, n):
    from genomics_rs_b200 import _lib
    return _lib.load().gx_check_scores(_lib.GxScores(*scores), m, n)


def _status(fn):
    """the library status fn() fails with (0 if it succeeds)"""
    from genomics_rs_b200 import _lib
    try:
        fn()
    except _lib.GxError as e:
        return e.status
    return 0


def _set_chain1(monkeypatch, chain1):
    if chain1 is None:
        monkeypatch.delenv("GX_CHAIN1", raising=False)
    else:
        monkeypatch.setenv("GX_CHAIN1", str(chain1))


_LUT = np.frombuffer(b"ACGT", np.uint8)

# local tables whose maximum is 0 (test_gpu_parity.py::test_local_all_zero_table): start (m, n) at every blocking
_ZERO_SHAPES = [(b"A" * 64, b"C"), (b"A" * 4096, b"C"), (b"A" * 8192, b"CC"), (b"A" * 64, b"C" * 3), (b"A" * 128, b"C" * 129),
                (b"A" * 256, b"C" * 513), (b"A" * 32, b"C" * 5), (b"A" * 31, b"C"), (b"A" * 4160, b"C" * 7), (b"AC" * 40, b"GT" * 33)]


# ================================================================================================ (a) local start cell
@functools.lru_cache(maxsize=None)
def _start_cell_pairs():
    rng = np.random.default_rng(2718)
    pairs = [random_pair(rng, 600, 500), random_pair(rng, 3000, 2600, sub=0.1, indel=0.02), random_pair(rng, 4500, 700)]
    pairs += [(np.frombuffer(a, np.uint8), np.frombuffer(b, np.uint8)) for a, b in _ZERO_SHAPES]
    # two equal local maxima (x against either copy of itself): in different panels (4096 rows) of one strip, and --
    # transposed -- in different strips of one row.  The LAST one in row-major order must win (algo.rs:311-322).
    x = _LUT[rng.integers(0, 4, size=300)]
    twice = np.concatenate([x, _LUT[rng.integers(0, 4, size=4300)], x])
    pairs += [(twice, x), (x, twice)]
    return tuple(pairs)


def _start_cell_scorings(pairs):
    m, n = widest(pairs)
    hgs = [-(1 << 27) + 1, -(1 << 27), -(1 << 27) - 1, -(1 << 28) + 1, -(1 << 28), -(1 << 28) - 1,
           -((1 << 28) + 10),        # K=8: keys straddle INT32_MAX, V = 10 lands on the INT32_MIN "no row" sentinel
           -((1 << 27) + 6),         # K=16: the same
           -300_000_001, -(max_h(m, n, 1) + 1)]
    return [(1, -1, -1, hg + 1) for hg in hgs] + [(50, -30, -1, -((1 << 28) + 9))]


@gpu
@pytest.mark.parametrize("chain1", [None, 0, 1])
@pytest.mark.parametrize("k,r", KR_COMBOS)
def test_local_start_cell_large_gaps(gx, oracle, k, r, chain1, monkeypatch):
    """gap penalties up to the contract's limit with a local start cell, with traceback, with the start cell only and
    score only, for every K and recurrence form: a plan whose CHAIN1 keys would not fit int32 runs the classic form"""
    force_kr(monkeypatch, k, r)
    _set_chain1(monkeypatch, chain1)
    pairs = list(_start_cell_pairs())
    wrong_form = []
    for scores in _start_cell_scorings(pairs):
        assert _check_scores(scores, *widest(pairs)) == 0
        for traceback, start_cell in ((True, False), (False, True), (False, False)):
            res, st = _run(gx, pairs, scores, True, traceback=traceback, start_cell=start_cell)
            _check(res, pairs, oracle, scores, True, traceback, start_cell, f"K={k} chain1={chain1}")
            assert st[15] == k
            keyed = traceback or start_cell
            if keyed and not chain1_keys_fit(k, scores):
                want = 0
            else:
                want = st[17] if chain1 is None else chain1
            if st[17] != want:
                wrong_form.append((scores, traceback, start_cell, st[17]))
    assert not wrong_form, wrong_form     # after the results: a wrong result is the more telling failure


@gpu
def test_local_start_cell_default_single_pair(gx, oracle, monkeypatch):
    """one short local pair takes K=8 and CHAIN1 by default: with -(h+g) = 300 000 001 its start-cell keys would wrap"""
    for v in ("GX_K", "GX_R", "GX_CHAIN1", "GX_TICKETS", "GX_RESIDENT"):
        monkeypatch.delenv(v, raising=False)
    rng = np.random.default_rng(31)
    a, b = random_pair(rng, 600, 500)
    for scores in ((1, -1, -1, -300_000_000), (1, -1, -1, -2)):
        o = oracle.align_linear(a, b, scores, True)
        _same(gx.align_batch([(a, b)], scores, True)[0], o, scores)
        res, st = _run(gx, [(a, b)], scores, True, traceback=False, start_cell=True)
        assert res[0].score == o.score and tuple(res[0].start) == tuple(o.start), scores
        assert st[15] == 8 and st[17] == (0 if scores[3] < -2 else 1), (scores, st)


# ================================================================================================ (b) global at the int32 edge
_GLOBAL_DIMS = [(4097, 300), (300, 4200), (8193, 770), (33, 1025), (1, 3000)]


@functools.lru_cache(maxsize=None)
def _global_pairs():
    rng = np.random.default_rng(4099)
    pairs = [random_pair(rng, m, n, similar=(x % 2 == 0)) for x, (m, n) in enumerate(_GLOBAL_DIMS)]
    # 2500 unrelated leading bases: the path runs up to 2500 columns right of the scaled diagonal, out of a 64-column band
    x = _LUT[rng.integers(0, 4, size=9000)]
    pairs.append((x, np.concatenate([_LUT[rng.integers(0, 4, size=2500)], x])))
    return tuple(pairs)


def _global_scorings(m, n):
    mx1, mx0 = max_mx(m, n, -1), max_mx(m, n, 0)
    return [(1, -1, -1, -max_h(m, n, 1)),    # E within m+n of -2^30: the I<<1 colbuf packing and the NEG32 ordering
            (mx1, -mx1, -mx1, -1), (mx0, -mx0, -1, 0)]


@gpu
@pytest.mark.parametrize("sched", ["tickets", "resident"])
@pytest.mark.parametrize("chain1", [0, 1])
@pytest.mark.parametrize("k,r", KR_COMBOS)
def test_global_int32_edge(gx, oracle, k, r, chain1, sched, monkeypatch):
    """global tables at the cell bound, ragged across strip, batch and panel boundaries (the widest pair sets the bound):
    traceback with the default code band, with codes everywhere and with a 64-column band (the fallback fires), and score
    only"""
    force_kr(monkeypatch, k, r)
    _set_chain1(monkeypatch, chain1)
    if sched == "tickets":
        monkeypatch.setenv("GX_TICKETS", "1")
        monkeypatch.delenv("GX_RESIDENT", raising=False)
    else:
        monkeypatch.delenv("GX_TICKETS", raising=False)
        monkeypatch.setenv("GX_RESIDENT", "1")
    pairs = list(_global_pairs())
    for scores in _global_scorings(*widest(pairs)):
        for band in (None, "0", "64", "score"):
            if band in (None, "score"):
                monkeypatch.delenv("GX_CODE_BAND", raising=False)
            else:
                monkeypatch.setenv("GX_CODE_BAND", band)
            traceback = band != "score"
            res, st = _run(gx, pairs, scores, False, traceback=traceback)
            what = f"K={k} chain1={chain1} {sched} band={band}"
            _check(res, pairs, oracle, scores, False, traceback, False, what)
            assert (st[15], st[17], st[21]) == (k, chain1, float(sched == "resident")), (what, st)
            if band == "0":
                assert st[23] == 1.0 and st[24] == 0, (what, st)
            if band == "64":
                assert st[24] >= 1, (what, st)          # a path left the band: the execute was repeated with codes everywhere
    monkeypatch.delenv("GX_CODE_BAND", raising=False)


@functools.lru_cache(maxsize=None)
def _long_pair():
    return random_pair(np.random.default_rng(40000), 2000, 40000, sub=0.1, indel=0.02)


@gpu
@pytest.mark.parametrize("k,r", KR_COMBOS)
def test_banded_at_cell_bound(gx, oracle, k, r, monkeypatch):
    """one 2000 x 40 000 pair at the cell bound through 1..8 column bands on one GPU: the row-0 formula
    h + (col0 + j)·g of the last band runs close to -2^29"""
    force_kr(monkeypatch, k, r)
    a, b = _long_pair()
    mx = max_mx(len(a), len(b), -1)
    for scores in ((mx, -mx, -mx, -1), (1, -1, -1, -max_h(len(a), len(b), 1))):
        key = ("banded", scores)
        if key not in _ORACLE:
            _ORACLE[key] = oracle.score_linear(a, b, scores, False)[0]
        for bands in range(1, 9):
            assert gx.nw_score_banded_local(a, b, scores, bands) == _ORACLE[key], (k, bands, scores)


# ================================================================================================ (c) local value range
@functools.lru_cache(maxsize=None)
def _identical_pairs():
    rng = np.random.default_rng(3000)
    x = _LUT[rng.integers(0, 4, size=3000)]
    y = x.copy()
    idx = rng.choice(3000, size=60, replace=False)
    y[idx] = _LUT[(rng.integers(1, 4, size=60) + np.searchsorted(_LUT, y[idx])) % 4]
    return ((x, x), (x, y))


@gpu
@pytest.mark.parametrize("chain1", [0, 1])
@pytest.mark.parametrize("k,r", KR_COMBOS)
def test_local_value_range(gx, oracle, k, r, chain1, monkeypatch):
    """identical 3000-base sequences with the largest match score the local bound accepts: V reaches just under 2^26
    and the classic K=16 start-cell key about 2^30.  The next match score is refused."""
    force_kr(monkeypatch, k, r)
    _set_chain1(monkeypatch, chain1)
    pairs = list(_identical_pairs())
    a = max_local_a(3000, 3000)
    scores = (a, -a, -a, -1)
    assert 3000 * a < LOCAL_LIM <= 3000 * (a + 1)
    for traceback, start_cell in ((True, False), (False, True), (False, False)):
        res, st = _run(gx, pairs, scores, True, traceback=traceback, start_cell=start_cell)
        assert (st[15], st[17]) == (k, chain1)
        _check(res, pairs, oracle, scores, True, traceback, start_cell, f"K={k} chain1={chain1}")
    assert res[0].score == 3000 * a
    assert _status(lambda: gx.align_batch(pairs, (a + 1, -a - 1, -a - 1, -1), True)) == 3


# ================================================================================================ (d) LCS pass
@functools.lru_cache(maxsize=None)
def _lcs_pairs():
    rng = np.random.default_rng(2602)
    pairs = [random_pair(rng, int(rng.integers(0, 90)), int(rng.integers(0, 90)), alphabet=b"ACGT" if q % 3 else b"AC",
                         similar=bool(q % 2)) for q in range(40)]
    pairs += [random_pair(rng, 700, 900), random_pair(rng, 2500, 300), random_pair(rng, 1200, 2500, similar=False)]
    return tuple(pairs)


@gpu
@pytest.mark.parametrize("chain1", [0, 1])
@pytest.mark.parametrize("k,r", KR_COMBOS)
def test_lcs_at_max_key_range(gx, oracle, k, r, chain1, monkeypatch):
    """GX_FLAG_LCS_AT_MAX keys the first maximum as (V << log2 K) | (K-1-k) in int32, global mode included: scorings just
    under its bound, global and local, against the oracle's max_matches at the first max cell.  One step past the bound
    is refused."""
    force_kr(monkeypatch, k, r)
    _set_chain1(monkeypatch, chain1)
    pairs = list(_lcs_pairs())
    L = max(max(len(a), len(b)) for a, b in pairs)
    mx = max_lcs_mx(L, -1)
    h1 = LCS_LIM - 1 - (2 * L + 2)
    for scores in ((mx, -mx, -mx, -1), (1, -1, -1, -h1)):
        for is_local in (False, True):
            res, st = _run(gx, pairs, scores, is_local, lcs_at_max=True)
            what = f"K={k} chain1={chain1} {scores} local={is_local}"
            assert st[15] == k, what
            _check(res, pairs, oracle, scores, is_local, True, False, what)
            for (a, b), rr in zip(pairs, res):
                assert rr.matches_at_max == _expect(oracle, a, b, scores, is_local).lcs_at_first_max, (what, len(a), len(b))
    for is_local in (False, True):
        for scores in ((mx + 1, -mx - 1, -mx - 1, -1), (1, -1, -1, -h1 - 1)):
            assert _status(lambda: gx.align_batch(pairs, scores, is_local, lcs_at_max=True)) == 3, (scores, is_local)


# ================================================================================================ (f) read kernels
def _read_set(seed, n_pairs, max_len):
    """n_pairs pairs of lengths 0..max_len (the first one max_len x max_len), every second one similar"""
    rng = np.random.default_rng(seed)
    pairs = []
    for q in range(n_pairs):
        m = max_len if q == 0 else int(rng.integers(0, max_len + 1))
        n = max_len if q == 0 else int(rng.integers(0, max_len + 1))
        pairs.append(random_pair(rng, m, n, similar=bool(q % 2), sub=0.06, indel=0.01))
    return pairs


def _reads16_edges(max_len):
    """(scores, lane width the plan must run) on both sides of each limit of the s16x2 kernel (reads16_ok)"""
    a = 8000 // (max_len + 1) + 1                  # the vmax limit binds before the beta limit
    beta = 15999 - (max_len + 1) * a               # vmax = max_len·a + beta + a = 15 999
    return [((a, -1, -1, -(beta - 1)), 16), ((a, -1, -1, -beta), 32),                 # vmax 15 999 / 16 000
            ((1, -1, -7999, 0), 16), ((1, -1, -8000, 0), 32),                         # -g 7 999 / 8 000
            ((1, -1, -1, -7998), 16), ((1, -1, -1, -7999), 32),                       # beta = -(h+g) 7 999 / 8 000
            ((1, -6, -1, -5), 16), ((1, -7, -1, -5), 32)]                             # b + beta 0 / -1


def _read_plan_scores(gx, packed, scores, is_local):
    blob, off1, len1, off2, len2 = packed
    plan = gx.Plan(len1, len2, scores, is_local, traceback=False)
    try:
        plan.upload(blob, off1, off2)
        plan.execute()
        return plan.fetch_scores(), plan.stat(9), plan.stat(26)
    finally:
        plan.close()


@gpu
@pytest.mark.parametrize("max_len", [152, 153, 320, 321, 640])
def test_read_kernels_s16_limits(gx, oracle, max_len, monkeypatch):
    """1024-pair read plans in every G x K class, local, with scorings on both sides of each s16x2 limit: against the
    oracle and against the 32-bit kernel (GX_READS32)"""
    monkeypatch.delenv("GX_READS32", raising=False)
    packed = gx.pack_pairs(_read_set(max_len, 1024, max_len))
    for scores, bits in _reads16_edges(max_len):
        exp = oracle.score_batch(*packed, scores, True, n_threads=8)
        got, kind, used = _read_plan_scores(gx, packed, scores, True)
        assert (kind, used) == (1, bits), (max_len, scores)
        assert np.array_equal(got, exp), (max_len, scores)
        monkeypatch.setenv("GX_READS32", "1")
        got32, kind, used = _read_plan_scores(gx, packed, scores, True)
        monkeypatch.delenv("GX_READS32")
        assert (kind, used) == (1, 32), (max_len, scores)
        assert np.array_equal(got32, exp), (max_len, scores)


@gpu
def test_read_kernel_global_cell_bound(gx, oracle):
    """the 32-bit read kernel in global mode at the cell bound of 640 x 640 pairs"""
    packed = gx.pack_pairs(_read_set(640, 1024, 640))
    mx = max_mx(640, 640, -1)
    for scores in ((mx, -mx, -mx, -1), (1, -1, -1, -max_h(640, 640, 1))):
        exp = oracle.score_batch(*packed, scores, False, n_threads=8)
        got, kind, used = _read_plan_scores(gx, packed, scores, False)
        assert (kind, used) == (1, 32), scores
        assert np.array_equal(got, exp), scores


@functools.lru_cache(maxsize=None)
def _stream_set():
    """2^18 + 4099 pairs of up to 60 bases (every chunk holds a 60 x 60 pair), laid out pair by pair; s2 is a trimmed,
    mutated copy of s1 for even pairs and random for odd ones"""
    rng = np.random.default_rng(1 << 18)
    n_pairs, L = (1 << 18) + 4099, 60
    len1 = rng.integers(0, L + 1, size=n_pairs).astype(np.uint64)
    len1[::1 << 18] = L
    trim = np.minimum(rng.integers(0, 4, size=n_pairs).astype(np.uint64), len1)
    trim[::1 << 18] = 0
    len2 = len1 - trim
    inter = np.empty(2 * n_pairs, np.uint64)
    inter[0::2], inter[1::2] = len1, len2
    ends = np.cumsum(inter)
    off1, off2 = ends[0::2] - len1, ends[1::2] - len2
    blob = _LUT[rng.integers(0, 4, size=int(ends[-1]))]
    even = np.arange(0, n_pairs, 2)
    cnt = len2[even].astype(np.int64)
    within = np.arange(int(cnt.sum())) - np.repeat(np.cumsum(cnt) - cnt, cnt)
    dst = np.repeat(off2[even].astype(np.int64), cnt) + within
    src = np.repeat((off1[even] + trim[even]).astype(np.int64), cnt) + within
    blob[dst] = blob[src]
    mut = dst[rng.random(dst.size) < 1 / 16]
    blob[mut] = _LUT[rng.integers(0, 4, size=mut.size)]
    return blob, off1, len1, off2, len2


@gpu
def test_read_stream_edges(gx, oracle, monkeypatch):
    """the streamed path (>= 2^18 pairs), which checks every batch against 640 x 640: one scoring at the s16x2 vmax
    limit (local) and one at the streamed cell bound (global), against the oracle and the 32-bit kernel"""
    blob, off1, len1, off2, len2 = _stream_set()
    a = 8000 // 61 + 1
    mx = max_mx(READS_MAX_LEN, READS_MAX_LEN, -1)
    for scores, is_local in (((a, -1, -1, -(15999 - 61 * a - 1)), True), ((mx, -mx, -mx, -1), False)):
        exp = oracle.score_batch(blob, off1, len1, off2, len2, scores, is_local, n_threads=8)
        monkeypatch.delenv("GX_READS32", raising=False)
        got = gx.score_batch(blob, off1, len1, off2, len2, scores, is_local)
        assert np.array_equal(got, exp), (scores, is_local)
        monkeypatch.setenv("GX_READS32", "1")
        got = gx.score_batch(blob, off1, len1, off2, len2, scores, is_local)
        monkeypatch.delenv("GX_READS32")
        assert np.array_equal(got, exp), (scores, is_local)


# ================================================================================================ (g) refusals
@gpu
def test_refusals_at_each_bound(gx):
    """the last scoring inside each bound is accepted and the first one past it returns status 3, through every entry
    point that checks one"""
    rng = np.random.default_rng(5)
    a, b = random_pair(rng, 700, 900)
    mx, hmax, la = max_mx(700, 900, -1), max_h(700, 900, 1), max_local_a(700, 900)
    cases = [(False, (mx, -mx, -mx, -1), (mx + 1, -mx, -mx, -1)),
             (False, (1, -1, -1, -hmax), (1, -1, -1, -hmax - 1)),
             (True, (la, -1, -1, -5), (la + 1, -1, -1, -5))]
    for is_local, inside, past in cases:
        for scores, want in ((inside, 0), (past, 3)):
            assert _status(lambda: gx.Plan([700], [900], scores, is_local).close()) == want, (scores, is_local)
            assert _status(lambda: gx.align_batch([(a, b)], scores, is_local)) == want, (scores, is_local)
            assert _status(lambda: gx.align_batch([(a, b)], scores, is_local, traceback=False, start_cell=True)) == want
    # LCS pass
    L = 900
    lmx = max_lcs_mx(L, -1)
    for is_local in (False, True):
        assert _status(lambda: gx.align_batch([(a, b)], (lmx, -lmx, -lmx, -1), is_local, lcs_at_max=True)) == 0
        assert _status(lambda: gx.align_batch([(a, b)], (lmx + 1, -lmx, -1, -1), is_local, lcs_at_max=True)) == 3
    # column bands
    assert _status(lambda: gx.nw_score_banded_local(a, b, (mx, -mx, -mx, -1), 3)) == 0
    assert _status(lambda: gx.nw_score_banded_local(a, b, (mx, -mx - 1, -mx, -1), 3)) == 3
    assert _status(lambda: gx.Band(700, 900, 2, 0, 2, (1, -1, -1, -hmax)).close()) == 0
    assert _status(lambda: gx.Band(700, 900, 2, 0, 2, (1, -1, -1, -hmax - 1)).close()) == 3
    # score batches: the plan path checks each pair, the streamed path (>= 2^18 pairs) checks 640 x 640
    packed = gx.pack_pairs(_read_set(7, 1024, 150))
    smx = max_mx(150, 150, -1)
    for is_local in (False, True):
        if not is_local:
            assert _status(lambda: gx.score_batch(*packed, (smx, -smx, -smx, -1), is_local)) == 0
            assert _status(lambda: gx.score_batch(*packed, (smx + 1, -smx, -smx, -1), is_local)) == 3
        sla = max_local_a(150, 150)
        assert _status(lambda: gx.score_batch(*packed, (sla, -1, -1, -1), True)) == 0
        assert _status(lambda: gx.score_batch(*packed, (sla + 1, -1, -1, -1), True)) == 3
    stream = _stream_set()
    rmx = max_mx(READS_MAX_LEN, READS_MAX_LEN, -1)
    assert _status(lambda: gx.score_batch(*stream, (rmx, -rmx, -rmx, -1), False)) == 0
    assert _status(lambda: gx.score_batch(*stream, (rmx + 1, -rmx, -rmx, -1), False)) == 3     # 60-base pairs, yet refused
    rla = max_local_a(READS_MAX_LEN, READS_MAX_LEN)
    assert _status(lambda: gx.score_batch(*stream, (rla, -1, -1, -1), True)) == 0
    assert _status(lambda: gx.score_batch(*stream, (rla + 1, -1, -1, -1), True)) == 3


# ================================================================================================ CPU: the bounds themselves
def test_check_scores_exact_boundaries():
    """gx_check_scores (local bounds included) at the exact edges the helpers above derive: the last scoring inside is
    accepted, the first one past is status 3; the sign rules are status 2"""
    from genomics_rs_b200 import _lib
    lib = _lib.load()

    def chk(scores, m, n):
        return lib.gx_check_scores(_lib.GxScores(*scores), m, n)

    for m, n in ((0, 0), (1, 3000), (700, 900), (8193, 770), (3000, 2600), (2000, 40000), (640, 640), (1 << 20, 5)):
        for h in (0, -1, -12345):
            mx = max_mx(m, n, h)
            assert chk((1, -mx, -1, h), m, n) == 0 and chk((1, -mx - 1, -1, h), m, n) == 3, (m, n, h)
            assert chk((1, -1, -mx, h), m, n) == 0 and chk((1, -1, -mx - 1, h), m, n) == 3, (m, n, h)
            assert chk((-mx, -mx, -1, h), m, n) == 0 and chk((-mx - 1, -1, -1, h), m, n) == 3, (m, n, h)
        hm = max_h(m, n, 1)
        assert chk((1, -1, -1, -hm), m, n) == 0 and chk((1, -1, -1, -hm - 1), m, n) == 3, (m, n)
    for m, n in ((3000, 3000), (3000, 2600), (8192, 8192), (640, 640)):
        a = max_local_a(m, n)
        assert (m + n + 2) * (a + 1) < CELL_LIM       # the local bound binds here, not the cell bound
        assert chk((a, -1, -1, -1), m, n) == 0 and chk((a + 1, -1, -1, -1), m, n) == 3, (m, n)
        assert chk((-1, -a - 1, -1, -1), m, n) == 0    # only a positive match score counts
    assert chk((1, -1, -1, 0), 1 << 28, 1) == 0 and chk((1, -1, -1, 0), (1 << 28) + 1, 1) == 3
    assert chk((1, -1, -1, 0), 10, 10) == 0           # h = 0 is allowed
    assert chk((1, -1, -1, 1), 10, 10) == 2           # h > 0
    assert chk((1, -1, 0, -1), 10, 10) == 2           # g = 0
    assert chk((1, -1, 0, 0), 10, 10) == 2            # h + g = 0


def test_chain1_key_rule():
    """where the CHAIN1 start-cell key of V = 0 reaches INT32_MIN, for every blocking (the classic form never does)"""
    for k, first_bad in ((4, 1 << 29), (8, 1 << 28), (16, 1 << 27)):
        assert chain1_keys_fit(k, (1, -1, -1, -(first_bad - 2)))
        assert not chain1_keys_fit(k, (1, -1, -1, -(first_bad - 1)))
        kb = k.bit_length() - 1
        assert ((-(first_bad - 1)) << kb) >= -(1 << 31) and ((-first_bad) << kb) == -(1 << 31)
    # K = 4 cannot reach it inside the contract: the largest |h+g| it allows is 2^29 - 2 (empty table, g = -1)
    assert chain1_keys_fit(4, (1, -1, -1, -max_h(0, 0, 1)))
