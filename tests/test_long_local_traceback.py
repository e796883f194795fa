"""Local traceback of pairs whose direction codes do not fit the device.  A compact local plan runs a score-only pass that
finds each pair's start cell first, then keeps codes only for the tiles of a band around the slope-1 line that ends there
(DESIGN.md section 2).  CPU: the diagonal construction that pins the config-5 pair's local alignment, and the band test
against the global one.  GPU: the 1 Mbp x 1 Mbp pair end to end, compact against dense storage, the goldens, interior start
cells with run-on tails, every kernel variant, edge tables, re-upload, the code budget and GX_FLAG_LCS_AT_MAX."""
import ctypes as C

import numpy as np
import pytest

from conftest import CONFIG_TOML, KR_COMBOS, force_kr, random_pair, read_fasta_gz
from test_long_traceback import _tile_in_band

FULL = 1_000_000
PANEL_H = 4096
# (L, score, start, n_ops) of the L x L prefix of the config-5 pair, local: the tail of the diagonal (end (1, 1))
TABLE = {FULL: (906128, 999998, 999998), 262144: (237285, 262143, 262143)}


def _config5():
    from genomics_rs_b200 import workloads as wl
    return wl.long_pair(FULL)


def _local_diagonal(a, b):
    """the local alignment of an m x m table of a substitution-only pair whose diagonal prefix sums c (+1 match, -2
    mismatch) stay >= 1: V(i, i) = c[i] never reaches 0, so the score is max c, the start cell (i*, i*) with i* the last
    index that attains it, and the walk is i* diagonal moves to (1, 1), the move at (i, i) labelled is_match(i, i) -- the
    characters after the cell, 0-based a[i] == b[i], None == None at i = m"""
    m = a.size
    eq = a == b
    c = np.concatenate([[0], np.cumsum(np.where(eq, 1, -2))])
    assert c[1:].min() >= 1
    score = int(c.max())
    i = int(np.flatnonzero(c == score)[-1])
    idx = np.arange(i, 0, -1)
    lab = np.where(idx < m, eq[np.minimum(idx, m - 1)], True)
    ops = np.where(lab, 0, 1).astype(np.uint8)
    return {"score": score, "start": (i, i), "ops": ops, "matches": int(np.count_nonzero(lab)),
            "mismatches": int(np.count_nonzero(~lab))}


def _line(end, local):
    """(a0, b0, a1, b1) of a pair's band line: global (0,0)-(m,n), local the slope-1 line back from the start cell"""
    i, j = end
    d = min(i, j) if local else 0
    return (i - d, j - d, i, j) if local else (0, 0, i, j)


def _tile_in_line(a0, b0, a1, b1, m, p, s, W, cw):
    """tile_in_code_band (csrc/gx_common.cuh)"""
    if p == 0 and s == 0:
        return True
    i0 = p * PANEL_H
    i1 = min(i0 + PANEL_H, m)
    c0 = s * W
    if i0 >= a1 or c0 >= b1:
        return False
    col = lambda i: b0 if (i <= a0 or a1 == a0) else b0 + (i - a0) * (b1 - b0) // (a1 - a0)
    return c0 + W + cw > col(i0) and c0 < col(i1) + cw + 1


def _band_tiles(m, n, end, K, cw, local=True):
    """in-band tiles of one pair; those that start at or beyond the end cell are out, so only the ones before it are tested"""
    W = 32 * K
    line = _line(end, local)
    return sum(_tile_in_line(*line, m, p, s, W, cw) for p in range(-(-end[0] // PANEL_H)) for s in range(-(-end[1] // W)))


def _tile_bytes(m, K):
    return (min(m, PANEL_H) + 62) // 32 * (K // 2) * 32 * 16


def _compact_bytes(dims, ends, K, widths, local=True):
    """bytes of compact code storage: in-band tiles x tile_code_bytes (32-step hand-off batches, 16-byte chunks per lane)"""
    return sum(_band_tiles(m, n, e, K, w, local) * _tile_bytes(m, K) for (m, n), e, w in zip(dims, ends, widths) if m and n)


# ------------------------------------------------------------------------------------------------ CPU
def test_local_diagonal_expectation_small(oracle):
    """the construction against the oracle's local traceback on prefixes it can run, one with its start cell inside"""
    a, b = _config5()
    for L, start in ((4096, (4096, 4096)), (20000, (20000, 20000)), (2005, (2004, 2004))):
        o = oracle.align_linear(a[:L], b[:L], CONFIG_TOML, True)
        d = _local_diagonal(a[:L], b[:L])
        assert o.score == d["score"] and tuple(o.start) == d["start"] == start and tuple(o.end) == (1, 1), L
        assert np.array_equal(o.ops, d["ops"]), L
        assert (o.matches, o.mismatches, o.gap_extensions, o.opening_gaps) == (d["matches"], d["mismatches"], 0, 0), L
    assert _local_diagonal(a[:2005], b[:2005])["score"] == 1779


def test_local_diagonal_table():
    """the full pair and the 262144 prefix: score, start cell and length of the path"""
    a, b = _config5()
    for L, (score, i, j) in TABLE.items():
        d = _local_diagonal(a[:L], b[:L])
        assert (d["score"], d["start"], d["ops"].size) == (score, (i, j), i), L


def test_band_line_generalises_the_diagonal():
    """the line test with the global end points (0,0)-(m,n) is the old diagonal test tile for tile"""
    rng = np.random.default_rng(5)
    shapes = [(1, 1), (5, 3000), (3000, 5), (4096, 4096), (4097, 4095), (12000, 700), (700, 12000), (20000, 19000),
              (50000, 50000), (65537, 1000)] + [tuple(int(v) for v in rng.integers(1, 40000, 2)) for _ in range(20)]
    for m, n in shapes:
        for K in (4, 8, 16):
            W = 32 * K
            S, P = -(-n // W), -(-m // PANEL_H)
            for cw in (0, 64, 300, 1024 + abs(m - n)):
                for p in range(P):
                    for s in range(S):
                        assert _tile_in_line(0, 0, m, n, m, p, s, W, cw) == _tile_in_band(m, n, p, s, W, cw), (m, n, K, cw, p, s)


def test_band_line_local_shape():
    """local lines: tiles beyond the end cell are out, tile (0,0) is in for every end cell, and widening always reaches
    the tile of any cell up and left of the end cell"""
    rng = np.random.default_rng(6)
    for _ in range(40):
        m, n = (int(v) for v in rng.integers(1, 60000, 2))
        end = (int(rng.integers(1, m + 1)), int(rng.integers(1, n + 1)))
        K = int(rng.choice([4, 8, 16]))
        W = 32 * K
        line = _line(end, True)
        S, P = -(-n // W), -(-m // PANEL_H)
        for cw in (64, 1024):
            assert _tile_in_line(*line, m, 0, 0, W, cw)
            for p in range(P):
                for s in range(S):
                    if p * PANEL_H >= end[0] or s * W >= end[1]:
                        assert not _tile_in_line(*line, m, p, s, W, cw) or (p, s) == (0, 0)
        i, j = int(rng.integers(1, end[0] + 1)), int(rng.integers(1, end[1] + 1))
        w = 64
        while not _tile_in_line(*line, m, (i - 1) // PANEL_H, (j - 1) // W, W, w):
            w *= 2
            assert w < 1 << 40


def test_local_compact_bytes_of_the_table():
    """the plan arithmetic at the default half-width 1024 for the two table rows (K as the plan picks it on a B200: 8 for
    the full pair, 4 for the prefix): 6,101 and 3,119 tiles hold codes, 1.6 GB and 0.41 GB against 251 GB and 17 GB dense"""
    full = _compact_bytes([(FULL, FULL)], [(999998, 999998)], 8, [1024])
    assert full == _compact_bytes([(FULL, FULL)], [(FULL, FULL)], 8, [1024]) == 6101 * 264_192 == 1_611_835_392
    pre = _compact_bytes([(262144, 262144)], [(262143, 262143)], 4, [1024])
    assert pre == 3119 * 132_096 == 412_007_424
    for b, (L, K) in ((full, (FULL, 8)), (pre, (262144, 4))):
        assert b % _tile_bytes(L, K) == 0
        assert b * 40 < -(-L // (32 * K)) * -(-L // PANEL_H) * _tile_bytes(L, K)


def test_brca2_local_path_within_the_default_band(oracle):
    """the BRCA2 local path, run-on tail included, stays within 232 columns of the slope-1 line through its start cell"""
    s = read_fasta_gz("Human-Mouse-BRCA2-cds")
    o = oracle.align_linear(s[0][1], s[1][1], CONFIG_TOML, True)
    assert tuple(o.start) == (10283, 10117)
    off = (o.ops_j.astype(np.int64) - 10117) - (o.ops_i.astype(np.int64) - 10283)
    assert np.abs(off).max() <= 232


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def gx():
    import genomics_rs_b200 as gx
    from genomics_rs_b200 import _lib
    _lib.ensure_init()
    return gx


def _align_pair_local(a, b, scores=CONFIG_TOML):
    from genomics_rs_b200 import _lib
    from genomics_rs_b200.alignment import _scores_struct
    lib = _lib.ensure_init()
    res = _lib.GxResult()
    ops = np.zeros(a.size + b.size + 1, np.uint8)
    rc = lib.gx_align_pair(a.ctypes.data, a.size, b.ctypes.data, b.size, _scores_struct(scores), 1, _lib.GX_FLAG_TRACEBACK,
                           C.byref(res), ops.ctypes.data, ops.size)
    return rc, res, ops[:res.n_ops]


def _ops_of(res, ops, ops_off, q):
    return ops[int(ops_off[q]):int(ops_off[q]) + int(res["n_ops"][q])].copy()


def _run(gx, pairs, executes=1, **kw):
    blob, off1, len1, off2, len2 = gx.pack_pairs(pairs)
    plan = gx.Plan(len1, len2, CONFIG_TOML, True, traceback=True, **kw)
    plan.upload(blob, off1, off2)
    for _ in range(executes):
        plan.execute()
    res, ops, ops_off = plan.fetch()
    return plan, res, [_ops_of(res, ops, ops_off, q) for q in range(len(pairs))]


def _same(res, q, ops, o, what=""):
    assert res["score"][q] == o.score, what
    assert (res["start_i"][q], res["start_j"][q]) == tuple(o.start) and (res["end_i"][q], res["end_j"][q]) == tuple(o.end), what
    assert (res["matches"][q], res["mismatches"][q], res["gap_extensions"][q], res["opening_gaps"][q]) == (
        o.matches, o.mismatches, o.gap_extensions, o.opening_gaps), what
    assert np.array_equal(ops, o.ops), what


@pytest.mark.gpu
def test_config5_full_local_traceback(gx):
    """the 10^6 x 10^6 pair, local with traceback, through gx_align_pair: dense codes (~251 GB) do not fit, the band
    around the start cell's line does; the result is the table's row exactly, and score and start cell are those of a
    score-only start-cell plan"""
    from genomics_rs_b200 import _lib
    a, b = _config5()
    rc, r, ops = _align_pair_local(a, b)
    assert rc == 0, _lib.load().gx_last_error()
    d = _local_diagonal(a, b)
    assert r.score == d["score"] == 906128
    assert (r.start_i, r.start_j, r.end_i, r.end_j) == (999998, 999998, 1, 1)
    assert (r.matches, r.mismatches, r.gap_extensions, r.opening_gaps) == (d["matches"], d["mismatches"], 0, 0)
    assert r.n_ops == 999998 and np.array_equal(ops, d["ops"])
    plan, res, _ = _run(gx, [(a, b)])
    K = int(plan.stat(15))
    assert plan.stat(27) == 2.0 and plan.stat(4) < 4e9 and plan.stat(24) == 0 and plan.stat(29) > 0
    assert plan.stat(0) >= plan.stat(29)
    assert plan.stat(4) == _compact_bytes([(FULL, FULL)], [(999998, 999998)], K, [int(plan.stat(28))])
    assert int(res["score"][0]) == 906128 and int(res["n_ops"][0]) == 999998
    plan.close()
    sc = gx.align_batch([(a, b)], CONFIG_TOML, True, traceback=False, start_cell=True)[0]
    assert sc.score == 906128 and tuple(sc.start) == (999998, 999998)


@pytest.mark.gpu
def test_local_compact_equals_dense_262144(gx, monkeypatch):
    """the 262144 x 262144 prefix (dense local codes fit): compact storage forced and dense storage give the same gx_result
    (less the timings) and the same ops; both code sizes match the plan arithmetic"""
    a, b = _config5()
    L = 262144
    out = {}
    for compact in (True, False):
        if compact:
            monkeypatch.setenv("GX_CODE_COMPACT", "1")
        else:
            monkeypatch.delenv("GX_CODE_COMPACT", raising=False)
        plan, res, ops = _run(gx, [(a[:L], b[:L])])
        assert plan.stat(27) == (2.0 if compact else 0.0)
        assert (plan.stat(29) > 0) == compact
        out[compact] = (res, ops[0], plan.stat(4), int(plan.stat(15)))
        plan.close()
    for f in (f for f in out[True][0].dtype.names if f not in ("fill_ms", "walk_ms")):
        assert out[True][0][f][0] == out[False][0][f][0], f
    assert np.array_equal(out[True][1], out[False][1])
    K = out[True][3]
    assert out[True][2] == _compact_bytes([(L, L)], [(262143, 262143)], K, [1024])
    assert out[False][2] == -(-L // (32 * K)) * -(-L // PANEL_H) * _tile_bytes(L, K) > 40 * out[True][2]
    d = _local_diagonal(a[:L], b[:L])
    r = out[True][0]
    assert (int(r["score"][0]), int(r["start_i"][0]), int(r["end_i"][0])) == (237285, 262143, 1)
    assert np.array_equal(out[True][1], d["ops"])


@pytest.mark.gpu
def test_local_goldens_compact(gx, oracle, goldens, monkeypatch):
    """compact storage forced: every local golden against oracle_goldens.json and the oracle; BRCA2 needs no widening"""
    monkeypatch.setenv("GX_CODE_COMPACT", "1")
    for g in (p for p in goldens["pairs"] if p["is_local"]):
        s = read_fasta_gz(g["fixture"])
        x, y = np.frombuffer(s[0][1].encode(), np.uint8), np.frombuffer(s[1][1].encode(), np.uint8)
        plan, res, ops = _run(gx, [(x, y)])
        assert plan.stat(27) == 2.0, g["fixture"]
        assert res["score"][0] == g["score"] and [res["start_i"][0], res["start_j"][0]] == g["start"], g["fixture"]
        assert [res["end_i"][0], res["end_j"][0]] == g["end"] and len(ops[0]) == g["n_ops"], g["fixture"]
        assert "%016x" % oracle.hash_ops(ops[0], g["start"]) == g["op_hash"], g["fixture"]
        assert (res["matches"][0], res["mismatches"][0], res["gap_extensions"][0], res["opening_gaps"][0]) == (
            g["matches"], g["mismatches"], g["gap_extensions"], g["opening_gaps"]), g["fixture"]
        _same(res, 0, ops[0], oracle.align_linear(x, y, CONFIG_TOML, True), g["fixture"])
        if g["fixture"] == "Human-Mouse-BRCA2-cds":
            assert plan.stat(24) == 0 and plan.stat(28) == 1024
        plan.close()


def _offset_pairs(rng):
    """a homologous segment at different offsets in each sequence, unrelated flanks: start cells inside the table with
    i* != j*, and run-on tails through unrelated sequence"""
    lut = np.frombuffer(b"ACGT", np.uint8)
    junk = lambda k: lut[rng.integers(0, 4, size=k)]
    out = []
    for core, (l1, r1, l2, r2) in ((3000, (500, 800, 2500, 100)), (6000, (3000, 400, 200, 3500)),
                                   (2000, (6000, 1000, 700, 300)), (4000, (100, 100, 4000, 4000)),
                                   (1500, (50, 2000, 60, 2500))):
        x, y = random_pair(rng, core, core, similar=True, sub=0.05, indel=0.01)
        out.append((np.concatenate([junk(l1), x, junk(r1)]), np.concatenate([junk(l2), y, junk(r2)])))
    # substitutions only, start cell on the main diagonal: stays inside any band
    x, y = random_pair(rng, 5000, 5000, similar=True, sub=0.05, indel=0.0)
    out.append((x, y))
    return out


_OFFSET = {}


@pytest.mark.gpu
def test_local_interior_start_cells(gx, oracle, monkeypatch):
    """interior start cells off the main diagonal, with a forced 64-column band and the default: the bands move to the
    start cells, walks whose run-on tails leave make the execute widen those pairs only, and every result is the
    oracle's; a second execute needs no repeat"""
    pairs = _offset_pairs(np.random.default_rng(41))
    exp = [oracle.align_linear(x, y, CONFIG_TOML, True) for x, y in pairs]
    assert sum(o.start[0] < len(x) and o.start[1] < len(y) and o.start[0] != o.start[1] for o, (x, y) in zip(exp, pairs)) >= 4
    dims = [(len(x), len(y)) for x, y in pairs]
    ends = [tuple(int(v) for v in o.start) for o in exp]
    monkeypatch.setenv("GX_CODE_COMPACT", "1")
    for band in ("64", None):
        if band:
            monkeypatch.setenv("GX_CODE_BAND", band)
        else:
            monkeypatch.delenv("GX_CODE_BAND", raising=False)
        plan, res, ops = _run(gx, pairs)
        K = int(plan.stat(15))
        for q, o in enumerate(exp):
            _same(res, q, ops[q], o, (band, q))
        if band:
            assert plan.stat(24) >= 1
            widest = int(plan.stat(28))
            assert widest >= 128
            assert _compact_bytes(dims, ends, K, [64] * len(pairs)) < plan.stat(4) < _compact_bytes(dims, ends, K, [widest] * len(pairs))
        n_rep = plan.stat(24)
        plan.execute()
        assert plan.stat(24) == n_rep
        res2, ops2, off2 = plan.fetch()
        for q in range(len(pairs)):
            assert np.array_equal(_ops_of(res2, ops2, off2, q), ops[q]) and res2["score"][q] == res["score"][q]
        plan.close()
    # the substitution-only pair alone keeps its 64-column band
    monkeypatch.setenv("GX_CODE_BAND", "64")
    plan, res, ops = _run(gx, pairs[-1:])
    _same(res, 0, ops[0], exp[-1])
    assert plan.stat(24) == 0 and plan.stat(28) == 64
    assert plan.stat(4) == _compact_bytes(dims[-1:], ends[-1:], int(plan.stat(15)), [64])
    plan.close()


def _ragged_pairs(rng):
    sim = [random_pair(rng, m, n, similar=True, sub=0.1, indel=0.01) for m, n in [(4200, 4200), (8193, 8193), (2000, 2100), (4096, 4096)]]
    lut = np.frombuffer(b"ACGT", np.uint8)
    x, y = random_pair(rng, 3000, 3000, similar=True, sub=0.08, indel=0.01)
    off = [(np.concatenate([lut[rng.integers(0, 4, size=1200)], x]), np.concatenate([y, lut[rng.integers(0, 4, size=900)]])),
           (np.concatenate([x, lut[rng.integers(0, 4, size=5000)]]), np.concatenate([lut[rng.integers(0, 4, size=4100)], y]))]
    any_ = [random_pair(rng, m, n, similar=False) for m, n in [(4097, 5300), (700, 9000), (5000, 400)]]
    return sim + off + any_


_RAGGED = {}


@pytest.mark.parametrize("mode", ["tickets", "resident"])
@pytest.mark.parametrize("chain1", [0, 1])
@pytest.mark.parametrize("k,r", KR_COMBOS)
@pytest.mark.gpu
def test_local_compact_kernel_ragged(gx, oracle, k, r, chain1, mode, monkeypatch):
    """the compact local fill for every register tile, both recurrence forms, ticket and resident-strips scheduling, on
    ragged tables with a forced 300-column band: similar pairs, offset homology and unrelated pairs"""
    force_kr(monkeypatch, k, r)
    monkeypatch.setenv("GX_CHAIN1", str(chain1))
    monkeypatch.setenv("GX_CODE_COMPACT", "1")
    monkeypatch.setenv("GX_CODE_BAND", "300")
    monkeypatch.setenv("GX_TICKETS" if mode == "tickets" else "GX_RESIDENT", "1")
    pairs = _ragged_pairs(np.random.default_rng(19))
    plan, res, ops = _run(gx, pairs)
    assert plan.stat(27) == 2.0 and plan.stat(21) == (1.0 if mode == "resident" else 0.0) and plan.stat(15) == k
    for q, (a, b) in enumerate(pairs):
        if q not in _RAGGED:
            _RAGGED[q] = oracle.align_linear(a, b, CONFIG_TOML, True)
        _same(res, q, ops[q], _RAGGED[q], (k, chain1, mode, q))
    plan.close()


@pytest.mark.parametrize("rows", [64, 128, 256, 512])
@pytest.mark.parametrize("k,r", [(4, 1), (8, 1)])
@pytest.mark.gpu
def test_local_compact_walk_window_sizes(gx, oracle, k, r, rows, monkeypatch):
    """the walk's loader on compact local storage for every window height, with a 128-column band"""
    force_kr(monkeypatch, k, r)
    monkeypatch.setenv("GX_WALK_ROWS", str(rows))
    monkeypatch.setenv("GX_CODE_COMPACT", "1")
    monkeypatch.setenv("GX_CODE_BAND", "128")
    pairs = _ragged_pairs(np.random.default_rng(19))[3:7]
    plan, res, ops = _run(gx, pairs)
    for q, (a, b) in enumerate(pairs):
        key = q + 3
        if key not in _RAGGED:
            _RAGGED[key] = oracle.align_linear(a, b, CONFIG_TOML, True)
        _same(res, q, ops[q], _RAGGED[key], (k, rows, q))
    plan.close()


def _edge_pairs(rng):
    """all-zero tables, empty and single-base pairs, and last-maximum ties across panels and strips: junk uses letters the
    other sequence never has, so that the only positive cells come from the planted copies"""
    lut = np.frombuffer(b"ACGT", np.uint8)
    x = lut[rng.integers(0, 4, size=300)]
    W = lambda k: np.full(k, ord("W"), np.uint8)
    S = lambda k: np.full(k, ord("S"), np.uint8)
    e = np.zeros(0, np.uint8)
    return [
        ("all_zero", np.full(300, ord("A"), np.uint8), np.full(2000, ord("C"), np.uint8)),
        ("all_zero_tall", np.full(5000, ord("A"), np.uint8), np.full(700, ord("C"), np.uint8)),
        ("m0", e, x[:10]), ("n0", x[:10], e), ("m0n0", e, e), ("1x1_match", x[:1], x[:1]),
        ("1x1_mismatch", np.array([ord("A")], np.uint8), np.array([ord("C")], np.uint8)), ("1xn", x[:1], x), ("mx1", x, x[:1]),
        ("rows_two_panels", np.concatenate([W(200), x, W(5000), x, W(100)]), np.concatenate([S(400), x, S(50)])),
        ("cols_two_strips", np.concatenate([W(90), x, W(10)]), np.concatenate([S(100), x, S(1500), x, S(700)])),
        ("both_ways", np.concatenate([x, W(4500), x]), np.concatenate([x, S(900), x])),
    ]


@pytest.mark.gpu
def test_local_compact_edge_tables(gx, oracle, monkeypatch):
    """all-zero tables (start (m, n), the walk runs along row m), empty and single-base pairs, and last-maximum ties
    across panels and strips, in one batch that mixes pairs whose start cells differ, and each tie pair alone"""
    monkeypatch.setenv("GX_CODE_COMPACT", "1")
    named = _edge_pairs(np.random.default_rng(3))
    pairs = [(a, b) for _, a, b in named]
    exp = [oracle.align_linear(a, b, CONFIG_TOML, True) for a, b in pairs]
    for (name, a, b), o in zip(named, exp):
        if name.startswith("all_zero"):
            assert o.score == 0 and tuple(o.start) == (len(a), len(b)), name
        if name == "rows_two_panels":    # the later copy wins the tie: the table cut after the first copy has the same score
            assert o.score == 300 and tuple(o.start) == (5800, 700)
            assert oracle.align_linear(a[:600], b, CONFIG_TOML, True).score == 300
    plan, res, ops = _run(gx, pairs)
    assert plan.stat(27) == 2.0
    for q, ((name, _, _), o) in enumerate(zip(named, exp)):
        _same(res, q, ops[q], o, name)
    plan.close()
    for name, a, b in named[9:]:
        plan, res, ops = _run(gx, [(a, b)])
        _same(res, 0, ops[0], exp[[n for n, _, _ in named].index(name)], name)
        plan.close()


@pytest.mark.gpu
def test_local_compact_reupload(gx, oracle, monkeypatch):
    """one plan, two uploads of different sequences of the same lengths: the start cells move, both uploads' results are
    the oracle's; executes without a new upload repeat the result and add no repeats"""
    monkeypatch.setenv("GX_CODE_COMPACT", "1")
    rng = np.random.default_rng(77)
    lut = np.frombuffer(b"ACGT", np.uint8)
    junk = lambda k: lut[rng.integers(0, 4, size=k)]
    x, y = random_pair(rng, 3000, 3000, similar=True, sub=0.05, indel=0.0)
    first = [(np.concatenate([x, junk(3000)]), np.concatenate([junk(1000), y, junk(1000)])), random_pair(rng, 4500, 4500)]
    second = [(np.concatenate([junk(2500), x, junk(500)]), np.concatenate([y, junk(2000)])), random_pair(rng, 4500, 4500)]
    blob, off1, len1, off2, len2 = gx.pack_pairs(first)
    plan = gx.Plan(len1, len2, CONFIG_TOML, True, traceback=True)
    starts = []
    for pairs in (first, second):
        blob, off1, _, off2, _ = gx.pack_pairs(pairs)
        plan.upload(blob, off1, off2)
        plan.execute()
        res, ops, ops_off = plan.fetch()
        for q, (a, b) in enumerate(pairs):
            _same(res, q, _ops_of(res, ops, ops_off, q), oracle.align_linear(a, b, CONFIG_TOML, True), q)
        starts.append((int(res["start_i"][0]), int(res["start_j"][0])))
        n_rep, snap = plan.stat(24), res.copy()
        for _ in range(2):
            plan.execute()
            again, ops2, _ = plan.fetch()
            assert plan.stat(24) == n_rep
            for f in (f for f in snap.dtype.names if f not in ("fill_ms", "walk_ms")):
                assert np.array_equal(again[f], snap[f]), f
            assert np.array_equal(ops2, ops)
    assert starts[0] != starts[1]
    plan.close()


@pytest.mark.gpu
def test_local_code_budget(gx, oracle, monkeypatch):
    """GX_CODE_BUDGET below what the widened band needs: the execute returns GX_ERR_NOMEM (7) naming the local pair, the
    half-width and the bytes; the next execute refuses; the device stays usable.  An all-zero table starts at (m, n) and
    its walk runs along row m, out of any narrow band."""
    from genomics_rs_b200 import _lib
    pairs = [(np.full(300, ord("A"), np.uint8), np.full(9000, ord("C"), np.uint8))]
    blob, off1, len1, off2, len2 = gx.pack_pairs(pairs)
    monkeypatch.setenv("GX_CODE_BAND", "64")
    monkeypatch.setenv("GX_CODE_COMPACT", "1")
    plan = gx.Plan(len1, len2, CONFIG_TOML, True, traceback=True)
    need64 = int(plan.stat(4))
    plan.close()
    monkeypatch.delenv("GX_CODE_COMPACT")
    monkeypatch.setenv("GX_CODE_BUDGET", str(need64))     # dense codes exceed it: compact storage, at 64 columns it fits
    plan = gx.Plan(len1, len2, CONFIG_TOML, True, traceback=True)
    assert plan.stat(27) == 2.0 and plan.stat(4) == need64
    plan.upload(blob, off1, off2)
    with pytest.raises(_lib.GxError) as e:
        plan.execute()
    assert e.value.status == 7
    msg = str(e.value)
    assert "local pair 0" in msg and "half-width" in msg and "bytes" in msg and "GX_CODE_BUDGET" in msg, msg
    with pytest.raises(_lib.GxError) as e:
        plan.execute()
    assert e.value.status == 7
    plan.close()
    monkeypatch.delenv("GX_CODE_BUDGET")
    monkeypatch.delenv("GX_CODE_BAND")
    r = gx.align_batch(pairs, CONFIG_TOML, True)[0]
    o = oracle.align_linear(pairs[0][0], pairs[0][1], CONFIG_TOML, True)
    assert r.score == o.score == 0 and tuple(r.start) == (300, 9000) and np.array_equal(r.ops, o.ops)


@pytest.mark.gpu
def test_local_compact_lcs_at_max(gx, monkeypatch):
    """GX_FLAG_LCS_AT_MAX on a compact local plan: the same result as dense, lcs_at_first_max included"""
    pairs = _offset_pairs(np.random.default_rng(41))[:3]
    out = {}
    for compact in (True, False):
        if compact:
            monkeypatch.setenv("GX_CODE_COMPACT", "1")
        else:
            monkeypatch.delenv("GX_CODE_COMPACT", raising=False)
        plan, res, ops = _run(gx, pairs, executes=2, lcs_at_max=True)
        assert plan.stat(27) == (2.0 if compact else 0.0)
        out[compact] = (res, ops)
        plan.close()
    for f in (f for f in out[True][0].dtype.names if f not in ("fill_ms", "walk_ms")):
        assert np.array_equal(out[True][0][f], out[False][0][f]), f
    assert all(np.array_equal(x, y) for x, y in zip(out[True][1], out[False][1]))
    assert all(out[True][0]["lcs_at_first_max"] > 0)
