"""Global traceback of pairs whose direction codes do not fit the device: compact code storage keeps codes only for the
tiles of the code band (DESIGN.md section 2), and a walk that leaves the band makes the execute repeat with a wider band for
that pair.  CPU: the pure-diagonal property of the config-5 pair that lets its full-size path be checked exactly.  GPU: the
1 Mbp x 1 Mbp pair end to end, compact against dense storage, compact storage against the oracle and the goldens, the
widening rounds and the code budget."""
import ctypes as C
import json
import os

import numpy as np
import pytest

from conftest import CONFIG_TOML, GOLDEN, KR_COMBOS, force_kr, random_pair, read_fasta_gz

FULL = 1_000_000
PANEL_H = 4096


def _config5():
    from genomics_rs_b200 import workloads as wl
    return wl.long_pair(FULL)


def _diagonal(a, b, L):
    """the global alignment of the L x L prefix when it is the pure diagonal: walk from (L, L), L diagonal moves, the move
    at (i, i) labelled is_match(i, i) -- the characters AFTER the cell, 0-based a[i] == b[i], with None == None at i = L"""
    eq = a[:L] == b[:L]
    lab = np.ones(L, bool)
    lab[1:] = eq[np.arange(L - 1, 0, -1)]          # moves at (L-1, L-1) .. (1, 1)
    ops = np.where(lab, 0, 1).astype(np.uint8)     # 0 Match, 1 Mismatch
    mism = int(np.count_nonzero(~eq[1:]))
    return {"score": L - 3 * int(np.count_nonzero(~eq)), "ops": ops, "matches": 1 + int(np.count_nonzero(eq[1:])),
            "mismatches": mism}


# ------------------------------------------------------------------------------------------------ CPU
def test_config5_prefix_scores_are_the_diagonal():
    """every frozen config-5 prefix score is the score of the pure diagonal, L - 3 * #mismatches (match 1, mismatch -2):
    V(i, i) is the diagonal prefix score for every i, so the reference's walk from (L, L) is L diagonal moves"""
    gold = json.load(open(os.path.join(GOLDEN, "config5_scores.json")))
    assert tuple(gold["scores"][k] for k in ("s_match", "s_mismatch", "g", "h")) == CONFIG_TOML
    a, b = _config5()
    for L, score in gold["prefix_scores"].items():
        L = int(L)
        d = _diagonal(a, b, L)
        assert d["score"] == score, L
        assert d["ops"].size == L and d["ops"][0] == 0
        assert d["matches"] + d["mismatches"] == L


def test_diagonal_expectation_small(oracle):
    """the expected-ops construction above against the oracle's traceback on a prefix it can run"""
    a, b = _config5()
    for L in (1, 2, 300, 4096):
        o = oracle.align_linear(a[:L], b[:L], CONFIG_TOML, False)
        d = _diagonal(a, b, L)
        assert o.score == d["score"], L
        assert np.array_equal(o.ops, d["ops"]), L
        assert (o.matches, o.mismatches, o.gap_extensions, o.opening_gaps) == (d["matches"], d["mismatches"], 0, 0), L
        assert tuple(o.start) == (L, L) and tuple(o.end) == (1, 1)


def _tile_in_band(m, n, p, s, W, cw):
    """tile_in_code_band (csrc/gx_common.cuh)"""
    i0 = p * PANEL_H
    i1 = min(i0 + PANEL_H, m)
    lo, hi = i0 * n // m, i1 * n // m
    c0 = s * W
    return c0 + W + cw > lo and c0 < hi + cw + 1


def _compact_bytes(dims, K, widths):
    """bytes of compact code storage: in-band tiles x tile_code_bytes (32-step hand-off batches, 16-byte chunks per lane)"""
    W, tot = 32 * K, 0
    for (m, n), cw in zip(dims, widths):
        if not m or not n:
            continue
        tile = (min(m, PANEL_H) + 62) // 32 * (K // 2) * 32 * 16
        S, P = -(-n // W), -(-m // PANEL_H)
        tot += tile * sum(_tile_in_band(m, n, p, s, W, cw) for p in range(P) for s in range(S))
    return tot


def test_compact_bytes_of_config5():
    """the plan arithmetic of the 1 Mbp pair at K = 8 and the default half-width 1024: 6,101 tiles of the 957,215 hold
    codes, about 1.6 GB instead of 251 GB"""
    W, S, P = 256, -(-FULL // 256), -(-FULL // PANEL_H)
    assert S * P == 957_215
    band = sum(_tile_in_band(FULL, FULL, p, s, W, 1024) for p in range(P) for s in range(S))
    assert band == 6101
    assert _compact_bytes([(FULL, FULL)], 8, [1024]) == band * 264_192 < 2e9


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def gx():
    import genomics_rs_b200 as gx
    from genomics_rs_b200 import _lib
    _lib.ensure_init()
    return gx


def _align_pair(a, b, scores=CONFIG_TOML):
    from genomics_rs_b200 import _lib
    from genomics_rs_b200.alignment import _scores_struct
    lib = _lib.ensure_init()
    res = _lib.GxResult()
    ops = np.zeros(a.size + b.size + 1, np.uint8)
    rc = lib.gx_align_pair(a.ctypes.data, a.size, b.ctypes.data, b.size, _scores_struct(scores), 0, _lib.GX_FLAG_TRACEBACK,
                           C.byref(res), ops.ctypes.data, ops.size)
    return rc, res, ops[:res.n_ops]


def _plan_run(gx, pairs, scores=CONFIG_TOML, executes=1):
    blob, off1, len1, off2, len2 = gx.pack_pairs(pairs)
    plan = gx.Plan(len1, len2, scores, False, traceback=True)
    plan.upload(blob, off1, off2)
    for _ in range(executes):
        plan.execute()
    res, ops, ops_off = plan.fetch()
    return plan, res, [ops[int(ops_off[q]):int(ops_off[q]) + int(res["n_ops"][q])].copy() for q in range(len(pairs))]


def _same(gpu, ora, what=""):
    assert gpu.score == ora.score, what
    assert tuple(gpu.start) == tuple(ora.start) and tuple(gpu.end) == tuple(ora.end), what
    assert (gpu.matches, gpu.mismatches, gpu.gap_extensions, gpu.opening_gaps) == (
        ora.matches, ora.mismatches, ora.gap_extensions, ora.opening_gaps), what
    assert np.array_equal(gpu.ops, ora.ops), what


@pytest.mark.gpu
def test_config5_full_traceback(gx):
    """the 10^6 x 10^6 pair, global with traceback, through gx_align_pair: its dense codes (~251 GB) do not fit, the compact
    band's (~1.6 GB) do; the path is the exact diagonal"""
    a, b = _config5()
    rc, r, ops = _align_pair(a, b)
    assert rc == 0
    d = _diagonal(a, b, FULL)
    assert r.score == d["score"] == 906127
    assert (r.start_i, r.start_j, r.end_i, r.end_j) == (FULL, FULL, 1, 1)
    assert (r.matches, r.mismatches, r.gap_extensions, r.opening_gaps) == (d["matches"], d["mismatches"], 0, 0)
    assert r.n_ops == FULL and np.array_equal(ops, d["ops"])
    plan, res, _ = _plan_run(gx, [(a, b)])
    assert plan.stat(27) == 2.0 and plan.stat(4) < 4e9 and plan.stat(24) == 0
    assert plan.stat(4) == _compact_bytes([(FULL, FULL)], int(plan.stat(15)), [int(plan.stat(28))])
    assert int(res["score"][0]) == 906127 and int(res["n_ops"][0]) == FULL
    plan.close()


@pytest.mark.gpu
def test_compact_equals_dense_262144(gx, monkeypatch):
    """the 262144 x 262144 prefix (dense codes fit): compact storage forced and dense storage give the same gx_result
    (less the timings) and the same ops"""
    a, b = _config5()
    L = 262144
    pair = [(a[:L], b[:L])]
    out = {}
    for compact in (True, False):
        if compact:
            monkeypatch.setenv("GX_CODE_COMPACT", "1")
        else:
            monkeypatch.delenv("GX_CODE_COMPACT", raising=False)
        plan, res, ops = _plan_run(gx, pair)
        assert plan.stat(27) == (2.0 if compact else 1.0)
        out[compact] = (res, ops[0], plan.stat(4), int(plan.stat(15)))
        plan.close()
    fields = [f for f in out[True][0].dtype.names if f not in ("fill_ms", "walk_ms")]
    for f in fields:
        assert out[True][0][f][0] == out[False][0][f][0], f
    assert np.array_equal(out[True][1], out[False][1])
    K = out[True][3]
    assert out[True][2] == _compact_bytes([(L, L)], K, [1024])           # compact: the band's tiles only
    assert out[False][2] == _compact_bytes([(L, L)], K, [2 * L]) > 40 * out[True][2]
    d = _diagonal(a, b, L)
    assert int(out[True][0]["score"][0]) == d["score"] == 237283 and np.array_equal(out[True][1], d["ops"])


@pytest.mark.gpu
def test_compact_reference_fixtures_and_corona(gx, oracle, goldens, ref_vectors, monkeypatch):
    """compact storage forced: the reference's vectors, every global fixture (BRCA2 included) and all 45 coronavirus pairs
    against the goldens and the oracle"""
    monkeypatch.setenv("GX_CODE_COMPACT", "1")
    sc = ref_vectors["scores"]
    scores = (sc["s_match"], sc["s_mismatch"], sc["g"], sc["h"])
    for case in ref_vectors["cases"]:
        r = gx.align_batch([(case["s1"], case["s2"])], scores, False)[0]
        assert [[c.name, i, j] for c, i, j in r.alignment] == case["alignment"], case["name"]
        assert (r.matches, r.mismatches, r.opening_gaps, r.gap_extensions) == (
            case["matches"], case["mismatches"], case["opening_gaps"], case["gap_extensions"]), case["name"]
        _same(r, oracle.align_faithful(case["s1"], case["s2"], scores, False), case["name"])
    for g in (p for p in goldens["pairs"] if not p["is_local"]):
        s = read_fasta_gz(g["fixture"])
        r = gx.align_batch([(s[0][1], s[1][1])], CONFIG_TOML, False)[0]
        assert r.score == g["score"] and list(r.start) == g["start"] and list(r.end) == g["end"], g["fixture"]
        assert len(r.ops) == g["n_ops"] and "%016x" % oracle.hash_ops(r.ops, r.start) == g["op_hash"], g["fixture"]
        assert (r.matches, r.mismatches, r.gap_extensions, r.opening_gaps) == (
            g["matches"], g["mismatches"], g["gap_extensions"], g["opening_gaps"]), g["fixture"]
        _same(r, oracle.align_linear(s[0][1], s[1][1], CONFIG_TOML, False), g["fixture"])
    order = goldens["corona_order"]
    seqs = [read_fasta_gz(name)[0][1] for name in order]
    jobs = [(x, y) for x in range(len(seqs)) for y in range(x + 1, len(seqs))]
    got = gx.align_batch([(seqs[x], seqs[y]) for x, y in jobs], CONFIG_TOML, False)
    gold = {tuple(c["pair"]): c for c in goldens["corona"]}
    for (x, y), r in zip(jobs, got):
        g = gold[(x, y)]
        assert r.score == g["score"] and len(r.ops) == g["n_ops"], (x, y)
        assert (r.matches, r.mismatches, r.gap_extensions, r.opening_gaps) == (
            g["matches"], g["mismatches"], g["gap_extensions"], g["opening_gaps"]), (x, y)
        assert "%016x" % oracle.hash_ops(r.ops, r.start) == g["op_hash"], (x, y)
    blob, off1, len1, off2, len2 = gx.pack_pairs([(seqs[x], seqs[y]) for x, y in jobs])
    plan = gx.Plan(len1, len2, CONFIG_TOML, False, traceback=True)
    assert plan.stat(27) == 2.0
    plan.close()


_RAGGED = {}


@pytest.mark.parametrize("mode", ["tickets", "resident"])
@pytest.mark.parametrize("chain1", [0, 1])
@pytest.mark.parametrize("k,r", KR_COMBOS)
@pytest.mark.gpu
def test_compact_kernel_ragged(gx, oracle, k, r, chain1, mode, monkeypatch):
    """the compact fill for every register tile, both recurrence forms, ticket and resident-strips scheduling, on ragged
    tables partly inside and partly outside a forced 300-column band: similar pairs stay inside, unrelated ones leave
    and widen"""
    force_kr(monkeypatch, k, r)
    monkeypatch.setenv("GX_CHAIN1", str(chain1))
    monkeypatch.setenv("GX_CODE_COMPACT", "1")
    monkeypatch.setenv("GX_CODE_BAND", "300")
    if mode == "tickets":
        monkeypatch.setenv("GX_TICKETS", "1")
    else:
        monkeypatch.setenv("GX_RESIDENT", "1")
    rng = np.random.default_rng(17)
    dims_sim = [(4200, 4200), (8193, 8193), (2000, 2000), (5000, 5000), (4096, 4096), (12000, 12000)]
    dims_any = [(4200, 4000), (4097, 5300), (8193, 7000), (2000, 2100), (5000, 4000), (4096, 4096), (700, 9000)]
    for similar in (True, False):
        pairs = [random_pair(rng, m, n, similar=similar, sub=0.1, indel=0.01) for m, n in (dims_sim if similar else dims_any)]
        plan, res, ops = _plan_run(gx, pairs)
        assert plan.stat(27) == 2.0 and plan.stat(21) == (1.0 if mode == "resident" else 0.0)
        if similar:
            assert plan.stat(23) < 0.9 and plan.stat(24) == 0, (plan.stat(23), plan.stat(24))
        for q, (a, b) in enumerate(pairs):
            key = (similar, q)
            if key not in _RAGGED:
                _RAGGED[key] = oracle.align_linear(a, b, CONFIG_TOML, False)
            o = _RAGGED[key]
            assert res["score"][q] == o.score and res["n_ops"][q] == len(o.ops), (k, chain1, mode, similar, q)
            assert np.array_equal(ops[q], o.ops), (k, chain1, mode, similar, q)
            assert (res["matches"][q], res["mismatches"][q], res["gap_extensions"][q], res["opening_gaps"][q]) == (
                o.matches, o.mismatches, o.gap_extensions, o.opening_gaps), (k, chain1, mode, similar, q)
        plan.close()


_WINDOW = {}


@pytest.mark.parametrize("rows", [64, 128, 256, 512])
@pytest.mark.parametrize("k,r", KR_COMBOS)
@pytest.mark.gpu
def test_compact_walk_window_sizes(gx, oracle, k, r, rows, monkeypatch):
    """the walk's loader on compact storage for every window height and strip width, with a 128-column band: windows
    it prefetches on the left and above lie partly outside the band, paths that wander out make the band widen"""
    force_kr(monkeypatch, k, r)
    monkeypatch.setenv("GX_WALK_ROWS", str(rows))
    monkeypatch.setenv("GX_CODE_COMPACT", "1")
    monkeypatch.setenv("GX_CODE_BAND", "128")
    rng = np.random.default_rng(23)
    pairs = [random_pair(rng, m, n, similar=True, sub=0.08, indel=0.02) for m, n in [(4300, 4250), (8200, 8300), (1500, 600), (700, 5000)]]
    a, b = random_pair(rng, 6000, 6000, similar=True, sub=0.05, indel=0.005)
    pairs += [(a, b[1500:4700]), (a[300:5100], b), (a[:4100], a[:4100]), (a[5000:], b[:900])]
    got = gx.align_batch(pairs, CONFIG_TOML, False)
    for x, ((s1, s2), res) in enumerate(zip(pairs, got)):
        if x not in _WINDOW:
            _WINDOW[x] = oracle.align_linear(s1, s2, CONFIG_TOML, False)
        _same(res, _WINDOW[x], f"pair {x} m={len(s1)} n={len(s2)} K={k} rows={rows}")


def _band_pairs():
    """the pairs of test_code_band_and_fallback: a 1500-base deletion, 2500 unrelated leading bases, substitutions only,
    the transposed deletion and a 200-base offset"""
    rng = np.random.default_rng(99)
    lut = np.frombuffer(b"ACGT", np.uint8)
    a = lut[rng.integers(0, 4, size=9000)]
    b1 = np.concatenate([a[:3000], a[4500:]])
    b2 = np.concatenate([lut[rng.integers(0, 4, size=2500)], a])
    b3 = a.copy(); b3[rng.choice(9000, 300, replace=False)] = lut[rng.integers(0, 4, size=300)]
    return [(a, b1), (a, b2), (a, b3), (b1, a), (a[:5000], a[200:5300])]


@pytest.mark.gpu
def test_compact_widening(gx, oracle, monkeypatch):
    """compact storage with a 64-column band: the walks that leave it make the execute repeat with a wider band for their
    pairs only -- results equal the oracle, the repeats are counted (stat 24), and the codes are fewer than if every pair
    had been widened to the widest band (the substitution-only pair stays at 64 columns)"""
    pairs = _band_pairs()
    exp = [oracle.align_linear(x, y, CONFIG_TOML, False) for x, y in pairs]
    dims = [(len(x), len(y)) for x, y in pairs]
    monkeypatch.setenv("GX_CODE_COMPACT", "1")
    monkeypatch.setenv("GX_CODE_BAND", "64")
    for mode in ("tickets", "resident"):
        if mode == "tickets":
            monkeypatch.setenv("GX_TICKETS", "1")
        else:
            monkeypatch.delenv("GX_TICKETS", raising=False)
        blob, off1, len1, off2, len2 = gx.pack_pairs(pairs)
        plan = gx.Plan(len1, len2, CONFIG_TOML, False, traceback=True)
        K = int(plan.stat(15))
        assert plan.stat(27) == 2.0 and plan.stat(28) == 64.0
        assert plan.stat(4) == _compact_bytes(dims, K, [64] * len(pairs))
        plan.upload(blob, off1, off2)
        for it in range(2):
            plan.execute()
            res, ops, ops_off = plan.fetch()
            for q, o in enumerate(exp):
                assert res["score"][q] == o.score and res["n_ops"][q] == len(o.ops), (mode, it, q)
                assert np.array_equal(ops[int(ops_off[q]):int(ops_off[q]) + len(o.ops)], o.ops), (mode, it, q)
                assert (res["end_i"][q], res["end_j"][q]) == tuple(o.end), (mode, it, q)
            if it == 0:
                assert plan.stat(24) >= 1
                widest = int(plan.stat(28))
                assert widest >= 128
                assert _compact_bytes(dims, K, [64] * len(pairs)) < plan.stat(4) < _compact_bytes(dims, K, [widest] * len(pairs))
            else:
                assert plan.stat(28) == widest      # the widths persist: the second execute needs no repeat
        n_rep = plan.stat(24)
        plan.execute()
        assert plan.stat(24) == n_rep
        plan.close()


@pytest.mark.gpu
def test_code_budget(gx, oracle, monkeypatch):
    """GX_CODE_BUDGET below what the widened band needs: the execute returns GX_ERR_NOMEM (7) naming the pair, the
    half-width and the bytes, never a wrong result; below the dense codes of a plan that cannot take compact storage (a
    local plan, or the code band off) plan creation returns it with the reason.  The device stays usable."""
    from genomics_rs_b200 import _lib
    pairs = _band_pairs()
    blob, off1, len1, off2, len2 = gx.pack_pairs(pairs)
    monkeypatch.setenv("GX_CODE_BAND", "64")
    monkeypatch.setenv("GX_CODE_COMPACT", "1")
    plan = gx.Plan(len1, len2, CONFIG_TOML, False, traceback=True)
    need64 = int(plan.stat(4))
    plan.close()
    monkeypatch.delenv("GX_CODE_COMPACT")
    monkeypatch.setenv("GX_CODE_BUDGET", str(need64))     # dense codes exceed it: compact storage, at 64 columns it fits
    plan = gx.Plan(len1, len2, CONFIG_TOML, False, traceback=True)
    assert plan.stat(27) == 2.0 and plan.stat(4) == need64
    plan.upload(blob, off1, off2)
    with pytest.raises(_lib.GxError) as e:
        plan.execute()
    assert e.value.status == 7
    msg = str(e.value)
    assert "pair" in msg and "half-width" in msg and "bytes" in msg and "GX_CODE_BUDGET" in msg, msg
    with pytest.raises(_lib.GxError) as e:              # the plan has no codes buffer now: it refuses to run
        plan.execute()
    assert e.value.status == 7
    plan.close()
    for env, local, why in ((("GX_CODE_BAND", "64"),), True, "local"), ((("GX_CODE_BAND", "0"),), False, "GX_CODE_BAND=0"):
        for kv in env:
            monkeypatch.setenv(*kv)
        monkeypatch.setenv("GX_CODE_BUDGET", "4096")
        with pytest.raises(_lib.GxError) as e:
            gx.Plan(len1, len2, CONFIG_TOML, local, traceback=True)
        assert e.value.status == 7 and why in str(e.value), str(e.value)
    monkeypatch.delenv("GX_CODE_BUDGET")
    monkeypatch.delenv("GX_CODE_BAND")
    r = gx.align_batch(pairs, CONFIG_TOML, False)
    for (x, y), got in zip(pairs, r):
        _same(got, oracle.align_linear(x, y, CONFIG_TOML, False))
