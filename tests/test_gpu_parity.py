"""GPU parity tests: the CUDA path (through the C ABI / the reference-shaped host mirror) against the
oracle and the committed golden vectors.  Integer work: every comparison is bit-exact."""
import numpy as np
import pytest

from conftest import CONFIG_TOML, KR_COMBOS, TEST_CONFIG, force_kr, random_pair, read_fasta_gz

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gx():
    import genomics_rs_b200 as gx
    from genomics_rs_b200 import _lib
    _lib.ensure_init()
    return gx


def _container(gx, s1, s2):
    return gx.SequenceContainer(sequences=[gx.Sequence("s1", s1), gx.Sequence("s2", s2)])


def _same(gpu, ora, oracle, what=""):
    assert gpu.score == ora.score, what
    assert tuple(gpu.start) == tuple(ora.start), what
    assert tuple(gpu.end) == tuple(ora.end), what
    assert (gpu.matches, gpu.mismatches, gpu.gap_extensions, gpu.opening_gaps) == (
        ora.matches, ora.mismatches, ora.gap_extensions, ora.opening_gaps), what
    assert np.array_equal(gpu.ops, ora.ops), what
    oi, oj = gpu.coords()
    assert np.array_equal(oi, ora.ops_i) and np.array_equal(oj, ora.ops_j), what


# ---- the reference's own tests (tests/test_alignment.rs:23-139), written the way the reference writes them
def test_reference_test_simple_matches(gx):
    sc = _container(gx, "ACGT", "ACGT")
    scores = gx.Scores(1, -2, -2, -5)
    table, _ = gx.alignment_table(sc, scores, False, False)
    aligned = gx.retrace(sc, table, False)
    M = gx.AlignmentChoice.Match
    assert aligned.score == 4
    assert (aligned.matches, aligned.mismatches, aligned.opening_gaps, aligned.gap_extensions) == (4, 0, 0, 0)
    assert aligned.alignment == [(M, 4, 4), (M, 3, 3), (M, 2, 2), (M, 1, 1)]


def test_reference_test_gaps(gx):
    sc = _container(gx, "ACGT", "AGCGT")
    table, _ = gx.alignment_table(sc, gx.Scores(1, -2, -2, -5), False, False)
    aligned = gx.retrace(sc, table, False)
    C = gx.AlignmentChoice
    assert (aligned.matches, aligned.mismatches, aligned.opening_gaps, aligned.gap_extensions) == (3, 1, 1, 0)
    assert aligned.alignment == [(C.Match, 4, 5), (C.Match, 3, 4), (C.Match, 2, 3), (C.OpenInsert, 1, 2), (C.Mismatch, 1, 1)]
    assert str(aligned).startswith("\n\n0-5:\n\nA-CGT\nx%|||\nAGCGT\n")


def test_reference_test_affine_gap(gx, ref_vectors):
    case = ref_vectors["cases"][2]
    sc = _container(gx, case["s1"], case["s2"])
    table, _ = gx.alignment_table(sc, gx.Scores(1, -2, -2, -5), False, False)
    aligned = gx.retrace(sc, table, False)
    assert (aligned.matches, aligned.mismatches, aligned.opening_gaps, aligned.gap_extensions) == (12, 0, 1, 3)
    assert [[c.name, i, j] for c, i, j in aligned.alignment] == case["alignment"]


# ---- fixtures vs committed goldens and vs the oracle, global and local (configs 1 and 2 of BASELINE.json)
@pytest.mark.parametrize("fixture", ["test1", "test2_short", "test3_short", "test4", "Opsin1_colorblindness_gene",
                                     "Human-Mouse-BRCA2-cds"])
@pytest.mark.parametrize("is_local", [False, True])
def test_fixture_parity(gx, oracle, goldens, fixture, is_local):
    g = next(p for p in goldens["pairs"] if p["fixture"] == fixture and p["is_local"] == is_local)
    s = read_fasta_gz(fixture)
    sc = gx.SequenceContainer(sequences=[gx.Sequence(*s[0]), gx.Sequence(*s[1])])
    a = gx.align(sc, gx.Scores(*CONFIG_TOML), is_local)
    assert a.score == g["score"] and list(a.start) == g["start"] and list(a.end) == g["end"]
    assert len(a.ops) == g["n_ops"]
    assert (a.matches, a.mismatches, a.gap_extensions, a.opening_gaps) == (
        g["matches"], g["mismatches"], g["gap_extensions"], g["opening_gaps"])
    assert "%016x" % oracle.hash_ops(a.ops, a.start) == g["op_hash"]
    o = oracle.align_linear(s[0][1], s[1][1], CONFIG_TOML, is_local)
    _same(a, o, oracle, fixture)


def test_edge_cases(gx, oracle):
    cases = [("", ""), ("", "ACG"), ("ACG", ""), ("A", "A"), ("A", "C"), ("AAAA", "TTTT"), ("ACGT" * 70, "ACGT" * 70),
             ("A" * 257, "A" * 256), ("ACGTTGCA" * 40, "TTTT"), ("G", "ACGT" * 100), ("\x00\xff\x80A", "\x00\xffA\x80")]
    for scores in (CONFIG_TOML, TEST_CONFIG, (2, 1, -1, 0)):
        for is_local in (False, True):
            pairs = [(a.encode("latin-1"), b.encode("latin-1")) for a, b in cases]
            got = gx.align_batch(pairs, scores, is_local)
            for (a, b), r in zip(pairs, got):
                o = oracle.align_faithful(a, b, scores, is_local)
                _same(r, o, oracle, f"{a[:12]!r} {b[:12]!r} {scores} local={is_local}")


@pytest.mark.parametrize("k,r", [(0, 0)] + KR_COMBOS)
@pytest.mark.parametrize("chain1", [0, 1])
def test_local_all_zero_table(gx, oracle, k, r, chain1, monkeypatch):
    """a local table whose maximum is 0: score 0, start (m, n) -- the LAST cell in row-major order (algo.rs:311-322) --
    and the run-on walk from there.  Shapes where a padded column right of the table runs through an unmasked batch
    (n mod 32K in [1, K-1], rows a multiple of the batch) for every register blocking and both recurrence forms."""
    if k:
        force_kr(monkeypatch, k, r)
    monkeypatch.setenv("GX_CHAIN1", str(chain1))
    pairs = [(b"A" * 64, b"C"), (b"A" * 4096, b"C"), (b"A" * 8192, b"CC"), (b"A" * 64, b"C" * 3), (b"A" * 128, b"C" * 129),
             (b"A" * 256, b"C" * 513), (b"A" * 32, b"C" * 5), (b"A" * 31, b"C"), (b"A" * 4160, b"C" * 7), (b"AC" * 40, b"GT" * 33)]
    for scores in (CONFIG_TOML, TEST_CONFIG):
        for traceback in (True, False):
            got = gx.align_batch(pairs, scores, True, traceback=traceback, start_cell=True)
            for (a, b), r in zip(pairs, got):
                o = oracle.align_linear(a, b, scores, True)
                assert r.score == 0 == o.score
                assert tuple(r.start) == (len(a), len(b)) == tuple(o.start), (len(a), len(b), k, chain1)
                if traceback:
                    _same(r, o, oracle, f"m={len(a)} n={len(b)} K={k} chain1={chain1}")


# scoring -> whether it takes the IDP.4A path: a, b, a-(h+g) and b-(h+g) must all fit a signed byte
_BYTE_PATH = {(120, -100, -20, -30): False, (127, -128, -1, 0): False, (60, -70, -50, -9): True, (-3, -7, -2, -4): True,
              (120, -5, -3, -4): True, (121, -5, -3, -4): False,        # a-(h+g) = 127 / 128
              (5, -128, -1, 0): True, (5, -129, -2, 0): False,          # b = -128 / -129
              (3, -130, -1, -1): False, (3, -131, -1, -1): False}       # b-(h+g) = -128 / -129 (b itself is out of range)


@pytest.mark.parametrize("scores", list(_BYTE_PATH))
def test_score_byte_range_paths(gx, oracle, scores):
    """4-letter batches score through one IDP.4A per cell when (score - (h+g)) fits a signed byte and through the compare
    path otherwise: scorings on both sides of each edge of that range (and an all-negative one) against the faithful
    oracle, and the path the plan took (gx_plan_stat 25)"""
    rng = np.random.default_rng(sum(scores) & 0xffff)
    pairs = [random_pair(rng, int(rng.integers(1, 90)), int(rng.integers(1, 90)), similar=bool(k % 2)) for k in range(120)]
    pairs += [random_pair(rng, 300, 520), random_pair(rng, 4100, 140)]
    for is_local in (False, True):
        got = gx.align_batch(pairs, scores, is_local)
        for (a, b), r in zip(pairs, got):
            o = oracle.align_faithful(a, b, scores, is_local) if len(a) < 1000 else oracle.align_linear(a, b, scores, is_local)
            _same(r, o, oracle, f"m={len(a)} n={len(b)} {scores} local={is_local}")
        blob, off1, len1, off2, len2 = gx.pack_pairs(pairs)
        plan = gx.Plan(len1, len2, scores, is_local, traceback=False)
        plan.upload(blob, off1, off2)
        assert plan.stat(25) == float(_BYTE_PATH[scores]), (scores, is_local)
        plan.close()


@pytest.mark.parametrize("scores", [CONFIG_TOML, TEST_CONFIG, (2, -1, -1, 0), (5, -4, -3, -10), (1, 0, -1, -1), (3, 1, -2, -2)])
def test_random_small_vs_faithful(gx, oracle, scores):
    rng = np.random.default_rng(hash(scores) & 0xffff)
    pairs = []
    for _ in range(200):
        m, n = int(rng.integers(0, 70)), int(rng.integers(0, 70))
        pairs.append(random_pair(rng, m, n, alphabet=b"ACGT" if rng.random() < 0.7 else b"AC", similar=bool(rng.integers(0, 2))))
    for is_local in (False, True):
        got = gx.align_batch(pairs, scores, is_local)
        for (a, b), r in zip(pairs, got):
            o = oracle.align_faithful(a, b, scores, is_local)
            _same(r, o, oracle, f"m={len(a)} n={len(b)} {scores} local={is_local}")


_RAGGED_ORACLE = {}


@pytest.mark.parametrize("chain1", [0, 1])
@pytest.mark.parametrize("k,r", KR_COMBOS)
def test_random_medium_ragged_vs_linear(gx, oracle, k, r, chain1, monkeypatch):
    """sizes that cross strip (32*K columns), batch (up to 32 rows) and panel (4096 rows) boundaries, for every
    K the library can pick (GX_K forces it) and both forms of the recurrence"""
    force_kr(monkeypatch, k, r)
    monkeypatch.setenv("GX_CHAIN1", str(chain1))
    rng = np.random.default_rng(11)
    dims = [(255, 256), (256, 257), (257, 255), (31, 600), (33, 1025), (1000, 31), (513, 513), (4095, 300), (4096, 300),
            (4097, 300), (4200, 520), (300, 4200), (8193, 770), (1, 3000), (3000, 1), (127, 129), (129, 127), (511, 512),
            (64, 1030), (2, 70), (3, 513), (5, 5), (7, 260), (4094, 140), (4099, 130), (8190, 40), (8197, 33), (33, 4100)]
    pairs = [random_pair(rng, m, n, similar=(x % 3 != 0)) for x, (m, n) in enumerate(dims)]
    for is_local in (False, True):
        got = gx.align_batch(pairs, CONFIG_TOML, is_local)
        for x, ((a, b), res) in enumerate(zip(pairs, got)):
            if (x, is_local) not in _RAGGED_ORACLE:     # the same seeded pairs for every (K, R, form): one oracle run each
                _RAGGED_ORACLE[(x, is_local)] = oracle.align_linear(a, b, CONFIG_TOML, is_local)
            _same(res, _RAGGED_ORACLE[(x, is_local)], oracle, f"m={len(a)} n={len(b)} local={is_local} K={k} R={r} chain1={chain1}")


def test_score_only_and_start_cell(gx, oracle):
    rng = np.random.default_rng(5)
    pairs = [random_pair(rng, int(rng.integers(1, 900)), int(rng.integers(1, 900))) for _ in range(40)]
    for is_local in (False, True):
        got = gx.align_batch(pairs, CONFIG_TOML, is_local, traceback=False, start_cell=True)
        for (a, b), r in zip(pairs, got):
            sc, si, sj = oracle.score_linear(a, b, CONFIG_TOML, is_local)
            assert r.score == sc and tuple(r.start) == (si, sj)
        got = gx.align_batch(pairs, CONFIG_TOML, is_local, traceback=False)
        for (a, b), r in zip(pairs, got):
            assert r.score == oracle.score_linear(a, b, CONFIG_TOML, is_local)[0]


@pytest.mark.parametrize("k,r", KR_COMBOS)
@pytest.mark.parametrize("is_local", [False, True])
def test_brca2_other_blockings(gx, oracle, goldens, k, r, is_local, monkeypatch):
    force_kr(monkeypatch, k, r)
    g = next(p for p in goldens["pairs"] if p["fixture"] == "Human-Mouse-BRCA2-cds" and p["is_local"] == is_local)
    s = read_fasta_gz("Human-Mouse-BRCA2-cds")
    a = gx.align_batch([(s[0][1], s[1][1])], CONFIG_TOML, is_local)[0]
    assert a.score == g["score"] and list(a.start) == g["start"] and list(a.end) == g["end"] and len(a.ops) == g["n_ops"]
    assert "%016x" % oracle.hash_ops(a.ops, a.start) == g["op_hash"]


def test_plan_reexecute_is_idempotent(gx, oracle):
    """the LL parity protocol must survive repeated executes of one plan (bench.py re-runs plans)"""
    rng = np.random.default_rng(9)
    pairs = [random_pair(rng, 1500, 1300), random_pair(rng, 700, 2100)]
    blob, off1, len1, off2, len2 = gx.pack_pairs(pairs)
    plan = gx.Plan(len1, len2, CONFIG_TOML, False, traceback=True)
    plan.upload(blob, off1, off2)
    ref = None
    for _ in range(5):
        plan.execute()
        res, ops, ops_off = plan.fetch()
        cur = (res["score"].tolist(), res["n_ops"].tolist(), ops.tobytes())
        if ref is None:
            ref = cur
            for q, (a, b) in enumerate(pairs):
                o = oracle.align_linear(a, b, CONFIG_TOML, False)
                assert res["score"][q] == o.score
                k = int(res["n_ops"][q])
                assert np.array_equal(ops[int(ops_off[q]):int(ops_off[q]) + k], o.ops)
        assert cur == ref
    plan.close()


def test_resident_abort_falls_back_to_tickets(gx, oracle, monkeypatch):
    """a resident-strips execute that gives up waiting (SPIN_LIMIT) is repeated once in ticket mode: same results,
    the plan stays usable (GX_TEST_ABORT fakes the abort word of the first execute)"""
    rng = np.random.default_rng(3)
    pairs = [random_pair(rng, 5000, 3000), random_pair(rng, 900, 2500)]
    blob, off1, len1, off2, len2 = gx.pack_pairs(pairs)
    monkeypatch.setenv("GX_TEST_ABORT", "1")
    plan = gx.Plan(len1, len2, CONFIG_TOML, False, traceback=True)
    monkeypatch.delenv("GX_TEST_ABORT")
    plan.upload(blob, off1, off2)
    assert plan.stat(21) == 1.0                       # few strips: resident mode (cooperative launch)
    for it in range(3):
        plan.execute()
        assert plan.stat(20) == 1.0 and plan.stat(21) == 0.0   # retried once, ticket mode from then on
        res, ops, ops_off = plan.fetch()
        for q, (a, b) in enumerate(pairs):
            o = oracle.align_linear(a, b, CONFIG_TOML, False)
            assert res["score"][q] == o.score
            assert np.array_equal(ops[int(ops_off[q]):int(ops_off[q]) + int(res["n_ops"][q])], o.ops)
    plan.close()


def test_code_band_and_fallback(gx, oracle, monkeypatch):
    """global traceback plans write direction codes only near the table's diagonal; a path that leaves the band makes the
    execute repeat with codes everywhere -- results are exact either way.  Pairs with a long terminal gap / big indels
    against a forced 64-column band (fallback must fire), the same pairs with the default band and with the band off."""
    rng = np.random.default_rng(99)
    lut = np.frombuffer(b"ACGT", np.uint8)
    a = lut[rng.integers(0, 4, size=9000)]
    b1 = np.concatenate([a[:3000], a[4500:]])                                    # one 1500-base deletion
    b2 = np.concatenate([lut[rng.integers(0, 4, size=2500)], a])                 # 2500 unrelated leading bases
    b3 = a.copy(); b3[rng.choice(9000, 300, replace=False)] = lut[rng.integers(0, 4, size=300)]   # substitutions only
    pairs = [(a, b1), (a, b2), (a, b3), (b1, a), (a[:5000], a[200:5300])]
    exp = [oracle.align_linear(x, y, CONFIG_TOML, False) for x, y in pairs]
    blob, off1, len1, off2, len2 = gx.pack_pairs(pairs)
    monkeypatch.setenv("GX_TICKETS", "1")
    for band, want_fallback in (("64", True), (None, None), ("0", False), ("64r", True)):
        if band == "64r":                       # the same through resident strips (cooperative launch)
            monkeypatch.delenv("GX_TICKETS", raising=False)
            band = "64"
        if band is None:
            monkeypatch.delenv("GX_CODE_BAND", raising=False)
        else:
            monkeypatch.setenv("GX_CODE_BAND", band)
        plan = gx.Plan(len1, len2, CONFIG_TOML, False, traceback=True)
        plan.upload(blob, off1, off2)
        for _ in range(2):
            plan.execute()
            res, ops, ops_off = plan.fetch()
            for q, o in enumerate(exp):
                assert res["score"][q] == o.score and res["n_ops"][q] == len(o.ops), (band, q)
                assert np.array_equal(ops[int(ops_off[q]):int(ops_off[q]) + len(o.ops)], o.ops), (band, q)
        if want_fallback is not None:
            assert (plan.stat(24) >= 1) == want_fallback, (band, plan.stat(24))
        if band == "0":
            assert plan.stat(23) == 1.0
        plan.close()
    monkeypatch.delenv("GX_CODE_BAND", raising=False)
    monkeypatch.delenv("GX_TICKETS", raising=False)


@pytest.mark.parametrize("chain1", [0, 1])
@pytest.mark.parametrize("k,r", KR_COMBOS)
def test_code_band_kernel_ragged(gx, oracle, k, r, chain1, monkeypatch):
    """the two-variant (code band) fill kernel for every register tile and both recurrence forms, on ragged tables whose
    tiles are partly inside and partly outside a forced 300-column band; similar pairs stay inside it, unrelated ones
    wander out and take the fallback"""
    force_kr(monkeypatch, k, r)
    monkeypatch.setenv("GX_CHAIN1", str(chain1))
    monkeypatch.setenv("GX_TICKETS", "1")
    monkeypatch.setenv("GX_CODE_BAND", "300")
    rng = np.random.default_rng(17)
    # equal-length similar pairs keep their path within a few dozen columns of the diagonal; ragged / unrelated ones do not
    dims_sim = [(4200, 4200), (8193, 8193), (2000, 2000), (5000, 5000), (4096, 4096), (12000, 12000)]
    dims_any = [(4200, 4000), (4097, 5300), (8193, 7000), (2000, 2100), (5000, 4000), (4096, 4096), (700, 9000)]
    for similar in (True, False):
        pairs = [random_pair(rng, m, n, similar=similar, sub=0.1, indel=0.01) for m, n in (dims_sim if similar else dims_any)]
        blob, off1, len1, off2, len2 = gx.pack_pairs(pairs)
        plan = gx.Plan(len1, len2, CONFIG_TOML, False, traceback=True)
        plan.upload(blob, off1, off2)
        plan.execute()
        res, ops, ops_off = plan.fetch()
        if similar:
            assert plan.stat(23) < 0.9 and plan.stat(24) == 0, (plan.stat(23), plan.stat(24))   # band in use, no fallback
        for q, (a, b) in enumerate(pairs):
            o = oracle.align_linear(a, b, CONFIG_TOML, False)
            assert res["score"][q] == o.score and res["n_ops"][q] == len(o.ops), (k, chain1, similar, q)
            assert np.array_equal(ops[int(ops_off[q]):int(ops_off[q]) + len(o.ops)], o.ops), (k, chain1, similar, q)
        plan.close()


_WINDOW_ORACLE = {}


@pytest.mark.parametrize("rows", [64, 128, 256, 512])
@pytest.mark.parametrize("k,r", KR_COMBOS)
def test_walk_window_sizes(gx, oracle, k, r, rows, monkeypatch):
    """the walk's code windows (GX_WALK_ROWS forces their height) for every strip width: paths that cross strip and panel
    (4096 rows) boundaries, leave a window on the left and at the top, run along long gaps (one sequence a fragment of the
    other: hundreds of consecutive Insert / Delete ops) and end on row 0 / column 0"""
    force_kr(monkeypatch, k, r)
    monkeypatch.setenv("GX_WALK_ROWS", str(rows))
    rng = np.random.default_rng(23)
    pairs = [random_pair(rng, m, n, similar=True, sub=0.08, indel=0.02) for m, n in [(4300, 4250), (8200, 8300), (1500, 600), (700, 5000)]]
    a, b = random_pair(rng, 6000, 6000, similar=True, sub=0.05, indel=0.005)
    pairs += [(a, b[1500:4700]), (a[300:5100], b), (a[:4100], a[:4100]), (a[5000:], b[:900])]
    for is_local in (False, True):
        got = gx.align_batch(pairs, CONFIG_TOML, is_local)
        for x, ((s1, s2), res) in enumerate(zip(pairs, got)):
            if (x, is_local) not in _WINDOW_ORACLE:
                _WINDOW_ORACLE[(x, is_local)] = oracle.align_linear(s1, s2, CONFIG_TOML, is_local)
            _same(res, _WINDOW_ORACLE[(x, is_local)], oracle, f"pair {x} m={len(s1)} n={len(s2)} local={is_local} K={k} rows={rows}")


def test_corona_all_vs_all(gx, oracle, goldens):
    """BASELINE config 3: 45 pairs of ~30 kb genomes, global, score + traceback, one batch."""
    order = goldens["corona_order"]
    seqs = [read_fasta_gz(name)[0][1] for name in order]
    jobs = [(a, b) for a in range(len(seqs)) for b in range(a + 1, len(seqs))]
    got = gx.align_batch([(seqs[a], seqs[b]) for a, b in jobs], CONFIG_TOML, False)
    gold = {tuple(c["pair"]): c for c in goldens["corona"]}
    for (a, b), r in zip(jobs, got):
        g = gold[(a, b)]
        assert r.score == g["score"], (a, b)
        assert len(r.ops) == g["n_ops"], (a, b)
        assert (r.matches, r.mismatches, r.gap_extensions, r.opening_gaps) == (
            g["matches"], g["mismatches"], g["gap_extensions"], g["opening_gaps"]), (a, b)
        assert "%016x" % oracle.hash_ops(r.ops, r.start) == g["op_hash"], (a, b)


def test_matches_at_max(gx, oracle, goldens):
    """alignment_table's second return value (algo.rs:279-281): max_matches (the LCS-length lanes, algo.rs:112-121,
    250-255) at the FIRST cell attaining the table maximum (algo.rs:258-262) -- against the faithful oracle on random
    pairs (ties are frequent in small tables) and against the goldens of every fixture, global and local"""
    for scores in (CONFIG_TOML, TEST_CONFIG, (2, -1, -1, 0)):
        rng = np.random.default_rng(31 + scores[0])
        pairs = [random_pair(rng, int(rng.integers(0, 90)), int(rng.integers(0, 90)), alphabet=b"ACGT" if k % 3 else b"AC",
                             similar=bool(k % 2)) for k in range(150)]
        pairs += [random_pair(rng, m, n) for m, n in ((700, 900), (4100, 300), (300, 4200), (2500, 2600))]
        pairs += [(b"\x00\xff\x80ABCDEFG" * 9, b"\xffA\x80CDXFG\x00" * 11)]
        for is_local in (False, True):
            got = gx.align_batch(pairs, scores, is_local, lcs_at_max=True)
            for (a, b), r in zip(pairs, got):
                o = oracle.align_faithful(a, b, scores, is_local)
                assert r.matches_at_max == o.lcs_at_first_max, (len(a), len(b), scores, is_local, o.first_max)
                assert r.score == o.score and np.array_equal(r.ops, o.ops)      # the extra passes leave the alignment alone
    for fixture in ("test1", "test2_short", "test3_short", "test4", "Opsin1_colorblindness_gene", "Human-Mouse-BRCA2-cds"):
        s = read_fasta_gz(fixture)
        for is_local in (False, True):
            g = next(p for p in goldens["pairs"] if p["fixture"] == fixture and p["is_local"] == is_local)
            sc = gx.SequenceContainer(sequences=[gx.Sequence(*s[0]), gx.Sequence(*s[1])])
            table, second = gx.alignment_table(sc, gx.Scores(*CONFIG_TOML), is_local, False, matches_at_max=True)
            assert second == g["lcs_at_first_max"], (fixture, is_local)
            assert gx.retrace(sc, table, is_local).score == g["score"]
    # tables wider than one 32768-column block of the bit-vector pass: the local maximum sits behind column 40000
    rng = np.random.default_rng(77)
    lut = np.frombuffer(b"ACGT", np.uint8)
    a = lut[rng.integers(0, 4, size=3000)]
    core = a.copy()
    idx = rng.choice(3000, size=150, replace=False)
    core[idx] = lut[rng.integers(0, 4, size=150)]
    b = np.concatenate([lut[rng.integers(0, 4, size=40000)], core[:1400], core[1430:], lut[rng.integers(0, 4, size=27000)]])
    for is_local in (True, False):
        r = gx.align_batch([(a, b)], CONFIG_TOML, is_local, traceback=False, lcs_at_max=True)[0]
        o = oracle.align_linear(a, b, CONFIG_TOML, is_local, traceback=False)
        assert r.score == o.score
        assert r.matches_at_max == o.lcs_at_first_max, (is_local, o.first_max, o.lcs_at_first_max)
        if is_local:
            assert o.first_max[1] > 32768


def test_align_all_directory(gx, goldens, tmp_path):
    """SURVEY 8f N3: directory ingestion + all-vs-all through one batch call, Python mirror and the C++ CLI"""
    import gzip, os, subprocess
    order = goldens["corona_order"][:3]
    for name in order:
        raw = gzip.open(os.path.join(os.path.dirname(__file__), "golden", "fasta", name + ".fasta.gz"), "rb").read()
        (tmp_path / (name + ".fasta")).write_bytes(raw)
    sc = gx.SequenceContainer()
    sc.from_fasta_dir(str(tmp_path))
    assert len(sc.sequences) == 3
    gold = {tuple(c["pair"]): c for c in goldens["corona"]}
    res = gx.align_all(sc, gx.Scores(*CONFIG_TOML), False)
    assert [j for j, _ in res] == [(0, 1), (0, 2), (1, 2)]
    for (a, b), r in res:
        g = gold[(a, b)]
        assert r.score == g["score"] and len(r.ops) == g["n_ops"] and r.matches == g["matches"]
    cli = os.path.join(os.path.dirname(os.path.dirname(__file__)), "genomics_rs_b200", "host", "gxalign_cli")
    if os.path.exists(cli):
        cfg = tmp_path / "config.toml"
        cfg.write_text("[scores]\ns_match = 1\ns_mismatch = -2\ng = -1\nh = -5\n")
        out = subprocess.run([cli, "--config-path", str(cfg), "align-all", "-a", "global", "--fasta-dir", str(tmp_path)],
                             capture_output=True, text=True, timeout=300)
        assert out.returncode == 0, out.stderr
        rows = [ln.split("\t") for ln in out.stdout.splitlines() if ln and not ln.startswith("#")][1:]
        assert [int(r[2]) for r in rows] == [gold[p]["score"] for p in ((0, 1), (0, 2), (1, 2))]


def test_score_planes_visualiser(gx, oracle, capsys):
    """SURVEY 8f N4: the insert/delete/sub planes the reference's small-table visualiser prints (display.rs:131-220)"""
    rng = np.random.default_rng(12)
    cases = [(b"ACGT", b"AGCGT"), (b"", b"ACG"), (b"A", b""), (b"", b"")]
    cases += [random_pair(rng, int(rng.integers(1, 199)), int(rng.integers(1, 400))) for _ in range(12)]
    for scores in (CONFIG_TOML, TEST_CONFIG):
        for is_local in (False, True):
            for a, b in cases:
                got = gx.score_planes(a, b, scores, is_local)
                exp = oracle.planes(a, b, scores, is_local)
                for g_, e_ in zip(got, exp):
                    assert np.array_equal(g_, e_), (len(a), len(b), scores, is_local)
    from genomics_rs_b200 import _lib
    with pytest.raises(_lib.GxError):
        gx.score_planes(b"A" * 200, b"A", CONFIG_TOML, False)          # the reference refuses these sizes too
    sc = _container(gx, "ACGT", "AGCGT")
    table, _ = gx.alignment_table(sc, gx.Scores(1, -2, -2, -5), False, False)
    gx.retrace(sc, table, False, print_table=True)
    out = capsys.readouterr().out
    assert "Sequence Table (S1 columns, S2 rows):" in out and "AXI..." in out and "Sub Scores" in out


def test_read_batch_scores(gx, oracle):
    """BASELINE config 4 shape: many 150 bp pairs, local score only (inter-task kernel), plus ragged lengths."""
    rng = np.random.default_rng(150)
    n_pairs = 20000
    pairs = [random_pair(rng, 150, 150, similar=(k % 4 != 0), sub=0.06, indel=0.01) for k in range(n_pairs)]
    blob, off1, len1, off2, len2 = gx.pack_pairs(pairs)
    for is_local in (True, False):
        got = gx.score_batch(blob, off1, len1, off2, len2, CONFIG_TOML, is_local)
        exp = oracle.score_batch(blob, off1, len1, off2, len2, CONFIG_TOML, is_local, n_threads=8)
        assert np.array_equal(got, exp)
    ragged = [random_pair(rng, int(rng.integers(0, 152)), int(rng.integers(0, 152))) for _ in range(5000)]
    ragged += [random_pair(rng, int(rng.integers(100, 600)), int(rng.integers(100, 600))) for _ in range(1500)]
    blob, off1, len1, off2, len2 = gx.pack_pairs(ragged)
    for is_local in (True, False):
        got = gx.score_batch(blob, off1, len1, off2, len2, TEST_CONFIG, is_local)
        exp = oracle.score_batch(blob, off1, len1, off2, len2, TEST_CONFIG, is_local, n_threads=8)
        assert np.array_equal(got, exp)


def test_config4_parity_sets(gx, oracle):
    """BASELINE config 4 as SURVEY 8d specifies its parity: EVERY score of the parity set's first 100 000 pairs
    (s2 = s1 with 1/16 substitutions) and a strided 1 % of the 10 M-pair throughput set, local SW score only --
    against the oracle run here and against the frozen fixture (tests/golden/config4_scores.npz), through the streamed
    host-buffer entry point and through a resident plan; the first pairs also against the FAITHFUL oracle variant."""
    import os
    from genomics_rs_b200 import workloads as wl
    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "config4_scores.npz"))
    sets = {"parity": wl.reads150(0, wl.CONFIG4_PARITY_PAIRS, parity_set=True),
            "strided": wl.reads150_pairs(np.arange(0, 10_000_000, wl.CONFIG4_STRIDE, dtype=np.uint64))}
    for name, (blob, off1, len1, off2, len2) in sets.items():
        exp = oracle.score_batch(blob, off1, len1, off2, len2, CONFIG_TOML, True, n_threads=8)
        assert np.array_equal(exp, gold[name].astype(np.int64)), name
        got = gx.score_batch(blob, off1, len1, off2, len2, CONFIG_TOML, True)                 # plan path (< 2^18 pairs)
        assert np.array_equal(got, exp), name
        plan = gx.Plan(len1, len2, CONFIG_TOML, True, traceback=False)
        plan.upload(blob, off1, off2)
        plan.execute()
        assert np.array_equal(plan.fetch_scores(), exp), name
        plan.close()
        for q in range(0, 300, 7):
            a = blob[int(off1[q]):int(off1[q]) + 150]
            b = blob[int(off2[q]):int(off2[q]) + 150]
            assert oracle.align_faithful(a, b, CONFIG_TOML, True).score == int(got[q]), (name, q)
    # the streamed path (>= 2^18 pairs): parity set followed by the strided set followed by the parity set again
    blobs = [sets["parity"], sets["strided"], sets["parity"]]
    blob = np.concatenate([b[0] for b in blobs])
    base = np.cumsum([0] + [b[0].size for b in blobs[:-1]]).astype(np.uint64)
    off1 = np.concatenate([b[1] + o for b, o in zip(blobs, base)])
    off2 = np.concatenate([b[3] + o for b, o in zip(blobs, base)])
    len1 = np.concatenate([b[2] for b in blobs])
    len2 = np.concatenate([b[4] for b in blobs])
    got = gx.score_batch(blob, off1, len1, off2, len2, CONFIG_TOML, True)
    exp = np.concatenate([gold["parity"], gold["strided"], gold["parity"]]).astype(np.int64)
    assert got.size >= (1 << 18) and np.array_equal(got, exp)


def test_read_stream_scores(gx, oracle):
    """large read sets take the streamed path of gx_score_batch (chunks of 2^20 pairs through two copy/compute lanes):
    more than one chunk, ragged lengths, both modes, offsets that are not multiples of anything"""
    rng = np.random.default_rng(4242)
    lut = np.frombuffer(b"ACGT", np.uint8)
    n_pairs = (1 << 20) + 70001
    lens1 = rng.integers(0, 61, size=n_pairs).astype(np.uint64)
    lens2 = rng.integers(0, 61, size=n_pairs).astype(np.uint64)
    lens1[:4] = (0, 0, 60, 1); lens2[:4] = (0, 60, 0, 1)
    tot = np.zeros(2 * n_pairs + 1, np.uint64)
    inter = np.empty(2 * n_pairs, np.uint64); inter[0::2] = lens1; inter[1::2] = lens2
    np.cumsum(inter, out=tot[1:])
    off1, off2 = tot[0:-1:2].copy(), tot[1::2].copy()
    blob = lut[rng.integers(0, 4, size=int(tot[-1]))]
    # make half of the pairs similar: copy s1 into s2 where the lengths allow, then mutate a few bases
    for q in range(0, n_pairs, 2):
        k = int(min(lens1[q], lens2[q]))
        if k:
            blob[int(off2[q]):int(off2[q]) + k] = blob[int(off1[q]):int(off1[q]) + k]
    idx = rng.integers(0, blob.size, size=blob.size // 16)
    blob[idx] = lut[rng.integers(0, 4, size=idx.size)]
    for is_local, scores in ((True, CONFIG_TOML), (False, TEST_CONFIG)):
        got = gx.score_batch(blob, off1, lens1, off2, lens2, scores, is_local)
        exp = oracle.score_batch(blob, off1, lens1, off2, lens2, scores, is_local, n_threads=8)
        assert np.array_equal(got, exp)


def test_large_properties(gx, oracle):
    """size-independent properties at sizes the oracle does not brute-force:
    identical sequences give m*match with an all-Match walk; transposing the pair (I <-> D) keeps the
    global and the local score; a substitution-only pair agrees with the oracle's score."""
    rng = np.random.default_rng(77)
    lut = np.frombuffer(b"ACGT", np.uint8)
    m = 60000
    a = lut[rng.integers(0, 4, size=m)]
    r = gx.align_batch([(a, a)], CONFIG_TOML, False)[0]
    assert r.score == m and r.matches == m and len(r.ops) == m and r.end == (1, 1)
    assert not r.ops.any()
    A, B = random_pair(rng, 50000, 48000, sub=0.1, indel=0.02)
    for is_local in (False, True):
        x = gx.align_batch([(A, B), (B, A)], CONFIG_TOML, is_local, traceback=False)
        assert x[0].score == x[1].score
    a4 = rng.integers(0, 4, size=20000)
    b4 = a4.copy()
    idx = rng.choice(20000, size=600, replace=False)
    b4[idx] = (b4[idx] + 1 + rng.integers(0, 3, size=600)) % 4
    r = gx.align_batch([(lut[a4], lut[b4])], CONFIG_TOML, False)[0]
    assert r.score == oracle.score_linear(lut[a4], lut[b4], CONFIG_TOML, False)[0]
