"""Device top-k (cudasw4_b200/csrc/topk.cuh) against an exact sort by (score descending, index ascending), the oracle's
topk. The harness (tests/topk_harness.cu) runs the engine's own dispatch, topk_enqueue, on scores chosen here: every
k around the warp, pass-1 and large-path limits, sizes around every block split, every shift 8..12 up to the top
level-1 bin, and tie patterns placed on the block boundaries. The engine tests run the same selection after real scans:
the short-block fallback of pass 1, k changing between scans of one handle, several shards and a shift-9 scan."""
import numpy as np
import pytest

from tests import topk_harness

SMALL_K = [1, 2, 31, 32, 33, 1000, 2048, 2049, 2730, 2731, 4095, 4096]
LARGE_K = [4097, 6000, 8192, 8193, 65536, 100000]
P1 = 148 * 4096
SM_CHOICES = [None, 1, 2, 3, 7]  # None: the device's own SM count
# every shift 8..12 at its upper edge (the maximum lands in level-1 bin 4095) and one above it
SHIFT_EDGES = [(1 << (12 + s)) - 1 for s in range(8, 13)] + [1 << (12 + s) for s in range(8, 12)]
PATTERNS = ["zero", "equal", "uniform", "bin_edges", "tied_kth", "k_positive", "fewer_positive", "max_first", "max_last",
            "ties_then_above"]


@pytest.fixture(scope="module")
def harness():
    return topk_harness.load()


def _sizes(k):
    return sorted({n for n in (k, k + 1, 4095, 4096, 4097, 2 * k - 1, 8191, 8193, P1 - 1, P1 + 1, 10**6) if n >= k})


def _block_ranges(h, n, k, sm):
    """[begin, end) of every block that splits the scores: pass 1's blocks, or the large path's count/emit blocks."""
    blocks = h.large_blocks if h.uses_large_path(k) else h.pass1_blocks(n, k, sm)
    per = -(-n // blocks)
    return [(min(n, b * per), min(n, (b + 1) * per)) for b in range(blocks)]


def _scores(pattern, rng, n, k, max_score, shift, ranges):
    """n scores in [0, max_score] (max_score >= 1) of one pattern; every pattern but "zero" and "fewer_positive"
    reaches max_score."""
    hi = max_score
    T = hi // 2
    s = np.zeros(n, np.int64)
    if pattern == "zero":
        return s.astype(np.int32)
    if pattern == "equal":
        return np.full(n, hi, np.int32)
    if pattern == "uniform":
        s = rng.integers(0, hi + 1, n)
    elif pattern == "bin_edges":  # m * 2^shift - 1, m * 2^shift, m * 2^shift + 1
        s = (rng.integers(0, (hi >> shift) + 1, n) << shift) + rng.integers(-1, 2, n)
    elif pattern == "tied_kth":
        # entries == T on both sides of every block boundary and every stride-th entry, about twice as many as the
        # k - above that are kept, so the first ties in index order come from several blocks; k // 3 entries above T
        above = k // 3
        s = rng.integers(0, T, n) if T > 0 else s
        stride = max(1, n // (2 * (k - above) + 8))
        s[::stride] = T
        for b, _ in ranges[1:]:
            s[max(0, b - 2): b + 2] = T
        s[rng.choice(n, above, replace=False)] = rng.integers(T + 1, hi + 1, above)
    elif pattern == "k_positive":
        s[rng.choice(n, k, replace=False)] = rng.integers(1, hi + 1, k)
    elif pattern == "fewer_positive":
        s[rng.choice(n, k // 2, replace=False)] = rng.integers(1, hi + 1, k // 2)
    elif pattern in ("max_first", "max_last"):
        s = rng.integers(0, min(hi - 1, 50) + 1, n)
        s[0 if pattern == "max_first" else n - 1] = hi
        return s.astype(np.int32)
    elif pattern == "ties_then_above":
        # every block: its first third == T (more ties than it keeps), then below T, and its last entries above T at
        # the end of its range, so the ties are done long before the entries above T are
        s = rng.integers(0, T, n) if T > 0 else s
        for b, e in ranges:
            if e > b:
                s[b: b + (e - b) // 3] = T
                m = min(e - b, k // 2 + 1)
                s[e - m: e] = rng.integers(T + 1, hi + 1, m)
    else:
        raise ValueError(pattern)
    s = np.clip(s, 0, hi)
    if pattern != "fewer_positive":
        s[rng.integers(n)] = hi
    return s.astype(np.int32)


def _check(h, oracle, scores, k, max_score, sm, global_ids=None):
    got = h.run(scores, k, max_score, sm, global_ids)
    assert got != topk_harness.REFUSED
    out_s, out_i, count, launches = got
    assert launches >= 9 if h.uses_large_path(k) else launches == 2
    ref_s, ref_i = oracle.topk(scores, k)
    if global_ids is not None:
        ref_i = np.asarray(global_ids, np.int32)[ref_i]
    assert count == k
    bad = np.flatnonzero((out_s != ref_s) | (out_i != ref_i))
    assert bad.size == 0, (f"{bad.size} of {k} entries differ, first at {bad[0]}: got ({out_s[bad[0]]}, {out_i[bad[0]]}), "
                           f"want ({ref_s[bad[0]]}, {ref_i[bad[0]]})")


def _gapped_ids(rng, n):
    return (np.cumsum(rng.integers(1, 4, n)) + 5).astype(np.int32)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the dispatch itself
# ---------------------------------------------------------------------------------------------------------------------

def test_shift_for_every_edge(harness):
    want = {0: 8, (1 << 20) - 1: 8, 1 << 20: 9, (1 << 24) - 1: 12, 1 << 24: -1, (1 << 40): -1}
    for s in range(8, 12):
        want[(1 << (12 + s)) - 1] = s
        want[1 << (12 + s)] = s + 1
    for max_score, shift in want.items():
        assert harness.shift_for(max_score) == shift, max_score
        if shift > 0:
            assert (max_score >> shift) < 4096
            assert shift == 8 or (max_score >> (shift - 1)) >= 4096  # the smallest shift that fits
    for max_score in SHIFT_EDGES:  # the upper edges put the maximum into the top level-1 bin
        if max_score & (max_score + 1) == 0:
            assert max_score >> harness.shift_for(max_score) == 4095


def test_dispatch_path_and_pass1_split(harness):
    """Which path runs, and pass 1's split: min(smCount, 8192 // k, ceil(n / 4096)) blocks, whose candidates all fit
    pass 2's kTopkMaxCandidates; the block ranges the GPU cases are built on come from the same function."""
    assert harness.max_candidates == 8192 and harness.large_blocks == 592
    for k in SMALL_K + LARGE_K:
        assert harness.uses_large_path(k) == (k > 4096), k
        if harness.uses_large_path(k):
            continue
        for n in _sizes(k):
            for sm in (148, 1, 2, 3, 7):
                blocks = harness.pass1_blocks(n, k, sm)
                assert blocks == max(1, min(sm, 8192 // k, -(-n // 4096))), (n, k, sm)
                assert blocks * k <= harness.max_candidates
                ranges = _block_ranges(harness, n, k, sm)
                assert ranges[0][0] == 0 and ranges[-1][1] == n
                assert all(a[1] == b[0] for a, b in zip(ranges, ranges[1:]))


def test_fallback_cases_reach_short_blocks(harness):
    """The tie cases below do reach the pass-1 fallback (a block with fewer than k entries) and, for contrast, splits
    where no block falls short; the large path gets empty block ranges at n = k = 4097."""
    short, full = set(), set()
    for k, n, sm in _boundary_cases():
        if harness.uses_large_path(k):
            continue
        ranges = _block_ranges(harness, n, k, sm or 148)
        (short if any(e - b < k for b, e in ranges) else full).add(k)
    assert {2049, 2731, 4096} <= short and 1000 in full and 2049 in full
    assert sum(e == b for b, e in _block_ranges(harness, 4097, 4097, 148)) > 0


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the harness against an exact sort
# ---------------------------------------------------------------------------------------------------------------------

def _sweep_cases():
    """Every k with every size. Pattern (period 10), maxScore (9) and global ids (3) cycle with the case number; the SM
    count steps on by one more every 10 cases, so that it meets every pattern."""
    cases, i = [], 0
    for k in SMALL_K + LARGE_K:
        for n in _sizes(k):
            sm = SM_CHOICES[(i + i // 10) % 5]
            cases.append((k, n, sm, PATTERNS[i % 10], SHIFT_EDGES[i % 9], i % 3 == 2))
            i += 1
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("k,n,sm,pattern,max_score,gids", _sweep_cases())
def test_every_k_and_size(harness, oracle, k, n, sm, pattern, max_score, gids):
    sm = sm or harness.sm_count()
    rng = np.random.default_rng(k * 1000003 + n)
    scores = _scores(pattern, rng, n, k, max_score, harness.shift_for(max_score), _block_ranges(harness, n, k, sm))
    _check(harness, oracle, scores, k, max_score, sm, _gapped_ids(rng, n) if gids else None)


def _boundary_cases():
    cases = []
    for k in (1000, 2049, 2731, 4096, 8193):
        for n in sorted({2 * k - 1, 4097, 8191, P1 + 1}):
            if n >= k:
                cases += [(k, n, sm) for sm in SM_CHOICES]
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", ["tied_kth", "ties_then_above", "max_last"])
@pytest.mark.parametrize("k,n,sm", _boundary_cases())
def test_ties_on_block_boundaries(harness, oracle, k, n, sm, pattern):
    """The k-th score tied across every block boundary, blocks whose ties are done before their entries above T, and
    scores of at most 50 (all in level-1 bin 0, as after a short query), at every SM count: pass 1's short blocks (2048 < k <= 4096, n < 2k) and the large path's 592 ranges."""
    sm = sm or harness.sm_count()
    rng = np.random.default_rng(k + 7 * n + sm)
    max_score = (1 << 20) - 1
    scores = _scores(pattern, rng, n, k, max_score, harness.shift_for(max_score), _block_ranges(harness, n, k, sm))
    _check(harness, oracle, scores, k, max_score, sm, _gapped_ids(rng, n) if sm % 2 else None)


@pytest.mark.gpu
@pytest.mark.parametrize("max_score", SHIFT_EDGES)
@pytest.mark.parametrize("k,n", [(33, 200_000), (2731, 5461), (6000, 300_000)])
@pytest.mark.parametrize("pattern", ["uniform", "bin_edges"])
def test_every_shift(harness, oracle, k, n, pattern, max_score):
    sm = harness.sm_count()
    rng = np.random.default_rng(max_score + k)
    scores = _scores(pattern, rng, n, k, max_score, harness.shift_for(max_score), _block_ranges(harness, n, k, sm))
    assert scores.max() == max_score
    _check(harness, oracle, scores, k, max_score, sm)


@pytest.mark.gpu
@pytest.mark.parametrize("k,n,pattern", [(8193, 3_000_001, "tied_kth"), (65536, 7_000_000, "tied_kth"),
                                         (4096, 3_000_001, "ties_then_above"), (100000, 7_000_000, "bin_edges")])
def test_millions(harness, oracle, k, n, pattern):
    sm = harness.sm_count()
    rng = np.random.default_rng(n + k)
    max_score = (1 << 22) - 1
    scores = _scores(pattern, rng, n, k, max_score, harness.shift_for(max_score), _block_ranges(harness, n, k, sm))
    _check(harness, oracle, scores, k, max_score, sm, _gapped_ids(rng, n))


@pytest.mark.gpu
@pytest.mark.parametrize("k", [10, 6000])
def test_refuses_scores_from_2_pow_24(harness, k):
    scores = np.zeros(10000, np.int32)
    assert harness.run(scores, k, 1 << 24, harness.sm_count()) == topk_harness.REFUSED
    out_s, out_i, count, _ = harness.run(scores, k, (1 << 24) - 1, harness.sm_count())
    assert count == k and (out_s == 0).all() and (out_i == np.arange(k)).all()


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the engine after real scans, against oracle.scan + oracle.topk
# ---------------------------------------------------------------------------------------------------------------------

def _db(seed, lengths):
    from cudasw4_b200 import dbformat, synth
    rng = np.random.default_rng(seed)
    return dbformat.from_sequences([synth.random_residues(rng, int(x)) for x in lengths]), rng


def _scan_matches(eng, oracle, query, ref, k):
    res = eng.scan(query)
    s, i = oracle.topk(ref, k)
    assert len(res.scores) == min(k, len(ref))
    assert res.scores == s.tolist(), k
    assert res.referenceIds == i.tolist(), k


@pytest.mark.gpu
def test_engine_pass1_fallback_band(oracle):
    """About 5000 short subjects: pass 1 splits them into two blocks of about 2500, fewer than k for k > 2500 (the
    fallback), not for k = 2049. A short query gives scores of a few values, so T is tied by many subjects in both
    blocks. n = 8191 with k = 4096: only the last block falls short."""
    import cudasw4_b200 as sw
    from cudasw4_b200 import dbformat, synth
    for n, ks in ((5003, (2049, 2600, 3000, 4096)), (8191, (4096,))):
        db, rng = _db(n, np.random.default_rng(n).integers(4, 16, n))
        with sw.CudaSW4(deviceIds=[0], numTop=ks[0], blosumType=62) as eng:
            eng.setDatabase(db)
            for qlen in (3, 8):
                q = synth.random_residues(rng, qlen)
                ref = oracle.scan(62, q, db, -11, -1)
                assert len(np.unique(ref)) < 40
                for k in ks:
                    eng.setNumTop(k)
                    _scan_matches(eng, oracle, dbformat.decode(q), ref, k)


@pytest.mark.gpu
def test_engine_k_changes_between_scans(oracle):
    """k = 10 -> 5000 -> 10 -> 20001 -> 3000 on one handle: both paths, and the top-k scratch regrown between them."""
    import cudasw4_b200 as sw
    from cudasw4_b200 import dbformat, synth
    db, rng = _db(21, np.random.default_rng(21).integers(5, 60, 20011))
    q = synth.random_residues(rng, 25)
    ref = oracle.scan(62, q, db, -11, -1)
    with sw.CudaSW4(deviceIds=[0], numTop=10, blosumType=62) as eng:
        eng.setDatabase(db)
        for k in (10, 5000, 10, 20001, 3000):
            eng.setNumTop(k)
            _scan_matches(eng, oracle, dbformat.decode(q), ref, k)


@pytest.mark.gpu
def test_engine_three_shards(oracle):
    """12,500 subjects on three shards of one GPU: interleaved blocks of 256 give shards of 4308, 4096 and 4096.
    k = 100 and 3000 run pass 1/2 on every shard; k = 4200 lies between the shard sizes (the large path on the first
    shard, pass 1/2 on the others after the clip to min(k, n)); k = 20000 is above the database size."""
    import cudasw4_b200 as sw
    from cudasw4_b200 import dbformat, synth
    db, rng = _db(33, np.random.default_rng(33).integers(5, 80, 12500))
    q = synth.random_residues(rng, 12)
    ref = oracle.scan(62, q, db, -11, -1)
    with sw.CudaSW4(deviceIds=[0, 0, 0], numTop=100, blosumType=62) as eng:
        eng.setDatabase(db)
        for k in (100, 3000, 4200, 20000):
            eng.setNumTop(k)
            _scan_matches(eng, oracle, dbformat.decode(q), ref, k)


@pytest.mark.gpu
def test_engine_shift_9(oracle, harness):
    """BLOSUM45 (largest entry 15), a 70,000-residue query and one 70,000-residue subject among 2000 short ones: the
    bound 15 x 70,000 >= 2^20 selects shift 9. Most query residues are W (self score 15), and 60,000 residues of the
    query are planted in the long subject, so its hit lands near the top of the level-1 bins the bound allows
    (15 x 70,000 >> 9 = 2050)."""
    import cudasw4_b200 as sw
    from cudasw4_b200 import dbformat, synth
    assert harness.shift_for(15 * 70_000) == 9
    rng = np.random.default_rng(45)
    q = synth.random_residues(rng, 70_000)
    q[rng.random(len(q)) < 0.7] = dbformat.encode("W")[0]
    long_subject = synth.random_residues(rng, 70_000)
    long_subject[4000:64000] = q[5000:65000]
    seqs = [synth.random_residues(rng, int(x)) for x in rng.integers(20, 80, 2000)]
    seqs.insert(1234, long_subject)
    db = dbformat.from_sequences(seqs)
    ref = oracle.scan(45, q, db, -11, -1)
    assert ref.max() >> 9 > 1400  # the level-1 bin of the planted hit
    with sw.CudaSW4(deviceIds=[0], numTop=50, blosumType=45) as eng:
        eng.setDatabase(db)
        _scan_matches(eng, oracle, dbformat.decode(q), ref, 50)
        scores, ids = eng.lastScanAllScores()
        got = np.empty_like(ref)
        got[ids] = scores
        assert (got == ref).all()
