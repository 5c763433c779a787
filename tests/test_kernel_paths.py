"""Every scoring-kernel path against the oracle, chosen by the kernel that runs rather than by database shape.

The engine picks one of about ten kernels per length class and query (engine.cu, Engine::enqueueBatch): the
two-rows-per-step kernel in one of its lane x column shapes, its multi-segment form, the full-warp one-row kernel, the
CTA-wide one-row array (kernels_s16_long.cuh, W = 2..16 warps) or the two-row array (kernels_s16_long2.cuh, W = 2..8),
and then one of two exact 32-bit re-scoring kernels (kernels_s32.cuh, kernels_s32_long.cuh). `kernel_path` restates
that choice in Python with the constants parsed from the sources; the CPU tests below keep the restatement tied to the
code and check that the GPU cases reach every (kernel, shape, re-scoring kernel) combination the GPU they run on can
reach. The GPU tests (-m gpu) then place queries on both sides of every threshold of the rule, run the gap scores at
the limits of the accepted range, put subjects exactly on the 16-bit overflow boundaries, and run every development
switch. Every GPU result is compared with the oracle on all scores, the top-k list (ties by ascending id) and
stats.numOverflows."""
import functools
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "cudasw4_b200", "csrc")


def _src(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


# ---------------------------------------------------------------------------------------------------------------------
# the path rule, restated from engine.cu (shapeForQuery, Engine::enqueueBatch) and s16_long2_warps
# ---------------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def constants():
    def get(src, name):
        return int(re.search(r"constexpr (?:int|short) %s = (-?\d+);" % name, src).group(1))

    s16, long1, long2, eng = _src("kernels_s16.cuh"), _src("kernels_s16_long.cuh"), _src("kernels_s16_long2.cuh"), _src("engine.cu")
    c = {k: get(long1, k) for k in ("kLongLag", "kLongMaxWarps", "kLongBatch", "kLongFifoRows")}
    c.update({k: get(long2, k) for k in ("kLag2", "kFifo2", "kLong2Warps", "kLong2MaxW")})
    c.update({k: get(s16, k) for k in ("kStatMaxLength", "kBatchSteps", "kNegS16")})
    c.update({k: get(eng, k) for k in ("kS16OverflowThreshold", "kHalf2Threshold")})
    c["kS16Warps"] = int(re.search(r"#define SW4_S16_THREADS (\d+)", s16).group(1)) // 32
    table = eng[eng.index("kLengthClasses[] = {"):]
    table = table[:table.index("};")]
    c["classes"] = tuple((int(g), int(r), int(cap), w == "true", m == "true")
                         for g, r, cap, w, m in re.findall(r"\{(\d+), (\d+), (\d+), (true|false), (true|false)\}", table))
    return c


def class_of(length):
    """Index of the length class a subject of `length` >= 1 residues belongs to (Engine::makeBatch)."""
    for i, (_, _, cap, _, multi) in enumerate(constants()["classes"]):
        if multi or length <= cap:
            return i
    raise AssertionError(length)


def long_class():
    return len(constants()["classes"]) - 1


def array_period(qlen):
    return (qlen + 32 + 15) // 16 * 16


def long2_warps(qlen):
    """s16_long2_warps: (W, period in steps); W = 0 when the query is too short for an array."""
    c = constants()
    p0 = ((qlen + 1) // 2 + 32 + 15) // 16 * 16
    w = c["kLong2MaxW"]
    while w > 1 and c["kLag2"] * w + 16 > p0:
        w //= 2
    return (w if w >= 2 else 0), p0


def long1_warps(qlen):
    c = constants()
    w = c["kLongMaxWarps"]
    while w > 1 and c["kLongLag"] * w + 64 > array_period(qlen):
        w //= 2
    return w


def rescoring_kernel(qlen, switches=None):
    c = constants()
    use_long = "SW4_NO_LONG_KERNEL" not in (switches or {})
    return "s32_long" if use_long and c["kLongLag"] * c["kLongMaxWarps"] + 64 <= array_period(qlen) else "s32"


def kernel_path(qlen, cls, num_items, sm_count, switches=None):
    """(score kernel, shape, re-scoring kernel) the engine runs for length class `cls` holding `num_items` subject
    pairs, a query of `qlen` residues, `sm_count` SMs and the development switches `switches` (environment).
    The shape is "lanes x columns" for the two-row and one-row kernels and the array width W (warps) for the array
    kernels. Assumes the default border-scratch budget, under which the multi-segment kernels get border slots."""
    c = constants()
    sw = switches or {}
    crossover = int(sw.get("SW4_CLASS256_CROSSOVER", 0x7FFFFFFF))
    use_long = "SW4_NO_LONG_KERNEL" not in sw
    use_long2 = "SW4_NO_LONG2_KERNEL" not in sw
    min_warps = max(2, int(sw.get("SW4_LONG_MIN_WARPS", 2)))
    two_row = "SW4_NO_TWO_ROW_MULTI" not in sw
    items_per_group = float(sw.get("SW4_LONG_ARRAY_ITEMS_PER_GROUP", 3.0))
    log_g, R, cap, wide, multi = c["classes"][cls]
    if cap == 256 and not wide and qlen < crossover:
        log_g, R = 3, 32
    rescore = rescoring_kernel(qlen, sw)
    w1 = 0
    if multi and use_long:
        w1 = long1_warps(qlen)
        if w1 < min_warps:
            w1 = 0
        if w1 and two_row and num_items > items_per_group * sm_count * c["kS16Warps"] * 2:
            w1 = 0
    w2 = long2_warps(qlen)[0] if (w1 and use_long2) else 0
    if w2 < min(w1, c["kLong2MaxW"]) or qlen < 256:
        w2 = 0
    if w2 and w1 > c["kLong2MaxW"] and num_items < 2 * sm_count:
        w2 = 0
    if w2:
        return ("long2", w2, rescore)
    if w1:
        return ("long", w1, rescore)
    if wide and two_row:
        return ("s16_seg", "16x%d" % R, rescore)
    if wide:
        return ("s16_wide_multi" if multi else "s16_wide", "32x%d" % R, rescore)
    return ("s16", "%dx%d" % (1 << log_g, R), rescore)


def db_combos(qlen, lengths, sm_count, switches=None):
    """Every (kernel, shape, re-scoring kernel) one scan of a database with these subject lengths runs."""
    counts = np.bincount([class_of(int(n)) for n in lengths if n > 0], minlength=len(constants()["classes"]))
    return {kernel_path(qlen, cls, (int(n) + 1) // 2, sm_count, switches) for cls, n in enumerate(counts) if n}


# ---------------------------------------------------------------------------------------------------------------------
# the cases of the GPU tests (functions of the SM count; shared with the CPU coverage test)
# ---------------------------------------------------------------------------------------------------------------------
SHORT_QUERIES = (1, 2, 3, 15, 16, 17, 18, 19, 31, 32, 33, 34, 35, 36, 63, 64, 65, 127, 128, 129)
NEAR_2000 = (1997, 2002)
SWEEP_GAPS = ((62, -11, -1), (62, -5, -3))
W_RICH_LENGTH = 3400
SWITCH_QUERIES = (60, 150, 300, 500, 700, W_RICH_LENGTH)
SWITCHES = ({"SW4_NO_LONG_KERNEL": "1"}, {"SW4_NO_LONG2_KERNEL": "1"}, {"SW4_LONG_MIN_WARPS": "16"},
            {"SW4_LONG_ARRAY_ITEMS_PER_GROUP": "0"}, {"SW4_LONG_ARRAY_ITEMS_PER_GROUP": "1e9"},
            {"SW4_CLASS256_CROSSOVER": "0"}, {"SW4_NO_TWO_ROW_MULTI": "1"}, {"SW4_NO_GAP_SETS": "1"},
            {"SW4_NO_CLUSTER": "1"}, {"SW4_PIPELINE": "1"}, {"SW4_PIPELINE": "16"}, {"SW4_BACKFILL_ITEMS": "1"},
            {"SW4_BACKFILL_ITEMS": "64"})
# gap pairs (blosum, gop, gex): the limits of the accepted range [-4096, 0], pairs next to a compiled-in gap set, and
# positive inputs (negated by the library: (11, 1) must run as gap set 1, -11 / -1)
GAP_MATRIX = ((62, 0, 0), (45, 0, -1), (80, -1, 0), (62, -1, -4096), (45, -4096, -1), (80, -4096, -4096),
              (62, -11, -2), (45, -12, -1), (80, -10, -2), (62, 11, 1), (45, 13, 2))
GAP_SETS = ((62, -11, -1), (45, -13, -2), (80, -10, -1), (50, -5, -3))


def few_long_items(sm_count):
    return sm_count // 3 + 1          # < 2 SMs: the array kernels take the long class, the one-row array at W = 16


def many_long_items(sm_count):
    return 2 * sm_count + 5           # 2 SMs .. 3 x 32 x SMs: still the arrays, the two-row one at W = 8


def long_items_kind(items, sm_count):
    if items < 2 * sm_count:
        return "few"
    assert items <= 3 * sm_count * 2 * constants()["kS16Warps"]
    return "many"


def long_path_breaks(sm_count, items, switches=None, qmax=2100):
    """Query lengths q at which the long class's path differs from that of q - 1."""
    prev, out = None, []
    for q in range(1, qmax + 1):
        p = kernel_path(q, long_class(), items, sm_count, switches)
        if prev is not None and p != prev:
            out.append(q)
        prev = p
    return out


def threshold_queries(sm_count):
    """Both sides of every threshold of the long class's path, with few and with many items."""
    qs = set()
    for items in (few_long_items(sm_count), many_long_items(sm_count)):
        for q in long_path_breaks(sm_count, items):
            qs.update((q - 1, q))
    return tuple(sorted(qs))


def sweep_queries(sm_count):
    return tuple(sorted(set(SHORT_QUERIES) | set(threshold_queries(sm_count)) | set(NEAR_2000)))


def gap_queries(sm_count):
    """One query per path of the long class with few items (the middle of the first q range of each path)."""
    items = few_long_items(sm_count)
    ranges = {}
    for q in range(1, 2101):
        ranges.setdefault(kernel_path(q, long_class(), items, sm_count), []).append(q)
    return {p: qs[len(qs) // 2] if qs[-1] < 2100 else qs[0] + 100 for p, qs in ranges.items()}


def sweep_lengths(sm_count, kind):
    """Subject lengths of the two sweep databases: both bounds of every length class, one class holding a single
    subject and one holding two, random fillers, and few or many long subjects."""
    rng = np.random.default_rng(4242 if kind == "few" else 4343)
    caps = sorted({cap for _, _, cap, _, multi in constants()["classes"] if not multi})
    one, two = (576, 640) if kind == "few" else (48, 256)        # capacities of the classes with one / two subjects
    lo_of = {cap: (caps[i - 1] + 1 if i else 1) for i, cap in enumerate(caps)}
    L = [1, 2]
    for cap in caps:
        if cap == one:
            L += [cap]
        elif cap == two:
            L += [lo_of[cap], cap]
        else:
            L += [lo_of[cap], cap] + rng.integers(lo_of[cap], cap + 1, 5).tolist()
    items = few_long_items(sm_count) if kind == "few" else many_long_items(sm_count)
    hi = 3000 if kind == "few" else 1500
    L += [1025] + rng.integers(1026, hi, 2 * items - 2).tolist()      # an odd number of long subjects: a half pair
    return np.array(L, dtype=np.int64)


def coverage_cases(sm_count):
    """(case name, combinations it reaches) for every GPU case of this file."""
    cases = []
    lengths = {kind: sweep_lengths(sm_count, kind) for kind in ("few", "many")}
    for kind in ("few", "many"):
        for q in sweep_queries(sm_count):
            cases.append(("sweep/%s/q=%d" % (kind, q), db_combos(q, lengths[kind], sm_count)))
    for q in gap_queries(sm_count).values():
        cases.append(("gaps/q=%d" % q, db_combos(q, lengths["few"], sm_count)))
    for kind in ("few", "many"):
        cases.append(("overflow/%s" % kind, db_combos(W_RICH_LENGTH, lengths[kind], sm_count)))
    for sw in SWITCHES:
        for q in SWITCH_QUERIES:
            cases.append(("switch/%s/q=%d" % (",".join("%s=%s" % kv for kv in sw.items()), q),
                          db_combos(q, lengths["few"], sm_count, sw)))
    return cases


def reachable_combos(sm_count):
    """Every combination the rule can produce for databases of both kinds, any query length and every switch setting
    the tests use (evaluated at the long class's breakpoints, where all classes' paths are constant in between)."""
    out = set()
    for kind in ("few", "many"):
        lengths = sweep_lengths(sm_count, kind)
        items = (int((lengths > 1024).sum()) + 1) // 2
        for sw in ({},) + SWITCHES:
            qs = {1, 2100, W_RICH_LENGTH, 35000}
            for q in long_path_breaks(sm_count, items, sw):
                qs.update((q - 1, q))
            for q in qs:
                out |= db_combos(q, lengths, sm_count, sw)
    return out


def _sm_counts():
    """The SM count of the GPU the tests run on; on a machine without one, the counts of current data-centre parts."""
    try:
        import torch
        if torch.cuda.is_available():
            return [torch.cuda.get_device_properties(0).multi_processor_count]
    except Exception:
        pass
    return [132, 148, 160]


# ---------------------------------------------------------------------------------------------------------------------
# CPU tests
# ---------------------------------------------------------------------------------------------------------------------
def test_path_rule_matches_engine_source():
    """The restatement above depends on these expressions; if one changes, kernel_path must change with it."""
    eng = _src("engine.cu")
    for expr in (
        'getenv("SW4_CLASS256_CROSSOVER"); return e ? atoi(e) : 0x7fffffff;',
        "if (lc.capacity == 256 && !lc.wide && qlen < crossover) return LengthClass{3, 32, 256, false, false};",
        "const int p0 = (qlen + 32 + 15) / 16 * 16;",
        "if (lc.multi && useLongKernel) {",
        "longWarps = kLongMaxWarps;",
        "while (longWarps > 1 && kLongLag * longWarps + 64 > p0) longWarps >>= 1;",
        "if (longWarps < longMinWarps) longWarps = 0;",
        "if (longWarps && twoRowMulti && cl.numItems > longArrayMaxItemsPerGroup * sh.smCount * kS16Warps * 2) longWarps = 0;",
        "int long2Warps = (longWarps && useLong2Kernel) ? s16_long2_warps(qlen, &long2Period) : 0;",
        "if (long2Warps < std::min(longWarps, kLong2MaxW) || qlen < 256) long2Warps = 0;",
        "if (long2Warps && longWarps > kLong2MaxW && cl.numItems < 2 * sh.smCount) long2Warps = 0;",
        "const bool segmented = lc.wide && twoRowMulti && ctx.borderSlots > 0;",
        "if (useLongKernel && kLongLag * kLongMaxWarps + 64 <= p0) {",
        'getenv("SW4_LONG_MIN_WARPS"); return e ? std::max(2, atoi(e)) : 2;',
        'getenv("SW4_LONG_ARRAY_ITEMS_PER_GROUP"); return e ? atof(e) : 3.0;',
        'getenv("SW4_NO_LONG_KERNEL"); return !e;',
        'getenv("SW4_NO_LONG2_KERNEL"); return !e;',
        'getenv("SW4_NO_TWO_ROW_MULTI"); return !e;',
        "const size_t e = lc.multi ? end : (size_t)(std::upper_bound(L + pos, L + end, lc.capacity) - L);",
        "bc.numItems = (bc.count + 1) / 2;",
        # the numOverflows rule: classes above 240 columns count, the multi-segment kernels up to kStatMaxLength
        "prm.statThreshold = (lc.capacity > 240) ? statThreshold() : 0x7fffffff;",
        "return kernelTypes[0] == SW4_KERNEL_HALF2 ? kHalf2Threshold : kS16OverflowThreshold;",
        # default border budget: every SM gets a border slot (kernel_path assumes slots exist)
        "ctx.borderSlots = needBorder ? (int)std::min<size_t>((size_t)sh.smCount, rows * 2 / 3 / groupsPerCta) : 0;",
    ):
        assert expr in eng, expr
    hdr = _src("kernels_s16_long2.cuh")
    for expr in ("const int p0 = ((qlen + 1) / 2 + 32 + 15) / 16 * 16;", "while (w > 1 && kLag2 * w + 16 > p0) w >>= 1;",
                 "return w >= 2 ? w : 0;"):
        assert expr in hdr, expr
    c = constants()
    assert len(c["classes"]) == 32 and c["classes"][-1][4] and not any(m for *_, m in c["classes"][:-1])
    assert [cap for _, _, cap, _, _ in c["classes"]] == sorted(cap for _, _, cap, _, _ in c["classes"])


def test_long_class_thresholds_restate_the_documented_table():
    """The long-class thresholds the sweep is built from, for any SM count: multi-segment up to 112, one-row W = 2 from
    113, W = 4 from 209, two-row W = 4 from 257, one-row W = 8 from 401, two-row W = 8 from 577, and from 785 one-row
    W = 16 (few items) or two-row W = 8 (many), re-scored by the array form of the exact kernel."""
    for sm in _sm_counts():
        few, many = few_long_items(sm), many_long_items(sm)
        assert long_items_kind(few, sm) == "few" and long_items_kind(many, sm) == "many"
        assert long_path_breaks(sm, few) == [113, 209, 257, 401, 577, 785]
        assert long_path_breaks(sm, many) == [113, 209, 257, 401, 577, 785]
        at = lambda q, n: kernel_path(q, long_class(), n, sm)
        assert at(112, few) == ("s16_seg", "16x32", "s32") and at(113, few) == ("long", 2, "s32")
        assert at(256, few) == ("long", 4, "s32") and at(257, few) == ("long2", 4, "s32")
        assert at(576, few) == ("long", 8, "s32") and at(577, few) == ("long2", 8, "s32")
        assert at(785, few) == ("long", 16, "s32_long") and at(785, many) == ("long2", 8, "s32_long")
        assert at(785, 3 * sm * 32 + 1) == ("s16_seg", "16x32", "s32_long")


@pytest.mark.parametrize("sm", _sm_counts())
def test_cases_reach_every_reachable_path(sm):
    cases = coverage_cases(sm)
    covered = set().union(*(combos for _, combos in cases))
    reachable = reachable_combos(sm)
    missing = reachable - covered
    assert not missing, sorted(missing, key=str)
    assert covered <= reachable
    # which case reaches what (pytest -rA -s shows it)
    first = {}
    for name, combos in cases:
        for cmb in combos:
            first.setdefault(cmb, name)
    for cmb in sorted(first, key=str):
        print("%-45s %s" % (cmb, first[cmb]))


NEG_INF = np.iinfo(np.int64).min // 4   # below any finite sum of scores the recurrence can form: a true minus infinity


def numpy_gotoh(M, q, s, gop, gex):
    """Plain int64 local Gotoh (same recurrence as oracle/sw_oracle.cpp, but with a true minus infinity)."""
    M = np.asarray(M, dtype=np.int64)
    n = len(s)
    H = np.zeros(n + 1, np.int64)
    F = np.full(n + 1, NEG_INF, np.int64)
    best = 0
    for qi in q:
        sub = M[qi][np.asarray(s, dtype=np.intp)]
        F = np.maximum(F + gex, H + gop)                      # vertical gap: from the previous row
        diag = H[:-1] + sub
        Hn = np.zeros(n + 1, np.int64)
        E = NEG_INF
        for j in range(1, n + 1):
            E = max(E + gex, int(Hn[j - 1]) + gop)
            Hn[j] = max(0, int(diag[j - 1]), E, int(F[j]))
        F[0] = NEG_INF
        H = Hn
        best = max(best, int(H.max()))
    return best


@pytest.mark.parametrize("blosum,gop,gex", GAP_MATRIX + GAP_SETS)
def test_oracle_matches_numpy_gotoh_at_gap_limits(oracle, blosum, gop, gex):
    """The C oracle's minus infinity is -10000 and it was pinned against the reference at ordinary gap scores only."""
    from cudasw4_b200 import synth
    gop, gex = -abs(gop), -abs(gex)
    M = oracle.matrix(blosum)
    rng = np.random.default_rng(1000 + blosum - gop - 7 * gex)
    for t in range(12):
        q = synth.random_residues(rng, int(rng.integers(1, 40)))
        s = synth.random_residues(rng, int(rng.integers(1, 40)))
        if t % 3 == 0:
            s[:: 5] = 17                                         # some W to make long gapped alignments worth it
            q[:: 4] = 17
        if t % 4 == 1:
            s[0] = 20
        assert oracle.score(blosum, q, s, gop, gex) == numpy_gotoh(M, q, s, gop, gex), (t, q.tolist(), s.tolist())


# ---------------------------------------------------------------------------------------------------------------------
# GPU tests
# ---------------------------------------------------------------------------------------------------------------------
def _sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _sprinkle_other(rng, seqs):
    for s in seqs[::13]:          # some code-20 letters
        if len(s):
            s[rng.integers(0, len(s))] = 20
    return seqs


def _sweep_db(sm, kind):
    from cudasw4_b200 import dbformat, synth
    L = sweep_lengths(sm, kind)
    rng = np.random.default_rng(int(L.sum()))
    seqs = _sprinkle_other(rng, [synth.random_residues(rng, int(n)) for n in L])
    return dbformat.from_sequences(seqs)


def _all_scores(eng, n):
    scores, ids = eng.lastScanAllScores()
    assert sorted(ids.tolist()) == list(range(n))
    got = np.empty(n, np.int32)
    got[ids] = scores
    return got


def _check_all(eng, oracle, db, q, blosum, gop, gex, k, res=None, ref=None, stat_threshold=25000):
    """Every score, the top-k list and stats.numOverflows of one scan against the oracle; returns the oracle scores."""
    from cudasw4_b200 import dbformat
    res = res or eng.scan(dbformat.decode(q))
    got = _all_scores(eng, db.num_sequences)
    if ref is None:
        ref = oracle.scan(blosum, q, db, -abs(gop), -abs(gex))
    bad = np.nonzero(got != ref)[0]
    assert len(bad) == 0, (len(q), blosum, gop, gex, bad[:8], got[bad[:8]], ref[bad[:8]], db.lengths[bad[:8]])
    s, i = oracle.topk(ref, k)
    assert res.scores == s.tolist() and res.referenceIds == i.tolist(), (len(q), blosum, gop, gex)
    L = db.lengths
    c = constants()
    assert res.stats.numOverflows == int(((ref >= stat_threshold) & (L > 240) & (L <= c["kStatMaxLength"])).sum()), len(q)
    return ref


def _assert_long_kind(db, sm, kind):
    items = (int((db.lengths > 1024).sum()) + 1) // 2
    assert long_items_kind(items, sm) == kind, (items, sm)


@pytest.fixture(scope="module")
def sweep_dbs():
    sm = _sm_count()
    return sm, {kind: _sweep_db(sm, kind) for kind in ("few", "many")}


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["few", "many"])
@pytest.mark.parametrize("blosum,gop,gex", SWEEP_GAPS)
def test_query_length_sweep(oracle, sweep_dbs, kind, blosum, gop, gex):
    """Query lengths at the two-row kernel's period floors and ring / batch edges, on both sides of every long-class
    threshold of the rule, and near 2000, against a database with few and one with many long subjects."""
    import cudasw4_b200 as sw
    from cudasw4_b200 import synth
    sm, dbs = sweep_dbs
    db = dbs[kind]
    _assert_long_kind(db, sm, kind)
    qs = sweep_queries(sm)
    assert {112, 113, 208, 209, 256, 257, 400, 401, 576, 577, 784, 785} <= set(qs)
    rng = np.random.default_rng(7 + gex)
    reached = set()
    with sw.CudaSW4(deviceIds=[0], numTop=17, blosumType=blosum, gop=gop, gex=gex) as eng:
        eng.setDatabase(db)
        for ql in qs:
            q = synth.random_residues(rng, ql)
            if ql > 30:
                q[ql // 3] = 20
            _check_all(eng, oracle, db, q, blosum, gop, gex, 17)
            reached |= db_combos(ql, db.lengths, sm)
    assert {p for p in reached if p[0] in ("long", "long2")} >= (
        {("long", w, "s32") for w in (2, 4, 8)} | {("long2", w, "s32") for w in (4, 8)}
        | ({("long", 16, "s32_long")} if kind == "few" else {("long2", 8, "s32_long")}))


@pytest.mark.gpu
def test_gap_scores_at_range_limits_on_every_array_path(oracle, sweep_dbs):
    """Gap pairs at the ends of [-4096, 0], next to a compiled-in gap set and given as positive numbers, on every path
    of the long class (multi-segment, one-row W = 2/4/8/16, two-row W = 4/8), then every gap set on the two-row array;
    an out-of-range pair is refused and leaves the previous pair in force."""
    import cudasw4_b200 as sw
    from cudasw4_b200 import dbformat, synth
    sm, dbs = sweep_dbs
    db = dbs["few"]
    paths = gap_queries(sm)
    assert {p[:2] for p in paths} == {("s16_seg", "16x32"), ("long", 2), ("long", 4), ("long", 8), ("long", 16),
                                      ("long2", 4), ("long2", 8)}
    rng = np.random.default_rng(99)
    queries = {ql: synth.random_residues(rng, ql) for ql in paths.values()}
    for q in queries.values():
        q[::7] = 17
    results = {}
    with sw.CudaSW4(deviceIds=[0], numTop=9, blosumType=62) as eng:
        eng.setDatabase(db)
        for blosum, gop, gex in GAP_MATRIX:
            eng.setBlosum(blosum)
            eng.setGapScores(gop, gex)
            for ql, q in queries.items():
                res = eng.scan(dbformat.decode(q))
                _check_all(eng, oracle, db, q, blosum, gop, gex, 9, res=res)
                results[(blosum, gop, gex, ql)] = (res.scores, res.referenceIds, _all_scores(eng, db.num_sequences))
        long2_qs = [ql for p, ql in paths.items() if p[0] == "long2"]
        for blosum, gop, gex in GAP_SETS:
            eng.setBlosum(blosum)
            eng.setGapScores(gop, gex)
            for ql in long2_qs:
                res = eng.scan(dbformat.decode(queries[ql]))
                _check_all(eng, oracle, db, queries[ql], blosum, gop, gex, 9, res=res)
                if (blosum, gop, gex) == (62, -11, -1):
                    a, b = results[(62, 11, 1, ql)], (res.scores, res.referenceIds, _all_scores(eng, db.num_sequences))
                    assert a[0] == b[0] and a[1] == b[1] and (a[2] == b[2]).all()
        eng.setBlosum(45)
        eng.setGapScores(-4096, -4096)
        for bad in ((-4097, -1), (-1, -4097), (4097, 1), (1, 4097), (-4097, -4097)):
            with pytest.raises(sw.SW4Error):
                eng.setGapScores(*bad)
        q = queries[long2_qs[0]]
        _check_all(eng, oracle, db, q, 45, -4096, -4096, 9)


def _w_rich_query():
    from cudasw4_b200 import synth
    rng = np.random.default_rng(2024)
    q = synth.random_residues(rng, W_RICH_LENGTH)
    q[rng.random(W_RICH_LENGTH) < 0.8] = 17
    return q


def _tune(oracle, q, blosum, targets):
    """For each target score: a prefix of q plus one tuning residue whose exact score against q is the target."""
    from cudasw4_b200 import dbformat
    found = {}
    for target in targets:
        lo, hi = 1, len(q)
        while lo < hi:                                   # shortest prefix scoring >= target - 12
            mid = (lo + hi) // 2
            if oracle.score(blosum, q, q[:mid], -11, -1) >= target - 12:
                hi = mid
            else:
                lo = mid + 1
        cands = [np.append(q[:n], np.uint8(r)) for n in range(max(1, lo - 2), min(len(q) - 1, lo + 6) + 1) for r in range(20)]
        scores = oracle.scan(blosum, q, dbformat.from_sequences(cands, presorted=True), -11, -1)
        hit = np.nonzero(scores == target)[0]
        assert len(hit), (target, sorted(set(scores.tolist())))
        found[target] = cands[int(hit[0])]
    return found


def _padded(core, length):
    """core followed by code-20 letters up to `length` (they score the matrix minimum against everything, so the
    subject scores what its core scores)."""
    s = np.full(length, 20, np.uint8)
    s[:len(core)] = core
    return s


@pytest.fixture(scope="module")
def overflow_setup(oracle, sweep_dbs):
    """The W-rich query, subjects scoring exactly 24999 / 25000 / 32767 / 32768 (long class) and 2047 / 2048 at 240,
    241, 8000 and 8001 residues, each twice in a row (so that it sits at an even and an odd position of its class),
    added to both sweep databases."""
    from cudasw4_b200 import dbformat
    sm, dbs = sweep_dbs
    q = _w_rich_query()
    cores = _tune(oracle, q, 62, (24999, 25000, 32767, 32768, 2047, 2048))
    special = {(t, len(cores[t])): cores[t] for t in (24999, 25000, 32767, 32768)}
    special.update({(t, n): _padded(cores[t], n) for t in (2047, 2048) for n in (240, 241, 8000, 8001)})
    for (target, _), s in special.items():
        assert oracle.score(62, q, s, -11, -1) == target
    assert all(n > 1024 for t, n in special if t > 20000)
    out = {}
    for kind, base in dbs.items():
        seqs = [base.sequence(i).copy() for i in range(base.num_sequences)]
        for s in special.values():
            seqs += [s.copy(), s.copy()]
        db = dbformat.from_sequences(seqs)
        _assert_long_kind(db, sm, kind)
        ref = oracle.scan(62, q, db, -11, -1)
        L = db.lengths
        cls = np.array([class_of(int(n)) if n else -1 for n in L])
        for (target, length), s in special.items():
            pos = [int(i) for i in np.nonzero((ref == target) & (L == length))[0] if np.array_equal(db.sequence(int(i)), s)]
            first = int(np.searchsorted(cls, class_of(length)))
            assert len(pos) == 2 and {(i - first) % 2 for i in pos} == {0, 1}, (target, length, pos, first)
        out[kind] = (db, ref)
    return sm, q, out


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["few", "many"])
def test_scores_on_the_16_bit_overflow_boundaries(oracle, overflow_setup, kind):
    """Exact scores 24999 / 25000 (re-scoring threshold) and 32767 / 32768 (16-bit range) in both halves of a packed
    pair, through the one-row W = 16 array (few long subjects) or the two-row W = 8 array (many), re-scored by the
    array form of the exact kernel; numOverflows counts exactly the subjects of 241..8000 residues at >= 25000."""
    import cudasw4_b200 as sw
    sm, q, dbs = overflow_setup
    db, ref = dbs[kind]
    expect = ("long", 16, "s32_long") if kind == "few" else ("long2", 8, "s32_long")
    assert kernel_path(len(q), long_class(), (int((db.lengths > 1024).sum()) + 1) // 2, sm) == expect
    for t in (24999, 25000, 32767, 32768):
        assert int((ref == t).sum()) >= 2, t
    with sw.CudaSW4(deviceIds=[0], numTop=12, blosumType=62) as eng:
        eng.setDatabase(db)
        _check_all(eng, oracle, db, q, 62, -11, -1, 12, ref=ref)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["few", "many"])
def test_half2_overflow_count_at_its_length_gates(oracle, overflow_setup, kind):
    """KernelTypeConfig(Half2, ...) counts scores >= 2048 instead of 25000, with the same length gates: subjects of
    240 residues are not counted, 241 are, 8000 are, 8001 are not (the last two on the two-row array with many long
    subjects). Scores stay exact."""
    import cudasw4_b200 as sw
    sm, q, dbs = overflow_setup
    db, ref = dbs[kind]
    L = db.lengths
    for n in (240, 241, 8000, 8001):
        assert int(((L == n) & (ref == 2048)).sum()) >= 2 and int(((L == n) & (ref == 2047)).sum()) >= 2, n
    cfg = sw.KernelTypeConfig(sw.KernelType.Half2, sw.KernelType.Half2, sw.KernelType.Float, sw.KernelType.Float)
    with sw.CudaSW4(deviceIds=[0], numTop=12, blosumType=62, kernelTypeConfig=cfg) as eng:
        eng.setDatabase(db)
        _check_all(eng, oracle, db, q, 62, -11, -1, 12, ref=ref, stat_threshold=constants()["kHalf2Threshold"])


_SWITCH_CHILD = r'''
import sys
import numpy as np
sys.path.insert(0, %(root)r)
import cudasw4_b200 as sw
from cudasw4_b200 import dbformat
d = np.load(sys.argv[1])
db = dbformat.SequenceDB(d["chars"], d["offsets"], d["lengths"], d["headers"], d["header_offsets"])
L = db.lengths
n, nq, k = db.num_sequences, int(d["nq"]), int(d["k"])
qs = [d["q%%d" %% i] for i in range(nq)]
def check(res, i, all_scores):
    ref = d["ref%%d" %% i]
    if all_scores:
        scores, ids = eng.lastScanAllScores()
        assert sorted(ids.tolist()) == list(range(n))
        got = np.empty(n, np.int32)
        got[ids] = scores
        bad = np.nonzero(got != ref)[0]
        assert len(bad) == 0, (len(qs[i]), bad[:8], got[bad[:8]], ref[bad[:8]], L[bad[:8]])
    assert res.scores == d["s%%d" %% i].tolist() and res.referenceIds == d["i%%d" %% i].tolist(), len(qs[i])
    assert res.stats.numOverflows == int(((ref >= 25000) & (L > 240) & (L <= 8000)).sum()), len(qs[i])
with sw.CudaSW4(deviceIds=[0], numTop=k, blosumType=62) as eng:
    eng.setDatabase(db)
    for i, q in enumerate(qs):
        check(eng.scan(dbformat.decode(q)), i, True)
    many, _ = eng.scanMany([dbformat.decode(q) for q in qs])
    for i, res in enumerate(many):
        check(res, i, False)
    check(many[-1], nq - 1, True)
print("ok")
'''


@pytest.fixture(scope="module")
def switch_inputs(oracle, overflow_setup, tmp_path_factory):
    """The database with few long subjects and the overflow subjects, the queries and their oracle results, written
    once for all child processes."""
    from cudasw4_b200 import synth
    sm, qw, dbs = overflow_setup
    db, ref_w = dbs["few"]
    rng = np.random.default_rng(55)
    qs = [synth.random_residues(rng, n) for n in SWITCH_QUERIES[:-1]] + [qw]
    assert qs[-1] is qw and len(qw) == SWITCH_QUERIES[-1]
    k = 11
    arrays = dict(chars=db.chars, offsets=db.offsets, lengths=db.lengths, headers=db.headers,
                  header_offsets=db.header_offsets, nq=len(qs), k=k)
    for i, q in enumerate(qs):
        ref = ref_w if q is qw else oracle.scan(62, q, db, -11, -1)
        s, ids = oracle.topk(ref, k)
        arrays.update({"q%d" % i: q, "ref%d" % i: ref, "s%d" % i: s, "i%d" % i: ids})
    path = str(tmp_path_factory.mktemp("switches") / "inputs.npz")
    np.savez(path, **arrays)
    return sm, db, path


@pytest.mark.gpu
@pytest.mark.parametrize("switch", SWITCHES, ids=lambda sw: ",".join("%s=%s" % kv for kv in sw.items()))
def test_development_switches_change_no_result(switch_inputs, switch):
    """The development switches (read once per process, hence one child process each) select other kernels, shapes,
    launch geometries and pipeline depths; none may change a score, the top-k list or numOverflows."""
    sm, db, path = switch_inputs
    combos = set().union(*(db_combos(q, db.lengths, sm, switch) for q in SWITCH_QUERIES))
    assert combos == set().union(*(db_combos(q, sweep_lengths(sm, "few"), sm, switch) for q in SWITCH_QUERIES))
    env = dict(os.environ, **switch)
    r = subprocess.run([sys.executable, "-c", _SWITCH_CHILD % {"root": ROOT}, path], env=env, capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0 and "ok" in r.stdout, (switch, r.stdout[-500:], r.stderr[-2000:])
