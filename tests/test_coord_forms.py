"""Every form of the alignment coordinate and traceback passes against the oracles, chosen by the plan that runs.

The three passes behind alignmentCoordinates / alignments (kernels_coords.cuh; Engine::coordPasses and
Engine::alignmentTraceback in engine.cu) run each pair either on one warp (16 pairs per CTA) or, when it has more than
one 512-column tile and at least kCoordCtaMinCells cells, on a CTA of W = min(tiles, 16) warps that hand the border
column to each other 32 rows at a time. Pass 2 keeps the form of the whole pair over the smaller rectangle
(qe + 1) x (re + 1); pass 3 picks its own form from the rectangle q[qb..qe] x s[rb..re]. Pairs are launched CTA form
first, in chunks whose scratch fits max_temp_bytes. `coord_plan` and `trace_plan` restate that plan in Python with the
constants parsed from the sources; the CPU tests keep the restatement tied to the code and check that the GPU cases reach
every (pass, form, W, tiles mod W, rows mod 32) combination. The GPU tests (-m gpu) compare every coordinate, count and
CIGAR with the CPU oracles and check kernel launches and cells against the plan.

The score bound (maxEntry x min(q, len) < 2^24) is tested on both sides, and a scan that refuses a query is checked to
leave the handle's last scan, its contexts and its statistics as they were."""
import functools
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "cudasw4_b200", "csrc")
DEFAULT_BUDGET = 4 << 30   # MemoryConfig.maxTempBytes


def _src(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


# ---------------------------------------------------------------------------------------------------------------------
# the plan, restated from engine.cu (Engine::coordPasses, Engine::alignmentTraceback) and kernels_coords.cuh
# ---------------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def constants():
    coords, s32, eng = _src("kernels_coords.cuh"), _src("kernels_s32.cuh"), _src("engine.cu")
    threads = int(re.search(r"constexpr int kCoordThreads = (\d+);", coords).group(1))
    r = int(re.search(r"constexpr int kS32R = (\d+);", s32).group(1))
    shift = int(re.search(r"constexpr long long kCoordCtaMinCells = 1ll << (\d+);", eng).group(1))
    return {"warps": threads // 32, "tile": 32 * r, "min_cells": 1 << shift}


def _up(x, a):
    return (x + a - 1) // a * a


def tiles_of(cols):
    return (cols + constants()["tile"] - 1) // constants()["tile"]


def form_warps(rows, cols):
    """W of a pair or rectangle: 1 (one warp) or the CTA width."""
    c, t = constants(), tiles_of(cols)
    return min(t, c["warps"]) if t > 1 and rows * cols >= c["min_cells"] else 1


def _chunks(order, scratch, budget, start):
    """The greedy chunk loop: lists of positions into `order`; None when one pair alone does not fit (SW4_ERR_NOMEM)."""
    out, pos = [], 0
    while pos < len(order):
        end, used = pos, start
        while end < len(order) and used + scratch[order[end]] <= budget:
            used += scratch[order[end]]
            end += 1
        if end == pos:
            return None
        out.append(order[pos:end])
        pos = end
    return out


def _groups(chunk, warps):
    """CoordGroups of one chunk: (first, count, W); one-warp pairs share a CTA up to kCoordWarps."""
    groups = []
    for k, i in enumerate(chunk):
        W = warps[i]
        if W == 1 and groups and groups[-1][2] == 1 and groups[-1][1] < constants()["warps"]:
            groups[-1][1] += 1
        else:
            groups.append([k, 1, W])
    return [tuple(g) for g in groups]


def coord_plan(qlen, lengths, budget=DEFAULT_BUDGET):
    """Passes 1 and 2: per pair W, the launch order, the scratch of each pair, the chunks and their groups."""
    lengths = [int(n) for n in lengths]
    warps = [form_warps(qlen, n) for n in lengths]
    stride = _up(max(qlen, 1), 32)
    scratch = [_up(n, 16) + (warps[i] * stride * 8 if tiles_of(n) > 1 else 0) for i, n in enumerate(lengths)]
    order = sorted(range(len(lengths)), key=lambda i: (warps[i] == 1, -lengths[i]))   # stable, CTA form first
    chunks = _chunks(order, scratch, budget, 0)
    return {"warps": warps, "order": order, "scratch": scratch, "chunks": chunks,
            "groups": None if chunks is None else [_groups(c, warps) for c in chunks]}


def rect(c):
    """(rows, cols) of pass 3 for oracle coordinates (S, qb, qe, rb, re)."""
    return int(c[2]) - int(c[1]) + 1, int(c[4]) - int(c[3]) + 1


def trace_plan(coords, budget=DEFAULT_BUDGET):
    """Pass 3 and the walk: the same for the traced pairs (score > 0), from their rectangles."""
    traced = [i for i in range(len(coords)) if coords[i][0] > 0]
    warps, scratch = {}, {}
    for i in traced:
        rows, cols = rect(coords[i])
        W = form_warps(rows, cols)
        border = W * _up(rows, 32) if tiles_of(cols) > 1 else 0
        words = tiles_of(cols) * (rows + 31) * 32
        warps[i] = W
        scratch[i] = _up(cols, 16) + border * 8 + words * 8 + _up(rows + cols, 16) + 16
    order = sorted(traced, key=lambda i: (warps[i] == 1, -rect(coords[i])[0] * rect(coords[i])[1]))
    chunks = _chunks(order, scratch, budget, 32)
    return {"warps": warps, "order": order, "scratch": scratch, "chunks": chunks,
            "groups": None if chunks is None else [_groups(c, warps) for c in chunks]}


def expected_stats(qlen, lengths, coords, budget=DEFAULT_BUDGET, trace=False):
    """(kernel launches, cells) of alignmentCoordinates (trace=False) or alignments."""
    cp = coord_plan(qlen, lengths, budget)
    launches = (1 if qlen > 0 else 0) + 2 * len(cp["chunks"])
    cells = sum(qlen * int(n) for n in lengths) + sum((int(c[2]) + 1) * (int(c[4]) + 1) for c in coords if c[0] > 0)
    if trace:
        tp = trace_plan(coords, budget)
        launches += 2 * len(tp["chunks"])
        cells += sum(rect(c)[0] * rect(c)[1] for c in coords if c[0] > 0)
    return launches, cells


def _tile_res(tiles, W):
    r = tiles % W
    return "0" if r == 0 else ("1" if r == 1 else "other")


def _row_res(rows):
    return "<32" if rows < 32 else {0: "0", 1: "1", 31: "31"}.get(rows % 32, "other")


def pass_keys(qlen, lengths, coords):
    """(pass, form, W, tiles mod W, rows mod 32) of every pair in every pass it runs."""
    keys = set()
    for n, c in zip(lengths, coords):
        W = form_warps(qlen, int(n))
        for p, rows, cols in ((1, qlen, int(n)), (2, int(c[2]) + 1, int(c[4]) + 1), (3,) + rect(c)):
            if p > 1 and c[0] <= 0:
                continue      # pass 2 runs no tile and pass 3 does not run for a score-0 pair
            if p == 3:
                W = form_warps(rows, cols)
            if rows <= 0 or cols <= 0:
                continue
            keys.add((p, "warp", 1, "-", "-") if W == 1 else (p, "cta", W, _tile_res(tiles_of(cols), W), _row_res(rows)))
    return keys


def required_items():
    """What the cases must reach: both forms in every pass, every W with every tile residue its pass allows (pass 1 and
    3 have W = tiles up to 16; pass 2 runs the pair's W over a rectangle of any smaller tile count), and the row
    residues of the border hand-over on the CTA form; and both forms in every pass of the PSSM kernels."""
    req = set()
    for p in (1, 2, 3):
        req |= {("form", p, "warp"), ("form", p, "cta"), ("pssm", p, "warp"), ("pssm", p, "cta")}
        req |= {("rows", p, r) for r in ("<32", "0", "1", "31")}
        for W in range(2, constants()["warps"] + 1):
            if p == 2:
                res = ("0", "1") if W == 2 else ("0", "1", "other")
            else:
                res = ("0", "1", "other") if W == constants()["warps"] else ("0",)
            req |= {("W", p, W, r) for r in res}
    return req


def items_of(key, pssm):
    p, form, W, tres, rres = key
    out = {("pssm" if pssm else "form", p, form)}
    if form == "cta" and not pssm:
        out |= {("W", p, W, tres), ("rows", p, rres)}
    return out


# ---------------------------------------------------------------------------------------------------------------------
# the cases of the GPU tests (shared with the CPU coverage test)
# ---------------------------------------------------------------------------------------------------------------------
BLOSUM = 62
CELLS = 1 << 24
THRESHOLD_PAIRS = ((1, CELLS - 1), (1, CELLS), (31, 541200), (31, 541201), (32, 524287), (32, 524288), (33, 508400),
                   (33, 508401), (4096, 4095), (4096, 4096), (40000, 512), (40000, 513))
SWEEP_TILES = tuple(range(2, 18)) + (31, 32, 33, 47)
SWEEP_EXTRA = (1, 16, 17, 512)          # lengths 512 (t - 1) + these
SWEEP_RES = (0, 1, 31)                  # q mod 32
SWEEP_GAPS = ((-11, -1), (-1, 0))
PSSM_SWEEP_TILES = (3, 9, 17, 33)
THIN_ROWS = (31, 32, 33)
THIN_COLS = 600_000
THIN_GAPS = ((0, 0), (-1, 0))


def _codes(s):
    from cudasw4_b200 import dbformat
    return dbformat.encode(s)[0]


def _make_db(seqs):
    """The database and, for each sequence, its id (from_sequences sorts by length)."""
    from cudasw4_b200 import dbformat
    order = np.argsort([len(s) for s in seqs], kind="stable")
    ids = np.empty(len(seqs), np.int64)
    ids[order] = np.arange(len(seqs))
    return dbformat.from_sequences(seqs), ids


def _plant(rng, s, src, end):
    """Put a mutated copy of src (substitutions and indels) into s so that it ends at position `end`."""
    from cudasw4_b200 import synth
    m = synth.mutate(rng, src, 0.1, indels=4)
    m = m[max(0, len(m) - (end + 1)):]
    s[end + 1 - len(m):end + 1] = m


def _sweep_query(t, res):
    """ceil(2^24 / shortest length) rounded up to q mod 32 = res: every pair of tile count t is on the CTA form."""
    q = -(-CELLS // (512 * (t - 1) + 1))
    return q + (res - q) % 32


@functools.lru_cache(maxsize=None)
def threshold_set():
    """One database holding both sides of every threshold pair; (db, [(q codes, ids)])."""
    from cudasw4_b200 import synth
    rng = np.random.default_rng(240)
    queries = {q: synth.random_residues(rng, q) for q in sorted({q for q, _ in THRESHOLD_PAIRS})}
    queries[1][0] = _codes("W")
    seqs = []
    for q, n in THRESHOLD_PAIRS:
        s = synth.random_residues(rng, n)
        if q > 1:   # a homolog of the query a long way into the subject (a large pass-2 rectangle)
            src = queries[q][q // 4: q // 4 + min(q // 2, 300)] if q > 64 else queries[q]
            _plant(rng, s, src, min(n - 1, n // 2 + 700))
        seqs.append(s)
    db, ids = _make_db(seqs)
    cases = [(queries[q], [int(ids[k]) for k, (qq, _) in enumerate(THRESHOLD_PAIRS) if qq == q]) for q in queries]
    return db, cases


@functools.lru_cache(maxsize=None)
def sweep_set():
    """Four subjects per tile count t (lengths 512 (t - 1) + 1 / 16 / 17 / 512), each with a homolog of the query
    crossing a tile edge and ending in tile 0, tile 1, the middle or the last tile; W (11) at both ends of every query
    and subject. (db, {t: ids}, {(t, res): q codes})."""
    from cudasw4_b200 import synth
    rng = np.random.default_rng(2424)
    W = _codes("W")
    queries = {}
    for t in SWEEP_TILES:
        for res in SWEEP_RES:
            q = synth.random_residues(rng, _sweep_query(t, res))
            q[0] = q[-1] = W
            queries[(t, res)] = q
    seqs, owner = [], []
    for t in SWEEP_TILES:
        src_q = queries[(t, 0)]
        for k, extra in enumerate(SWEEP_EXTRA):
            n = 512 * (t - 1) + extra
            s = synth.random_residues(rng, n)
            end_tile = (0, 1, (t - 1) // 2 + 1, t - 1)[k]
            end = min(n - 2, end_tile * 512 + 300)
            plen = min(len(src_q) - 2, 400 if end_tile == 0 else 1500, end - 10)
            a = int(rng.integers(1, len(src_q) - plen))
            _plant(rng, s, src_q[a:a + plen], end)
            s[0] = s[-1] = W
            seqs.append(s)
            owner.append(t)
    db, ids = _make_db(seqs)
    by_t = {t: [int(ids[k]) for k in range(len(seqs)) if owner[k] == t] for t in SWEEP_TILES}
    return db, by_t, queries


@functools.lru_cache(maxsize=None)
def thin_set():
    """Queries of 31 / 32 / 33 residues of W and C, each spread over a 600 k subject whose other residues score <= 0
    against W and C: the alignment spans the whole pair, a rectangle of <= 33 rows and >= 2^24 cells."""
    rng = np.random.default_rng(31)
    W, C = _codes("W"), _codes("C")
    filler = np.array([r for r in range(20) if r not in (W, C, _codes("Y"), _codes("F"))], np.uint8)
    queries, seqs = {}, []
    for rows in THIN_ROWS:
        q = np.where(rng.random(rows) < 0.5, W, C).astype(np.uint8)
        s = filler[rng.integers(0, len(filler), THIN_COLS)]
        s[np.round(np.linspace(0, THIN_COLS - 1, rows)).astype(np.int64)] = q
        queries[rows] = q
        seqs.append(s)
    db, ids = _make_db(seqs)
    return db, {rows: [int(ids[k])] for k, rows in enumerate(THIN_ROWS)}, queries


@functools.lru_cache(maxsize=None)
def mixed_set():
    """One call that mixes CTA pairs of W = 5, 6, 8, 12 and 16 (two of them with homologs whose rectangles are on the
    CTA form in pass 3 too), 37 one-warp pairs (groups of 16, 16 and 5), zero-length subjects, score-0 subjects (all
    code 20) on both forms and duplicate ids, in shuffled order. (db, q codes, ids)."""
    from cudasw4_b200 import synth
    rng = np.random.default_rng(37)
    q = synth.random_residues(rng, 8209)
    cta = [synth.random_residues(rng, n) for n in (2049, 3000, 4000, 6000, 9000)]
    _plant(rng, cta[3], q[1000:5600], 5800)
    _plant(rng, cta[4], q[500:6700], 8500)
    zero = [np.full(2500, 20, np.uint8), np.full(300, 20, np.uint8)]
    warp = [synth.random_residues(rng, int(n)) for n in rng.integers(1, 2000, 32)] + [np.zeros(0, np.uint8)] * 2
    db, ids = _make_db(cta + zero + warp)
    cta_ids = [int(i) for i in ids[:5]] + [int(ids[5])]
    warp_ids = [int(i) for i in ids[6:]]
    order = cta_ids + [cta_ids[3]] + warp_ids + [warp_ids[3], warp_ids[-1]]
    order = [order[i] for i in rng.permutation(len(order))]
    return db, q, order


def _pssm_of(rng, q, spread=2):
    """A positional PSSM around the BLOSUM62 rows of q: each entry moved by up to `spread`, column 20 <= 0."""
    from tests import oracle_lib
    M = oracle_lib.load().matrix(BLOSUM).astype(np.int64)
    P = M[np.minimum(q, 20)] + rng.integers(-spread, spread + 1, (len(q), 21))
    P[:, 20] = np.minimum(P[:, 20], 0)
    return np.clip(P, -128, 127).astype(np.int8)


@functools.lru_cache(maxsize=None)
def pssm_tables():
    """PSSMs of the threshold queries, a subset of the sweep queries and the thin queries (thin: the self score of each
    position drawn from 3..20, every other entry as BLOSUM62, so the spread-out alignment stays the only one)."""
    rng = np.random.default_rng(2112)
    _, thr = threshold_set()
    _, _, sq = sweep_set()
    _, _, tq = thin_set()
    out = {("threshold", len(q)): _pssm_of(rng, q) for q, _ in thr}
    out.update({("sweep", t): _pssm_of(rng, sq[(t, 1)]) for t in PSSM_SWEEP_TILES})
    for rows, q in tq.items():
        P = _pssm_of(rng, q, spread=0)
        P[np.arange(rows), q] = rng.integers(3, 21, rows)
        out[("thin", rows)] = P
    return out


def cases():
    """(name, db, q codes, pssm or None, ids, gop, gex) of every GPU case with oracle coordinates."""
    out = []
    db, thr = threshold_set()
    P = pssm_tables()
    for q, ids in thr:
        out.append(("threshold/q=%d" % len(q), db, q, None, ids, -11, -1))
        out.append(("threshold-pssm/q=%d" % len(q), db, q, P[("threshold", len(q))], ids, -11, -1))
    db, by_t, sq = sweep_set()
    for gop, gex in SWEEP_GAPS:
        for t in SWEEP_TILES:
            for res in SWEEP_RES:
                out.append(("sweep/%d,%d/t=%d/q%%32=%d" % (gop, gex, t, res), db, sq[(t, res)], None, by_t[t], gop, gex))
        for t in PSSM_SWEEP_TILES:
            out.append(("sweep-pssm/%d,%d/t=%d" % (gop, gex, t), db, sq[(t, 1)], P[("sweep", t)], by_t[t], gop, gex))
    db, by_rows, tq = thin_set()
    for gop, gex in THIN_GAPS:
        for rows in THIN_ROWS:
            out.append(("thin/%d,%d/rows=%d" % (gop, gex, rows), db, tq[rows], None, by_rows[rows], gop, gex))
        out.append(("thin-pssm/%d,%d/rows=32" % (gop, gex), db, tq[32], P[("thin", 32)], by_rows[32], gop, gex))
    db, q, ids = mixed_set()
    out.append(("mixed", db, q, None, ids, -11, -1))
    return out


@functools.lru_cache(maxsize=None)
def _oracles():
    from tests import coords_oracle, oracle_lib, pssm_oracle, traceback_oracle
    co = coords_oracle.load(oracle_lib.load())
    return co, traceback_oracle.load(co), pssm_oracle.load()


_WANT = {}


def want_of(name, db, q, pssm, ids, gop, gex):
    """The oracle's Traceback (coordinates, counts, CIGARs) of q against the subjects `ids` (memoised per case)."""
    if name not in _WANT:
        _, tb, po = _oracles()
        subjects = [db.sequence(int(i)) for i in ids]
        _WANT[name] = (tb.traceback(BLOSUM, q, subjects, gop, gex) if pssm is None
                       else po.traceback(pssm, q, subjects, gop, gex))
    return _WANT[name]


def lengths_of(db, ids):
    return [int(db.lengths[int(i)]) for i in ids]


# ---------------------------------------------------------------------------------------------------------------------
# CPU tests
# ---------------------------------------------------------------------------------------------------------------------
def _flat(s):
    return re.sub(r"\s+", " ", s)


def test_plan_matches_engine_source():
    """coord_plan and trace_plan depend on these expressions; if one changes, the restatement must change with it."""
    eng, hdr = _flat(_src("engine.cu")), _flat(_src("kernels_coords.cuh"))
    for expr, count in (
        ("constexpr long long kCoordCtaMinCells = 1ll << 24;", 1),
        # forms: passes 1 and 2 from the pair, pass 3 from the rectangle
        ("return (tiles > 1 && (long long)qlen * len >= kCoordCtaMinCells) ? std::min(tiles, kCoordWarps) : 1;", 1),
        ("return (tiles > 1 && (long long)rowsOf(i) * colsOf(i) >= kCoordCtaMinCells) ? std::min(tiles, kCoordWarps) : 1;", 1),
        ("auto tilesOf = [](int len) { return (len + kCoordTileCols - 1) / kCoordTileCols; };", 1),
        ("auto tilesOf = [](int cols) { return (cols + kCoordTileCols - 1) / kCoordTileCols; };", 1),
        # scratch of the two chunk loops
        ("const size_t borderStride = alignUp((size_t)std::max(qlen, 1), 32);", 1),
        ("size_t b = alignUp((size_t)len, 16); if (tilesOf(len) > 1) b += (size_t)warpsOf(len) * borderStride * sizeof(int2); return b;", 1),
        ("return tilesOf(colsOf(i)) > 1 ? (size_t)warpsOf(i) * alignUp((size_t)rowsOf(i), 32) : 0;", 1),
        ("auto wordsOf = [&](int i) { return (size_t)tilesOf(colsOf(i)) * ((size_t)rowsOf(i) + 31) * 32; };", 1),
        ("auto opsOf = [&](int i) { return alignUp((size_t)rowsOf(i) + (size_t)colsOf(i), 16); };", 1),
        ("return alignUp((size_t)colsOf(i), 16) + borderOf(i) * sizeof(int2) + wordsOf(i) * sizeof(unsigned long long) + opsOf(i) + sizeof(int4);", 1),
        # launch order: stable sorts, CTA form first
        ("std::stable_sort(order.begin(), order.end(), [&](int a, int b) { const int la = lengthOf(a), lb = lengthOf(b); "
         "const bool ca = warpsOf(la) > 1, cb = warpsOf(lb) > 1; if (ca != cb) return ca; return la > lb; });", 1),
        ("std::stable_sort(traced.begin(), traced.end(), [&](int a, int b) { const bool ca = warpsOf(a) > 1, cb = warpsOf(b) > 1; "
         "if (ca != cb) return ca; return (long long)rowsOf(a) * colsOf(a) > (long long)rowsOf(b) * colsOf(b); });", 1),
        ("if (coords[i].score > 0) traced.push_back(i);", 1),
        # chunk loops
        ("size_t bytes = 0; while (end < n && bytes + scratchOf(lengthOf(order[end])) <= budget) bytes += scratchOf(lengthOf(order[end++]));", 1),
        ("size_t bytes = 2 * sizeof(int4); // error counters (padded) while (end < nt && bytes + scratchOf(traced[end]) <= budget) "
         "bytes += scratchOf(traced[end++]);", 1),
        ("if (end == pos) fail(SW4_ERR_NOMEM,", 2),
        # grouping
        ("if (W == 1 && last && last->warps == 1 && last->count < kCoordWarps) last->count++; "
         "else cs.hGroups.p[numGroups++] = CoordGroup{k, 1, W};", 2),
        # stats
        ("cells += (double)qlen * (double)len;", 1),
        ("if (r[0] > 0) cells += (double)(r[2] + 1) * (double)(r[4] + 1);", 1),
        ("cells += (double)rowsOf(i) * (double)colsOf(i);", 1),
        ("launches += 2;", 2),
        ("if (qpad > 0) { convert_query_kernel<<<(qpad + 255) / 256, 256, 0, st>>>(cs.dQueryLetters.p, cs.dQueryCodes.p, qlen, qpad); "
         "SW4_CUDA(cudaGetLastError()); launches++; }", 1),
    ):
        assert eng.count(expr) == count, expr
    for expr in ("constexpr int kCoordWarps = kCoordThreads / 32;", "constexpr int kCoordR = kS32R;",
                 "constexpr int kCoordTileCols = 32 * kCoordR;", "const int W = g.warps;",
                 "const int slot = warp / W, wi = warp % W;", "q = S > 0 ? qe + 1 : 0;", "len = S > 0 ? re + 1 : 0;",
                 "const int tiles = q > 0 ? (len + kCoordTileCols - 1) / kCoordTileCols : 0;",
                 "for (int tile = wi; tile < tiles; tile += W) {",
                 "const int borderStride = TRACE ? (q + 31) & ~31 : prm.borderStride;"):
        assert expr in hdr, expr
    assert constants() == {"warps": 16, "tile": 512, "min_cells": 1 << 24}


def test_plan_of_the_threshold_and_mixed_cases():
    """The forms the threshold pairs are chosen for, and the groups of the mixed launch."""
    for q, n in THRESHOLD_PAIRS:
        want = 1 if q * n < CELLS or n <= 512 else min(tiles_of(n), 16)
        assert form_warps(q, n) == want and (want > 1) == (q * n >= CELLS and n > 512), (q, n)
    assert form_warps(40000, 512) == 1 and form_warps(40000, 513) == 2
    for t in SWEEP_TILES:
        for res in SWEEP_RES:
            q = _sweep_query(t, res)
            assert q % 32 == res and all(form_warps(q, 512 * (t - 1) + e) == min(t, 16) for e in SWEEP_EXTRA), (t, res)
    db, q, ids = mixed_set()
    plan = coord_plan(len(q), lengths_of(db, ids))
    assert len(plan["chunks"]) == 1
    groups = plan["groups"][0]
    assert sorted(W for _, _, W in groups if W > 1) == [5, 5, 6, 8, 12, 12, 16]
    assert [c for _, c, W in groups if W == 1] == [16, 16, 5]
    L = lengths_of(db, ids)
    assert L.count(0) >= 3 and len(set(ids)) < len(ids)


def test_oracle_coordinates_of_the_constructed_cases():
    """Each case does what it was built for (from the oracle): the thin rectangles span the subject on <= 33 rows, the
    planted homologs of the mixed case are traced on the CTA form, and the all-code-20 subjects score 0."""
    for name, db, q, pssm, ids, gop, gex in cases():
        if name.startswith("thin"):
            c = want_of(name, db, q, pssm, ids, gop, gex).coordinates[0]
            rows, cols = rect(c)
            assert rows == len(q) <= 33 and rows * cols >= CELLS and cols == THIN_COLS, (name, c.tolist())
            assert form_warps(rows, cols) == 16
        if name == "mixed":
            coords = want_of(name, db, q, pssm, ids, gop, gex).coordinates
            tp = trace_plan(coords)
            assert sum(W > 1 for W in tp["warps"].values()) >= 3, tp["warps"]   # (one of the two planted pairs appears twice)
            L = lengths_of(db, ids)
            assert [int(c[0]) for c, n in zip(coords, L) if n in (0, 300, 2500)] == [0] * sum(n in (0, 300, 2500) for n in L)


def test_cases_reach_every_reachable_path():
    covered, first = set(), {}
    for name, db, q, pssm, ids, gop, gex in cases():
        want = want_of(name, db, q, pssm, ids, gop, gex)
        for key in pass_keys(len(q), lengths_of(db, ids), want.coordinates):
            items = items_of(key, pssm is not None)
            covered |= items
            first.setdefault(key + (("pssm",) if pssm is not None else ()), name)
    missing = required_items() - covered
    assert not missing, sorted(missing, key=str)
    # which case reaches what (pytest -rA -s shows it)
    for key in sorted(first, key=str):
        print("%-42s %s" % (key, first[key]))


# ---------------------------------------------------------------------------------------------------------------------
# GPU tests
# ---------------------------------------------------------------------------------------------------------------------
def _engine(**kw):
    import cudasw4_b200 as sw
    return sw.CudaSW4(deviceIds=[0], **kw)


def _assert_same(got, want, ctx=None):
    from tests.test_traceback import _assert_same as same
    same(got, want, ctx)


def _check_case(eng, name, db, q, pssm, ids, gop, gex, budget=DEFAULT_BUDGET):
    """alignmentCoordinates and alignments of one case against the oracle, with launches and cells from the plan."""
    import cudasw4_b200 as sw
    from cudasw4_b200 import dbformat
    want = want_of(name, db, q, pssm, ids, gop, gex)
    letters = dbformat.decode(q)
    L = lengths_of(db, ids)
    st = sw.BenchmarkStats()
    got = eng.alignmentCoordinates(letters, ids, stats=st, pssm=pssm)
    assert (got == want.coordinates).all(), (name, np.nonzero((got != want.coordinates).any(axis=1))[0][:4])
    assert (st.kernelLaunches, st.cells) == expected_stats(len(q), L, want.coordinates, budget), name
    got = eng.alignments(letters, ids, stats=st, pssm=pssm)
    _assert_same(got, want, name)
    assert (st.kernelLaunches, st.cells) == expected_stats(len(q), L, want.coordinates, budget, trace=True), name


def _run_cases(prefixes, gaps=None):
    byname = {}
    for c in cases():
        if c[0].split("/")[0] in prefixes and (gaps is None or (c[5], c[6]) == gaps):
            byname.setdefault(id(c[1]), []).append(c)
    for group in byname.values():
        with _engine(numTop=4, gop=group[0][5], gex=group[0][6]) as eng:
            eng.setDatabase(group[0][1])
            for c in group:
                eng.setGapScores(c[5], c[6])
                _check_case(eng, *c)


@pytest.mark.gpu
def test_threshold_pairs():
    """Both sides of kCoordCtaMinCells at q = 1, 31, 32, 33 and 4096, and one tile with >= 2^24 cells (one warp)
    against two tiles (W = 2), for sequence and PSSM queries."""
    _run_cases(("threshold", "threshold-pssm"))


@pytest.mark.gpu
@pytest.mark.parametrize("gaps", SWEEP_GAPS)
def test_tile_sweep(gaps):
    """W = 2..16 and tiles = kW, kW + 1, kW - 1 in every pass, q mod 32 = 0, 1, 31; homologs ending in tile 0, tile 1,
    the middle and the last tile (pass 2 on a W = 16 pair whose rectangle has one or two tiles)."""
    _run_cases(("sweep", "sweep-pssm"), gaps)


@pytest.mark.gpu
def test_thin_rectangles():
    """31 / 32 / 33-row alignments across 600 k columns: the border arrives as one partial 32-row chunk on the CTA
    form, in all three passes."""
    _run_cases(("thin", "thin-pssm"))


@pytest.mark.gpu
def test_mixed_launch():
    _run_cases(("mixed",))


def _prefix_budgets(plan, start):
    """Budgets exactly equal to the scratch of the first j pairs of the launch order: one inside the CTA block (j = 2),
    one at the form boundary, and each of those minus 1."""
    order, scratch, warps = plan["order"], plan["scratch"], plan["warps"]
    ncta = sum(warps[i] > 1 for i in order)
    assert ncta >= 3
    out = []
    for j in (2, ncta):
        b = start + sum(scratch[i] for i in order[:j])
        out += [(b, j), (b - 1, j - 1)]   # (budget, pairs of the first chunk)
    return out


@pytest.mark.gpu
def test_chunk_edges():
    """Both chunk loops at budgets on the edges of the mixed case's pairs give the same arrays, with the predicted
    number of chunks in kernelLaunches; a budget one byte short of the largest single pair is SW4_ERR_NOMEM."""
    import cudasw4_b200 as sw
    from cudasw4_b200 import dbformat
    db, q, ids = mixed_set()
    L = lengths_of(db, ids)
    want = want_of("mixed", db, q, None, ids, -11, -1)
    letters = dbformat.decode(q)
    cplan = coord_plan(len(q), L)
    tplan = trace_plan(want.coordinates)
    with _engine(numTop=4) as eng:
        eng.setDatabase(db)
        for budget, first in _prefix_budgets(cplan, 0):
            eng.setMemoryConfig(sw.MemoryConfig(maxTempBytes=budget))
            p = coord_plan(len(q), L, budget)
            assert p["chunks"] is not None and len(p["chunks"][0]) == first and len(p["chunks"]) > 1
            st = sw.BenchmarkStats()
            got = eng.alignmentCoordinates(letters, ids, stats=st)
            assert (got == want.coordinates).all(), budget
            assert (st.kernelLaunches, st.cells) == expected_stats(len(q), L, want.coordinates, budget), budget
        for budget, first in _prefix_budgets(tplan, 32):
            eng.setMemoryConfig(sw.MemoryConfig(maxTempBytes=budget))
            assert coord_plan(len(q), L, budget)["chunks"] is not None
            p = trace_plan(want.coordinates, budget)
            assert p["chunks"] is not None and len(p["chunks"][0]) == first and len(p["chunks"]) > 1
            st = sw.BenchmarkStats()
            _assert_same(eng.alignments(letters, ids, stats=st), want, budget)
            assert (st.kernelLaunches, st.cells) == expected_stats(len(q), L, want.coordinates, budget, trace=True), budget
        # one byte short of the largest pair of each loop
        big = cplan["order"][0]
        eng.setMemoryConfig(sw.MemoryConfig(maxTempBytes=cplan["scratch"][big] - 1))
        with pytest.raises(sw.SW4Error) as e:
            eng.alignmentCoordinates(letters, [ids[big]])
        assert e.value.code == -4
        big = tplan["order"][0]
        budget = 32 + tplan["scratch"][big] - 1
        assert coord_plan(len(q), [L[big]], budget)["chunks"] is not None
        eng.setMemoryConfig(sw.MemoryConfig(maxTempBytes=budget))
        with pytest.raises(sw.SW4Error) as e:
            eng.alignments(letters, [ids[big]])
        assert e.value.code == -4
        assert (eng.alignmentCoordinates(letters, [ids[big]]) == want.coordinates[[big]]).all()


@pytest.mark.gpu
def test_empty_query():
    import cudasw4_b200 as sw
    db, _, ids = mixed_set()
    with _engine(numTop=4) as eng:
        eng.setDatabase(db)
        st = sw.BenchmarkStats()
        got = eng.alignments("", ids, stats=st)
        assert (got.coordinates == [[0, -1, -1, -1, -1]] * len(ids)).all()
        assert got.cigars == [""] * len(ids) and (got.counts == 0).all()
        assert (st.kernelLaunches, st.cells) == (2, 0)
        assert (eng.alignmentCoordinates("", ids, stats=st) == got.coordinates).all()
        assert (st.kernelLaunches, st.cells) == (2, 0)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the 2^24 score bound on both sides, and a refused scan
# ---------------------------------------------------------------------------------------------------------------------
BOUND_OK = (1 << 24) // 127            # 127 x 132104 = 16777208
BLOSUM_REFUSED = (1 << 24) // 11 + 1   # 11 x 1525202 >= 2^24


def _single_entry_pssm(n, p, r):
    P = np.full((n, 21), -1, np.int8)
    P[p, r] = 127
    return P


@pytest.mark.gpu
def test_score_bound_accepted_side():
    """A PSSM whose only positive entry is pssm[p][r] = 127, q = len = 132104 (127 x 132104 = 16777208 < 2^24): the
    subject holds r only at position j, so the answer is S = 127 at (p, p, j, j). The largest CTA-form pair here (259
    tiles, q mod 32 = 8), through scan, alignmentCoordinates and alignments."""
    from cudasw4_b200 import dbformat, synth
    n, p, j = BOUND_OK, 70001, 91234
    assert 127 * n < 1 << 24 and tiles_of(n) == 259 and n % 32 == 8 and form_warps(n, n) == 16
    rng = np.random.default_rng(127)
    r = _codes("W")
    others = np.array([c for c in range(20) if c != r], np.uint8)
    s = others[rng.integers(0, len(others), n)]
    s[j] = r
    q = synth.random_residues(rng, n)
    q[p] = r
    P = _single_entry_pssm(n, p, r)
    db = dbformat.from_sequences([s])
    with _engine(numTop=1) as eng:
        eng.setDatabase(db)
        res = eng.scan(dbformat.decode(q), pssm=P)
        assert res.scores == [127] and res.referenceIds == [0]
        assert (eng.alignmentCoordinates(dbformat.decode(q), [0], pssm=P) == [[127, p, p, j, j]]).all()
        for letter, cigar, counts in ((r, "1=", [1, 1, 1, 0]), (_codes("A"), "1X", [1, 0, 1, 0])):
            q[p] = letter
            got = eng.alignments(dbformat.decode(q), [0], pssm=P)
            assert got.coordinates.tolist() == [[127, p, p, j, j]] and got.cigars == [cigar] and got.counts.tolist() == [counts]


@pytest.mark.gpu
def test_score_bound_refused_side():
    """One residue more is refused by all three calls (SW4_ERR_INVALID), and so is BLOSUM62 at 11 x 1525202."""
    import cudasw4_b200 as sw
    from cudasw4_b200 import dbformat, synth
    rng = np.random.default_rng(128)
    n = BOUND_OK + 1
    P = _single_entry_pssm(n, 5, 0)
    q = dbformat.decode(synth.random_residues(rng, n))
    with _engine(numTop=1) as eng:
        eng.setDatabase(dbformat.from_sequences([synth.random_residues(rng, n)]))
        for call in (lambda: eng.scan(q, pssm=P), lambda: eng.alignmentCoordinates(q, [0], pssm=P),
                     lambda: eng.alignments(q, [0], pssm=P)):
            with pytest.raises(sw.SW4Error) as e:
                call()
            assert e.value.code == -1 and "2^24" in str(e.value)
    qb = dbformat.decode(synth.random_residues(rng, BLOSUM_REFUSED))
    with _engine(numTop=1) as eng:
        eng.setDatabase(dbformat.from_sequences([synth.random_residues(rng, BLOSUM_REFUSED)]))
        for call in (lambda: eng.scan(qb), lambda: eng.alignmentCoordinates(qb, [0])):
            with pytest.raises(sw.SW4Error) as e:
                call()
            assert e.value.code == -1 and "2^24" in str(e.value)


def _refusal_scenarios(oracle):
    """A refused scan or scanMany leaves the handle as it was: the last scan's scores, histogram and statistics, and
    every following scan equals the oracle. The refusals: the score bound of a PSSM query (the last of four queries),
    and max_temp_bytes too small for the border rows of a 70 k query (also the last)."""
    import cudasw4_b200 as sw
    from cudasw4_b200 import dbformat, synth
    rng = np.random.default_rng(1184)
    seqs = [synth.random_residues(rng, int(n)) for n in rng.integers(30, 900, 300)]
    seqs.append(synth.random_residues(rng, BOUND_OK + 1))
    db = dbformat.from_sequences(seqs)
    qs = [synth.random_residues(rng, int(n)) for n in (180, 260, 333)]
    M = oracle.matrix(BLOSUM)
    ps = [M[np.minimum(x, 20)].astype(np.int8) for x in qs]       # PSSMs that score as the matrix does
    big = synth.random_residues(rng, BOUND_OK + 1)
    big_p = _single_entry_pssm(len(big), 9, 3)
    refs = [oracle.scan(BLOSUM, x, db, -11, -1) for x in qs]
    letters = [dbformat.decode(x) for x in qs]

    def all_scores(eng):
        scores, ids = eng.lastScanAllScores()
        got = np.empty(db.num_sequences, np.int32)
        got[ids] = scores
        return got

    def check(res, ref):
        s, i = oracle.topk(ref, 10)
        assert res.scores == s.tolist() and res.referenceIds == i.tolist()

    def state(eng):
        return all_scores(eng), [h.copy() for h in eng.lastScoreHistogram()], repr(eng.lastScoreStatistics())  # (repr: NaN == NaN)

    def same_state(a, b):
        assert (a[0] == b[0]).all() and all((x == y).all() for x, y in zip(a[1], b[1])) and a[2] == b[2]

    for temp, refused in ((4 << 30, "bound"), (4 << 20, "scratch")):
        with _engine(numTop=10, memoryConfig=sw.MemoryConfig(maxTempBytes=temp)) as eng:
            eng.setDatabase(db)
            eng.setScoreStatistics(True)
            check(eng.scan(letters[0]), refs[0])
            before = state(eng)
            assert (before[0] == refs[0]).all()
            for attempt in range(2):
                with pytest.raises(sw.SW4Error) as e:
                    if refused == "bound" and attempt == 0:
                        eng.scan(dbformat.decode(big), pssm=big_p)
                    elif refused == "bound":
                        eng.scanMany(letters + [dbformat.decode(big)], pssm=ps + [big_p])
                    else:
                        eng.scanMany(letters + [dbformat.decode(synth.random_residues(rng, 70000))])
                assert e.value.code == (-1 if refused == "bound" else -4), str(e.value)
                same_state(state(eng), before)
            check(eng.scan(letters[0]), refs[0])
            assert (all_scores(eng) == refs[0]).all()
            res, _ = eng.scanMany(letters[:2])
            check(res[0], refs[0])
            check(res[1], refs[1])
            assert (all_scores(eng) == refs[1]).all()
            res, _ = eng.scanMany(letters, pssm=ps)
            for r, ref in zip(res, refs):
                check(r, ref)


@pytest.mark.gpu
def test_refused_scan_changes_nothing(oracle):
    _refusal_scenarios(oracle)


_CHILD = """
import sys
sys.path.insert(0, %(root)r)
from tests import oracle_lib
from tests.test_coord_forms import _refusal_scenarios
_refusal_scenarios(oracle_lib.load())
print("ok")
"""


@pytest.mark.gpu
@pytest.mark.parametrize("depth", ["1", "16"])
def test_refused_scan_changes_nothing_at_pipeline_depth(depth):
    env = dict(os.environ, SW4_PIPELINE=depth)
    r = subprocess.run([sys.executable, "-c", _CHILD % {"root": ROOT}], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "ok" in r.stdout, (depth, r.stdout[-500:], r.stderr[-2000:])
