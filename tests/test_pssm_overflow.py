"""PSSM scores on the 16-bit overflow boundaries in every length class and on every scoring-kernel path.

With a sequence query no subject of at most 1024 residues can reach the re-scoring threshold (25000): the largest BLOSUM
entry is 15. A PSSM entry can be 127, so from 197 residues on a subject of any single-segment class can cross it, wrap
the packed 16-bit scores and land on the overflow list of a short-class kernel. These tests build, for each query
length, a PSSM whose rows give 127 to one consensus residue and a clearly negative score to most others (at gap scores
of -11 / -1, random subjects still chain consensus matches through gaps and score in the thousands, so most of them
pass 2048 and the longer ones 25000 against long queries), and subjects
whose exact score is a chosen boundary value: both sides of 25000, 25126 (24999 + 127, the alignment ending on the
crossing cell), the first and second 16-bit wrap, the class maximum, and 2047 / 2048 at 240 / 241 residues (Half2's
numOverflows rule and its length gate). Each subject sits twice in a row in its class, in both halves of a packed pair,
next to the subjects of both sweep databases of test_kernel_paths.py. The GPU tests (-m gpu) compare every score, the
top-k list and numOverflows with tests/pssm_oracle.cpp on every kernel path, under every development switch, in every
database mode, through scanMany, and compare the coordinates and traceback of the boundary subjects."""
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

from tests import pssm_oracle as pssm_oracle_lib
from tests.test_kernel_paths import (SWITCHES, _all_scores, _sm_counts, class_of, constants, db_combos,  # noqa: F401
                                     kernel_path, long_items_kind, reachable_combos, sweep_dbs, sweep_lengths)
from tests.test_pssm import valid_column20

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
THRESHOLD = 25000
# both sides of every long-class threshold (785 moves re-scoring to the s32 array), 196 / 197 (the first length at which
# a full diagonal passes 25000), 258 / 259 and 516 / 517 (where 32767 and 65536 first fit), and long queries
SWEEP_QUERIES = (112, 113, 196, 197, 208, 209, 256, 257, 258, 259, 400, 401, 516, 517, 576, 577, 784, 785, 1024, 2002,
                 3400)
# (112: the long class's one-row multi-segment kernel under SW4_NO_TWO_ROW_MULTI runs only below 113)
SWITCH_QUERIES = (112, 300, 784, 1100)
BOUNDARY_QUERIES = tuple(sorted(set(SWEEP_QUERIES) | set(SWITCH_QUERIES)))
# (query length, gop, gex): the ends of the accepted gap range with rows that hold -128 (the sentinel and the E / F floors)
GAP_CASES = ((259, -4096, -4096), (259, 0, 0), (785, -4096, -4096), (785, 0, 0))
TRACEBACK_QUERIES = (259, 1024)
WRAP_TARGETS = (24999, 25000, 25126, 32767, 32768, 32894, 65535, 65536)
GATE_TARGETS = (2047, 2048)   # Half2's numOverflows threshold, at 240 (not counted) and 241 (counted) residues
ODD_CLASS_CAP = 224           # the class whose last subject is a boundary subject without a partner (subject1 = -1)
COL20_ZERO_QUERY = 401        # column 20 = 0, the largest value allowed: padding and code-20 letters then score 0


# ---------------------------------------------------------------------------------------------------------------------
# boundary PSSMs and the placement of their subjects (pure functions of the query length)
# ---------------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def boundary_pssm(n):
    """(consensus residues, second residues, PSSM) of an n-residue query. Row p scores 127 for consensus[p] and a
    random 1..126 for second[p] (so that changing one or two residues of a consensus stretch can take any amount off its
    score); the other columns 0-19 are uniform in [-127, 8] with 3 % at -128, a mean of about -60, so that random
    subjects score a few hundred at most. Column 20 is -128, or 0 (the largest value allowed: padding and code-20
    letters then score 0) for COL20_ZERO_QUERY."""
    rng = np.random.default_rng(9000 + n)
    consensus = rng.integers(0, 20, n).astype(np.uint8)
    second = ((consensus + rng.integers(1, 20, n)) % 20).astype(np.uint8)
    P = rng.integers(-127, 9, (n, 21))
    P[rng.random((n, 21)) < 0.03] = -128
    P[:, 20] = 0 if n == COL20_ZERO_QUERY else -128
    P[np.arange(n), second] = rng.integers(1, 127, n)
    P[np.arange(n), consensus] = 127
    return consensus, second, valid_column20(P).astype(np.int8)


def _class_bounds():
    """(lowest length, capacity) of every length class; the long class has capacity None."""
    out, lo = [], 1
    for _, _, cap, _, multi in constants()["classes"]:
        out.append((lo, None if multi else cap))
        lo = cap + 1
    return out


def residues_needed(target):
    return -(-target // 127)


def placements(n):
    """(target, subject length) of every boundary subject of the n-residue query. Every class from 193 residues on gets
    the wrap targets that fit min(n, capacity) residues; each class gets its maximum 127 x min(capacity, n) (classes
    above n only the first of them and the long class); 240 and 241 residues get 2047 and 2048."""
    out = []
    first_above = True
    for ci, (lo, cap) in enumerate(_class_bounds()):
        room = n if cap is None else min(n, cap)
        if cap is not None and cap >= n:
            if not first_above:
                continue
            first_above = False
        targets = [t for t in WRAP_TARGETS if residues_needed(t) <= room] + [127 * room]
        for i, t in enumerate(dict.fromkeys(targets)):
            m = residues_needed(t)
            if cap is None:
                length = max(m, lo) + 7 * i
            else:
                length = cap if i % 2 == 0 else max(lo, m)
            out.append((t, length))
    out += [(t, length) for t in GATE_TARGETS for length in (240, 241)]
    return out


def _tune(pssm_oracle, n, target, length, rng):
    """A subject of `length` residues whose exact score against the boundary PSSM of n residues is `target`: a stretch
    of ceil(target / 127) consensus residues, with one or two inner residues changed to their row's second residue so
    that the stretch loses 127 - (target mod 127), between code-20 letters (with gap scores as cheap as -11 / -1 against
    entries of 127, random flanks would add to the score through gapped chains of consensus matches). The oracle chooses
    among the candidates."""
    consensus, second, P = boundary_pssm(n)
    m = residues_needed(target)
    loss = 127 * m - target
    gain = P[np.arange(n), second].astype(np.int64)
    cands = []
    for _ in range(40):
        a = int(rng.integers(0, n - m + 1))
        s = np.full(length, 20, np.uint8)
        b = int(rng.integers(0, length - m + 1))
        s[b:b + m] = consensus[a:a + m]
        if loss:
            # the first and last cells stay 127, so that the best alignment spans the stretch and ends on its last cell
            inner = np.arange(1, m - 1)
            lost = 127 - gain[a + inner]
            one = inner[lost == loss]
            if len(one):
                i = int(one[int(rng.integers(0, len(one)))])
                s[b + i] = second[a + i]
            else:
                pairs = [(int(i), int(j)) for i in inner for j in inner[(inner > i) & (lost == loss - lost[i - 1])]]
                if not pairs:
                    continue
                i, j = pairs[int(rng.integers(0, len(pairs)))]
                s[b + i], s[b + j] = second[a + i], second[a + j]
        cands.append(s)
        if len(cands) == 8:
            break
    assert cands, (n, target, length)
    scores = pssm_oracle.coords(P, cands, -11, -1)[:, 0]
    hit = np.nonzero(scores == target)[0]
    assert len(hit), (n, target, length, sorted(set(scores.tolist())))
    return cands[int(hit[0])]


def _class_index(cap):
    return next(i for i, (_, c) in enumerate(_class_bounds()) if c == cap)


def layout(sm, kind):
    """Subject lengths of the sweep database `kind` (ascending, as stored) followed by the boundary subjects, each twice
    in a row, and one more copy at the end of the ODD_CLASS_CAP class if that leaves it with an even count; and the
    (query length, target) of every boundary subject (None for the sweep subjects)."""
    lengths = sorted(int(x) for x in sweep_lengths(sm, kind))
    tags = [None] * len(lengths)
    for n in BOUNDARY_QUERIES:
        for t, length in placements(n):
            lengths += [length, length]
            tags += [(n, t, length)] * 2
    odd = _class_index(ODD_CLASS_CAP)
    if sum(class_of(x) == odd for x in lengths) % 2 == 0:
        n = max(BOUNDARY_QUERIES)
        t = max(t for t, length in placements(n) if length == ODD_CLASS_CAP)
        lengths.append(ODD_CLASS_CAP)
        tags.append((n, t, ODD_CLASS_CAP))
    return lengths, tags


def stored_order(lengths, tags):
    """Lengths and tags in the order of the database (a stable sort by length) and the class of every subject."""
    order = np.argsort(np.asarray(lengths), kind="stable")
    L = np.asarray(lengths)[order]
    return L, [tags[i] for i in order], np.array([class_of(int(x)) for x in L])


def _items(L):
    return (int((np.asarray(L) > 1024).sum()) + 1) // 2


def coverage_cases(sm):
    """(case name, combinations it reaches) for every GPU case of this file."""
    cases = []
    L = {kind: layout(sm, kind)[0] for kind in ("few", "many")}
    for kind in ("few", "many"):
        for q in SWEEP_QUERIES:
            cases.append(("sweep/%s/q=%d" % (kind, q), db_combos(q, L[kind], sm)))
    for q, gop, gex in GAP_CASES:
        cases.append(("gaps/%d,%d/q=%d" % (gop, gex, q), db_combos(q, L["few"], sm)))
    for sw in SWITCHES:
        for q in SWITCH_QUERIES:
            cases.append(("switch/%s/q=%d" % (",".join("%s=%s" % kv for kv in sw.items()), q),
                          db_combos(q, L["few"], sm, sw)))
    return cases


@functools.lru_cache(maxsize=None)
def boundary_subjects(n):
    """{(target, length): subject} for the n-residue boundary PSSM."""
    oracle = pssm_oracle_lib.load()
    rng = np.random.default_rng(77 + n)
    return {(t, length): _tune(oracle, n, t, length, rng) for t, length in placements(n)}


@pytest.fixture(scope="module")
def pssm_oracle():
    return pssm_oracle_lib.load()


# ---------------------------------------------------------------------------------------------------------------------
# CPU tests
# ---------------------------------------------------------------------------------------------------------------------
def test_placements_reach_every_boundary():
    for n in BOUNDARY_QUERIES:
        got = placements(n)
        for t, length in got:
            assert residues_needed(t) <= min(n, length), (n, t, length)
        targets = {t for t, _ in got}
        for t in WRAP_TARGETS:
            assert (t in targets) == (residues_needed(t) <= n), (n, t)
        assert {(t, length) for t in GATE_TARGETS for length in (240, 241)} <= set(got)
    # 25126 ends on the cell that crosses 25000 from 24999: ceil(25126 / 127) residues
    assert residues_needed(25126) == 198 and residues_needed(25000) == 197 and 127 * 196 < 25000
    assert [n for n in BOUNDARY_QUERIES if residues_needed(32767) <= n][0] == 259 and residues_needed(32894) == 260
    assert [n for n in BOUNDARY_QUERIES if residues_needed(65536) <= n][0] == 517


def test_boundary_subjects_score_their_targets(pssm_oracle):
    for n in BOUNDARY_QUERIES:
        consensus, second, P = boundary_pssm(n)
        assert (P[np.arange(n), consensus] == 127).all() and (P[:, 20] == (0 if n == COL20_ZERO_QUERY else -128)).all()
        assert P[:, :20].astype(np.int64).mean() < -40 and (P == -128).any()
        subjects = boundary_subjects(n)
        keys = list(subjects)
        scores = pssm_oracle.coords(P, [subjects[key] for key in keys], -11, -1)[:, 0]
        assert scores.tolist() == [t for t, _ in keys], n
        assert [len(subjects[key]) for key in keys] == [length for _, length in keys]


def _numpy_gotoh_rows(P, s, gop, gex):
    from tests.test_kernel_paths import numpy_gotoh
    return numpy_gotoh(P, np.arange(len(P)), s, gop, gex)   # query position i scores row i


def test_oracle_matches_numpy_gotoh_on_boundary_subjects(pssm_oracle):
    """The restatement against a plain int64 Gotoh given the PSSM rows, on boundary subjects and random ones, at the
    default gap scores and at both ends of the accepted range."""
    rng = np.random.default_rng(12)
    checked = 0
    for n in (q for q in BOUNDARY_QUERIES if q <= 300):
        consensus, _, P = boundary_pssm(n)
        subjects = list(boundary_subjects(n).items())
        pick = [subjects[int(i)] for i in rng.choice(len(subjects), min(4, len(subjects)), replace=False)]
        pick.append(((None, 60), rng.integers(0, 21, 60).astype(np.uint8)))
        for gop, gex in ((-11, -1), (-4096, -4096), (0, 0)):
            got = pssm_oracle.coords(P, [s for _, s in pick], gop, gex)[:, 0]
            for ((t, _), s), g in zip(pick, got):
                assert g == _numpy_gotoh_rows(P, s, gop, gex), (n, t, gop, gex)
                if t is not None and (gop, gex) == (-11, -1):
                    assert g == t
                checked += 1
    assert checked >= 60


@pytest.mark.parametrize("sm", _sm_counts())
def test_cases_reach_every_reachable_path(sm):
    """The GPU cases below reach every (kernel, shape, re-scoring kernel) combination the rule can produce, and every
    class from 208 columns on holds, in one case at least, subjects of >= 25000 in both halves of a packed pair."""
    for kind in ("few", "many"):
        assert long_items_kind(_items(layout(sm, kind)[0]), sm) == kind
    cases = coverage_cases(sm)
    covered = set().union(*(combos for _, combos in cases))
    reachable = reachable_combos(sm)
    assert not reachable - covered, sorted(reachable - covered, key=str)
    assert covered <= reachable
    # both halves: position parity inside the class, for one query's subjects of >= 25000
    for kind in ("few", "many"):
        L, tags, cls = stored_order(*layout(sm, kind))
        first = {c: int(np.searchsorted(cls, c)) for c in set(cls.tolist())}
        for ci, (lo, cap) in enumerate(_class_bounds()):
            if cap is not None and cap < 208:
                continue
            halves = {}
            for i, tag in enumerate(tags):
                if tag and cls[i] == ci and tag[1] >= THRESHOLD and tag[0] in SWEEP_QUERIES:
                    halves.setdefault(tag[0], set()).add((i - first[ci]) % 2)
            assert any(h == {0, 1} for h in halves.values()), (kind, ci, cap, halves)
        # the lone half of the last pair of ODD_CLASS_CAP's class is a subject of >= 25000
        odd = _class_index(ODD_CLASS_CAP)
        members = np.nonzero(cls == odd)[0]
        assert len(members) % 2 == 1 and tags[members[-1]] and tags[members[-1]][1] >= THRESHOLD, kind
    first = {}
    for name, combos in cases:
        for cmb in combos:
            first.setdefault(cmb, name)
    for cmb in sorted(first, key=str):
        print("%-45s %s" % (cmb, first[cmb]))


# ---------------------------------------------------------------------------------------------------------------------
# GPU tests
# ---------------------------------------------------------------------------------------------------------------------
class BoundaryDB:
    """A sweep database with the boundary subjects, their (query length, target, length) tags in database order, and
    the oracle's scores per (query length, gop, gex), computed on first use."""

    def __init__(self, sm, kind, base, pssm_oracle):
        from cudasw4_b200 import dbformat
        lengths, tags = layout(sm, kind)
        assert lengths[:base.num_sequences] == base.lengths.tolist()
        seqs = [base.sequence(i).copy() for i in range(base.num_sequences)]
        seqs += [boundary_subjects(n)[(t, length)].copy() for n, t, length in tags[base.num_sequences:]]
        self.db = dbformat.from_sequences(seqs)
        self.L, self.tags, self.cls = stored_order(lengths, tags)
        assert (self.L == self.db.lengths).all()
        assert long_items_kind(_items(self.L), sm) == kind
        self.sm, self.kind, self.oracle, self._refs = sm, kind, pssm_oracle, {}

    def ref(self, n, gop=-11, gex=-1):
        if (n, gop, gex) not in self._refs:
            ref = self.oracle.coords(boundary_pssm(n)[2], self.db, gop, gex)[:, 0]
            if (gop, gex) == (-11, -1):
                mine = [i for i, tag in enumerate(self.tags) if tag and tag[0] == n]
                assert ref[mine].tolist() == [self.tags[i][1] for i in mine], n
            self._refs[(n, gop, gex)] = ref
        return self._refs[(n, gop, gex)]

    def ids_of(self, n):
        return np.array([i for i, tag in enumerate(self.tags) if tag and tag[0] == n], dtype=np.int64)

    def describe(self, n, idx, got, ref, switches=None):
        """class, half of the packed pair, kernel path, reported and true score of the subjects at idx"""
        first = {c: int(np.searchsorted(self.cls, c)) for c in set(self.cls.tolist())}
        out = []
        for i in idx[:8]:
            c = int(self.cls[i])
            count = int((self.cls == c).sum())
            out.append(dict(id=int(i), length=int(self.L[i]), cls=c, half=(int(i) - first[c]) % 2,
                            path=kernel_path(n, c, (count + 1) // 2, self.sm, switches), got=int(got[i]),
                            true=int(ref[i]), tag=self.tags[i]))
        return out


@pytest.fixture(scope="module")
def boundary_dbs(pssm_oracle, sweep_dbs):
    sm, dbs = sweep_dbs
    return {kind: BoundaryDB(sm, kind, dbs[kind], pssm_oracle) for kind in ("few", "many")}


def _query(n):
    from cudasw4_b200 import dbformat
    consensus, _, P = boundary_pssm(n)
    return dbformat.decode(consensus), P


def _check_scan(eng, bd, n, k, stat_threshold=THRESHOLD, res=None, gop=-11, gex=-1, switches=None):
    """Every score, the top-k list (ties by ascending id) and numOverflows of one PSSM scan against the oracle."""
    letters, P = _query(n)
    res = res or eng.scan(letters, pssm=P)
    ref = bd.ref(n, gop, gex)
    got = _all_scores(eng, bd.db.num_sequences)
    bad = np.nonzero(got != ref)[0]
    assert len(bad) == 0, (n, gop, gex, len(bad), bd.describe(n, bad, got, ref, switches))
    order = np.lexsort((np.arange(len(ref)), -ref.astype(np.int64)))[:k]
    assert res.scores == ref[order].tolist() and res.referenceIds == order.tolist(), (n, gop, gex)
    L = bd.db.lengths
    want = int(((ref >= stat_threshold) & (L > 240) & (L <= constants()["kStatMaxLength"])).sum())
    assert res.stats.numOverflows == want, (n, gop, gex, stat_threshold, res.stats.numOverflows, want)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["few", "many"])
def test_boundary_scores_on_every_kernel_path(boundary_dbs, kind):
    """Every query length of SWEEP_QUERIES: all scores, the top-k list and numOverflows under the 25000 rule, then
    the same scans under Half2's rule (>= 2048) with KernelTypeConfig(Half2, ...)."""
    import cudasw4_b200 as sw
    bd = boundary_dbs[kind]
    L = bd.db.lengths
    for n in SWEEP_QUERIES:
        ref = bd.ref(n)
        if n >= 197:  # overflows in the single-segment classes too
            assert ((ref >= THRESHOLD) & (L <= 1024)).sum() >= 4, n
    with sw.CudaSW4(deviceIds=[0], numTop=17, blosumType=62) as eng:
        eng.setDatabase(bd.db)
        for n in SWEEP_QUERIES:
            _check_scan(eng, bd, n, 17)
    cfg = sw.KernelTypeConfig(sw.KernelType.Half2, sw.KernelType.Half2, sw.KernelType.Float, sw.KernelType.Float)
    with sw.CudaSW4(deviceIds=[0], numTop=17, blosumType=62, kernelTypeConfig=cfg) as eng:
        eng.setDatabase(bd.db)
        for n in SWEEP_QUERIES:
            _check_scan(eng, bd, n, 17, stat_threshold=constants()["kHalf2Threshold"])


@pytest.mark.gpu
def test_boundary_scores_at_gap_range_limits(boundary_dbs):
    """(-4096, -4096) and (0, 0) with rows holding -128: the -16000 sentinel of the gap rows and the E / F floors take
    the largest steps downwards, and free gaps send most subjects through re-scoring."""
    import cudasw4_b200 as sw
    bd = boundary_dbs["few"]
    for n, gop, gex in GAP_CASES:
        assert (boundary_pssm(n)[2] == -128).any()
        with sw.CudaSW4(deviceIds=[0], numTop=9, blosumType=62, gop=gop, gex=gex) as eng:
            eng.setDatabase(bd.db)
            _check_scan(eng, bd, n, 9, gop=gop, gex=gex)


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
qs = [dbformat.decode(d["q%%d" %% i]) for i in range(nq)]
ps = [d["p%%d" %% i] for i in range(nq)]
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
    for i in range(nq):
        check(eng.scan(qs[i], pssm=ps[i]), i, True)
    many, _ = eng.scanMany(qs, pssm=ps)
    for i, res in enumerate(many):
        check(res, i, False)
print("ok")
'''


@pytest.fixture(scope="module")
def switch_inputs(boundary_dbs, tmp_path_factory):
    bd = boundary_dbs["few"]
    db, k = bd.db, 11
    arrays = dict(chars=db.chars, offsets=db.offsets, lengths=db.lengths, headers=db.headers,
                  header_offsets=db.header_offsets, nq=len(SWITCH_QUERIES), k=k)
    for i, n in enumerate(SWITCH_QUERIES):
        consensus, _, P = boundary_pssm(n)
        ref = bd.ref(n)
        order = np.lexsort((np.arange(len(ref)), -ref.astype(np.int64)))[:k]
        arrays.update({"q%d" % i: consensus, "p%d" % i: P, "ref%d" % i: ref, "s%d" % i: ref[order], "i%d" % i: order})
    path = str(tmp_path_factory.mktemp("pssm_switches") / "inputs.npz")
    np.savez(path, **arrays)
    return bd, path


@pytest.mark.gpu
@pytest.mark.parametrize("switch", SWITCHES, ids=lambda sw: ",".join("%s=%s" % kv for kv in sw.items()))
def test_development_switches_with_saturating_pssms(switch_inputs, switch):
    """Every development switch (read once per process, hence a child process each) on the database with few long
    subjects: all scores, the top-k lists and numOverflows of saturating PSSM queries, alone and through scanMany."""
    bd, path = switch_inputs
    env = dict(os.environ, **switch)
    r = subprocess.run([sys.executable, "-c", _SWITCH_CHILD % {"root": ROOT}, path], env=env, capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0 and "ok" in r.stdout, (switch, r.stdout[-500:], r.stderr[-2000:])


MODE_QUERIES = (401, 1024)   # re-scored by sw_s32_pssm_kernel / by the s32 array


@pytest.mark.gpu
def test_saturating_pssm_in_every_database_mode(boundary_dbs):
    """Streamed (at least 4 batches), three shards on one GPU, sw4_set_shard and a pre-sharded handle: every score of
    every subject a handle scanned, and its top-k list, equal the oracle's."""
    import cudasw4_b200 as sw
    from cudasw4_b200 import dbformat
    bd = boundary_dbs["few"]
    db, N, k = bd.db, bd.db.num_sequences, 13

    def check(eng, ctx, expect_ids=None):
        for n in MODE_QUERIES:
            letters, P = _query(n)
            ref = bd.ref(n)
            res = eng.scan(letters, pssm=P)
            scores, ids = eng.lastScanAllScores()
            ids = np.asarray(ids, dtype=np.int64)
            assert len(set(ids.tolist())) == len(ids), ctx
            if expect_ids is not None:
                assert sorted(ids.tolist()) == sorted(expect_ids), ctx
            bad = np.nonzero(scores != ref[ids])[0]
            assert len(bad) == 0, (ctx, n, ids[bad[:8]], scores[bad[:8]], ref[ids[bad[:8]]])
            top = ids[np.lexsort((ids, -ref[ids].astype(np.int64)))[:k]]
            assert res.scores == ref[top].tolist() and res.referenceIds == top.tolist(), (ctx, n)
            assert (ref[ids] >= THRESHOLD).any(), (ctx, n)
        return set(ids.tolist())

    with sw.CudaSW4(deviceIds=[0], numTop=k, blosumType=62, memoryConfig=sw.MemoryConfig(maxGpuMem=3 << 20)) as eng:
        eng.setDatabase(db)
        eng.prefetchDBToGpus()
        assert eng.dbInfo().num_batches >= 4
        check(eng, "streamed", list(range(N)))
    with sw.CudaSW4(deviceIds=[0, 0, 0], numTop=k, blosumType=62) as eng:
        eng.setDatabase(db)
        check(eng, "three shards", list(range(N)))
    seen = set()
    for rank in range(3):
        with sw.CudaSW4(deviceIds=[0], numTop=k, blosumType=62) as eng:
            eng.setShard(rank, 3)
            eng.setDatabase(db)
            part = check(eng, "setShard %d/3" % rank)
            assert not part & seen
            seen |= part
    assert seen == set(range(N))
    gids = np.array([i for i in range(N) if (i // 256) % 3 == 1 or bd.tags[i]], dtype=np.int32)
    local = dbformat.from_sequences([db.sequence(int(i)) for i in gids])
    with sw.CudaSW4(deviceIds=[0], numTop=k, blosumType=62) as eng:
        eng.setDatabaseShard(local, gids, N)
        check(eng, "pre-sharded", gids.tolist())


@pytest.mark.gpu
def test_scan_many_interleaves_saturating_and_sequence_queries(oracle, boundary_dbs):
    """Saturating PSSM queries between sequence queries (as PSSMs of their matrix rows, which score exactly like the
    sequence) in one scanMany: each result equals its single scan, and the saturating ones equal the oracle."""
    import cudasw4_b200 as sw
    from cudasw4_b200 import dbformat, synth
    from tests.test_pssm import seq_pssm
    bd = boundary_dbs["many"]
    M = oracle.matrix(62)
    rng = np.random.default_rng(3)
    queries = []
    for n, m in ((197, 150), (517, 900), (785, 1200), (2002, 300)):
        letters, P = _query(n)
        queries.append((n, letters, P))
        q = synth.random_residues(rng, m)
        queries.append((None, dbformat.decode(q), seq_pssm(M, q)))
    with sw.CudaSW4(deviceIds=[0], numTop=15, blosumType=62) as eng:
        eng.setDatabase(bd.db)
        many, _ = eng.scanMany([q for _, q, _ in queries], pssm=[P for _, _, P in queries])
        for (n, letters, P), res in zip(queries, many):
            one = eng.scan(letters, pssm=P)
            assert (res.scores, res.referenceIds, res.stats.numOverflows) == \
                (one.scores, one.referenceIds, one.stats.numOverflows), (n, len(letters))
            if n is None:
                plain = eng.scan(letters)
                assert (plain.scores, plain.referenceIds) == (one.scores, one.referenceIds)
            else:
                _check_scan(eng, bd, n, 15, res=res)


@pytest.mark.gpu
@pytest.mark.parametrize("n", TRACEBACK_QUERIES)
def test_boundary_coordinates_and_traceback(pssm_oracle, boundary_dbs, n):
    """Coordinates and CIGARs of every boundary subject of the query (both copies) equal the restatement's."""
    import cudasw4_b200 as sw
    from tests.test_pssm import _assert_same
    from tests.traceback_oracle import Traceback
    bd = boundary_dbs["few"]
    consensus, _, P = boundary_pssm(n)
    letters, _ = _query(n)
    ids = bd.ids_of(n)
    want = pssm_oracle.traceback(P, consensus, [bd.db.sequence(int(i)) for i in ids], -11, -1)
    assert want.coordinates[:, 0].tolist() == [bd.tags[int(i)][1] for i in ids]
    with sw.CudaSW4(deviceIds=[0], numTop=5, blosumType=62) as eng:
        eng.setDatabase(bd.db)
        assert (eng.alignmentCoordinates(letters, ids, pssm=P) == want.coordinates).all()
        _assert_same(eng.alignments(letters, ids, pssm=P), Traceback(want.coordinates, want.counts, want.cigars), n)
