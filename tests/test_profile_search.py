"""Iterative profile search: sw4_build_pssm / CudaSW4.buildPssm, sw4_search_iterative / CudaSW4.searchIterative and
align --iterations / --outPssm.

CPU: the numpy restatement (tests/profile_oracle.py) on cases with known answers. GPU: buildPssm against the
restatement fed with alignments(), the no-hit profile, chunking and errors, the round driver against its rounds redone
through public calls, the sensitivity gain on a planted family, and the CLI."""
import math
import subprocess
from fractions import Fraction

import numpy as np
import pytest

import cudasw4_b200 as sw
from cudasw4_b200 import dbformat, synth
from tests import profile_oracle as po
from tests.test_cli import ALIGN, MAKEDB, _build_cli, _run_align

TABLES = (45, 50, 62, 80)


def _engine(**kw):
    kw.setdefault("deviceIds", [0])
    return sw.CudaSW4(**kw)


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("blosum", TABLES)
def test_oracle_without_hits_is_the_matrix_rows(oracle, blosum):
    M = oracle.matrix(blosum)
    q = po.query_codes(po.LETTERS + "XBZ*acdwy")  # X, other letters and lower case are code 20
    assert (q[20:] == 20).all()
    for beta in (0.5, 10.0, 1000.0):
        got, _ = po.profile(q, [], M, beta)
        assert (got == M[q]).all(), blosum


def test_oracle_weights_on_a_hand_made_msa():
    # query ACDE; row 1 = ACG over query 0..2 (2=1X); row 2 = A-DE (1=1I2=)
    q = po.query_codes("ACDE")
    alignments = [((9, 0, 2, 0, 2), "2=1X", po.query_codes("ACG")), ((9, 0, 3, 0, 2), "1=1I2=", po.query_codes("ADE")),
                  ((0, -1, -1, -1, -1), "", po.query_codes("W"))]
    msa = po.build_msa(q, alignments)
    C, D, E, G = (po.LETTERS.index(c) for c in "CDEG")
    assert msa.tolist() == [[0, C, D, E], [0, C, G, po.EMPTY], [0, po.GAP, D, E]]
    # column 0: r = 1, n = 3; column 1: r = 2 (C x2, gap); column 2: r = 2 (D x2, G); column 3: r = 1, n = 2
    want = [Fraction(1, 3) + Fraction(1, 4) + Fraction(1, 4) + Fraction(1, 2),
            Fraction(1, 3) + Fraction(1, 4) + Fraction(1, 2),
            Fraction(1, 3) + Fraction(1, 2) + Fraction(1, 4) + Fraction(1, 2)]
    assert want == [Fraction(4, 3), Fraction(13, 12), Fraction(19, 12)]
    got = po.henikoff_weights(msa)
    assert np.allclose(got, [float(x) for x in want], rtol=0, atol=1e-15)


def test_oracle_lambda_is_the_ungapped_lambda_of_test_evalue(oracle):
    p = np.bincount(synth._PSEUDO_TABLE, minlength=20) / 256.0
    M = oracle.matrix(62)[:20, :20].astype(np.float64)
    lo, hi = 1e-3, 2.0
    for _ in range(200):
        mid = (lo + hi) / 2
        lo, hi = (mid, hi) if (np.outer(p, p) * np.exp(mid * M)).sum() < 1 else (lo, mid)
    assert po.ungapped_lambda(oracle.matrix(62)) == lo
    lam, q = po.target_frequencies(oracle.matrix(62))
    assert lam == lo and abs(q.sum() - 1) < 1e-12 and 0.3 < lam < 0.33


# ---------------------------------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------------------------------
def _family_db(seed=1, n=3000):
    """C1-like records plus a planted family of the first query (substitutions and indels, some with non-standard
    letters) and one all-X subject (score 0 against everything). Returns (db, query letters, ids of the family)."""
    recs, queries = synth.config_c1(seed=seed, n=n)
    rng = np.random.default_rng(seed + 100)
    query = queries[0][1]
    qc = dbformat.encode(query)
    fam = []
    for k, rate in enumerate((0.1, 0.25, 0.35, 0.45, 0.55, 0.6)):
        c = synth.mutate(rng, qc, rate, indels=3)
        if k % 2:
            c[rng.integers(0, len(c), 6)] = 20
        fam.append(c)
    seqs = [dbformat.encode(s) for _, s in recs] + fam + [np.full(50, 20, np.uint8)]
    headers = [h for h, _ in recs] + [f"fam{k}" for k in range(len(fam))] + ["allx"]
    db = dbformat.from_sequences(seqs, headers)
    hb = bytes(db.headers)
    names = [hb[int(db.header_offsets[i]):int(db.header_offsets[i + 1])].decode() for i in range(len(db.lengths))]
    fam_ids = [names.index(f"fam{k}") for k in range(len(fam))]
    return db, query, fam_ids, names.index("allx")


def _ref_codes(db, i):
    o = int(db.offsets[i])
    return np.asarray(db.chars[o:o + int(db.lengths[i])])


def _oracle_profile(eng, db, query, ids, M, beta, pssm=None):
    al = eng.alignments(query, ids, pssm=pssm)
    rows = [(al.coordinates[k], al.cigars[k], _ref_codes(db, int(i))) for k, i in enumerate(ids)]
    return po.profile(po.query_codes(query), rows, M, beta)


def _compare(got, want, x):
    """Every entry equal, except entries whose x lies within 1e-9 of k + 1/2 may differ by 1. Returns the number of such
    near-tie entries."""
    near = np.zeros(got.shape, dtype=bool)
    frac = np.abs(x - np.floor(x) - 0.5)
    near[:, :20] = np.nan_to_num(frac, nan=1.0) < 1e-9
    diff = got.astype(np.int64) - want.astype(np.int64)
    assert ((diff == 0) | (near & (np.abs(diff) == 1))).all(), np.argwhere(diff != 0)[:10]
    return int(near.sum())


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_build_pssm_equals_the_oracle(oracle):
    db, query, fam, allx = _family_db()
    near_total = checked = 0
    for blosum in TABLES:
        M = oracle.matrix(blosum)
        for gop, gex in ((-11, -1), (-6, -3)):
            with _engine(numTop=40, blosumType=blosum, gop=gop, gex=gex) as eng:
                eng.setDatabase(db)
                top = eng.scan(query).referenceIds
                ids = top[:25] + fam + [allx, 0, top[0], top[0], fam[1]]
                for beta in (0.5, 10.0, 1000.0):
                    got = eng.buildPssm(query, ids, pseudocountWeight=beta)
                    want, x = _oracle_profile(eng, db, query, ids, M, beta)
                    near_total += _compare(got, want, x)
                    checked += got.size
                # the PSSM query form: align the hits with the profile just built
                P = eng.buildPssm(query, ids)
                top2 = eng.scan(query, pssm=P).referenceIds
                ids2 = top2[:20] + fam + [allx, top2[0]]
                for beta in (0.5, 10.0, 1000.0):
                    got = eng.buildPssm(query, ids2, pssm=P, pseudocountWeight=beta)
                    want, x = _oracle_profile(eng, db, query, ids2, M, beta, pssm=P)
                    near_total += _compare(got, want, x)
                    checked += got.size
    print(f"buildPssm vs oracle: {checked} entries, {near_total} within 1e-9 of a rounding tie")


@pytest.mark.gpu
@pytest.mark.parametrize("blosum", TABLES)
def test_no_hits_gives_the_matrix_rows_and_the_sequence_scan(oracle, blosum):
    db, _, _, _ = _family_db()
    M = oracle.matrix(blosum)
    query = synth.load_queries()[1][1][:150] + "XBZacdx*"
    with _engine(numTop=25, blosumType=blosum) as eng:
        eng.setDatabase(db)
        P = eng.buildPssm(query, [])
        assert (P == M[po.query_codes(query)]).all()
        r_seq = eng.scan(query)
        s_seq, i_seq = eng.lastScanAllScores()
        r_pssm = eng.scan(query, pssm=P)
        s_pssm, i_pssm = eng.lastScanAllScores()
    assert r_seq.scores == r_pssm.scores and r_seq.referenceIds == r_pssm.referenceIds
    assert (s_seq == s_pssm).all() and (i_seq == i_pssm).all()


@pytest.mark.gpu
def test_chunking_determinism_and_errors():
    db, query, fam, allx = _family_db()
    with _engine(numTop=60, blosumType=62) as eng:
        eng.setDatabase(db)
        ids = eng.scan(query).referenceIds + fam + [allx]
        st_full, st_small = sw.BenchmarkStats(), sw.BenchmarkStats()
        full = eng.buildPssm(query, ids, stats=st_full)
        assert (eng.buildPssm(query, ids) == full).all()  # the same call, the same bytes
        eng.setMemoryConfig(sw.MemoryConfig(maxTempBytes=600_000))
        st_align = sw.BenchmarkStats()
        eng.alignments(query, ids, stats=st_align)
        small = eng.buildPssm(query, ids, stats=st_small)
        # alignments: convert + 2 per coordinate chunk + 2 per traceback chunk; buildPssm adds one scatter per
        # traceback chunk and 3 kernels for the scores
        trace_chunks = st_small.kernelLaunches - st_align.kernelLaunches - 3
        print(f"traceback chunks at 600 kB: {trace_chunks}; launches {st_full.kernelLaunches} -> {st_small.kernelLaunches}")
        assert trace_chunks >= 3
        assert (small == full).all()
        eng.setMemoryConfig(sw.MemoryConfig(maxTempBytes=500_000))
        dups = 500_000 // len(query) + 1
        with pytest.raises(sw.SW4Error) as e:  # the MSA: (1 + dups) x m bytes > 500 kB; one pair's trace scratch fits
            eng.buildPssm(query, [fam[0]] * dups)
        assert e.value.code == -4
        eng.setMemoryConfig(sw.MemoryConfig())
        for beta in (0.0, -1.0, math.nan, math.inf):
            with pytest.raises(sw.SW4Error) as e:
                eng.buildPssm(query, ids, pseudocountWeight=beta)
            assert e.value.code == -1
        for bad in ([-1], [len(db.lengths)]):
            with pytest.raises(sw.SW4Error) as e:
                eng.buildPssm(query, bad)
            assert e.value.code == -1
        assert (eng.buildPssm(query, ids) == full).all()  # refusals leave nothing behind
    with _engine(numTop=10, blosumType=62) as eng:
        with pytest.raises(sw.SW4Error) as e:
            eng.buildPssm(query, [])
        assert e.value.code == -1


def family_members(rng, query_len=300, extra=(3, 6), grades=((0.5, 0.0), (0.7, 0.05), (0.8, 0.05), (0.85, 0.1), (0.9, 0.1),
                   (0.95, 0.1), (1.0, 0.1), (1.0, 0.15)), copies=4):
    """A planted family whose columns differ in what they allow: column c of the ancestor (the query) admits its own
    residue and 3..6 others. A member of grade (d, noise) draws each position from the column's residues with
    probability d, takes a background residue with probability `noise`, and gets two indels. The far grades are what a
    profile of the near ones finds. Returns (ancestor codes, [(grade, member codes)])."""
    anc = synth._PSEUDO_TABLE[rng.integers(0, 256, query_len)]
    allowed = [np.concatenate([[anc[c]], synth._PSEUDO_TABLE[rng.integers(0, 256, int(rng.integers(extra[0], extra[1] + 1)))]])
               for c in range(query_len)]
    members = []
    for d, noise in grades:
        for _ in range(copies):
            c = anc.copy()
            for j in np.nonzero(rng.random(query_len) < d)[0]:
                c[j] = allowed[j][rng.integers(0, len(allowed[j]))]
            m = rng.random(query_len) < noise
            c[m] = synth._PSEUDO_TABLE[rng.integers(0, 256, int(m.sum()))]
            members.append(((d, noise), synth.mutate(rng, c, 0.0, indels=2)))
    return anc, members


def plant(lengths, members):
    """The ascending lengths of a database with one more slot per member, and where the members go: (lengths,
    {id: codes} for setPseudoDatabaseLengths, {grade: ids})."""
    L = np.sort(np.concatenate([np.asarray(lengths, dtype=np.int64), [len(c) for _, c in members]])).astype(np.int32)
    planted, by_grade = {}, {}
    for grade, c in members:
        i = int(np.searchsorted(L, len(c)))
        while i in planted or L[i] != len(c):
            i += 1
        planted[i] = c
        by_grade.setdefault(grade, []).append(i)
    return L, planted, by_grade


def _planted_family(rng, n_null):
    """A null database of n_null lognormal lengths with one planted family: (lengths, planted, query letters, ids by
    grade)."""
    anc, members = family_members(rng)
    L, planted, by_grade = plant(synth.lognormal_lengths(rng, n_null, 5.683, 0.636, 2, 35213), members)
    return L, planted, dbformat.decode(anc), by_grade


def _manual_rounds(eng, query, rounds, incl=0.002, beta=10.0):
    """The driver restated through public calls: [(ScanResult, pssm searched with, included ids)] per round."""
    out, P, prev = [], None, None
    for i in range(1, rounds + 1):
        r = eng.scan(query, pssm=P)
        hits = [j for j, e in zip(r.referenceIds, r.evalues) if e <= incl]
        out.append((r, P, hits))
        if i == rounds or not hits or (prev is not None and sorted(hits) == sorted(prev)):
            break
        P = eng.buildPssm(query, hits, pssm=P, pseudocountWeight=beta)
        prev = hits
    return out


@pytest.mark.gpu
def test_driver_equals_its_rounds_through_public_calls(oracle):
    rng = np.random.default_rng(31)
    L, planted, query, _ = _planted_family(rng, 30_000)
    M = oracle.matrix(62)
    with _engine(numTop=200, blosumType=62) as eng:
        eng.setPseudoDatabaseLengths(L, seed=41, planted=planted)
        with pytest.raises(sw.SW4Error) as e:  # statistics off
            eng.searchIterative(query)
        assert e.value.code == -1
        eng.setScoreStatistics(True)
        manual = _manual_rounds(eng, query, 4)
        print(f"manual rounds: {[len(h) for _, _, h in manual]} included hits")
        assert len(manual) >= 2
        for k in range(1, len(manual) + 1):
            it = eng.searchIterative(query, iterations=k)
            r, P, hits = manual[k - 1]
            assert it.iterations == k
            assert it.result.scores == r.scores and it.result.referenceIds == r.referenceIds
            assert it.result.evalues == r.evalues
            want_P = M[po.query_codes(query)] if P is None else P
            assert (it.pssm == want_P).all()
            again = eng.scan(query, pssm=it.pssm)
            assert again.scores == it.result.scores and again.referenceIds == it.result.referenceIds
        last = eng.searchIterative(query, iterations=10)
        assert last.iterations <= 10 and (last.converged or last.iterations == 10 or not last.result.evalues)
        plain = eng.scan(query)
        one = eng.searchIterative(query, iterations=1)
        assert one.result.scores == plain.scores and one.result.referenceIds == plain.referenceIds
        assert one.result.evalues == plain.evalues and not one.converged
        # the rounds take their hits before the cutoff; the reported list has it
        eng.setScoreStatistics(True, 1e-30)
        cut = eng.searchIterative(query, iterations=k)
        r = manual[k - 1][0]
        keep = [e <= 1e-30 for e in r.evalues]
        assert cut.result.referenceIds == [i for i, ok in zip(r.referenceIds, keep) if ok]
        assert (cut.pssm == it.pssm).all()
        eng.setScoreStatistics(True)
        for bad in (dict(iterations=0), dict(pseudocountWeight=0.0), dict(inclusionEvalue=math.nan)):
            with pytest.raises(sw.SW4Error) as e:
                eng.searchIterative(query, **bad)
            assert e.value.code == -1
    with _engine(deviceIds=[0, 0, 0], numTop=200, blosumType=62) as eng:
        eng.setPseudoDatabaseLengths(L, seed=41, planted=planted)
        eng.setScoreStatistics(True)
        three = eng.searchIterative(query, iterations=3)
    with _engine(numTop=200, blosumType=62) as eng:
        eng.setPseudoDatabaseLengths(L, seed=41, planted=planted)
        eng.setScoreStatistics(True)
        single = eng.searchIterative(query, iterations=3)
    assert three.result.scores == single.result.scores and three.result.referenceIds == single.result.referenceIds
    assert (three.pssm == single.pssm).all() and three.iterations == single.iterations
    with _engine(numTop=200, blosumType=62) as eng:
        eng.setShard(0, 2)
        eng.setPseudoDatabaseLengths(L, seed=41, planted=planted)
        eng.setScoreStatistics(True)
        with pytest.raises(sw.SW4Error) as e:
            eng.searchIterative(query)
        assert e.value.code == -1


@pytest.mark.gpu
def test_rounds_find_distant_members_the_first_scan_misses():
    rng = np.random.default_rng(77)
    L, planted, query, by_grade = _planted_family(rng, 200_000)
    members = set(planted)
    with _engine(numTop=500, blosumType=62) as eng:
        eng.setPseudoDatabaseLengths(L, seed=78, planted=planted)
        eng.setScoreStatistics(True)
        found = []
        for k in (1, 2, 3, 4, 5):
            it = eng.searchIterative(query, iterations=k)
            inc = {i for i, e in zip(it.result.referenceIds, it.result.evalues) if e <= 0.002}
            found.append(inc & members)
            if it.iterations < k:
                break
    print("planted members with E <= 0.002 per round:", [len(f) for f in found], "of", len(members))
    for grade, ids in by_grade.items():
        print(f"  grade {grade}: per round {[len(f & set(ids)) for f in found]} of {len(ids)}")
    assert found[-1] - found[0], "the last round includes no planted member that round 1 missed"


@pytest.mark.gpu
def test_align_iterations_and_out_pssm(tmp_path):
    _build_cli()
    recs, queries = synth.config_c1(seed=3, n=4000)
    dbformat.write_fasta(str(tmp_path / "db.fa"), recs)
    dbformat.write_fasta(str(tmp_path / "q.fa"), queries[:3])
    subprocess.run([MAKEDB, str(tmp_path / "db.fa"), str(tmp_path / "db")], check=True, stdout=subprocess.DEVNULL)
    common = ["--query", "q.fa", "--db", "db", "--top", "30", "--mat", "blosum62"]
    cwd = str(tmp_path)
    _run_align(ALIGN, common + ["--tsv", "--cigar", "--of", "plain.tsv"], cwd)
    _run_align(ALIGN, common + ["--tsv", "--cigar", "--iterations", "1", "--of", "one.tsv"], cwd)
    assert open(tmp_path / "one.tsv", "rb").read() == open(tmp_path / "plain.tsv", "rb").read()
    out = _run_align(ALIGN, common + ["--tsv", "--evalue", "--cigar", "--coordinates", "--iterations", "3", "--batchQueries", "2",
                                      "--outPssm", "final", "--of", "it.tsv"], cwd)
    lines = [ln for ln in out.splitlines() if ln.startswith("Query ") and "round" in ln]
    assert len(lines) == 3, out[-2000:]
    rows = [r.split("\t") for r in open(tmp_path / "it.tsv").read().splitlines()[1:]]
    with _engine(numTop=30, blosumType=62) as eng:
        eng.setDatabase(str(tmp_path / "db"))
        eng.setScoreStatistics(True)
        for qi, (_, q) in enumerate(queries[:3]):
            it = eng.searchIterative(q, iterations=3)
            assert f"Query {qi}: {it.iterations} round" in lines[qi]
            assert ("not converged" not in lines[qi]) == it.converged
            mine = [r for r in rows if int(r[0]) == qi]
            assert [int(r[4]) for r in mine] == it.result.scores
            assert [int(r[7]) for r in mine] == it.result.referenceIds
            for r, e in zip(mine, it.result.evalues):
                assert math.isclose(float(r[-2]), e, rel_tol=1e-5)
            al = eng.alignments(q, it.result.referenceIds, pssm=it.pssm)
            assert [r[8] for r in mine] == [str(c[1] + 1) for c in al.coordinates]  # query begin
            assert [r[-3] for r in mine] == al.cigars
            # the written file: the same PSSM, and align --pssm on it reproduces the hits
            P = np.loadtxt(tmp_path / f"final.{qi}.pssm", skiprows=2, usecols=range(2, 22), dtype=np.int64, ndmin=2)
            assert (P == it.pssm[:, :20]).all()
            _run_align(ALIGN, ["--pssm", f"final.{qi}.pssm", "--db", "db", "--top", "30", "--mat", "blosum62", "--tsv",
                               "--of", f"re{qi}.tsv"], cwd)
            re_rows = [x.split("\t") for x in open(tmp_path / f"re{qi}.tsv").read().splitlines()[1:]]
            assert [int(x[4]) for x in re_rows] == it.result.scores and [int(x[7]) for x in re_rows] == it.result.referenceIds
    r = subprocess.run([ALIGN, "--pssm", "final.0.pssm", "--db", "db", "--iterations", "2"], cwd=cwd, capture_output=True, text=True)
    assert r.returncode != 0 and "--pssm" in r.stderr
