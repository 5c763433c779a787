"""Alignment coordinates (sw4_alignment_coordinates / CudaSW4.alignmentCoordinates / align --coordinates).

CPU: the restatement of the coordinates (tests/coords_oracle.cpp) against a brute force over every (begin, end) pair
of tiny inputs, and its score against the oracle's sw4o_gotoh_score. GPU: every result, score and four positions,
against that restatement, in every database mode, on tie-heavy and on very long pairs, and through the CLI."""
import itertools
import os
import subprocess

import numpy as np
import pytest

import cudasw4_b200 as sw
from cudasw4_b200 import dbformat, synth
from tests import coords_oracle as coords_oracle_lib
from tests.test_cli import ALIGN, ALIGN_CASES, _run_align, align_case_inputs, pseudodb_case_inputs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MATRICES = [(62, -11, -1), (45, -13, -2), (50, -13, -2), (80, -10, -1), (62, -5, -3), (45, -9, -3), (80, -14, -2)]
EXTRA_GAPS = [(62, 0, 0), (62, -4096, -4096), (62, 0, -4096)]
BRUTE_GAPS = [(0, 0), (0, -1), (-1, 0), (-11, -1), (-4096, -4096)]
NEG = float("-inf")


@pytest.fixture(scope="module")
def coords_oracle(oracle):
    return coords_oracle_lib.load(oracle)


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def _anchored_from(M, q, s, b1, b2, gop, gex):
    """P[i][j] = best score of an alignment that starts with the pair (b1, b2) and ends with the pair (i, j), by a full
    matrix over q[b1:] x s[b2:] (three states: pair, gap along s, gap along q)."""
    n, m = len(q) - b1, len(s) - b2
    P = [[NEG] * m for _ in range(n)]
    E = [[NEG] * m for _ in range(n)]
    F = [[NEG] * m for _ in range(n)]
    for i in range(n):
        for j in range(m):
            if i == 0 and j == 0:
                P[i][j] = M[q[b1]][s[b2]]
            elif i > 0 and j > 0:
                P[i][j] = M[q[b1 + i]][s[b2 + j]] + max(P[i - 1][j - 1], E[i - 1][j - 1], F[i - 1][j - 1])
            if j > 0:
                E[i][j] = max(max(P[i][j - 1], E[i][j - 1], F[i][j - 1]) + gop, E[i][j - 1] + gex)
            if i > 0:
                F[i][j] = max(max(P[i - 1][j], E[i - 1][j], F[i - 1][j]) + gop, F[i - 1][j] + gex)
    return P


def _brute_force(M, q, s, gop, gex):
    """(S, qb, qe, rb, re) by enumerating every (begin, end) pair: the smallest end among the optimal pairs, then the
    largest begin among the optimal pairs with that end."""
    best, pairs = 0, []
    for b1, b2 in itertools.product(range(len(q)), range(len(s))):
        P = _anchored_from(M, q, s, b1, b2, gop, gex)
        for i, row in enumerate(P):
            for j, v in enumerate(row):
                if v > best:
                    best, pairs = v, []
                if v == best and v > 0:
                    pairs.append((b1, b2, b1 + i, b2 + j))
    if best == 0:
        return (0, -1, -1, -1, -1)
    qe, re = min((p[2], p[3]) for p in pairs)
    qb, rb = max((p[0], p[1]) for p in pairs if (p[2], p[3]) == (qe, re))
    return (best, qb, qe, rb, re)


@pytest.mark.parametrize("blosum", [45, 50, 62, 80])
def test_oracle_coordinates_equal_brute_force(coords_oracle, oracle, blosum):
    M = oracle.matrix(blosum).astype(int).tolist()
    rng = np.random.default_rng(blosum)
    cases = 0
    for gop, gex in BRUTE_GAPS:
        for letters in (2, 3):
            for _ in range(5):
                alphabet = rng.choice(20, letters, replace=False)
                q = alphabet[rng.integers(0, letters, int(rng.integers(1, 10)))].astype(np.uint8)
                s = alphabet[rng.integers(0, letters, int(rng.integers(1, 10)))].astype(np.uint8)
                got = tuple(coords_oracle.coords(blosum, q, [s], gop, gex)[0].tolist())
                want = _brute_force(M, q.tolist(), s.tolist(), gop, gex)
                assert got == want, (blosum, gop, gex, q.tolist(), s.tolist())
                if want[0] > 0:  # the anchored score of the reported rectangle is the score
                    P = _anchored_from(M, q.tolist(), s.tolist(), want[1], want[3], gop, gex)
                    assert P[want[2] - want[1]][want[4] - want[3]] == want[0]
                cases += 1
    assert cases == 50


def test_oracle_coordinates_score_equals_gotoh_score(coords_oracle, oracle):
    rng = np.random.default_rng(7)
    for blosum, gop, gex in MATRICES + EXTRA_GAPS + [(45, 0, -1), (80, -1, 0)]:
        subjects = [synth.random_residues(rng, int(n)) for n in rng.integers(0, 120, 40)]
        q = synth.random_residues(rng, int(rng.integers(1, 150)))
        got = coords_oracle.coords(blosum, q, subjects, gop, gex)
        for s, row in zip(subjects, got):
            assert row[0] == oracle.score(blosum, q, s, gop, gex)
            if row[0] == 0:
                assert row[1:].tolist() == [-1, -1, -1, -1]
            else:
                assert 0 <= row[1] <= row[2] < len(q) and 0 <= row[3] <= row[4] < len(s)


def test_facade_coordinates_compile_standalone(tmp_path):
    import shutil
    gxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else shutil.which("g++")
    if not gxx:
        pytest.skip("no host compiler")
    src = tmp_path / "coords.cpp"
    src.write_text('#include "cudasw4.cuh"\n'
                   'int main() {\n'
                   '  cudasw4::KernelTypeConfig k; cudasw4::MemoryConfig m;\n'
                   '  cudasw4::CudaSW4 sw({0}, 10, cudasw4::BlosumType::BLOSUM62_20, k, m, false);\n'
                   '  std::vector<cudasw4::ReferenceIdT> ids{0, 3};\n'
                   '  std::vector<cudasw4::AlignmentCoordinates> c = sw.computeAlignmentCoordinates("ACDE", 4, ids);\n'
                   '  return c[0].score + c[0].queryBegin + c[0].queryEnd + c[0].referenceBegin + c[0].referenceEnd;\n'
                   '}\n')
    r = subprocess.run([gxx, "-std=c++17", "-Wall", "-Werror", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), str(src)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
CLASS_EDGES = [32, 48, 64, 80, 96, 112, 128, 144, 160, 176, 192, 208, 224, 240, 256, 288, 320, 352, 384, 416, 448, 480,
               512, 576, 640, 704, 768, 832, 896, 960, 1024]
QUERY_LENGTHS = [1, 3, 37, 144, 300, 517, 1500]


def _engine(**kw):
    return sw.CudaSW4(deviceIds=kw.pop("deviceIds", [0]), **kw)


def _mixed_db(seed=11):
    rng = np.random.default_rng(seed)
    lengths = [0, 1, 2] + sorted({x for c in CLASS_EDGES for x in (c - 1, c, c + 1)}) + [1500, 2500]
    seqs = [synth.random_residues(rng, n) for n in lengths]
    for s in seqs[::7]:
        if len(s):
            s[rng.integers(0, len(s))] = 20
    return dbformat.from_sequences(seqs), rng


def _queries(rng, db):
    out = []
    for n in QUERY_LENGTHS:
        q = synth.random_residues(rng, n)
        if n >= 37:  # a fragment of a database sequence so that some pairs align over long stretches
            src = db.sequence(int(rng.integers(db.num_sequences // 2, db.num_sequences)))
            k = min(len(src), n // 2)
            q[n // 4:n // 4 + k] = src[:k]
        out.append(q)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("blosum,gop,gex", MATRICES + EXTRA_GAPS)
def test_every_subject_matches_oracle_and_scan(coords_oracle, blosum, gop, gex):
    db, rng = _mixed_db()
    ids = np.arange(db.num_sequences)
    with _engine(numTop=25, blosumType=blosum, gop=gop, gex=gex) as eng:
        eng.setDatabase(db)
        for q in _queries(rng, db):
            letters = dbformat.decode(q)
            got = eng.alignmentCoordinates(letters, ids)
            want = coords_oracle.coords(blosum, q, db, gop, gex)
            assert got.dtype == np.int32 and got.shape == (db.num_sequences, 5)
            bad = np.nonzero((got != want).any(axis=1))[0]
            assert len(bad) == 0, (len(q), [(int(i), got[i].tolist(), want[i].tolist()) for i in bad[:5]])
            res = eng.scan(letters)
            top = eng.alignmentCoordinates(letters, res.referenceIds)
            assert top[:, 0].tolist() == res.scores
            assert (top == want[res.referenceIds]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("blosum,gop,gex", [(62, 0, 0), (62, 0, -1), (62, -1, 0), (62, -11, -1), (45, -4096, -4096)])
def test_tie_heavy_inputs(coords_oracle, blosum, gop, gex):
    rng = np.random.default_rng(3)
    A, W, L = dbformat.encode("A")[0], dbformat.encode("W")[0], dbformat.encode("L")[0]
    motif = dbformat.encode("GAVL")
    q_base = synth.random_residues(rng, 60)
    subjects = [np.full(n, A, np.uint8) for n in (1, 5, 100, 700, 1300)]
    subjects += [np.tile(np.array([A, W], np.uint8), n) for n in (3, 250, 600)]
    subjects += [np.tile(motif, n) for n in (10, 200)]
    planted = synth.random_residues(rng, 2000)
    for pos in (5, 600, 1400, 1900):  # duplicates of the query at several positions of one subject
        planted[pos:pos + len(q_base)] = q_base[:min(len(q_base), 2000 - pos)]
    subjects += [planted, np.concatenate([q_base, q_base, q_base])]
    db = dbformat.from_sequences(subjects)
    queries = [np.full(40, A, np.uint8), np.tile(np.array([A, W], np.uint8), 300), np.tile(motif, 30),
               np.full(700, L, np.uint8), q_base, np.concatenate([q_base, q_base])]
    with _engine(numTop=5, blosumType=blosum, gop=gop, gex=gex) as eng:
        eng.setDatabase(db)
        for q in queries:
            got = eng.alignmentCoordinates(dbformat.decode(q), np.arange(db.num_sequences))
            want = coords_oracle.coords(blosum, q, db, gop, gex)
            assert (got == want).all(), (len(q), got.tolist(), want.tolist())


@pytest.mark.gpu
def test_long_pairs(coords_oracle):
    """35 k x 20-35 k pairs with planted copies (scores above 100,000) and a 70 k query against 1-5 k subjects: the
    CTA-wide form (DESIGN.md 3.6)."""
    rng = np.random.default_rng(35)
    q = synth.random_residues(rng, 35000)
    s0 = synth.random_residues(rng, 20000)
    s1 = synth.random_residues(rng, 35000)
    s1[2000:2000 + 30000] = q[1000:31000]
    s2 = np.concatenate([q[:15000], synth.random_residues(rng, 3000), synth.mutate(rng, q[20000:], 0.05, indels=3)])
    s3 = synth.random_residues(rng, 27000)
    s3[100:100 + 26000] = q[5000:31000]
    db = dbformat.from_sequences([s0, s1, s2, s3])
    with _engine(numTop=4, blosumType=45, gop=-9, gex=-3) as eng:
        eng.setDatabase(db)
        ids = np.arange(4)
        got = eng.alignmentCoordinates(dbformat.decode(q), ids)
        want = coords_oracle.coords(45, q, db, -9, -3)
        assert (got == want).all(), (got.tolist(), want.tolist())
        assert (want[[1, 3], 0] > 100000).all()
        q70 = synth.random_residues(rng, 70000)
        small = [synth.random_residues(rng, int(n)) for n in (1000, 2500, 5000)]
        small[1][200:2200] = q70[50000:52000]
        db2 = dbformat.from_sequences(small)
        eng.setDatabase(db2)
        got = eng.alignmentCoordinates(dbformat.decode(q70), np.arange(3))
        want = coords_oracle.coords(45, q70, db2, -9, -3)
        assert (got == want).all(), (got.tolist(), want.tolist())


def _modes_db():
    db, rng = _mixed_db(21)
    more = dbformat.from_sequences([db.sequence(i) for i in range(db.num_sequences)] +
                                   [synth.random_residues(rng, int(n)) for n in rng.integers(1, 1200, 12000)])
    return more, rng


@pytest.mark.gpu
def test_database_modes_give_identical_arrays(coords_oracle):
    db, rng = _modes_db()
    q = synth.random_residues(rng, 250)
    letters = dbformat.decode(q)
    ids = np.concatenate([np.arange(db.num_sequences), [5, 5, 17]])
    want = coords_oracle.coords(62, q, db, -11, -1)[ids]
    with _engine(numTop=30) as eng:  # before any upload
        eng.setDatabase(db)
        assert (eng.alignmentCoordinates(letters, ids) == want).all()
        eng.prefetchDBToGpus()
        assert (eng.alignmentCoordinates(letters, ids) == want).all()
    with _engine(numTop=30, memoryConfig=sw.MemoryConfig(maxGpuMem=3 << 20)) as eng:  # streamed
        eng.setDatabase(db)
        eng.prefetchDBToGpus()
        assert eng.dbInfo().num_batches >= 4
        first = eng.scan(letters)
        assert (eng.alignmentCoordinates(letters, ids) == want).all()
        second = eng.scan(letters)
        assert first.scores == second.scores and first.referenceIds == second.referenceIds
    with _engine(numTop=30, deviceIds=[0, 0, 0]) as eng:  # multi-shard on one GPU
        eng.setDatabase(db)
        assert (eng.alignmentCoordinates(letters, ids) == want).all()
    with _engine(numTop=30) as eng:
        eng.setShard(1, 3)
        eng.setDatabase(db)
        assert (eng.alignmentCoordinates(letters, ids) == want).all()


@pytest.mark.gpu
def test_presharded_handle_chunking_and_errors(coords_oracle):
    db, rng = _modes_db()
    q = synth.random_residues(rng, 400)
    letters = dbformat.decode(q)
    want = coords_oracle.coords(62, q, db, -11, -1)
    gids = np.array([i for i in range(db.num_sequences) if (i // 256) % 3 == 1], dtype=np.int32)
    local = dbformat.from_sequences([db.sequence(int(i)) for i in gids])
    with _engine(numTop=10) as eng:
        eng.setDatabaseShard(local, gids, db.num_sequences)
        assert (eng.alignmentCoordinates(letters, gids) == want[gids]).all()
        assert eng.alignmentCoordinates(letters, []).shape == (0, 5)
        for bad in ([int(gids[0]) - 1], [-1], [db.num_sequences]):
            with pytest.raises(sw.SW4Error) as e:
                eng.alignmentCoordinates(letters, bad)
            assert e.value.code == -1
    # a budget that holds a few pairs at a time gives the same arrays; one below a single long pair is refused
    with _engine(numTop=10, memoryConfig=sw.MemoryConfig(maxTempBytes=40_000)) as eng:
        eng.setDatabaseShard(local, gids, db.num_sequences)
        assert (eng.alignmentCoordinates(letters, gids) == want[gids]).all()
        longest = int(gids[np.argmax(local.lengths)])
        eng.setMemoryConfig(sw.MemoryConfig(maxTempBytes=1000))
        with pytest.raises(sw.SW4Error) as e:
            eng.alignmentCoordinates(letters, [longest])
        assert e.value.code == -4


# ---------------------------------------------------------------------------------------------------------------------
# CLI
# ---------------------------------------------------------------------------------------------------------------------
def _split_tsv(text, extra):
    base, tail = [], []
    for line in text.splitlines():
        cols = line.split("\t")
        base.append("\t".join(cols[:len(cols) - extra]))
        tail.append(cols[len(cols) - extra:])
    return "\n".join(base) + "\n", tail


@pytest.mark.gpu
@pytest.mark.parametrize("mat,extra", ALIGN_CASES)
def test_align_tsv_coordinates(coords_oracle, tmp_path, golden_dir, mat, extra):
    common = align_case_inputs(str(tmp_path), mat, extra)
    _run_align(ALIGN, common + ["--dpx", "--coordinates", "--of", "coords.tsv"], str(tmp_path))
    base, tail = _split_tsv(open(tmp_path / "coords.tsv").read(), 4)
    with open(os.path.join(golden_dir, "align", f"{mat}.tsv")) as f:
        assert base == f.read()
    assert tail[0] == ["Query begin", "Query end", "Reference begin", "Reference end"]
    blosum = int(mat[-2:])
    gop = int(extra[1]) if extra else (-13 if blosum == 45 else -11)
    gex = int(extra[3]) if extra else (-2 if blosum == 45 else -1)
    db = dbformat.read_db(str(tmp_path / "db"))
    queries = [dbformat.encode(s) for _, s in dbformat.read_fasta(str(tmp_path / "q.fa"))]
    rows = [line.split("\t") for line in base.splitlines()[1:]]
    for row, t in zip(rows, tail[1:]):
        q, rid = queries[int(row[0])], int(row[7])
        want = coords_oracle.coords(blosum, q, [db.sequence(rid)], gop, gex)[0]
        assert int(row[4]) == want[0]
        assert [int(x) for x in t] == [int(want[1]) + 1, int(want[2]) + 1, int(want[3]) + 1, int(want[4]) + 1]


@pytest.mark.gpu
def test_align_plain_coordinates_pseudodb(tmp_path, golden_dir):
    common = pseudodb_case_inputs(str(tmp_path))
    _run_align(ALIGN, common + ["--coordinates", "--of", "res.txt"], str(tmp_path))
    lines = open(tmp_path / "res.txt").read().splitlines()
    stripped = []
    for line in lines:
        if line.startswith("Result "):
            head, sep, tail = line.partition(" Query ")
            assert sep and tail.count("Reference ") == 1 and tail.endswith(".")
            line = head
        stripped.append(line)
    with open(os.path.join(golden_dir, "align", "pseudodb.txt")) as f:
        assert "\n".join(stripped) + "\n" == f.read()


@pytest.mark.gpu
def test_align_coordinates_batch_and_streaming_write_the_same_file(tmp_path):
    from tests.test_cli import MAKEDB
    recs, queries = synth.config_c1(seed=2, n=12000)
    dbformat.write_fasta(str(tmp_path / "db.fa"), recs)
    dbformat.write_fasta(str(tmp_path / "q.fa"), queries[:9])
    subprocess.run([MAKEDB, str(tmp_path / "db.fa"), str(tmp_path / "db")], check=True, stdout=subprocess.DEVNULL)
    common = ["--query", "q.fa", "--db", "db", "--top", "12", "--mat", "blosum62", "--dpx", "--coordinates"]
    _run_align(ALIGN, common + ["--of", "plain.txt"], str(tmp_path))
    _run_align(ALIGN, common + ["--of", "batched.txt", "--batchQueries", "4"], str(tmp_path))
    _run_align(ALIGN, common + ["--of", "streamed.txt", "--maxGpuMem", "5M", "--batchQueries", "16"], str(tmp_path))
    plain = open(tmp_path / "plain.txt").read()
    assert plain.count(" Reference ") == 9 * 12
    assert open(tmp_path / "batched.txt").read() == plain
    assert open(tmp_path / "streamed.txt").read() == plain
