"""Alignment traceback (sw4_alignment_traceback / CudaSW4.alignments / align --cigar).

CPU: the restatement of the traceback (tests/traceback_oracle.cpp) against a plain Python statement of the rule over
full P/E/F matrices on tiny inputs, and every CIGAR it gives rescored to the score. GPU: every coordinate, count and
CIGAR against that restatement, in every database mode, on tie-heavy and on very long pairs, and through the CLI."""
import os
import re
import subprocess

import numpy as np
import pytest

import cudasw4_b200 as sw
from cudasw4_b200 import dbformat, synth
from tests import coords_oracle as coords_oracle_lib
from tests import traceback_oracle as traceback_oracle_lib
from tests.test_cli import ALIGN, ALIGN_CASES, _run_align, align_case_inputs, pseudodb_case_inputs
from tests.test_coordinates import (BRUTE_GAPS, EXTRA_GAPS, MATRICES, NEG, _anchored_from, _engine, _mixed_db, _modes_db,
                                    _queries, _split_tsv)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def coords_oracle(oracle):
    return coords_oracle_lib.load(oracle)


@pytest.fixture(scope="module")
def tb_oracle(coords_oracle):
    return traceback_oracle_lib.load(coords_oracle)


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def _anchored_states(M, q, s, qb, rb, qe, re_, gop, gex):
    """P, E, F over the rectangle q[qb..qe] x s[rb..re], started with the pair (qb, rb) (full matrices, -inf borders)."""
    n, m = qe - qb + 1, re_ - rb + 1
    P = [[NEG] * m for _ in range(n)]
    E = [[NEG] * m for _ in range(n)]
    F = [[NEG] * m for _ in range(n)]
    for i in range(n):
        for j in range(m):
            sub = M[q[qb + i]][s[rb + j]]
            if i == 0 and j == 0:
                P[i][j] = sub
            elif i > 0 and j > 0:
                P[i][j] = sub + max(P[i - 1][j - 1], E[i - 1][j - 1], F[i - 1][j - 1])
            if j > 0:
                E[i][j] = max(max(P[i][j - 1], E[i][j - 1], F[i][j - 1]) + gop, E[i][j - 1] + gex)
            if i > 0:
                F[i][j] = max(max(P[i - 1][j], E[i - 1][j], F[i - 1][j]) + gop, F[i - 1][j] + gex)
    return P, E, F


def _python_rule(M, q, s, c, gop, gex):
    """(CIGAR, [length, identities, positives, gaps]) by the walk of include/sw4b200.h over full matrices."""
    S, qb, qe, rb, re_ = c
    if S == 0:
        return "", [0, 0, 0, 0]
    P, E, F = _anchored_states(M, q, s, qb, rb, qe, re_, gop, gex)
    assert P == [row[:re_ - rb + 1] for row in _anchored_from(M, q, s, qb, rb, gop, gex)[:qe - qb + 1]]
    assert P[qe - qb][re_ - rb] == S
    states = (P, E, F)

    def first(i, j):
        x = max(P[i][j], E[i][j], F[i][j])
        return next(k for k in range(3) if states[k][i][j] == x)

    i, j, st, ops = qe - qb, re_ - rb, 0, []
    counts = [0, 0, 0, 0]
    while True:
        if st == 0:
            a, b = min(q[qb + i], 20), min(s[rb + j], 20)
            ops.append("=" if a == b else "X")
            counts[1] += a == b
            counts[2] += M[a][b] > 0
            if (i, j) == (0, 0):
                break
            i, j = i - 1, j - 1
            assert i >= 0 and j >= 0
            st = first(i, j)
        elif st == 1:
            ops.append("D")
            counts[3] += 1
            ext = E[i][j - 1] + gex == E[i][j]
            j -= 1
            assert j >= 0
            st = 1 if ext else first(i, j)
        else:
            ops.append("I")
            counts[3] += 1
            ext = F[i - 1][j] + gex == F[i][j]
            i -= 1
            assert i >= 0
            st = 2 if ext else first(i, j)
    counts[0] = len(ops)
    return traceback_oracle_lib.cigar_of("".join(reversed(ops)).encode()), counts


def _rescore(M, q, s, c, cigar, gop, gex):
    """Score of a CIGAR by the rescoring rule of include/sw4b200.h, and the query and reference residues it consumes."""
    S, qb, qe, rb, re_ = c
    i, j, score = qb, rb, 0
    for run, op in re.findall(r"(\d+)([=XID])", cigar):
        k = int(run)
        if op in "=X":
            for _ in range(k):
                assert (op == "=") == (min(q[i], 20) == min(s[j], 20))
                score += M[q[i]][s[j]]
                i, j = i + 1, j + 1
        else:
            score += gop + (k - 1) * max(gop, gex)
            if op == "I":
                i += k
            else:
                j += k
    return score, i - qb, j - rb


def _counts_of(M, q, s, c, cigar):
    """(length, identities, positives, gaps) read off a CIGAR and the sequences."""
    i, j, out = c[1], c[3], [0, 0, 0, 0]
    for run, op in re.findall(r"(\d+)([=XID])", cigar):
        k = int(run)
        out[0] += k
        if op in "=X":
            for _ in range(k):
                a, b = min(q[i], 20), min(s[j], 20)
                out[1] += a == b
                out[2] += M[a][b] > 0
                i, j = i + 1, j + 1
        else:
            out[3] += k
            i, j = (i + k, j) if op == "I" else (i, j + k)
    return out


@pytest.mark.parametrize("blosum", [45, 50, 62, 80])
def test_oracle_traceback_equals_python_rule(tb_oracle, oracle, blosum):
    M = oracle.matrix(blosum).astype(int).tolist()
    rng = np.random.default_rng(100 + blosum)
    cases = 0
    for gop, gex in BRUTE_GAPS:
        for letters in (2, 3):
            for _ in range(8):
                alphabet = rng.choice(20, letters, replace=False)
                q = alphabet[rng.integers(0, letters, int(rng.integers(1, 12)))].astype(np.uint8)
                s = alphabet[rng.integers(0, letters, int(rng.integers(1, 12)))].astype(np.uint8)
                got = tb_oracle.traceback(blosum, q, [s], gop, gex)
                c = got.coordinates[0].tolist()
                cigar, counts = _python_rule(M, q.tolist(), s.tolist(), c, gop, gex)
                assert (got.cigars[0], got.counts[0].tolist()) == (cigar, counts), (blosum, gop, gex, q.tolist(), s.tolist())
                cases += 1
    assert cases == 80


def test_oracle_cigars_rescore_to_the_score(tb_oracle, oracle):
    rng = np.random.default_rng(17)
    gapped = 0
    for blosum, gop, gex in MATRICES + EXTRA_GAPS:
        M = oracle.matrix(blosum).astype(int).tolist()
        q = synth.random_residues(rng, int(rng.integers(50, 300)))
        subjects = [synth.random_residues(rng, int(n)) for n in rng.integers(0, 200, 20)]
        subjects += [synth.mutate(rng, q[int(a):int(a) + 150], 0.2, indels=4) for a in rng.integers(0, 40, 10)]
        subjects[-1][::13] = 20  # non-standard residues compare as code 20
        got = tb_oracle.traceback(blosum, q, subjects, gop, gex)
        for s, c, counts, cigar in zip(subjects, got.coordinates.tolist(), got.counts.tolist(), got.cigars):
            if c[0] == 0:
                assert cigar == "" and counts == [0, 0, 0, 0]
                continue
            score, used_q, used_s = _rescore(M, q.tolist(), s.tolist(), c, cigar, gop, gex)
            assert (score, used_q, used_s) == (c[0], c[2] - c[1] + 1, c[4] - c[3] + 1), (blosum, gop, gex, c, cigar)
            assert counts == _counts_of(M, q.tolist(), s.tolist(), c, cigar)
            assert cigar[-1] in "=X" and re.match(r"^\d+[=X]", cigar)
            gapped += counts[3] > 0
    assert gapped >= 20


def test_facade_alignments_compile_standalone(tmp_path):
    import shutil
    gxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else shutil.which("g++")
    if not gxx:
        pytest.skip("no host compiler")
    src = tmp_path / "alignments.cpp"
    src.write_text('#include "cudasw4.cuh"\n'
                   'int main() {\n'
                   '  cudasw4::KernelTypeConfig k; cudasw4::MemoryConfig m;\n'
                   '  cudasw4::CudaSW4 sw({0}, 10, cudasw4::BlosumType::BLOSUM62_20, k, m, false);\n'
                   '  std::vector<cudasw4::ReferenceIdT> ids{0, 3};\n'
                   '  std::vector<cudasw4::Alignment> a = sw.computeAlignments("ACDE", 4, ids);\n'
                   '  return a[0].coordinates.score + a[0].length + a[0].identities + a[0].positives + a[0].gaps +\n'
                   '         (int)a[0].cigar.size();\n'
                   '}\n')
    r = subprocess.run([gxx, "-std=c++17", "-Wall", "-Werror", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), str(src)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _assert_same(got, want, ctx=None):
    assert got.coordinates.dtype == np.int32 and got.counts.dtype == np.int32
    assert got.coordinates.shape == want.coordinates.shape and got.counts.shape == want.counts.shape
    bad = [k for k in range(len(want.cigars)) if (got.coordinates[k] != want.coordinates[k]).any()
           or (got.counts[k] != want.counts[k]).any() or got.cigars[k] != want.cigars[k]]
    assert not bad, (ctx, [(k, got.coordinates[k].tolist(), want.coordinates[k].tolist(), got.counts[k].tolist(),
                            want.counts[k].tolist(), got.cigars[k][:200], want.cigars[k][:200]) for k in bad[:3]])


def _select(t, ids):
    return traceback_oracle_lib.Traceback(t.coordinates[ids], t.counts[ids], [t.cigars[int(i)] for i in ids])


@pytest.mark.gpu
@pytest.mark.parametrize("blosum,gop,gex", MATRICES + EXTRA_GAPS)
def test_every_subject_matches_oracle_and_scan(tb_oracle, blosum, gop, gex):
    db, rng = _mixed_db()
    ids = np.arange(db.num_sequences)
    with _engine(numTop=25, blosumType=blosum, gop=gop, gex=gex) as eng:
        eng.setDatabase(db)
        for q in _queries(rng, db):
            letters = dbformat.decode(q)
            st = sw.BenchmarkStats()
            got = eng.alignments(letters, ids, stats=st)
            want = tb_oracle.traceback(blosum, q, db, gop, gex)
            _assert_same(got, want, len(q))
            assert len(got.cigars) == db.num_sequences and st.kernelLaunches >= 5
            first = eng.scan(letters)
            top = eng.alignments(letters, first.referenceIds)
            assert (top.coordinates == eng.alignmentCoordinates(letters, first.referenceIds)).all()
            assert top.coordinates[:, 0].tolist() == first.scores
            _assert_same(top, _select(want, first.referenceIds), len(q))
            second = eng.scan(letters)
            assert (first.scores, first.referenceIds) == (second.scores, second.referenceIds)


@pytest.mark.gpu
@pytest.mark.parametrize("blosum,gop,gex", [(62, 0, 0), (62, 0, -1), (62, -1, 0), (62, -11, -1), (45, -4096, -4096)])
def test_tie_heavy_inputs(tb_oracle, blosum, gop, gex):
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
            got = eng.alignments(dbformat.decode(q), np.arange(db.num_sequences))
            _assert_same(got, tb_oracle.traceback(blosum, q, db, gop, gex), len(q))


@pytest.mark.gpu
def test_long_pairs(tb_oracle):
    """A 35 k query against 20-35 k subjects with planted copies carrying substitutions and indels (rectangles of up to
    35 k x 35 k on the CTA form), and a 70 k query against 1-5 k subjects."""
    rng = np.random.default_rng(36)
    q = synth.random_residues(rng, 35000)
    s0 = synth.random_residues(rng, 20000)
    s1 = np.concatenate([synth.random_residues(rng, 1000), synth.mutate(rng, q[1000:31000], 0.1, indels=12)])
    s1 = np.concatenate([s1, synth.random_residues(rng, 35000 - len(s1))]) if len(s1) < 35000 else s1[:35000]
    s2 = np.concatenate([q[:15000], synth.random_residues(rng, 3000), synth.mutate(rng, q[20000:], 0.05, indels=6)])
    s3 = synth.mutate(rng, q[4000:31000], 0.15, indels=20)
    db = dbformat.from_sequences([s0, s1, s2, s3])
    with _engine(numTop=4, blosumType=45, gop=-9, gex=-3) as eng:
        eng.setDatabase(db)
        st = sw.BenchmarkStats()
        got = eng.alignments(dbformat.decode(q), np.arange(4), stats=st)
        want = tb_oracle.traceback(45, q, db, -9, -3, threads=2)
        _assert_same(got, want)
        big = want.coordinates[:, 0] > 50000
        assert big.sum() >= 3 and (want.counts[big, 3] > 0).all()
        assert ((want.coordinates[big, 2] - want.coordinates[big, 1]) > 20000).all()
        q70 = synth.random_residues(rng, 70000)
        small = [synth.random_residues(rng, int(n)) for n in (1000, 2500, 5000)]
        small[1][200:2200] = synth.mutate(rng, q70[50000:52000], 0.1, indels=4)[:2000]
        db2 = dbformat.from_sequences(small)
        eng.setDatabase(db2)
        got = eng.alignments(dbformat.decode(q70), np.arange(3))
        _assert_same(got, tb_oracle.traceback(45, q70, db2, -9, -3))


@pytest.mark.gpu
def test_database_modes_give_identical_results(tb_oracle):
    db, rng = _modes_db()
    q = synth.random_residues(rng, 250)
    src = db.sequence(db.num_sequences - 3)
    copy = synth.mutate(rng, src[:150], 0.1, indels=2)[:150]
    q[50:50 + len(copy)] = copy
    letters = dbformat.decode(q)
    ids = np.concatenate([np.arange(db.num_sequences), [5, 5, 17]])
    want = _select(tb_oracle.traceback(62, q, db, -11, -1), ids)
    with _engine(numTop=30) as eng:  # before any upload
        eng.setDatabase(db)
        _assert_same(eng.alignments(letters, ids), want, "before upload")
        eng.prefetchDBToGpus()
        _assert_same(eng.alignments(letters, ids), want, "resident")
    with _engine(numTop=30, memoryConfig=sw.MemoryConfig(maxGpuMem=3 << 20)) as eng:  # streamed
        eng.setDatabase(db)
        eng.prefetchDBToGpus()
        assert eng.dbInfo().num_batches >= 4
        first = eng.scan(letters)
        _assert_same(eng.alignments(letters, ids), want, "streamed")
        second = eng.scan(letters)
        assert first.scores == second.scores and first.referenceIds == second.referenceIds
    with _engine(numTop=30, deviceIds=[0, 0, 0]) as eng:  # multi-shard on one GPU
        eng.setDatabase(db)
        _assert_same(eng.alignments(letters, ids), want, "multi-shard")
    with _engine(numTop=30) as eng:
        eng.setShard(1, 3)
        eng.setDatabase(db)
        _assert_same(eng.alignments(letters, ids), want, "sharded")


@pytest.mark.gpu
def test_presharded_handle_chunking_and_errors(tb_oracle):
    db, rng = _modes_db()
    q = synth.random_residues(rng, 400)
    src = db.sequence(db.num_sequences - 1)
    q[100:100 + min(250, len(src))] = src[:min(250, len(src))]
    letters = dbformat.decode(q)
    want = tb_oracle.traceback(62, q, db, -11, -1)
    gids = np.unique([i for i in range(db.num_sequences) if (i // 256) % 3 == 1] + [db.num_sequences - 1]).astype(np.int32)
    local = dbformat.from_sequences([db.sequence(int(i)) for i in gids])
    with _engine(numTop=10) as eng:
        eng.setDatabaseShard(local, gids, db.num_sequences)
        st = sw.BenchmarkStats()
        _assert_same(eng.alignments(letters, gids, stats=st), _select(want, gids), "pre-sharded")
        whole = st.kernelLaunches
        empty = eng.alignments(letters, [])
        assert empty.coordinates.shape == (0, 5) and empty.counts.shape == (0, 4) and empty.cigars == []
        for bad in ([int(gids[0]) - 1], [-1], [db.num_sequences]):
            with pytest.raises(sw.SW4Error) as e:
                eng.alignments(letters, bad)
            assert e.value.code == -1
    # the largest rectangle: its trace scratch is a little more than half a byte per cell of 32-row-padded tiles
    c = want.coordinates[gids]
    rows, cols = c[:, 2] - c[:, 1] + 1, c[:, 4] - c[:, 3] + 1
    big = int(np.argmax(np.where(c[:, 0] > 0, rows * cols, 0)))
    assert rows[big] >= 200
    trace_big = ((cols[big] + 511) // 512) * (rows[big] + 31) * 256
    with _engine(numTop=10, memoryConfig=sw.MemoryConfig(maxTempBytes=int(trace_big) + 40_000)) as eng:
        eng.setDatabaseShard(local, gids, db.num_sequences)
        st = sw.BenchmarkStats()
        _assert_same(eng.alignments(letters, gids, stats=st), _select(want, gids), "chunked")
        assert st.kernelLaunches > whole + 10  # more chunks, two kernels each
        # a budget that holds the coordinate passes of the pair but not its rectangle's trace
        eng.setMemoryConfig(sw.MemoryConfig(maxTempBytes=int(trace_big) // 2))
        with pytest.raises(sw.SW4Error) as e:
            eng.alignments(letters, [int(gids[big])])
        assert e.value.code == -4
        assert (eng.alignmentCoordinates(letters, [int(gids[big])]) == want.coordinates[[int(gids[big])]]).all()


@pytest.mark.gpu
def test_score_zero_pairs_give_empty_cigars():
    A, W = dbformat.encode("A")[0], dbformat.encode("W")[0]
    db = dbformat.from_sequences([np.zeros(0, np.uint8), np.full(5, A, np.uint8), np.full(30, W, np.uint8)])
    with _engine(numTop=3) as eng:
        eng.setDatabase(db)
        got = eng.alignments(dbformat.decode(np.full(20, A, np.uint8)), [0, 2, 1, 0])
        assert got.cigars == ["", "", "5=", ""]
        assert got.coordinates[[0, 1, 3]].tolist() == [[0, -1, -1, -1, -1]] * 3
        assert got.coordinates[2].tolist() == [20, 0, 4, 0, 4]
        assert got.counts[[0, 1, 3]].tolist() == [[0, 0, 0, 0]] * 3
        assert got.counts[2].tolist() == [5, 5, 5, 0]


# ---------------------------------------------------------------------------------------------------------------------
# CLI
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mat,extra", ALIGN_CASES)
def test_align_tsv_cigar(tb_oracle, tmp_path, golden_dir, mat, extra):
    common = align_case_inputs(str(tmp_path), mat, extra)
    _run_align(ALIGN, common + ["--dpx", "--coordinates", "--cigar", "--of", "cigar.tsv"], str(tmp_path))
    base, tail = _split_tsv(open(tmp_path / "cigar.tsv").read(), 9)
    with open(os.path.join(golden_dir, "align", f"{mat}.tsv")) as f:
        assert base == f.read()
    assert tail[0] == ["Query begin", "Query end", "Reference begin", "Reference end", "Alignment length", "Identities",
                       "Positives", "Gaps", "CIGAR"]
    blosum = int(mat[-2:])
    gop = int(extra[1]) if extra else (-13 if blosum == 45 else -11)
    gex = int(extra[3]) if extra else (-2 if blosum == 45 else -1)
    db = dbformat.read_db(str(tmp_path / "db"))
    queries = [dbformat.encode(s) for _, s in dbformat.read_fasta(str(tmp_path / "q.fa"))]
    rows = [line.split("\t") for line in base.splitlines()[1:]]
    assert rows
    for row, t in zip(rows, tail[1:]):
        q, rid = queries[int(row[0])], int(row[7])
        want = tb_oracle.traceback(blosum, q, [db.sequence(rid)], gop, gex)
        c = want.coordinates[0]
        assert int(row[4]) == c[0]
        assert [int(x) for x in t[:4]] == [int(c[1]) + 1, int(c[2]) + 1, int(c[3]) + 1, int(c[4]) + 1]
        assert [int(x) for x in t[4:8]] == want.counts[0].tolist() and t[8] == want.cigars[0]
    # without --coordinates the five columns follow the base columns directly
    _run_align(ALIGN, common + ["--dpx", "--cigar", "--of", "cigar_only.tsv"], str(tmp_path))
    base2, tail2 = _split_tsv(open(tmp_path / "cigar_only.tsv").read(), 5)
    assert base2 == base and tail2 == [t[4:] for t in tail]


@pytest.mark.gpu
def test_align_plain_cigar_pseudodb(tmp_path, golden_dir):
    common = pseudodb_case_inputs(str(tmp_path))
    _run_align(ALIGN, common + ["--cigar", "--of", "res.txt"], str(tmp_path))
    lines = open(tmp_path / "res.txt").read().splitlines()
    stripped = []
    pattern = re.compile(r" Identities (\d+)/(\d+)\. Positives (\d+)/(\d+)\. Gaps (\d+)/(\d+)\. CIGAR ((?:\d+[=XID])*)\.$")
    for line in lines:
        if line.startswith("Result "):
            m = pattern.search(line)
            assert m, line
            assert m.group(2) == m.group(4) == m.group(6)
            assert sum(int(k) for k in re.findall(r"(\d+)[=XID]", m.group(7))) == int(m.group(2))
            line = line[:m.start()]
        stripped.append(line)
    with open(os.path.join(golden_dir, "align", "pseudodb.txt")) as f:
        assert "\n".join(stripped) + "\n" == f.read()


@pytest.mark.gpu
def test_align_cigar_batch_and_streaming_write_the_same_file(tmp_path):
    from tests.test_cli import MAKEDB
    recs, queries = synth.config_c1(seed=2, n=12000)
    dbformat.write_fasta(str(tmp_path / "db.fa"), recs)
    dbformat.write_fasta(str(tmp_path / "q.fa"), queries[:9])
    subprocess.run([MAKEDB, str(tmp_path / "db.fa"), str(tmp_path / "db")], check=True, stdout=subprocess.DEVNULL)
    common = ["--query", "q.fa", "--db", "db", "--top", "12", "--mat", "blosum62", "--dpx", "--coordinates", "--cigar"]
    _run_align(ALIGN, common + ["--of", "plain.txt"], str(tmp_path))
    _run_align(ALIGN, common + ["--of", "batched.txt", "--batchQueries", "4"], str(tmp_path))
    _run_align(ALIGN, common + ["--of", "streamed.txt", "--maxGpuMem", "5M", "--batchQueries", "16"], str(tmp_path))
    plain = open(tmp_path / "plain.txt").read()
    assert plain.count(" CIGAR ") == 9 * 12
    assert open(tmp_path / "batched.txt").read() == plain
    assert open(tmp_path / "streamed.txt").read() == plain
