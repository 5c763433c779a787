"""Search with a position-specific scoring matrix (sw4_*_pssm / CudaSW4 pssm= / align --pssm).

CPU: the PSSM restatement (tests/pssm_oracle.cpp) against the sequence oracles with pssm[p] = M[q_p] and against a
brute force on tiny inputs with random PSSMs; every CIGAR it gives rescored with positional scores; the facade's
overloads; the Python argument checks; align --pssm refusing malformed files. GPU: a PSSM built as M[q_p] gives what
the sequence query gives on every kernel path; truly positional PSSMs against the restatement in every database mode;
saturating PSSMs on both exact re-scoring kernels; the CLI against align --query."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import cudasw4_b200 as sw
from cudasw4_b200 import dbformat, synth
from tests import coords_oracle as coords_oracle_lib
from tests import pssm_oracle as pssm_oracle_lib
from tests import traceback_oracle as traceback_oracle_lib
from tests.test_cli import ALIGN, MAKEDB, _build_cli, _run_align
from tests.test_coordinates import BRUTE_GAPS, EXTRA_GAPS, MATRICES, _brute_force, _engine, _mixed_db, _modes_db, _queries
from tests.test_kernel_paths import (SWITCH_QUERIES, _all_scores, _sm_count, constants, overflow_setup,  # noqa: F401
                                     sweep_dbs, sweep_queries)
from tests.test_traceback import _python_rule

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# (blosum for the letters' table, gop, gex): the compiled-in gap sets, a run-time pair and the limits of the range
PSSM_GAPS = [(62, -11, -1), (45, -13, -2), (80, -10, -1), (62, -5, -3), (62, 0, 0), (62, -4096, -4096)]


@pytest.fixture(scope="module")
def pssm_oracle():
    return pssm_oracle_lib.load()


@pytest.fixture(scope="module")
def coords_oracle(oracle):
    return coords_oracle_lib.load(oracle)


@pytest.fixture(scope="module")
def tb_oracle(coords_oracle):
    return traceback_oracle_lib.load(coords_oracle)


def seq_pssm(M, q):
    """The PSSM that scores like the sequence query q under the 21 x 21 table M: row p = M[q_p]."""
    return np.ascontiguousarray(np.asarray(M, dtype=np.int8)[np.minimum(np.asarray(q, dtype=np.int64), 20)])


def valid_column20(P):
    """Column 20 (any other letter, also the padding code of the device layout) clipped to <= 0, as sw4b200.h requires."""
    P[:, 20] = np.minimum(P[:, 20], 0)
    return P


def random_pssm(rng, n, lo=-6, hi=6, extremes=0.02):
    """Random positional scores, a small share of them at -128 / 127."""
    P = rng.integers(lo, hi + 1, (n, 21))
    P[rng.random((n, 21)) < extremes / 2] = -128
    P[rng.random((n, 21)) < extremes / 2] = 127
    return valid_column20(P).astype(np.int8)


def biased_pssm(rng, target, noise=3, bonus=5):
    """Scores that favour the residues of `target` position by position (a planted subject aligns along it)."""
    P = rng.integers(-noise, noise + 1, (len(target), 21))
    P[np.arange(len(target)), np.minimum(target, 20)] += bonus
    return valid_column20(P).astype(np.int8)


def _rescore_pssm(P, q, s, c, cigar, gop, gex):
    """Score of a CIGAR with positional scores, the residues it consumes, and its counts (length, identities,
    positives, gaps); '=' / 'X' must match the residue codes."""
    S, qb, qe, rb, re_ = c
    i, j, score, counts = qb, rb, 0, [0, 0, 0, 0]
    for run, op in re.findall(r"(\d+)([=XID])", cigar):
        k = int(run)
        counts[0] += k
        if op in "=X":
            for _ in range(k):
                a, b = min(int(q[i]), 20), min(int(s[j]), 20)
                assert (op == "=") == (a == b)
                score += int(P[i][b])
                counts[1] += a == b
                counts[2] += int(P[i][b]) > 0
                i, j = i + 1, j + 1
        else:
            score += gop + (k - 1) * max(gop, gex)
            counts[3] += k
            i, j = (i + k, j) if op == "I" else (i, j + k)
    return score, i - qb, j - rb, counts


def _columns(cigar):
    """The column string of a CIGAR with = and X both written as M."""
    return "".join(("M" if op in "=X" else op) * int(run) for run, op in re.findall(r"(\d+)([=XID])", cigar))


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("blosum,gop,gex", MATRICES + EXTRA_GAPS)
def test_oracle_with_matrix_rows_equals_sequence_oracles(pssm_oracle, coords_oracle, tb_oracle, oracle, blosum, gop, gex):
    M = oracle.matrix(blosum)
    rng = np.random.default_rng(blosum * 7 - gop)
    q = synth.random_residues(rng, int(rng.integers(50, 300)))
    q[::17] = 20
    subjects = [synth.random_residues(rng, int(n)) for n in rng.integers(0, 250, 25)]
    subjects += [synth.mutate(rng, q[int(a):int(a) + 150], 0.2, indels=4) for a in rng.integers(0, 40, 8)]
    P = seq_pssm(M, q)
    got = pssm_oracle.traceback(P, q, subjects, gop, gex)
    want = tb_oracle.traceback(blosum, q, subjects, gop, gex)
    assert (got.coordinates == want.coordinates).all() and (got.counts == want.counts).all() and got.cigars == want.cigars
    assert (got.coordinates[:, 0] == coords_oracle.coords(blosum, q, subjects, gop, gex)[:, 0]).all()
    assert got.coordinates[:, 0].tolist() == [oracle.score(blosum, q, s, gop, gex) for s in subjects]


def test_oracle_equals_brute_force_on_tiny_inputs(pssm_oracle):
    """Two- and three-letter inputs with random PSSMs whose entries include -128 and 127: the coordinates by
    enumerating every (begin, end) pair, the columns by the walk over full matrices (both restated in Python)."""
    rng = np.random.default_rng(2025)
    cases = extremes = 0
    for gop, gex in BRUTE_GAPS:
        for letters in (2, 3):
            for _ in range(10):
                alphabet = rng.choice(20, letters, replace=False)
                q = alphabet[rng.integers(0, letters, int(rng.integers(1, 10)))].astype(np.uint8)
                s = alphabet[rng.integers(0, letters, int(rng.integers(1, 10)))].astype(np.uint8)
                P = random_pssm(rng, len(q), -8, 8, extremes=0.2)
                extremes += int((P == -128).any() and (P == 127).any())
                # the brute force indexes M[q_i][s_j]: positions as the query and one PSSM row per position
                rows = P.astype(int).tolist()
                pos = list(range(len(q)))
                want = _brute_force(rows, pos, s.tolist(), gop, gex)
                got = pssm_oracle.traceback(P, q, [s], gop, gex)
                assert tuple(got.coordinates[0].tolist()) == want, (gop, gex, q.tolist(), s.tolist(), rows)
                # the walk decides on the states only, so its ops up to = / X come from the positional restatement
                cigar, _ = _python_rule(rows, pos, s.tolist(), list(want), gop, gex)
                assert _columns(got.cigars[0]) == _columns(cigar)
                if want[0] > 0:
                    score, _, _, counts = _rescore_pssm(P, q, s, want, got.cigars[0], gop, gex)
                    assert score == want[0] and counts == got.counts[0].tolist()
                cases += 1
    assert cases == 100 and extremes >= 10


def test_oracle_cigars_rescore_with_positional_scores(pssm_oracle):
    rng = np.random.default_rng(31)
    gapped = 0
    for _, gop, gex in PSSM_GAPS + [(62, 0, -4096)]:
        q = synth.random_residues(rng, int(rng.integers(80, 300)))
        P = biased_pssm(rng, q)
        P[rng.random(P.shape) < 0.01] = 127
        P[rng.random(P.shape) < 0.01] = -128
        subjects = [synth.random_residues(rng, int(n)) for n in rng.integers(0, 200, 15)]
        subjects += [synth.mutate(rng, q[int(a):int(a) + 150], 0.2, indels=4) for a in rng.integers(0, 40, 10)]
        got = pssm_oracle.traceback(P, q, subjects, gop, gex)
        for s, c, counts, cigar in zip(subjects, got.coordinates.tolist(), got.counts.tolist(), got.cigars):
            if c[0] == 0:
                assert cigar == "" and counts == [0, 0, 0, 0] and c[1:] == [-1, -1, -1, -1]
                continue
            score, used_q, used_s, recount = _rescore_pssm(P, q, s, c, cigar, gop, gex)
            assert (score, used_q, used_s) == (c[0], c[2] - c[1] + 1, c[4] - c[3] + 1), (gop, gex, c, cigar)
            assert recount == counts
            gapped += counts[3] > 0
    assert gapped >= 15


def test_facade_pssm_overloads_compile_standalone(tmp_path):
    import shutil
    gxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else shutil.which("g++")
    if not gxx:
        pytest.skip("no host compiler")
    src = tmp_path / "pssm.cpp"
    src.write_text('#include "cudasw4.cuh"\n'
                   'int main() {\n'
                   '  cudasw4::KernelTypeConfig k; cudasw4::MemoryConfig m;\n'
                   '  cudasw4::CudaSW4 sw({0}, 10, cudasw4::BlosumType::BLOSUM62_20, k, m, false);\n'
                   '  std::vector<cudasw4::ReferenceIdT> ids{0, 3};\n'
                   '  std::int8_t pssm[4 * 21] = {};\n'
                   '  cudasw4::ScanResult r = sw.scan("ACDE", pssm, 4);\n'
                   '  std::vector<cudasw4::ScanResult> many = sw.scanMany({std::string_view("ACDE")}, {pssm});\n'
                   '  std::vector<cudasw4::AlignmentCoordinates> c = sw.computeAlignmentCoordinates("ACDE", pssm, 4, ids);\n'
                   '  std::vector<cudasw4::Alignment> a = sw.computeAlignments("ACDE", pssm, 4, ids);\n'
                   '  return (int)r.scores.size() + (int)many.size() + c[0].score + a[0].positives + (int)a[0].cigar.size();\n'
                   '}\n')
    r = subprocess.run([gxx, "-std=c++17", "-Wall", "-Werror", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), str(src)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_python_refuses_bad_pssms_before_the_call():
    for bad, n in ((np.zeros((3, 20)), 3), (np.zeros((2, 21)), 3), (np.zeros(63), 3), (np.full((3, 21), 128), 3),
                   (np.full((3, 21), -129), 3), (np.full((3, 21), 0.5), 3), (np.eye(3, 21, 18, dtype=np.int8), 3)):
        with pytest.raises(ValueError):
            sw._pssm_array(bad, n)
    ok = sw._pssm_array(np.full((3, 21), -128, dtype=np.int64), 3)
    assert ok.dtype == np.int8 and (ok == -128).all()


def write_ascii_pssm(path, letters, rows20):
    """A PSI-BLAST style ASCII PSSM: a title, the header of 20 letters (twice, as PSI-BLAST prints it), rows of
    position, letter, 20 scores and extra columns, then the statistics that end the matrix."""
    order = "ARNDCQEGHILKMFPSTWYV"
    with open(path, "w") as f:
        f.write("\nLast position-specific scoring matrix computed, weighted observed percentages rounded down\n")
        f.write("           " + " ".join(f"{c:>3}" for c in order) + " " + " ".join(f"{c:>3}" for c in order) + "\n")
        for p, (a, row) in enumerate(zip(letters, rows20)):
            f.write(f"{p + 1:>5} {a} " + " ".join(f"{int(v):>3}" for v in row) + "   " + " ".join(["0"] * 20) + "  0.50 0.10\n")
        f.write("\n                      K         Lambda\nStandard Ungapped    0.1337     0.3176\n")


def test_align_refuses_malformed_pssm_files(tmp_path):
    _build_cli()
    good = [[1] * 20, [2] * 20]
    cases = {}
    write_ascii_pssm(tmp_path / "order.pssm", "AC", good)
    text = open(tmp_path / "order.pssm").read()
    cases["order"] = text.replace(" A   R   N", " R   A   N", 1)
    cases["noheader"] = "\n".join(line for line in text.splitlines() if " R " not in line) + "\n"
    cases["gap"] = text.replace("    2 C", "    3 C")
    cases["missing"] = "\n".join(line for line in text.splitlines() if not line.startswith("    1 ")) + "\n"
    cases["range"] = text.replace("    2 C   2", "    2 C 128")
    cases["range_low"] = text.replace("    2 C   2", "    2 C -129")
    cases["short"] = "\n".join(line if not line.startswith("    2 ") else "    2 C 1 2 3" for line in text.splitlines()) + "\n"
    cases["norows"] = "\n".join(line for line in text.splitlines() if not line.startswith(("    1 ", "    2 "))) + "\n"
    for name, content in cases.items():
        assert content != text, name
        (tmp_path / f"{name}.pssm").write_text(content)
        r = subprocess.run([ALIGN, "--pssm", f"{name}.pssm", "--db", "nodb"], cwd=tmp_path, capture_output=True, text=True,
                           timeout=60)
        assert r.returncode != 0 and "PSSM file" in r.stderr, (name, r.stdout[-300:], r.stderr[-300:])
        assert "usable CUDA device" not in r.stderr
    r = subprocess.run([ALIGN, "--pssm", "order.pssm", "--query", "q.fa", "--db", "nodb"], cwd=tmp_path, capture_output=True,
                       text=True, timeout=60)
    assert r.returncode != 0 and "--query and --pssm" in r.stderr


# ---------------------------------------------------------------------------------------------------------------------
# GPU: a PSSM built from the matrix gives exactly what the sequence query gives
# ---------------------------------------------------------------------------------------------------------------------
def _same_scan(eng, n, letters, P, k):
    a = eng.scan(letters)
    all_a = _all_scores(eng, n)
    b = eng.scan(letters, pssm=P)
    all_b = _all_scores(eng, n)
    bad = np.nonzero(all_a != all_b)[0]
    assert len(bad) == 0, (len(letters), bad[:8], all_a[bad[:8]], all_b[bad[:8]])
    assert (a.scores, a.referenceIds) == (b.scores, b.referenceIds) and len(a.scores) == k
    assert a.stats.numOverflows == b.stats.numOverflows
    return b


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["few", "many"])
def test_matrix_rows_equal_sequence_scan_on_every_kernel_path(oracle, sweep_dbs, kind):
    sm, dbs = sweep_dbs
    db = dbs[kind]
    M = oracle.matrix(62)
    rng = np.random.default_rng(71)
    with sw.CudaSW4(deviceIds=[0], numTop=17, blosumType=62) as eng:
        eng.setDatabase(db)
        for ql in sweep_queries(sm):
            q = synth.random_residues(rng, ql)
            if ql > 30:
                q[ql // 3] = 20
            _same_scan(eng, db.num_sequences, dbformat.decode(q), seq_pssm(M, q), 17)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["few", "many"])
def test_matrix_rows_equal_sequence_scan_with_overflows(oracle, overflow_setup, kind):  # noqa: F811
    """The W-rich query whose subjects score 24999..32768: the array re-scoring kernels and numOverflows."""
    sm, q, dbs = overflow_setup
    db, ref = dbs[kind]
    with sw.CudaSW4(deviceIds=[0], numTop=12, blosumType=62) as eng:
        eng.setDatabase(db)
        b = _same_scan(eng, db.num_sequences, dbformat.decode(q), seq_pssm(oracle.matrix(62), q), 12)
        assert b.stats.numOverflows > 0 and (_all_scores(eng, db.num_sequences) == ref).all()


_SWITCH_CHILD = r'''
import sys
import numpy as np
sys.path.insert(0, %(root)r)
import cudasw4_b200 as sw
from cudasw4_b200 import dbformat
d = np.load(sys.argv[1])
db = dbformat.SequenceDB(d["chars"], d["offsets"], d["lengths"], d["headers"], d["header_offsets"])
n, nq, M = db.num_sequences, int(d["nq"]), d["M"]
def all_scores(eng):
    s, i = eng.lastScanAllScores()
    out = np.empty(n, np.int32)
    out[i] = s
    return out
with sw.CudaSW4(deviceIds=[0], numTop=11, blosumType=62) as eng:
    eng.setDatabase(db)
    qs = [d["q%%d" %% i] for i in range(nq)]
    for q in qs:
        a = eng.scan(dbformat.decode(q)); sa = all_scores(eng)
        b = eng.scan(dbformat.decode(q), pssm=M[q]); sb = all_scores(eng)
        assert (sa == sb).all() and a.scores == b.scores and a.referenceIds == b.referenceIds, len(q)
        assert a.stats.numOverflows == b.stats.numOverflows, len(q)
    assert (sb == d["ref_last"]).all()
    many, _ = eng.scanMany([dbformat.decode(q) for q in qs], pssm=[M[q] for q in qs])
    for q, r in zip(qs, many):
        assert r.scores == eng.scan(dbformat.decode(q)).scores
print("ok")
'''


@pytest.mark.gpu
@pytest.mark.parametrize("switch", [{"SW4_NO_LONG_KERNEL": "1"}, {"SW4_NO_TWO_ROW_MULTI": "1"}],
                         ids=lambda s: ",".join(s))
def test_matrix_rows_equal_sequence_scan_under_switches(oracle, overflow_setup, tmp_path, switch):  # noqa: F811
    sm, qw, dbs = overflow_setup
    db, ref_w = dbs["few"]
    rng = np.random.default_rng(56)
    qs = [synth.random_residues(rng, n) for n in SWITCH_QUERIES[:-1]] + [qw]
    arrays = dict(chars=db.chars, offsets=db.offsets, lengths=db.lengths, headers=db.headers, header_offsets=db.header_offsets,
                  nq=len(qs), M=oracle.matrix(62).astype(np.int8), ref_last=ref_w)
    arrays.update({"q%d" % i: q for i, q in enumerate(qs)})
    path = str(tmp_path / "inputs.npz")
    np.savez(path, **arrays)
    r = subprocess.run([sys.executable, "-c", _SWITCH_CHILD % {"root": ROOT}, path], env=dict(os.environ, **switch),
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "ok" in r.stdout, (switch, r.stdout[-500:], r.stderr[-2000:])


@pytest.mark.gpu
@pytest.mark.parametrize("blosum,gop,gex", [(62, -11, -1), (45, -13, -2), (80, -4096, -4096)])
def test_matrix_rows_equal_sequence_coordinates_and_traceback(oracle, blosum, gop, gex):
    db, rng = _mixed_db()
    ids = np.arange(db.num_sequences)
    M = oracle.matrix(blosum)
    with _engine(numTop=25, blosumType=blosum, gop=gop, gex=gex) as eng:
        eng.setDatabase(db)
        for q in _queries(rng, db):
            letters, P = dbformat.decode(q), seq_pssm(M, q)
            assert (eng.alignmentCoordinates(letters, ids, pssm=P) == eng.alignmentCoordinates(letters, ids)).all()
            a, b = eng.alignments(letters, ids), eng.alignments(letters, ids, pssm=P)
            assert (a.coordinates == b.coordinates).all() and (a.counts == b.counts).all() and a.cigars == b.cigars


# ---------------------------------------------------------------------------------------------------------------------
# GPU: truly positional PSSMs against the restatement
# ---------------------------------------------------------------------------------------------------------------------
def _assert_same(got, want, ctx=None):
    bad = [k for k in range(len(want.cigars)) if (got.coordinates[k] != want.coordinates[k]).any()
           or (got.counts[k] != want.counts[k]).any() or got.cigars[k] != want.cigars[k]]
    assert not bad, (ctx, [(k, got.coordinates[k].tolist(), want.coordinates[k].tolist(), got.counts[k].tolist(),
                            want.counts[k].tolist(), got.cigars[k][:200], want.cigars[k][:200]) for k in bad[:3]])


def _positional_queries(rng, db):
    """(letters codes, PSSM) pairs: random PSSMs and PSSMs biased towards a planted database subject."""
    out = []
    for n in (1, 37, 300, 517, 1500):
        q = synth.random_residues(rng, n)
        out.append((q, random_pssm(rng, n)))
        src = db.sequence(int(rng.integers(db.num_sequences // 2, db.num_sequences)))
        k = min(len(src), n)
        target = q.copy()
        target[:k] = src[:k]
        out.append((q, biased_pssm(rng, target)))
    return out


def _check_positional(eng, pssm_oracle, db, q, P, gop, gex, k, ids=None):
    letters = dbformat.decode(q)
    want = pssm_oracle.traceback(P, q, db, gop, gex)
    res = eng.scan(letters, pssm=P)
    scores = _all_scores(eng, db.num_sequences)
    bad = np.nonzero(scores != want.coordinates[:, 0])[0]
    assert len(bad) == 0, (len(q), bad[:8], scores[bad[:8]], want.coordinates[bad[:8], 0])
    order = np.lexsort((np.arange(db.num_sequences), -want.coordinates[:, 0].astype(np.int64)))[:k]
    assert res.scores == want.coordinates[order, 0].tolist() and res.referenceIds == order.tolist()
    L = db.lengths
    assert res.stats.numOverflows == int(((scores >= 25000) & (L > 240) & (L <= 8000)).sum())
    ids = np.arange(db.num_sequences) if ids is None else ids
    assert (eng.alignmentCoordinates(letters, ids, pssm=P) == want.coordinates[ids]).all()
    got = eng.alignments(letters, ids, pssm=P)
    _assert_same(got, traceback_oracle_lib.Traceback(want.coordinates[ids], want.counts[ids], [want.cigars[int(i)] for i in ids]),
                 len(q))
    return want


@pytest.mark.gpu
@pytest.mark.parametrize("blosum,gop,gex", PSSM_GAPS)
def test_positional_pssms_match_oracle(pssm_oracle, blosum, gop, gex):
    db, rng = _mixed_db(13)
    with _engine(numTop=20, blosumType=blosum, gop=gop, gex=gex) as eng:
        eng.setDatabase(db)
        queries = _positional_queries(rng, db)
        for q, P in queries:
            _check_positional(eng, pssm_oracle, db, q, P, gop, gex, 20)
        # sw4_scan_many_pssm against single PSSM scans
        many, _ = eng.scanMany([dbformat.decode(q) for q, _ in queries], pssm=[P for _, P in queries])
        for (q, P), r in zip(queries, many):
            one = eng.scan(dbformat.decode(q), pssm=P)
            assert (r.scores, r.referenceIds, r.stats.numOverflows) == (one.scores, one.referenceIds, one.stats.numOverflows)


@pytest.mark.gpu
def test_positional_pssm_in_every_database_mode(pssm_oracle):
    db, rng = _modes_db()
    src = db.sequence(db.num_sequences - 3)
    q = synth.random_residues(rng, 250)
    target = q.copy()
    target[50:50 + min(150, len(src))] = src[:min(150, len(src))]
    P = biased_pssm(rng, target)
    letters = dbformat.decode(q)
    ids = np.concatenate([np.arange(0, db.num_sequences, 7), [db.num_sequences - 3] * 2])
    want = pssm_oracle.traceback(P, q, db, -11, -1)
    want_ids = traceback_oracle_lib.Traceback(want.coordinates[ids], want.counts[ids], [want.cigars[int(i)] for i in ids])
    top = np.lexsort((np.arange(db.num_sequences), -want.coordinates[:, 0].astype(np.int64)))[:30]

    def check(eng, ctx):
        res = eng.scan(letters, pssm=P)
        assert res.scores == want.coordinates[top, 0].tolist() and res.referenceIds == top.tolist(), ctx
        _assert_same(eng.alignments(letters, ids, pssm=P), want_ids, ctx)

    with _engine(numTop=30) as eng:
        eng.setDatabase(db)
        check(eng, "resident")
        assert (_all_scores(eng, db.num_sequences) == want.coordinates[:, 0]).all()
    with _engine(numTop=30, memoryConfig=sw.MemoryConfig(maxGpuMem=3 << 20)) as eng:
        eng.setDatabase(db)
        eng.prefetchDBToGpus()
        assert eng.dbInfo().num_batches >= 4
        check(eng, "streamed")
    with _engine(numTop=30, deviceIds=[0, 0, 0]) as eng:
        eng.setDatabase(db)
        check(eng, "multi-shard")
    gids = np.unique([i for i in range(db.num_sequences) if (i // 256) % 3 == 1] + [db.num_sequences - 3]).astype(np.int32)
    local = dbformat.from_sequences([db.sequence(int(i)) for i in gids])
    with _engine(numTop=10) as eng:
        eng.setDatabaseShard(local, gids, db.num_sequences)
        res = eng.scan(letters, pssm=P)
        lt = gids[np.lexsort((gids, -want.coordinates[gids, 0].astype(np.int64)))[:10]]
        assert res.scores == want.coordinates[lt, 0].tolist() and res.referenceIds == lt.tolist()
        sel = gids[::5]
        _assert_same(eng.alignments(letters, sel, pssm=P), traceback_oracle_lib.Traceback(
            want.coordinates[sel], want.counts[sel], [want.cigars[int(i)] for i in sel]), "pre-sharded")
    c = want.coordinates[ids]
    rows, cols = c[:, 2] - c[:, 1] + 1, c[:, 4] - c[:, 3] + 1
    big = int(np.max(np.where(c[:, 0] > 0, ((cols + 511) // 512) * (rows + 31) * 256, 0)))
    with _engine(numTop=10, memoryConfig=sw.MemoryConfig(maxTempBytes=big + 40_000)) as eng:  # chunked
        eng.setDatabase(db)
        st = sw.BenchmarkStats()
        _assert_same(eng.alignments(letters, ids, stats=st, pssm=P), want_ids, "chunked")
        assert st.kernelLaunches > 12


@pytest.mark.gpu
def test_positional_pssm_long_pairs(pssm_oracle):
    """A 35 k PSSM query against 20-35 k subjects, planted copies with substitutions and indels: the CTA form of the
    coordinate passes and of the traceback pass."""
    rng = np.random.default_rng(37)
    q = synth.random_residues(rng, 35000)
    s0 = synth.random_residues(rng, 20000)
    s1 = np.concatenate([synth.random_residues(rng, 1000), synth.mutate(rng, q[1000:31000], 0.1, indels=12)])
    s1 = np.concatenate([s1, synth.random_residues(rng, 35000 - len(s1))]) if len(s1) < 35000 else s1[:35000]
    s2 = synth.mutate(rng, q[4000:31000], 0.15, indels=20)
    db = dbformat.from_sequences([s0, s1, s2])
    P = biased_pssm(rng, q, noise=4, bonus=6)
    with _engine(numTop=3, gop=-9, gex=-3) as eng:
        eng.setDatabase(db)
        want = pssm_oracle.traceback(P, q, db, -9, -3, threads=3)
        got = eng.alignments(dbformat.decode(q), np.arange(3), pssm=P)
        _assert_same(got, want)
        assert (want.coordinates[1:, 0] > 50000).all() and (want.counts[1:, 3] > 0).all()
        assert ((want.coordinates[1:, 2] - want.coordinates[1:, 1]) > 20000).all()


# ---------------------------------------------------------------------------------------------------------------------
# GPU: saturation, bounds and empty alignments
# ---------------------------------------------------------------------------------------------------------------------
def _saturating_db(rng, consensus, lengths):
    """Random subjects plus copies of prefixes of `consensus` (at most 8000 residues), each padded to a given length."""
    seqs = [synth.random_residues(rng, int(n)) for n in rng.integers(1, 1200, 600)]
    for n in lengths:
        s = synth.random_residues(rng, n)
        k = min(n, len(consensus))
        s[:k] = consensus[:k]
        seqs.append(s)
    return dbformat.from_sequences(seqs)


@pytest.mark.gpu
@pytest.mark.parametrize("qlen", [200, 400, 780, 785, 1200])
def test_saturating_pssm_rescores_exactly(pssm_oracle, qlen):
    """Entries of 127 along a consensus drive planted subjects past the 16-bit threshold: queries below about 785
    residues re-score on sw_s32_kernel, longer ones on the s32 array. Every score equals the restatement's, numOverflows
    follows its rule (and Half2's threshold of 2048), and the coordinates and CIGARs of the top hits match."""
    rng = np.random.default_rng(qlen)
    consensus = synth.random_residues(rng, qlen)
    P = valid_column20(rng.integers(-4, 3, (qlen, 21))).astype(np.int8)
    P[np.arange(qlen), consensus] = 127
    db = _saturating_db(rng, consensus, [qlen // 2, qlen, qlen + 1, 239, 241, 900, 2500])
    q = synth.random_residues(rng, qlen)
    want = pssm_oracle.traceback(P, q, db, -11, -1)
    assert int((want.coordinates[:, 0] >= 25000).sum()) >= 3
    with _engine(numTop=12) as eng:
        eng.setDatabase(db)
        _check_positional(eng, pssm_oracle, db, q, P, -11, -1, 12, ids=np.arange(db.num_sequences - 7, db.num_sequences))
    cfg = sw.KernelTypeConfig(sw.KernelType.Half2, sw.KernelType.Half2, sw.KernelType.Float, sw.KernelType.Float)
    with _engine(numTop=12, kernelTypeConfig=cfg) as eng:
        eng.setDatabase(db)
        res = eng.scan(dbformat.decode(q), pssm=P)
        L, ref = db.lengths, want.coordinates[:, 0]
        assert res.stats.numOverflows == int(((ref >= 2048) & (L > 240) & (L <= 8000)).sum())


@pytest.mark.gpu
def test_all_negative_pssm_and_the_score_bound():
    rng = np.random.default_rng(5)
    db = dbformat.from_sequences([synth.random_residues(rng, int(n)) for n in (0, 1, 50, 700, 3000)])
    q = synth.random_residues(rng, 400)
    P = rng.integers(-128, 0, (400, 21)).astype(np.int8)
    with _engine(numTop=5) as eng:
        eng.setDatabase(db)
        res = eng.scan(dbformat.decode(q), pssm=P)
        assert res.scores == [0] * 5 and (_all_scores(eng, 5) == 0).all()
        got = eng.alignments(dbformat.decode(q), np.arange(5), pssm=P)
        assert (got.coordinates == [[0, -1, -1, -1, -1]] * 5).all() and got.cigars == [""] * 5 and (got.counts == 0).all()
        out = np.empty(5, np.int32)
        with pytest.raises(sw.SW4Error) as e:  # NULL pssm through the C ABI
            eng._check(eng._lib.sw4_scan_pssm(eng._h, b"ACD", None, 3, out.ctypes.data, out.ctypes.data, None, None))
        assert e.value.code == -1 and "pssm" in str(e.value)
        # a positive score for code 20 (also the padding code of the device layout) is refused by the C ABI itself
        bad = np.zeros((3, 21), np.int8)
        bad[1, 20] = 1
        coords = np.empty((1, 5), np.int32)
        ids = np.zeros(1, np.int32)
        for rc in (eng._lib.sw4_scan_pssm(eng._h, b"ACD", bad.ctypes.data, 3, out.ctypes.data, out.ctypes.data, None, None),
                   eng._lib.sw4_alignment_coordinates_pssm(eng._h, b"ACD", bad.ctypes.data, 3, ids.ctypes.data, 1,
                                                           coords.ctypes.data, None)):
            with pytest.raises(sw.SW4Error) as e:
                eng._check(rc)
            assert e.value.code == -1 and "pssm[1][20]" in str(e.value)
    # 127 x min(query, subject) >= 2^24 is refused; the handle's BLOSUM bound would have accepted the pair
    n = (1 << 24) // 127 + 1
    big = dbformat.from_sequences([synth.random_residues(rng, n)])
    qb = synth.random_residues(rng, n)
    Pb = np.zeros((n, 21), np.int8)
    Pb[0, 0] = 127
    with _engine(numTop=1) as eng:
        eng.setDatabase(big)
        for call in (eng.alignmentCoordinates, eng.alignments):
            with pytest.raises(sw.SW4Error) as e:
                call(dbformat.decode(qb), [0], pssm=Pb)
            assert e.value.code == -1 and "2^24" in str(e.value)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the CLI
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_align_pssm_equals_align_query(oracle, tmp_path):
    _build_cli()
    recs, queries = synth.config_c1(seed=3, n=6000)
    dbformat.write_fasta(str(tmp_path / "db.fa"), recs)
    subprocess.run([MAKEDB, str(tmp_path / "db.fa"), str(tmp_path / "db")], check=True, stdout=subprocess.DEVNULL)
    queries = queries[:5]
    dbformat.write_fasta(str(tmp_path / "q.fa"), queries)
    for mat in ("blosum62", "blosum45"):
        M = oracle.matrix(int(mat[-2:]))
        files = []
        for i, (_, letters) in enumerate(queries):
            codes = dbformat.encode(letters)
            f = f"{mat}_q{i}.pssm"
            write_ascii_pssm(tmp_path / f, letters, seq_pssm(M, codes)[:, :20])
            files.append(f)
        pssm_args = [a for f in files for a in ("--pssm", f)]
        headers = [h for h, _ in queries]
        for extra in (["--tsv"], [], ["--tsv", "--coordinates", "--cigar"], ["--coordinates", "--cigar"],
                      ["--tsv", "--batchQueries", "3"], ["--coordinates", "--cigar", "--batchQueries", "4"]):
            common = ["--db", "db", "--top", "9", "--mat", mat] + extra
            _run_align(ALIGN, common + ["--query", "q.fa", "--of", "a.out"], str(tmp_path))
            _run_align(ALIGN, common + pssm_args + ["--of", "b.out"], str(tmp_path))
            a, b = open(tmp_path / "a.out").read(), open(tmp_path / "b.out").read()
            assert a.count("\n") > 9
            for h, f in zip(headers, files):
                if "--tsv" in extra:
                    a = a.replace(f"\t{h}\t", f"\t{f}\t")
                else:
                    a = a.replace(f", header{h}, ", f", header{f}, ")
            assert a == b, (mat, extra)
