"""CPU tests: pin the oracle (oracle/sw_oracle.cpp) against fixtures produced by the reference's own code
(tools/make_golden.py) and against the SURVEY.md §8c known-answer tables."""
import json
import os

import numpy as np
import pytest

from cudasw4_b200 import dbformat, synth


def _load(golden_dir, name):
    with open(os.path.join(golden_dir, name)) as f:
        return json.load(f)


def test_substitution_tables_match_reference(oracle, golden_dir):
    g = _load(golden_dir, "blosum_tables.json")
    for t in (45, 50, 62, 80):
        ref = np.array(g["tables"][str(t)], dtype=np.int8)
        assert (oracle.matrix(t) == ref).all()
        assert (ref == ref.T).all() and (ref[20] == ref[20, 20]).all()
    assert [int(np.array(g["tables"][str(t)]).max()) for t in (45, 50, 62, 80)] == [15, 15, 11, 11]
    assert [int(np.array(g["tables"][str(t)]).min()) for t in (45, 50, 62, 80)] == [-5, -5, -4, -6]


def test_letter_map_matches_reference(oracle, golden_dir):
    g = _load(golden_dir, "ref_misc.json")
    ref = np.array(g["convert_256"], dtype=np.uint8)
    assert (oracle.convert(bytes(range(256))) == ref).all()
    assert (dbformat.encode(bytes(range(256))) == ref).all()
    assert dbformat.decode(np.arange(22)) == "ARNDCQEGHILKMFPSTWYV--"


def test_partition_boundaries(oracle, golden_dir):
    g = _load(golden_dir, "ref_misc.json")
    assert g["boundaries"] == dbformat.BOUNDARIES.tolist()
    assert oracle.lib.sw4o_num_length_partitions() == 36
    assert [oracle.lib.sw4o_length_partition_boundary(i) for i in range(36)] == g["boundaries"]
    for L, p in ((0, 0), (1, 0), (48, 0), (49, 1), (240, 12), (241, 13), (256, 13), (257, 14), (1280, 33), (1281, 34),
                 (8000, 34), (8001, 35), (35000, 35)):
        assert oracle.partition(L) == p


def test_pseudodb_generator(oracle, golden_dir):
    g = _load(golden_dir, "ref_misc.json")["pseudodb"]
    for key, v in g.items():
        L, seed = map(int, key.split("_"))
        Lp = (L + 3) // 4 * 4
        chars = np.array(v["chars"], dtype=np.uint8).reshape(3, Lp)
        assert v["lengths"] == [L] * 3 and v["offsets"] == [0, Lp, 2 * Lp, 3 * Lp]
        assert (chars[0] == chars[1]).all() and (chars[:, L:] == 20).all()
        assert (oracle.pseudo_subject(L, seed) == chars[0, :L]).all()
        assert (synth.pseudo_subject(L, seed) == chars[0, :L]).all()
    db = synth.config_c2(n=5, length=77)
    assert db.num_sequences == 5 and (db.chars.reshape(5, 80)[:, 77:] == 20).all()


def test_oracle_matches_reference_cpu_gotoh(oracle, golden_dir):
    g = _load(golden_dir, "ref_cpu_gotoh.json")
    tiny = dbformat.read_db(os.path.join(golden_dir, "tinydb", "db"))
    queries = [dbformat.encode(s) for _, s in synth.load_queries()]
    for c in g["tinydb_cases"]:
        got = oracle.scan(62, queries[c["query"]], tiny, c["gop"], c["gex"])
        assert got.tolist() == c["scores"], c
    for c in g["random_cases"]:
        assert oracle.score(62, c["q"], c["s"], c["gop"], c["gex"]) == c["score"]
    assert g["random_cases"][-1]["score"] > 2048  # above the half2 envelope


def test_oracle_matches_survey_known_answers(oracle, golden_dir):
    kat = _load(golden_dir, "survey_kat.json")
    tiny = dbformat.read_db(os.path.join(golden_dir, "tinydb", "db"))
    queries = [dbformat.encode(s) for _, s in synth.load_queries()]
    for c in kat["tinydb"]:
        got = oracle.scan(c["blosum"], queries[c["query"]], tiny, c["gop"], c["gex"])
        assert got[: len(c["scores"])].tolist() == c["scores"], c
    for L, scores in kat["pseudodb_blosum62_gop-11_gex-1"].items():
        subj = oracle.pseudo_subject(int(L), 42)
        assert [oracle.score(62, q, subj, -11, -1) for q in queries] == scores


def test_reference_makedb_files_roundtrip(golden_dir, tmp_path):
    """dbformat reads what the reference makedb wrote and writes it back byte-identically."""
    for name in ("tinydb", "tiesdb"):
        d = os.path.join(golden_dir, name)
        db = dbformat.read_db(os.path.join(d, "db"))
        recs = dbformat.read_fasta(os.path.join(d, "input.fasta"))
        assert db.num_sequences == len(recs)
        assert (np.diff(db.lengths) >= 0).all()
        by_header = {h: s for h, s in recs}
        for i in range(db.num_sequences):
            s = by_header[db.header(i)]
            assert int(db.lengths[i]) == len(s)
            assert (db.sequence(i) == dbformat.encode(s)).all()
            assert int(db.offsets[i + 1] - db.offsets[i]) == (len(s) + 3) // 4 * 4
        out = str(tmp_path / name / "db")
        dbformat.write_db(out, db)
        for suffix in ("0chars", "0offsets", "0lengths", "0headers", "0headeroffsets", "0metadata", "metadata"):
            with open(os.path.join(d, "db" + suffix), "rb") as a, open(out + suffix, "rb") as b:
                assert a.read() == b.read(), (name, suffix)
    tiny = dbformat.read_db(os.path.join(golden_dir, "tinydb", "db"))
    assert tiny.lengths.tolist() == [70, 144, 189, 222, 375, 464, 567]
    assert tiny.offsets.tolist() == [0, 72, 216, 408, 632, 1008, 1472, 2040]


def test_topk_tie_rule(oracle):
    scores = np.array([5, 9, 9, 1, 9, 5, 0], dtype=np.int32)
    s, i = oracle.topk(scores, 4)
    assert s.tolist() == [9, 9, 9, 5] and i.tolist() == [1, 2, 4, 0]
    s, i = oracle.topk(scores, 100)
    assert len(s) == 7 and i.tolist() == [1, 2, 4, 0, 5, 3, 6]


def test_oracle_properties(oracle):
    rng = np.random.default_rng(0)
    for _ in range(20):
        q = synth.random_residues(rng, int(rng.integers(1, 200)))
        s = synth.random_residues(rng, int(rng.integers(1, 200)))
        for blosum, gop, gex in ((62, -11, -1), (45, -13, -2), (80, -10, -1), (50, -9, -3)):
            a = oracle.score(blosum, q, s, gop, gex)
            assert a == oracle.score(blosum, s, q, gop, gex)              # symmetric matrices => symmetric score
            assert a == oracle.score(blosum, q[::-1], s[::-1], gop, gex)  # reversal invariance
            assert a >= 0
            padded = np.concatenate([s, np.full(7, 20, np.uint8)])
            assert a == oracle.score(blosum, q, padded, gop, gex)          # padding code never raises the max
    q = synth.random_residues(rng, 50)
    m = oracle.matrix(62)
    assert oracle.score(62, q, q, -11, -1) == sum(int(m[c, c]) for c in q)
    assert oracle.score(62, q, np.zeros(0, np.uint8), -11, -1) == 0


def live_scan_cases():
    """The random database and (query, gop, gex) cases of test_oracle_scan_matches_reference_cpu_routine_live."""
    rng = np.random.default_rng(123)
    seqs = [synth.random_residues(rng, int(n)) for n in rng.integers(1, 900, 1500)]
    seqs += [np.full(40, 20, np.uint8), synth.random_residues(rng, 2500)]
    db = dbformat.from_sequences(seqs)
    cases = [(synth.random_residues(rng, ql), gop, gex) for ql, (gop, gex) in zip((1, 37, 400), ((-11, -1), (-5, -3), (-11, -1)))]
    return db, cases


def test_oracle_scan_matches_reference_cpu_routine_live(oracle, golden_dir):
    """The oracle's scan equals the reference's own scalar CPU Gotoh on a random database, subject by subject: against
    the stored scores of tests/golden/ref_cpu_scan_live.json, and live when oracle/_ref/libref_harness.so has been built
    from the reference sources (oracle/Makefile). tests/golden/ref_cpu_gotoh.json pins the same routine on other inputs."""
    import bench
    with open(os.path.join(golden_dir, "ref_cpu_scan_live.json")) as f:
        stored = json.load(f)["cases"]
    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref", "libref_harness.so")
    ref = bench._ReferenceCpuScan(path) if os.path.exists(path) else None
    db, cases = live_scan_cases()
    assert len(stored) == len(cases)
    for (q, gop, gex), s in zip(cases, stored):
        got = oracle.scan(62, q, db, gop, gex)
        assert [len(q), gop, gex] == [s["query_length"], s["gop"], s["gex"]]
        assert got.tolist() == s["scores"]
        if ref is not None:
            assert (ref.scan(62, q, db, gop, gex) == got).all()
