"""E-values and bit scores from each query's own score statistics (sw4_set_score_statistics, sw4_last_score_statistics,
sw4_last_score_histogram, sw4_fit_score_statistics; CudaSW4.setScoreStatistics; align --evalue / --maxEvalue).

CPU: the library's fit against its numpy restatement (tests/evalue_oracle.py) on random and edge-case histograms; the
fit recovers lambda and K from scores drawn from its own model; a two-rank gloo gather_score_statistics equals the fit
of the summed histograms. GPU: the device histogram equals a numpy histogram of all scores in every database mode;
disabled statistics change nothing; sharded histograms sum to the unsharded fit bit for bit; calibration on a null
database; the gapless limit against the exact ungapped lambda; planted homologs and the cutoff; the CLI columns."""
import math
import os
import socket
import subprocess

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

import cudasw4_b200 as sw
from cudasw4_b200 import dbformat, synth
from cudasw4_b200.distributed import gather_score_statistics
from tests import evalue_oracle as eo
from tests.test_cli import ALIGN, MAKEDB, _build_cli, _run_align

BINS = 4096
FIELDS = ["query_length", "db_residues", "num_subjects", "fitted", "left_censored", "right_censored", "c_lo", "c_hi"]


def _assert_fit_equal(got: sw.ScoreStatistics, want: dict):
    assert got.ok == want["ok"]
    for f in FIELDS:
        assert getattr(got, f) == want[f], f
    if want["ok"]:
        assert abs(got.lambda_ - want["lambda_"]) <= 1e-12 * want["lambda_"]
        assert abs(got.K - want["K"]) <= 1e-12 * want["K"]
    else:
        assert math.isnan(got.lambda_) and math.isnan(got.K)


def _model_histogram(rng, n, lam, K, m, bins=BINS):
    L = synth.lognormal_lengths(rng, n, 5.6, 0.6, 20, 5000)
    return eo.histogram(eo.sample_scores(rng, L, lam, K, m), L, bins)


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def _edge_histograms():
    z = np.zeros(BINS + 1, np.int64)
    out = [("empty", z.copy(), z.copy())]
    c = z.copy(); c[0] = 5000
    out.append(("all zero", c, c * 300))
    rng = np.random.default_rng(11)
    for u in (99, 100):  # exactly u fitted subjects: the median bin holds them, the rest sits below
        c = z.copy(); c[10] = u; c[5] = u - 1
        out.append((f"U={u}", c, c * 250))
    c, L = _model_histogram(rng, 300_000, 0.003, 0.04, 300)  # lambda this small reaches the overflow bin: c_hi = B
    out.append(("overflow", c, L))
    c = z.copy(); c[BINS] = 1000; c[3] = 10
    out.append(("median in the overflow bin", c, c * 100))
    c = z.copy(); c[40:80] = 500; c[BINS] = 900
    out.append(("mass in the overflow bin", c, c * 350))
    return out


def test_fit_equals_restatement_on_random_and_edge_histograms():
    rng = np.random.default_rng(1)
    cases = _edge_histograms()
    assert any(e == "overflow" and eo.fit(c, L, 300)["c_hi"] == BINS for e, c, L in cases)
    assert [eo.fit(c, L, 300)["ok"] for e, c, L in cases if e.startswith("U=")] == [False, True]
    for i in range(40):
        bins = int(rng.choice([8, 64, 300, BINS]))
        n = int(rng.integers(0, 50_000))
        lam, K = float(rng.uniform(0.05, 1.5)), float(rng.uniform(0.005, 0.5))
        c, L = _model_histogram(rng, n, lam, K, int(rng.integers(20, 2000)), bins)
        if i % 4 == 0:  # arbitrary shapes too
            c = rng.integers(0, 50, bins + 1) * (rng.random(bins + 1) < 0.3)
            L = c * rng.integers(1, 900, bins + 1)
        cases.append((f"random {i}", c, L))
    for name, c, L in cases:
        for m in (0, 1, 300):
            _assert_fit_equal(sw.fit_score_statistics(c, L, m), eo.fit(c, L, m))
    with pytest.raises(ValueError):
        bad = np.zeros(BINS + 1, np.int64); bad[3] = -1
        sw.fit_score_statistics(bad, np.zeros(BINS + 1, np.int64), 300)


def test_fit_recovers_the_model():
    rng = np.random.default_rng(2026)
    c, L = _model_histogram(rng, 10**6, 0.267, 0.041, 300)
    st = sw.fit_score_statistics(c, L, 300)
    assert st.ok and st.num_subjects == 10**6
    assert abs(st.lambda_ / 0.267 - 1) <= 0.02, st
    assert abs(st.K / 0.041 - 1) <= 0.15, st
    assert st.evalue(60) == st.K * 300.0 * float(L.sum()) * math.exp(-st.lambda_ * 60)


class _HistogramOnly:
    """Stands in for a CudaSW4 handle: gather_score_statistics only reads the local histogram."""
    def __init__(self, counts, lensums):
        self.h = (counts, lensums)

    def lastScoreHistogram(self, query_index):
        return self.h


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _gather_worker(rank, world, port, hists, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        st = gather_score_statistics(_HistogramOnly(*hists[rank]), 0, 350)
        q.put((rank, st))
    finally:
        dist.destroy_process_group()


def test_gather_score_statistics_two_ranks_equals_fit_of_the_sum():
    rng = np.random.default_rng(5)
    hists = [_model_histogram(rng, 200_000, 0.3, 0.05, 350) for _ in range(2)]
    want = sw.fit_score_statistics(hists[0][0] + hists[1][0], hists[0][1] + hists[1][1], 350)
    assert want.ok
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gather_worker, args=(r, 2, port, hists, q)) for r in range(2)]
    for p in procs:
        p.start()
    results = [q.get(timeout=120) for _ in range(2)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, st in results:
        assert st == want, rank


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _engine(**kw):
    kw.setdefault("deviceIds", [0])
    return sw.CudaSW4(**kw)


def _mixed_db(seed, n, lo, hi, extra=()):
    rng = np.random.default_rng(seed)
    L = np.concatenate([rng.integers(lo, hi + 1, n), np.array(extra, dtype=np.int64), np.zeros(7, np.int64)])
    return dbformat.from_sequences([synth.random_residues(rng, int(x)) for x in L]), rng


def _check_histogram(eng, lengths_by_id, query_index=0):
    """The device histogram of the last scan equals numpy's over lastScanAllScores (which holds the last query)."""
    scores, ids = eng.lastScanAllScores()
    counts, lensums = eng.lastScoreHistogram(query_index)
    c, L = eo.histogram(scores, np.asarray(lengths_by_id)[ids])
    assert (counts == c).all() and (lensums == L).all(), (np.nonzero(counts != c)[0][:8], np.nonzero(lensums != L)[0][:8])
    return counts, lensums


def _null_queries(rng, n, lo=100, hi=1000):
    return [dbformat.decode(synth._PSEUDO_TABLE[rng.integers(0, 256, int(m))]) for m in rng.integers(lo, hi + 1, n)]


def _null_lengths(rng, n):
    return np.sort(synth.lognormal_lengths(rng, n, 5.683, 0.636, 2, 35213)).astype(np.int32)


@pytest.mark.gpu
def test_histogram_equals_numpy_in_every_mode():
    db, rng = _mixed_db(3, 20_000, 1, 900, [1500, 3000, 6000])
    qs = [dbformat.decode(synth.random_residues(rng, int(m))) for m in (40, 300, 1200)]
    with _engine(numTop=10, blosumType=62) as eng:
        eng.setDatabase(db)
        eng.setScoreStatistics(True)
        resident = []
        for q in qs:
            r = eng.scan(q)
            resident.append(_check_histogram(eng, db.lengths))
            st = eng.lastScoreStatistics()
            assert r.statistics == st and st.whole_database and st.num_subjects == db.num_sequences - 7
            assert st.db_residues == int(db.lengths.sum()) and st.query_length == len(q)
            assert st.ok and len(r.evalues) == len(r.scores) == 10
            assert r.evalues == [st.evalue(s) for s in r.scores] and r.evalues == sorted(r.evalues)
        many, _ = eng.scanMany(qs)
        for i, m in enumerate(many):
            counts, lensums = eng.lastScoreHistogram(i)
            assert (counts == resident[i][0]).all() and (lensums == resident[i][1]).all()
            assert m.statistics == eng.lastScoreStatistics(i)
        _check_histogram(eng, db.lengths, len(qs) - 1)
        # PSSM query
        P = rng.integers(-4, 5, (300, 21)).astype(np.int8)
        P[:, 20] = -1
        eng.scan(qs[1], pssm=P)
        _check_histogram(eng, db.lengths)
        assert eng.lastScoreStatistics().query_length == 300
    with _engine(numTop=10, blosumType=62, memoryConfig=sw.MemoryConfig(maxGpuMem=4 << 20)) as eng:
        eng.setDatabase(db)
        eng.setScoreStatistics(True)
        for q, h in zip(qs, resident):
            eng.scan(q)
            counts, lensums = _check_histogram(eng, db.lengths)
            assert (counts == h[0]).all() and (lensums == h[1]).all()
        info = eng.dbInfo()
        print(f"streamed: {info.num_batches} batches")
        assert info.streaming == 1 and info.num_batches >= 4
    with _engine(deviceIds=[0, 0, 0], numTop=10, blosumType=62) as eng:  # three shards: summed on the host
        eng.setDatabase(db)
        eng.setScoreStatistics(True)
        for q, h in zip(qs, resident):
            eng.scan(q)
            counts, lensums = _check_histogram(eng, db.lengths)
            assert (counts == h[0]).all() and (lensums == h[1]).all()
    recs, queries = synth.config_c1(seed=1, n=10_000)  # C1
    c1 = dbformat.from_sequences([dbformat.encode(s) for _, s in recs], [h for h, _ in recs])
    with _engine(numTop=10, blosumType=62) as eng:
        eng.setDatabase(c1)
        eng.setScoreStatistics(True)
        for _, q in queries[:5]:
            eng.scan(q)
            _check_histogram(eng, c1.lengths)


@pytest.mark.gpu
def test_disabled_statistics_change_nothing():
    db, rng = _mixed_db(4, 8000, 1, 1300, [2500, 30_000])
    qs = [dbformat.decode(synth.random_residues(rng, int(m))) for m in (50, 500, 3000)]

    def run(setup):
        with _engine(numTop=20, blosumType=62) as eng:
            eng.setDatabase(db)
            setup(eng)
            out = [eng.scan(q) for q in qs]
            many, total = eng.scanMany(qs)
            return out + many, total

    fresh, total0 = run(lambda eng: None)
    toggled, total1 = run(lambda eng: (eng.setScoreStatistics(True, 1e-3), eng.setScoreStatistics(False)))
    enabled, total2 = run(lambda eng: eng.setScoreStatistics(True))
    for a, b, c in zip(fresh, toggled, enabled):
        assert (a.scores, a.referenceIds, a.stats.numOverflows, a.stats.kernelLaunches) == \
               (b.scores, b.referenceIds, b.stats.numOverflows, b.stats.kernelLaunches)
        assert b.evalues == [] and b.bitScores == [] and b.statistics is None
        assert (c.scores, c.referenceIds, c.stats.numOverflows) == (a.scores, a.referenceIds, a.stats.numOverflows)
        assert c.stats.kernelLaunches == a.stats.kernelLaunches + 1
    assert total0.kernelLaunches == total1.kernelLaunches == total2.kernelLaunches - len(qs)
    with _engine(numTop=20, blosumType=62) as eng:
        eng.setDatabase(db)
        eng.scan(qs[0])
        with pytest.raises(sw.SW4Error):
            eng.lastScoreStatistics()
        with pytest.raises(sw.SW4Error):
            eng.setScoreStatistics(True, float("nan"))


@pytest.mark.gpu
def test_sharded_histograms_sum_to_the_unsharded_fit():
    rng = np.random.default_rng(6)
    L = _null_lengths(rng, 200_000)
    qs = _null_queries(rng, 3)
    with _engine(numTop=10, blosumType=62) as eng:
        eng.setPseudoDatabaseLengths(L, seed=9)
        eng.setScoreStatistics(True)
        whole, _ = eng.scanMany(qs)
    parts = []
    for rank in range(2):
        with _engine(numTop=10, blosumType=62) as eng:
            eng.setShard(rank, 2)
            eng.setPseudoDatabaseLengths(L, seed=9)
            eng.setScoreStatistics(True, 1e-30)  # never applied to a shard
            res, _ = eng.scanMany(qs)
            assert all(not r.statistics.whole_database for r in res)
            assert all(len(r.scores) == 10 for r in res)
            parts.append([eng.lastScoreHistogram(i) for i in range(len(qs))])
    for i, q in enumerate(qs):
        c = parts[0][i][0] + parts[1][i][0]
        lens = parts[0][i][1] + parts[1][i][1]
        st = sw.fit_score_statistics(c, lens, len(q))
        assert st.ok and st == whole[i].statistics, i


@pytest.mark.gpu
def test_calibration_on_a_null_database():
    rng = np.random.default_rng(7)
    L = _null_lengths(rng, 1_000_000)
    qs = _null_queries(rng, 20)
    with _engine(numTop=300, blosumType=62, gop=-11, gex=-1) as eng:
        eng.setPseudoDatabaseLengths(L, seed=21)
        eng.setScoreStatistics(True)
        res, _ = eng.scanMany(qs)
    e10 = [sum(e <= 10 for e in r.evalues) for r in res]
    e1 = [sum(e <= 1 for e in r.evalues) for r in res]
    lam = [round(r.statistics.lambda_, 4) for r in res]
    print(f"null database, 20 queries: E <= 10: {sum(e10)} (expected 200), E <= 1: {sum(e1)} (expected 20); "
          f"per query E <= 10 {e10}, lambda {lam}")
    assert all(r.statistics.ok for r in res) and max(e10) < 300
    assert 200 / 3 <= sum(e10) <= 600


@pytest.mark.gpu
def test_gapless_limit_matches_the_ungapped_lambda(oracle):
    p = np.bincount(synth._PSEUDO_TABLE, minlength=20) / 256.0
    M = oracle.matrix(62)[:20, :20].astype(np.float64)
    lo, hi = 1e-3, 2.0
    for _ in range(200):  # sum p_a p_b e^(lambda s_ab) = 1: below the root the sum is < 1
        mid = (lo + hi) / 2
        lo, hi = (mid, hi) if (np.outer(p, p) * np.exp(mid * M)).sum() < 1 else (lo, mid)
    exact = lo
    rng = np.random.default_rng(8)
    L = _null_lengths(rng, 1_000_000)
    qs = _null_queries(rng, 6, 200, 1000)
    with _engine(numTop=1, blosumType=62, gop=-4096, gex=-4096) as eng:
        eng.setPseudoDatabaseLengths(L, seed=22)
        eng.setScoreStatistics(True)
        res, _ = eng.scanMany(qs)
    lam = [r.statistics.lambda_ for r in res]
    print(f"gapless: exact ungapped lambda {exact:.4f}, fitted {[round(x, 4) for x in lam]}")
    for x in lam:
        assert abs(x / exact - 1) <= 0.10, (x, exact)


@pytest.mark.gpu
def test_planted_homologs_and_the_cutoff():
    rng = np.random.default_rng(9)
    base = _null_lengths(rng, 1_000_000)
    q = synth._PSEUDO_TABLE[rng.integers(0, 256, 400)]
    copies = [synth.mutate(rng, q, 0.2, indels=0) for _ in range(5)]
    L = np.sort(np.concatenate([base, np.full(len(copies), len(q))])).astype(np.int32)
    first = int(np.searchsorted(L, len(q)))
    planted = {first + 3 * k: c for k, c in enumerate(copies)}
    assert all(L[i] == len(q) for i in planted)
    with _engine(numTop=50, blosumType=62) as eng:
        eng.setPseudoDatabaseLengths(L, seed=23, planted=planted)
        eng.setScoreStatistics(True)
        full = eng.scan(dbformat.decode(q))
        assert sorted(full.referenceIds[:len(copies)]) == sorted(planted)
        assert all(e < 1e-10 for e in full.evalues[:len(copies)]), full.evalues[:8]
        keep = [e <= 1e-3 for e in full.evalues]
        n = sum(keep)
        assert keep == [True] * n + [False] * (len(keep) - n) and n >= len(copies)
        eng.setScoreStatistics(True, 1e-3)
        cut = eng.scan(dbformat.decode(q))
        assert cut.scores == full.scores[:n] and cut.referenceIds == full.referenceIds[:n]
        assert cut.evalues == full.evalues[:n] and cut.statistics == full.statistics
        many, _ = eng.scanMany([dbformat.decode(q)] * 2)
        assert all(m.referenceIds == cut.referenceIds for m in many)


@pytest.mark.gpu
def test_align_evalue_columns(tmp_path):
    _build_cli()
    recs, queries = synth.config_c1(seed=3, n=4000)
    dbformat.write_fasta(str(tmp_path / "db.fa"), recs)
    dbformat.write_fasta(str(tmp_path / "q.fa"), queries[:4])
    subprocess.run([MAKEDB, str(tmp_path / "db.fa"), str(tmp_path / "db")], check=True, stdout=subprocess.DEVNULL)
    common = ["--query", "q.fa", "--db", "db", "--top", "30", "--mat", "blosum62"]
    cwd = str(tmp_path)
    _run_align(ALIGN, common + ["--tsv", "--of", "plain.tsv"], cwd)
    _run_align(ALIGN, common + ["--tsv", "--evalue", "--of", "ev.tsv"], cwd)
    _run_align(ALIGN, common + ["--tsv", "--maxEvalue", "1e-5", "--batchQueries", "4", "--of", "cut.tsv"], cwd)
    _run_align(ALIGN, common + ["--of", "plain.txt"], cwd)
    _run_align(ALIGN, common + ["--evalue", "--cigar", "--of", "ev.txt"], cwd)
    plain = open(tmp_path / "plain.tsv").read().splitlines()
    ev = [line.split("\t") for line in open(tmp_path / "ev.tsv").read().splitlines()]
    assert ev[0][-2:] == ["E-value", "Bit score"] and ["\t".join(r[:-2]) for r in ev] == plain
    with _engine(numTop=30, blosumType=62) as eng:
        eng.setDatabase(str(tmp_path / "db"))
        eng.setScoreStatistics(True)
        stats = [eng.scan(q).statistics for _, q in queries[:4]]
    kept = [ev[0]]
    for r in ev[1:]:
        st, score = stats[int(r[0])], int(r[4])
        assert st.ok and math.isclose(float(r[-2]), st.evalue(score), rel_tol=1e-5)
        assert math.isclose(float(r[-1]), st.bit_score(score), rel_tol=1e-5, abs_tol=1e-4)
        if st.evalue(score) <= 1e-5:
            kept.append(r)
    cut = [line.split("\t") for line in open(tmp_path / "cut.tsv").read().splitlines()]
    assert cut == kept and len(kept) > 4
    txt = open(tmp_path / "ev.txt").read().splitlines()
    plain_txt = open(tmp_path / "plain.txt").read().splitlines()
    assert len(txt) == len(plain_txt)
    for a, b in zip(txt, plain_txt):
        if b.startswith("Result"):
            assert a.startswith(b + " Identities ") and " E-value " in a and a.endswith(".")
        else:
            assert a == b
