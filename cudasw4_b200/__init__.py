"""cudasw4_b200 - B200-native Smith-Waterman protein database search (the scan hot path of CUDASW++4.0).

`CudaSW4` mirrors the reference's host class `cudasw4::CudaSW4` (reference src/cudasw4.cuh:244-2454): same method
names, argument meaning and error behaviour (exceptions instead of std::runtime_error), implemented as a thin ctypes
layer over the C ABI of include/sw4b200.h. All compute happens in libsw4b200.so on the GPU; there is no fallback.
"""
from __future__ import annotations

import ctypes
import enum
import math
from dataclasses import dataclass, field

import numpy as np

from . import _lib, dbformat

__all__ = ["CudaSW4", "ScanResult", "Alignments", "IterativeResult", "BenchmarkStats", "ScoreStatistics", "fit_score_statistics", "KernelType", "KernelTypeConfig", "MemoryConfig", "BlosumType",
           "SW4Error", "dbformat"]


class SW4Error(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"sw4 error {code}: {message}")
        self.code = code


class KernelType(enum.IntEnum):  # reference src/types.hpp:11-16
    Half2 = 0
    DPXs16 = 1
    DPXs32 = 2
    Float = 3


class BlosumType(enum.IntEnum):  # reference src/types.hpp:18-27 (only the 21x21 "_20" tables are live)
    BLOSUM45 = 45
    BLOSUM50 = 50
    BLOSUM62 = 62
    BLOSUM80 = 80
    BLOSUM45_20 = 45
    BLOSUM50_20 = 50
    BLOSUM62_20 = 62
    BLOSUM80_20 = 80


@dataclass
class KernelTypeConfig:  # reference src/cudasw4.cuh:88-93 (defaults of `align --dpx`)
    singlePassType: KernelType = KernelType.DPXs16
    manyPassType_small: KernelType = KernelType.DPXs16
    manyPassType_large: KernelType = KernelType.DPXs32
    overflowType: KernelType = KernelType.DPXs32


@dataclass
class MemoryConfig:  # reference src/cudasw4.cuh:95-100, defaults src/options.hpp:33-37
    maxBatchBytes: int = 128 * 1024 * 1024
    maxBatchSequences: int = 10_000_000
    maxTempBytes: int = 4 * 1024 * 1024 * 1024
    maxGpuMem: int = 2**64 - 1


@dataclass
class BenchmarkStats:  # reference src/cudasw4.cuh:76-80
    numOverflows: int = 0
    seconds: float = 0.0
    gcups: float = 0.0
    kernelSeconds: float = 0.0
    cells: float = 0.0
    kernelLaunches: int = 0


@dataclass
class ScoreStatistics:
    """The fit of a query's score histogram (sw4_score_statistics in include/sw4b200.h). `ok` is False when too few
    subjects could be fitted; lambda_ and K are then NaN."""
    ok: bool
    whole_database: bool
    lambda_: float
    K: float
    query_length: int
    db_residues: int
    num_subjects: int
    fitted: int
    left_censored: int
    right_censored: int
    c_lo: int
    c_hi: int

    def evalue(self, score: int) -> float:
        """E = K m D e^(-lambda S): the expected number of subjects with a score >= S under the fitted model."""
        return self.K * float(self.query_length) * float(self.db_residues) * math.exp(-self.lambda_ * score)

    def bit_score(self, score: int) -> float:
        return (self.lambda_ * score - math.log(self.K)) / math.log(2.0)


@dataclass
class ScanResult:  # reference src/cudasw4.cuh:82-86
    scores: list = field(default_factory=list)
    referenceIds: list = field(default_factory=list)
    stats: BenchmarkStats = field(default_factory=BenchmarkStats)
    # with score statistics enabled (CudaSW4.setScoreStatistics): one E-value and bit score per hit (empty when the
    # fit had too few subjects) and the fit itself; empty / None otherwise
    evalues: list = field(default_factory=list)
    bitScores: list = field(default_factory=list)
    statistics: ScoreStatistics | None = None


@dataclass
class Alignments:
    """What CudaSW4.alignments returns, one row per id: `coordinates` (n, 5) int32 as alignmentCoordinates, `counts`
    (n, 4) int32 (alignment length, identities, positives, gaps) and `cigars` (SAM-style run-length ops =, X, I, D in
    query order, with the query as the read; "" when the score is 0)."""
    coordinates: np.ndarray
    counts: np.ndarray
    cigars: list


@dataclass
class IterativeResult:
    """What CudaSW4.searchIterative returns: the last round's hits (`result`, with E-values, exactly as that round's
    scan reports them), the (m, 21) int8 PSSM that round searched with (`pssm`; after one round the matrix rows), the
    number of rounds and whether they stopped because the included hits repeated (`converged`)."""
    result: ScanResult
    pssm: np.ndarray
    iterations: int
    converged: bool


def _pssm_array(pssm, length: int) -> np.ndarray:
    """A (length, 21) position-specific scoring matrix as a contiguous int8 array (row p: the scores of query position p
    against residue codes 0..19 = ARNDCQEGHILKMFPSTWYV and 20 = any other letter). Refuses a wrong shape, a non-integer
    array, values outside the int8 range and a positive column 20 (code 20 also pads the subjects on the device, see
    include/sw4b200.h) with ValueError; values are never wrapped."""
    a = np.asarray(pssm)
    if a.ndim != 2 or a.shape != (length, 21):
        raise ValueError(f"pssm must have shape ({length}, 21) for a query of {length} residues, got {a.shape}")
    if a.size and not (np.issubdtype(a.dtype, np.integer) or np.issubdtype(a.dtype, np.bool_)):
        raise ValueError(f"pssm must hold integers, got {a.dtype}")
    if a.size and (int(a.min()) < -128 or int(a.max()) > 127):
        raise ValueError(f"pssm values must lie in [-128, 127], got [{int(a.min())}, {int(a.max())}]")
    if a.size and int(a[:, 20].max()) > 0:
        raise ValueError(f"pssm column 20 (any other letter) must be <= 0, got {int(a[:, 20].max())}")
    return np.ascontiguousarray(a, dtype=np.int8)


def _score_statistics(s: _lib.ScoreStatistics) -> ScoreStatistics:
    return ScoreStatistics(int(s.status) == 0, bool(s.whole_database), float(s.lambda_), float(s.K), int(s.query_length),
                           int(s.db_residues), int(s.num_subjects), int(s.fitted), int(s.left_censored),
                           int(s.right_censored), int(s.c_lo), int(s.c_hi))


def fit_score_statistics(counts, lensums, query_length: int) -> ScoreStatistics:
    """The E-value fit of sw4_fit_score_statistics on a histogram of len(counts) - 1 score bins plus the overflow bin
    (for example one summed over the ranks of a sharded search). Host code only: needs no device."""
    c = np.ascontiguousarray(counts, dtype=np.int64)
    L = np.ascontiguousarray(lensums, dtype=np.int64)
    if c.ndim != 1 or c.shape != L.shape or len(c) < 2:
        raise ValueError("counts and lensums must be 1-D arrays of equal length >= 2")
    out = _lib.ScoreStatistics()
    rc = _lib.load().sw4_fit_score_statistics(c.ctypes.data, L.ctypes.data, len(c) - 1, int(query_length), ctypes.byref(out))
    if rc != 0:
        raise ValueError("invalid histogram (negative entries?)")
    return _score_statistics(out)


def _stats(s: _lib.Stats) -> BenchmarkStats:
    return BenchmarkStats(int(s.num_overflows), float(s.seconds), float(s.gcups), float(s.kernel_seconds),
                          float(s.cells), int(s.kernel_launches))


class CudaSW4:
    """Host-side mirror of cudasw4::CudaSW4 (constructor: reference src/cudasw4.cuh:496-531)."""

    def __init__(self, deviceIds=None, numTop: int = 10, blosumType=BlosumType.BLOSUM62,
                 kernelTypeConfig: KernelTypeConfig | None = None, memoryConfig: MemoryConfig | None = None,
                 verbose: bool = False, gop: int | None = None, gex: int | None = None):
        self._lib = _lib.load()
        self._h = ctypes.c_void_p()
        self._keep = None
        ids = list(deviceIds) if deviceIds is not None else []
        arr = (ctypes.c_int * max(1, len(ids)))(*ids)
        mc = memoryConfig or MemoryConfig()
        mem = _lib.MemConfig(mc.maxBatchBytes, mc.maxBatchSequences, mc.maxTempBytes, min(mc.maxGpuMem, 2**64 - 1))
        # the reference constructs with gop=-11, gex=-1 whatever the matrix (src/cudasw4.cuh:2443-2444); callers use
        # setGapOpenScore/setGapExtendScore to change them. gop/gex keyword arguments are a convenience.
        rc = self._lib.sw4_create(arr if ids else None, len(ids), int(numTop), int(blosumType),
                                  -11 if gop is None else int(gop), -1 if gex is None else int(gex),
                                  ctypes.byref(mem), int(verbose), ctypes.byref(self._h))
        if rc != 0:
            raise SW4Error(rc, (self._lib.sw4_last_error(None) or b"").decode())
        self.numTop = int(numTop)
        self._scoreStatistics = False
        self._gop = -11 if gop is None else int(gop)
        self._gex = -1 if gex is None else int(gex)
        if kernelTypeConfig is not None:
            self.setKernelTypeConfig(kernelTypeConfig)

    # -- plumbing ---------------------------------------------------------------------------------------------
    def _check(self, rc: int):
        if rc != 0:
            raise SW4Error(rc, (self._lib.sw4_last_error(self._h) or b"").decode())

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.sw4_destroy(self._h)
            self._h = ctypes.c_void_p()
            self._keep = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- configuration (reference src/cudasw4.cuh:539-611) --------------------------------------------------------
    def setGapOpenScore(self, score: int):
        self.setGapScores(int(score), self._gex)

    def setGapExtendScore(self, score: int):
        self.setGapScores(self._gop, int(score))

    def setGapScores(self, gop: int, gex: int):
        self._check(self._lib.sw4_set_gap_scores(self._h, int(gop), int(gex)))
        self._gop, self._gex = int(gop), int(gex)  # only after the library accepted them

    def setBlosum(self, blosumType):
        self._check(self._lib.sw4_set_blosum(self._h, int(blosumType)))

    def setNumTop(self, value: int):
        self._check(self._lib.sw4_set_num_top(self._h, int(value)))
        self.numTop = int(value)

    def setKernelTypeConfig(self, val: KernelTypeConfig):
        self._check(self._lib.sw4_set_kernel_types(self._h, int(val.singlePassType), int(val.manyPassType_small),
                                                   int(val.manyPassType_large), int(val.overflowType)))

    def setMemoryConfig(self, val: MemoryConfig):
        mem = _lib.MemConfig(val.maxBatchBytes, val.maxBatchSequences, val.maxTempBytes, min(val.maxGpuMem, 2**64 - 1))
        self._check(self._lib.sw4_set_mem_config(self._h, ctypes.byref(mem)))

    def setScoreStatistics(self, enabled: bool = True, maxEvalue: float = math.inf):
        """Report E-values and bit scores: every following scan also builds the query's score histogram on the GPU and
        fits lambda and K to it (include/sw4b200.h). A finite maxEvalue drops the hits with E > maxEvalue, when this
        handle holds the whole database. Off by default."""
        self._check(self._lib.sw4_set_score_statistics(self._h, int(bool(enabled)), float(maxEvalue)))
        self._scoreStatistics = bool(enabled)

    def lastScoreStatistics(self, queryIndex: int = 0) -> ScoreStatistics:
        """The fit of query `queryIndex` of the last scan call (0 after scan())."""
        out = _lib.ScoreStatistics()
        self._check(self._lib.sw4_last_score_statistics(self._h, int(queryIndex), ctypes.byref(out)))
        return _score_statistics(out)

    def lastScoreHistogram(self, queryIndex: int = 0):
        """(counts, lensums): int64 arrays of SCORE_BINS + 1 entries (the last one is the overflow bin) over the
        subjects this handle scanned for query `queryIndex` of the last scan call."""
        counts = np.zeros(_lib.SCORE_BINS + 1, dtype=np.int64)
        lensums = np.zeros(_lib.SCORE_BINS + 1, dtype=np.int64)
        self._check(self._lib.sw4_last_score_histogram(self._h, int(queryIndex), counts.ctypes.data, lensums.ctypes.data,
                                                       _lib.SCORE_BINS))
        return counts, lensums

    def _with_statistics(self, r: ScanResult, queryIndex: int) -> ScanResult:
        if self._scoreStatistics:
            st = self.lastScoreStatistics(queryIndex)
            r.statistics = st
            if st.ok:
                r.evalues = [st.evalue(s) for s in r.scores]
                r.bitScores = [st.bit_score(s) for s in r.scores]
        return r

    def setShard(self, rank: int, world: int):
        """One process per GPU: scan only shard `rank` of `world`; ids stay global (no reference equivalent: the
        reference drives all GPUs from one process, src/cudasw4.cuh:928-1004)."""
        self._check(self._lib.sw4_set_shard(self._h, int(rank), int(world)))

    # -- database (reference src/cudasw4.cuh:552-568, 651-696) ----------------------------------------------------
    def setDatabase(self, db):
        """db: path prefix written by makedb (str), or a dbformat.SequenceDB held in host memory."""
        if isinstance(db, (str, bytes)):
            prefix = db.encode() if isinstance(db, str) else db
            self._check(self._lib.sw4_set_database_files(self._h, prefix, 1))
            self._keep = None
            return
        chars = np.ascontiguousarray(db.chars, dtype=np.uint8)
        offsets = np.ascontiguousarray(db.offsets, dtype=np.uint64)
        lengths = np.ascontiguousarray(db.lengths, dtype=np.int32)
        headers = np.ascontiguousarray(db.headers, dtype=np.uint8)
        hoff = np.ascontiguousarray(db.header_offsets, dtype=np.uint64)
        self._keep = (chars, offsets, lengths, headers, hoff)  # borrowed by the library
        self._check(self._lib.sw4_set_database_memory(self._h, chars.ctypes.data, offsets.ctypes.data,
                                                      lengths.ctypes.data, headers.ctypes.data, hoff.ctypes.data,
                                                      len(lengths)))

    def setDatabaseShard(self, db, globalIds, numSequencesGlobal: int):
        """One process per GPU, every rank holding only its own shard in host memory: `db` (dbformat.SequenceDB,
        ascending length) are the local sequences, `globalIds` their (strictly ascending) ids in the whole database."""
        chars = np.ascontiguousarray(db.chars, dtype=np.uint8)
        offsets = np.ascontiguousarray(db.offsets, dtype=np.uint64)
        lengths = np.ascontiguousarray(db.lengths, dtype=np.int32)
        gids = np.ascontiguousarray(globalIds, dtype=np.int32)
        if len(gids) != len(lengths):
            raise ValueError("one global id per local sequence")
        self._keep = (chars, offsets, lengths, gids)
        self._check(self._lib.sw4_set_database_shard_memory(self._h, chars.ctypes.data, offsets.ctypes.data, lengths.ctypes.data,
                                                            None, None, len(lengths), gids.ctypes.data, int(numSequencesGlobal)))

    def setPseudoDatabase(self, num: int, length: int, seed: int = 42):
        """loadPseudoDB(num, length) + setDatabase (reference src/dbdata.hpp:219-272, src/main.cu:193-203)."""
        self._check(self._lib.sw4_set_pseudo_database(self._h, int(num), int(length), int(seed)))
        self._keep = None

    def setPseudoDatabaseLengths(self, lengths, seed: int, planted: dict | None = None):
        """Synthetic database with the given (ascending) length array; this handle generates its own shard only
        (setShard). `planted` maps a global id to the residue codes that replace that sequence (same length)."""
        L = np.ascontiguousarray(lengths, dtype=np.int32)
        planted = planted or {}
        ids = np.array(sorted(planted), dtype=np.int32)
        codes = [np.ascontiguousarray(planted[int(i)], dtype=np.uint8) for i in ids]
        for i, c in zip(ids, codes):
            if len(c) != int(L[i]):
                raise ValueError(f"planted sequence {i} has length {len(c)}, slot has {int(L[i])}")
        ptrs = (ctypes.c_void_p * max(1, len(codes)))(*[c.ctypes.data for c in codes])
        self._check(self._lib.sw4_set_pseudo_database_lengths(self._h, L.ctypes.data, len(L), int(seed) & (2**64 - 1),
                                                              ids.ctypes.data if len(ids) else None, ptrs, len(codes)))
        self._keep = None

    def prefetchDBToGpus(self):
        self._check(self._lib.sw4_upload_database(self._h))

    # -- the hot path (reference src/cudasw4.cuh:698-765) ---------------------------------------------------------
    def scan(self, query, length: int | None = None, pssm=None) -> ScanResult:
        """query: residue letters (str/bytes). Returns the top-`numTop` (score, reference id) pairs.
        pssm: a (length, 21) integer array scoring each query position against each residue code instead of the
        handle's matrix (include/sw4b200.h); the letters then only serve the identities of alignments()."""
        q = query.encode() if isinstance(query, str) else bytes(query)
        n = len(q) if length is None else int(length)
        k = max(self.numTop, 1)
        scores = np.empty(k, dtype=np.int32)
        ids = np.empty(k, dtype=np.int32)
        count = ctypes.c_int32(0)
        st = _lib.Stats()
        if pssm is None:
            self._check(self._lib.sw4_scan(self._h, q, n, scores.ctypes.data, ids.ctypes.data, ctypes.byref(count),
                                           ctypes.byref(st)))
        else:
            p = _pssm_array(pssm, n)
            self._check(self._lib.sw4_scan_pssm(self._h, q, p.ctypes.data, n, scores.ctypes.data, ids.ctypes.data,
                                                ctypes.byref(count), ctypes.byref(st)))
        c = int(count.value)
        return self._with_statistics(ScanResult(scores[:c].tolist(), ids[:c].tolist(), _stats(st)), 0)

    def scanMany(self, queries, pssm=None):
        """Query batching (sw4_scan_many): all `queries` (letters) with several scans in flight per GPU. Returns
        (list of ScanResult in query order, BenchmarkStats of the whole call: device-timed span, total GCUPS).
        pssm: a list of (len(query), 21) arrays, one per query (as scan's pssm)."""
        qs = [q.encode() if isinstance(q, str) else bytes(q) for q in queries]
        nq = len(qs)
        if pssm is not None:
            if len(pssm) != nq:
                raise ValueError(f"one pssm per query: {len(pssm)} for {nq} queries")
            ps = [_pssm_array(p, len(q)) for p, q in zip(pssm, qs)]
        k = max(self.numTop, 1)
        arr = (ctypes.c_char_p * max(nq, 1))(*qs)
        lens = (ctypes.c_int32 * max(nq, 1))(*[len(q) for q in qs])
        scores = np.empty((max(nq, 1), k), dtype=np.int32)
        ids = np.empty((max(nq, 1), k), dtype=np.int32)
        counts = np.zeros(max(nq, 1), dtype=np.int32)
        per = (_lib.Stats * max(nq, 1))()
        total = _lib.Stats()
        if pssm is None:
            self._check(self._lib.sw4_scan_many(self._h, arr, lens, nq, scores.ctypes.data, ids.ctypes.data,
                                                counts.ctypes.data, per, ctypes.byref(total)))
        else:
            parr = (ctypes.c_void_p * max(nq, 1))(*[p.ctypes.data for p in ps])
            self._check(self._lib.sw4_scan_many_pssm(self._h, arr, parr, lens, nq, scores.ctypes.data, ids.ctypes.data,
                                                     counts.ctypes.data, per, ctypes.byref(total)))
        out = []
        for i in range(nq):
            c = int(counts[i]) if self.numTop > 0 else 0
            out.append(self._with_statistics(ScanResult(scores[i, :c].tolist(), ids[i, :c].tolist(), _stats(per[i])), i))
        return out, _stats(total)

    def alignmentCoordinates(self, query, ids, stats: BenchmarkStats | None = None, pssm=None) -> np.ndarray:
        """Where each hit aligns: for every database id in `ids`, one row (score, query_begin, query_end,
        reference_begin, reference_end) of an int32 array of shape (len(ids), 5). Positions are 0-based and inclusive,
        -1 when the score is 0; the end is the first cell holding the maximum, the begin that of the shortest optimal
        alignment ending there (include/sw4b200.h). `stats`, when given, receives the call's device-timed figures.
        pssm: a (len(query), 21) array, as scan's."""
        q = query.encode() if isinstance(query, str) else bytes(query)
        idv = np.ascontiguousarray(np.asarray(ids, dtype=np.int64).reshape(-1))
        if len(idv) and (idv.min() < -2**31 or idv.max() >= 2**31):
            raise SW4Error(-1, "database id out of range")
        idv = idv.astype(np.int32)
        out = np.empty((max(len(idv), 1), 5), dtype=np.int32)
        st = _lib.Stats()
        if pssm is None:
            self._check(self._lib.sw4_alignment_coordinates(self._h, q, len(q), idv.ctypes.data, len(idv), out.ctypes.data,
                                                            ctypes.byref(st)))
        else:
            p = _pssm_array(pssm, len(q))
            self._check(self._lib.sw4_alignment_coordinates_pssm(self._h, q, p.ctypes.data, len(q), idv.ctypes.data, len(idv),
                                                                 out.ctypes.data, ctypes.byref(st)))
        if stats is not None:
            for k, v in vars(_stats(st)).items():
                setattr(stats, k, v)
        return out[:len(idv)].copy()

    def alignments(self, query, ids, stats: BenchmarkStats | None = None, pssm=None) -> Alignments:
        """How each hit aligns: the coordinates of alignmentCoordinates, and the CIGAR and counts of the one alignment
        they locate, traced back on the GPU (the rule is in include/sw4b200.h). `stats`, when given, receives the
        call's device-timed figures (cells and kernel launches of all three passes). pssm: a (len(query), 21) array, as
        scan's; positives are then the pairs it scores above 0."""
        q = query.encode() if isinstance(query, str) else bytes(query)
        idv = np.ascontiguousarray(np.asarray(ids, dtype=np.int64).reshape(-1))
        if len(idv) and (idv.min() < -2**31 or idv.max() >= 2**31):
            raise SW4Error(-1, "database id out of range")
        idv = idv.astype(np.int32)
        n = len(idv)
        out = (_lib.AlignmentSummary * max(n, 1))()
        st = _lib.Stats()
        if pssm is None:
            self._check(self._lib.sw4_alignment_traceback(self._h, q, len(q), idv.ctypes.data, n, out, ctypes.byref(st)))
        else:
            p = _pssm_array(pssm, len(q))
            self._check(self._lib.sw4_alignment_traceback_pssm(self._h, q, p.ctypes.data, len(q), idv.ctypes.data, n, out,
                                                               ctypes.byref(st)))
        p = ctypes.c_void_p()
        size = ctypes.c_size_t(0)
        self._check(self._lib.sw4_last_cigars(self._h, ctypes.byref(p), ctypes.byref(size)))
        text = ctypes.string_at(p.value, size.value).decode() if size.value else ""
        raw = np.frombuffer(out, dtype=np.dtype([("coordinates", "<i4", 5), ("counts", "<i4", 4),
                                                 ("offset", "<u8"), ("length", "<u8")], align=True))[:n]
        if stats is not None:
            for k, v in vars(_stats(st)).items():
                setattr(stats, k, v)
        cigars = [text[int(o):int(o) + int(L)] for o, L in zip(raw["offset"], raw["length"])]
        return Alignments(raw["coordinates"].copy(), raw["counts"].copy(), cigars)

    def buildPssm(self, query, ids, pssm=None, pseudocountWeight: float = 10.0, stats: BenchmarkStats | None = None) -> np.ndarray:
        """The profile of the query and the hits `ids`, built on the GPU (sw4_build_pssm, include/sw4b200.h): the
        alignments of alignments() for that query form, a query-anchored MSA, Henikoff position-based weights and
        pseudocounts of weight `pseudocountWeight`. Returns an (m, 21) int8 array that scan(pssm=...) takes. `ids` may
        be empty (then the rows are the matrix rows of the query's residues); pssm: the query form to align with."""
        q = query.encode() if isinstance(query, str) else bytes(query)
        idv = np.ascontiguousarray(np.asarray(ids, dtype=np.int64).reshape(-1))
        if len(idv) and (idv.min() < -2**31 or idv.max() >= 2**31):
            raise SW4Error(-1, "database id out of range")
        idv = idv.astype(np.int32)
        out = np.zeros((max(len(q), 1), 21), dtype=np.int8)
        p = None if pssm is None else _pssm_array(pssm, len(q))
        st = _lib.Stats()
        self._check(self._lib.sw4_build_pssm(self._h, q, None if p is None else p.ctypes.data, len(q), idv.ctypes.data, len(idv),
                                             float(pseudocountWeight), out.ctypes.data, ctypes.byref(st)))
        if stats is not None:
            for k, v in vars(_stats(st)).items():
                setattr(stats, k, v)
        return out[:len(q)].copy()

    def searchIterative(self, query, iterations: int = 3, inclusionEvalue: float = 0.002,
                        pseudocountWeight: float = 10.0) -> IterativeResult:
        """Iterative profile search (sw4_search_iterative): scan, take the hits with E <= inclusionEvalue (before the
        handle's maxEvalue cutoff), build their profile with buildPssm and scan again with it, for at most `iterations`
        rounds or until no hit is included or the included set repeats. Needs setScoreStatistics(True) and a handle
        that scans the whole database."""
        q = query.encode() if isinstance(query, str) else bytes(query)
        k = max(self.numTop, 1)
        scores = np.empty(k, dtype=np.int32)
        ids = np.empty(k, dtype=np.int32)
        pssm = np.zeros((max(len(q), 1), 21), dtype=np.int8)
        count, rounds, converged = ctypes.c_int32(0), ctypes.c_int32(0), ctypes.c_int32(0)
        st = _lib.Stats()
        self._check(self._lib.sw4_search_iterative(self._h, q, len(q), int(iterations), float(inclusionEvalue),
                                                   float(pseudocountWeight), scores.ctypes.data, ids.ctypes.data,
                                                   ctypes.byref(count), pssm.ctypes.data, ctypes.byref(rounds),
                                                   ctypes.byref(converged), ctypes.byref(st)))
        c = int(count.value)
        r = self._with_statistics(ScanResult(scores[:c].tolist(), ids[:c].tolist(), _stats(st)), 0)
        return IterativeResult(r, pssm[:len(q)].copy(), int(rounds.value), bool(converged.value))

    def lastScanAllScores(self):
        """(scores, global ids) of every subject this handle scanned in the last scan() (parity helper)."""
        info = self.dbInfo()
        n = int(info.shard_sequences)
        scores = np.empty(max(n, 1), dtype=np.int32)
        ids = np.empty(max(n, 1), dtype=np.int32)
        got = ctypes.c_size_t(0)
        self._check(self._lib.sw4_last_scan_all_scores(self._h, scores.ctypes.data, ids.ctypes.data, n, ctypes.byref(got)))
        return scores[:got.value], ids[:got.value]

    # -- accessors (reference src/cudasw4.cuh:613-639, 799-839) -----------------------------------------------------
    def getReferenceHeader(self, referenceId: int) -> str:
        p = ctypes.c_void_p()
        n = ctypes.c_size_t(0)
        self._check(self._lib.sw4_reference_header(self._h, int(referenceId), ctypes.byref(p), ctypes.byref(n)))
        return ctypes.string_at(p.value, n.value).decode(errors="replace") if n.value else ""

    def getReferenceLength(self, referenceId: int) -> int:
        v = ctypes.c_int32(0)
        self._check(self._lib.sw4_reference_length(self._h, int(referenceId), ctypes.byref(v)))
        return int(v.value)

    def getReferenceSequence(self, referenceId: int) -> str:
        L = self.getReferenceLength(referenceId)
        buf = ctypes.create_string_buffer(L + 1)
        n = ctypes.c_size_t(0)
        self._check(self._lib.sw4_reference_sequence(self._h, int(referenceId), buf, L, ctypes.byref(n)))
        return buf.raw[:n.value].decode()

    def totalTimerStart(self):
        self._check(self._lib.sw4_total_timer_start(self._h))

    def totalTimerStop(self) -> BenchmarkStats:
        st = _lib.Stats()
        self._check(self._lib.sw4_total_timer_stop(self._h, ctypes.byref(st)))
        return _stats(st)

    def dbInfo(self) -> _lib.DbInfo:
        info = _lib.DbInfo()
        self._check(self._lib.sw4_get_db_info(self._h, ctypes.byref(info)))
        return info

    def printDBInfo(self):
        i = self.dbInfo()
        print(f"{i.num_sequences} sequences, {i.num_residues} characters")

    def printDBLengthPartitions(self):
        i = self.dbInfo()
        for b, c in zip(dbformat.BOUNDARIES.tolist(), list(i.partition_counts)):
            print(f"<= {b}: {c}")
