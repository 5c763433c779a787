// cudasw4.cuh - source-compatible C++ facade of the reference's host class cudasw4::CudaSW4
// (reference src/cudasw4.cuh:244-2454, types src/types.hpp:11-27, src/config.hpp:12-15) on top of the C ABI of
// sw4b200.h. A caller written against the reference (its src/main.cu) compiles against this header unchanged for the
// scan path: same namespace, type names, member names, argument meaning and exceptions (std::runtime_error).
// Pure host C++17: no CUDA headers needed; link with -lsw4b200.
//
// Differences, all deliberate (SURVEY.md 0 / 9):
//   * setGapOpenScore/setGapExtendScore work (the shipped align never calls them; our CLI does).
//   * a database that fits MemoryConfig::maxGpuMem is resident on the GPUs (--uploadFull); a larger one is streamed in
//     batches on every scan with all scores kept (the reference's streaming mode loses scores, SURVEY.md 0-2).
//   * result order is (score desc, id asc) for any database size / GPU count (the reference's order above 1e6
//     subjects is a thrust artefact, SURVEY.md 0-3); length-0 subjects score 0 instead of -1.
#ifndef CUDASW4_B200_FACADE_CUH
#define CUDASW4_B200_FACADE_CUH

#include <cmath>
#include <cstdint>
#include <iostream>
#include <limits>
#include <memory>
#include <stdexcept>
#include <string>
#include <string_view>
#include <vector>

#include "sw4b200.h"

namespace cudasw4 {

using ReferenceIdT = std::int32_t;      // src/config.hpp:12
using SequenceLengthT = std::int32_t;   // src/config.hpp:15

enum class KernelType { Half2, DPXs16, DPXs32, Float };  // src/types.hpp:11-16
enum class BlosumType { BLOSUM45, BLOSUM50, BLOSUM62, BLOSUM80, BLOSUM45_20, BLOSUM50_20, BLOSUM62_20, BLOSUM80_20 };

inline std::string to_string(KernelType t) {
    switch (t) { case KernelType::Half2: return "Half2"; case KernelType::DPXs16: return "DPXs16";
                 case KernelType::DPXs32: return "DPXs32"; case KernelType::Float: return "Float"; }
    return "Unnamed kernel type";
}
inline std::string to_string_nodim(BlosumType t) {
    switch (t) { case BlosumType::BLOSUM45: case BlosumType::BLOSUM45_20: return "BLOSUM45";
                 case BlosumType::BLOSUM50: case BlosumType::BLOSUM50_20: return "BLOSUM50";
                 case BlosumType::BLOSUM62: case BlosumType::BLOSUM62_20: return "BLOSUM62";
                 case BlosumType::BLOSUM80: case BlosumType::BLOSUM80_20: return "BLOSUM80"; }
    return "Unnamed blosum type";
}
inline int blosumNumber(BlosumType t) {
    switch (t) { case BlosumType::BLOSUM45: case BlosumType::BLOSUM45_20: return 45;
                 case BlosumType::BLOSUM50: case BlosumType::BLOSUM50_20: return 50;
                 case BlosumType::BLOSUM62: case BlosumType::BLOSUM62_20: return 62;
                 default: return 80; }
}

struct BenchmarkStats { int numOverflows{}; double seconds{}; double gcups{}; };                       // :76-80
struct ScanResult { std::vector<int> scores{}; std::vector<ReferenceIdT> referenceIds{}; BenchmarkStats stats{}; };
// Extension (no reference counterpart): where a hit aligns, 0-based inclusive, -1 when score == 0 (sw4b200.h)
struct AlignmentCoordinates { int score, queryBegin, queryEnd, referenceBegin, referenceEnd; };
// Extension: how a hit aligns (sw4b200.h): its coordinates, counts and SAM-style CIGAR (=, X, I, D; "" when score == 0)
struct Alignment { AlignmentCoordinates coordinates; int length, identities, positives, gaps; std::string cigar; };
// Extension: the score statistics of one query's search (sw4_score_statistics in sw4b200.h); ok == false: too few
// subjects to fit, lambda and K are NaN
struct ScoreStatistics {
    bool ok, wholeDatabase;
    double lambda, K;
    std::int64_t queryLength, dbResidues, numSubjects, fitted, leftCensored, rightCensored;
    int cLo, cHi;
    // E = K m D e^(-lambda S) and the bit score (lambda S - ln K) / ln 2 of a hit with score S
    double evalue(int score) const { return K * (double)queryLength * (double)dbResidues * std::exp(-lambda * score); }
    double bitScore(int score) const { return (lambda * score - std::log(K)) / std::log(2.0); }
};
// Extension: what searchIterative returns (sw4_search_iterative in sw4b200.h): the last round's hits, the [length][21]
// PSSM that round searched with, the number of rounds and whether they converged
struct IterativeSearchResult { ScanResult result; std::vector<std::int8_t> pssm; int iterations; bool converged; };
struct KernelTypeConfig {                                                                             // :88-93
    KernelType singlePassType = KernelType::Half2;
    KernelType manyPassType_small = KernelType::Half2;
    KernelType manyPassType_large = KernelType::Float;
    KernelType overflowType = KernelType::Float;
};
struct MemoryConfig {                                                                                 // :95-100
    size_t maxBatchBytes = 128ull * 1024ull * 1024ull;
    size_t maxBatchSequences = 10'000'000;
    size_t maxTempBytes = 4ull * 1024ull * 1024ull * 1024ull;
    size_t maxGpuMem = std::numeric_limits<size_t>::max();
};

// Stand-ins for the reference's database holders (src/dbdata.hpp): they only carry what setDatabase needs.
struct LoadDBException : public std::runtime_error { using std::runtime_error::runtime_error; };
struct DB { std::string prefix; bool prefetchSeq = false; };
struct DBWithVectors { std::string prefix; };
struct PseudoDB { size_t num = 0; SequenceLengthT length = 0; int randomseed = 42; };
inline DB loadDB(const std::string& prefix, bool /*writeAccess*/, bool prefetchSeq) { return DB{prefix, prefetchSeq}; }
inline DBWithVectors loadDBWithVectors(const std::string& prefix) { return DBWithVectors{prefix}; }
inline PseudoDB loadPseudoDB(size_t num, SequenceLengthT length, int randomseed = 42) { return PseudoDB{num, length, randomseed}; }

class CudaSW4 {
public:
    CudaSW4(std::vector<int> deviceIds_, int numTop_, BlosumType blosumType, const KernelTypeConfig& kernelTypeConfig,
            const MemoryConfig& memoryConfig, bool verbose_) : numTop(numTop_), verbose(verbose_) {                    // :496-531
        sw4_mem_config mem{memoryConfig.maxBatchBytes, memoryConfig.maxBatchSequences, memoryConfig.maxTempBytes,
                           memoryConfig.maxGpuMem};
        const int rc = sw4_create(deviceIds_.data(), (int)deviceIds_.size(), numTop_, blosumNumber(blosumType), gop, gex,
                                  &mem, verbose_ ? 1 : 0, &handle);
        if (rc != SW4_OK) throw std::runtime_error(sw4_last_error(nullptr));
        setKernelTypeConfig(kernelTypeConfig);
    }
    CudaSW4() = delete;
    CudaSW4(const CudaSW4&) = delete;
    CudaSW4(CudaSW4&& o) noexcept : handle(o.handle), numTop(o.numTop), gop(o.gop), gex(o.gex), verbose(o.verbose) { o.handle = nullptr; }
    CudaSW4& operator=(const CudaSW4&) = delete;
    CudaSW4& operator=(CudaSW4&& o) noexcept { std::swap(handle, o.handle); numTop = o.numTop; gop = o.gop; gex = o.gex; return *this; }
    ~CudaSW4() { if (handle) sw4_destroy(handle); }

    void setGapOpenScore(int score) {                                                                 // :539-544
        if (verbose && score >= 0) std::cout << "Warning, gap open score set to non-negative value. Is this intended?\n";
        gop = score; check(sw4_set_gap_scores(handle, gop, gex));
    }
    void setGapExtendScore(int score) {                                                               // :545-550
        if (verbose && score >= 0) std::cout << "Warning, gap extend score set to non-negative value. Is this intended?\n";
        gex = score; check(sw4_set_gap_scores(handle, gop, gex));
    }
    void setDatabase(std::shared_ptr<DB> db) {                                                        // :552-556
        if (sw4_set_database_files(handle, db->prefix.c_str(), db->prefetchSeq ? 1 : 0) != SW4_OK)
            throw LoadDBException(sw4_last_error(handle));
    }
    void setDatabase(std::shared_ptr<DBWithVectors> db) {                                             // :558-562
        if (sw4_set_database_files(handle, db->prefix.c_str(), 1) != SW4_OK) throw LoadDBException(sw4_last_error(handle));
    }
    void setDatabase(std::shared_ptr<PseudoDB> db) {                                                  // :564-568
        check(sw4_set_pseudo_database(handle, db->num, db->length, db->randomseed));
    }
    void setBlosum(BlosumType blosumType) { check(sw4_set_blosum(handle, blosumNumber(blosumType))); } // :570
    void setNumTop(int value) { if (value >= 0) { check(sw4_set_num_top(handle, value)); numTop = value; } }              // :574
    void setKernelTypeConfig(const KernelTypeConfig& val) {                                           // :589-607
        check(sw4_set_kernel_types(handle, (int)val.singlePassType, (int)val.manyPassType_small, (int)val.manyPassType_large,
                                   (int)val.overflowType));
    }
    void setMemoryConfig(const MemoryConfig& val) {                                                   // :609-611
        sw4_mem_config mem{val.maxBatchBytes, val.maxBatchSequences, val.maxTempBytes, val.maxGpuMem};
        check(sw4_set_mem_config(handle, &mem));
    }

    std::string_view getReferenceHeader(ReferenceIdT referenceId) const {                             // :613
        const char* p = nullptr; size_t n = 0;
        check(sw4_reference_header(handle, referenceId, &p, &n));
        return std::string_view(p, n);
    }
    int getReferenceLength(ReferenceIdT referenceId) const {                                          // :620
        int32_t len = 0; check(sw4_reference_length(handle, referenceId, &len)); return len;
    }
    std::string getReferenceSequence(ReferenceIdT referenceId) const {                                // :625
        std::string s((size_t)getReferenceLength(referenceId), '\0');
        size_t n = 0; check(sw4_reference_sequence(handle, referenceId, s.data(), s.size(), &n)); return s;
    }
    void prefetchDBToGpus() { check(sw4_upload_database(handle)); }                                   // :651

    ScanResult scan(const char* query, SequenceLengthT queryLength) {                                 // :698-765
        return scanImpl(query, nullptr, false, queryLength);
    }

    // Extension (SURVEY.md 8-f4; no reference counterpart: its align scans one query at a time, src/main.cu:228-255):
    // all queries with several scans in flight per GPU. Results equal one scan() per query, in query order.
    std::vector<ScanResult> scanMany(const std::vector<std::string_view>& queries, BenchmarkStats* total = nullptr) {
        return scanManyImpl(queries, nullptr, false, total);
    }
    // Extension (sw4b200.h): the same scans with position-specific scoring matrices. pssm is [length][21], row p
    // scoring query position p against residue codes 0..20; query holds the residue letters.
    ScanResult scan(const char* query, const std::int8_t* pssm, SequenceLengthT queryLength) {
        return scanImpl(query, pssm, true, queryLength);
    }
    // pssms[i] ([queries[i].size()][21]) belongs to queries[i]
    std::vector<ScanResult> scanMany(const std::vector<std::string_view>& queries, const std::vector<const std::int8_t*>& pssms,
                                     BenchmarkStats* total = nullptr) {
        if (pssms.size() != queries.size()) throw std::runtime_error("scanMany: one PSSM per query");
        return scanManyImpl(queries, pssms.data(), true, total);
    }

    // Extension: score, begin and end of one optimal local alignment of the query against each database id.
    std::vector<AlignmentCoordinates> computeAlignmentCoordinates(const char* query, SequenceLengthT length,
                                                                  const std::vector<ReferenceIdT>& ids) {
        return coordinatesImpl(query, nullptr, false, length, ids);
    }
    std::vector<AlignmentCoordinates> computeAlignmentCoordinates(const char* query, const std::int8_t* pssm, SequenceLengthT length,
                                                                  const std::vector<ReferenceIdT>& ids) {
        return coordinatesImpl(query, pssm, true, length, ids);
    }

    // Extension: coordinates, CIGAR and counts of one optimal local alignment of the query against each database id.
    std::vector<Alignment> computeAlignments(const char* query, SequenceLengthT length, const std::vector<ReferenceIdT>& ids) {
        return alignmentsImpl(query, nullptr, false, length, ids);
    }
    std::vector<Alignment> computeAlignments(const char* query, const std::int8_t* pssm, SequenceLengthT length,
                                             const std::vector<ReferenceIdT>& ids) {
        return alignmentsImpl(query, pssm, true, length, ids);
    }

    // Extension (sw4b200.h): E-values. enabled: every following scan also fits its score statistics; a finite maxEvalue
    // drops the hits with E > maxEvalue when the handle holds the whole database.
    void setScoreStatistics(bool enabled, double maxEvalue = INFINITY) { check(sw4_set_score_statistics(handle, enabled ? 1 : 0, maxEvalue)); }
    // the statistics of query queryIndex of the last scan() / scanMany() call
    ScoreStatistics lastScoreStatistics(int queryIndex = 0) const {
        sw4_score_statistics s{};
        check(sw4_last_score_statistics(handle, queryIndex, &s));
        return ScoreStatistics{s.status == SW4_STATS_OK, s.whole_database != 0, s.lambda, s.K, s.query_length, s.db_residues,
                               s.num_subjects, s.fitted, s.left_censored, s.right_censored, s.c_lo, s.c_hi};
    }
    // its histogram over this handle's subjects: SW4_SCORE_BINS + 1 entries each (the last is the overflow bin)
    void lastScoreHistogram(int queryIndex, std::vector<std::int64_t>& counts, std::vector<std::int64_t>& lensums) const {
        counts.assign(SW4_SCORE_BINS + 1, 0);
        lensums.assign(SW4_SCORE_BINS + 1, 0);
        check(sw4_last_score_histogram(handle, queryIndex, counts.data(), lensums.data(), SW4_SCORE_BINS));
    }

    // Extension (sw4b200.h): the [length][21] profile of the query and the hits `ids`, aligned with the sequence or
    // with a PSSM query form; pseudocountWeight is beta
    std::vector<std::int8_t> buildPssm(const char* query, SequenceLengthT length, const std::vector<ReferenceIdT>& ids,
                                       double pseudocountWeight = 10.0) {
        return buildPssmImpl(query, nullptr, length, ids, pseudocountWeight);
    }
    std::vector<std::int8_t> buildPssm(const char* query, const std::int8_t* pssm, SequenceLengthT length,
                                       const std::vector<ReferenceIdT>& ids, double pseudocountWeight = 10.0) {
        return buildPssmImpl(query, pssm, length, ids, pseudocountWeight);
    }
    // Extension: rounds of scan -> hits with E <= inclusionEvalue -> buildPssm -> scan (needs setScoreStatistics(true))
    IterativeSearchResult searchIterative(const char* query, SequenceLengthT length, int maxIterations = 3,
                                          double inclusionEvalue = 0.002, double pseudocountWeight = 10.0) {
        sw4_db_info info{};
        check(sw4_get_db_info(handle, &info));
        const size_t cap = (size_t)std::max<uint64_t>(1, std::min<uint64_t>(info.num_sequences, (uint64_t)std::max(numTop, 0)));
        std::vector<int32_t> scores(cap), ids(cap);
        IterativeSearchResult r{};
        r.pssm.assign((size_t)std::max(length, 1) * 21, 0);
        int32_t count = 0, iterations = 0, converged = 0;
        sw4_stats st{};
        check(sw4_search_iterative(handle, query, length, maxIterations, inclusionEvalue, pseudocountWeight, scores.data(), ids.data(),
                                   &count, r.pssm.data(), &iterations, &converged, &st));
        r.pssm.resize((size_t)std::max(length, 0) * 21);
        r.result.scores.assign(scores.begin(), scores.begin() + count);
        r.result.referenceIds.assign(ids.begin(), ids.begin() + count);
        r.result.stats = BenchmarkStats{st.num_overflows, st.seconds, st.gcups};
        r.iterations = iterations;
        r.converged = converged != 0;
        return r;
    }

    void printDBInfo() const {                                                                      // :799-807
        sw4_db_info info{}; check(sw4_get_db_info(handle, &info));
        std::cout << info.num_sequences << " sequences, " << info.num_residues << " characters\n";
    }
    void printDBLengthPartitions() const {                                                            // :809-816
        static const int b[36] = {48, 64, 80, 96, 112, 128, 144, 160, 176, 192, 208, 224, 240, 256, 288, 320, 352, 384, 416,
                                  448, 480, 512, 576, 640, 704, 768, 832, 896, 960, 1024, 1088, 1152, 1216, 1280, 8000, 2147483646};
        sw4_db_info info{}; check(sw4_get_db_info(handle, &info));
        for (int i = 0; i < 36; i++) std::cout << "<= " << b[i] << ": " << info.partition_counts[i] << "\n";
    }
    void totalTimerStart() { check(sw4_total_timer_start(handle)); }                                  // :818
    BenchmarkStats totalTimerStop() {                                                                 // :826
        sw4_stats st{}; check(sw4_total_timer_stop(handle, &st));
        return BenchmarkStats{st.num_overflows, st.seconds, st.gcups};
    }
    bool isValidSinglePassType(KernelType) const { return true; }                                     // :841-855
    bool isValidMultiPassType_small(KernelType) const { return true; }
    bool isValidMultiPassType_large(KernelType t) const { return t == KernelType::Float || t == KernelType::DPXs32; }
    bool isValidOverflowType(KernelType t) const { return t == KernelType::Float || t == KernelType::DPXs32; }

    sw4_handle* nativeHandle() const { return handle; }

private:
    // (pssmForm: the query comes with pssm, [length][21]; otherwise it is scored with the handle's matrix)
    ScanResult scanImpl(const char* query, const std::int8_t* pssm, bool pssmForm, SequenceLengthT queryLength) {
        sw4_db_info info{};
        check(sw4_get_db_info(handle, &info));
        ScanResult result;
        const size_t cap = (size_t)std::max<uint64_t>(1, std::min<uint64_t>(info.num_sequences, (uint64_t)std::max(numTop, 0)));
        std::vector<int32_t> scores(cap), ids(cap);
        int32_t count = 0; sw4_stats st{};
        check(pssmForm ? sw4_scan_pssm(handle, query, pssm, queryLength, scores.data(), ids.data(), &count, &st)
                       : sw4_scan(handle, query, queryLength, scores.data(), ids.data(), &count, &st));
        result.scores.assign(scores.begin(), scores.begin() + count);
        result.referenceIds.assign(ids.begin(), ids.begin() + count);
        result.stats.numOverflows = st.num_overflows; result.stats.seconds = st.seconds; result.stats.gcups = st.gcups;
        return result;
    }
    std::vector<AlignmentCoordinates> coordinatesImpl(const char* query, const std::int8_t* pssm, bool pssmForm, SequenceLengthT length,
                                                      const std::vector<ReferenceIdT>& ids) {
        std::vector<sw4_alignment> raw(std::max<size_t>(1, ids.size()));
        check(pssmForm ? sw4_alignment_coordinates_pssm(handle, query, pssm, length, ids.data(), (int32_t)ids.size(), raw.data(), nullptr)
                   : sw4_alignment_coordinates(handle, query, length, ids.data(), (int32_t)ids.size(), raw.data(), nullptr));
        std::vector<AlignmentCoordinates> out(ids.size());
        for (size_t i = 0; i < ids.size(); i++)
            out[i] = AlignmentCoordinates{raw[i].score, raw[i].query_begin, raw[i].query_end, raw[i].reference_begin, raw[i].reference_end};
        return out;
    }
    std::vector<Alignment> alignmentsImpl(const char* query, const std::int8_t* pssm, bool pssmForm, SequenceLengthT length,
                                          const std::vector<ReferenceIdT>& ids) {
        std::vector<sw4_alignment_summary> raw(std::max<size_t>(1, ids.size()));
        check(pssmForm ? sw4_alignment_traceback_pssm(handle, query, pssm, length, ids.data(), (int32_t)ids.size(), raw.data(), nullptr)
                   : sw4_alignment_traceback(handle, query, length, ids.data(), (int32_t)ids.size(), raw.data(), nullptr));
        const char* text = nullptr; size_t textLength = 0;
        check(sw4_last_cigars(handle, &text, &textLength));
        std::vector<Alignment> out(ids.size());
        for (size_t i = 0; i < ids.size(); i++) {
            const sw4_alignment& c = raw[i].coordinates;
            out[i] = Alignment{AlignmentCoordinates{c.score, c.query_begin, c.query_end, c.reference_begin, c.reference_end},
                               raw[i].length, raw[i].identities, raw[i].positives, raw[i].gaps,
                               std::string(text + raw[i].cigar_offset, raw[i].cigar_length)};
        }
        return out;
    }
    std::vector<ScanResult> scanManyImpl(const std::vector<std::string_view>& queries, const std::int8_t* const* pssms, bool pssmForm,
                                         BenchmarkStats* total) {
        sw4_db_info info{};
        check(sw4_get_db_info(handle, &info));
        const size_t nq = queries.size();
        const size_t stride = (size_t)std::max(numTop, 0);
        std::vector<const char*> ptrs(nq);
        std::vector<int32_t> lens(nq), counts(nq, 0);
        for (size_t i = 0; i < nq; i++) { ptrs[i] = queries[i].data(); lens[i] = (int32_t)queries[i].size(); }
        std::vector<int32_t> scores(std::max<size_t>(1, nq * stride)), ids(std::max<size_t>(1, nq * stride));
        std::vector<sw4_stats> per(std::max<size_t>(1, nq));
        sw4_stats tot{};
        check(pssmForm ? sw4_scan_many_pssm(handle, ptrs.data(), pssms, lens.data(), (int32_t)nq, scores.data(), ids.data(), counts.data(),
                                            per.data(), &tot)
                       : sw4_scan_many(handle, ptrs.data(), lens.data(), (int32_t)nq, scores.data(), ids.data(), counts.data(), per.data(), &tot));
        std::vector<ScanResult> out(nq);
        for (size_t i = 0; i < nq; i++) {
            out[i].scores.assign(scores.begin() + i * stride, scores.begin() + i * stride + counts[i]);
            out[i].referenceIds.assign(ids.begin() + i * stride, ids.begin() + i * stride + counts[i]);
            out[i].stats = BenchmarkStats{per[i].num_overflows, per[i].seconds, per[i].gcups};
        }
        if (total) *total = BenchmarkStats{tot.num_overflows, tot.seconds, tot.gcups};
        return out;
    }

    std::vector<std::int8_t> buildPssmImpl(const char* query, const std::int8_t* pssm, SequenceLengthT length,
                                           const std::vector<ReferenceIdT>& ids, double pseudocountWeight) {
        std::vector<std::int8_t> out((size_t)std::max(length, 1) * 21, 0);
        check(sw4_build_pssm(handle, query, pssm, length, ids.data(), (int32_t)ids.size(), pseudocountWeight, out.data(), nullptr));
        out.resize((size_t)std::max(length, 0) * 21);
        return out;
    }

    void check(int rc) const { if (rc != SW4_OK) throw std::runtime_error(sw4_last_error(handle)); }
    sw4_handle* handle = nullptr;
    int numTop = 10;
    int gop = -11, gex = -1;                                                                          // :2443-2444
    bool verbose = false;
};

}  // namespace cudasw4
#endif
