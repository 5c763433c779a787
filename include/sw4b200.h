/*
 * sw4b200.h - C ABI of the B200-native Smith-Waterman database search engine (libsw4b200.so).
 *
 * This is the drop-in boundary for the one hot path of CUDASW++4.0: CudaSW4::scan() -> score kernels -> top-k ->
 * multi-GPU merge. The reference has no FFI layer; its boundary is the header-only C++ class cudasw4::CudaSW4
 * (reference src/cudasw4.cuh:244-2454) used by src/main.cu:157-410. Every entry point below names the reference
 * member it replaces. include/cudasw4.cuh is a source-compatible C++ facade of that class on top of this ABI.
 *
 * Conventions: plain pointers and sizes only; every function returns SW4_OK (0) or a negative error code and never
 * throws; sw4_last_error() returns the message of the last failure on that handle (or globally for h == NULL).
 * device_ids may name the same GPU more than once: every entry gets its own shard (useful to exercise the multi-shard
 * path on a single-GPU machine).
 * Not thread-safe per handle (same as the reference, SURVEY.md 8b). All scores are exact Gotoh local-alignment
 * scores (int32); result lists are ordered by (score descending, database id ascending).
 * There is no CPU fallback: sw4_create() fails when no CUDA device is usable.
 */
#ifndef SW4B200_H
#define SW4B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SW4_OK 0
#define SW4_ERR_INVALID (-1)   /* bad argument / state (std::runtime_error in the reference)          */
#define SW4_ERR_CUDA (-2)      /* CUDA runtime failure (CUERR -> exit(1) in the reference)             */
#define SW4_ERR_IO (-3)        /* database files unreadable (LoadDBException in the reference)         */
#define SW4_ERR_NOMEM (-4)     /* device/host allocation failure (std::bad_alloc in the reference)     */

typedef struct sw4_handle sw4_handle;

/* cudasw4::KernelType (src/types.hpp:11-16). The engine computes in s16x2 DPX + exact s32 DPX; Half2/Float are
 * accepted for option compatibility and select the same exact-integer kernels (scores are identical by definition),
 * only the overflow accounting threshold follows the requested type (2048 for Half2, 25000 for DPXs16). */
enum { SW4_KERNEL_HALF2 = 0, SW4_KERNEL_DPX_S16 = 1, SW4_KERNEL_DPX_S32 = 2, SW4_KERNEL_FLOAT = 3 };

/* cudasw4::MemoryConfig (src/cudasw4.cuh:95-100) */
typedef struct sw4_mem_config {
    size_t max_batch_bytes;      /* accepted, unused: streaming batches are sized from max_gpu_mem (see below)   */
    size_t max_batch_sequences;  /* accepted, unused                                                             */
    size_t max_temp_bytes;       /* cap for the border-row scratch of the long-subject kernels, per query in     *
                                  * flight and GPU (fewer rows = fewer CTAs on those kernels; a query whose 16    *
                                  * row arrays do not fit is refused with SW4_ERR_NOMEM)                          */
    size_t max_gpu_mem;          /* cap for the DATABASE-related device memory per GPU (kernel-ready layout +    *
                                  * per-sequence arrays; SIZE_MAX = whatever is free). A shard that fits is kept  *
                                  * resident (--uploadFull); otherwise it is cut into batches that are streamed   *
                                  * through two device slots on every scan, the upload of the next batch          *
                                  * overlapping the kernels of the current one (src/cudasw4.cuh:1558-1712)        */
} sw4_mem_config;

/* cudasw4::BenchmarkStats (src/cudasw4.cuh:76-80) + device-side breakdown used by bench.py */
typedef struct sw4_stats {
    int32_t num_overflows;   /* subjects whose packed 16-bit score saturated and were re-scored in 32 bit         */
    double seconds;          /* device-timed: query upload -> top-k on host (CUDA events), as src/cudasw4.cuh:707 */
    double gcups;            /* sum(true subject lengths) * query length / 1e9 / seconds (src/cudasw4.cuh:2264)   */
    double kernel_seconds;   /* device time of the score kernels alone (max over GPUs)                            */
    double cells;            /* DP cells of this scan                                                             */
    int32_t kernel_launches; /* kernels launched by this scan (all GPUs)                                          */
} sw4_stats;

typedef struct sw4_db_info {
    uint64_t num_sequences;      /* sequences of the whole database (also for a pre-sharded handle)              */
    uint64_t num_residues;       /* sum of true lengths of the sequences this handle HOLDS (the whole database    *
                                  * unless it was set with sw4_set_database_shard_memory / _pseudo_database_lengths; *
                                  * the same goes for min/max_length and partition_counts)                        */
    int32_t min_length, max_length;
    uint64_t partition_counts[36]; /* sequences per reference length partition (src/length_partitions.hpp) */
    int32_t shard_rank, shard_world;
    uint64_t shard_sequences, shard_residues; /* what this handle actually scans */
    int32_t streaming;           /* after the upload: 1 when some GPU streams its shard in batches (max_gpu_mem) */
    int32_t num_batches;         /* after the upload: largest number of batches on one GPU (1 = resident)       */
} sw4_db_info;

/* CudaSW4::CudaSW4(deviceIds, numTop, blosumType, kernelTypeConfig, memoryConfig, verbose)  src/cudasw4.cuh:496-531.
 * blosum is 45, 50, 62 or 80 (the 21x21 "_20" tables, the only ones the shipped align can reach). gop/gex are the
 * (negative) gap-open / gap-extend scores: the first residue of a gap costs gop, each further one gex.
 * mem may be NULL (defaults = src/options.hpp:33-37). */
int sw4_create(const int* device_ids, int num_devices, int num_top, int blosum, int gop, int gex,
               const sw4_mem_config* mem, int verbose, sw4_handle** out);
/* ~CudaSW4 */
int sw4_destroy(sw4_handle* h);
const char* sw4_last_error(const sw4_handle* h);

/* CudaSW4::setGapOpenScore / setGapExtendScore  src/cudasw4.cuh:539-550 (positive values are negated like there) */
int sw4_set_gap_scores(sw4_handle* h, int gop, int gex);
/* CudaSW4::setNumTop  src/cudasw4.cuh:574-587 */
int sw4_set_num_top(sw4_handle* h, int num_top);
/* CudaSW4::setBlosum  src/cudasw4.cuh:570-572 */
int sw4_set_blosum(sw4_handle* h, int blosum);
/* CudaSW4::setKernelTypeConfig  src/cudasw4.cuh:589-607 (validity rules 841-855) */
int sw4_set_kernel_types(sw4_handle* h, int single_pass, int many_pass_small, int many_pass_large, int overflow);

/* CudaSW4::setMemoryConfig  src/cudasw4.cuh:609-611. Takes effect at the next upload / scan: the device layout is
 * planned again (resident or streamed) and the database is uploaded again. */
int sw4_set_mem_config(sw4_handle* h, const sw4_mem_config* mem);

/* One-process-per-GPU deployments (torch.distributed / MPI): this handle scans only shard `rank` of `world`
 * (interleaved blocks of the length-sorted database, so every shard sees the same length mix, cf. the per-partition
 * split of src/cudasw4.cuh:928-1004) and reports GLOBAL database ids. Must be called before a database is set. */
int sw4_set_shard(sw4_handle* h, int rank, int world);

/* CudaSW4::setDatabase(shared_ptr<DB>) after loadDB(prefix)  src/cudasw4.cuh:552-556, src/dbdata.cpp:207-222:
 * maps the six files written by makedb (<prefix>0chars, 0offsets, 0lengths, 0headers, 0headeroffsets; metadata is
 * ignored as in the reference). prefetch != 0 populates the mapping eagerly (--prefetchDBFile). */
int sw4_set_database_files(sw4_handle* h, const char* db_prefix, int prefetch);
/* CudaSW4::setDatabase(shared_ptr<DBWithVectors>)  src/cudasw4.cuh:558-562: borrowed host arrays in makedb layout;
 * they must stay valid until the handle is destroyed or another database is set. headers may be NULL. */
int sw4_set_database_memory(sw4_handle* h, const char* chars, const size_t* offsets, const int32_t* lengths,
                            const char* headers, const size_t* header_offsets, size_t num_sequences);
/* One-process-per-GPU deployments where every rank already holds ONLY its own shard in host memory (e.g. generated or
 * read per rank): same arrays as sw4_set_database_memory for the local sequences (ascending length), plus their
 * global database ids (strictly ascending) and the size of the whole database. Results carry global ids; the
 * sw4_reference_* accessors only know the local sequences. sw4_set_shard is ignored for such a database (it is
 * already sharded); the handle's own GPUs still split it. global_ids == NULL is sw4_set_database_memory. */
int sw4_set_database_shard_memory(sw4_handle* h, const char* chars, const size_t* offsets, const int32_t* lengths,
                                  const char* headers, const size_t* header_offsets, size_t num_sequences,
                                  const int32_t* global_ids, size_t num_sequences_global);
/* CudaSW4::setDatabase(shared_ptr<PseudoDB>) after loadPseudoDB(num, length)  src/dbdata.hpp:219-272 (seed 42) */
int sw4_set_pseudo_database(sw4_handle* h, size_t num_sequences, int length, int seed);

/* PseudoDB with a length distribution (benchmark shapes, SURVEY.md 8-d): `lengths` (ascending) describes the WHOLE
 * database; the handle generates and keeps only its own shard (sw4_set_shard rank/world, global ids in the results).
 * Residue p of sequence id = table[byte (p & 7) of mix64(mix64(seed + id) + (p >> 3))] (splitmix64 finaliser, table =
 * UniProt background frequencies in 1/256 steps; restated in cudasw4_b200/synth.py for checkers).
 * planted_codes[k] (residue CODES 0..20, exactly lengths[planted_ids[k]] of them) replaces sequence planted_ids[k]. */
int sw4_set_pseudo_database_lengths(sw4_handle* h, const int32_t* lengths, size_t num_sequences, uint64_t seed,
                                    const int32_t* planted_ids, const uint8_t* const* planted_codes, int32_t num_planted);

/* CudaSW4::prefetchDBToGpus  src/cudasw4.cuh:651-696. Builds the device-resident, length-classed, pair-interleaved
 * layout on every GPU. Called implicitly by the first sw4_scan() if omitted. */
int sw4_upload_database(sw4_handle* h);

/* ScanResult CudaSW4::scan(const char* query, SequenceLengthT length)  src/cudasw4.cuh:698-765.
 * query = residue LETTERS (converted on the device like setQuery, src/cudasw4.cuh:1280-1310). out_scores/out_ids must
 * hold num_top entries; *out_count receives min(num_top, database size). stats may be NULL. */
int sw4_scan(sw4_handle* h, const char* query, int32_t query_length, int32_t* out_scores, int32_t* out_ids,
             int32_t* out_count, sw4_stats* stats);

/* Query batching (SURVEY.md 8-f4; the reference scans one query at a time, src/main.cu:228-255): scans `num_queries`
 * queries with several of them in flight per GPU, so that the tail of one scan is back-filled by the next one and
 * the host never waits between queries; when the database is streamed (max_gpu_mem), every batch is uploaded once
 * per group of up to 16 queries instead of once per query. Results are identical to num_queries sw4_scan calls.
 * out_scores / out_ids: [num_queries][num_top] (row stride num_top), out_counts[num_queries].
 * per_query_stats (may be NULL): device-timed per query (the intervals of queries in flight overlap);
 * total_stats (may be NULL): seconds = device-timed span of the whole call (CUDA events: first query's upload ->
 * last result on the host, max over the GPUs), gcups = all cells / that time. */
int sw4_scan_many(sw4_handle* h, const char* const* queries, const int32_t* query_lengths, int32_t num_queries,
                  int32_t* out_scores, int32_t* out_ids, int32_t* out_counts, sw4_stats* per_query_stats,
                  sw4_stats* total_stats);

/* Where each hit aligns (no reference counterpart): for every id, the exact score and the begin and end of one optimal
 * local alignment in the query and in the reference, computed on the handle's first GPU on a stream of its own, with
 * the current matrix and gap scores. Positions are 0-based and inclusive. With H the local Gotoh matrix (i: query,
 * j: reference) and S = max H:
 *   end   (query_end, reference_end)     = the smallest (i, j) in (i, j) order with H(i, j) == S;
 *   begin (query_begin, reference_begin) = the largest (i, j) such that an alignment starting with the pair (i, j) and
 *                                          ending with the pair at the end scores S (the shortest optimal alignment);
 *   S == 0 (no positive substitution, empty query or subject): all four positions are -1.
 * query = residue LETTERS (converted as sw4_scan converts them). ids are global database ids, duplicates allowed;
 * num_ids == 0 does nothing. Subjects come from the host copy, so the call works before sw4_upload_database and in
 * every database mode, and leaves the results of later scans unchanged. Pairs whose scratch (subjects + border
 * columns) does not fit max_temp_bytes at once are processed in chunks; a single pair that cannot fit is
 * SW4_ERR_NOMEM. SW4_ERR_INVALID: no database, num_ids < 0, an id < 0 or >= num_sequences or not held by a pre-sharded
 * handle, query_length > 2^24, or a pair whose score could reach 2^24 (max matrix entry x min(query, subject) length).
 * stats may be NULL: seconds is device-timed (CUDA events), cells counts both passes, kernel_launches the kernels. */
typedef struct sw4_alignment {
    int32_t score;                           /* exact Gotoh score (== what sw4_scan reports for this id) */
    int32_t query_begin, query_end;          /* 0-based, inclusive; -1 when score == 0 */
    int32_t reference_begin, reference_end;  /* 0-based, inclusive; -1 when score == 0 */
} sw4_alignment;

int sw4_alignment_coordinates(sw4_handle* h, const char* query, int32_t query_length, const int32_t* ids, int32_t num_ids,
                              sw4_alignment* out, sw4_stats* stats);

/* How each hit aligns (no reference counterpart): the coordinates of sw4_alignment_coordinates, and the columns of the
 * one alignment they locate, traced back on the same GPU.
 *
 * The reported alignment is the one that sw4_alignment_coordinates locates: it starts with the pair (qb, rb), ends
 * with the pair (qe, re) and scores S. When several alignments qualify, this rule picks exactly one.
 * Over the rectangle, use the anchored recurrences started at (qb, rb):
 *   P is the pair state.
 *   E is a gap column that consumes a reference residue only. Its CIGAR op is D.
 *   F is a gap column that consumes a query residue only. Its CIGAR op is I.
 *   X = max(P, E, F).
 *   E(i,j) = max(X(i,j-1) + gop, E(i,j-1) + gex), and F likewise along i.
 * Walk back from (qe, re) in state P:
 *   In P at (i, j): emit the pair (= if the two residue codes are equal, else X). Unless this is (qb, rb), step to
 *     (i-1, j-1) and take the first state of P, E, F whose value equals X(i-1, j-1).
 *   In E at (i, j): emit D. Step to (i, j-1). If E(i,j-1) + gex == E(i,j), extend: stay in E. Extend wins a tie.
 *     Otherwise open: take the first of P, E, F equal to X(i, j-1).
 *   In F: do the same along i, emitting I.
 * The walk ends at (qb, rb) in state P. Score 0 gives coordinates of -1, an empty CIGAR and zero counts.
 *
 * Per hit, report the coordinates (identical to sw4_alignment_coordinates), the CIGAR and four counts:
 *   CIGAR: run-length ops =, X, I, D, in query order. I consumes the query only and D the reference only, as in SAM
 *     with the query as the read.
 *   length: the number of columns.
 *   identities: the number of = columns. These compare residue codes, so every non-standard letter counts as code 20.
 *   positives: pairs with a substitution score > 0.
 *   gaps: I + D columns.
 * A CIGAR rescores as follows. A pair scores M[q][r]. A maximal run of k gap columns of one kind scores
 * gop + (k-1) * max(gop, gex). Adjacent I and D runs each pay their own open. This is what the Gotoh recurrence
 * computes: H includes E, so when gop > gex (for example 0 / -4096) a gap is "re-opened" rather than extended.
 * Rescoring every CIGAR gives exactly S.
 *
 * Arguments, errors and chunking are those of sw4_alignment_coordinates; the traceback chunks the pairs again by their
 * trace scratch (about half a byte per cell of the rectangle plus rows + columns bytes; DESIGN.md 3.7), and a single
 * rectangle that does not fit max_temp_bytes is SW4_ERR_NOMEM. stats may be NULL: seconds is device-timed, cells
 * counts all three passes, kernel_launches every kernel. */
typedef struct sw4_alignment_summary {
    sw4_alignment coordinates;          /* == sw4_alignment_coordinates for this id */
    int32_t length, identities, positives, gaps;
    size_t cigar_offset, cigar_length;  /* into the text of sw4_last_cigars */
} sw4_alignment_summary;
int sw4_alignment_traceback(sw4_handle* h, const char* query, int32_t query_length, const int32_t* ids,
                            int32_t num_ids, sw4_alignment_summary* out, sw4_stats* stats);
/* CIGAR text of the last sw4_alignment_traceback on this handle; valid until the next call or sw4_destroy */
int sw4_last_cigars(const sw4_handle* h, const char** text, size_t* length);

/* Search with a position-specific scoring matrix (PSSM; no reference counterpart), such as PSI-BLAST's
 * -out_ascii_pssm writes it.
 *
 * A PSSM query is query_length residue letters plus int8_t pssm[query_length][21], row-major. pssm[p][r] is the score
 * of query position p against residue code r. Codes 0..19 are ARNDCQEGHILKMFPSTWYV (the order in which letters are
 * converted); code 20 is every other letter. Columns 0..19 take the whole int8 range; column 20 takes [-128, 0], and a
 * positive pssm[p][20] is SW4_ERR_INVALID. Code 20 also pads every subject in the engine's device layout, so a padded
 * column scores like a non-standard residue; it cannot raise a score or move a first maximum only while that score is
 * <= 0 against every query position (the BLOSUM tables give it their negative `low`).
 *
 * Every score, coordinate and CIGAR definition above holds with M[q_i][r] replaced by pssm[i][r]. Positives are the
 * pair columns with pssm[i][r] > 0. Identities and the =/X ops still compare residue codes; that is the only use of
 * the letters, and scores never depend on them. The handle's gap scores apply; its BLOSUM table is not used. The bound
 * that keeps scores below 2^24 uses the PSSM's own largest entry (at least 1) x min(query, subject) length, per query.
 *
 * Why the 16-bit scan stays exact with any int8 entries: every s16 kernel (two-row, multi-segment, one-row wide and
 * both array kernels) keeps, per subject of a packed pair, a running maximum of the diagonal term H[i-1][j-1] +
 * pssm[i][s_j] of every cell, and compares it with the re-scoring threshold 25000 once, when the pair is finished (the
 * array kernels fold the maxima of a pair's column blocks with a max first). Until some H reaches 25000 every value is
 * exact, and the first H to reach it is a diagonal term (E and F never exceed an earlier H), of at most 24999 + 127 <
 * 32767: it enters the running maximum before any 16-bit wrap, and a maximum never decreases, so the subject is
 * re-scored in 32 bit whatever wraps after it. Downwards, the gap rows' sentinel -16000 and
 * the E / F floors take at most -128 (one entry) or -4096 (one gap score) per step before the local floor at 0 or the
 * maximum with the sentinel resets them, far from -32768.
 *
 * The calls below behave as their sequence forms (arguments, outputs, errors, chunking, streaming, sharding, query
 * batching, sw4_last_cigars and sw4_last_scan_all_scores). query and pssm may be NULL only when query_length == 0;
 * otherwise a NULL one is SW4_ERR_INVALID, as is a positive entry in column 20. pssms[i] of sw4_scan_many_pssm belongs to queries[i]. */
int sw4_scan_pssm(sw4_handle* h, const char* query, const int8_t* pssm, int32_t query_length, int32_t* out_scores,
                  int32_t* out_ids, int32_t* out_count, sw4_stats* stats);
int sw4_scan_many_pssm(sw4_handle* h, const char* const* queries, const int8_t* const* pssms,
                       const int32_t* query_lengths, int32_t num_queries, int32_t* out_scores, int32_t* out_ids,
                       int32_t* out_counts, sw4_stats* per_query_stats, sw4_stats* total_stats);
int sw4_alignment_coordinates_pssm(sw4_handle* h, const char* query, const int8_t* pssm, int32_t query_length,
                                   const int32_t* ids, int32_t num_ids, sw4_alignment* out, sw4_stats* stats);
int sw4_alignment_traceback_pssm(sw4_handle* h, const char* query, const int8_t* pssm, int32_t query_length,
                                 const int32_t* ids, int32_t num_ids, sw4_alignment_summary* out, sw4_stats* stats);

/* Significance of the hits (no reference counterpart): E-values and bit scores from score statistics that each query's
 * own search yields. Every scan with statistics enabled also builds, on the GPU, a histogram of the scores of the
 * subjects it scanned: count[s] subjects and lensum[s] residues (the sum of their lengths) per score s, for
 * s = 0 .. SW4_SCORE_BINS - 1, and an overflow bin s = SW4_SCORE_BINS for all higher scores. Subjects of length 0 are
 * left out. In a database almost every subject is unrelated to the query, so this is the null distribution, and the fit
 * below turns it into lambda and K. It needs no tabulated constants and serves PSSM queries at any score scale.
 *
 * Model: with m the query length and n_j the length of subject j, its score behaves like x_j = s_j + 1/2 with
 * P(x_j >= x) = 1 - exp(-K m n_j e^(-lambda x)).
 * Censoring, with N the subjects of length >= 1:
 *   c_lo = the median score: the smallest s with #(score <= s) >= N / 2. Lower scores are left-censored.
 *   c_hi = the smallest s > c_lo with #(score >= s) <= floor(N / 1000); SW4_SCORE_BINS when no such s is below it.
 *          Scores >= c_hi are right-censored (the homologs end up there).
 * Maximum likelihood: U subjects with c_lo <= s < c_hi contribute ln lambda + ln(K m n_j) - lambda x_j - K m n_j
 * e^(-lambda x_j); a left-censored one -K m n_j e^(-lambda c_lo); the R right-censored ones ln(K m n_j) - lambda c_hi.
 * dlnL/dK = 0 gives K = (U + R) / (m A(lambda)) with A(lambda) = sum_fitted lensum[s] e^(-lambda (s + 1/2)) +
 * e^(-lambda c_lo) sum_{s < c_lo} lensum[s]. The profile likelihood is strictly concave in lambda; its derivative
 * U / lambda - sum_fitted count[s] (s + 1/2) - R c_hi + (U + R) B(lambda) / A(lambda), with B = A with each term
 * weighted by its x (s + 1/2, or c_lo), is bisected on [1e-4, 10] until the interval cannot shrink in double.
 * status SW4_STATS_TOO_FEW (lambda = K = NaN: no E-values, no cutoff) when U < 100, c_lo >= SW4_SCORE_BINS or m < 1.
 *
 * A hit with score S has E = K m D e^(-lambda S) (D = sum of lensum: the residues of the subjects; E is the expected
 * number of subjects with a score >= S under the model) and the bit score (lambda S - ln K) / ln 2. E decreases with S,
 * so a cutoff on E only shortens a result list. */
#define SW4_SCORE_BINS 4096
#define SW4_STATS_OK 0
#define SW4_STATS_TOO_FEW 1
typedef struct sw4_score_statistics {
    int32_t status;          /* SW4_STATS_OK or SW4_STATS_TOO_FEW                                                    */
    int32_t whole_database;  /* 1 when the histogram covers the whole database; 0 when the handle scans only a shard   *
                              * (sw4_set_shard with world > 1, or a database of which it holds only some sequences:    *
                              * sw4_set_database_shard_memory, sw4_set_pseudo_database_lengths under sw4_set_shard)     */
    double lambda, K;        /* NaN unless status == SW4_STATS_OK                                                     */
    int64_t query_length;    /* m */
    int64_t db_residues;     /* D = sum of lensum */
    int64_t num_subjects;    /* N = sum of count */
    int64_t fitted, left_censored, right_censored;  /* U, the subjects below c_lo, R */
    int32_t c_lo, c_hi;
} sw4_score_statistics;

/* The fit above, on a histogram of bins + 1 entries per array (entry `bins` is the overflow bin), for example one summed
 * over the shards of a sharded search. Pure host code: it needs no handle and no device. whole_database is set to 1.
 * SW4_ERR_INVALID: NULL arrays or out, bins < 1, or a negative entry. */
int sw4_fit_score_statistics(const int64_t* counts, const int64_t* lensums, int32_t bins, int64_t query_length,
                             sw4_score_statistics* out);

/* enabled != 0: every following scan also builds the score histogram of each query (one more kernel per query and GPU)
 * and fits it. max_evalue (INFINITY: no cutoff) then drops the hits with E > max_evalue from out_scores / out_ids /
 * *out_count of every scan call (sw4_scan, sw4_scan_many and their _pssm forms), but only when the handle holds the
 * whole database and the fit succeeded. enabled == 0 (the default): a scan does exactly what it did without statistics.
 * SW4_ERR_INVALID: max_evalue NaN or < 0. */
int sw4_set_score_statistics(sw4_handle* h, int enabled, double max_evalue);
/* The statistics of query `query_index` of the last scan call (0 after sw4_scan). A handle on several GPUs sums their
 * histograms before the fit. SW4_ERR_INVALID when the last scan ran without statistics or query_index is out of range. */
int sw4_last_score_statistics(const sw4_handle* h, int32_t query_index, sw4_score_statistics* out);
/* The histogram behind sw4_last_score_statistics (this handle's shards summed): counts and lensums hold bins + 1 entries,
 * and bins must be SW4_SCORE_BINS. A sharded search sums these over its ranks and calls sw4_fit_score_statistics. */
int sw4_last_score_histogram(const sw4_handle* h, int32_t query_index, int64_t* counts, int64_t* lensums, int32_t bins);

/* Iterative profile search (no reference counterpart): a PSSM built on the GPU from a search's own hits, and rounds of
 * scan -> significant hits -> profile -> scan, in the manner of PSI-BLAST (its numbers are not reproduced).
 *
 * sw4_build_pssm writes out[query_length][21], the profile of the query and the hits `ids`. M is the handle's table, its
 * gap scores apply, and `pssm` (NULL: the sequence query, scored with M) is the query form the hits are aligned with.
 *   1. Alignments: for each id, the alignment sw4_alignment_traceback(_pssm) reports for that query form. Ids whose
 *      score is 0 add no row.
 *   2. Query-anchored MSA over the query's m positions (columns c): row 0 is the query, x_0c = q_c (its codes, converted
 *      as every call converts them). Then one row per remaining id, in the order of `ids` (duplicates each add a row).
 *      Row k covers columns qb..qe of its alignment: an = or X column puts the reference code paired with query position
 *      c into x_kc; an I column (query position c in a gap) puts GAP there; D columns leave nothing; columns outside
 *      [qb, qe] are empty. The symbols are codes 0..20 and GAP.
 *   3. Henikoff position-based weights over the whole MSA: r_c = the number of distinct symbols in column c,
 *      n_{c,s} = the number of rows with symbol s there, w_k = sum over the non-empty c of row k of 1 / (r_c n_{c,x_kc}).
 *   4. Frequencies from the rows with x_kc in 0..19: W_c = sum w_k over those rows, f_ca = sum_{x_kc = a} w_k / W_c. If
 *      W_c = 0 (q_c = 20 and no standard residue in the column), output row c is M[20][.].
 *   5. Background p_a = the generated databases' frequencies (sw4_set_pseudo_database_lengths, 1/256 steps). lambda_u is
 *      the root of sum_{a,b<20} p_a p_b e^(lambda M[a][b]) = 1, bisected in double on [1e-3, 2] until the interval
 *      stops shrinking; q_ab = p_a p_b e^(lambda_u M[a][b]) / Z with Z that sum.
 *   6. r'_c = the number of distinct codes 0..19 in column c; N = the mean of r'_c over the columns with r'_c >= 1 and
 *      alpha = N - 1 (0 when there is no such column); g_ca = sum_b f_cb q_ab / p_b;
 *      Q_ca = (alpha f_ca + beta g_ca) / (alpha + beta);
 *      out[c][a] = clamp(floor(ln(Q_ca / p_a) / lambda_u + 1/2), -128, 127) for a < 20, and out[c][20] = M's `low`.
 * With no hits alpha = 0 and every row is M[q_c][.]: a scan with that PSSM equals the sequence scan.
 * The arguments, errors and chunking are those of sw4_alignment_traceback(_pssm), and sw4_last_cigars is left as it was.
 * The MSA, (1 + rows) x query_length bytes, is allocated apart from the traceback scratch: when it alone exceeds
 * max_temp_bytes the call is SW4_ERR_NOMEM. beta (the pseudocount weight, PSI-BLAST's default is 10) <= 0, NaN or
 * infinite is SW4_ERR_INVALID. The same call always returns the same bytes, however the pairs are chunked. stats may be
 * NULL: it covers every pass and kernel of the call.
 *
 * sw4_search_iterative runs the rounds on the query letters:
 *   P_1 = the sequence;
 *   round i: scan with P_i; H_i = the ids of the top-num_top list, taken before the handle's max_evalue cutoff, with
 *   E <= inclusion_evalue; stop when i == max_iterations, H_i is empty or set(H_i) == set(H_{i-1}) (then converged = 1,
 *   for i >= 2 and a non-empty H_i); else P_{i+1} = sw4_build_pssm(query, P_i, H_i in list order, beta).
 * It reports the last scan's list exactly as that scan reports it (the max_evalue cutoff applies) in out_scores /
 * out_ids / *out_count (num_top entries), the PSSM that scan searched with in out_pssm[query_length][21] (after one
 * round: the profile without hits, the matrix rows), the number of rounds and the converged flag.
 * sw4_last_score_statistics then describes the last scan. SW4_ERR_INVALID: statistics not enabled, a handle that does
 * not scan the whole database (sw4_set_shard with world > 1, a partly held database), max_iterations < 1, a NaN or
 * negative inclusion_evalue, a bad beta, or null outputs. stats may be NULL: it sums every scan, pass and kernel. */
int sw4_build_pssm(sw4_handle* h, const char* query, const int8_t* pssm, int32_t query_length, const int32_t* ids, int32_t num_ids,
                   double beta, int8_t* out, sw4_stats* stats);
int sw4_search_iterative(sw4_handle* h, const char* query, int32_t query_length, int32_t max_iterations, double inclusion_evalue,
                         double beta, int32_t* out_scores, int32_t* out_ids, int32_t* out_count, int8_t* out_pssm,
                         int32_t* out_iterations, int32_t* out_converged, sw4_stats* stats);

/* Debug / parity helper (the reference's CUDASW_DEBUG_CHECK_CORRECTNESS mode sets numTop to the whole database,
 * src/cudasw4.cuh:505-507): all scores of the last scan for this handle's shard, plus their global ids, in shard
 * order. capacity is in entries; returns the number written in *out_count. */
int sw4_last_scan_all_scores(sw4_handle* h, int32_t* out_scores, int32_t* out_ids, size_t capacity, size_t* out_count);

/* CudaSW4::getReferenceHeader / getReferenceLength / getReferenceSequence  src/cudasw4.cuh:613-639 */
int sw4_reference_header(const sw4_handle* h, int32_t id, const char** ptr, size_t* len);
int sw4_reference_length(const sw4_handle* h, int32_t id, int32_t* len);
int sw4_reference_sequence(const sw4_handle* h, int32_t id, char* out, size_t capacity, size_t* len);

/* CudaSW4::totalTimerStart / totalTimerStop  src/cudasw4.cuh:818-839 */
int sw4_total_timer_start(sw4_handle* h);
int sw4_total_timer_stop(sw4_handle* h, sw4_stats* stats);

/* CudaSW4::printDBInfo / printDBLengthPartitions  src/cudasw4.cuh:799-816 (as data instead of stdout) */
int sw4_get_db_info(const sw4_handle* h, sw4_db_info* info);

/* library / build identification, e.g. "sw4b200 0.1 sm_100a" */
const char* sw4_version(void);

#ifdef __cplusplus
}
#endif
#endif /* SW4B200_H */
