// Host engine behind the C ABI of include/sw4b200.h: database handling, sharding, per-GPU working sets, the scan
// pipeline (query -> profile -> score kernels -> exact re-scoring -> top-k -> merge) and timing.
// Mirrors the responsibilities of the reference's cudasw4::CudaSW4 (src/cudasw4.cuh:244-2454) with a different
// design:
//   * a shard lives on its GPU in a kernel-ready layout (length-classed pair-blocks built on the device); when it does
//     not fit `max_gpu_mem` it is cut into batches that are streamed through two device slots, the upload of batch
//     b+1 overlapping the kernels of batch b (the reference's streaming mode, src/cudasw4.cuh:1558-1712,
//     src/dbbatching.cuh:16-99, 238-276 - without its score-index bug, SURVEY.md 0-2);
//   * every query in flight owns a context (stream, profile, scores, scratch): sw4_scan_many keeps several queries in
//     flight so that the tail of one scan is back-filled by the next one, and in streaming mode one pass over the
//     database serves a whole group of queries (the reference scans one query at a time, src/main.cu:228-255);
//   * one persistent launch per length class, device-side top-k for any k, only k (score, id) pairs per GPU reach the
//     host; one host thread per GPU.
#include <algorithm>
#include <cerrno>
#include <cmath>
#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <memory>
#include <random>
#include <string>
#include <thread>
#include <vector>

#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <cuda_runtime.h>

#include "../../include/sw4b200.h"
#include "blosum_tables.hpp"
#include "device_db.cuh"
#include "launch.hpp"
#include "profile.cuh"
#include "stats.cuh"
#include "topk.cuh"

namespace sw4 {

// ---------------------------------------------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------------------------------------------
struct Error {
    int code;
    std::string msg;
};

[[noreturn]] static void fail(int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    throw Error{code, buf};
}

#define SW4_CUDA(expr)                                                                                   \
    do {                                                                                                 \
        cudaError_t e_ = (expr);                                                                         \
        if (e_ != cudaSuccess)                                                                           \
            ::sw4::fail(e_ == cudaErrorMemoryAllocation ? SW4_ERR_NOMEM : SW4_ERR_CUDA, "%s failed: %s (%s:%d)", \
                        #expr, cudaGetErrorString(e_), __FILE__, __LINE__);                              \
    } while (0)

// ---------------------------------------------------------------------------------------------------------------
// length classes of the packed 16-bit kernel: G lanes x R columns, capacity G*R
// ---------------------------------------------------------------------------------------------------------------
// G = 1<<logG lanes x R columns per lane; capacity = G*R columns per pair-block. Subjects up to 512 residues run on the
// two-rows-per-step kernel (G = 8 or 16, kernels_s16.cuh); 513..1024 and the multi-segment class (1024-column segments,
// any length) on the full-warp one-row-per-step variant (G = 32, kernels_s16_wide.cuh).
struct LengthClass { int logG, R, capacity; bool wide, multi; };
static const LengthClass kLengthClasses[] = {
    {3, 4, 32, false, false}, {3, 6, 48, false, false}, {3, 8, 64, false, false}, {3, 10, 80, false, false},
    {3, 12, 96, false, false}, {3, 14, 112, false, false}, {3, 16, 128, false, false}, {3, 18, 144, false, false},
    {3, 20, 160, false, false}, {3, 22, 176, false, false}, {3, 24, 192, false, false}, {3, 26, 208, false, false},
    {3, 28, 224, false, false}, {3, 30, 240, false, false}, {4, 16, 256, false, false}, {4, 18, 288, false, false},
    {4, 20, 320, false, false}, {4, 22, 352, false, false}, {4, 24, 384, false, false}, {4, 26, 416, false, false},
    {4, 28, 448, false, false}, {4, 30, 480, false, false}, {4, 32, 512, false, false}, {5, 18, 576, true, false},
    {5, 20, 640, true, false}, {5, 22, 704, true, false}, {5, 24, 768, true, false}, {5, 26, 832, true, false},
    {5, 28, 896, true, false}, {5, 30, 960, true, false}, {5, 32, 1024, true, false}, {5, 32, 1024, true, true},
};
constexpr int kNumLengthClasses = sizeof(kLengthClasses) / sizeof(kLengthClasses[0]);
constexpr int kS16OverflowThreshold = 25000;  // reference MAX_ACC_SHORT, src/kernels.cuh:5
constexpr int kHalf2Threshold = 2048;         // reference MAX_ACC_HALF2, src/kernels.cuh:4
constexpr int kNumCounters = 8 + 32;          // [0] overflow [1] stat [2],[3] s32 tickets [4] top-k count [8+c] class tickets
constexpr int kShardBlock = 256;              // subjects per interleaving block (even => pairs never straddle)
constexpr int kMaxClassStreams = 32;
constexpr int kProfileRows = kFused + 63;     // 441 fused-pair rows + two s16 single-residue planes + one int32 plane
constexpr int kMaxContexts = 16;              // queries in flight per GPU (streaming mode: queries served per pass)
constexpr size_t kStageChunkBytes = (size_t)32 << 20;  // pinned staging buffers of the database upload (two of them)

static const int kRefBoundaries[36] = {48,  64,  80,  96,  112, 128, 144, 160, 176, 192,  208,  224,
                                       240, 256, 288, 320, 352, 384, 416, 448, 480, 512,  576,  640,
                                       704, 768, 832, 896, 960, 1024, 1088, 1152, 1216, 1280, 8000, 2147483646};

static inline size_t alignUp(size_t v, size_t a) { return (v + a - 1) / a * a; }

// UniProt background frequencies in 1/256 steps (cumulative), residue codes 0..19: the residues of generated databases
// (sw4_set_pseudo_database_lengths) and the background p_a of the profile construction (sw4_build_pssm)
static const int kPseudoCumulative[20] = {21, 35, 46, 60, 63, 73, 91, 109, 115, 130, 155, 170, 176, 186, 198, 214, 228, 231, 238, 256};

// ---------------------------------------------------------------------------------------------------------------
// host database (makedb format)
// ---------------------------------------------------------------------------------------------------------------
struct MappedFile {
    void* ptr = nullptr;
    size_t size = 0;
    MappedFile() = default;
    MappedFile(const MappedFile&) = delete;
    MappedFile& operator=(const MappedFile&) = delete;
    ~MappedFile() { if (ptr && size) munmap(ptr, size); }
    void open(const std::string& path, bool populate) {
        int fd = ::open(path.c_str(), O_RDONLY);
        if (fd < 0) fail(SW4_ERR_IO, "cannot open %s: %s", path.c_str(), strerror(errno));
        struct stat st;
        if (fstat(fd, &st) != 0) { ::close(fd); fail(SW4_ERR_IO, "cannot stat %s", path.c_str()); }
        size = (size_t)st.st_size;
        if (size > 0) {
            ptr = mmap(nullptr, size, PROT_READ, MAP_PRIVATE | (populate ? MAP_POPULATE : 0), fd, 0);
            if (ptr == MAP_FAILED) { ptr = nullptr; ::close(fd); fail(SW4_ERR_IO, "cannot mmap %s", path.c_str()); }
        }
        ::close(fd);
    }
};

struct HostDB {
    const uint8_t* chars = nullptr;
    const size_t* offsets = nullptr;
    const int32_t* lengths = nullptr;
    const char* headers = nullptr;
    const size_t* headerOffsets = nullptr;
    const int32_t* globalIds = nullptr;  // pre-sharded database: global id of every local sequence (ascending); else null
    size_t n = 0;                        // sequences held by this handle
    size_t nGlobal = 0;                  // sequences of the whole database (== n unless pre-sharded)
    uint64_t residues = 0;
    int minLen = 0, maxLen = 0;
    // owners
    MappedFile fChars, fOffsets, fLengths, fHeaders, fHeaderOffsets;
    std::vector<uint8_t> vChars;
    std::vector<size_t> vOffsets, vHeaderOffsets;
    std::vector<int32_t> vLengths, vGlobalIds;
    std::vector<char> vHeaders;

    void finish() {
        residues = 0; minLen = n ? lengths[0] : 0; maxLen = 0;
        for (size_t i = 0; i < n; i++) {
            if (lengths[i] < 0) fail(SW4_ERR_INVALID, "negative sequence length at %zu", i);
            if (i && lengths[i] < lengths[i - 1]) fail(SW4_ERR_INVALID, "database is not sorted by length (id %zu)", i);
            if (globalIds && i && globalIds[i] <= globalIds[i - 1]) fail(SW4_ERR_INVALID, "global ids must be ascending (entry %zu)", i);
            residues += (uint64_t)lengths[i];
            minLen = std::min(minLen, lengths[i]);
            maxLen = std::max(maxLen, lengths[i]);
        }
        if (!globalIds) nGlobal = n;
        if (n > (size_t)0x7ffffffe || nGlobal > (size_t)0x7ffffffe) fail(SW4_ERR_INVALID, "too many sequences");
        if (globalIds && n && ((size_t)globalIds[n - 1] >= nGlobal || globalIds[0] < 0)) fail(SW4_ERR_INVALID, "global id out of range");
    }
    // position of global id `id` in this handle's arrays, or n when the handle does not hold it
    size_t localIndex(int32_t id) const {
        if (!globalIds) return (size_t)id < n ? (size_t)id : n;
        const int32_t* p = std::lower_bound(globalIds, globalIds + n, id);
        return (p != globalIds + n && *p == id) ? (size_t)(p - globalIds) : n;
    }
};

// ---------------------------------------------------------------------------------------------------------------
// device buffers
// ---------------------------------------------------------------------------------------------------------------
template <class T>
struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { release(); }
    void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
    void alloc(size_t count) {
        release();
        if (count == 0) count = 1;
        SW4_CUDA(cudaMalloc(&p, count * sizeof(T)));
        n = count;
    }
    void ensure(size_t count) { if (count > n) alloc(count + count / 4); }
    size_t bytes() const { return n * sizeof(T); }
};

template <class T>
struct PinnedBuf {
    T* p = nullptr;
    size_t n = 0;
    PinnedBuf() = default;
    PinnedBuf(const PinnedBuf&) = delete;
    PinnedBuf& operator=(const PinnedBuf&) = delete;
    ~PinnedBuf() { if (p) cudaFreeHost(p); }
    void ensure(size_t count) {
        if (count <= n) return;
        if (p) cudaFreeHost(p);
        p = nullptr; n = 0;
        SW4_CUDA(cudaMallocHost(&p, count * sizeof(T)));
        n = count;
    }
};

// ---------------------------------------------------------------------------------------------------------------
// batches (what is resident in one device slot at a time) and their per-class layout
// ---------------------------------------------------------------------------------------------------------------
struct BatchClass {
    int cls = 0;               // index into kLengthClasses
    int first = 0, count = 0;  // shard-local subject range
    int numItems = 0, numBlocks = 0;
    size_t colsOff = 0, itemsOff = 0, blockItemOff = 0;  // byte offsets inside the slot arena
    std::vector<S16Item> hostItems;       // multi-segment class only (the others are generated on the device)
    std::vector<int32_t> hostBlockItem;   // multi-segment class only
};

struct Batch {
    size_t first = 0, count = 0;   // shard-local subject range [first, first+count)
    size_t numZeroLength = 0;      // leading subjects of length 0 (they score 0 by definition)
    size_t charsBytes = 0;         // padded residues of the range
    size_t offsetsOff = 0;         // arena byte offset of the size_t[count+1] offsets (chars are at offset 0)
    size_t arenaBytes = 0;
    std::vector<BatchClass> classes;
};

struct Slot {
    DevBuf<uint8_t> arena;
    cudaEvent_t evReady = nullptr;
    int batch = -1;  // which batch the arena holds
    ~Slot() { if (evReady) cudaEventDestroy(evReady); }
};

// ---------------------------------------------------------------------------------------------------------------
// per-query context: everything one scan in flight owns on one GPU
// ---------------------------------------------------------------------------------------------------------------
struct Ctx {
    cudaStream_t stream = nullptr;
    cudaStream_t classStreams[kMaxClassStreams] = {}, oddStreams[kMaxClassStreams] = {};
    cudaEvent_t evStart = nullptr, evK0 = nullptr, evK1 = nullptr, evStop = nullptr, evFork = nullptr;
    cudaEvent_t evJoin[kMaxClassStreams] = {}, evJoinOdd[kMaxClassStreams] = {};
    cudaEvent_t evBatchDone[2] = {};
    DevBuf<int32_t> dScores, dOvfList;
    DevBuf<int> dCounters;
    DevBuf<char> dQueryLetters;
    DevBuf<uint8_t> dQueryCodes;
    DevBuf<uint32_t> dProfile;
    DevBuf<int8_t> dMatrix;
    // Border rows of the long-subject kernels: row arrays of borderStride (H, E) pairs. The first borderSlots * 32 arrays
    // belong to the multi-segment two-row kernels (several length classes run concurrently: a CTA takes a free slot of 32
    // arrays, dBorderSlots holds the flags); the remaining borderRowArrays arrays (from borderB on) serve the kernels that
    // run one at a time per scan (array kernels, one-warp-per-pair kernels, exact 32-bit kernels).
    DevBuf<uint2> dBorder;
    DevBuf<int> dBorderSlots;
    uint2* borderB = nullptr;
    size_t borderRowArrays = 0, borderStride = 0;
    int borderSlots = 0;
    DevBuf<unsigned long long> dClassNs;
    DevBuf<TopkCand> dCand;
    DevBuf<int32_t> dTopScores, dTopIds;
    DevBuf<int> dTopkWork;
    DevBuf<unsigned long long> dTopkKeys;
    PinnedBuf<char> hQuery;
    PinnedBuf<int32_t> hTop;        // scores[k], ids[k], counters[8]
    // a PSSM query's [qlen][21] table (allocated by the first PSSM query, grown with queryCapacity)
    PinnedBuf<int8_t> hPssm;
    DevBuf<int8_t> dPssm;
    // score histogram of the query (statistics enabled; allocated by the first such scan): counts, then lensums
    DevBuf<unsigned long long> dHist;
    PinnedBuf<unsigned long long> hHist;
    int queryCapacity = 0;
    size_t topCapacity = 0;
    // the query in flight
    bool busy = false;
    int queryIndex = -1, qlen = 0, k = 0, profStride = 0, launches = 0;
    bool pssm = false;
    bool stats = false;  // the scan also builds the score histogram
    int maxEntry = 1;  // largest score of one residue pair (at least 1): bounds the scores by maxEntry * min(qlen, len)
    bool largeK = false;

    void create() {
        SW4_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        SW4_CUDA(cudaEventCreate(&evStart));
        SW4_CUDA(cudaEventCreate(&evK0));
        SW4_CUDA(cudaEventCreate(&evK1));
        SW4_CUDA(cudaEventCreate(&evStop));
        SW4_CUDA(cudaEventCreateWithFlags(&evFork, cudaEventDisableTiming));
        for (auto& e : evBatchDone) SW4_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        for (int i = 0; i < kMaxClassStreams; i++) {
            SW4_CUDA(cudaStreamCreateWithFlags(&classStreams[i], cudaStreamNonBlocking));
            SW4_CUDA(cudaStreamCreateWithFlags(&oddStreams[i], cudaStreamNonBlocking));
            SW4_CUDA(cudaEventCreateWithFlags(&evJoin[i], cudaEventDisableTiming));
            SW4_CUDA(cudaEventCreateWithFlags(&evJoinOdd[i], cudaEventDisableTiming));
        }
        dCounters.alloc(kNumCounters);
        dClassNs.alloc(96);
        dMatrix.alloc(441);
        dCand.alloc(kTopkMaxCandidates);
        SW4_CUDA(topk_configure());  // every context sets it on its shard's device (runShard selects it before creating them)
        SW4_CUDA(score_histogram_configure());
    }
    ~Ctx() {
        for (cudaEvent_t e : {evStart, evK0, evK1, evStop, evFork, evBatchDone[0], evBatchDone[1]})
            if (e) cudaEventDestroy(e);
        for (int i = 0; i < kMaxClassStreams; i++) {
            if (evJoin[i]) cudaEventDestroy(evJoin[i]);
            if (evJoinOdd[i]) cudaEventDestroy(evJoinOdd[i]);
            if (classStreams[i]) cudaStreamDestroy(classStreams[i]);
            if (oddStreams[i]) cudaStreamDestroy(oddStreams[i]);
        }
        if (stream) cudaStreamDestroy(stream);
    }
};

// what one shard reports for one query
struct ShardResult {
    std::vector<int32_t> scores, ids;
    std::vector<int64_t> hist;  // counts then lensums, 2 * kHistEntries (statistics enabled only)
    int statCount = 0, launches = 0;
    double seconds = 0, kernelSeconds = 0;
};

struct Shard {
    int device = 0;
    int smCount = 148;
    size_t deviceFree = 0;
    // which part of the handle's database this shard scans: blocks firstBlock, firstBlock+blockStride, ... of
    // kShardBlock consecutive sequences
    size_t firstBlock = 0, blockStride = 1;
    size_t n = 0;
    uint64_t residues = 0;
    int maxLen = 0;
    std::vector<int32_t> lengths;          // [n]
    std::vector<size_t> blockCharPrefix;   // padded residues before local block j (local blocks of kShardBlock subjects)
    bool uploaded = false;
    bool streaming = false;
    bool hasMulti = false;
    // resident for the whole shard
    DevBuf<int32_t> dLengths, dGlobalIds;
    std::vector<Batch> batches;
    Slot slots[2];
    cudaStream_t copyStream = nullptr;
    cudaEvent_t evManyStart = nullptr, evManyStop = nullptr;  // device-timed span of one scan / scan_many call
    double lastSpanSeconds = 0;
    PinnedBuf<uint8_t> stage[2];
    cudaEvent_t evStageFree[2] = {};
    std::vector<std::unique_ptr<Ctx>> ctxs;
    int lastCtx = -1;  // context of the most recent scan (sw4_last_scan_all_scores)

    ~Shard() {
        cudaSetDevice(device);
        ctxs.clear();
        for (auto& e : evStageFree)
            if (e) cudaEventDestroy(e);
        if (evManyStart) cudaEventDestroy(evManyStart);
        if (evManyStop) cudaEventDestroy(evManyStop);
        if (copyStream) cudaStreamDestroy(copyStream);
    }
    size_t numLocalBlocks() const { return (n + kShardBlock - 1) / kShardBlock; }
    // position of shard-local subject i in the handle's host arrays
    size_t srcIndex(size_t i) const { return (firstBlock + (i / kShardBlock) * blockStride) * kShardBlock + i % kShardBlock; }
};

// steps (row pairs) between two alignments of a group: ceil(q/2) + G - 1 rounded up to a batch, at least 16 so that
// no lane of a half-warp starts before step 0
// The 256-column class can run as 16 lanes x 16 columns or as 8 lanes x 32 columns on the same pair-blocks (a block is
// 256 consecutive column codes either way). 8 x 32 has 8 fewer fill steps per alignment and half the per-pair hand-over
// work; with the gap scores as immediates it is the faster shape at every query length (1 M x 256: 8.04 vs 7.59 TCUPS),
// so it is the default. SW4_CLASS256_CROSSOVER=q sends queries of q residues and more to 16 x 16 (round 1: 1200).
static inline LengthClass shapeForQuery(const LengthClass& lc, int qlen) {
    static const int crossover = [] { const char* e = getenv("SW4_CLASS256_CROSSOVER"); return e ? atoi(e) : 0x7fffffff; }();
    if (lc.capacity == 256 && !lc.wide && qlen < crossover) return LengthClass{3, 32, 256, false, false};
    return lc;
}

static inline int s16Period(int qlen, int G) { return std::max(16, ((qlen + 1) / 2 + G - 1 + 7) / 8 * 8); }
// the wide variant advances one row per step: q + G - 1 rounded up to 8, at least 32
static inline int s16WidePeriod(int qlen, int G) { return std::max(32, (qlen + G - 1 + 7) / 8 * 8); }

// pssm: nullptr for a sequence query; otherwise the query's [length][21] position-specific scores (the letters then
// only serve the identities of the traceback)
struct QueryRef { const char* letters; int length; const int8_t* pssm = nullptr; };

// the largest entry of a [qlen][21] PSSM, at least 1 (the bound of sw4b200.h)
static inline int pssmMaxEntry(const int8_t* pssm, int qlen) {
    int m = 1;
    for (size_t i = 0; i < (size_t)qlen * 21; i++) m = std::max(m, (int)pssm[i]);
    return m;
}

// Code 20 also pads every subject in the device layouts (pair-blocks, tiles of the exact kernels), and the kernels take
// the maximum over padded columns too. A padded column cannot raise a score or move a first maximum only while it scores
// <= 0 against every query position, which the BLOSUM tables guarantee (their `low`) and a PSSM must state: column 20
// (any other letter) > 0 is refused. `what` names the query in the message.
static inline void checkPssmColumn20(const int8_t* pssm, int qlen, const char* what) {
    for (int p = 0; p < qlen; p++)
        if (pssm[(size_t)p * 21 + 20] > 0)
            fail(SW4_ERR_INVALID, "%s: pssm[%d][20] = %d; the score of residue code 20 (any other letter) must be <= 0", what, p,
                 (int)pssm[(size_t)p * 21 + 20]);
}

// Everything sw4_alignment_coordinates and sw4_alignment_traceback own on the handle's first GPU: it shares nothing with the scan (slots, contexts,
// results), so a scan after the call returns what it would have returned without it.
struct CoordState {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t evStart = nullptr, evStop = nullptr;
    DevBuf<char> dQueryLetters;
    DevBuf<uint8_t> dQueryCodes, dSubjects;
    DevBuf<int8_t> dMatrix;
    DevBuf<CoordGroup> dGroups;
    DevBuf<CoordItem> dItems;
    DevBuf<int2> dBorder;
    DevBuf<int4> dEnds;
    DevBuf<int32_t> dOut;  // [item][5] + error count
    PinnedBuf<char> hQuery;
    PinnedBuf<int8_t> hPssm;  // a PSSM query's table (allocated by the first PSSM query)
    DevBuf<int8_t> dPssm;
    PinnedBuf<uint8_t> hSubjects;
    PinnedBuf<CoordGroup> hGroups;
    PinnedBuf<CoordItem> hItems;
    PinnedBuf<int32_t> hOut;
    // traceback: per-pair rectangles, and the ops, counts and error counters copied back
    DevBuf<TraceItem> dTraceItems;
    PinnedBuf<TraceItem> hTraceItems;
    PinnedBuf<char> hTraceOut;
    // profile construction (sw4_build_pssm): the MSA (apart from the arena), each traced pair's MSA row per chunk, the
    // column statistics, row weights, background tables and the [m][21] result
    DevBuf<uint8_t> dMsa;
    DevBuf<int> dMsaRows, dProfileCounts;
    PinnedBuf<int> hMsaRows;
    DevBuf<int2> dProfileDistinct;
    DevBuf<unsigned long long> dProfileNsum;
    DevBuf<double> dProfileWeights, dProfileTables;  // tables: q_ab / p_b [400], then p_a [20]
    PinnedBuf<double> hProfileTables;
    DevBuf<int8_t> dProfileOut;
    PinnedBuf<int8_t> hProfileOut;

    void create(int dev) {
        device = dev;
        SW4_CUDA(cudaSetDevice(device));
        SW4_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        SW4_CUDA(cudaEventCreate(&evStart));
        SW4_CUDA(cudaEventCreate(&evStop));
        dMatrix.alloc(441);
    }
    ~CoordState() {
        cudaSetDevice(device);
        if (evStart) cudaEventDestroy(evStart);
        if (evStop) cudaEventDestroy(evStop);
        if (stream) cudaStreamDestroy(stream);
    }
};

// The ungapped background of a substitution table M (sw4_build_pssm): p_a from kPseudoCumulative, lambda_u the root of
// sum_{a,b<20} p_a p_b e^(lambda M[a][b]) = 1, bisected in double on [1e-3, 2] until the interval stops shrinking, and
// q_ab = p_a p_b e^(lambda_u M[a][b]) / Z with Z that sum. qOverP[a][b] = q_ab / p_b.
struct ProfileBackground {
    int blosum = 0;  // the table it was computed for (0: none yet)
    double lambda = 0, p[20] = {}, qOverP[400] = {};
    void compute(int id, const int8_t* matrix) {
        for (int a = 0; a < 20; a++) p[a] = (kPseudoCumulative[a] - (a ? kPseudoCumulative[a - 1] : 0)) / 256.0;
        auto sum = [&](double lam) {
            double z = 0;
            for (int a = 0; a < 20; a++)
                for (int b = 0; b < 20; b++) z += p[a] * p[b] * std::exp(lam * matrix[a * 21 + b]);
            return z;
        };
        double lo = 1e-3, hi = 2.0;  // below the root the sum is < 1
        for (;;) {
            const double mid = (lo + hi) / 2;
            if (!(mid > lo && mid < hi)) break;
            (sum(mid) < 1 ? lo : hi) = mid;
        }
        lambda = lo;
        const double z = sum(lambda);
        for (int a = 0; a < 20; a++)
            for (int b = 0; b < 20; b++) qOverP[a * 20 + b] = p[a] * p[b] * std::exp(lambda * matrix[a * 21 + b]) / z / p[b];
        blosum = id;
    }
};

// A pair runs on a CTA of up to 16 warps (one per 512-column tile) when it has this many cells and more than one tile;
// below that one warp per pair, 16 pairs per CTA. One warp needs about 0.3 s for 35 k x 35 k (DESIGN.md 3.2).
constexpr long long kCoordCtaMinCells = 1ll << 24;

struct Engine {
    std::vector<int> deviceIds;
    int numTop = 10;
    int blosum = 62;
    int gop = -11, gex = -1;
    int kernelTypes[4] = {SW4_KERNEL_DPX_S16, SW4_KERNEL_DPX_S16, SW4_KERNEL_DPX_S32, SW4_KERNEL_DPX_S32};
    sw4_mem_config mem{};
    bool verbose = false;
    // development switches
    bool useLongKernel = [] { const char* e = getenv("SW4_NO_LONG_KERNEL"); return !e; }();
    bool useLong2Kernel = [] { const char* e = getenv("SW4_NO_LONG2_KERNEL"); return !e; }();  // two rows per step
    int longMinWarps = [] { const char* e = getenv("SW4_LONG_MIN_WARPS"); return e ? std::max(2, atoi(e)) : 2; }();
    int backfillItems = [] { const char* e = getenv("SW4_BACKFILL_ITEMS"); return e ? std::max(1, atoi(e)) : 2; }();  // C3: 6.77 vs 6.68 TCUPS at 4
    // classes above 512 columns: the multi-segment two-rows-per-step kernel (default) or the older full-warp one-row kernel
    bool twoRowMulti = [] { const char* e = getenv("SW4_NO_TWO_ROW_MULTI"); return !e; }();
    // the long class goes to the CTA-wide array kernel when it has fewer items than this per group of the GPU (latency
    // bound: few very long alignments), else to the multi-segment kernel (throughput bound)
    double longArrayMaxItemsPerGroup = [] { const char* e = getenv("SW4_LONG_ARRAY_ITEMS_PER_GROUP"); return e ? atof(e) : 3.0; }();
    int pipelineDepth = [] { const char* e = getenv("SW4_PIPELINE"); return e ? std::min(kMaxContexts, std::max(1, atoi(e))) : 3; }();
    int shardRank = 0, shardWorld = 1;
    std::unique_ptr<HostDB> db;
    std::vector<std::unique_ptr<Shard>> shards;
    std::unique_ptr<CoordState> coord;  // created by the first sw4_alignment_coordinates / _traceback call
    int8_t matrix[441];
    int maxMatrixEntry = 11;
    std::string lastError;
    std::string lastCigars;  // CIGAR text of the last sw4_alignment_traceback (sw4_last_cigars)
    // score statistics (sw4_set_score_statistics) and, per query of the last scan call, the histogram and its fit
    bool statsEnabled = false;
    double maxEvalue = INFINITY;
    std::vector<std::vector<int64_t>> lastHists;
    std::vector<sw4_score_statistics> lastStats;
    ProfileBackground profileBg;  // of the current table, computed by the first sw4_build_pssm that needs it
    // total timer
    std::chrono::steady_clock::time_point totalStart;
    double totalCells = 0;
    int totalOverflows = 0;

    void buildMatrix() {
        const SubstitutionTriangle* t = nullptr;
        for (const auto& cand : kSubstitutionTriangles)
            if (cand.id == blosum) t = &cand;
        if (!t) fail(SW4_ERR_INVALID, "unsupported substitution matrix blosum%d (45, 50, 62, 80)", blosum);
        maxMatrixEntry = 1;
        for (int r = 0; r < 21; r++)
            for (int c = 0; c < 21; c++) {
                int v = t->low;
                if (r < 20 && c < 20) { const int a = std::max(r, c), b = std::min(r, c); v = t->tri[a * (a + 1) / 2 + b]; }
                matrix[r * 21 + c] = (int8_t)v;
                maxMatrixEntry = std::max(maxMatrixEntry, v);
            }
    }

    void checkGaps() const {
        if (gop > 0 || gex > 0 || gop < -4096 || gex < -4096)
            fail(SW4_ERR_INVALID, "gap scores must be in [-4096, 0] (gop=%d gex=%d)", gop, gex);
    }

    // ---- sharding: interleaved blocks of kShardBlock consecutive subjects of the length-sorted database ----
    // Every shard gets the same length mix (the purpose of the reference's per-partition split, src/cudasw4.cuh:928-1004)
    // and shard-local order is ascending in global id (needed by the tie rule). A pre-sharded database (the caller
    // already holds only its rank's sequences, sw4_set_database_shard_memory) is split among this handle's GPUs only.
    void assignShards() {
        shards.clear();
        const int perHandle = (int)deviceIds.size();
        const bool presharded = db->globalIds != nullptr;
        const size_t totalShards = (size_t)perHandle * (presharded ? 1 : shardWorld);
        const size_t n = db->n;
        const size_t numBlocks = (n + kShardBlock - 1) / kShardBlock;
        for (int d = 0; d < perHandle; d++) {
            auto sh = std::make_unique<Shard>();
            sh->device = deviceIds[d];
            sh->firstBlock = (size_t)(presharded ? 0 : shardRank) * perHandle + d;
            sh->blockStride = totalShards;
            size_t cnt = 0;
            for (size_t b = sh->firstBlock; b < numBlocks; b += totalShards) cnt += std::min<size_t>(kShardBlock, n - b * kShardBlock);
            sh->n = cnt;
            sh->lengths.resize(cnt);
            sh->blockCharPrefix.assign(sh->numLocalBlocks() + 1, 0);
            for (size_t i = 0; i < cnt; i++) {
                const int len = db->lengths[sh->srcIndex(i)];
                sh->lengths[i] = len;
                sh->residues += (uint64_t)len;
                sh->blockCharPrefix[i / kShardBlock + 1] += ((size_t)len + 3) / 4 * 4;
            }
            for (size_t j = 0; j < sh->numLocalBlocks(); j++) sh->blockCharPrefix[j + 1] += sh->blockCharPrefix[j];
            sh->maxLen = cnt ? sh->lengths[cnt - 1] : 0;
            shards.push_back(std::move(sh));
        }
    }
    int32_t globalIdOf(const Shard& sh, size_t i) const {
        const size_t src = sh.srcIndex(i);
        return db->globalIds ? db->globalIds[src] : (int32_t)src;
    }

    // ---- batch layout ----
    // Upper bound of the arena bytes a batch over local subjects [first, end) needs (first, end multiples of kShardBlock
    // or end == n). The multi-segment class pads every pair to whole 1024-column segments of its longer subject; with
    // sorted lengths the sum of (longer - shorter) over consecutive pairs telescopes to at most the longest length.
    size_t arenaBound(const Shard& sh, size_t first, size_t end) const {
        const size_t chars = sh.blockCharPrefix[(end + kShardBlock - 1) / kShardBlock] - sh.blockCharPrefix[first / kShardBlock];
        size_t bytes = alignUp(chars + 16, 256) + alignUp((end - first + 1) * sizeof(size_t), 256);
        const int32_t* L = sh.lengths.data();
        size_t pos = std::upper_bound(L + first, L + end, 0) - L;
        for (int c = 0; c < kNumLengthClasses && pos < end; c++) {
            const LengthClass& lc = kLengthClasses[c];
            const size_t e = lc.multi ? end : (size_t)(std::upper_bound(L + pos, L + end, lc.capacity) - L);
            if (e > pos) {
                const size_t pairs = (e - pos + 1) / 2;
                if (!lc.multi) {
                    bytes += alignUp(pairs * (size_t)lc.capacity * 2, 256) + alignUp(pairs * sizeof(S16Item), 256);
                } else {
                    const size_t multiChars = sh.blockCharPrefix[(end + kShardBlock - 1) / kShardBlock] - sh.blockCharPrefix[pos / kShardBlock];
                    const size_t cols = multiChars + 2 * (size_t)lc.capacity * pairs + (size_t)L[end - 1] + lc.capacity;
                    bytes += alignUp(cols * 2, 256) + alignUp(pairs * sizeof(S16Item), 256) + alignUp((cols / lc.capacity + pairs) * 4, 256);
                }
            }
            pos = std::max(pos, e);
        }
        return bytes;
    }

    Batch makeBatch(const Shard& sh, size_t first, size_t end) const {
        Batch b;
        b.first = first;
        b.count = end - first;
        b.charsBytes = sh.blockCharPrefix[(end + kShardBlock - 1) / kShardBlock] - sh.blockCharPrefix[first / kShardBlock];
        size_t off = alignUp(b.charsBytes + 16, 256);
        b.offsetsOff = off;
        off += alignUp((b.count + 1) * sizeof(size_t), 256);
        const int32_t* L = sh.lengths.data();
        size_t pos = std::upper_bound(L + first, L + end, 0) - L;
        b.numZeroLength = pos - first;
        for (int c = 0; c < kNumLengthClasses && pos < end; c++) {
            const LengthClass& lc = kLengthClasses[c];
            const size_t e = lc.multi ? end : (size_t)(std::upper_bound(L + pos, L + end, lc.capacity) - L);
            if (e > pos) {
                BatchClass bc;
                bc.cls = c;
                bc.first = (int)pos;
                bc.count = (int)(e - pos);
                bc.numItems = (bc.count + 1) / 2;
                bc.numBlocks = bc.numItems;
                if (lc.multi) {
                    bc.hostItems.reserve(bc.numItems);
                    for (size_t i = pos; i < e; i += 2) {
                        S16Item it;
                        it.subject0 = (int)i;
                        it.subject1 = (i + 1 < e) ? (int)(i + 1) : -1;
                        const int maxLen = std::max(L[i], (i + 1 < e) ? L[i + 1] : 0);
                        it.numSegments = (maxLen + lc.capacity - 1) / lc.capacity;
                        it.firstBlock = 0;
                        bc.hostItems.push_back(it);
                    }
                    std::reverse(bc.hostItems.begin(), bc.hostItems.end());  // longest first: they bound the makespan
                    int blk = 0;
                    for (size_t k = 0; k < bc.hostItems.size(); k++) {
                        bc.hostItems[k].firstBlock = blk;
                        for (int sgm = 0; sgm < bc.hostItems[k].numSegments; sgm++) bc.hostBlockItem.push_back((int32_t)k);
                        blk += bc.hostItems[k].numSegments;
                    }
                    bc.numBlocks = blk;
                }
                bc.colsOff = off;
                off += alignUp((size_t)bc.numBlocks * lc.capacity * 2, 256);
                bc.itemsOff = off;
                off += alignUp((size_t)bc.numItems * sizeof(S16Item), 256);
                if (lc.multi) { bc.blockItemOff = off; off += alignUp((size_t)bc.numBlocks * 4, 256); }
                b.classes.push_back(std::move(bc));
            }
            pos = std::max(pos, e);
        }
        b.arenaBytes = off;
        return b;
    }

    void initShardDevice(Shard& sh) {
        SW4_CUDA(cudaSetDevice(sh.device));
        cudaDeviceProp prop;
        SW4_CUDA(cudaGetDeviceProperties(&prop, sh.device));
        if (prop.major < 10)
            fail(SW4_ERR_CUDA, "device %d (%s, sm_%d%d) cannot run this library: it is built for sm_100a only", sh.device, prop.name,
                 prop.major, prop.minor);
        sh.smCount = prop.multiProcessorCount;
        if (!sh.copyStream) {
            SW4_CUDA(cudaStreamCreateWithFlags(&sh.copyStream, cudaStreamNonBlocking));
            SW4_CUDA(cudaEventCreate(&sh.evManyStart));
            SW4_CUDA(cudaEventCreate(&sh.evManyStop));
            for (auto& e : sh.evStageFree) SW4_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            for (auto& sl : sh.slots) SW4_CUDA(cudaEventCreateWithFlags(&sl.evReady, cudaEventDisableTiming));
        }
    }

    // Decide between the resident layout (one batch) and streaming (batches through two slots) and allocate.
    // max_gpu_mem bounds the database-related device memory of a GPU (slots + the per-subject length / id arrays);
    // the per-query scratch is bounded separately (max_temp_bytes for the border rows).
    void planShard(Shard& sh) {
        initShardDevice(sh);
        size_t freeB = 0, totalB = 0;
        SW4_CUDA(cudaMemGetInfo(&freeB, &totalB));
        sh.deviceFree = freeB;
        const size_t n = sh.n;
        const size_t perSubject = n * 2 * sizeof(int32_t);
        // keep room for the query contexts (scores + overflow list per subject, profile, border rows) and the runtime
        const size_t reserve = ((size_t)1 << 30) + (size_t)pipelineDepth * (n * 8 + ((size_t)256 << 20));
        const size_t usable = freeB > reserve ? freeB - reserve : 0;
        const size_t budget = std::min(usable, mem.max_gpu_mem);
        sh.batches.clear();
        const size_t whole = arenaBound(sh, 0, n);
        if (perSubject + whole <= budget) {
            sh.streaming = false;
            sh.batches.push_back(makeBatch(sh, 0, n));
        } else {
            sh.streaming = true;
            if (budget <= perSubject + ((size_t)64 << 10))
                fail(SW4_ERR_NOMEM, "device %d: %zu MiB usable for the database (max_gpu_mem), the per-sequence arrays alone need %zu MiB",
                     sh.device, budget >> 20, perSubject >> 20);
            const size_t slotBytes = (budget - perSubject) / 2;
            size_t first = 0;
            while (first < n) {
                // largest end (multiple of kShardBlock, or n) whose arena bound fits a slot
                size_t lo = first / kShardBlock + 1, hi = sh.numLocalBlocks();
                auto endOf = [&](size_t blk) { return std::min(n, blk * (size_t)kShardBlock); };
                if (arenaBound(sh, first, endOf(lo)) > slotBytes)
                    fail(SW4_ERR_NOMEM, "device %d: a block of %d sequences around local index %zu (longest %d residues) does not fit a "
                         "streaming slot of %zu MiB; raise max_gpu_mem", sh.device, kShardBlock, first, sh.lengths[endOf(lo) - 1], slotBytes >> 20);
                while (lo < hi) {
                    const size_t mid = (lo + hi + 1) / 2;
                    if (arenaBound(sh, first, endOf(mid)) <= slotBytes) lo = mid; else hi = mid - 1;
                }
                sh.batches.push_back(makeBatch(sh, first, endOf(lo)));
                first = endOf(lo);
            }
            if (n == 0) sh.batches.push_back(makeBatch(sh, 0, 0));
        }
        size_t maxArena = 0;
        sh.hasMulti = false;
        for (const Batch& b : sh.batches) {
            maxArena = std::max(maxArena, b.arenaBytes);
            for (const BatchClass& bc : b.classes) sh.hasMulti |= kLengthClasses[bc.cls].multi;
        }
        const int numSlots = sh.streaming && sh.batches.size() > 1 ? 2 : 1;
        for (int s = 0; s < numSlots; s++) { sh.slots[s].arena.alloc(maxArena + 256); sh.slots[s].batch = -1; }
        if (verbose)
            fprintf(stderr, "[sw4] device %d: %zu subjects, %llu residues, %s, %zu batch(es), slot %zu MiB\n", sh.device, n,
                    (unsigned long long)sh.residues, sh.streaming ? "streaming" : "resident", sh.batches.size(), maxArena >> 20);
    }

    // Copy batch `bi` into slot `si` and build its kernel-ready layout there; everything is enqueued on sh.copyStream
    // (the host only blocks on the pinned staging buffers). Records slot.evReady.
    void stageBatch(Shard& sh, int bi, int si) {
        Batch& b = sh.batches[bi];
        Slot& slot = sh.slots[si];
        cudaStream_t cs = sh.copyStream;
        uint8_t* arena = slot.arena.p;
        // local offsets of the batch (padded to 4)
        std::vector<size_t> offsets(b.count + 1);
        offsets[0] = 0;
        for (size_t i = 0; i < b.count; i++) offsets[i + 1] = offsets[i] + ((size_t)sh.lengths[b.first + i] + 3) / 4 * 4;
        // residues through two pinned staging buffers, gathered by host threads (a block of kShardBlock consecutive
        // sequences is one memcpy when the caller's offsets are tight, as makedb writes them)
        const int nt = (int)std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
        size_t i0 = 0;
        int chunk = 0;
        while (i0 < b.count) {
            size_t i1 = i0;
            while (i1 < b.count && offsets[std::min(b.count, i1 + kShardBlock)] - offsets[i0] <= kStageChunkBytes) i1 = std::min(b.count, i1 + kShardBlock);
            if (i1 == i0) i1 = std::min(b.count, i0 + kShardBlock);  // one oversized block: the staging buffer grows below
            const size_t bytes = offsets[i1] - offsets[i0];
            const int p = chunk & 1;
            SW4_CUDA(cudaEventSynchronize(sh.evStageFree[p]));
            sh.stage[p].ensure(std::max(bytes, kStageChunkBytes));
            uint8_t* dst = sh.stage[p].p;
            const size_t blocks = (i1 - i0 + kShardBlock - 1) / kShardBlock;
            auto work = [&](int t) {
                for (size_t blk = (size_t)t; blk < blocks; blk += (size_t)nt) {
                    const size_t a = i0 + blk * kShardBlock, e = std::min(i1, a + kShardBlock);
                    const size_t srcA = sh.srcIndex(b.first + a);
                    bool tight = true;  // the caller's layout of this block equals ours (every sequence padded to 4)
                    for (size_t i = a; i < e && tight; i++)
                        tight = db->offsets[srcA + (i - a) + 1] - db->offsets[srcA + (i - a)] == offsets[i + 1] - offsets[i];
                    if (tight) {
                        memcpy(dst + (offsets[a] - offsets[i0]), db->chars + db->offsets[srcA], offsets[e] - offsets[a]);
                    } else {
                        for (size_t i = a; i < e; i++)
                            memcpy(dst + (offsets[i] - offsets[i0]), db->chars + db->offsets[srcA + (i - a)], (size_t)sh.lengths[b.first + i]);
                    }
                }
            };
            if (blocks < 8 || nt == 1) { work(0); if (nt > 1) for (int t = 1; t < nt; t++) work(t); }
            else {
                std::vector<std::thread> th;
                for (int t = 1; t < nt; t++) th.emplace_back(work, t);
                work(0);
                for (auto& t : th) t.join();
            }
            SW4_CUDA(cudaMemcpyAsync(arena + offsets[i0], dst, bytes, cudaMemcpyHostToDevice, cs));
            SW4_CUDA(cudaEventRecord(sh.evStageFree[p], cs));
            i0 = i1;
            chunk++;
        }
        size_t* dOffsets = reinterpret_cast<size_t*>(arena + b.offsetsOff);
        SW4_CUDA(cudaMemcpyAsync(dOffsets, offsets.data(), (b.count + 1) * sizeof(size_t), cudaMemcpyHostToDevice, cs));
        if (b.count) {
            const size_t words = (b.charsBytes + 3) / 4;
            if (words) sanitize_codes_kernel<<<(unsigned)((words + 255) / 256), 256, 0, cs>>>(reinterpret_cast<uint32_t*>(arena), words);
            pad_codes_kernel<<<(unsigned)((b.count + 255) / 256), 256, 0, cs>>>(arena, dOffsets, sh.dLengths.p + b.first, (int)b.count);
        }
        // the items index subjects by shard-local index: shift the offsets pointer accordingly
        const size_t* offsetsBySubject = dOffsets - b.first;
        for (BatchClass& bc : b.classes) {
            const LengthClass& lc = kLengthClasses[bc.cls];
            PairItem* dItems = reinterpret_cast<PairItem*>(arena + bc.itemsOff);
            const int32_t* dBlockItem = nullptr;
            if (lc.multi) {
                SW4_CUDA(cudaMemcpyAsync(dItems, bc.hostItems.data(), bc.hostItems.size() * sizeof(S16Item), cudaMemcpyHostToDevice, cs));
                SW4_CUDA(cudaMemcpyAsync(arena + bc.blockItemOff, bc.hostBlockItem.data(), bc.hostBlockItem.size() * 4, cudaMemcpyHostToDevice, cs));
                dBlockItem = reinterpret_cast<const int32_t*>(arena + bc.blockItemOff);
            } else {
                make_pair_items_kernel<<<(bc.numItems + 255) / 256, 256, 0, cs>>>(dItems, bc.numItems, bc.first, bc.count);
            }
            const long long total = (long long)bc.numBlocks * (lc.capacity / 4);
            build_pair_blocks_kernel<<<(unsigned)((total + 255) / 256), 256, 0, cs>>>(
                arena, offsetsBySubject, sh.dLengths.p, dItems, dBlockItem, bc.numBlocks, lc.capacity,
                reinterpret_cast<uint16_t*>(arena + bc.colsOff));
        }
        SW4_CUDA(cudaGetLastError());
        SW4_CUDA(cudaEventRecord(slot.evReady, cs));
        slot.batch = bi;
    }

    void uploadShard(Shard& sh) {
        planShard(sh);
        const size_t n = sh.n;
        sh.dLengths.alloc(n);
        sh.dGlobalIds.alloc(n);
        SW4_CUDA(cudaMemcpyAsync(sh.dLengths.p, sh.lengths.data(), n * sizeof(int32_t), cudaMemcpyHostToDevice, sh.copyStream));
        {
            std::vector<int32_t> ids(std::min<size_t>(n, (size_t)1 << 22));
            for (size_t base = 0; base < n; base += ids.size()) {
                const size_t m = std::min(ids.size(), n - base);
                for (size_t i = 0; i < m; i++) ids[i] = globalIdOf(sh, base + i);
                SW4_CUDA(cudaMemcpyAsync(sh.dGlobalIds.p + base, ids.data(), m * sizeof(int32_t), cudaMemcpyHostToDevice, sh.copyStream));
                SW4_CUDA(cudaStreamSynchronize(sh.copyStream));  // `ids` is reused
            }
        }
        sh.ctxs.clear();
        sh.lastCtx = -1;
        if (!sh.streaming) stageBatch(sh, 0, 0);
        SW4_CUDA(cudaStreamSynchronize(sh.copyStream));
        sh.uploaded = true;
    }

    void upload() {
        if (!db) fail(SW4_ERR_INVALID, "no database set");
        bool fresh = false;
        for (auto& sh : shards)
            if (!sh->uploaded) { uploadShard(*sh); fresh = true; }
        if (fresh) {  // untimed warm-up scan: loads every kernel this database will launch and sizes the scratch buffers
            std::string warm;
            for (int i = 0; i < 320; i++) warm.push_back("ARNDCQEGHILKMFPSTWYV"[(i * 7) % 20]);
            // (as many copies as queries can be in flight, so that every context exists before the first timed scan)
            std::vector<QueryRef> q((size_t)pipelineDepth, QueryRef{warm.data(), (int)warm.size()});
            const int k = (int)std::min<size_t>((size_t)std::max(numTop, 1), std::min<size_t>(std::max<size_t>(db->nGlobal, 1), 16));
            std::vector<std::vector<ShardResult>> res;
            runAllShards(q.data(), (int)q.size(), k, res);
        }
    }

    int statThreshold() const { return kernelTypes[0] == SW4_KERNEL_HALF2 ? kHalf2Threshold : kS16OverflowThreshold; }

    Ctx& context(Shard& sh, int c) {
        while ((int)sh.ctxs.size() <= c) {
            auto ctx = std::make_unique<Ctx>();
            ctx->create();
            sh.ctxs.push_back(std::move(ctx));
        }
        return *sh.ctxs[c];
    }

    // The query capacity a context grows to for a qlen-residue query (from `current`, 0 for a new context), by doubling.
    static int queryCapacityFor(int qlen, int current) {
        int cap = std::max(current, 8192);
        while (cap < qlen) cap *= 2;
        return cap;
    }
    static size_t borderStrideFor(int cap) { return (size_t)(cap + 31) / 32 * 32 + 128; }
    // Every scan needs at least kS16Warps border row arrays of its context's capacity within max_temp_bytes. Contexts are
    // recreated when the memory configuration changes, so a query that passes at its own capacity,
    // queryCapacityFor(qlen, 0), passes in any context that a later query of the same call grows.
    void checkBorderRows(int cap, int qlen) const {
        const size_t stride = borderStrideFor(cap);
        if (mem.max_temp_bytes / (stride * sizeof(uint2)) < (size_t)kS16Warps)
            fail(SW4_ERR_NOMEM, "max_temp_bytes (%zu MiB) cannot hold the border rows of a %d-residue query (%zu MiB needed at least)",
                 mem.max_temp_bytes >> 20, qlen, (kS16Warps * stride * sizeof(uint2)) >> 20);
    }

    // All device scratch of a context is sized here, BEFORE the timed region, for a query capacity that only grows by
    // doubling: cudaMalloc/cudaFree inside the event-bracketed region stall the stream for up to hundreds of ms.
    void ensureCtx(Shard& sh, Ctx& ctx, int qlen, int k, bool pssm, bool stats) {
        if ((size_t)qlen > ctx.hQuery.n) ctx.hQuery.ensure(std::max<size_t>((size_t)qlen * 2, 65536));
        const size_t topWords = (size_t)2 * k + 8;
        if (topWords > ctx.hTop.n) ctx.hTop.ensure(topWords + 64);
        if (ctx.dScores.n < std::max<size_t>(sh.n, 1)) { ctx.dScores.alloc(sh.n); ctx.dOvfList.alloc(sh.n); }
        if (qlen > ctx.queryCapacity || (size_t)k > ctx.topCapacity) {
            SW4_CUDA(cudaStreamSynchronize(ctx.stream));
            const int cap = queryCapacityFor(qlen, ctx.queryCapacity);
            ctx.queryCapacity = cap;
            ctx.topCapacity = std::max(ctx.topCapacity, (size_t)std::max(k, 64));
            const size_t capStride = (size_t)(cap + 96 + 31) / 32 * 32;
            ctx.dQueryLetters.ensure((size_t)cap + 16);
            ctx.dQueryCodes.ensure((size_t)cap + 16);
            ctx.dProfile.ensure((size_t)kProfileRows * capStride);
            ctx.dTopScores.ensure(ctx.topCapacity);
            ctx.dTopIds.ensure(ctx.topCapacity);
            if (topk_uses_large_path(k)) {
                ctx.dTopkWork.ensure(topk_large_work_ints());
                ctx.dTopkKeys.ensure((size_t)topk_large_num_keys(k));
            }
            // border rows of the long-subject kernels: one row array per warp (one-warp-per-pair kernels) or per CTA (array
            // kernels); the kernels of one scan that use them run one after the other, so they share one buffer. Its
            // size is bounded by max_temp_bytes: fewer row arrays = fewer CTAs on those kernels.
            // (one row array = cap + 128 (H, E) pairs; the two-row multi-segment kernel keeps one per GROUP, two per warp, as
            // cap / 2 + 64 entries of both rows of a step)
            checkBorderRows(cap, qlen);
            ctx.borderStride = borderStrideFor(cap);
            const bool needBorder = sh.maxLen > 512;
            const size_t groupsPerCta = (size_t)kS16Warps * 2;
            size_t rows = needBorder ? (size_t)sh.smCount * (groupsPerCta + kS16Warps) : (size_t)kS16Warps;
            const size_t maxRows = mem.max_temp_bytes / (ctx.borderStride * sizeof(uint2));
            rows = std::min(rows, maxRows / kS16Warps * kS16Warps);
            // two thirds for the slots of the multi-segment kernels (none when the budget is that small: those classes
            // then fall back to the one-warp-per-pair kernel)
            ctx.borderSlots = needBorder ? (int)std::min<size_t>((size_t)sh.smCount, rows * 2 / 3 / groupsPerCta) : 0;
            ctx.borderRowArrays = rows - (size_t)ctx.borderSlots * groupsPerCta;
            ctx.dBorder.ensure(rows * ctx.borderStride);
            // test hook: border rows full of large positive scores make any read of a stale entry show up in the results
            if (getenv("SW4_DEBUG_POISON_BORDER")) SW4_CUDA(cudaMemset(ctx.dBorder.p, 0x7f, ctx.dBorder.bytes()));
            ctx.borderB = ctx.dBorder.p + (size_t)ctx.borderSlots * groupsPerCta * ctx.borderStride;
            ctx.dBorderSlots.ensure((size_t)std::max(ctx.borderSlots, 1));
        }
        if (pssm && ctx.dPssm.n < (size_t)ctx.queryCapacity * 21) {
            SW4_CUDA(cudaStreamSynchronize(ctx.stream));
            ctx.hPssm.ensure((size_t)ctx.queryCapacity * 21);
            ctx.dPssm.alloc((size_t)ctx.queryCapacity * 21);
        }
        if (stats && !ctx.dHist.p) {
            ctx.dHist.alloc(2 * kHistEntries);
            ctx.hHist.ensure(2 * kHistEntries);
        }
    }

    // ---- one query on one shard, part 1: query upload, profile, score reset (enqueued on ctx.stream) ----
    void enqueuePrologue(Shard& sh, Ctx& ctx, const QueryRef& q, int queryIndex, int k) {
        const int qlen = q.length;
        ensureCtx(sh, ctx, qlen, k, q.pssm != nullptr, statsEnabled);
        ctx.busy = true;
        ctx.queryIndex = queryIndex;
        ctx.qlen = qlen;
        ctx.k = k;
        ctx.launches = 0;
        ctx.pssm = q.pssm != nullptr;
        ctx.stats = statsEnabled;
        ctx.maxEntry = ctx.pssm ? pssmMaxEntry(q.pssm, qlen) : maxMatrixEntry;
        const int qpad = (qlen + 3) / 4 * 4;
        // rows of the positional profile start on 128-byte lines: the ring refill copies 64 contiguous bytes per row, which
        // then always fall into two sectors of one line (a stride of 4 mod 8 words cost 3-4 % on the peak benchmark)
        ctx.profStride = (qlen + 96 + 31) / 32 * 32;  // (the two-row array kernel reads up to q + 80 gap rows)
        cudaStream_t st = ctx.stream;
        SW4_CUDA(cudaEventRecord(ctx.evStart, st));
        if (ctx.pssm) {
            // the scan reads only the profile: the letters of a PSSM query are not needed
            if (qlen) {
                memcpy(ctx.hPssm.p, q.pssm, (size_t)qlen * 21);
                SW4_CUDA(cudaMemcpyAsync(ctx.dPssm.p, ctx.hPssm.p, (size_t)qlen * 21, cudaMemcpyHostToDevice, st));
            }
        } else {
            if (qlen) memcpy(ctx.hQuery.p, q.letters, (size_t)qlen);
            if (qlen) SW4_CUDA(cudaMemcpyAsync(ctx.dQueryLetters.p, ctx.hQuery.p, (size_t)qlen, cudaMemcpyHostToDevice, st));
            SW4_CUDA(cudaMemcpyAsync(ctx.dMatrix.p, matrix, 441, cudaMemcpyHostToDevice, st));
        }
        SW4_CUDA(cudaMemsetAsync(ctx.dCounters.p, 0, kNumCounters * sizeof(int), st));
        if (ctx.borderSlots) SW4_CUDA(cudaMemsetAsync(ctx.dBorderSlots.p, 0, (size_t)ctx.borderSlots * sizeof(int), st));
        // every scan starts from "-1 = not scored" so that a subject the kernels missed can never keep an old score;
        // empty subjects (and everything, for an empty query) score 0 by definition
        SW4_CUDA(cudaMemsetAsync(ctx.dScores.p, qlen == 0 ? 0 : 0xff, std::max<size_t>(sh.n, 1) * sizeof(int32_t), st));
        const size_t numZero = std::upper_bound(sh.lengths.begin(), sh.lengths.end(), 0) - sh.lengths.begin();
        if (qlen > 0 && numZero) SW4_CUDA(cudaMemsetAsync(ctx.dScores.p, 0, numZero * sizeof(int32_t), st));
        const dim3 profGrid((ctx.profStride + 127) / 128, kProfileRows);
        if (ctx.pssm) {
            build_profile_pssm_kernel<<<profGrid, 128, 0, st>>>(ctx.dPssm.p, qlen, ctx.dProfile.p, ctx.profStride);
        } else {
            if (qpad > 0) {
                convert_query_kernel<<<(qpad + 255) / 256, 256, 0, st>>>(ctx.dQueryLetters.p, ctx.dQueryCodes.p, qlen, qpad);
                ctx.launches++;
            }
            build_profile_kernel<<<profGrid, 128, 0, st>>>(ctx.dQueryCodes.p, qlen, ctx.dMatrix.p, ctx.dProfile.p, ctx.profStride);
        }
        SW4_CUDA(cudaGetLastError());
        ctx.launches++;
        SW4_CUDA(cudaEventRecord(ctx.evK0, st));
    }

    // ---- part 2: the score kernels of one batch (the whole shard when it is resident) ----
    // All length classes run CONCURRENTLY: every non-empty class is launched at (up to) full width, longest subjects
    // first, on its own stream; one CTA fits per SM, so a later class's CTAs (and the next query's) start as earlier
    // CTAs retire and the dynamic tickets even out the rest. No SM goes idle before the last class runs dry.
    // (The reference: 36 launches over 10 streams per query, src/cudasw4.cuh:1745-2103.)
    void enqueueBatch(Shard& sh, Ctx& ctx, int bi, int si, bool firstBatch) {
        Batch& b = sh.batches[bi];
        Slot& slot = sh.slots[si];
        cudaStream_t st = ctx.stream;
        const int qlen = ctx.qlen;
        if (sh.streaming) SW4_CUDA(cudaStreamWaitEvent(st, slot.evReady, 0));
        if (qlen > 0 && !b.classes.empty()) {
            if (!firstBatch) {  // tickets and the overflow list start from zero for every batch; [1] (statistics) accumulates
                SW4_CUDA(cudaMemsetAsync(ctx.dCounters.p, 0, sizeof(int), st));
                SW4_CUDA(cudaMemsetAsync(ctx.dCounters.p + 2, 0, 2 * sizeof(int), st));
                SW4_CUDA(cudaMemsetAsync(ctx.dCounters.p + 8, 0, 32 * sizeof(int), st));
            }
            uint8_t* arena = slot.arena.p;
            const size_t* offsetsBySubject = reinterpret_cast<const size_t*>(arena + b.offsetsOff) - b.first;
            const int profStride = ctx.profStride;
            const uint32_t gop2 = ((uint32_t)(uint16_t)(int16_t)gop << 16) | (uint16_t)(int16_t)gop;
            const uint32_t gex2 = ((uint32_t)(uint16_t)(int16_t)gex << 16) | (uint16_t)(int16_t)gex;
            const int numClasses = (int)b.classes.size();
            const int width = sh.smCount >= 2 ? (sh.smCount & ~1) : 1;
            SW4_CUDA(cudaEventRecord(ctx.evFork, st));
            for (int ci = numClasses - 1; ci >= 0; ci--) {
                const BatchClass& cl = b.classes[ci];
                const LengthClass lc = shapeForQuery(kLengthClasses[cl.cls], qlen);
                const int G = 1 << lc.logG;
                const int groupsPerCta = kS16Warps * (32 >> lc.logG);
                int grid = (cl.numItems + groupsPerCta * backfillItems - 1) / (groupsPerCta * backfillItems);
                grid = std::max(1, std::min(width, grid));
                if (grid > 1) grid = (grid + 1) & ~1;
                grid = std::min(grid, width);
                if (lc.multi) grid = std::max(1, std::min<int>(grid, (int)(ctx.borderRowArrays / kS16Warps)));
                cudaStream_t cst = ctx.classStreams[ci % kMaxClassStreams];
                SW4_CUDA(cudaStreamWaitEvent(cst, ctx.evFork, 0));
                const int activeGroups = std::min(groupsPerCta, std::max(1, (cl.numItems + grid - 1) / grid));
                const uint16_t* cols = reinterpret_cast<const uint16_t*>(arena + cl.colsOff);
                const S16Item* items = reinterpret_cast<const S16Item*>(arena + cl.itemsOff);
                auto fillCommon = [&](auto& prm) {
                    prm.cols = cols;
                    prm.items = items;
                    prm.numItems = cl.numItems;
                    prm.ticket = ctx.dCounters.p + 8 + cl.cls;
                    prm.logG = lc.logG;
                    prm.profile = ctx.dProfile.p;
                    prm.profStride = profStride;
                    prm.qlen = qlen;
                    prm.gop2 = gop2;
                    prm.gex2 = gex2;
                    prm.ovfThreshold = kS16OverflowThreshold;
                    prm.statThreshold = (lc.capacity > 240) ? statThreshold() : 0x7fffffff;
                    prm.scores = ctx.dScores.p;
                    prm.ovfList = ctx.dOvfList.p;
                    prm.ovfCount = ctx.dCounters.p + 0;
                    prm.statCount = ctx.dCounters.p + 1;
                    prm.elapsedNs = ctx.dClassNs.p;
                    prm.activeGroups = activeGroups;
                };
                // the long class runs on the CTA-wide array kernel when the query is long enough to keep at least two warps of
                // an array busy (kernels_s16_long.cuh) AND the class is too small to fill the GPU's groups a few times over
                int longWarps = 0;
                const int p0 = (qlen + 32 + 15) / 16 * 16;
                if (lc.multi && useLongKernel) {
                    longWarps = kLongMaxWarps;
                    while (longWarps > 1 && kLongLag * longWarps + 64 > p0) longWarps >>= 1;
                    if (longWarps < longMinWarps) longWarps = 0;
                    if (longWarps && twoRowMulti && cl.numItems > longArrayMaxItemsPerGroup * sh.smCount * kS16Warps * 2) longWarps = 0;
                }
                // The two-rows-per-step form of the array kernel (kernels_s16_long2.cuh) has 20 % fewer instructions per cell but
                // fits at most 8 warps - and only half as many as the one-row form at a given query length - into an array.
                // It wins whenever that does not cost array width (measured on C5, per query: +9..+12 % at W = 8 vs 8 or 16,
                // +9 % at 4 vs 4; -28 % at 4 vs 8, -43 % at 2 vs 4), unless there are too few items to keep its 2 x 148
                // arrays of 8 warps busy (then the 16-warp array finishes the few long alignments sooner).
                int long2Period = 0;
                int long2Warps = (longWarps && useLong2Kernel) ? s16_long2_warps(qlen, &long2Period) : 0;
                if (long2Warps < std::min(longWarps, kLong2MaxW) || qlen < 256) long2Warps = 0;
                if (long2Warps && longWarps > kLong2MaxW && cl.numItems < 2 * sh.smCount) long2Warps = 0;
                if (long2Warps) {
                    S16Long2Params lp{};
                    lp.cols = cols;
                    lp.items = items;
                    lp.lengths = sh.dLengths.p;
                    lp.numItems = cl.numItems;
                    lp.ticket = ctx.dCounters.p + 8 + cl.cls;
                    lp.warps = long2Warps;
                    lp.ringSlots = s16_long2_ring_slots(long2Warps);
                    lp.profLo = ctx.dProfile.p + (size_t)kFused * profStride;
                    lp.profHi = ctx.dProfile.p + (size_t)(kFused + 21) * profStride;
                    lp.profStride = profStride;
                    lp.qlen = qlen;
                    lp.period = long2Period;
                    lp.gop2 = gop2;
                    lp.gex2 = gex2;
                    lp.ovfThreshold = kS16OverflowThreshold;
                    lp.statThreshold = statThreshold();
                    lp.scores = ctx.dScores.p;
                    lp.ovfList = ctx.dOvfList.p;
                    lp.ovfCount = ctx.dCounters.p + 0;
                    lp.statCount = ctx.dCounters.p + 1;
                    lp.border = reinterpret_cast<uint4*>(ctx.borderB);
                    lp.borderStride = (int)(ctx.borderStride / 2);
                    const int arrays = kLong2Warps / long2Warps;
                    int g = std::max(1, std::min(sh.smCount, (cl.numItems + arrays - 1) / arrays));
                    g = std::max(1, (int)std::min<size_t>((size_t)g, ctx.borderRowArrays / arrays));
                    SW4_CUDA(launch_s16_long2(lp, g, cst));
                    ctx.launches++;
                    SW4_CUDA(cudaEventRecord(ctx.evJoin[ci % kMaxClassStreams], cst));
                    SW4_CUDA(cudaStreamWaitEvent(st, ctx.evJoin[ci % kMaxClassStreams], 0));
                    continue;
                }
                if (longWarps) {
                    S16LongParams lp{};
                    lp.cols = cols;
                    lp.items = items;
                    lp.lengths = sh.dLengths.p;
                    lp.numItems = cl.numItems;
                    lp.ticket = ctx.dCounters.p + 8 + cl.cls;
                    lp.warps = longWarps;
                    lp.ringSlots = s16_long_ring_slots(longWarps);
                    lp.profLo = ctx.dProfile.p + (size_t)kFused * profStride;
                    lp.profHi = ctx.dProfile.p + (size_t)(kFused + 21) * profStride;
                    lp.profStride = profStride;
                    lp.qlen = qlen;
                    lp.period = p0;
                    lp.gop2 = gop2;
                    lp.gex2 = gex2;
                    lp.ovfThreshold = kS16OverflowThreshold;
                    lp.statThreshold = statThreshold();
                    lp.scores = ctx.dScores.p;
                    lp.ovfList = ctx.dOvfList.p;
                    lp.ovfCount = ctx.dCounters.p + 0;
                    lp.statCount = ctx.dCounters.p + 1;
                    lp.elapsedNs = ctx.dClassNs.p;
                    lp.border = ctx.borderB;
                    lp.borderStride = (int)ctx.borderStride;
                    const int smemBytes = s16_long_smem_bytes(longWarps);
                    const int ctasPerSm = std::max(1, std::min(kLongMaxWarps / longWarps, (227 * 1024) / (smemBytes + 1024)));
                    int g = std::max(1, std::min(cl.numItems, std::min(sh.smCount * ctasPerSm, sh.smCount * 8)));
                    g = (int)std::min<size_t>((size_t)g, ctx.borderRowArrays);
                    SW4_CUDA(launch_s16_long(lp, g, cst));
                    ctx.launches++;
                    SW4_CUDA(cudaEventRecord(ctx.evJoin[ci % kMaxClassStreams], cst));
                    SW4_CUDA(cudaStreamWaitEvent(st, ctx.evJoin[ci % kMaxClassStreams], 0));
                    continue;
                }
                // classes above 512 columns (576..1024 and the long class): the two-rows-per-step kernel over 16 x R-column
                // segments, the border column handed from segment to segment (kernels_s16.cuh, MULTI)
                const bool segmented = lc.wide && twoRowMulti && ctx.borderSlots > 0;
                S16Params narrow{};
                S16WideParams wide{};
                if (segmented) {
                    const int groupsPerCta2 = kS16Warps * 2;
                    grid = (cl.numItems + groupsPerCta2 * backfillItems - 1) / (groupsPerCta2 * backfillItems);
                    grid = std::max(1, std::min(width, grid));
                    if (grid > 1) grid = (grid + 1) & ~1;
                    grid = std::max(1, std::min(grid, width));
                    fillCommon(narrow);
                    narrow.logG = 4;
                    narrow.activeGroups = std::min(groupsPerCta2, std::max(1, (cl.numItems + grid - 1) / grid));
                    narrow.period = std::max(32, s16Period(qlen, 16));
                    narrow.statThreshold = statThreshold();
                    narrow.lengths = sh.dLengths.p;
                    narrow.border = reinterpret_cast<uint4*>(ctx.dBorder.p);
                    narrow.borderStride = (int)(ctx.borderStride / 2);
                    narrow.borderSlots = ctx.dBorderSlots.p;
                    narrow.numBorderSlots = ctx.borderSlots;
                    narrow.blockScale = 2;
                } else if (lc.wide) {
                    fillCommon(wide);
                    wide.period = s16WidePeriod(qlen, G);
                    wide.lengths = sh.dLengths.p;
                    wide.border = ctx.borderB;
                    wide.borderStride = (int)ctx.borderStride;
                } else {
                    fillCommon(narrow);
                    narrow.period = s16Period(qlen, G);
                    narrow.firstSubject = cl.first;
                    narrow.numSubjects = cl.count;
                }
                auto launchClass = [&](int g, cudaStream_t strm, int ctaOffset) {
                    cudaError_t e;
                    if (segmented) { narrow.ctaOffset = ctaOffset; e = launch_s16_multi(lc.R, narrow, g, strm); }
                    else if (lc.wide) { wide.ctaOffset = ctaOffset; e = launch_s16_wide(lc.R, lc.multi, wide, g, strm); }
                    else { narrow.ctaOffset = ctaOffset; e = launch_s16(lc.R, narrow, g, strm); }
                    if (e == cudaErrorInvalidValue) { cudaGetLastError(); fail(SW4_ERR_INVALID, "no kernel for class G=%d R=%d", G, lc.R); }
                    SW4_CUDA(e);
                    ctx.launches++;
                };
                // even part as clusters of 2 (same code on both SMs of a TPC), an odd leftover CTA on a second stream;
                // both launches share the class's ticket counter
                const int evenPart = grid & ~1;
                if (evenPart > 0) launchClass(evenPart, cst, 0);
                SW4_CUDA(cudaEventRecord(ctx.evJoin[ci % kMaxClassStreams], cst));
                SW4_CUDA(cudaStreamWaitEvent(st, ctx.evJoin[ci % kMaxClassStreams], 0));
                if (grid & 1) {
                    cudaStream_t ost = ctx.oddStreams[ci % kMaxClassStreams];
                    SW4_CUDA(cudaStreamWaitEvent(ost, ctx.evFork, 0));
                    launchClass(1, ost, evenPart);
                    SW4_CUDA(cudaEventRecord(ctx.evJoinOdd[ci % kMaxClassStreams], ost));
                    SW4_CUDA(cudaStreamWaitEvent(st, ctx.evJoinOdd[ci % kMaxClassStreams], 0));
                }
            }

            // exact 32-bit path for whatever saturated in 16 bit (the list and its length live on the device)
            const int p0 = (qlen + 32 + 15) / 16 * 16;
            if (useLongKernel && kLongLag * kLongMaxWarps + 64 <= p0) {
                // long queries re-score on the CTA-wide array, 16 warps per subject, whatever the subject's length (with a
                // PSSM, subjects of any class from 197 residues on can saturate 16 bits)
                S32LongParams lp{};
                lp.chars = arena; lp.offsets = offsetsBySubject; lp.lengths = sh.dLengths.p;
                lp.list = ctx.dOvfList.p; lp.listCountPtr = ctx.dCounters.p + 0; lp.ticket = ctx.dCounters.p + 3;
                lp.warps = kLongMaxWarps;
                lp.ringSlots = s16_long_ring_slots(kLongMaxWarps);
                lp.prof = reinterpret_cast<const int32_t*>(ctx.dProfile.p + (size_t)(kFused + 42) * profStride);
                lp.profStride = profStride; lp.qlen = qlen; lp.period = p0; lp.gop = gop; lp.gex = gex;
                lp.scores = ctx.dScores.p;
                lp.border = reinterpret_cast<int2*>(ctx.borderB);
                lp.borderStride = (int)ctx.borderStride;
                SW4_CUDA(launch_s32_long(lp, (int)std::min<size_t>((size_t)sh.smCount, ctx.borderRowArrays), st));
            } else {
                S32Params p{};
                p.chars = arena; p.offsets = offsetsBySubject; p.lengths = sh.dLengths.p;
                p.list = ctx.dOvfList.p; p.listCountPtr = ctx.dCounters.p + 0; p.listCountHost = 0;
                p.query = ctx.dQueryCodes.p; p.qlen = qlen; p.matrix = ctx.dMatrix.p; p.gop = gop; p.gex = gex;
                p.border = reinterpret_cast<int2*>(ctx.borderB); p.borderStride = (int)ctx.borderStride;
                p.ticket = ctx.dCounters.p + 3; p.scores = ctx.dScores.p;
                p.statThreshold = 0x7fffffff;
                p.statCount = ctx.dCounters.p + 1;
                const int blocks = std::max(1, (int)(ctx.borderRowArrays / kS32WarpsPerBlock));
                if (ctx.pssm) {  // scores from the profile's int32 plane: the PSSM query has no matrix rows
                    const int32_t* prof = reinterpret_cast<const int32_t*>(ctx.dProfile.p + (size_t)(kFused + 42) * profStride);
                    SW4_CUDA(launch_s32_pssm(p, prof, profStride, blocks, st));
                } else {
                    SW4_CUDA(launch_s32(p, blocks, st));
                }
            }
            ctx.launches++;
        }
        if (sh.streaming) SW4_CUDA(cudaEventRecord(ctx.evBatchDone[bi & 1], st));
    }

    // ---- part 3: top-k of the shard and the copy of k (score, id) pairs + counters to pinned host memory ----
    void enqueueEpilogue(Shard& sh, Ctx& ctx) {
        cudaStream_t st = ctx.stream;
        SW4_CUDA(cudaEventRecord(ctx.evK1, st));
        const long long n = (long long)sh.n;
        const int k = ctx.k;
        if (k > 0 && n > 0) {
            const long long bound = scanScoreBound(ctx.maxEntry, ctx.qlen, sh);
            const int launches = topk_enqueue(ctx.dScores.p, n, k, bound, sh.smCount, sh.dGlobalIds.p, ctx.dCand.p, ctx.dTopkWork.p,
                                              ctx.dTopkKeys.p, ctx.dTopScores.p, ctx.dTopIds.p, ctx.dCounters.p + 4, st);
            if (launches < 0) refuseScoreBound(bound);  // (checkScanQueries refuses the call before this can happen)
            ctx.launches += launches;
            SW4_CUDA(cudaGetLastError());
            SW4_CUDA(cudaMemcpyAsync(ctx.hTop.p, ctx.dTopScores.p, (size_t)k * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
            SW4_CUDA(cudaMemcpyAsync(ctx.hTop.p + k, ctx.dTopIds.p, (size_t)k * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        }
        if (ctx.stats) {  // the histogram of the scores and lengths of the shard (stats.cuh), next to the top-k
            SW4_CUDA(cudaMemsetAsync(ctx.dHist.p, 0, ctx.dHist.bytes(), st));
            ctx.launches += score_histogram_enqueue(ctx.dScores.p, sh.dLengths.p, n, sh.smCount, ctx.dHist.p, st);
            SW4_CUDA(cudaGetLastError());
            SW4_CUDA(cudaMemcpyAsync(ctx.hHist.p, ctx.dHist.p, ctx.dHist.bytes(), cudaMemcpyDeviceToHost, st));
        }
        SW4_CUDA(cudaMemcpyAsync(ctx.hTop.p + 2 * k, ctx.dCounters.p, 8 * sizeof(int), cudaMemcpyDeviceToHost, st));
        SW4_CUDA(cudaEventRecord(ctx.evStop, st));
    }

    // the result of the context's query goes to results[ctx.queryIndex]
    void collect(Shard& sh, Ctx& ctx, std::vector<ShardResult>& results) {
        if (ctx.queryIndex < 0 || (size_t)ctx.queryIndex >= results.size())
            fail(SW4_ERR_CUDA, "internal error: a context holds query %d of a call with %zu queries", ctx.queryIndex, results.size());
        ShardResult& out = results[(size_t)ctx.queryIndex];
        SW4_CUDA(cudaEventSynchronize(ctx.evStop));
        float ms = 0, kms = 0;
        SW4_CUDA(cudaEventElapsedTime(&ms, ctx.evStart, ctx.evStop));
        SW4_CUDA(cudaEventElapsedTime(&kms, ctx.evK0, ctx.evK1));
        const int k = ctx.k;
        const int* counters = ctx.hTop.p + 2 * k;
        const int cnt = (k > 0 && sh.n > 0) ? counters[4] : 0;
        out.scores.assign(ctx.hTop.p, ctx.hTop.p + cnt);
        out.ids.assign(ctx.hTop.p + k, ctx.hTop.p + k + cnt);
        out.statCount = counters[1];
        out.launches = ctx.launches;
        if (ctx.stats) out.hist.assign(ctx.hHist.p, ctx.hHist.p + 2 * kHistEntries);
        out.seconds = (double)ms * 1e-3;
        out.kernelSeconds = (double)kms * 1e-3;
        ctx.busy = false;
    }

    // ---- all queries on one shard ----
    // Resident shard: a rolling pipeline of `pipelineDepth` contexts; the host only blocks on the oldest query in flight.
    // Streaming shard: groups of up to kMaxContexts queries; every batch is uploaded once per group and scanned by all of
    // its queries while the next batch is on its way into the other slot.
    // An exception (a CUDA error: checkScanQueries has refused every bad query up front) waits for the work of the
    // shard's busy contexts and marks them idle before it leaves, so that the next call neither collects a query of this
    // one nor reuses buffers that are still being written.
    void runShard(Shard& sh, const QueryRef* queries, int nq, int kGlobal, std::vector<ShardResult>& results) {
        try {
            runShardQueries(sh, queries, nq, kGlobal, results);
        } catch (...) {
            cudaSetDevice(sh.device);
            for (auto& c : sh.ctxs) {
                if (!c->busy) continue;
                for (int i = 0; i < kMaxClassStreams; i++) {  // (errors ignored: the first one is on its way out)
                    cudaStreamSynchronize(c->classStreams[i]);
                    cudaStreamSynchronize(c->oddStreams[i]);
                }
                cudaStreamSynchronize(c->stream);
                c->busy = false;
            }
            cudaStreamSynchronize(sh.copyStream);
            throw;
        }
    }

    void runShardQueries(Shard& sh, const QueryRef* queries, int nq, int kGlobal, std::vector<ShardResult>& results) {
        SW4_CUDA(cudaSetDevice(sh.device));
        results.assign(nq, ShardResult{});
        sh.lastSpanSeconds = 0;
        if (nq == 0) return;
        const int k = (int)std::min<size_t>((size_t)kGlobal, sh.n);
        // device-timed span of the whole call: from the first query's first operation to the last stop event of any context
        auto spanStart = [&](Ctx& first) { SW4_CUDA(cudaEventRecord(sh.evManyStart, first.stream)); };
        auto spanStop = [&] {
            for (auto& c : sh.ctxs) SW4_CUDA(cudaStreamWaitEvent(sh.copyStream, c->evStop, 0));
            SW4_CUDA(cudaEventRecord(sh.evManyStop, sh.copyStream));
            SW4_CUDA(cudaEventSynchronize(sh.evManyStop));
            float ms = 0;
            SW4_CUDA(cudaEventElapsedTime(&ms, sh.evManyStart, sh.evManyStop));
            sh.lastSpanSeconds = (double)ms * 1e-3;
        };
        if (!sh.streaming) {
            const int depth = std::max(1, std::min(pipelineDepth, nq));
            for (int qi = 0; qi < nq; qi++) {
                Ctx& ctx = context(sh, qi % depth);
                if (qi == 0) spanStart(ctx);
                if (ctx.busy) collect(sh, ctx, results);
                enqueuePrologue(sh, ctx, queries[qi], qi, k);
                enqueueBatch(sh, ctx, 0, 0, true);
                enqueueEpilogue(sh, ctx);
                sh.lastCtx = qi % depth;
            }
            for (int c = 0; c < depth; c++) {
                Ctx& ctx = context(sh, (nq + c) % depth);  // oldest first
                if (ctx.busy) collect(sh, ctx, results);
            }
            spanStop();
            return;
        }
        const int numBatches = (int)sh.batches.size();
        const int group = std::max(1, std::min(kMaxContexts, nq));
        for (int q0 = 0; q0 < nq; q0 += group) {
            const int q1 = std::min(nq, q0 + group);
            if (q0 == 0) spanStart(context(sh, 0));
            for (int qi = q0; qi < q1; qi++) enqueuePrologue(sh, context(sh, qi - q0), queries[qi], qi, k);
            auto stage = [&](int bi) {
                const int si = bi & 1;
                if (sh.slots[si].batch == bi) return;  // still there from the previous group (single-batch case)
                // the slot's previous tenant (batch bi-2 of this group, or a batch of the previous group) must be done
                for (auto& c : sh.ctxs) SW4_CUDA(cudaStreamWaitEvent(sh.copyStream, c->evBatchDone[si], 0));
                stageBatch(sh, bi, si);
            };
            stage(0);
            for (int bi = 0; bi < numBatches; bi++) {
                for (int qi = q0; qi < q1; qi++) enqueueBatch(sh, context(sh, qi - q0), bi, bi & 1, bi == 0);
                if (bi + 1 < numBatches) stage(bi + 1);
            }
            for (int qi = q0; qi < q1; qi++) enqueueEpilogue(sh, context(sh, qi - q0));
            for (int qi = q0; qi < q1; qi++) collect(sh, context(sh, qi - q0), results);
            sh.lastCtx = q1 - q0 - 1;
        }
        spanStop();
    }

    // One host thread per GPU issues that GPU's work (the reference drives all GPUs from a single thread in lock-step
    // phases, src/cudasw4.cuh:1509-2259: ~35 launches x 8 GPUs back to back before the last GPU starts).
    void runAllShards(const QueryRef* queries, int nq, int k, std::vector<std::vector<ShardResult>>& results) {
        results.assign(shards.size(), {});
        if (shards.size() == 1) { runShard(*shards[0], queries, nq, k, results[0]); return; }
        std::vector<std::thread> workers;
        std::vector<Error> errors(shards.size(), Error{SW4_OK, ""});
        auto body = [&](size_t i) {
            try { runShard(*shards[i], queries, nq, k, results[i]); }
            catch (const Error& e) { errors[i] = e; }
            catch (const std::exception& e) { errors[i] = Error{SW4_ERR_INVALID, e.what()}; }
        };
        for (size_t i = 1; i < shards.size(); i++) workers.emplace_back(body, i);
        body(0);
        for (auto& w : workers) w.join();
        for (auto& e : errors)
            if (e.code != SW4_OK) throw e;
    }

    // The scores of a query whose largest pair score is maxEntry stay below this bound on the shard; the device top-k
    // is exact only while it is below 2^24.
    static long long scanScoreBound(int maxEntry, int qlen, const Shard& sh) { return (long long)maxEntry * std::min(qlen, sh.maxLen); }
    [[noreturn]] static void refuseScoreBound(long long bound) {
        fail(SW4_ERR_INVALID, "scores of this scan may reach %lld; the device top-k is exact below 2^24", bound);
    }

    // Every per-query refusal of a scan call (the top-k bound of enqueueEpilogue, the border rows of ensureCtx), decided
    // before the first query is enqueued: a refused call leaves the contexts, the last scan's scores and its statistics
    // as they were. kGlobal: the call's k.
    void checkScanQueries(const QueryRef* queries, int nq, int kGlobal) const {
        for (int i = 0; i < nq; i++) {
            const QueryRef& q = queries[i];
            checkBorderRows(queryCapacityFor(q.length, 0), q.length);
            const int maxEntry = q.pssm ? pssmMaxEntry(q.pssm, q.length) : maxMatrixEntry;
            for (const auto& sh : shards) {
                const int k = (int)std::min<size_t>((size_t)kGlobal, sh->n);
                if (k > 0 && sh->n > 0 && topk_shift_for(scanScoreBound(maxEntry, q.length, *sh)) < 0)
                    refuseScoreBound(scanScoreBound(maxEntry, q.length, *sh));
            }
        }
    }

    // ---- the public scans ----
    // outScores/outIds: [nq][numTop] (row stride numTop), outCounts[nq]; perQuery[nq] and total may be null.
    void scanMany(const QueryRef* queries, int nq, int32_t* outScores, int32_t* outIds, int32_t* outCounts, sw4_stats* perQuery,
                  sw4_stats* total) {
        if (!db) fail(SW4_ERR_INVALID, "no database set");
        for (int i = 0; i < nq; i++) {
            if (queries[i].length < 0 || (queries[i].length > 0 && !queries[i].letters)) fail(SW4_ERR_INVALID, "invalid query %d", i);
            if (queries[i].length > (1 << 24)) fail(SW4_ERR_INVALID, "query %d too long (%d)", i, queries[i].length);
            if (queries[i].pssm) checkPssmColumn20(queries[i].pssm, queries[i].length, ("query " + std::to_string(i)).c_str());
        }
        checkGaps();
        const size_t nTotal = db->nGlobal;
        const int k = (int)std::min<size_t>((size_t)std::max(numTop, 0), nTotal);
        checkScanQueries(queries, nq, k);
        lastHists.clear();
        lastStats.clear();
        upload();
        std::vector<std::vector<ShardResult>> results;
        runAllShards(queries, nq, k, results);
        double span = 0;  // device-timed, max over the GPUs
        for (auto& sh : shards) span = std::max(span, sh->lastSpanSeconds);
        uint64_t residues = 0;
        for (auto& sh : shards) residues += sh->residues;
        double sumCells = 0;
        int sumOverflows = 0, sumLaunches = 0;
        double sumKernel = 0;
        struct Entry { int32_t score, id; };
        std::vector<Entry> merged;
        for (int qi = 0; qi < nq; qi++) {
            merged.clear();
            double seconds = 0, kernelSeconds = 0;
            int overflows = 0, launches = 0;
            for (size_t s = 0; s < shards.size(); s++) {
                const ShardResult& r = results[s][qi];
                for (size_t i = 0; i < r.scores.size(); i++) merged.push_back(Entry{r.scores[i], r.ids[i]});
                seconds = std::max(seconds, r.seconds);
                kernelSeconds = std::max(kernelSeconds, r.kernelSeconds);
                overflows += r.statCount;
                launches += r.launches;
            }
            int got = (int)std::min<size_t>((size_t)k, merged.size());
            if (shards.size() > 1)
                std::partial_sort(merged.begin(), merged.begin() + got, merged.end(), [](const Entry& a, const Entry& b) {
                    if (a.score != b.score) return a.score > b.score;
                    return a.id < b.id;
                });
            if (statsEnabled) {  // the shards' histograms summed, their fit, and the E-value cutoff
                std::vector<int64_t> hist(2 * kHistEntries, 0);
                for (size_t s = 0; s < shards.size(); s++)
                    for (size_t b = 0; b < hist.size(); b++) hist[b] += results[s][qi].hist[b];
                sw4_score_statistics st;
                sw4_fit_score_statistics(hist.data(), hist.data() + kHistEntries, SW4_SCORE_BINS, queries[qi].length, &st);
                st.whole_database = holdsWholeDatabase() ? 1 : 0;
                if (st.whole_database && st.status == SW4_STATS_OK && std::isfinite(maxEvalue)) {
                    int keep = 0;  // E grows as the score falls: the hits to keep are a prefix
                    while (keep < got && evalueOf(st, merged[keep].score) <= maxEvalue) keep++;
                    got = keep;
                }
                lastHists.push_back(std::move(hist));
                lastStats.push_back(st);
            }
            for (int i = 0; i < got; i++) {
                outScores[(size_t)qi * numTop + i] = merged[i].score;
                outIds[(size_t)qi * numTop + i] = merged[i].id;
            }
            if (outCounts) outCounts[qi] = got;
            const double cells = (double)residues * (double)queries[qi].length;
            sumCells += cells;
            sumOverflows += overflows;
            sumLaunches += launches;
            sumKernel += kernelSeconds;
            if (perQuery) {
                perQuery[qi].num_overflows = overflows;
                perQuery[qi].seconds = seconds;
                perQuery[qi].gcups = seconds > 0 ? cells / 1e9 / seconds : 0;
                perQuery[qi].kernel_seconds = kernelSeconds;
                perQuery[qi].cells = cells;
                perQuery[qi].kernel_launches = launches;
            }
        }
        totalCells += sumCells;
        totalOverflows += sumOverflows;
        if (total) {
            total->num_overflows = sumOverflows;
            total->seconds = span;
            total->gcups = span > 0 ? sumCells / 1e9 / span : 0;
            total->kernel_seconds = sumKernel;
            total->cells = sumCells;
            total->kernel_launches = sumLaunches;
        }
    }

    // Does this handle scan every sequence of the database? Not when sw4_set_shard splits it (world > 1), and not when
    // the handle holds only some of the sequences (sw4_set_database_shard_memory, or the generated shard of
    // sw4_set_pseudo_database_lengths, which gives every database global ids, sharded or not).
    bool holdsWholeDatabase() const { return db->globalIds ? db->n == db->nGlobal : shardWorld == 1; }

    // E = K m D e^(-lambda S) (sw4b200.h)
    static double evalueOf(const sw4_score_statistics& st, int score) {
        return st.K * (double)st.query_length * (double)st.db_residues * std::exp(-st.lambda * score);
    }

    void scan(const char* query, int qlen, const int8_t* pssm, int32_t* outScores, int32_t* outIds, int32_t* outCount, sw4_stats* stats) {
        QueryRef q{query, qlen, pssm};
        scanMany(&q, 1, outScores, outIds, outCount, stats, nullptr);
    }

    // ---- alignment coordinates: score, end and begin of one optimal local alignment per (query, id) pair ----
    // Subjects come from the host copy (any database mode, before or after the upload) and go through pinned staging to
    // the handle's first GPU. Pass 1 leaves the ends on the device for pass 2; the host waits once per chunk of pairs
    // whose scratch (gathered subjects + border columns) fits max_temp_bytes.
    // Checks the arguments shared by sw4_alignment_coordinates and sw4_alignment_traceback; returns the position of
    // every id in the handle's host arrays.
    // pssm: nullptr (sequence query) or the query's [qlen][21] table (the caller has checked it is there)
    std::vector<size_t> alignmentPairs(const char* query, int qlen, const int8_t* pssm, const int32_t* ids, int n, const void* out) {
        if (!db) fail(SW4_ERR_INVALID, "no database set");
        if (n < 0) fail(SW4_ERR_INVALID, "num_ids must be >= 0 (got %d)", n);
        if (n > 0 && (!ids || !out)) fail(SW4_ERR_INVALID, "null id or output array");
        if (qlen < 0 || (qlen > 0 && !query)) fail(SW4_ERR_INVALID, "invalid query");
        if (qlen > (1 << 24)) fail(SW4_ERR_INVALID, "query too long (%d residues, at most 2^24)", qlen);
        checkGaps();
        if (pssm) checkPssmColumn20(pssm, qlen, "query");
        const int maxEntry = pssm ? pssmMaxEntry(pssm, qlen) : maxMatrixEntry;
        std::vector<size_t> local((size_t)n);
        for (int i = 0; i < n; i++) {
            const int32_t id = ids[i];
            if (id < 0 || (size_t)id >= db->nGlobal)
                fail(SW4_ERR_INVALID, "database id %d out of range (the database has %zu sequences)", id, db->nGlobal);
            local[i] = db->localIndex(id);
            if (local[i] >= db->n) fail(SW4_ERR_INVALID, "database id %d is not held by this handle (pre-sharded database)", id);
            const long long bound = (long long)maxEntry * std::min(qlen, db->lengths[local[i]]);
            if (topk_shift_for(bound) < 0)
                fail(SW4_ERR_INVALID, "the score of the query against id %d may reach %lld; scores are exact below 2^24", id, bound);
        }
        return local;
    }

    // the CoordState on the handle's first GPU (made current) with the query codes and the matrix uploaded on its stream,
    // and a PSSM query's table in cs.dPssm
    CoordState& coordQuery(const char* query, int qlen, const int8_t* pssm, int& launches) {
        if (!coord) {
            auto c = std::make_unique<CoordState>();
            c->create(deviceIds[0]);
            coord = std::move(c);
        }
        CoordState& cs = *coord;
        SW4_CUDA(cudaSetDevice(cs.device));
        cudaStream_t st = cs.stream;
        SW4_CUDA(cudaEventRecord(cs.evStart, st));
        const int qpad = (qlen + 3) / 4 * 4;
        cs.hQuery.ensure((size_t)std::max(qlen, 1));
        if (qlen) memcpy(cs.hQuery.p, query, (size_t)qlen);
        if ((size_t)qpad + 16 > cs.dQueryCodes.n) { cs.dQueryLetters.alloc((size_t)qpad + 16); cs.dQueryCodes.alloc((size_t)qpad + 16); }
        if (qlen) SW4_CUDA(cudaMemcpyAsync(cs.dQueryLetters.p, cs.hQuery.p, (size_t)qlen, cudaMemcpyHostToDevice, st));
        SW4_CUDA(cudaMemcpyAsync(cs.dMatrix.p, matrix, 441, cudaMemcpyHostToDevice, st));
        if (pssm && qlen) {
            const size_t bytes = (size_t)qlen * 21;
            if (bytes > cs.dPssm.n) {  // (the previous call has synchronised: nothing in flight reads the old buffers)
                const size_t cap = std::max(bytes * 2, (size_t)8192 * 21);
                cs.hPssm.ensure(cap);
                cs.dPssm.alloc(cap);
            }
            memcpy(cs.hPssm.p, pssm, bytes);
            SW4_CUDA(cudaMemcpyAsync(cs.dPssm.p, cs.hPssm.p, bytes, cudaMemcpyHostToDevice, st));
        }
        if (qpad > 0) {
            convert_query_kernel<<<(qpad + 255) / 256, 256, 0, st>>>(cs.dQueryLetters.p, cs.dQueryCodes.p, qlen, qpad);
            SW4_CUDA(cudaGetLastError());
            launches++;
        }
        return cs;
    }

    // stats of a coordinate / traceback call: device time from coordQuery's start event to now
    void coordStats(CoordState& cs, double cells, int launches, sw4_stats* stats) {
        SW4_CUDA(cudaEventRecord(cs.evStop, cs.stream));
        SW4_CUDA(cudaEventSynchronize(cs.evStop));
        float ms = 0;
        SW4_CUDA(cudaEventElapsedTime(&ms, cs.evStart, cs.evStop));
        if (stats) {
            stats->seconds = (double)ms * 1e-3;
            stats->cells = cells;
            stats->gcups = ms > 0 ? cells / 1e9 / stats->seconds : 0;
            stats->kernel_launches = launches;
        }
    }

    // passes 1 and 2 for the pairs (query, local[i]), in chunks under max_temp_bytes; out[i] receives the coordinates
    // (pssm: the device table of a PSSM query, or nullptr)
    void coordPasses(CoordState& cs, int qlen, const int8_t* pssm, const std::vector<size_t>& local, sw4_alignment* out, double& cells,
                     int& launches) {
        const int n = (int)local.size();
        cudaStream_t st = cs.stream;
        auto lengthOf = [&](int i) { return (int)db->lengths[local[i]]; };
        auto tilesOf = [](int len) { return (len + kCoordTileCols - 1) / kCoordTileCols; };
        auto warpsOf = [&](int len) {
            const int tiles = tilesOf(len);
            return (tiles > 1 && (long long)qlen * len >= kCoordCtaMinCells) ? std::min(tiles, kCoordWarps) : 1;
        };
        const size_t borderStride = alignUp((size_t)std::max(qlen, 1), 32);
        auto scratchOf = [&](int len) {
            size_t b = alignUp((size_t)len, 16);
            if (tilesOf(len) > 1) b += (size_t)warpsOf(len) * borderStride * sizeof(int2);
            return b;
        };
        // CTA-form pairs first, then the one-warp pairs; longest first within each form
        std::vector<int> order((size_t)n);
        for (int i = 0; i < n; i++) order[i] = i;
        std::stable_sort(order.begin(), order.end(), [&](int a, int b) {
            const int la = lengthOf(a), lb = lengthOf(b);
            const bool ca = warpsOf(la) > 1, cb = warpsOf(lb) > 1;
            if (ca != cb) return ca;
            return la > lb;
        });

        const size_t budget = mem.max_temp_bytes;
        for (int pos = 0; pos < n;) {
            int end = pos;
            size_t bytes = 0;
            while (end < n && bytes + scratchOf(lengthOf(order[end])) <= budget) bytes += scratchOf(lengthOf(order[end++]));
            if (end == pos)
                fail(SW4_ERR_NOMEM, "max_temp_bytes (%zu bytes) cannot hold the scratch of one pair (%d x %d residues: %zu bytes)", budget,
                     qlen, lengthOf(order[pos]), scratchOf(lengthOf(order[pos])));
            const int m = end - pos;
            cs.hItems.ensure((size_t)m);
            cs.hGroups.ensure((size_t)m);
            size_t subjectBytes = 0, borderEntries = 0;
            int numGroups = 0;
            for (int k = 0; k < m; k++) {
                const int len = lengthOf(order[pos + k]), W = warpsOf(len);
                CoordItem& it = cs.hItems.p[k];
                it.subjectOffset = subjectBytes;
                it.subjectLength = len;
                it.borderOffset = borderEntries;
                subjectBytes += alignUp((size_t)len, 16);
                if (tilesOf(len) > 1) borderEntries += (size_t)W * borderStride;
                CoordGroup* last = numGroups ? &cs.hGroups.p[numGroups - 1] : nullptr;
                if (W == 1 && last && last->warps == 1 && last->count < kCoordWarps) last->count++;
                else cs.hGroups.p[numGroups++] = CoordGroup{k, 1, W};
                cells += (double)qlen * (double)len;
            }
            cs.hSubjects.ensure(std::max<size_t>(subjectBytes, 1));
            for (int k = 0; k < m; k++) {
                const size_t li = local[order[pos + k]];
                memcpy(cs.hSubjects.p + cs.hItems.p[k].subjectOffset, db->chars + db->offsets[li], (size_t)db->lengths[li]);
            }
            // one scratch arena: subjects, then border columns (16-byte aligned: every subject is padded to 16)
            const size_t scratchBytes = subjectBytes + borderEntries * sizeof(int2);
            if (std::max<size_t>(scratchBytes, 16) > cs.dSubjects.n) cs.dSubjects.alloc(std::max<size_t>(scratchBytes, 16));
            if ((size_t)m > cs.dItems.n) { cs.dItems.alloc((size_t)m); cs.dGroups.alloc((size_t)m); cs.dEnds.alloc((size_t)m); }
            if ((size_t)m * 5 + 1 > cs.dOut.n) cs.dOut.alloc((size_t)m * 5 + 1);
            cs.hOut.ensure((size_t)m * 5 + 1);
            if (subjectBytes) SW4_CUDA(cudaMemcpyAsync(cs.dSubjects.p, cs.hSubjects.p, subjectBytes, cudaMemcpyHostToDevice, st));
            SW4_CUDA(cudaMemcpyAsync(cs.dItems.p, cs.hItems.p, (size_t)m * sizeof(CoordItem), cudaMemcpyHostToDevice, st));
            SW4_CUDA(cudaMemcpyAsync(cs.dGroups.p, cs.hGroups.p, (size_t)numGroups * sizeof(CoordGroup), cudaMemcpyHostToDevice, st));
            SW4_CUDA(cudaMemsetAsync(cs.dOut.p + (size_t)m * 5, 0, sizeof(int32_t), st));
            CoordParams p{};
            p.groups = cs.dGroups.p; p.items = cs.dItems.p; p.subjects = cs.dSubjects.p;
            p.query = cs.dQueryCodes.p; p.qlen = qlen; p.matrix = cs.dMatrix.p; p.gop = gop; p.gex = gex;
            p.border = reinterpret_cast<int2*>(cs.dSubjects.p + subjectBytes); p.borderStride = (int)borderStride;
            p.ends = cs.dEnds.p; p.out = cs.dOut.p; p.errors = cs.dOut.p + (size_t)m * 5;
            SW4_CUDA(launch_coords(false, p, numGroups, st, pssm));
            SW4_CUDA(launch_coords(true, p, numGroups, st, pssm));
            launches += 2;
            SW4_CUDA(cudaMemcpyAsync(cs.hOut.p, cs.dOut.p, ((size_t)m * 5 + 1) * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
            SW4_CUDA(cudaStreamSynchronize(st));
            if (cs.hOut.p[(size_t)m * 5] != 0)
                fail(SW4_ERR_CUDA, "internal error: the begin pass of %d pairs did not reach the anchored score", cs.hOut.p[(size_t)m * 5]);
            for (int k = 0; k < m; k++) {
                const int32_t* r = cs.hOut.p + (size_t)k * 5;
                out[order[pos + k]] = sw4_alignment{r[0], r[1], r[2], r[3], r[4]};
                if (r[0] > 0) cells += (double)(r[2] + 1) * (double)(r[4] + 1);
            }
            pos = end;
        }
    }

    void alignmentCoordinates(const char* query, int qlen, const int8_t* pssm, const int32_t* ids, int n, sw4_alignment* out,
                              sw4_stats* stats) {
        const std::vector<size_t> local = alignmentPairs(query, qlen, pssm, ids, n, out);
        if (stats) memset(stats, 0, sizeof(*stats));
        if (n == 0) return;
        int launches = 0;
        double cells = 0;
        CoordState& cs = coordQuery(query, qlen, pssm, launches);
        coordPasses(cs, qlen, pssm ? cs.dPssm.p : nullptr, local, out, cells, launches);
        coordStats(cs, cells, launches, stats);
    }

    // ---- alignment traceback: the columns of the alignment that sw4_alignment_coordinates locates ----
    // After the coordinate passes, the pairs with a positive score are chunked again by their trace scratch (subject
    // slice, border columns, 4-bit direction words, rows + cols op bytes, counts) under max_temp_bytes. Each chunk runs
    // pass 3 and the walk and copies the ops and counts back: one host synchronisation per chunk.
    // profile: the pseudocount weight of sw4_build_pssm, whose MSA the chunks then fill (each pair's row right after the
    // walk) and whose PSSM follows the last chunk into cs.hProfileOut; nullptr: the traceback alone, which leaves
    // sw4_last_cigars to this call. Without a profile the call enqueues nothing else.
    void alignmentTraceback(const char* query, int qlen, const int8_t* pssm, const int32_t* ids, int n, sw4_alignment_summary* out,
                            sw4_stats* stats, const double* profile = nullptr) {
        if (!profile) lastCigars.clear();
        const std::vector<size_t> local = alignmentPairs(query, qlen, pssm, ids, n, out);
        if (stats) memset(stats, 0, sizeof(*stats));
        if (n == 0 && !profile) return;
        int launches = 0;
        double cells = 0;
        CoordState& cs = coordQuery(query, qlen, pssm, launches);
        const int8_t* dPssm = pssm ? cs.dPssm.p : nullptr;
        std::vector<sw4_alignment> coords((size_t)n);
        coordPasses(cs, qlen, dPssm, local, coords.data(), cells, launches);
        cudaStream_t st = cs.stream;

        std::vector<int> traced;
        for (int i = 0; i < n; i++) {
            out[i] = sw4_alignment_summary{};
            out[i].coordinates = coords[i];
            if (coords[i].score > 0) traced.push_back(i);
        }
        auto rowsOf = [&](int i) { return coords[i].query_end - coords[i].query_begin + 1; };
        auto colsOf = [&](int i) { return coords[i].reference_end - coords[i].reference_begin + 1; };
        auto tilesOf = [](int cols) { return (cols + kCoordTileCols - 1) / kCoordTileCols; };
        auto warpsOf = [&](int i) {  // the form of pass 3, from the rectangle
            const int tiles = tilesOf(colsOf(i));
            return (tiles > 1 && (long long)rowsOf(i) * colsOf(i) >= kCoordCtaMinCells) ? std::min(tiles, kCoordWarps) : 1;
        };
        auto borderOf = [&](int i) {  // int2 entries
            return tilesOf(colsOf(i)) > 1 ? (size_t)warpsOf(i) * alignUp((size_t)rowsOf(i), 32) : 0;
        };
        auto wordsOf = [&](int i) { return (size_t)tilesOf(colsOf(i)) * ((size_t)rowsOf(i) + 31) * 32; };
        auto opsOf = [&](int i) { return alignUp((size_t)rowsOf(i) + (size_t)colsOf(i), 16); };
        auto scratchOf = [&](int i) {
            return alignUp((size_t)colsOf(i), 16) + borderOf(i) * sizeof(int2) + wordsOf(i) * sizeof(unsigned long long) + opsOf(i) +
                   sizeof(int4);
        };
        // the profile's MSA: row 0 the query, then one row per traced id in call order, allocated apart from the arena
        std::vector<int> msaRow;
        int msaRows = 1;
        if (profile) {
            msaRow.assign((size_t)n, 0);
            for (int i : traced) msaRow[i] = msaRows++;
            const size_t msaBytes = (size_t)msaRows * (size_t)qlen;
            if (msaBytes > mem.max_temp_bytes)
                fail(SW4_ERR_NOMEM, "max_temp_bytes (%zu bytes) cannot hold the MSA of the profile (%d rows x %d columns)",
                     mem.max_temp_bytes, msaRows, qlen);
            cs.dMsa.ensure(std::max<size_t>(msaBytes, 1));
            if (qlen) {
                SW4_CUDA(cudaMemsetAsync(cs.dMsa.p, kMsaEmpty, msaBytes, st));
                SW4_CUDA(cudaMemcpyAsync(cs.dMsa.p, cs.dQueryCodes.p, (size_t)qlen, cudaMemcpyDeviceToDevice, st));
            }
        }
        // CTA-form pairs first, then the one-warp pairs; largest rectangle first within each form
        std::stable_sort(traced.begin(), traced.end(), [&](int a, int b) {
            const bool ca = warpsOf(a) > 1, cb = warpsOf(b) > 1;
            if (ca != cb) return ca;
            return (long long)rowsOf(a) * colsOf(a) > (long long)rowsOf(b) * colsOf(b);
        });

        const size_t budget = mem.max_temp_bytes;
        const int nt = (int)traced.size();
        for (int pos = 0; pos < nt;) {
            int end = pos;
            size_t bytes = 2 * sizeof(int4);  // error counters (padded)
            while (end < nt && bytes + scratchOf(traced[end]) <= budget) bytes += scratchOf(traced[end++]);
            if (end == pos)
                fail(SW4_ERR_NOMEM, "max_temp_bytes (%zu bytes) cannot hold the traceback scratch of one pair (%d x %d rectangle: %zu bytes)",
                     budget, rowsOf(traced[pos]), colsOf(traced[pos]), scratchOf(traced[pos]) + 2 * sizeof(int4));
            const int m = end - pos;
            cs.hItems.ensure((size_t)m);
            cs.hGroups.ensure((size_t)m);
            cs.hTraceItems.ensure((size_t)m);
            size_t subjectBytes = 0, borderEntries = 0, words = 0, opsBytes = 0;
            int numGroups = 0;
            for (int k = 0; k < m; k++) {
                const int i = traced[pos + k], W = warpsOf(i);
                CoordItem& it = cs.hItems.p[k];
                it.subjectOffset = subjectBytes;
                it.subjectLength = colsOf(i);
                it.borderOffset = borderEntries;
                TraceItem& ti = cs.hTraceItems.p[k];
                ti.words = words;
                ti.ops = opsBytes;
                ti.queryBegin = coords[i].query_begin;
                ti.rows = rowsOf(i);
                ti.score = coords[i].score;
                subjectBytes += alignUp((size_t)colsOf(i), 16);
                borderEntries += borderOf(i);
                words += wordsOf(i);
                opsBytes += opsOf(i);
                CoordGroup* last = numGroups ? &cs.hGroups.p[numGroups - 1] : nullptr;
                if (W == 1 && last && last->warps == 1 && last->count < kCoordWarps) last->count++;
                else cs.hGroups.p[numGroups++] = CoordGroup{k, 1, W};
                cells += (double)rowsOf(i) * (double)colsOf(i);
            }
            cs.hSubjects.ensure(std::max<size_t>(subjectBytes, 1));
            for (int k = 0; k < m; k++) {
                const int i = traced[pos + k];
                const size_t li = local[i];
                memcpy(cs.hSubjects.p + cs.hItems.p[k].subjectOffset, db->chars + db->offsets[li] + coords[i].reference_begin,
                       (size_t)colsOf(i));
            }
            // one scratch arena: subject slices | border columns | direction words | ops | counts | 2 error counters
            // (every part is a multiple of 16 bytes)
            const size_t borderAt = subjectBytes, wordsAt = borderAt + borderEntries * sizeof(int2);
            const size_t opsAt = wordsAt + words * sizeof(unsigned long long), countsAt = opsAt + opsBytes;
            const size_t errorsAt = countsAt + (size_t)m * sizeof(int4), scratchBytes = errorsAt + 2 * sizeof(int4);
            if (scratchBytes > cs.dSubjects.n) cs.dSubjects.alloc(scratchBytes);
            if ((size_t)m > cs.dItems.n) { cs.dItems.alloc((size_t)m); cs.dGroups.alloc((size_t)m); cs.dEnds.alloc((size_t)m); }
            if ((size_t)m > cs.dTraceItems.n) cs.dTraceItems.alloc((size_t)m);
            cs.hTraceOut.ensure(scratchBytes - opsAt);
            uint8_t* arena = cs.dSubjects.p;
            SW4_CUDA(cudaMemcpyAsync(arena, cs.hSubjects.p, subjectBytes, cudaMemcpyHostToDevice, st));
            SW4_CUDA(cudaMemcpyAsync(cs.dItems.p, cs.hItems.p, (size_t)m * sizeof(CoordItem), cudaMemcpyHostToDevice, st));
            SW4_CUDA(cudaMemcpyAsync(cs.dTraceItems.p, cs.hTraceItems.p, (size_t)m * sizeof(TraceItem), cudaMemcpyHostToDevice, st));
            SW4_CUDA(cudaMemcpyAsync(cs.dGroups.p, cs.hGroups.p, (size_t)numGroups * sizeof(CoordGroup), cudaMemcpyHostToDevice, st));
            SW4_CUDA(cudaMemsetAsync(arena + errorsAt, 0, 2 * sizeof(int), st));
            CoordParams p{};
            p.groups = cs.dGroups.p; p.items = cs.dItems.p; p.subjects = arena;
            p.query = cs.dQueryCodes.p; p.qlen = qlen; p.matrix = cs.dMatrix.p; p.gop = gop; p.gex = gex;
            p.border = reinterpret_cast<int2*>(arena + borderAt);
            p.errors = reinterpret_cast<int*>(arena + errorsAt);
            p.traceItems = cs.dTraceItems.p;
            p.trace = reinterpret_cast<unsigned long long*>(arena + wordsAt);
            p.ops = reinterpret_cast<char*>(arena + opsAt);
            p.counts = reinterpret_cast<int4*>(arena + countsAt);
            p.numItems = m;
            SW4_CUDA(launch_coords_trace(p, numGroups, st, dPssm));
            SW4_CUDA(launch_coords_walk(p, st, dPssm));
            launches += 2;
            if (profile && qlen) {  // the chunk's MSA rows, while its subject slices and ops are in the arena
                cs.hMsaRows.ensure((size_t)m);
                for (int k = 0; k < m; k++) cs.hMsaRows.p[k] = msaRow[traced[pos + k]];
                cs.dMsaRows.ensure((size_t)m);
                SW4_CUDA(cudaMemcpyAsync(cs.dMsaRows.p, cs.hMsaRows.p, (size_t)m * sizeof(int), cudaMemcpyHostToDevice, st));
                SW4_CUDA(launch_profile_scatter(p, cs.dMsaRows.p, cs.dMsa.p, qlen, st));
                launches++;
            }
            SW4_CUDA(cudaMemcpyAsync(cs.hTraceOut.p, arena + opsAt, scratchBytes - opsAt, cudaMemcpyDeviceToHost, st));
            SW4_CUDA(cudaStreamSynchronize(st));
            const char* ops = cs.hTraceOut.p;
            const int4* counts = reinterpret_cast<const int4*>(ops + (countsAt - opsAt));
            const int* errors = reinterpret_cast<const int*>(ops + (errorsAt - opsAt));
            if (errors[0] != 0)
                fail(SW4_ERR_CUDA, "internal error: the traceback pass of %d pairs did not reach the anchored score", errors[0]);
            if (errors[1] != 0) fail(SW4_ERR_CUDA, "internal error: the walk of %d pairs did not end at the begin", errors[1]);
            for (int k = 0; k < m; k++) {
                sw4_alignment_summary& o = out[traced[pos + k]];
                const int4 c = counts[k];
                o.length = c.x; o.identities = c.y; o.positives = c.z; o.gaps = c.w;
                if (profile) continue;
                // the walk wrote the ops from the end: run-length encode them backwards, in query order
                const char* r = ops + cs.hTraceItems.p[k].ops;
                o.cigar_offset = lastCigars.size();
                for (int e = c.x - 1; e >= 0;) {
                    const char op = r[e];
                    int run = 0;
                    while (e >= 0 && r[e] == op) { run++; e--; }
                    lastCigars += std::to_string(run);
                    lastCigars += op;
                }
                o.cigar_length = lastCigars.size() - o.cigar_offset;
            }
            pos = end;
        }
        if (profile) profileScores(cs, qlen, msaRows, *profile, launches);
        coordStats(cs, cells, launches, stats);
    }

    // steps 3-6 of the profile over the finished MSA of msaRows rows (profile.cuh); the result lands in cs.hProfileOut
    // once the stream is synchronised
    void profileScores(CoordState& cs, int qlen, int msaRows, double beta, int& launches) {
        if (qlen == 0) return;
        cudaStream_t st = cs.stream;
        if (profileBg.blosum != blosum) profileBg.compute(blosum, matrix);
        cs.hProfileTables.ensure(420);
        memcpy(cs.hProfileTables.p, profileBg.qOverP, 400 * sizeof(double));
        memcpy(cs.hProfileTables.p + 400, profileBg.p, 20 * sizeof(double));
        cs.dProfileTables.ensure(420);
        cs.dProfileCounts.ensure((size_t)kMsaSymbols * qlen);
        cs.dProfileDistinct.ensure((size_t)qlen);
        cs.dProfileNsum.ensure(2);
        cs.dProfileWeights.ensure((size_t)msaRows);
        cs.dProfileOut.ensure((size_t)qlen * 21);
        cs.hProfileOut.ensure((size_t)qlen * 21);
        SW4_CUDA(cudaMemcpyAsync(cs.dProfileTables.p, cs.hProfileTables.p, 420 * sizeof(double), cudaMemcpyHostToDevice, st));
        SW4_CUDA(cudaMemsetAsync(cs.dProfileNsum.p, 0, 2 * sizeof(unsigned long long), st));
        ProfileParams p{};
        p.msa = cs.dMsa.p; p.rows = msaRows; p.m = qlen;
        p.counts = cs.dProfileCounts.p; p.distinct = cs.dProfileDistinct.p; p.nsum = cs.dProfileNsum.p;
        p.weights = cs.dProfileWeights.p; p.qOverP = cs.dProfileTables.p; p.p = cs.dProfileTables.p + 400;
        p.lambda = profileBg.lambda; p.beta = beta; p.low = matrix[20 * 21 + 20];
        p.out = cs.dProfileOut.p;
        SW4_CUDA(launch_profile_build(p, st, &launches));
        SW4_CUDA(cudaMemcpyAsync(cs.hProfileOut.p, cs.dProfileOut.p, (size_t)qlen * 21, cudaMemcpyDeviceToHost, st));
    }

    // ---- profile construction and the iterative search (sw4_build_pssm, sw4_search_iterative) ----
    static void checkBeta(double beta) {
        if (!(beta > 0) || !std::isfinite(beta)) fail(SW4_ERR_INVALID, "the pseudocount weight must be a finite number > 0 (got %g)", beta);
    }

    void buildPssm(const char* query, int qlen, const int8_t* pssm, const int32_t* ids, int n, double beta, int8_t* out, sw4_stats* stats) {
        checkBeta(beta);
        if (qlen > 0 && !out) fail(SW4_ERR_INVALID, "null output array");
        std::vector<sw4_alignment_summary> alignments((size_t)std::max(n, 1));
        alignmentTraceback(query, qlen, pssm, ids, n, alignments.data(), stats, &beta);
        if (qlen > 0) memcpy(out, coord->hProfileOut.p, (size_t)qlen * 21);
    }

    // P_1 = the sequence; round i scans with P_i (statistics on, no E-value cutoff), H_i = the ids of its list with
    // E <= inclusionE; the rounds stop at maxIt, at an empty H_i or at set(H_i) == set(H_{i-1}) (converged), else
    // P_{i+1} = the profile of H_i aligned with P_i. The last scan's list is reported with the handle's cutoff applied.
    void searchIterative(const char* query, int qlen, int maxIt, double inclusionE, double beta, int32_t* outScores, int32_t* outIds,
                         int32_t* outCount, int8_t* outPssm, int32_t* outIterations, int32_t* outConverged, sw4_stats* stats) {
        if (!db) fail(SW4_ERR_INVALID, "no database set");
        if (!statsEnabled) fail(SW4_ERR_INVALID, "the iterative search needs score statistics (sw4_set_score_statistics)");
        if (!holdsWholeDatabase()) fail(SW4_ERR_INVALID, "the iterative search needs a handle that scans the whole database");
        if (maxIt < 1) fail(SW4_ERR_INVALID, "max_iterations must be >= 1 (got %d)", maxIt);
        if (std::isnan(inclusionE) || inclusionE < 0) fail(SW4_ERR_INVALID, "inclusion_evalue must be >= 0 (got %g)", inclusionE);
        checkBeta(beta);
        if (qlen < 0 || (qlen > 0 && (!query || !outPssm))) fail(SW4_ERR_INVALID, "invalid query or null PSSM output");
        if (numTop > 0 && (!outScores || !outIds)) fail(SW4_ERR_INVALID, "null output arrays");
        if (!outCount || !outIterations || !outConverged) fail(SW4_ERR_INVALID, "null output");
        sw4_stats total{};
        auto add = [&](const sw4_stats& s) {
            total.num_overflows += s.num_overflows;
            total.seconds += s.seconds;
            total.kernel_seconds += s.kernel_seconds;
            total.cells += s.cells;
            total.kernel_launches += s.kernel_launches;
        };
        const size_t k = (size_t)std::max(numTop, 1);
        std::vector<int32_t> scores(k), ids(k), hits, prev;
        std::vector<int8_t> P, next((size_t)std::max(qlen, 1) * 21);
        int32_t count = 0;
        int iteration = 1;
        bool converged = false;
        const double cutoff = maxEvalue;
        struct RestoreCutoff { double& v; double keep; ~RestoreCutoff() { v = keep; } } restore{maxEvalue, cutoff};
        maxEvalue = INFINITY;  // the rounds take their hits before the cutoff
        for (;; iteration++) {
            sw4_stats s{};
            scan(query, qlen, P.empty() ? nullptr : P.data(), scores.data(), ids.data(), &count, &s);
            add(s);
            const sw4_score_statistics& st = lastStats[0];
            hits.clear();
            if (st.status == SW4_STATS_OK)
                for (int i = 0; i < count && evalueOf(st, scores[i]) <= inclusionE; i++) hits.push_back(ids[i]);
            std::vector<int32_t> sorted = hits;
            std::sort(sorted.begin(), sorted.end());
            converged = iteration > 1 && !hits.empty() && sorted == prev;
            if (iteration == maxIt || hits.empty() || converged) break;
            buildPssm(query, qlen, P.empty() ? nullptr : P.data(), hits.data(), (int)hits.size(), beta, next.data(), &s);
            add(s);
            P.assign(next.begin(), next.begin() + (size_t)qlen * 21);
            prev = std::move(sorted);
        }
        maxEvalue = cutoff;  // (restore does it on an error)
        if (P.empty()) {  // one round: the sequence's profile, the matrix rows
            sw4_stats s{};
            buildPssm(query, qlen, nullptr, nullptr, 0, beta, next.data(), &s);
            add(s);
            P.assign(next.begin(), next.begin() + (size_t)qlen * 21);
        }
        const sw4_score_statistics& st = lastStats[0];
        if (st.status == SW4_STATS_OK && std::isfinite(maxEvalue))
            while (count > 0 && evalueOf(st, scores[count - 1]) > maxEvalue) count--;
        for (int i = 0; i < count; i++) { outScores[i] = scores[i]; outIds[i] = ids[i]; }
        *outCount = count;
        if (qlen > 0) memcpy(outPssm, P.data(), (size_t)qlen * 21);
        *outIterations = iteration;
        *outConverged = converged ? 1 : 0;
        if (stats) {
            *stats = total;
            stats->gcups = total.seconds > 0 ? total.cells / 1e9 / total.seconds : 0;
        }
    }
};

}  // namespace sw4

// =================================================================================================================
// C ABI
// =================================================================================================================
struct sw4_handle {
    sw4::Engine eng;
};

static std::string g_globalError;

template <class Fn>
static int guarded(sw4_handle* h, Fn&& fn) {
    try {
        fn();
        return SW4_OK;
    } catch (const sw4::Error& e) {
        (h ? h->eng.lastError : g_globalError) = e.msg;
        return e.code;
    } catch (const std::bad_alloc&) {
        (h ? h->eng.lastError : g_globalError) = "out of host memory";
        return SW4_ERR_NOMEM;
    } catch (const std::exception& e) {
        (h ? h->eng.lastError : g_globalError) = e.what();
        return SW4_ERR_INVALID;
    }
}

extern "C" {

const char* sw4_version(void) { return "sw4b200 0.2 sm_100a"; }

const char* sw4_last_error(const sw4_handle* h) { return h ? h->eng.lastError.c_str() : g_globalError.c_str(); }

int sw4_create(const int* device_ids, int num_devices, int num_top, int blosum, int gop, int gex, const sw4_mem_config* mem,
               int verbose, sw4_handle** out) {
    if (!out) return SW4_ERR_INVALID;
    *out = nullptr;
    sw4_handle* h = nullptr;
    int rc = guarded(nullptr, [&] {
        // the length classes (and the queries in flight) run on their own streams: give them their own hardware queues
        // (only effective when this process has not initialised CUDA yet; never overrides the caller's setting)
        setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0);
        int count = 0;
        cudaError_t e = cudaGetDeviceCount(&count);
        if (e != cudaSuccess || count == 0)
            sw4::fail(SW4_ERR_CUDA, "no usable CUDA device (%s); this engine has no CPU fallback",
                      e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
        h = new sw4_handle();
        sw4::Engine& eng = h->eng;
        if (device_ids && num_devices > 0) {
            for (int i = 0; i < num_devices; i++) {
                if (device_ids[i] < 0 || device_ids[i] >= count) sw4::fail(SW4_ERR_INVALID, "invalid device id %d", device_ids[i]);
                eng.deviceIds.push_back(device_ids[i]);
            }
        } else {
            for (int i = 0; i < count; i++) eng.deviceIds.push_back(i);  // all visible GPUs, like src/main.cu:110-128
        }
        eng.numTop = num_top;
        eng.blosum = blosum;
        eng.gop = gop > 0 ? -gop : gop;
        eng.gex = gex > 0 ? -gex : gex;
        eng.verbose = verbose != 0;
        eng.mem.max_batch_bytes = 128ull << 20;
        eng.mem.max_batch_sequences = 10000000;
        eng.mem.max_temp_bytes = 4ull << 30;
        eng.mem.max_gpu_mem = SIZE_MAX;
        if (mem) eng.mem = *mem;
        if (eng.mem.max_temp_bytes == 0) eng.mem.max_temp_bytes = 4ull << 30;
        if (eng.mem.max_gpu_mem == 0) eng.mem.max_gpu_mem = SIZE_MAX;
        eng.buildMatrix();
        eng.checkGaps();
        if (num_top < 0) sw4::fail(SW4_ERR_INVALID, "num_top must be >= 0");
    });
    if (rc != SW4_OK) { delete h; return rc; }
    *out = h;
    return SW4_OK;
}

int sw4_destroy(sw4_handle* h) {
    delete h;
    return SW4_OK;
}

int sw4_set_gap_scores(sw4_handle* h, int gop, int gex) {
    if (!h) return SW4_ERR_INVALID;
    return guarded(h, [&] {
        const int a = gop > 0 ? -gop : gop, b = gex > 0 ? -gex : gex;  // src/cudasw4.cuh:539-550 negates positives
        const int oa = h->eng.gop, ob = h->eng.gex;
        h->eng.gop = a; h->eng.gex = b;
        try { h->eng.checkGaps(); } catch (...) { h->eng.gop = oa; h->eng.gex = ob; throw; }
    });
}

int sw4_set_num_top(sw4_handle* h, int num_top) {
    if (!h) return SW4_ERR_INVALID;
    return guarded(h, [&] {
        if (num_top < 0) sw4::fail(SW4_ERR_INVALID, "num_top must be >= 0");
        h->eng.numTop = num_top;
    });
}

int sw4_set_blosum(sw4_handle* h, int blosum) {
    if (!h) return SW4_ERR_INVALID;
    return guarded(h, [&] {
        const int old = h->eng.blosum;
        h->eng.blosum = blosum;
        try { h->eng.buildMatrix(); } catch (...) { h->eng.blosum = old; h->eng.buildMatrix(); throw; }
    });
}

int sw4_set_kernel_types(sw4_handle* h, int single_pass, int many_pass_small, int many_pass_large, int overflow) {
    if (!h) return SW4_ERR_INVALID;
    return guarded(h, [&] {
        const int v[4] = {single_pass, many_pass_small, many_pass_large, overflow};
        for (int x : v)
            if (x < 0 || x > 3) sw4::fail(SW4_ERR_INVALID, "invalid kernel type %d", x);
        // validity rules of src/cudasw4.cuh:841-855
        if (many_pass_large != SW4_KERNEL_FLOAT && many_pass_large != SW4_KERNEL_DPX_S32)
            sw4::fail(SW4_ERR_INVALID, "many_pass_large must be Float or DPXs32");
        if (overflow != SW4_KERNEL_FLOAT && overflow != SW4_KERNEL_DPX_S32)
            sw4::fail(SW4_ERR_INVALID, "overflow type must be Float or DPXs32");
        for (int i = 0; i < 4; i++) h->eng.kernelTypes[i] = v[i];
    });
}

int sw4_set_mem_config(sw4_handle* h, const sw4_mem_config* mem) {
    if (!h || !mem) return SW4_ERR_INVALID;
    return guarded(h, [&] {
        h->eng.mem = *mem;
        if (h->eng.mem.max_temp_bytes == 0) h->eng.mem.max_temp_bytes = 4ull << 30;
        if (h->eng.mem.max_gpu_mem == 0) h->eng.mem.max_gpu_mem = SIZE_MAX;
        for (auto& sh : h->eng.shards) sh->uploaded = false;  // planned and uploaded again on the next use
    });
}

int sw4_set_shard(sw4_handle* h, int rank, int world) {
    if (!h) return SW4_ERR_INVALID;
    return guarded(h, [&] {
        if (world < 1 || rank < 0 || rank >= world) sw4::fail(SW4_ERR_INVALID, "invalid shard %d of %d", rank, world);
        if (h->eng.db) sw4::fail(SW4_ERR_INVALID, "sw4_set_shard must be called before a database is set");
        h->eng.shardRank = rank;
        h->eng.shardWorld = world;
    });
}

int sw4_set_database_files(sw4_handle* h, const char* db_prefix, int prefetch) {
    if (!h || !db_prefix) return SW4_ERR_INVALID;
    return guarded(h, [&] {
        auto db = std::make_unique<sw4::HostDB>();
        const std::string p = std::string(db_prefix) + "0";
        db->fChars.open(p + "chars", prefetch != 0);
        db->fOffsets.open(p + "offsets", true);
        db->fLengths.open(p + "lengths", true);
        db->fHeaders.open(p + "headers", false);
        db->fHeaderOffsets.open(p + "headeroffsets", false);
        db->n = db->fLengths.size / sizeof(int32_t);
        if (db->fOffsets.size != (db->n + 1) * sizeof(size_t) || db->fHeaderOffsets.size != (db->n + 1) * sizeof(size_t))
            sw4::fail(SW4_ERR_IO, "inconsistent database files for prefix %s", db_prefix);
        db->chars = (const uint8_t*)db->fChars.ptr;
        db->offsets = (const size_t*)db->fOffsets.ptr;
        db->lengths = (const int32_t*)db->fLengths.ptr;
        db->headers = (const char*)db->fHeaders.ptr;
        db->headerOffsets = (const size_t*)db->fHeaderOffsets.ptr;
        if (db->n && db->offsets[db->n] > db->fChars.size) sw4::fail(SW4_ERR_IO, "chars file too small for prefix %s", db_prefix);
        db->finish();
        h->eng.db = std::move(db);
        h->eng.assignShards();
    });
}

int sw4_set_database_memory(sw4_handle* h, const char* chars, const size_t* offsets, const int32_t* lengths, const char* headers,
                            const size_t* header_offsets, size_t num_sequences) {
    return sw4_set_database_shard_memory(h, chars, offsets, lengths, headers, header_offsets, num_sequences, nullptr, num_sequences);
}

int sw4_set_database_shard_memory(sw4_handle* h, const char* chars, const size_t* offsets, const int32_t* lengths, const char* headers,
                                  const size_t* header_offsets, size_t num_sequences, const int32_t* global_ids,
                                  size_t num_sequences_global) {
    if (!h) return SW4_ERR_INVALID;
    return guarded(h, [&] {
        if (num_sequences && (!chars || !offsets || !lengths)) sw4::fail(SW4_ERR_INVALID, "null database arrays");
        if (global_ids && num_sequences_global < num_sequences) sw4::fail(SW4_ERR_INVALID, "num_sequences_global < num_sequences");
        auto db = std::make_unique<sw4::HostDB>();
        db->chars = (const uint8_t*)chars;
        db->offsets = offsets;
        db->lengths = lengths;
        db->headers = headers;
        db->headerOffsets = headers ? header_offsets : nullptr;
        db->n = num_sequences;
        db->globalIds = global_ids;
        db->nGlobal = global_ids ? num_sequences_global : num_sequences;
        db->finish();
        h->eng.db = std::move(db);
        h->eng.assignShards();
    });
}

int sw4_set_pseudo_database(sw4_handle* h, size_t num_sequences, int length, int seed) {
    if (!h) return SW4_ERR_INVALID;
    return guarded(h, [&] {
        if (length < 0) sw4::fail(SW4_ERR_INVALID, "negative length");
        auto db = std::make_unique<sw4::HostDB>();
        // reference src/dbdata.hpp:219-246: one random subject, replicated
        static const char letters[] = "ARNDCQEGHILKMFPSTWYV";
        std::mt19937 gen(seed);
        std::uniform_int_distribution<> dist(0, 19);
        std::vector<uint8_t> one(length);
        for (int i = 0; i < length; i++) {
            const char c = letters[dist(gen)];
            one[i] = (uint8_t)(strchr(letters, c) - letters);
        }
        const size_t padded = ((size_t)length + 3) / 4 * 4;
        db->vChars.assign(num_sequences * padded, 20);
        db->vOffsets.resize(num_sequences + 1);
        db->vLengths.assign(num_sequences, length);
        db->vHeaders.assign(num_sequences, 'H');
        db->vHeaderOffsets.resize(num_sequences + 1);
        for (size_t i = 0; i < num_sequences; i++) {
            db->vOffsets[i] = i * padded;
            db->vHeaderOffsets[i] = i;
            if (length) memcpy(db->vChars.data() + i * padded, one.data(), (size_t)length);
        }
        db->vOffsets[num_sequences] = num_sequences * padded;
        db->vHeaderOffsets[num_sequences] = num_sequences;
        db->chars = db->vChars.data();
        db->offsets = db->vOffsets.data();
        db->lengths = db->vLengths.data();
        db->headers = db->vHeaders.data();
        db->headerOffsets = db->vHeaderOffsets.data();
        db->n = num_sequences;
        db->finish();
        h->eng.db = std::move(db);
        h->eng.assignShards();
    });
}

// Deterministic synthetic database with a given length distribution (the benchmark shapes SURVEY.md 8-d names: no
// network, so the real UniProt files are not available). A generalisation of the reference's PseudoDB
// (src/dbdata.hpp:219-272), which can only replicate one sequence: residue p of sequence `id` is
//   kPseudoResidue[ byte (p & 7) of mix64(mix64(seed + id) + (p >> 3)) ]
// (splitmix64 finaliser; byte -> residue code by UniProt background frequencies in 1/256 steps), so every rank of a
// multi-process run can generate exactly its own shard (sw4_set_shard) of the same database, and a checker can
// re-create any single sequence (cudasw4_b200/synth.py: pseudo_lengths_sequence).
static inline uint64_t sw4_mix64(uint64_t z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

int sw4_set_pseudo_database_lengths(sw4_handle* h, const int32_t* lengths, size_t num_sequences, uint64_t seed,
                                    const int32_t* planted_ids, const uint8_t* const* planted_codes, int32_t num_planted) {
    if (!h) return SW4_ERR_INVALID;
    return guarded(h, [&] {
        if (num_sequences && !lengths) sw4::fail(SW4_ERR_INVALID, "null lengths");
        if (num_planted < 0 || (num_planted > 0 && (!planted_ids || !planted_codes))) sw4::fail(SW4_ERR_INVALID, "invalid planted list");
        if (num_sequences > (size_t)0x7ffffffe) sw4::fail(SW4_ERR_INVALID, "too many sequences");
        uint8_t table[256];
        for (int b = 0, c = 0; b < 256; b++) { while (b >= sw4::kPseudoCumulative[c]) c++; table[b] = (uint8_t)c; }
        auto db = std::make_unique<sw4::HostDB>();
        const size_t rank = (size_t)h->eng.shardRank, world = (size_t)h->eng.shardWorld;
        const size_t numBlocks = (num_sequences + sw4::kShardBlock - 1) / sw4::kShardBlock;
        // this rank's sequences: blocks rank, rank + world, ... of the length-sorted database (as assignShards cuts it)
        std::vector<int32_t>& ids = db->vGlobalIds;
        for (size_t b = rank; b < numBlocks; b += world)
            for (size_t i = b * sw4::kShardBlock; i < std::min(num_sequences, (b + 1) * sw4::kShardBlock); i++) ids.push_back((int32_t)i);
        const size_t n = ids.size();
        db->vLengths.resize(n);
        db->vOffsets.resize(n + 1);
        db->vOffsets[0] = 0;
        for (size_t i = 0; i < n; i++) {
            const int32_t len = lengths[ids[i]];
            if (len < 0) sw4::fail(SW4_ERR_INVALID, "negative length at %d", ids[i]);
            db->vLengths[i] = len;
            db->vOffsets[i + 1] = db->vOffsets[i] + ((size_t)len + 3) / 4 * 4;
        }
        db->vChars.resize(db->vOffsets[n]);
        const int nt = (int)std::max(1u, std::min(32u, std::thread::hardware_concurrency()));
        auto work = [&](int t) {
            for (size_t i = (size_t)t * sw4::kShardBlock; i < n; i += (size_t)nt * sw4::kShardBlock)
                for (size_t j = i; j < std::min(n, i + sw4::kShardBlock); j++) {
                    uint8_t* dst = db->vChars.data() + db->vOffsets[j];
                    const size_t len = (size_t)db->vLengths[j], padded = db->vOffsets[j + 1] - db->vOffsets[j];
                    const uint64_t key = sw4_mix64(seed + (uint64_t)ids[j]);
                    for (size_t p = 0; p < len; p += 8) {
                        uint64_t w = sw4_mix64(key + (p >> 3));
                        const size_t m = std::min<size_t>(8, len - p);
                        for (size_t x = 0; x < m; x++, w >>= 8) dst[p + x] = table[w & 0xff];
                    }
                    for (size_t p = len; p < padded; p++) dst[p] = 20;
                }
        };
        {
            std::vector<std::thread> th;
            for (int t = 1; t < nt; t++) th.emplace_back(work, t);
            work(0);
            for (auto& t : th) t.join();
        }
        for (int k = 0; k < num_planted; k++) {  // planted sequences overwrite their slot (same length by construction)
            const int32_t gid = planted_ids[k];
            if (gid < 0 || (size_t)gid >= num_sequences) sw4::fail(SW4_ERR_INVALID, "planted id %d out of range", gid);
            const auto it = std::lower_bound(ids.begin(), ids.end(), gid);
            if (it == ids.end() || *it != gid) continue;  // another rank's sequence
            const size_t j = (size_t)(it - ids.begin());
            memcpy(db->vChars.data() + db->vOffsets[j], planted_codes[k], (size_t)db->vLengths[j]);
        }
        db->chars = db->vChars.data();
        db->offsets = db->vOffsets.data();
        db->lengths = db->vLengths.data();
        db->globalIds = ids.data();
        db->n = n;
        db->nGlobal = num_sequences;
        db->finish();
        h->eng.db = std::move(db);
        h->eng.assignShards();
    });
}

int sw4_upload_database(sw4_handle* h) {
    if (!h) return SW4_ERR_INVALID;
    return guarded(h, [&] { h->eng.upload(); });
}

int sw4_scan(sw4_handle* h, const char* query, int32_t query_length, int32_t* out_scores, int32_t* out_ids, int32_t* out_count,
             sw4_stats* stats) {
    if (!h) return SW4_ERR_INVALID;
    return guarded(h, [&] {
        if (h->eng.numTop > 0 && (!out_scores || !out_ids)) sw4::fail(SW4_ERR_INVALID, "null output arrays");
        h->eng.scan(query, query_length, nullptr, out_scores, out_ids, out_count, stats);
    });
}

// (pssms == nullptr: sequence queries)
static int scanManyQueries(sw4_handle* h, const char* const* queries, const int8_t* const* pssms, const int32_t* query_lengths,
                           int32_t num_queries, int32_t* out_scores, int32_t* out_ids, int32_t* out_counts, sw4_stats* per_query_stats,
                           sw4_stats* total_stats) {
    if (!h) return SW4_ERR_INVALID;
    return guarded(h, [&] {
        if (num_queries < 0 || (num_queries > 0 && (!queries || !query_lengths))) sw4::fail(SW4_ERR_INVALID, "invalid query list");
        if (h->eng.numTop > 0 && num_queries > 0 && (!out_scores || !out_ids)) sw4::fail(SW4_ERR_INVALID, "null output arrays");
        std::vector<sw4::QueryRef> q((size_t)num_queries);
        for (int i = 0; i < num_queries; i++) {
            q[i] = sw4::QueryRef{queries[i], query_lengths[i], pssms ? pssms[i] : nullptr};
            if (pssms && query_lengths[i] > 0 && !pssms[i]) sw4::fail(SW4_ERR_INVALID, "null pssm of query %d", i);
        }
        if (total_stats) memset(total_stats, 0, sizeof(*total_stats));
        h->eng.scanMany(q.data(), num_queries, out_scores, out_ids, out_counts, per_query_stats, total_stats);
    });
}

int sw4_scan_many(sw4_handle* h, const char* const* queries, const int32_t* query_lengths, int32_t num_queries, int32_t* out_scores,
                  int32_t* out_ids, int32_t* out_counts, sw4_stats* per_query_stats, sw4_stats* total_stats) {
    return scanManyQueries(h, queries, nullptr, query_lengths, num_queries, out_scores, out_ids, out_counts, per_query_stats, total_stats);
}

int sw4_alignment_coordinates(sw4_handle* h, const char* query, int32_t query_length, const int32_t* ids, int32_t num_ids,
                              sw4_alignment* out, sw4_stats* stats) {
    if (!h) return SW4_ERR_INVALID;
    return guarded(h, [&] { h->eng.alignmentCoordinates(query, query_length, nullptr, ids, num_ids, out, stats); });
}

int sw4_alignment_traceback(sw4_handle* h, const char* query, int32_t query_length, const int32_t* ids, int32_t num_ids,
                            sw4_alignment_summary* out, sw4_stats* stats) {
    if (!h) return SW4_ERR_INVALID;
    const int rc = guarded(h, [&] { h->eng.alignmentTraceback(query, query_length, nullptr, ids, num_ids, out, stats); });
    if (rc != SW4_OK) h->eng.lastCigars.clear();
    return rc;
}

// ---- PSSM queries: the same calls with a [query_length][21] position-specific scoring matrix ----
// (an empty query may come with a NULL pssm: it still runs as a PSSM query, with no rows)
static const int8_t kNoPssmRows[1] = {0};
static const int8_t* pssmQuery(const char* query, const int8_t* pssm, int32_t query_length) {
    if (query_length > 0 && (!query || !pssm)) sw4::fail(SW4_ERR_INVALID, "null query letters or pssm");
    return pssm ? pssm : kNoPssmRows;
}

int sw4_scan_pssm(sw4_handle* h, const char* query, const int8_t* pssm, int32_t query_length, int32_t* out_scores, int32_t* out_ids,
                  int32_t* out_count, sw4_stats* stats) {
    if (!h) return SW4_ERR_INVALID;
    return guarded(h, [&] {
        const int8_t* rows = pssmQuery(query, pssm, query_length);
        if (h->eng.numTop > 0 && (!out_scores || !out_ids)) sw4::fail(SW4_ERR_INVALID, "null output arrays");
        h->eng.scan(query, query_length, rows, out_scores, out_ids, out_count, stats);
    });
}

int sw4_scan_many_pssm(sw4_handle* h, const char* const* queries, const int8_t* const* pssms, const int32_t* query_lengths,
                       int32_t num_queries, int32_t* out_scores, int32_t* out_ids, int32_t* out_counts, sw4_stats* per_query_stats,
                       sw4_stats* total_stats) {
    if (!h) return SW4_ERR_INVALID;
    if (num_queries > 0 && !pssms) return guarded(h, [] { sw4::fail(SW4_ERR_INVALID, "null pssm list"); });
    std::vector<const int8_t*> p((size_t)std::max(num_queries, 0));  // (scanManyQueries refuses a NULL pssm of a non-empty query)
    for (size_t i = 0; i < p.size(); i++) p[i] = pssms[i] || (query_lengths && query_lengths[i] > 0) ? pssms[i] : kNoPssmRows;
    return scanManyQueries(h, queries, p.data(), query_lengths, num_queries, out_scores, out_ids, out_counts, per_query_stats, total_stats);
}

int sw4_alignment_coordinates_pssm(sw4_handle* h, const char* query, const int8_t* pssm, int32_t query_length, const int32_t* ids,
                                   int32_t num_ids, sw4_alignment* out, sw4_stats* stats) {
    if (!h) return SW4_ERR_INVALID;
    return guarded(h, [&] {
        h->eng.alignmentCoordinates(query, query_length, pssmQuery(query, pssm, query_length), ids, num_ids, out, stats);
    });
}

int sw4_alignment_traceback_pssm(sw4_handle* h, const char* query, const int8_t* pssm, int32_t query_length, const int32_t* ids,
                                 int32_t num_ids, sw4_alignment_summary* out, sw4_stats* stats) {
    if (!h) return SW4_ERR_INVALID;
    const int rc = guarded(h, [&] {
        h->eng.alignmentTraceback(query, query_length, pssmQuery(query, pssm, query_length), ids, num_ids, out, stats);
    });
    if (rc != SW4_OK) h->eng.lastCigars.clear();
    return rc;
}

int sw4_build_pssm(sw4_handle* h, const char* query, const int8_t* pssm, int32_t query_length, const int32_t* ids, int32_t num_ids,
                   double beta, int8_t* out, sw4_stats* stats) {
    if (!h) return SW4_ERR_INVALID;
    return guarded(h, [&] {
        h->eng.buildPssm(query, query_length, pssm ? pssmQuery(query, pssm, query_length) : nullptr, ids, num_ids, beta, out, stats);
    });
}

int sw4_search_iterative(sw4_handle* h, const char* query, int32_t query_length, int32_t max_iterations, double inclusion_evalue,
                         double beta, int32_t* out_scores, int32_t* out_ids, int32_t* out_count, int8_t* out_pssm,
                         int32_t* out_iterations, int32_t* out_converged, sw4_stats* stats) {
    if (!h) return SW4_ERR_INVALID;
    return guarded(h, [&] {
        h->eng.searchIterative(query, query_length, max_iterations, inclusion_evalue, beta, out_scores, out_ids, out_count, out_pssm,
                               out_iterations, out_converged, stats);
    });
}

int sw4_last_cigars(const sw4_handle* h, const char** text, size_t* length) {
    if (!h || !text || !length) return SW4_ERR_INVALID;
    *text = h->eng.lastCigars.c_str();
    *length = h->eng.lastCigars.size();
    return SW4_OK;
}

int sw4_set_score_statistics(sw4_handle* h, int enabled, double max_evalue) {
    if (!h) return SW4_ERR_INVALID;
    return guarded(h, [&] {
        if (std::isnan(max_evalue) || max_evalue < 0) sw4::fail(SW4_ERR_INVALID, "max_evalue must be >= 0 or INFINITY (got %g)", max_evalue);
        h->eng.statsEnabled = enabled != 0;
        h->eng.maxEvalue = max_evalue;
    });
}

// (query_index of the last scan call; fails when it ran without statistics)
static const char* lastStatsError(const sw4_handle* h, int32_t query_index) {
    if (h->eng.lastStats.empty()) return "the last scan ran without score statistics (sw4_set_score_statistics)";
    if (query_index < 0 || (size_t)query_index >= h->eng.lastStats.size()) return "query_index out of range";
    return nullptr;
}

int sw4_last_score_statistics(const sw4_handle* h, int32_t query_index, sw4_score_statistics* out) {
    if (!h || !out) return SW4_ERR_INVALID;
    if (const char* e = lastStatsError(h, query_index)) { const_cast<sw4_handle*>(h)->eng.lastError = e; return SW4_ERR_INVALID; }
    *out = h->eng.lastStats[(size_t)query_index];
    return SW4_OK;
}

int sw4_last_score_histogram(const sw4_handle* h, int32_t query_index, int64_t* counts, int64_t* lensums, int32_t bins) {
    if (!h || !counts || !lensums) return SW4_ERR_INVALID;
    const char* e = lastStatsError(h, query_index);
    if (!e && bins != SW4_SCORE_BINS) e = "bins must be SW4_SCORE_BINS";
    if (e) { const_cast<sw4_handle*>(h)->eng.lastError = e; return SW4_ERR_INVALID; }
    const std::vector<int64_t>& hist = h->eng.lastHists[(size_t)query_index];
    memcpy(counts, hist.data(), sw4::kHistEntries * sizeof(int64_t));
    memcpy(lensums, hist.data() + sw4::kHistEntries, sw4::kHistEntries * sizeof(int64_t));
    return SW4_OK;
}

int sw4_last_scan_all_scores(sw4_handle* h, int32_t* out_scores, int32_t* out_ids, size_t capacity, size_t* out_count) {
    if (!h) return SW4_ERR_INVALID;
    return guarded(h, [&] {
        size_t total = 0;
        for (auto& sh : h->eng.shards) total += sh->n;
        if (capacity < total) sw4::fail(SW4_ERR_INVALID, "capacity %zu < %zu", capacity, total);
        size_t pos = 0;
        for (auto& shp : h->eng.shards) {
            sw4::Shard& sh = *shp;
            if (!sh.uploaded || sh.lastCtx < 0) sw4::fail(SW4_ERR_INVALID, "no scan has run yet");
            SW4_CUDA(cudaSetDevice(sh.device));
            SW4_CUDA(cudaMemcpy(out_scores + pos, sh.ctxs[sh.lastCtx]->dScores.p, sh.n * sizeof(int32_t), cudaMemcpyDeviceToHost));
            if (out_ids)
                for (size_t i = 0; i < sh.n; i++) out_ids[pos + i] = h->eng.globalIdOf(sh, i);
            pos += sh.n;
        }
        if (out_count) *out_count = total;
    });
}

// (a pre-sharded handle only knows the sequences of its own shard: other ids are SW4_ERR_INVALID)
int sw4_reference_header(const sw4_handle* h, int32_t gid, const char** ptr, size_t* len) {
    if (!h || !h->eng.db || gid < 0 || !ptr || !len) return SW4_ERR_INVALID;
    const sw4::HostDB& db = *h->eng.db;
    const size_t id = db.localIndex(gid);
    if (id >= db.n) return SW4_ERR_INVALID;
    if (!db.headers) { *ptr = ""; *len = 0; return SW4_OK; }
    *ptr = db.headers + db.headerOffsets[id];
    *len = db.headerOffsets[id + 1] - db.headerOffsets[id];
    return SW4_OK;
}

int sw4_reference_length(const sw4_handle* h, int32_t gid, int32_t* len) {
    if (!h || !h->eng.db || gid < 0 || !len) return SW4_ERR_INVALID;
    const size_t id = h->eng.db->localIndex(gid);
    if (id >= h->eng.db->n) return SW4_ERR_INVALID;
    *len = h->eng.db->lengths[id];
    return SW4_OK;
}

int sw4_reference_sequence(const sw4_handle* h, int32_t gid, char* out, size_t capacity, size_t* len) {
    if (!h || !h->eng.db || gid < 0) return SW4_ERR_INVALID;
    const sw4::HostDB& db = *h->eng.db;
    const size_t id = db.localIndex(gid);
    if (id >= db.n) return SW4_ERR_INVALID;
    const size_t L = (size_t)db.lengths[id];
    if (len) *len = L;
    if (!out) return SW4_OK;
    if (capacity < L) return SW4_ERR_INVALID;
    static const char inv[] = "ARNDCQEGHILKMFPSTWYV-";  // src/convert.cuh:36-64
    const uint8_t* s = db.chars + db.offsets[id];
    for (size_t i = 0; i < L; i++) out[i] = inv[s[i] > 20 ? 20 : s[i]];
    return SW4_OK;
}

int sw4_total_timer_start(sw4_handle* h) {
    if (!h) return SW4_ERR_INVALID;
    h->eng.totalStart = std::chrono::steady_clock::now();
    h->eng.totalCells = 0;
    h->eng.totalOverflows = 0;
    return SW4_OK;
}

int sw4_total_timer_stop(sw4_handle* h, sw4_stats* stats) {
    if (!h || !stats) return SW4_ERR_INVALID;
    const double s = std::chrono::duration<double>(std::chrono::steady_clock::now() - h->eng.totalStart).count();
    memset(stats, 0, sizeof(*stats));
    stats->seconds = s;
    stats->cells = h->eng.totalCells;
    stats->gcups = s > 0 ? h->eng.totalCells / 1e9 / s : 0;
    stats->num_overflows = h->eng.totalOverflows;
    return SW4_OK;
}

int sw4_get_db_info(const sw4_handle* h, sw4_db_info* info) {
    if (!h || !info || !h->eng.db) return SW4_ERR_INVALID;
    const sw4::HostDB& db = *h->eng.db;
    memset(info, 0, sizeof(*info));
    info->num_sequences = db.nGlobal;
    info->num_residues = db.residues;
    info->min_length = db.minLen;
    info->max_length = db.maxLen;
    size_t pos = 0;
    for (int p = 0; p < 36; p++) {  // membership b[i-1] < len <= b[i], src/cudasw4.cuh:904-926
        const size_t end = std::upper_bound(db.lengths + pos, db.lengths + db.n, sw4::kRefBoundaries[p]) - db.lengths;
        info->partition_counts[p] = end - pos;
        pos = end;
    }
    info->shard_rank = h->eng.shardRank;
    info->shard_world = h->eng.shardWorld;
    for (auto& sh : h->eng.shards) {
        info->shard_sequences += sh->n;
        info->shard_residues += sh->residues;
        if (sh->uploaded) {
            info->streaming |= sh->streaming ? 1 : 0;
            info->num_batches = std::max<int32_t>(info->num_batches, (int32_t)sh->batches.size());
        }
    }
    return SW4_OK;
}

}  // extern "C"
