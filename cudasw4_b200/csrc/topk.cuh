// Device-side top-k selection under the total order (score descending, database id ascending).
//
// Replaces the reference's "write 8 bytes per subject, radix-sort everything in chunks of 1e6, merge"
// (src/cudasw4.cuh:1365-1401, src/util.cuh:159-192) by a two-pass selection that reads the int32 score array once
// per pass and never materialises more than k candidates per block:
//   pass 1  every block owns a contiguous range of subjects. It finds the exact k-th largest score T of its range with
//           two shared-memory histograms (score >> shift, then the low `shift` bits inside the deciding bin) and emits
//           all entries above T plus the first (k - #above) entries equal to T in index order: exactly its local
//           top-k. The host picks shift (8..12) from an upper bound of the scan's scores (15 x min(query, longest
//           subject)) so that no score is ever clipped; scans whose bound reaches 2^24 are refused (topk_shift_for).
//   pass 2  one block bitonic-sorts the <= 8192 surviving (score, index) keys and writes the k best with global ids.
// Shard-local indices are ascending in global id, so "first in index order" is the reference's tie rule
// (ascending DB id, SURVEY.md 0-3) without the 1e6-chunk artefact.
#pragma once
#include <algorithm>
#include <cstdint>
#include <cuda_runtime.h>

namespace sw4 {

constexpr int kTopkThreads = 1024;
constexpr int kTopkHiBins = 4096;     // score >> shift; level 2 has 1 << shift <= 4096 bins
constexpr int kTopkMaxShift = 12;     // => exact for scores below 2^24
constexpr int kTopkMaxCandidates = 8192;

struct TopkCand { int32_t score; int32_t index; };

__device__ __forceinline__ int topk_hi(int s, int shift) { return min(max(s, 0) >> shift, kTopkHiBins - 1); }

// smallest shift in [8, 12] such that (maxScore >> shift) < 4096, or -1 when even 12 is not enough
static inline int topk_shift_for(long long maxScore) {
    for (int sh = 8; sh <= kTopkMaxShift; sh++)
        if ((maxScore >> sh) < kTopkHiBins) return sh;
    return -1;
}


// Block-wide: given hist[0..nbins) in shared memory, find the highest bin b such that (count of entries in bins > b) < k
// <= (count in bins >= b), or b = 0 when even all bins together hold fewer than k. Returns (b, count above b) in
// sBin/sAbove. Every thread owns nbins/blockDim consecutive bins; the suffix sums come from a reverse block scan.
// baseAbove (entries above all of hist) is below k. Both barriers are unconditional: every thread derives the total
// from warpTotals itself, so no thread decides anything from sBin/sAbove while another one may be writing them.
__device__ __forceinline__ void topk_find_bin(const int* hist, int nbins, int k, int baseAbove, int* warpTotals, int* sBin,
                                              int* sAbove) {
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nthreads = blockDim.x;
    const int per = (nbins + nthreads - 1) / nthreads;
    // thread t owns bins [lo, hi) counted from the TOP: logical index i <-> bin nbins-1-i
    const int lo = tid * per, hi = min(nbins, lo + per);
    int mine = 0;
    for (int i = lo; i < hi; i++) mine += hist[nbins - 1 - i];
    // inclusive prefix over threads (in top-down order)
    int incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) warpTotals[w] = incl;
    __syncthreads();
    int before = baseAbove, total = baseAbove;
    for (int x = 0; x < (nthreads + 31) / 32; x++) {
        if (x < w) before += warpTotals[x];
        total += warpTotals[x];
    }
    const int exclusive = before + incl - mine;  // entries in bins above this thread's range
    if (exclusive < k && exclusive + mine >= k) {   // the crossing is inside this thread's bins (exactly one thread)
        int above = exclusive;
        for (int i = lo; i < hi; i++) {
            const int c = hist[nbins - 1 - i];
            if (above + c >= k) { *sBin = nbins - 1 - i; *sAbove = above; break; }
            above += c;
        }
    }
    if (total < k && tid == 0) {  // no crossing (fewer than k entries in total): bin 0 decides, everything above it is kept
        *sBin = 0;
        *sAbove = total - hist[0];
    }
    __syncthreads();
}

// scores[begin+i]; indexOf = begin+i (or indices[begin+i] when indices != nullptr, which must be ascending)
__global__ void __launch_bounds__(kTopkThreads) topk_pass1_kernel(const int32_t* __restrict__ scores,
                                                                  const int32_t* __restrict__ indices, long long n,
                                                                  int k, int shift, TopkCand* __restrict__ out) {
    __shared__ int hist[kTopkHiBins];
    __shared__ int warpTotals[kTopkThreads / 32];
    __shared__ int sBin, sAbove, sRunning, sEmitted, sDone;
    const int tid = threadIdx.x;
    const long long per = (n + gridDim.x - 1) / gridDim.x;
    const long long begin = per * blockIdx.x;
    const long long end = min(n, begin + per);
    TopkCand* myOut = out + (size_t)blockIdx.x * k;
    for (int i = tid; i < k; i += blockDim.x) myOut[i] = TopkCand{-1, 0x7fffffff};
    const long long cnt = end - begin;
    if (cnt <= 0) return;

    // ---- level 1: histogram of score >> shift ----
    for (int i = tid; i < kTopkHiBins; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    for (long long i = begin + tid; i < end; i += blockDim.x) atomicAdd(&hist[topk_hi(scores[i], shift)], 1);
    __syncthreads();
    topk_find_bin(hist, kTopkHiBins, k, 0, warpTotals, &sBin, &sAbove);  // bin b decides (or everything fits: b == 0)
    const int bin = sBin;
    const int aboveBin = sAbove;
    // ---- level 2: exact threshold inside the deciding bin (scores are never clipped, see topk_shift_for) ----
    __syncthreads();
    const int lowBins = 1 << shift;
    for (int i = tid; i < lowBins; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    for (long long i = begin + tid; i < end; i += blockDim.x) {
        const int s = scores[i];
        if (topk_hi(s, shift) == bin) atomicAdd(&hist[max(s, 0) & (lowBins - 1)], 1);
    }
    __syncthreads();
    topk_find_bin(hist, lowBins, k, aboveBin, warpTotals, &sBin, &sAbove);
    if (tid == 0) { sRunning = 0; sEmitted = 0; }
    __syncthreads();
    const int T = (bin << shift) | sBin;  // k-th largest score of this range (0 when the range holds fewer than k)
    const int need = k - sAbove;          // how many entries == T to keep
    // ---- emit: everything above T (unordered), then the first `need` entries equal to T in index order ----
    for (long long base = begin; base < end; base += blockDim.x) {
        const long long i = base + tid;
        int s = -1;
        if (i < end) s = scores[i];
        const bool isAbove = i < end && s > T;
        const bool isEq = i < end && max(s, 0) == T;
        if (isAbove) {
            const int pos = atomicAdd(&sEmitted, 1);
            myOut[pos] = TopkCand{s, indices ? indices[i] : (int32_t)i};
        }
        const unsigned bal = __ballot_sync(0xffffffffu, isEq);
        const int lane = tid & 31, w = tid >> 5;
        if (lane == 0) warpTotals[w] = __popc(bal);
        __syncthreads();
        int before = sRunning;
        for (int x = 0; x < w; x++) before += warpTotals[x];
        const int rank = before + __popc(bal & ((1u << lane) - 1u));
        if (isEq && rank < need) myOut[sAbove + rank] = TopkCand{s, indices ? indices[i] : (int32_t)i};
        __syncthreads();
        if (tid == 0) {
            int tot = 0;
            for (int x = 0; x < kTopkThreads / 32; x++) tot += warpTotals[x];
            sRunning += tot;
            // decided once, between barriers: the next chunk's atomicAdd on sEmitted must not reach a slower warp's test
            sDone = sRunning >= need && sEmitted >= sAbove;
        }
        __syncthreads();
        if (sDone) break;  // uniform: written before the barrier, next written after two more barriers
    }
}

// One block: sort numCand (<= 8192) candidates by (score desc, index asc), write the k best; index -> global id.
__global__ void __launch_bounds__(kTopkThreads) topk_pass2_kernel(const TopkCand* __restrict__ cand, int numCand, int k,
                                                                  const int32_t* __restrict__ globalIds,
                                                                  int32_t* __restrict__ outScores,
                                                                  int32_t* __restrict__ outIds, int* outCount) {
    extern __shared__ unsigned long long keys[];  // pow2 >= numCand
    int n2 = 1;
    while (n2 < numCand) n2 <<= 1;
    for (int i = threadIdx.x; i < n2; i += blockDim.x) {
        unsigned long long key = 0;  // sorts last
        if (i < numCand && cand[i].score >= 0)
            key = ((unsigned long long)(unsigned)(cand[i].score + 1) << 32) | (unsigned)(0x7fffffff - cand[i].index);
        keys[i] = key;
    }
    __syncthreads();
    for (int size = 2; size <= n2; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int i = threadIdx.x; i < n2 / 2; i += blockDim.x) {
                const int lo = 2 * i - (i & (stride - 1));
                const int hi = lo + stride;
                const bool desc = ((lo & size) == 0);
                const unsigned long long a = keys[lo], b = keys[hi];
                if ((a < b) == desc) { keys[lo] = b; keys[hi] = a; }
            }
            __syncthreads();
        }
    }
    int valid = 0;
    for (int i = threadIdx.x; i < k; i += blockDim.x) {
        const unsigned long long key = (i < n2) ? keys[i] : 0ull;
        if (key != 0) {
            const int idx = 0x7fffffff - (int)(unsigned)(key & 0xffffffffu);
            outScores[i] = (int)(key >> 32) - 1;
            outIds[i] = globalIds ? globalIds[idx] : idx;
        } else {
            outScores[i] = -1;
            outIds[i] = -1;
        }
    }
    if (threadIdx.x == 0) {
        for (int i = 0; i < k && i < n2; i++) valid += keys[i] != 0;
        *outCount = valid;
    }
}

// -----------------------------------------------------------------------------------------------------------------
// Result lists longer than pass 2 can sort in shared memory (k > kTopkMaxCandidates / 2; the reference accepts any
// --top, src/cudasw4.cuh:1365-1401): device-wide exact selection + global bitonic sort, nothing goes through the host.
//   1. two global histograms (score >> shift, then the low bits inside the deciding bin) give the exact k-th largest
//      score T and the number of entries above it;
//   2. every block counts its entries == T; an exclusive scan over the blocks ranks them in index order;
//   3. entries > T are appended in any order, the first (k - #above) entries == T in index order (= ascending id);
//   4. the k keys (score << 32 | ~index) are sorted descending by a bitonic network (2048-key chunks in shared memory,
//      larger strides in global memory) and written out with global ids.
// -----------------------------------------------------------------------------------------------------------------
constexpr int kTopkLargeBlocks = 592;     // blocks of the histogram / count / emit kernels (4 per SM)
constexpr int kTopkChunk = 2048;          // keys sorted per block in shared memory

struct TopkLargeState {   // device-resident scalars of one selection
    int bin, aboveBin;    // level 1 result
    int T, above;         // exact threshold and number of entries > T
    int emitted;          // append counter for entries > T
    int pad[3];
};

__global__ void __launch_bounds__(kTopkThreads) topkL_hist_kernel(const int32_t* __restrict__ scores, long long n, int shift,
                                                                  int level, const TopkLargeState* __restrict__ st,
                                                                  int* __restrict__ hist) {
    __shared__ int h[kTopkHiBins];
    for (int i = threadIdx.x; i < kTopkHiBins; i += blockDim.x) h[i] = 0;
    __syncthreads();
    const int bin = level ? st->bin : 0;
    const int lowMask = (1 << shift) - 1;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int s = scores[i];
        if (level == 0) atomicAdd(&h[topk_hi(s, shift)], 1);
        else if (topk_hi(s, shift) == bin) atomicAdd(&h[max(s, 0) & lowMask], 1);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < kTopkHiBins; i += blockDim.x)
        if (h[i]) atomicAdd(&hist[i], h[i]);
}

__global__ void __launch_bounds__(kTopkThreads) topkL_find_kernel(int* __restrict__ hist, int nbins, int k, int shift, int level,
                                                                  TopkLargeState* __restrict__ st) {
    __shared__ int h[kTopkHiBins];
    __shared__ int warpTotals[kTopkThreads / 32];
    __shared__ int sBin, sAbove;
    for (int i = threadIdx.x; i < nbins; i += blockDim.x) { h[i] = hist[i]; hist[i] = 0; }  // zeroed for the next level
    __syncthreads();
    topk_find_bin(h, nbins, k, level ? st->aboveBin : 0, warpTotals, &sBin, &sAbove);
    if (threadIdx.x == 0) {
        if (level == 0) { st->bin = sBin; st->aboveBin = sAbove; }
        else { st->T = (st->bin << shift) | sBin; st->above = sAbove; st->emitted = 0; }
    }
}

// blockEq[b] = number of entries == T in block b's contiguous range
__global__ void __launch_bounds__(kTopkThreads) topkL_count_kernel(const int32_t* __restrict__ scores, long long n,
                                                                   const TopkLargeState* __restrict__ st, int* __restrict__ blockEq) {
    __shared__ int cnt;
    if (threadIdx.x == 0) cnt = 0;
    __syncthreads();
    const long long per = (n + gridDim.x - 1) / gridDim.x;
    const long long begin = per * blockIdx.x, end = min(n, begin + per);
    const int T = st->T;
    int mine = 0;
    for (long long i = begin + threadIdx.x; i < end; i += blockDim.x) mine += (max(scores[i], 0) == T);
    if (mine) atomicAdd(&cnt, mine);
    __syncthreads();
    if (threadIdx.x == 0) blockEq[blockIdx.x] = cnt;
}

// in place: blockEq[b] <- sum of blockEq[0..b)   (one block, numBlocks <= 1024)
__global__ void __launch_bounds__(kTopkThreads) topkL_scan_kernel(int* __restrict__ blockEq, int numBlocks) {
    __shared__ int v[kTopkThreads];
    const int t = threadIdx.x;
    v[t] = t < numBlocks ? blockEq[t] : 0;
    __syncthreads();
    for (int o = 1; o < kTopkThreads; o <<= 1) {
        const int add = t >= o ? v[t - o] : 0;
        __syncthreads();
        v[t] += add;
        __syncthreads();
    }
    if (t < numBlocks) blockEq[t] = t ? v[t - 1] : 0;
}

__device__ __forceinline__ unsigned long long topk_key(int score, long long index) {
    return ((unsigned long long)(unsigned)(max(score, 0) + 1) << 32) | (unsigned)(0x7fffffff - (int)index);
}

__global__ void __launch_bounds__(kTopkThreads) topkL_emit_kernel(const int32_t* __restrict__ scores, long long n, int k,
                                                                  TopkLargeState* __restrict__ st, const int* __restrict__ blockEqExcl,
                                                                  unsigned long long* __restrict__ keys) {
    __shared__ int warpTotals[kTopkThreads / 32];
    __shared__ int sRunning;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const long long per = (n + gridDim.x - 1) / gridDim.x;
    const long long begin = per * blockIdx.x, end = min(n, begin + per);
    const int T = st->T, above = st->above, need = k - above;
    if (tid == 0) sRunning = blockEqExcl[blockIdx.x];
    __syncthreads();
    for (long long base = begin; base < end; base += blockDim.x) {
        const long long i = base + tid;
        const int s = i < end ? scores[i] : -1;
        if (i < end && s > T) keys[atomicAdd(&st->emitted, 1)] = topk_key(s, i);
        const bool isEq = i < end && max(s, 0) == T;
        const unsigned bal = __ballot_sync(0xffffffffu, isEq);
        if (lane == 0) warpTotals[w] = __popc(bal);
        __syncthreads();
        int before = sRunning;
        for (int x = 0; x < w; x++) before += warpTotals[x];
        const int rank = before + __popc(bal & ((1u << lane) - 1u));
        if (isEq && rank < need) keys[above + rank] = topk_key(s, i);
        __syncthreads();
        if (tid == 0) {
            int tot = 0;
            for (int x = 0; x < kTopkThreads / 32; x++) tot += warpTotals[x];
            sRunning += tot;
        }
        __syncthreads();
    }
}

// Bitonic network, descending overall. Element i is compared with i ^ stride; the pair is ordered descending when
// (i & size) == 0. One block handles one chunk of 2048 keys in shared memory for all strides below 2048:
// firstSize == 2: full sort of the chunk (sizes 2..2048); otherwise the tail (strides 1024..1) of merge step `firstSize`.
__global__ void __launch_bounds__(kTopkThreads) bitonic_chunk_kernel(unsigned long long* __restrict__ keys, long long firstSize) {
    __shared__ unsigned long long sh[kTopkChunk];
    const long long base = (long long)blockIdx.x * kTopkChunk;
    const int t = threadIdx.x;
    sh[t] = keys[base + t];
    sh[t + kTopkThreads] = keys[base + t + kTopkThreads];
    __syncthreads();
    const long long lastSize = firstSize == 2 ? kTopkChunk : firstSize;
    for (long long size = firstSize; size <= lastSize; size <<= 1) {
        for (int stride = (int)min((long long)kTopkChunk / 2, size >> 1); stride > 0; stride >>= 1) {
            const int lo = 2 * t - (t & (stride - 1));
            const int hi = lo + stride;
            const bool desc = (((base + lo) & size) == 0);
            const unsigned long long a = sh[lo], b = sh[hi];
            if ((a < b) == desc) { sh[lo] = b; sh[hi] = a; }
            __syncthreads();
        }
        if (firstSize != 2) break;
    }
    keys[base + t] = sh[t];
    keys[base + t + kTopkThreads] = sh[t + kTopkThreads];
}

__global__ void bitonic_global_kernel(unsigned long long* __restrict__ keys, long long half, long long size, long long stride) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= half) return;
    const long long lo = 2 * i - (i & (stride - 1));
    const long long hi = lo + stride;
    const bool desc = ((lo & size) == 0);
    const unsigned long long a = keys[lo], b = keys[hi];
    if ((a < b) == desc) { keys[lo] = b; keys[hi] = a; }
}

__global__ void topkL_write_kernel(const unsigned long long* __restrict__ keys, int k, const int32_t* __restrict__ globalIds,
                                   int32_t* __restrict__ outScores, int32_t* __restrict__ outIds, int* __restrict__ outCount) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) *outCount = k;
    if (i >= k) return;
    const unsigned long long key = keys[i];
    const int idx = 0x7fffffff - (int)(unsigned)(key & 0xffffffffu);
    outScores[i] = (int)(key >> 32) - 1;
    outIds[i] = globalIds ? globalIds[idx] : idx;
}

// Enqueue the whole large-k selection on `stream`. Scratch: hist[4096] ints, state, blockEq[kTopkLargeBlocks] ints
// (all inside `work`, >= topk_large_work_ints() ints, zero-initialised here), keys[pow2 >= max(k, 2048)].
static inline size_t topk_large_work_ints() { return kTopkHiBins + 16 + kTopkLargeBlocks; }
static inline long long topk_large_num_keys(long long k) {
    long long n2 = kTopkChunk;
    while (n2 < k) n2 <<= 1;
    return n2;
}
static inline int topk_large_enqueue(const int32_t* scores, long long n, int k, int shift, const int32_t* globalIds, int* work,
                                     unsigned long long* keys, int32_t* outScores, int32_t* outIds, int* outCount,
                                     cudaStream_t stream) {
    int launches = 0;
    int* hist = work;
    TopkLargeState* st = reinterpret_cast<TopkLargeState*>(work + kTopkHiBins);
    int* blockEq = work + kTopkHiBins + 16;
    const long long n2 = topk_large_num_keys(k);
    cudaMemsetAsync(work, 0, topk_large_work_ints() * sizeof(int), stream);
    cudaMemsetAsync(keys, 0, (size_t)n2 * sizeof(unsigned long long), stream);  // key 0 sorts last
    topkL_hist_kernel<<<kTopkLargeBlocks, kTopkThreads, 0, stream>>>(scores, n, shift, 0, st, hist);
    topkL_find_kernel<<<1, kTopkThreads, 0, stream>>>(hist, kTopkHiBins, k, shift, 0, st);
    topkL_hist_kernel<<<kTopkLargeBlocks, kTopkThreads, 0, stream>>>(scores, n, shift, 1, st, hist);
    topkL_find_kernel<<<1, kTopkThreads, 0, stream>>>(hist, 1 << shift, k, shift, 1, st);
    topkL_count_kernel<<<kTopkLargeBlocks, kTopkThreads, 0, stream>>>(scores, n, st, blockEq);
    topkL_scan_kernel<<<1, kTopkThreads, 0, stream>>>(blockEq, kTopkLargeBlocks);
    topkL_emit_kernel<<<kTopkLargeBlocks, kTopkThreads, 0, stream>>>(scores, n, k, st, blockEq, keys);
    launches += 7;
    const unsigned chunks = (unsigned)(n2 / kTopkChunk);
    bitonic_chunk_kernel<<<chunks, kTopkThreads, 0, stream>>>(keys, 2ll);
    launches++;
    for (long long size = 2 * kTopkChunk; size <= n2; size <<= 1) {
        for (long long stride = size >> 1; stride >= kTopkChunk; stride >>= 1) {
            bitonic_global_kernel<<<(unsigned)((n2 / 2 + 255) / 256), 256, 0, stream>>>(keys, n2 / 2, size, stride);
            launches++;
        }
        bitonic_chunk_kernel<<<chunks, kTopkThreads, 0, stream>>>(keys, size);
        launches++;
    }
    topkL_write_kernel<<<(k + 255) / 256, 256, 0, stream>>>(keys, k, globalIds, outScores, outIds, outCount);
    return launches + 1;
}

// -----------------------------------------------------------------------------------------------------------------
// Dispatch: the one place that picks the path, the shift and the pass-1 split.
// -----------------------------------------------------------------------------------------------------------------
static inline bool topk_uses_large_path(int k) { return k > kTopkMaxCandidates / 2; }

// Pass-1 blocks: at most one per SM, at most kTopkMaxCandidates / k (pass 2 sorts all their candidates in shared
// memory), and no more than one per 4096 entries. Block b owns [b * per, min(n, (b + 1) * per)), per = ceil(n / blocks).
static inline int topk_pass1_blocks(long long n, int k, int smCount) {
    const long long blocks = std::min<long long>(std::min<long long>(smCount, kTopkMaxCandidates / k), (n + 4095) / 4096);
    return (int)std::max<long long>(blocks, 1);
}

// On the current device, before its first topk_enqueue (repeating it is harmless): pass 2 sorts up to
// kTopkMaxCandidates keys in dynamic shared memory.
static inline cudaError_t topk_configure() {
    return cudaFuncSetAttribute(topk_pass2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kTopkMaxCandidates * 8);
}

// Top-k of scores[0..n) (all >= 0 and <= maxScore, 1 <= k <= n) under (score desc, index asc), written to
// outScores/outIds[0..k) (index -> globalIds[index] when globalIds != nullptr) and *outCount, enqueued on `stream`.
// Scratch: cand[kTopkMaxCandidates]; for the large path (topk_uses_large_path) also work[topk_large_work_ints()] and
// keys[topk_large_num_keys(k)]. Returns the number of kernels launched, or -1 (nothing launched) when maxScore >= 2^24.
static inline int topk_enqueue(const int32_t* scores, long long n, int k, long long maxScore, int smCount,
                               const int32_t* globalIds, TopkCand* cand, int* work, unsigned long long* keys,
                               int32_t* outScores, int32_t* outIds, int* outCount, cudaStream_t stream) {
    const int shift = topk_shift_for(maxScore);
    if (shift < 0) return -1;
    if (topk_uses_large_path(k))
        return topk_large_enqueue(scores, n, k, shift, globalIds, work, keys, outScores, outIds, outCount, stream);
    const int blocks = topk_pass1_blocks(n, k, smCount);
    topk_pass1_kernel<<<blocks, kTopkThreads, 0, stream>>>(scores, nullptr, n, k, shift, cand);
    const int numCand = blocks * k;
    int n2 = 1;
    while (n2 < numCand) n2 <<= 1;
    topk_pass2_kernel<<<1, kTopkThreads, (size_t)n2 * 8, stream>>>(cand, numCand, k, globalIds, outScores, outIds, outCount);
    return 2;
}

}  // namespace sw4
