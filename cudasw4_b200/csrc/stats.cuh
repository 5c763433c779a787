// Score histogram of one query's shard: the input of the E-value fit (sw4_fit_score_statistics, include/sw4b200.h).
// For every subject of length >= 1, bin s = min(score, SW4_SCORE_BINS) gets count += 1 and lensum += length; bin
// SW4_SCORE_BINS is the overflow bin. Length-0 subjects score 0 by definition, not by chance, and are left out.
//
// Null scores crowd into a few dozen bins, so every CTA keeps its own copy of the histogram in shared memory and a warp
// adds the lanes that hit the same bin in one step (__match_any_sync): the lowest lane of a group adds the group's count
// and the sum of its lengths. The CTA then adds its non-zero bins to the global int64 arrays. Integer sums make the
// result exact and independent of the schedule.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/sw4b200.h"

namespace sw4 {

constexpr int kHistThreads = 256;
constexpr int kHistEntries = SW4_SCORE_BINS + 1;                                  // bins + overflow bin
constexpr int kHistSmemBytes = kHistEntries * 2 * (int)sizeof(unsigned long long);  // count[] then lensum[]

// hist: [count[kHistEntries], lensum[kHistEntries]] in global memory (kHistSmemBytes), zeroed by the caller
__global__ void __launch_bounds__(kHistThreads) score_histogram_kernel(const int32_t* __restrict__ scores,
                                                                       const int32_t* __restrict__ lengths, long long n,
                                                                       unsigned long long* __restrict__ hist) {
    extern __shared__ unsigned long long sHist[];
    __shared__ int32_t sLen[kHistThreads];
    unsigned long long* sCount = sHist;
    unsigned long long* sLensum = sHist + kHistEntries;
    for (int b = threadIdx.x; b < 2 * kHistEntries; b += kHistThreads) sHist[b] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    // every lane of a warp runs the same number of iterations (__match_any_sync needs the whole warp)
    const long long stride = (long long)gridDim.x * kHistThreads;
    for (long long base = (long long)blockIdx.x * kHistThreads + (threadIdx.x & ~31); base < n; base += stride) {
        const long long i = base + lane;
        int bin = -1, len = 0;
        if (i < n) {
            len = lengths[i];
            if (len >= 1) bin = min(max(scores[i], 0), SW4_SCORE_BINS);
        }
        const unsigned peers = __match_any_sync(0xffffffffu, bin);
        sLen[threadIdx.x] = len;
        __syncwarp();
        if (bin >= 0 && lane == __ffs(peers) - 1) {
            unsigned long long sum = 0;
            for (unsigned m = peers; m; m &= m - 1) sum += (unsigned long long)sLen[(threadIdx.x & ~31) + __ffs(m) - 1];
            atomicAdd(&sCount[bin], (unsigned long long)__popc(peers));
            atomicAdd(&sLensum[bin], sum);
        }
        __syncwarp();
    }
    __syncthreads();
    for (int b = threadIdx.x; b < kHistEntries; b += kHistThreads) {
        if (sCount[b]) {
            atomicAdd(&hist[b], sCount[b]);
            atomicAdd(&hist[kHistEntries + b], sLensum[b]);
        }
    }
}

static inline cudaError_t score_histogram_configure() {
    return cudaFuncSetAttribute(score_histogram_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kHistSmemBytes);
}

// Enqueues the kernel over scores/lengths[0..n) on `stream` (hist zeroed before); returns the number of kernels launched.
// Three CTAs of 64 KiB fit an SM; a CTA takes at least 4096 subjects, so small shards use few CTAs and few flushes.
static inline int score_histogram_enqueue(const int32_t* scores, const int32_t* lengths, long long n, int smCount,
                                          unsigned long long* hist, cudaStream_t stream) {
    if (n <= 0) return 0;
    const long long want = (n + 4095) / 4096;
    const int grid = (int)(want < 3ll * smCount ? want : 3ll * smCount);
    score_histogram_kernel<<<grid, kHistThreads, kHistSmemBytes, stream>>>(scores, lengths, n, hist);
    return 1;
}

}  // namespace sw4
