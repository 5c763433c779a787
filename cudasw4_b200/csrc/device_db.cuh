// Device-resident database layout + per-query preparation kernels.
//
// Replaces the reference's GpuDatabaseAllocation / batch copy plans (src/gpudatabaseallocation.cuh:22-61,
// src/dbbatching.cuh:16-99) and the per-block LUT expansion + query staging (src/dpx_s16_kernels.cuh:55-69,
// src/cudasw4.cuh:1280-1310):
//   * raw shard      chars / offsets / lengths exactly as makedb stores them (used by the exact 32-bit kernel)
//   * pair-blocks    for every length class (G lanes x R columns): consecutive subjects of the length-sorted shard are
//                    paired, and column c of the pair is stored as the fused code f = s0[c] + 21*s1[c] (u16), padded
//                    with the 'other' code 20; one block = G*R*2 contiguous bytes = one coalesced cp.async burst
//   * query profile  prof[f][p] = (M[q_p][s1] << 16) | (M[q_p][s0] & 0xffff) for every query position p, built once per
//                    scan (441 x q words); positions >= q hold -16000 ("gap rows" of the kernel's schedule)
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace sw4 {

// letters -> residue codes (reference src/convert.cuh:6-34): the 20 upper-case letters in NCBI order, all else 20
__global__ void convert_query_kernel(const char* __restrict__ letters, uint8_t* __restrict__ codes, int n, int padTo) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= padTo) return;
    uint8_t c = 20;
    if (i < n) {
        const char a = letters[i];
        const char order[21] = "ARNDCQEGHILKMFPSTWYV";
#pragma unroll
        for (int k = 0; k < 20; k++)
            if (a == order[k]) c = (uint8_t)k;
    }
    codes[i] = c;
}

// Entry (f, p) of the profile. `scores` holds the 21 scores of query position p against residue codes 0..20: the
// matrix row of its residue code (sequence query) or row p of a position-specific scoring matrix (PSSM query).
template <bool PSSM>
__device__ __forceinline__ void build_profile_entry(const uint8_t* __restrict__ qcodes, int qlen, const int8_t* __restrict__ scores,
                                                    uint32_t* __restrict__ profile, int stride) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    const int f = blockIdx.y;  // fused pair: s0 = f % 21 (low half), s1 = f / 21 (high half)
    if (p >= stride) return;
    // (only for p < qlen) the first of the 21 scores, as an index into `scores`
    auto base = [&] { return (PSSM ? p : (int)qcodes[p]) * 21; };
    uint32_t v = 0xc180c180u;  // (-16000, -16000)
    if (f >= 483) {
        // rows 483..503: plain int32 plane for the exact 32-bit kernels (sw_s32_long_kernel, and sw_s32_kernel's PSSM form)
        v = p < qlen ? (uint32_t)(int32_t)scores[base() + (f - 483)] : (uint32_t)(-(1 << 28));
    } else if (f >= 441) {
        // rows 441..461: single-residue plane with the score in the low half, rows 462..482: the same in the high half
        // (sw_s16_long_kernel adds one entry of each)
        const int s = (f - 441) % 21;
        const bool high = f >= 462;
        const uint32_t m = p < qlen ? (uint32_t)(uint16_t)(int16_t)scores[base() + s] : 0xc180u;
        v = high ? (m << 16) : m;
    } else if (p < qlen) {
        const int b = base();
        const int lo = scores[b + f % 21], hi = scores[b + f / 21];
        v = ((uint32_t)(uint16_t)(int16_t)hi << 16) | (uint16_t)(int16_t)lo;
    }
    profile[(size_t)f * stride + p] = v;
}

__global__ void build_profile_kernel(const uint8_t* __restrict__ qcodes, int qlen, const int8_t* __restrict__ matrix,
                                     uint32_t* __restrict__ profile, int stride) {
    build_profile_entry<false>(qcodes, qlen, matrix, profile, stride);
}

// the profile of a PSSM query: pssm is [qlen][21], row p scoring query position p against residue codes 0..20
__global__ void build_profile_pssm_kernel(const int8_t* __restrict__ pssm, int qlen, uint32_t* __restrict__ profile, int stride) {
    build_profile_entry<true>(nullptr, qlen, pssm, profile, stride);
}

// Work items of a single-segment length class, generated on the device: consecutive subjects [first, first+count) are
// paired; item k = (first+2k, first+2k+1 or none) and owns pair-block k.
struct PairItem { int subject0, subject1, firstBlock, numSegments; };  // same layout as sw4::S16Item

__global__ void make_pair_items_kernel(PairItem* __restrict__ items, int numItems, int first, int count) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= numItems) return;
    const int s0 = first + 2 * k;
    items[k] = PairItem{s0, (2 * k + 1 < count) ? s0 + 1 : -1, k, 1};
}

// Residue codes above 20 become 20 and the padding bytes behind every sequence (up to the next multiple of 4) are set to
// 20, whatever the caller's arrays held there. One thread per 4-byte word; `wordSubject` is not needed: the padding is
// fixed per subject by a second launch dimension (one thread per subject).
__global__ void sanitize_codes_kernel(uint32_t* __restrict__ words, size_t numWords) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= numWords) return;
    const uint32_t w = words[i];
    uint32_t r = 0;
#pragma unroll
    for (int b = 0; b < 4; b++) {
        const uint32_t c = (w >> (8 * b)) & 0xffu;
        r |= (c > 20u ? 20u : c) << (8 * b);
    }
    if (r != w) words[i] = r;
}
__global__ void pad_codes_kernel(uint8_t* __restrict__ chars, const size_t* __restrict__ offsets,
                                 const int32_t* __restrict__ lengths, int count) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const size_t end = offsets[i + 1];
    for (size_t p = offsets[i] + (size_t)lengths[i]; p < end; p++) chars[p] = 20;
}

// One thread per (pair-block, 4 columns). blockItem[b] names the work item (a pair of subjects) block b belongs to
// (nullptr: block b belongs to item b); the block covers columns [seg*columns, (seg+1)*columns) of the pair,
// seg = b - item.firstBlock. `offsets` and `lengths` are indexed by the items' subject indices (the caller shifts the
// pointers when the block of sequences at `chars` does not start at subject 0). Sequences start on 4-byte boundaries
// and are padded with code 20 to a multiple of 4, so four columns of one subject are one aligned 32-bit load.
__global__ void build_pair_blocks_kernel(const uint8_t* __restrict__ chars, const size_t* __restrict__ offsets,
                                         const int32_t* __restrict__ lengths, const PairItem* __restrict__ items,
                                         const int32_t* __restrict__ blockItem, int numBlocks, int columns,
                                         uint16_t* __restrict__ cols) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int quads = columns >> 2;
    const long long total = (long long)numBlocks * quads;
    if (gid >= total) return;
    const int b = (int)(gid / quads), c = (int)(gid % quads) * 4;
    const PairItem it = items[blockItem ? blockItem[b] : b];
    const long long col = (long long)(b - it.firstBlock) * columns + c;
    uint32_t w0 = 0x14141414u, w1 = 0x14141414u;  // 20 20 20 20
    if (it.subject0 >= 0 && col < lengths[it.subject0]) w0 = *reinterpret_cast<const uint32_t*>(chars + offsets[it.subject0] + col);
    if (it.subject1 >= 0 && col < lengths[it.subject1]) w1 = *reinterpret_cast<const uint32_t*>(chars + offsets[it.subject1] + col);
    uint32_t f[4];
#pragma unroll
    for (int x = 0; x < 4; x++) f[x] = ((w0 >> (8 * x)) & 0xffu) + 21u * ((w1 >> (8 * x)) & 0xffu);
    uint2 out;
    out.x = f[0] | (f[1] << 16);
    out.y = f[2] | (f[3] << 16);
    *reinterpret_cast<uint2*>(cols + (size_t)b * columns + c) = out;
}

}  // namespace sw4
