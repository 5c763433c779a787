// Exact 32-bit Gotoh score kernel: one subject per warp, any subject / query length.
//
// Role (SURVEY.md 8-a3): (1) re-scoring of subjects whose packed 16-bit score saturated, (2) subjects longer than the
// register tile of the s16x2 kernel, (3) the always-correct path every other kernel is tested against on the device.
// It replaces the reference's NW_local_affine_{single,multi}_pass_dpx_s32 + device-side launcher
// (src/dpx_s32_kernels.cuh:273-1232) without dynamic parallelism: the work list is consumed by a persistent grid
// through an atomic ticket, longest subject first.
//
// Organisation: intra-sequence anti-diagonal wavefront. The subject is cut into tiles of 32*R columns; lane l owns
// R consecutive columns and is l query rows behind lane l-1 (values flow with __shfl_up). Between tiles the last
// column's (H, E) for every query row goes through a per-warp border array in global memory (read and written 32 rows
// at a time, coalesced). F never crosses a tile border (it runs along the query), so the result is the textbook
// recurrence bit for bit.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace sw4 {

constexpr int kS32Threads = 128;
constexpr int kS32WarpsPerBlock = kS32Threads / 32;
constexpr int kS32R = 16;                      // columns per lane -> 512 columns per tile
constexpr int kNegS32 = -(1 << 28);

struct S32Params {
    const uint8_t* chars;       // residue codes, makedb layout (shard-local)
    const size_t* offsets;      // [n+1]
    const int32_t* lengths;     // [n]
    const int32_t* list;        // local subject indices to score, ascending length (consumed from the back)
    const int* listCountPtr;    // number of entries (device memory: the overflow list is filled by another kernel)
    int listCountHost;          // used when listCountPtr == nullptr
    const uint8_t* query;       // query residue codes
    int qlen;
    const int8_t* matrix;       // 21x21 substitution scores
    int gop, gex;
    int2* border;               // [gridWarps][borderStride] (H, E) of the tile's last column per query row
    int borderStride;           // >= roundup32(qlen) + 32
    int* ticket;                // zero-initialised work counter
    int32_t* scores;            // [n]
    int statThreshold;          // subjects of reference partition 34 (240 < len <= 8000) scoring >= this are counted
    int* statCount;
};

// The body of both forms. Sequence form: row `row` scores Msm[21 * query[row] + code] (the matrix in shared memory).
// PSSM form: it scores prof[code * profStride + row], the int32 plane of the query profile (rows 483..503 of
// build_profile_kernel), so the query may have any length.
template <bool PSSM>
__device__ __forceinline__ void sw_s32_body(const S32Params& prm, const int32_t* __restrict__ prof, int profStride) {
    constexpr int R = kS32R;
    __shared__ int Msm[PSSM ? 1 : 21 * 21];
    if (!PSSM) {
        for (int i = threadIdx.x; i < 441; i += blockDim.x) Msm[i] = prm.matrix[i];
        __syncthreads();
    }
    const int lane = threadIdx.x & 31;
    const int warpGlobal = blockIdx.x * kS32WarpsPerBlock + (threadIdx.x >> 5);
    int2* border = prm.border + (size_t)warpGlobal * prm.borderStride;
    const int count = prm.listCountPtr ? *prm.listCountPtr : prm.listCountHost;
    const int q = prm.qlen, gop = prm.gop, gex = prm.gex;

    for (;;) {
        int item = 0;
        if (lane == 0) item = atomicAdd(prm.ticket, 1);
        item = __shfl_sync(0xffffffffu, item, 0);
        if (item >= count) break;
        const int subj = prm.list[count - 1 - item];
        const int len = prm.lengths[subj];
        const uint8_t* s = prm.chars + prm.offsets[subj];
        int best = 0;
        const int tiles = (len + 32 * R - 1) / (32 * R);
        for (int tile = 0; tile < tiles; tile++) {
            const int col0 = tile * 32 * R + lane * R;
            int srow[R];  // residue code (PSSM form: code * profStride); the query row is added per row
#pragma unroll
            for (int j = 0; j < R; j++) srow[j] = ((col0 + j < len) ? s[col0 + j] : 20) * (PSSM ? profStride : 1);
            int Hp[R], F[R];
#pragma unroll
            for (int j = 0; j < R; j++) { Hp[j] = 0; F[j] = kNegS32; }
            int Hlast = 0, Elast = kNegS32, HinPrev = 0;
            int2 inBuf = make_int2(0, kNegS32), outBuf = make_int2(0, 0);
            const bool firstTile = tile == 0, lastTile = tile == tiles - 1;
            const int steps = q + 31;
            for (int t = 0; t < steps; t++) {
                if (!firstTile && (t & 31) == 0) {  // next 32 rows of the left border, coalesced
                    const int r = t + lane;
                    inBuf = (r < q) ? border[r] : make_int2(0, kNegS32);
                }
                int Hin = __shfl_up_sync(0xffffffffu, Hlast, 1);
                int Ein = __shfl_up_sync(0xffffffffu, Elast, 1);
                const int bH = __shfl_sync(0xffffffffu, inBuf.x, t & 31);
                const int bE = __shfl_sync(0xffffffffu, inBuf.y, t & 31);
                if (lane == 0) { Hin = firstTile ? 0 : bH; Ein = firstTile ? kNegS32 : bE; }
                const int row = t - lane;
                if (row >= 0 && row < q) {
                    const int* Mrow = PSSM ? prof + row : Msm + 21 * prm.query[row];
                    int E = Ein, diag = HinPrev;
#pragma unroll
                    for (int j = 0; j < R; j++) {
                        const int d = diag + (PSSM ? __ldg(Mrow + srow[j]) : Mrow[srow[j]]);
                        diag = Hp[j];
                        const int h = __vimax3_s32_relu(d, E, F[j]);
                        Hp[j] = h;
                        const int tt = h + gop;
                        E = __viaddmax_s32(E, gex, tt);
                        F[j] = __viaddmax_s32(F[j], gex, tt);
                        best = max(best, h);
                    }
                    Hlast = Hp[R - 1];
                    Elast = E;
                    HinPrev = Hin;
                }
                if (!lastTile) {  // lane 31 finished row t-31: collect 32 rows, then store them coalesced
                    const int r31 = t - 31;
                    const int vH = __shfl_sync(0xffffffffu, Hlast, 31);
                    const int vE = __shfl_sync(0xffffffffu, Elast, 31);
                    if (r31 >= 0) {
                        if (lane == (r31 & 31)) outBuf = make_int2(vH, vE);
                        if ((r31 & 31) == 31 || r31 == q - 1) {
                            const int r = (r31 & ~31) + lane;
                            if (lane <= (r31 & 31)) border[r] = outBuf;
                        }
                    }
                }
            }
            __syncwarp();
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) best = max(best, __shfl_xor_sync(0xffffffffu, best, o));
        if (lane == 0) {
            prm.scores[subj] = best;
            if (best >= prm.statThreshold && len > 240 && len <= 8000) atomicAdd(prm.statCount, 1);
        }
    }
}

// (templates only so that the header can be included by several translation units)
template <int kInstance = 0>
__global__ void __launch_bounds__(kS32Threads) sw_s32_kernel(const S32Params prm) {
    sw_s32_body<false>(prm, nullptr, 0);
}

// PSSM queries: prof = the profile's int32 plane (profile + 483 * profStride); prm.query and prm.matrix are not read
template <int kInstance = 0>
__global__ void __launch_bounds__(kS32Threads) sw_s32_pssm_kernel(const S32Params prm, const int32_t* prof, int profStride) {
    sw_s32_body<true>(prm, prof, profStride);
}

}  // namespace sw4
