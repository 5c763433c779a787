// Alignment coordinates and traceback: exact 32-bit Gotoh passes that locate one optimal local alignment of a
// (query, subject) pair and recover its columns.
//
// Pass 1 (forward, kCoordEnds) runs the local recurrence over q x s and keeps the maximum S together with its first
// cell in (i, j) order: the end (qe, re). Pass 2 (kCoordBegins) runs over the reversed prefixes q[qe..0] x s[re..0]
// with the corner H(-1, -1) = kCoordAnchor, every other border H = 0 and E/F borders at minus infinity. A path from the
// corner carries kCoordAnchor + (score of an alignment that ends with the pair (qe, re)); a path restarted at the floor
// reaches at most S < kCoordAnchor. The optimal anchored alignments never dip below the anchor (a prefix of a score-S
// alignment scores >= 0, because its suffix is itself an alignment scoring <= S), so the maximum of pass 2 is exactly
// kCoordAnchor + S and its first cell in reversed (i, j) order is the lexicographically largest begin (qb, rb).
// The first cell holding a maximum is always a substitution cell: a gap cell with that value has a predecessor with the
// same value that comes earlier in (i, j) order.
//
// Pass 3 (kCoordTrace, sw4_alignment_traceback) is pass 2's argument mirrored: it runs forward over the rectangle
// q[qb..qe] x s[rb..re] with the corner H(-1, -1) = kCoordAnchor, every other border H = 0 and E/F at minus infinity.
// Every state value on an optimal anchored path is kCoordAnchor + (score of a prefix of a score-S alignment) >= the
// anchor: a prefix that ends in a gap column scores >= 0 as well, since dropping the gap columns at the head of its
// suffix leaves an alignment that scores at least as much as the suffix and at most S. A value connected to the floor is
// the score of some local alignment fragment, <= S < kCoordAnchor. So on the path the floor never ties, each H, E and F
// equals its anchored value, and the directions recorded there are exactly those of the anchored recurrence; the value
// at (qe, re) is kCoordAnchor + S (checked on the device). Per cell the pass records 4 bits:
//   bits 0-1  which state H takes, the first of P (0, diagonal), E (1), F (2) equal to it;
//   bit 2     E of the cell to the right extends this cell's E:  E + gex >= H + gop  (extend wins a tie);
//   bit 3     F of the cell below extends this cell's F:         F + gex >= H + gop.
// (The extension bits sit with the cell whose values decide them, so a walk that steps left or up reads one nibble for
// both its extension test and the next source.) Lane l's 16 columns of one row form one 64-bit word (column j in
// nibble j), stored in wavefront order: word ((tile * (rows + 31) + step) * 32 + lane), so every step of a warp is one
// 256-byte store and cell (i, c) is at tile c / 512, lane (c % 512) / 16, step i + lane.
//
// The walk (sw_coords_walk_kernel, one thread per pair) starts at (qe, re) in state P and follows the nibbles back to
// (qb, rb), writing the ops in reverse and counting identities, positives and gaps.
//
// Organisation: the wavefront of kernels_s32.cuh (lane l owns 16 consecutive columns of a 512-column tile and runs l
// query rows behind lane l-1; the last column's (H, E) crosses to the next tile through a border array in global memory).
// A CTA of 16 warps holds either up to 16 short pairs, one warp each (W = 1), or one long pair whose tiles are dealt
// round robin to W <= 16 warps: warp w runs tile t = w, w + W, ... and reads the border that warp w - 1 writes for tile
// t - 1, 32 rows at a time, after that warp has published them in shared memory. A warp overwrites its border array for
// tile t + W only after the W - 1 warps in between have advanced past those rows, so each border array is read before it
// is reused.
#pragma once
#include <climits>
#include <cstdint>
#include <cuda_runtime.h>

#include "kernels_s32.cuh"

namespace sw4 {

constexpr int kCoordThreads = 512;
constexpr int kCoordWarps = kCoordThreads / 32;
constexpr int kCoordR = kS32R;                    // columns per lane -> 512 columns per tile
constexpr int kCoordTileCols = 32 * kCoordR;
constexpr int kCoordAnchor = 1 << 24;             // scores stay below 2^24 (checked by the host)

struct CoordGroup { int firstItem, count, warps; };    // one per CTA: items [firstItem, firstItem + count), W warps each
struct CoordItem {
    size_t subjectOffset;   // into CoordParams::subjects
    size_t borderOffset;    // into CoordParams::border (warps * borderStride entries; unused for single-tile subjects)
    int subjectLength;
};

// pass 3 and the walk: one per traced pair (its rectangle; CoordItem holds the subject slice s[rb..re] and its length)
struct TraceItem {
    size_t words;           // first trace word of the pair in CoordParams::trace
    size_t ops;             // first op byte of the pair in CoordParams::ops (rows + cols bytes)
    int queryBegin, rows;   // qb, qe - qb + 1
    int score;              // S
};

struct CoordParams {
    const CoordGroup* groups;
    const CoordItem* items;
    const uint8_t* subjects;    // residue codes, gathered per call
    const uint8_t* query;       // query residue codes
    int qlen;
    const int8_t* matrix;       // 21x21
    int gop, gex;
    int2* border;
    int borderStride;           // >= qlen
    int4* ends;                 // [item] pass 1 writes (S, qe, re, 0); pass 2 reads it
    int32_t* out;               // [item][5] pass 2 writes (S, qb, qe, rb, re), -1 positions when S == 0
    int* errors;                // [0] pass 2 / pass 3: pairs whose anchored value is not kCoordAnchor + S; [1] the walk:
                                // pairs whose walk does not end at (qb, rb) in state P (both must stay 0)
    // pass 3 and the walk
    const TraceItem* traceItems;
    unsigned long long* trace;
    char* ops;                  // the walk writes the ops of each pair from its end: '=', 'X', 'I', 'D'
    int4* counts;               // [item] the walk writes (length, identities, positives, gaps)
    int numItems;
};

enum CoordMode { kCoordEnds = 0, kCoordBegins = 1, kCoordTrace = 2 };

// order of the tracker: value descending, then i ascending, then j ascending
__device__ __forceinline__ bool coord_better(int v, int i, int j, int bv, int bi, int bj) {
    return v > bv || (v == bv && (i < bi || (i == bi && j < bj)));
}

// PSSM: query position i scores pssm[21 * i + code] (a [qlen][21] table in global memory) instead of the matrix row
// of its residue code; prm.matrix is not read.
template <int MODE, bool PSSM = false>
__device__ __forceinline__ void coords_pass(const CoordParams& prm, const int8_t* __restrict__ pssm = nullptr) {
    constexpr bool REV = MODE == kCoordBegins, TRACE = MODE == kCoordTrace;
    constexpr int R = kCoordR;
    __shared__ int Msm[PSSM ? 1 : 21 * 21];
    __shared__ long long progress[kCoordWarps];  // (tile << 32) | rows of that tile's right border already stored
    __shared__ int redV[kCoordWarps], redI[kCoordWarps], redJ[kCoordWarps];
    if (!PSSM)
        for (int i = threadIdx.x; i < 441; i += blockDim.x) Msm[i] = prm.matrix[i];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) progress[warp] = -1;
    __syncthreads();
    const CoordGroup g = prm.groups[blockIdx.x];
    const int W = g.warps;
    const int slot = warp / W, wi = warp % W;
    const int item = g.firstItem + slot;
    const bool active = slot < g.count;
    int best = 0, bi = INT_MAX, bj = INT_MAX;
    int S = 0, qe = 0, re = 0;
    if (active) {
        const CoordItem it = prm.items[item];
        int q = prm.qlen, len = it.subjectLength;
        int q0 = 0;
        unsigned long long* trace = nullptr;
        if (REV) {
            const int4 e = prm.ends[item];
            S = e.x; qe = e.y; re = e.z;
            q = S > 0 ? qe + 1 : 0;
            len = S > 0 ? re + 1 : 0;
        }
        if (TRACE) {
            const TraceItem ti = prm.traceItems[item];
            S = ti.score; q0 = ti.queryBegin; q = ti.rows;
            trace = prm.trace + ti.words;
        }
        const uint8_t* s = prm.subjects + it.subjectOffset;
        const int borderStride = TRACE ? (q + 31) & ~31 : prm.borderStride;  // pass 3: rows of the pair's rectangle
        int2* outBorder = prm.border + it.borderOffset + (size_t)wi * borderStride;
        const int2* inBorder = prm.border + it.borderOffset + (size_t)((wi + W - 1) % W) * borderStride;
        volatile long long* leftProgress = progress + (warp - wi) + (wi + W - 1) % W;
        volatile long long* myProgress = progress + warp;
        const int gop = prm.gop, gex = prm.gex;
        const int tiles = q > 0 ? (len + kCoordTileCols - 1) / kCoordTileCols : 0;
        for (int tile = wi; tile < tiles; tile += W) {
            const int col0 = tile * kCoordTileCols + lane * R;
            int srow[R];
#pragma unroll
            for (int j = 0; j < R; j++) {
                const int c = col0 + j;
                const int code = c < len ? (int)s[REV ? re - c : c] : 20;
                srow[j] = min(code, 20);
            }
            int Hp[R], F[R];
#pragma unroll
            for (int j = 0; j < R; j++) { Hp[j] = 0; F[j] = kNegS32; }
            int Hlast = 0, Elast = kNegS32;
            int HinPrev = ((REV || TRACE) && tile == 0 && lane == 0) ? kCoordAnchor : 0;  // H(-1, -1)
            int2 inBuf = make_int2(0, kNegS32), outBuf = make_int2(0, 0);
            const bool firstTile = tile == 0, lastTile = tile == tiles - 1;
            const int steps = q + 31;
            for (int t = 0; t < steps; t++) {
                if (!firstTile && (t & 31) == 0) {  // next 32 rows of the left border, once the left warp stored them
                    if (W > 1) {
                        const long long need = ((long long)(tile - 1) << 32) | (long long)min(q, t + 32);
                        if (lane == 0)
                            while (*leftProgress < need) __nanosleep(32);
                        __syncwarp();
                        __threadfence_block();
                    }
                    const int r = t + lane;
                    inBuf = (r < q) ? __ldcg(inBorder + r) : make_int2(0, kNegS32);
                }
                int Hin = __shfl_up_sync(0xffffffffu, Hlast, 1);
                int Ein = __shfl_up_sync(0xffffffffu, Elast, 1);
                const int bH = __shfl_sync(0xffffffffu, inBuf.x, t & 31);
                const int bE = __shfl_sync(0xffffffffu, inBuf.y, t & 31);
                if (lane == 0) { Hin = firstTile ? 0 : bH; Ein = firstTile ? kNegS32 : bE; }
                const int row = t - lane;
                if (row >= 0 && row < q) {
                    const int qrow = REV ? qe - row : (TRACE ? q0 + row : row);
                    const int* Mrow = PSSM ? nullptr : Msm + 21 * prm.query[qrow];
                    const int8_t* Prow = PSSM ? pssm + 21 * (size_t)qrow : nullptr;
                    int E = Ein, diag = HinPrev;
                    int rowBest = 0, rowJ = 0;  // first maximum of this row segment
                    unsigned dirs[2] = {0u, 0u};  // pass 3: nibbles of columns 0-7 and 8-15
#pragma unroll
                    for (int j = 0; j < R; j++) {
                        const int d = diag + (PSSM ? (int)__ldg(Prow + srow[j]) : Mrow[srow[j]]);
                        diag = Hp[j];
                        const int h = __vimax3_s32_relu(d, E, F[j]);
                        Hp[j] = h;
                        const int tt = h + gop;
                        if (TRACE) {
                            const unsigned nib = (d == h ? 0u : (E == h ? 1u : 2u)) | (E + gex >= tt ? 4u : 0u) |
                                                 (F[j] + gex >= tt ? 8u : 0u);
                            dirs[j / 8] |= nib << (4 * (j % 8));
                        }
                        E = __viaddmax_s32(E, gex, tt);
                        F[j] = __viaddmax_s32(F[j], gex, tt);
                        if (!TRACE && h > rowBest) { rowBest = h; rowJ = j; }
                    }
                    if (TRACE) {
                        trace[((size_t)tile * (q + 31) + t) * 32 + lane] = ((unsigned long long)dirs[1] << 32) | dirs[0];
                    } else {
                        // a lane sees its rows in order and its tiles left to right: on a tie only a smaller row wins
                        if (rowBest > best || (rowBest == best && row < bi)) { best = rowBest; bi = row; bj = col0 + rowJ; }
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
                            if (lane <= (r31 & 31)) outBorder[r] = outBuf;
                            if (W > 1) {
                                __syncwarp();
                                if (lane == 0) {
                                    __threadfence_block();
                                    *myProgress = ((long long)tile << 32) | (long long)(r31 + 1);
                                }
                            }
                        }
                    }
                }
            }
            if (TRACE && lastTile) {  // every lane's Hp holds row q - 1: the value at (qe, re) must be the anchored score
#pragma unroll
                for (int j = 0; j < R; j++)
                    if (col0 + j == len - 1 && Hp[j] != kCoordAnchor + S) atomicAdd(prm.errors, 1);
            }
            __syncwarp();
        }
    }
    if constexpr (!TRACE) {  // passes 1 and 2: combine the trackers of the lanes and warps of the pair
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const int v = __shfl_xor_sync(0xffffffffu, best, o);
            const int i = __shfl_xor_sync(0xffffffffu, bi, o);
            const int j = __shfl_xor_sync(0xffffffffu, bj, o);
            if (coord_better(v, i, j, best, bi, bj)) { best = v; bi = i; bj = j; }
        }
        if (lane == 0) { redV[warp] = best; redI[warp] = bi; redJ[warp] = bj; }
        __syncthreads();
        if (!active || wi != 0 || lane != 0) return;
        for (int w = warp + 1; w < warp + W; w++)
            if (coord_better(redV[w], redI[w], redJ[w], best, bi, bj)) { best = redV[w]; bi = redI[w]; bj = redJ[w]; }
        if (!REV) {
            prm.ends[item] = best > 0 ? make_int4(best, bi, bj, 0) : make_int4(0, -1, -1, 0);
            return;
        }
        int32_t* o = prm.out + (size_t)item * 5;
        if (S <= 0) {
            o[0] = 0; o[1] = -1; o[2] = -1; o[3] = -1; o[4] = -1;
            return;
        }
        if (best != kCoordAnchor + S) atomicAdd(prm.errors, 1);
        o[0] = S; o[1] = qe - bi; o[2] = qe; o[3] = re - bj; o[4] = re;
    }
}

// passes 1 and 2 (REV)
template <bool REV>
__global__ void __launch_bounds__(kCoordThreads, 1) sw_coords_kernel(const CoordParams prm) {
    coords_pass<REV ? kCoordBegins : kCoordEnds>(prm);
}
// the same for a PSSM query (pssm: [qlen][21])
template <bool REV>
__global__ void __launch_bounds__(kCoordThreads, 1) sw_coords_pssm_kernel(const CoordParams prm, const int8_t* pssm) {
    coords_pass<REV ? kCoordBegins : kCoordEnds, true>(prm, pssm);
}

// pass 3: the same wavefront over each pair's rectangle, storing the 4-bit directions instead of tracking a maximum
// (this kernel and the walk are templates only so that the header can be included by several translation units)
template <int kInstance = 0>
__global__ void __launch_bounds__(kCoordThreads, 1) sw_coords_trace_kernel(const CoordParams prm) {
    coords_pass<kCoordTrace>(prm);
}
template <int kInstance = 0>
__global__ void __launch_bounds__(kCoordThreads, 1) sw_coords_trace_pssm_kernel(const CoordParams prm, const int8_t* pssm) {
    coords_pass<kCoordTrace, true>(prm, pssm);
}

constexpr int kWalkThreads = 128;

// The walk: one thread per traced pair, from (qe, re) in state P back to (qb, rb), by the rule of include/sw4b200.h.
// PSSM: a pair at query position i is a positive when pssm[21 * i + code] > 0.
template <bool PSSM>
__device__ __forceinline__ void coords_walk(const CoordParams& prm, const int8_t* __restrict__ pssm) {
    __shared__ int Msm[PSSM ? 1 : 21 * 21];
    if (!PSSM)
        for (int i = threadIdx.x; i < 441; i += blockDim.x) Msm[i] = prm.matrix[i];
    __syncthreads();
    const int item = blockIdx.x * blockDim.x + threadIdx.x;
    if (item >= prm.numItems) return;
    const CoordItem it = prm.items[item];
    const TraceItem ti = prm.traceItems[item];
    const uint8_t* s = prm.subjects + it.subjectOffset;
    const uint8_t* qy = prm.query + ti.queryBegin;
    const unsigned long long* tr = prm.trace + ti.words;
    char* ops = prm.ops + ti.ops;
    const int n = ti.rows, m = it.subjectLength;
    const size_t tileWords = (size_t)(n + 31) * 32;
    auto nibble = [&](int i, int c) -> unsigned {
        const int lane = (c / kCoordR) % 32;
        const unsigned long long w = tr[(size_t)(c / kCoordTileCols) * tileWords + (size_t)(i + lane) * 32 + lane];
        return (unsigned)(w >> (4 * (c % kCoordR))) & 15u;
    };
    int i = n - 1, c = m - 1, state = 0, len = 0, idents = 0, pos = 0, gaps = 0;
    bool ok = false;
    while (len < n + m) {
        if (state == 0) {  // P: a pair; then the first state equal to X(i - 1, c - 1)
            const int a = min((int)qy[i], 20), b = min((int)s[c], 20);
            ops[len++] = a == b ? '=' : 'X';
            idents += a == b;
            pos += (PSSM ? (int)pssm[21 * ((size_t)ti.queryBegin + i) + b] : Msm[21 * a + b]) > 0;
            if (i == 0 && c == 0) { ok = true; break; }
            if (--i < 0 || --c < 0) break;
            state = (int)(nibble(i, c) & 3u);
        } else if (state == 1) {  // E: consumes a reference residue; extend, else open from X(i, c - 1)
            ops[len++] = 'D';
            gaps++;
            if (--c < 0) break;
            const unsigned w = nibble(i, c);
            state = (w & 4u) ? 1 : (int)(w & 3u);
        } else {  // F: consumes a query residue; extend, else open from X(i - 1, c)
            ops[len++] = 'I';
            gaps++;
            if (--i < 0) break;
            const unsigned w = nibble(i, c);
            state = (w & 8u) ? 2 : (int)(w & 3u);
        }
    }
    prm.counts[item] = make_int4(len, idents, pos, gaps);
    if (!ok) atomicAdd(prm.errors + 1, 1);
}

template <int kInstance = 0>
__global__ void __launch_bounds__(kWalkThreads) sw_coords_walk_kernel(const CoordParams prm) {
    coords_walk<false>(prm, nullptr);
}
template <int kInstance = 0>
__global__ void __launch_bounds__(kWalkThreads) sw_coords_walk_pssm_kernel(const CoordParams prm, const int8_t* pssm) {
    coords_walk<true>(prm, pssm);
}

}  // namespace sw4
