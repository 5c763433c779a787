// Profile construction (sw4_build_pssm, include/sw4b200.h): a query-anchored multiple alignment of the traced hits,
// Henikoff position-based weights, pseudocount-mixed residue frequencies and log-odds scores, all on the GPU.
//
// The MSA is row-major, (1 + rows) x m bytes: row 0 is the query's codes, row k the k-th traced id with a positive score
// (ids in call order). A byte is a residue code 0..20, kMsaGap (the query position sits in a gap of that row: an I column)
// or kMsaEmpty (outside the row's [qb, qe]). Columns are query positions, so a thread per column reads a row's bytes
// coalesced.
//
// 1. profile_scatter_kernel runs in every traceback chunk right after the walk, while the chunk's subject slices and op
//    bytes are still in the arena: one thread per pair follows its ops from (qe, re) backwards and fills its MSA row.
// 2. profile_columns_kernel, one thread per column: n_{c,s} per symbol, r_c (distinct symbols) and r'_c (distinct codes
//    0..19); the sum of r'_c over the columns with r'_c >= 1 and their number go to two 64-bit integer counters.
// 3. profile_weights_kernel, one CTA per row: w_k = sum over the row's non-empty columns of 1 / (r_c n_{c,x_kc}), in
//    double, each thread over a fixed column stride and then a fixed tree.
// 4. profile_scores_kernel, one thread per column: W_c and f_ca over the rows with a code 0..19, then
//    g_ca = sum_b f_cb q_ab / p_b with the 20 x 20 table in shared memory, Q_ca = (alpha f_ca + beta g_ca) / (alpha + beta)
//    and out[c][a] = clamp(floor(ln(Q_ca / p_a) / lambda_u + 1/2), -128, 127); column 20 is the table's `low`.
// Every sum runs in an order fixed by the MSA alone (integer atomics for the counters), so the bytes do not depend on
// the chunking or on the schedule.
//
// The kernels are templates only so that the header can be included by several translation units.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "kernels_coords.cuh"

namespace sw4 {

constexpr uint8_t kMsaGap = 21;      // symbol of a query position in a gap (an I column)
constexpr uint8_t kMsaEmpty = 255;   // no symbol: outside the row's alignment
constexpr int kMsaSymbols = 22;      // codes 0..20 and the gap
constexpr int kProfileThreads = 128;

struct ProfileParams {
    const uint8_t* msa;       // [rows][m]
    int rows, m;
    int* counts;              // [kMsaSymbols][m]: n_{c,s}
    int2* distinct;           // [m]: (r_c, r'_c)
    unsigned long long* nsum; // [2]: sum of r'_c over the columns with r'_c >= 1, the number of those columns (zeroed)
    double* weights;          // [rows]
    const double* qOverP;     // [20][20]: q_ab / p_b
    const double* p;          // [20]: background frequencies
    double lambda, beta;
    int low;                  // the table's score of code 20
    int8_t* out;              // [m][21]
};

// 1. one thread per traced pair of the chunk: row msaRow[item] of the MSA from the walk's ops (written from the end)
template <int kInstance = 0>
__global__ void __launch_bounds__(kProfileThreads) profile_scatter_kernel(const CoordParams prm, const int* __restrict__ msaRow,
                                                                         uint8_t* __restrict__ msa, int m) {
    const int item = blockIdx.x * blockDim.x + threadIdx.x;
    if (item >= prm.numItems) return;
    const CoordItem it = prm.items[item];
    const TraceItem ti = prm.traceItems[item];
    const uint8_t* s = prm.subjects + it.subjectOffset;
    const char* ops = prm.ops + ti.ops;
    const int len = prm.counts[item].x;
    uint8_t* row = msa + (size_t)msaRow[item] * m + ti.queryBegin;
    int i = ti.rows - 1, c = it.subjectLength - 1;
    for (int e = 0; e < len; e++) {
        const char op = ops[e];
        if (op == 'D') { c--; continue; }
        if (op == 'I') row[i] = kMsaGap;
        else row[i] = (uint8_t)min((int)s[c--], 20);
        i--;
    }
}

// 2. one thread per column
template <int kInstance = 0>
__global__ void __launch_bounds__(kProfileThreads) profile_columns_kernel(const ProfileParams prm) {
    __shared__ int cnt[kMsaSymbols][kProfileThreads];
    const int c = blockIdx.x * kProfileThreads + threadIdx.x;
    int r = 0, r20 = 0;
    if (c < prm.m) {
        for (int s = 0; s < kMsaSymbols; s++) cnt[s][threadIdx.x] = 0;
        for (int k = 0; k < prm.rows; k++) {
            const int x = prm.msa[(size_t)k * prm.m + c];
            if (x != kMsaEmpty) cnt[x][threadIdx.x]++;
        }
        for (int s = 0; s < kMsaSymbols; s++) {
            const int v = cnt[s][threadIdx.x];
            prm.counts[(size_t)s * prm.m + c] = v;
            r += v > 0;
            if (s < 20) r20 += v > 0;
        }
        prm.distinct[c] = make_int2(r, r20);
    }
    unsigned long long sum = r20, cols = r20 > 0;
    for (int o = 16; o > 0; o >>= 1) {
        sum += __shfl_xor_sync(0xffffffffu, sum, o);
        cols += __shfl_xor_sync(0xffffffffu, cols, o);
    }
    if ((threadIdx.x & 31) == 0 && cols) {
        atomicAdd(prm.nsum, sum);
        atomicAdd(prm.nsum + 1, cols);
    }
}

// 3. one CTA per row
template <int kInstance = 0>
__global__ void __launch_bounds__(kProfileThreads) profile_weights_kernel(const ProfileParams prm) {
    __shared__ double part[kProfileThreads];
    const int k = blockIdx.x;
    const uint8_t* row = prm.msa + (size_t)k * prm.m;
    double w = 0;
    for (int c = threadIdx.x; c < prm.m; c += kProfileThreads) {
        const int x = row[c];
        if (x != kMsaEmpty) w += 1.0 / ((double)prm.distinct[c].x * (double)prm.counts[(size_t)x * prm.m + c]);
    }
    part[threadIdx.x] = w;
    __syncthreads();
    for (int o = kProfileThreads / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) part[threadIdx.x] += part[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) prm.weights[k] = part[0];
}

// 4. one thread per column
template <int kInstance = 0>
__global__ void __launch_bounds__(kProfileThreads) profile_scores_kernel(const ProfileParams prm) {
    __shared__ double qp[400], pa[20];
    __shared__ double f[20][kProfileThreads];
    for (int i = threadIdx.x; i < 400; i += kProfileThreads) qp[i] = prm.qOverP[i];
    if (threadIdx.x < 20) pa[threadIdx.x] = prm.p[threadIdx.x];
    __syncthreads();
    const int c = blockIdx.x * kProfileThreads + threadIdx.x;
    if (c >= prm.m) return;
    const int t = threadIdx.x;
    for (int a = 0; a < 20; a++) f[a][t] = 0;
    double W = 0;
    for (int k = 0; k < prm.rows; k++) {
        const int x = prm.msa[(size_t)k * prm.m + c];
        if (x < 20) {
            const double w = prm.weights[k];
            f[x][t] += w;
            W += w;
        }
    }
    int8_t* o = prm.out + (size_t)c * 21;
    o[20] = (int8_t)prm.low;
    if (W == 0) {  // no standard residue in the column: the row of code 20
        for (int a = 0; a < 20; a++) o[a] = (int8_t)prm.low;
        return;
    }
    for (int a = 0; a < 20; a++) f[a][t] /= W;
    const unsigned long long cols = prm.nsum[1];
    const double alpha = cols ? (double)prm.nsum[0] / (double)cols - 1.0 : 0.0;
    for (int a = 0; a < 20; a++) {
        double g = 0;
        for (int b = 0; b < 20; b++) g += f[b][t] * qp[a * 20 + b];
        const double Q = (alpha * f[a][t] + prm.beta * g) / (alpha + prm.beta);
        const double v = floor(log(Q / pa[a]) / prm.lambda + 0.5);
        o[a] = (int8_t)fmin(fmax(v, -128.0), 127.0);
    }
}

// launchers (launch_profile.cu)
cudaError_t launch_profile_scatter(const CoordParams& prm, const int* msaRow, uint8_t* msa, int m, cudaStream_t stream);
// steps 2-4 over the finished MSA; returns the number of kernels launched in *launches
cudaError_t launch_profile_build(const ProfileParams& prm, cudaStream_t stream, int* launches);

}  // namespace sw4
