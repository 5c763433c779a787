// TEST INFRASTRUCTURE ONLY. CPU restatement of the alignment coordinates that sw4_alignment_coordinates reports
// (definitions in include/sw4b200.h), written from the definition in int64 with a true minus infinity and two rolling
// rows. tests/coords_oracle.py compiles and binds it; tests/test_coordinates.py checks it against a brute force over
// every (begin, end) pair and its score against the oracle's sw4o_gotoh_score. The 21x21 substitution table is passed
// in (taken from the oracle's table), so this file has no data of its own.
#include <algorithm>
#include <cstddef>
#include <cstdint>
#include <vector>
#ifdef _OPENMP
#include <omp.h>
#endif

namespace {

// out = (S, qb, qe, rb, re); returns false if the begin pass does not reach S (cannot happen: a check of the restatement)
bool gotoh_coords(const signed char* M, const unsigned char* q, int qlen, const unsigned char* s, int slen, int gop, int gex,
                  std::int32_t* out) {
    typedef long long i64;
    const i64 NEG = -(1ll << 60);
    // end: H(i, j) = max(0, H(i-1, j-1) + M, E, F); the first (i, j) in row-major order holding max H
    std::vector<i64> H(slen + 1, 0), F(slen + 1, NEG);
    i64 S = 0;
    int qe = -1, re = -1;
    for (int i = 0; i < qlen; i++) {
        i64 diag = 0, left = 0, E = NEG;
        for (int j = 1; j <= slen; j++) {
            const i64 up = H[j];
            E = std::max(E + gex, left + gop);
            F[j] = std::max(F[j] + gex, up + gop);
            const i64 h = std::max<i64>(0, std::max(diag + M[21 * q[i] + s[j - 1]], std::max(E, F[j])));
            diag = up;
            H[j] = h;
            left = h;
            if (h > S) { S = h; qe = i; re = j - 1; }
        }
    }
    out[0] = (std::int32_t)S;
    out[1] = out[2] = out[3] = out[4] = -1;
    if (S == 0) return true;
    // begin: over the reversed prefixes, P(a, b) = best score of an alignment that starts with the pair (qe, re) and
    // ends with the pair (qe - a, re - b) (no floor: both ends are anchored). X = max(P, E, F); X(-1, -1) = 0 and every
    // other border is minus infinity. The first (a, b) in row-major order with P == S is the largest (qb, rb).
    const int n = qe + 1, m = re + 1;
    std::vector<i64> X(m + 1, NEG), G(m + 1, NEG);  // X, F of the previous row (index b + 1)
    i64 best = NEG;
    int ba = -1, bb = -1;
    for (int a = 0; a < n; a++) {
        i64 diag = a == 0 ? 0 : NEG, left = NEG, E = NEG;
        for (int b = 1; b <= m; b++) {
            const i64 up = X[b];
            E = std::max(E + gex, left + gop);
            G[b] = std::max(G[b] + gex, up + gop);
            const i64 p = diag + M[21 * q[qe - a] + s[re - (b - 1)]];
            const i64 x = std::max(p, std::max(E, G[b]));
            diag = up;
            X[b] = x;
            left = x;
            if (p > best) { best = p; ba = a; bb = b - 1; }
        }
    }
    out[1] = qe - ba; out[2] = qe; out[3] = re - bb; out[4] = re;
    return best == S;
}

}  // namespace

extern "C" {

// q against n subjects stored makedb-style (codes + byte offsets + true lengths), OpenMP over subjects. matrix441 is
// the 21x21 table, row = query code. out is [n][5] = (score, query_begin, query_end, reference_begin, reference_end),
// 0-based inclusive, -1 positions when score == 0. Returns the number of pairs whose begin pass failed (0).
long sw4c_gotoh_coords_batch(const signed char* matrix441, const unsigned char* q, int qlen, const unsigned char* chars,
                             const std::size_t* offsets, const std::int32_t* lengths, long n, int gop, int gex,
                             std::int32_t* out, int threads) {
    long failed = 0;
#ifdef _OPENMP
    if (threads <= 0) threads = omp_get_max_threads();
#pragma omp parallel for schedule(dynamic, 1) num_threads(threads) reduction(+ : failed)
#endif
    for (long i = 0; i < n; i++)
        if (!gotoh_coords(matrix441, q, qlen, chars + offsets[i], lengths[i], gop, gex, out + 5 * i)) failed++;
    return failed;
}

}  // extern "C"
