// TEST INFRASTRUCTURE ONLY. CPU restatement of the score, the coordinates and the traceback of a query scored with a
// position-specific scoring matrix (PSSM; include/sw4b200.h), in int64 with a true minus infinity. It is the rule of
// tests/coords_oracle.cpp and tests/traceback_oracle.cpp with the substitution score M[q_i][r] replaced by
// pssm[21 * i + r]; positives are the pairs with pssm[21 * i + r] > 0, identities compare residue codes.
// tests/pssm_oracle.py compiles and binds it; tests/test_pssm.py checks it against those oracles with pssm[i] = M[q_i]
// and against a brute force on tiny inputs.
#include <algorithm>
#include <cstddef>
#include <cstdint>
#include <vector>
#ifdef _OPENMP
#include <omp.h>
#endif

namespace {

typedef long long i64;
const i64 NEG = -(1ll << 60);

// out = (S, qb, qe, rb, re), -1 positions when S == 0; false if the begin pass does not reach S
bool pssm_coords(const signed char* P, int qlen, const unsigned char* s, int slen, int gop, int gex, std::int32_t* out) {
    // end: H(i, j) = max(0, H(i-1, j-1) + P[i][s_j], E, F); the first (i, j) in row-major order holding max H
    std::vector<i64> H(slen + 1, 0), F(slen + 1, NEG);
    i64 S = 0;
    int qe = -1, re = -1;
    for (int i = 0; i < qlen; i++) {
        i64 diag = 0, left = 0, E = NEG;
        for (int j = 1; j <= slen; j++) {
            const i64 up = H[j];
            E = std::max(E + gex, left + gop);
            F[j] = std::max(F[j] + gex, up + gop);
            const i64 h = std::max<i64>(0, std::max(diag + P[21 * (i64)i + s[j - 1]], std::max(E, F[j])));
            diag = up;
            H[j] = h;
            left = h;
            if (h > S) { S = h; qe = i; re = j - 1; }
        }
    }
    out[0] = (std::int32_t)S;
    out[1] = out[2] = out[3] = out[4] = -1;
    if (S == 0) return true;
    // begin: over the reversed prefixes, the best alignment starting with the pair (qe, re) and ending with the pair
    // (qe - a, re - b), no floor; the first (a, b) in row-major order reaching S is the largest (qb, rb)
    const int n = qe + 1, m = re + 1;
    std::vector<i64> X(m + 1, NEG), G(m + 1, NEG);
    i64 best = NEG;
    int ba = -1, bb = -1;
    for (int a = 0; a < n; a++) {
        i64 diag = a == 0 ? 0 : NEG, left = NEG, E = NEG;
        for (int b = 1; b <= m; b++) {
            const i64 up = X[b];
            E = std::max(E + gex, left + gop);
            G[b] = std::max(G[b] + gex, up + gop);
            const i64 p = diag + P[21 * (i64)(qe - a) + s[re - (b - 1)]];
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

inline unsigned char first_max(i64 p, i64 e, i64 f) {
    const i64 x = std::max(p, std::max(e, f));
    return p == x ? 0 : (e == x ? 1 : 2);
}

// The walk of include/sw4b200.h over the rectangle c = (S, qb, qe, rb, re); ops in query order, counts = (length,
// identities, positives, gaps). False if the anchored value at (qe, re) is not S or the walk does not end at (qb, rb).
bool pssm_traceback(const signed char* P, const unsigned char* q, const unsigned char* s, const std::int32_t* c, int gop, int gex,
                    char* ops, std::int32_t* counts) {
    counts[0] = counts[1] = counts[2] = counts[3] = 0;
    if (c[0] <= 0) return true;
    const int qb = c[1], rb = c[3], n = c[2] - c[1] + 1, m = c[4] - c[3] + 1;
    auto score = [&](int i, int j) -> i64 { return P[21 * (i64)(qb + i) + s[rb + j]]; };
    std::vector<unsigned char> dir((size_t)n * m);
    std::vector<i64> Pp(m, NEG), Ep(m, NEG), Fp(m, NEG), Pc(m), Ec(m), Fc(m);
    for (int i = 0; i < n; i++) {
        for (int j = 0; j < m; j++) {
            i64 p = NEG;
            if (i == 0 && j == 0) p = score(0, 0);
            else if (i > 0 && j > 0) {
                const i64 x = std::max(Pp[j - 1], std::max(Ep[j - 1], Fp[j - 1]));
                if (x > NEG) p = x + score(i, j);
            }
            i64 e = NEG, f = NEG;
            bool eExt = false, fExt = false;
            if (j > 0) {
                const i64 x = std::max(Pc[j - 1], std::max(Ec[j - 1], Fc[j - 1]));
                const i64 open = x > NEG ? x + gop : NEG, ext = Ec[j - 1] > NEG ? Ec[j - 1] + gex : NEG;
                e = std::max(open, ext);
                eExt = e > NEG && ext == e;
            }
            if (i > 0) {
                const i64 x = std::max(Pp[j], std::max(Ep[j], Fp[j]));
                const i64 open = x > NEG ? x + gop : NEG, ext = Fp[j] > NEG ? Fp[j] + gex : NEG;
                f = std::max(open, ext);
                fExt = f > NEG && ext == f;
            }
            Pc[j] = p; Ec[j] = e; Fc[j] = f;
            dir[(size_t)i * m + j] = (unsigned char)(first_max(p, e, f) | (eExt ? 4 : 0) | (fExt ? 8 : 0));
        }
        if (i == n - 1 && Pc[m - 1] != c[0]) return false;
        std::swap(Pp, Pc); std::swap(Ep, Ec); std::swap(Fp, Fc);
    }
    int i = n - 1, j = m - 1, state = 0;
    std::vector<char> rev;
    for (;;) {
        if ((int)rev.size() > n + m) return false;
        if (state == 0) {
            const int a = std::min<int>(q[qb + i], 20), b = std::min<int>(s[rb + j], 20);
            rev.push_back(a == b ? '=' : 'X');
            counts[1] += a == b;
            counts[2] += score(i, j) > 0;
            if (i == 0 && j == 0) break;
            if (--i < 0 || --j < 0) return false;
            state = dir[(size_t)i * m + j] & 3;
        } else if (state == 1) {
            rev.push_back('D');
            counts[3]++;
            const bool ext = dir[(size_t)i * m + j] & 4;
            if (--j < 0) return false;
            state = ext ? 1 : (dir[(size_t)i * m + j] & 3);
        } else {
            rev.push_back('I');
            counts[3]++;
            const bool ext = dir[(size_t)i * m + j] & 8;
            if (--i < 0) return false;
            state = ext ? 2 : (dir[(size_t)i * m + j] & 3);
        }
    }
    const int len = (int)rev.size();
    counts[0] = len;
    for (int k = 0; k < len; k++) ops[k] = rev[len - 1 - k];
    return true;
}

}  // namespace

extern "C" {

// The PSSM query (pssm [qlen][21], residue codes q for the identities) against n subjects stored makedb-style (codes,
// byte offsets, true lengths), OpenMP over subjects. out is [n][5] = (score, qb, qe, rb, re). Returns the number of
// pairs whose check failed (0).
long sw4p_coords_batch(const signed char* pssm, int qlen, const unsigned char* chars, const std::size_t* offsets,
                       const std::int32_t* lengths, long n, int gop, int gex, std::int32_t* out, int threads) {
    long failed = 0;
#ifdef _OPENMP
    if (threads <= 0) threads = omp_get_max_threads();
#pragma omp parallel for schedule(dynamic, 1) num_threads(threads) reduction(+ : failed)
#endif
    for (long k = 0; k < n; k++)
        if (!pssm_coords(pssm, qlen, chars + offsets[k], lengths[k], gop, gex, out + 5 * k)) failed++;
    return failed;
}

// coords as sw4p_coords_batch gives them; pair k writes its ops at ops + ops_offsets[k]; counts is [n][4]
long sw4p_traceback_batch(const signed char* pssm, const unsigned char* q, const unsigned char* chars, const std::size_t* offsets,
                          long n, const std::int32_t* coords, int gop, int gex, char* ops, const std::size_t* ops_offsets,
                          std::int32_t* counts, int threads) {
    long failed = 0;
#ifdef _OPENMP
    if (threads <= 0) threads = omp_get_max_threads();
#pragma omp parallel for schedule(dynamic, 1) num_threads(threads) reduction(+ : failed)
#endif
    for (long k = 0; k < n; k++)
        if (!pssm_traceback(pssm, q, chars + offsets[k], coords + 5 * k, gop, gex, ops + ops_offsets[k], counts + 4 * k)) failed++;
    return failed;
}

}  // extern "C"
