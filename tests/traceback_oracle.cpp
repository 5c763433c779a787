// TEST INFRASTRUCTURE ONLY. CPU restatement of the alignment that sw4_alignment_traceback reports (the rule in
// include/sw4b200.h), written from the rule in int64 with a true minus infinity. The coordinates are an input: they come
// from tests/coords_oracle.cpp, which restates their definition. Over the rectangle the anchored recurrences fill full
// rows of P, E and F, and one byte per cell keeps the decisions the walk needs; then the walk runs from (qe, re) back to
// (qb, rb). tests/traceback_oracle.py compiles and binds it; tests/test_traceback.py checks it against a plain Python
// statement of the rule on tiny inputs and by rescoring every CIGAR.
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

// the first of P (0), E (1), F (2) equal to X = max(P, E, F)
inline unsigned char first_max(i64 p, i64 e, i64 f) {
    const i64 x = std::max(p, std::max(e, f));
    return p == x ? 0 : (e == x ? 1 : 2);
}

// c = (S, qb, qe, rb, re). ops receives the columns in query order ('=', 'X', 'I', 'D'), counts = (length, identities,
// positives, gaps). Returns false if the value at (qe, re) is not S or the walk does not end at (qb, rb) in state P.
bool traceback(const signed char* M, const unsigned char* q, const unsigned char* s, const std::int32_t* c, int gop, int gex,
               char* ops, std::int32_t* counts) {
    counts[0] = counts[1] = counts[2] = counts[3] = 0;
    if (c[0] <= 0) return true;
    const int qb = c[1], rb = c[3], n = c[2] - c[1] + 1, m = c[4] - c[3] + 1;
    // dir(i, j): bits 0-1 the first state equal to X(i, j); bit 2 E(i, j) extends E(i, j-1) (E(i,j-1) + gex == E(i,j));
    // bit 3 F(i, j) extends F(i-1, j)
    std::vector<unsigned char> dir((size_t)n * m);
    std::vector<i64> Pp(m, NEG), Ep(m, NEG), Fp(m, NEG), Pc(m), Ec(m), Fc(m);  // previous and current row
    for (int i = 0; i < n; i++) {
        for (int j = 0; j < m; j++) {
            const i64 sub = M[21 * q[qb + i] + s[rb + j]];
            i64 p = NEG;
            if (i == 0 && j == 0) p = sub;
            else if (i > 0 && j > 0) {
                const i64 x = std::max(Pp[j - 1], std::max(Ep[j - 1], Fp[j - 1]));
                if (x > NEG) p = x + sub;
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
    // the walk, from (qe, re) in state P
    int i = n - 1, j = m - 1, state = 0, len = 0;
    std::vector<char> rev;
    rev.reserve((size_t)n + m);
    for (;;) {
        if ((int)rev.size() > n + m) return false;
        if (state == 0) {
            const int a = std::min<int>(q[qb + i], 20), b = std::min<int>(s[rb + j], 20);
            rev.push_back(a == b ? '=' : 'X');
            counts[1] += a == b;
            counts[2] += M[21 * a + b] > 0;
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
    len = (int)rev.size();
    counts[0] = len;
    for (int k = 0; k < len; k++) ops[k] = rev[len - 1 - k];
    return true;
}

}  // namespace

extern "C" {

// q against n subjects stored makedb-style (codes + byte offsets + true lengths), OpenMP over subjects. coords is
// [n][5] (score, qb, qe, rb, re) as tests/coords_oracle.cpp computes them. ops: pair k writes its columns at
// ops + ops_offsets[k] (room for (qe - qb + 1) + (re - rb + 1) bytes); counts is [n][4]. Returns the number of pairs whose
// check failed (0).
long sw4t_traceback_batch(const signed char* matrix441, const unsigned char* q, const unsigned char* chars,
                          const std::size_t* offsets, long n, const std::int32_t* coords, int gop, int gex, char* ops,
                          const std::size_t* ops_offsets, std::int32_t* counts, int threads) {
    long failed = 0;
#ifdef _OPENMP
    if (threads <= 0) threads = omp_get_max_threads();
#pragma omp parallel for schedule(dynamic, 1) num_threads(threads) reduction(+ : failed)
#endif
    for (long k = 0; k < n; k++)
        if (!traceback(matrix441, q, chars + offsets[k], coords + 5 * k, gop, gex, ops + ops_offsets[k], counts + 4 * k)) failed++;
    return failed;
}

}  // extern "C"
