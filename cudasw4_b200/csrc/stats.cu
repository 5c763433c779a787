// The E-value fit (sw4_fit_score_statistics, defined in include/sw4b200.h): maximum likelihood for lambda and K on a
// censored score histogram. Pure host code; tests/evalue_oracle.py restates it.
#include <cmath>
#include <cstring>

#include "../../include/sw4b200.h"

namespace {

constexpr int64_t kMinFitted = 100;  // fewer fitted subjects than this: SW4_STATS_TOO_FEW

// The derivative of the profile log-likelihood in lambda. A and B are taken times e^(lambda c_lo), which keeps every
// exponent <= 0 and leaves B / A unchanged; *aShifted receives that A (K needs it).
struct ProfileSlope {
    const int64_t *counts, *lensums;
    int cLo, cHi;
    double leftLen, sumX, fitted, right;
    double operator()(double lambda, double* aShifted = nullptr) const {
        double a = leftLen, b = (double)cLo * leftLen;
        for (int s = cLo; s < cHi; s++) {
            if (!lensums[s]) continue;
            const double x = s + 0.5;
            const double w = (double)lensums[s] * std::exp(-lambda * (x - cLo));
            a += w;
            b += w * x;
        }
        if (aShifted) *aShifted = a;
        return fitted / lambda - sumX - right * cHi + (fitted + right) * b / a;
    }
};

}  // namespace

extern "C" int sw4_fit_score_statistics(const int64_t* counts, const int64_t* lensums, int32_t bins, int64_t query_length,
                                        sw4_score_statistics* out) {
    if (!counts || !lensums || !out || bins < 1) return SW4_ERR_INVALID;
    for (int s = 0; s <= bins; s++)
        if (counts[s] < 0 || lensums[s] < 0) return SW4_ERR_INVALID;
    memset(out, 0, sizeof(*out));
    out->status = SW4_STATS_TOO_FEW;
    out->whole_database = 1;
    out->lambda = out->K = std::nan("");
    out->query_length = query_length;
    int64_t n = 0, d = 0;
    for (int s = 0; s <= bins; s++) { n += counts[s]; d += lensums[s]; }
    out->num_subjects = n;
    out->db_residues = d;
    // c_lo: the median; c_hi: the first score above it that at most floor(N / 1000) subjects reach
    int cLo = bins;
    int64_t below = 0;  // subjects below the score under consideration
    for (int s = 0; s < bins; s++) {
        below += counts[s];
        if (2 * below >= n) { cLo = s; break; }
    }
    int cHi = bins;
    for (int s = cLo + 1; s < bins; s++) {
        if (n - below <= n / 1000) { cHi = s; break; }
        below += counts[s];
    }
    int64_t left = 0, fitted = 0;
    double leftLen = 0, sumX = 0;
    for (int s = 0; s < cLo && s < bins; s++) { left += counts[s]; leftLen += (double)lensums[s]; }
    for (int s = cLo; s < cHi; s++) { fitted += counts[s]; sumX += (double)counts[s] * (s + 0.5); }
    out->c_lo = cLo;
    out->c_hi = cHi;
    out->left_censored = left;
    out->fitted = fitted;
    out->right_censored = n - left - fitted;
    if (fitted < kMinFitted || cLo >= bins || query_length < 1) return SW4_OK;

    const ProfileSlope slope{counts, lensums, cLo, cHi, leftLen, sumX, (double)fitted, (double)out->right_censored};
    double lo = 1e-4, hi = 10.0, lambda;
    if (slope(lo) <= 0) {
        lambda = lo;
    } else if (slope(hi) >= 0) {
        lambda = hi;
    } else {
        for (;;) {  // the slope decreases: keep it > 0 at lo and <= 0 at hi until no double lies between them
            const double mid = lo + (hi - lo) / 2;
            if (mid <= lo || mid >= hi) break;
            if (slope(mid) > 0) lo = mid; else hi = mid;
        }
        lambda = lo + (hi - lo) / 2;
    }
    double aShifted = 0;
    slope(lambda, &aShifted);
    out->lambda = lambda;
    out->K = std::exp(std::log((double)(fitted + out->right_censored)) + lambda * cLo - std::log((double)query_length) -
                      std::log(aShifted));
    out->status = SW4_STATS_OK;
    return SW4_OK;
}
