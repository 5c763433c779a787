"""The E-value fit of include/sw4b200.h (sw4_fit_score_statistics, cudasw4_b200/csrc/stats.cu) restated in numpy, and a
sampler of the model it fits. The tests hold the library's fit against this restatement."""
from __future__ import annotations

import math

import numpy as np


def fit(counts, lensums, query_length: int) -> dict:
    """Fit of a histogram with len(counts) - 1 score bins and an overflow bin. Returns the fields of
    sw4_score_statistics (ok instead of status, lambda_ for lambda)."""
    c = np.asarray(counts, dtype=np.int64)
    L = np.asarray(lensums, dtype=np.int64)
    bins = len(c) - 1
    n, d = int(c.sum()), int(L.sum())
    cum = np.cumsum(c[:bins])
    hit = np.nonzero(2 * cum >= n)[0]
    c_lo = int(hit[0]) if len(hit) else bins
    c_hi = bins
    if c_lo < bins:
        tail = n - np.concatenate([[0], cum])[:bins]  # tail[s] = #(score >= s)
        s = np.arange(bins)
        hit = np.nonzero((s > c_lo) & (tail <= n // 1000))[0]
        c_hi = int(hit[0]) if len(hit) else bins
    left = int(c[:c_lo].sum())
    fitted = int(c[c_lo:c_hi].sum())
    right = n - left - fitted
    out = dict(ok=False, lambda_=math.nan, K=math.nan, query_length=int(query_length), db_residues=d, num_subjects=n,
               fitted=fitted, left_censored=left, right_censored=right, c_lo=c_lo, c_hi=c_hi)
    if fitted < 100 or c_lo >= bins or query_length < 1:
        return out
    x = np.arange(c_lo, c_hi) + 0.5
    lens = L[c_lo:c_hi].astype(np.float64)
    left_len = float(L[:c_lo].sum())
    sum_x = float((c[c_lo:c_hi] * x).sum())

    def slope(lam):
        w = lens * np.exp(-lam * (x - c_lo))
        a = left_len + w.sum()
        b = c_lo * left_len + (w * x).sum()
        return fitted / lam - sum_x - right * c_hi + (fitted + right) * b / a, a

    lo, hi = 1e-4, 10.0
    if slope(lo)[0] <= 0:
        lam = lo
    elif slope(hi)[0] >= 0:
        lam = hi
    else:
        while True:
            mid = lo + (hi - lo) / 2
            if mid <= lo or mid >= hi:
                break
            if slope(mid)[0] > 0:
                lo = mid
            else:
                hi = mid
        lam = lo + (hi - lo) / 2
    a = slope(lam)[1]
    out.update(ok=True, lambda_=lam,
               K=math.exp(math.log(fitted + right) + lam * c_lo - math.log(query_length) - math.log(a)))
    return out


def histogram(scores, lengths, bins: int = 4096):
    """(counts, lensums) of subjects with length >= 1, scores >= bins in the overflow bin: what the device builds."""
    s = np.asarray(scores, dtype=np.int64)
    L = np.asarray(lengths, dtype=np.int64)
    keep = L >= 1
    b = np.minimum(s[keep], bins)
    return (np.bincount(b, minlength=bins + 1).astype(np.int64),
            np.bincount(b, weights=L[keep], minlength=bins + 1).astype(np.int64))


def sample_scores(rng, lengths, lam: float, K: float, m: int):
    """Integer scores drawn from the model: x with P(x >= t) = 1 - exp(-K m n e^(-lambda t)), floored."""
    u = rng.random(len(lengths))
    x = np.log(K * m * np.asarray(lengths, dtype=np.float64) / -np.log1p(-u)) / lam
    return np.maximum(np.floor(x), 0).astype(np.int64)
