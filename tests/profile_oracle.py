"""numpy restatement of the profile construction of sw4_build_pssm (include/sw4b200.h, steps 2-6).

It takes what alignments() reports (coordinates and CIGARs) plus the reference codes, so it checks everything after
the traceback: the query-anchored MSA, the Henikoff weights, the frequencies, the pseudocounts and the rounding."""
import re

import numpy as np

from cudasw4_b200 import synth

LETTERS = "ARNDCQEGHILKMFPSTWYV"
GAP = 21
EMPTY = -1


def query_codes(query: str) -> np.ndarray:
    """Letters -> codes as the device converts a query: the 20 upper-case letters, everything else 20."""
    return np.array([LETTERS.index(c) if c in LETTERS else 20 for c in query], dtype=np.int64)


def background() -> np.ndarray:
    """p_a: the generated databases' residue frequencies (synth._PSEUDO_TABLE, 1/256 steps)."""
    return np.bincount(synth._PSEUDO_TABLE, minlength=20) / 256.0


def ungapped_lambda(M: np.ndarray) -> float:
    """The root of sum_{a,b<20} p_a p_b e^(lambda M[a][b]) = 1, by the bisection of test_evalue.py."""
    p = background()
    M = np.asarray(M)[:20, :20].astype(np.float64)
    lo, hi = 1e-3, 2.0
    for _ in range(200):  # sum p_a p_b e^(lambda s_ab) = 1: below the root the sum is < 1
        mid = (lo + hi) / 2
        lo, hi = (mid, hi) if (np.outer(p, p) * np.exp(mid * M)).sum() < 1 else (lo, mid)
    return lo


def target_frequencies(M: np.ndarray):
    """(lambda_u, q) with q_ab = p_a p_b e^(lambda_u M[a][b]) / Z."""
    p = background()
    lam = ungapped_lambda(M)
    t = np.outer(p, p) * np.exp(lam * np.asarray(M)[:20, :20].astype(np.float64))
    return lam, t / t.sum()


def build_msa(qcodes, alignments) -> np.ndarray:
    """Row 0 the query, then one row per alignment with a positive score, in order. alignments: (coordinates
    (score, qb, qe, rb, re), CIGAR, reference codes). Symbols: codes 0..20, GAP, EMPTY."""
    m = len(qcodes)
    rows = [np.asarray(qcodes, dtype=np.int64)]
    for coords, cigar, ref in alignments:
        score, qb, qe, rb, re_ = (int(v) for v in coords)
        if score <= 0:
            continue
        row = np.full(m, EMPTY, dtype=np.int64)
        i, j = qb, rb
        for run, op in re.findall(r"(\d+)([=XID])", cigar):
            for _ in range(int(run)):
                if op in "=X":
                    row[i] = min(int(ref[j]), 20)
                    i += 1
                    j += 1
                elif op == "I":
                    row[i] = GAP
                    i += 1
                else:
                    j += 1
        assert i == qe + 1 and j == re_ + 1, (coords, cigar)
        rows.append(row)
    return np.array(rows, dtype=np.int64).reshape(len(rows), m)


def henikoff_weights(msa: np.ndarray) -> np.ndarray:
    """w_k = sum over the non-empty columns c of row k of 1 / (r_c n_{c, x_kc})."""
    msa = np.asarray(msa)
    w = np.zeros(msa.shape[0])
    for c in range(msa.shape[1]):
        col = msa[:, c]
        present = col != EMPTY
        syms, counts = np.unique(col[present], return_counts=True)
        n = dict(zip(syms.tolist(), counts.tolist()))
        r = len(syms)
        for k in np.nonzero(present)[0]:
            w[k] += 1.0 / (r * n[int(col[k])])
    return w


def profile(qcodes, alignments, M: np.ndarray, beta: float):
    """(pssm (m, 21) int8, x (m, 20) float64): x = ln(Q_ca / p_a) / lambda_u before the rounding."""
    M = np.asarray(M).astype(np.int64)
    low = int(M[20, 20])
    msa = build_msa(qcodes, alignments)
    m = msa.shape[1]
    w = henikoff_weights(msa)
    p = background()
    lam, q = target_frequencies(M)
    rprime = np.array([len(np.unique(msa[:, c][(msa[:, c] >= 0) & (msa[:, c] < 20)])) for c in range(m)], dtype=np.int64)
    alpha = float(rprime[rprime >= 1].mean()) - 1.0 if (rprime >= 1).any() else 0.0
    out = np.empty((m, 21), dtype=np.int64)
    x = np.full((m, 20), np.nan)
    for c in range(m):
        col = msa[:, c]
        std = (col >= 0) & (col < 20)
        W = w[std].sum()
        if W == 0:
            out[c] = M[20]
            continue
        f = np.array([w[std & (col == a)].sum() for a in range(20)]) / W
        g = q @ (f / p)  # g_a = sum_b f_b q_ab / p_b
        Q = (alpha * f + beta * g) / (alpha + beta)
        x[c] = np.log(Q / p) / lam
        out[c, :20] = np.clip(np.floor(x[c] + 0.5), -128, 127)
    out[:, 20] = low
    return out.astype(np.int8), x
