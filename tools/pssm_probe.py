"""PSSM-query timings (sw4_scan_pssm, sw4_alignment_coordinates_pssm, sw4_alignment_traceback_pssm) beside the
sequence forms of the same calls, in one process on one GPU.
  python tools/pssm_probe.py [OUT_JSON]

1. The peak benchmark (PseudoDB 1,000,000 x 256, BLOSUM62 -11/-1): every query scanned as letters and as the PSSM
   pssm[p] = M[q_p], alternating, median of 5 device-timed scans each. The scan kernels are the same; the PSSM form
   differs only in its prologue (PSSM upload and profile build instead of letters, conversion and profile build).
2. The coordinates and traceback cases of tools/coords_probe.py / tools/traceback_probe.py (DESIGN.md 3.6 / 3.7):
   top-10 and top-1000 on the peak benchmark, and one 35 k x 35 k pair, sequence form against PSSM form.
3. A PSSM that saturates 16 bits on short queries (entries of 127 along a consensus that 5 % of a 1 M x 256 database
   carries): the overflows re-score on sw_s32_kernel's PSSM form. Reported with numOverflows and the same scan with
   pssm = M[q_p] (no overflow) on the same database.
Every time is the call's device-timed stats (CUDA events) after one warm-up call."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import cudasw4_b200 as sw  # noqa: E402
from cudasw4_b200 import dbformat, synth  # noqa: E402
from tests import oracle_lib  # noqa: E402
from tools.coords_probe import card  # noqa: E402

REPS = 5


def med(values):
    values = sorted(values)
    return values[len(values) // 2]


def stat_call(call):
    call(None)  # warm-up
    runs = []
    for _ in range(3):
        st = sw.BenchmarkStats()
        call(st)
        runs.append(st.seconds)
    return med(runs)


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else None
    info = card()
    print("card (name, power limit, max SM clock):", info, flush=True)
    M = oracle_lib.load().matrix(62).astype(np.int8)
    queries = synth.load_queries()
    res = {"card": info, "scan": [], "alignments": [], "saturation": []}
    with sw.CudaSW4(deviceIds=[0], numTop=1000, blosumType=62) as eng:
        eng.setPseudoDatabase(1_000_000, 256)
        eng.prefetchDBToGpus()
        tot_s = tot_p = 0.0
        for qi, (_, q) in enumerate(queries):
            P = M[dbformat.encode(q)]
            a, b = eng.scan(q), eng.scan(q, pssm=P)  # warm-up
            assert (a.scores, a.referenceIds) == (b.scores, b.referenceIds)
            ts, tp = [], []
            for _ in range(REPS):
                ts.append(eng.scan(q).stats.seconds)
                tp.append(eng.scan(q, pssm=P).stats.seconds)
            s, p = med(ts), med(tp)
            tot_s, tot_p = tot_s + s, tot_p + p
            res["scan"].append({"query": qi, "length": len(q), "sequence_seconds": s, "pssm_seconds": p})
            print(f"peak q{qi:>2} len {len(q):>5}: sequence {s * 1e3:8.3f} ms  pssm {p * 1e3:8.3f} ms  ({(p / s - 1) * 100:+.2f} %)",
                  flush=True)
        cells = 1e6 * 256 * sum(len(q) for _, q in queries)
        print(f"peak, all 20 queries: sequence {cells / tot_s / 1e12:.3f} TCUPS, pssm {cells / tot_p / 1e12:.3f} TCUPS", flush=True)
        res["scan_total"] = {"sequence_seconds": tot_s, "pssm_seconds": tot_p}
        for qi in (0, 9, 19):
            q = queries[qi][1]
            P = M[dbformat.encode(q)]
            ids = eng.scan(q).referenceIds
            for k in (10, 1000):
                row = {"case": f"peak, query {qi}, top-{k}", "query_length": len(q)}
                for form, kw in (("sequence", {}), ("pssm", {"pssm": P})):
                    row[f"coords_{form}"] = stat_call(lambda st, kw=kw: eng.alignmentCoordinates(q, ids[:k], stats=st, **kw))
                    row[f"traceback_{form}"] = stat_call(lambda st, kw=kw: eng.alignments(q, ids[:k], stats=st, **kw))
                res["alignments"].append(row)
                print(row, flush=True)
    rng = np.random.default_rng(5)
    _, c5q = synth.config_c5(n_subjects=2)
    qc = c5q[-1]
    with sw.CudaSW4(deviceIds=[0], numTop=1, blosumType=62) as eng:
        eng.setDatabase(dbformat.from_sequences([synth.mutate(rng, qc, 0.1, indels=10)]))
        ql, P = dbformat.decode(qc), M[qc]
        row = {"case": "35 k x 35 k pair", "query_length": len(qc)}
        for form, kw in (("sequence", {}), ("pssm", {"pssm": P})):
            row[f"coords_{form}"] = stat_call(lambda st, kw=kw: eng.alignmentCoordinates(ql, [0], stats=st, **kw))
            row[f"traceback_{form}"] = stat_call(lambda st, kw=kw: eng.alignments(ql, [0], stats=st, **kw))
        res["alignments"].append(row)
        print(row, flush=True)
    # saturation: 5 % of 1 M x 256 subjects carry the consensus; short queries re-score them on sw_s32_kernel
    n, L = 1_000_000, 256
    lengths = np.full(n, L, np.int32)
    consensus = synth.random_residues(rng, L)
    planted = {int(i): consensus for i in range(0, n, 20)}
    with sw.CudaSW4(deviceIds=[0], numTop=10, blosumType=62) as eng:
        eng.setPseudoDatabaseLengths(lengths, 7, planted)
        eng.prefetchDBToGpus()
        for ql in (200, 256):
            q = synth.random_residues(rng, ql)
            P = rng.integers(-4, 1, (ql, 21)).astype(np.int8)
            P[np.arange(ql), consensus[:ql]] = 127
            eng.scan(dbformat.decode(q), pssm=P)
            r = [eng.scan(dbformat.decode(q), pssm=P) for _ in range(REPS)]
            eng.scan(dbformat.decode(q), pssm=M[q])
            base = med([eng.scan(dbformat.decode(q), pssm=M[q]).stats.seconds for _ in range(REPS)])
            row = {"query_length": ql, "saturating_seconds": med([x.stats.seconds for x in r]), "top_score": r[0].scores[0],
                   "num_overflows": r[0].stats.numOverflows, "rescored_subjects": len(planted), "matrix_rows_seconds": base}
            res["saturation"].append(row)
            print(row, flush=True)
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
