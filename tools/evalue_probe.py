"""Cost of score statistics (sw4_set_score_statistics): device time of the same scans with statistics on and off, in one
process on one GPU.
  python tools/evalue_probe.py [OUT_JSON]

1. The peak benchmark (PseudoDB 1,000,000 x 256, BLOSUM62 -11/-1), its 20 queries.
2. A C3-shaped database (570,000 subjects of Swiss-Prot-like lengths, 205 M residues, 25 of 8-35 k residues; generated
   on the device with sw4_set_pseudo_database_lengths), the same 20 queries.
Per query, scans with statistics on and off alternate on one handle after a warm-up of each; the median of REPS
device-timed scans (CUDA events: query upload -> results on the host) is reported per mode. Scores and ids are checked
to be the same in both modes."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import cudasw4_b200 as sw  # noqa: E402
from cudasw4_b200 import synth  # noqa: E402
from tools.coords_probe import card  # noqa: E402

REPS = 7


def med(values):
    values = sorted(values)
    return values[len(values) // 2]


def c3_lengths(seed=3, n=570_000, total=205e6):
    rng = np.random.default_rng(seed)
    L = synth.lognormal_lengths(rng, n - 25, 5.683, 0.636, 2, 35213, total=total)
    return np.sort(np.concatenate([L, rng.integers(8001, 35214, 25)])).astype(np.int32)


def probe(eng, label, queries, residues):
    rows, tot_off, tot_on = [], 0.0, 0.0
    for qi, (_, q) in enumerate(queries):
        eng.setScoreStatistics(False)
        a = eng.scan(q)
        eng.setScoreStatistics(True)
        b = eng.scan(q)
        assert (a.scores, a.referenceIds) == (b.scores, b.referenceIds) and b.statistics.ok
        off, on = [], []
        for _ in range(REPS):
            eng.setScoreStatistics(False)
            off.append(eng.scan(q).stats.seconds)
            eng.setScoreStatistics(True)
            on.append(eng.scan(q).stats.seconds)
        t0, t1 = med(off), med(on)
        tot_off, tot_on = tot_off + t0, tot_on + t1
        st = b.statistics
        rows.append({"query": qi, "length": len(q), "off_seconds": t0, "on_seconds": t1, "lambda": st.lambda_, "K": st.K,
                     "c_lo": st.c_lo, "c_hi": st.c_hi, "top_evalue": b.evalues[0] if b.evalues else None})
        print(f"{label} q{qi:>2} len {len(q):>5}: off {t0 * 1e3:8.3f} ms  on {t1 * 1e3:8.3f} ms  ({(t1 / t0 - 1) * 100:+.2f} %)"
              f"  lambda {st.lambda_:.4f} K {st.K:.4f}", flush=True)
    cells = residues * sum(len(q) for _, q in queries)
    print(f"{label}, all {len(queries)} queries: off {tot_off * 1e3:.2f} ms ({cells / tot_off / 1e12:.3f} TCUPS), "
          f"on {tot_on * 1e3:.2f} ms ({cells / tot_on / 1e12:.3f} TCUPS), {(tot_on / tot_off - 1) * 100:+.2f} %", flush=True)
    return {"queries": rows, "off_seconds": tot_off, "on_seconds": tot_on}


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else None
    info = card()
    print("card (name, power limit, max SM clock):", info, flush=True)
    queries = synth.load_queries()
    res = {"card": info}
    with sw.CudaSW4(deviceIds=[0], numTop=10, blosumType=62) as eng:
        eng.setPseudoDatabase(1_000_000, 256)
        eng.prefetchDBToGpus()
        res["peak"] = probe(eng, "peak", queries, 1e6 * 256)
    L = c3_lengths()
    with sw.CudaSW4(deviceIds=[0], numTop=10, blosumType=62) as eng:
        eng.setPseudoDatabaseLengths(L, 3)
        eng.prefetchDBToGpus()
        res["c3"] = probe(eng, "c3", queries, float(L.sum()))
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
