"""Cost of the iterative profile search per round: device time of the scan, the traceback of the included hits and the
profile construction, in one process on one GPU.
  python tools/iterate_probe.py [OUT_JSON]

Database: C3-shaped (570,000 subjects of Swiss-Prot-like lengths, 205 M residues, 25 of 8-35 k residues; generated on
the device with sw4_set_pseudo_database_lengths) with QUERIES planted families of 32 members each, from near to
distant (tests/test_profile_search.py: family_members); the queries are the families' ancestors, of 150, 300 and 600
residues. BLOSUM62 -11/-1, numTop 500, statistics on.
Per query, 3 rounds are redone through the public calls that searchIterative's rounds consist of:
  scan (with the previous round's PSSM), the hits with E <= 0.002, alignments() of those hits (the traceback: coordinate
  passes, pass 3 and the walk) and buildPssm() of the same hits (the same passes plus the scatter and the profile
  kernels). Each step is device-timed (CUDA events, median of REPS after a warm-up); "build" is buildPssm's time, and
  "build - traceback" what the profile adds to the traceback it runs. searchIterative(iterations=3) is checked to return
  the last manual round, and its own device time (the sum over its scans and builds) is reported."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import cudasw4_b200 as sw  # noqa: E402
from cudasw4_b200 import dbformat  # noqa: E402
from tools.coords_probe import card  # noqa: E402
from tools.evalue_probe import c3_lengths, med  # noqa: E402
from tests.test_profile_search import family_members, plant  # noqa: E402

REPS = 3
QUERIES = 3
INCLUSION = 0.002


def planted_c3(seed=3):
    rng = np.random.default_rng(seed + 1000)
    queries, members = [], []
    for k, qlen in enumerate((150, 300, 600)[:QUERIES]):
        anc, fam = family_members(rng, qlen)
        queries.append((f"family{k}", dbformat.decode(anc)))
        members += fam
    L, planted, _ = plant(c3_lengths(seed), members)
    return queries, L, planted


def timed(fn):
    fn()  # warm-up
    values = []
    for _ in range(REPS):
        st = sw.BenchmarkStats()
        fn(st)
        values.append(st.seconds)
    return med(values)


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else None
    info = card()
    print("card (name, power limit, max SM clock):", info, flush=True)
    queries, L, planted = planted_c3()
    res = {"card": info, "subjects": int(len(L)), "residues": int(L.sum()), "queries": []}
    with sw.CudaSW4(deviceIds=[0], numTop=500, blosumType=62) as eng:
        eng.setPseudoDatabaseLengths(L, 3, planted=planted)
        eng.prefetchDBToGpus()
        eng.setScoreStatistics(True)
        for qi, (_, q) in enumerate(queries):
            P, rounds = None, []
            for i in range(1, 4):
                r = eng.scan(q, pssm=P)
                hits = [j for j, e in zip(r.referenceIds, r.evalues) if e <= INCLUSION]

                def scan(st=None, P=P):
                    s = eng.scan(q, pssm=P).stats
                    if st is not None:
                        st.seconds = s.seconds

                t_scan = timed(scan)
                row = {"round": i, "hits": len(hits), "hit_residues": int(sum(int(L[h]) for h in hits)), "scan_seconds": t_scan}
                if i < 3 and hits:
                    t_tb = timed(lambda st=None: eng.alignments(q, hits, pssm=P, stats=st))
                    t_build = timed(lambda st=None: eng.buildPssm(q, hits, pssm=P, stats=st))
                    row.update(traceback_seconds=t_tb, build_seconds=t_build)
                    P = eng.buildPssm(q, hits, pssm=P)
                rounds.append(row)
                print(f"q{qi} len {len(q):>5} round {i}: {len(hits):>4} hits ({row['hit_residues']} residues)  scan "
                      f"{t_scan * 1e3:8.3f} ms" + (f"  traceback {row['traceback_seconds'] * 1e3:8.3f} ms  build "
                                                  f"{row['build_seconds'] * 1e3:8.3f} ms (build - traceback "
                                                  f"{(row['build_seconds'] - row['traceback_seconds']) * 1e3:.3f} ms)"
                                                  if "build_seconds" in row else ""), flush=True)
                if not hits:
                    break
            it = eng.searchIterative(q, iterations=3, inclusionEvalue=INCLUSION)
            if len(rounds) == 3:
                assert it.iterations == 3 or it.converged
                if it.iterations == 3:
                    assert it.result.referenceIds == r.referenceIds and (it.pssm == P).all()
            print(f"q{qi}: searchIterative {it.iterations} rounds, converged {it.converged}, device time "
                  f"{it.result.stats.seconds * 1e3:.3f} ms", flush=True)
            res["queries"].append({"query": qi, "length": len(q), "rounds": rounds, "iterative_rounds": it.iterations,
                                   "converged": it.converged, "iterative_seconds": it.result.stats.seconds})
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
