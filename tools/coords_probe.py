"""Alignment-coordinate timings (sw4_alignment_coordinates) beside the scan of the same query, on one GPU.
  python tools/coords_probe.py [OUT_JSON]

Cases (DESIGN.md 3.6): the peak-benchmark shape (PseudoDB 1 M x 256) with queries 0, 9 and 19 of allqueries, top-10
and top-1000 hits; the long-subject shape of scale_probe.py c5 (2,024 subjects of 2-35 k residues) with query 19 and
a 35,000-residue query, top-10; the Swiss-Prot-shaped database (synth.config_c3) with a ~500-residue query, 4,096
hits. Every time is the call's device-timed stats (CUDA events) after one warm-up call, median of 3."""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import cudasw4_b200 as sw  # noqa: E402
from cudasw4_b200 import dbformat, synth  # noqa: E402

REPS = 3


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                       text=True, check=True)
    return r.stdout.strip().splitlines()[1]


def measure(eng, label, query, ids, results):
    eng.scan(query)  # warm-up of the scan of this query
    scans = sorted(eng.scan(query).stats.seconds for _ in range(REPS))
    eng.alignmentCoordinates(query, ids)  # warm-up
    runs = []
    for _ in range(REPS):
        st = sw.BenchmarkStats()
        eng.alignmentCoordinates(query, ids, stats=st)
        runs.append(st)
    runs.sort(key=lambda s: s.seconds)
    st = runs[len(runs) // 2]
    row = {"case": label, "query_length": len(query), "ids": len(ids), "cells": st.cells, "seconds": st.seconds,
           "gcups": st.gcups, "kernel_launches": st.kernelLaunches, "scan_seconds": scans[len(scans) // 2]}
    row["share_of_scan"] = row["seconds"] / row["scan_seconds"]
    results.append(row)
    print(f"{label:<44} q={len(query):>6} ids={len(ids):>5} cells={st.cells:.3e} {st.seconds * 1e3:9.3f} ms "
          f"{st.gcups:8.1f} GCUPS | scan {row['scan_seconds'] * 1e3:9.3f} ms ({100 * row['share_of_scan']:.2f} %)", flush=True)


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else None
    info = card()
    print("card (name, power limit, max SM clock):", info, flush=True)
    queries = synth.load_queries()
    results = []
    with sw.CudaSW4(deviceIds=[0], numTop=1000, blosumType=62) as eng:
        eng.setPseudoDatabase(1_000_000, 256)
        eng.prefetchDBToGpus()
        for qi in (0, 9, 19):
            q = queries[qi][1]
            ids = eng.scan(q).referenceIds
            for k in (10, 1000):
                measure(eng, f"PseudoDB 1M x 256, query {qi}, top-{k}", q, ids[:k], results)
    db, c5q = synth.config_c5(n_subjects=2000)
    with sw.CudaSW4(deviceIds=[0], numTop=10, blosumType=62) as eng:
        eng.setDatabase(db)
        eng.prefetchDBToGpus()
        for label, q in (("query 19", queries[19][1]), ("35,000-residue query", dbformat.decode(c5q[-1]))):
            ids = eng.scan(q).referenceIds
            measure(eng, f"C5 {db.num_sequences} x 2-35 k, {label}, top-10", q, ids, results)
    del db
    db = synth.config_c3()
    lengths = [len(s) for _, s in queries]
    qi = int(np.argmin([abs(n - 500) for n in lengths]))
    with sw.CudaSW4(deviceIds=[0], numTop=4096, blosumType=62) as eng:
        eng.setDatabase(db)
        eng.prefetchDBToGpus()
        q = queries[qi][1]
        ids = eng.scan(q).referenceIds
        measure(eng, f"Swiss-Prot-shaped, query {qi}, 4,096 hits", q, ids, results)
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            json.dump({"card": info, "results": results}, f, indent=1)


if __name__ == "__main__":
    main()
