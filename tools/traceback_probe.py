"""Alignment-traceback timings (sw4_alignment_traceback) beside the coordinates call and the scan of the same query.
  python tools/traceback_probe.py [OUT_JSON]

Cases: those of tools/coords_probe.py (DESIGN.md 3.6). Every time is the call's device-timed stats (CUDA events) after
one warm-up call, median of 3. For the 35,000-residue query, one further traceback call runs under torch.profiler and
the device time of every kernel is summed by name: passes 1-2 (sw_coords_kernel), pass 3 (sw_coords_trace_kernel) and
the walk (sw_coords_walk_kernel)."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import cudasw4_b200 as sw  # noqa: E402
from cudasw4_b200 import dbformat, synth  # noqa: E402
from tools.coords_probe import REPS, card  # noqa: E402


def median_stats(call):
    call()  # warm-up
    runs = []
    for _ in range(REPS):
        st = sw.BenchmarkStats()
        call(st)
        runs.append(st)
    runs.sort(key=lambda s: s.seconds)
    return runs[len(runs) // 2]


def measure(eng, label, query, ids, results):
    eng.scan(query)
    scan = sorted(eng.scan(query).stats.seconds for _ in range(REPS))[REPS // 2]
    co = median_stats(lambda st=None: eng.alignmentCoordinates(query, ids, stats=st))
    tb = median_stats(lambda st=None: eng.alignments(query, ids, stats=st))
    row = {"case": label, "query_length": len(query), "ids": len(ids), "scan_seconds": scan,
           "coords_seconds": co.seconds, "coords_cells": co.cells, "traceback_seconds": tb.seconds,
           "traceback_cells": tb.cells, "traceback_launches": tb.kernelLaunches}
    results.append(row)
    print(f"{label:<44} q={len(query):>6} ids={len(ids):>5} | scan {scan * 1e3:9.3f} ms | coords {co.seconds * 1e3:9.3f} ms"
          f" | traceback {tb.seconds * 1e3:9.3f} ms ({tb.cells:.3e} cells, {tb.kernelLaunches} launches)", flush=True)


def kernel_split(eng, query, ids):
    """Device time per kernel name of one traceback call, from torch.profiler (CUPTI sees every kernel of the process)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.zeros(1, device="cuda")
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        eng.alignments(query, ids)
        torch.cuda.synchronize()
    out = {}
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            for key in ("sw_coords_walk_kernel", "sw_coords_trace_kernel", "sw_coords_kernel", "convert_query_kernel"):
                if key in ev.name:
                    out[key] = out.get(key, 0.0) + ev.device_time * 1e-6
                    break
    return out


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else None
    info = card()
    print("card (name, power limit, max SM clock):", info, flush=True)
    queries = synth.load_queries()
    results, split = [], {}
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
        # one 35 k x 35 k pair: the query against a copy of itself with substitutions and indels
        rng = np.random.default_rng(5)
        qc = c5q[-1]
        planted = synth.mutate(rng, qc, 0.1, indels=10)
        db2 = dbformat.from_sequences([planted])
        eng.setDatabase(db2)
        ql = dbformat.decode(qc)
        measure(eng, "35 k x 35 k pair (10 % substitutions, 10 indels)", ql, [0], results)
        split = kernel_split(eng, ql, [0])
        print("35 k x 35 k pair, device seconds per kernel:", split, flush=True)
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
            json.dump({"card": info, "results": results, "split_35k": split}, f, indent=1)


if __name__ == "__main__":
    main()
