#!/usr/bin/env python3
"""Headline benchmark: GCUPS of the database scan hot path on BASELINE.json config[1]
(the reference's "peak benchmark": PseudoDB of 1,000,000 equal-length subjects (256 aa) vs the 20 queries of
allqueries.fasta, BLOSUM62 -11/-1, database resident, `runpeakbenchmark.sh:26-54`).

  python bench.py --gpus N --steps K --warmup W            (N>1: launched by torchrun, one rank per GPU)
  python bench.py --impl reference ...                       (CPU arm: the oracle port on the host cores)
  python bench.py ... --dump-outputs DIR                     (also writes the last timed step's top-k lists as .npy)

A *step* = one pass of the hot path over the whole query batch: all 20 queries scanned against the resident database
(20 sw4_scan calls through the C ABI, each: query H2D -> profile -> score kernels -> top-k -> k results D2H).
Weak scaling: every rank holds 1,000,000 subjects (shard `rank` of a N x 1M-subject database, global ids); the only
exchange is an all_gather of k (score, id) pairs per rank per query, merged on rank 0.

Two more legs run after the timed region of the headline metric (they never change `value`):
  c4           STRONG scaling on ONE fixed UniRef50-shaped database (C4: 65,000,000 subjects / 17.0 G residues, seed 4,
               sw4_set_pseudo_database_lengths): every rank generates and uploads only its own shard (blocks of 256
               subjects, rank, rank+N, ...), queries 0/5/9/14/19, one pass, per-query GCUPS = cells / max-over-ranks
               device time; `checked` = planted copies found with their self score and a >= 3,000-subject sample of
               every rank's scores equal to the CPU oracle (the reference's multi-GPU use, rununiref50benchmark.sh).
  ref_gpu      the reference's OWN align binary (oracle/_ref/align, built for sm_100a from /root/reference), --dpx and
               default half2 kernels, on the same PseudoDB (runpeakbenchmark.sh:27,44-50), timed on the same GPU
               right after ours (rank 0, N = 1 only).

  value        GCUPS from the device-timed scan regions (CUDA events inside libsw4b200.so on its own stream, the
               reference's own "Scan time" definition, src/cudasw4.cuh:707-726), max over ranks
  e2e          GCUPS from host wall-clock around the same C-ABI calls with HOST query buffers (pinned staging, H2D,
               D2H of the results inside the timed region), max over ranks
  roofline     score kernels only, against the ALU(DPX)-pipe roofline measured with tools/ubench (see DESIGN.md)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_SUBJECTS = 1_000_000
SUBJECT_LEN = 256
TOP_K = 10
CONFIG_NAME = "peak benchmark: PseudoDB 1,000,000 x 256 aa per GPU vs allqueries.fasta (20 queries, 41,752 aa), BLOSUM62 gop=-11 gex=-1, top-10, DB resident"


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback"


def _traffic():
    """dram__bytes_read+write of the dominant kernel per launch, from the committed ncu capture (profiles/)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f)
    except Exception:
        return None


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop_evt = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for n, v in zip(names, out[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=3)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


class _ReferenceCpuScan:
    """The reference's OWN scalar CPU Gotoh (src/cudasw4.cuh:2331-2392, BLOSUM62), compiled from /root/reference into
    oracle/_ref/libref_harness.so by oracle/Makefile and driven one OpenMP task per subject like its
    computeAllScoresCPU_blosum62 (src/cudasw4.cuh:767-796). Present when the harness travelled with the repository."""

    def __init__(self, path):
        import ctypes
        self.lib = ctypes.CDLL(path)
        self.fn = self.lib.ref_cpu_scan_blosum62
        self.fn.restype = ctypes.c_int
        self.last_threads = 0

    def scan(self, blosum, q, db, gop, gex, threads=0):
        import ctypes
        import numpy as np
        assert blosum == 62
        q = np.ascontiguousarray(q, dtype=np.uint8)
        chars = np.ascontiguousarray(db.chars, dtype=np.uint8)
        offsets = np.ascontiguousarray(db.offsets, dtype=np.uint64)
        lengths = np.ascontiguousarray(db.lengths, dtype=np.int32)
        out = np.empty(len(lengths), dtype=np.int32)
        p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
        self.last_threads = self.fn(p(q), ctypes.c_int(len(q)), p(chars), p(offsets), p(lengths), ctypes.c_long(len(lengths)),
                                    ctypes.c_int(gop), ctypes.c_int(gex), p(out), ctypes.c_int(threads))
        return out


def _cpu_scanner():
    """(scanner, kind): the reference's own CPU routine when oracle/_ref holds it, else the oracle port."""
    path = os.path.join(ROOT, "oracle", "_ref", "libref_harness.so")
    if os.path.exists(path) and not os.environ.get("SW4_BENCH_CPU_PORT"):
        try:
            return _ReferenceCpuScan(path), "reference"
        except (OSError, AttributeError):
            pass
    from tests import oracle_lib
    return oracle_lib.load(), "port"


def host_threads() -> int:
    """Threads for the CPU arm: every core this process may run on. (torchrun exports OMP_NUM_THREADS=1, which would
    silently turn an `omp_get_max_threads()` default into a 1-core baseline.)"""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_baseline(seconds_budget: float = 20.0, threads: int = 0):
    """CPU Gotoh (the reference's own scalar routine if built, else the oracle port; OpenMP over subjects) on a bounded
    sample of the same workload."""
    import numpy as np
    threads = threads or host_threads()
    from cudasw4_b200 import dbformat, synth
    oracle, kind = _cpu_scanner()
    queries = [dbformat.encode(s) for _, s in synth.load_queries()]
    subj = synth.pseudo_subject(SUBJECT_LEN, 42)
    # calibrate: 256 subjects x shortest query
    db = dbformat.from_equal_length_matrix(np.broadcast_to(subj, (256, SUBJECT_LEN)).copy())
    t0 = time.perf_counter()
    oracle.scan(62, queries[0], db, -11, -1, threads=threads)
    dt = max(time.perf_counter() - t0, 1e-4)
    rate = 256 * SUBJECT_LEN * len(queries[0]) / dt
    total_q = sum(len(q) for q in queries)
    n = int(max(64, min(N_SUBJECTS, seconds_budget * rate / (SUBJECT_LEN * total_q))))
    db = dbformat.from_equal_length_matrix(np.broadcast_to(subj, (n, SUBJECT_LEN)).copy())
    t0 = time.perf_counter()
    for q in queries:
        oracle.scan(62, q, db, -11, -1, threads=threads)
    dt = time.perf_counter() - t0
    cells = float(n) * SUBJECT_LEN * total_q
    return {"value": cells / 1e9 / dt, "unit": "GCUPS", "cores": int(oracle.last_threads), "kind": kind,
            "sample": f"first {n} of {N_SUBJECTS} subjects x all 20 queries ({cells:.3g} cells, {dt:.1f} s)"}, dt, cells


def run_reference(args, rank, world):
    if rank != 0:
        return
    steps_dt, steps_cells = [], []
    base = None
    for i in range(args.warmup + args.steps):
        base, dt, cells = cpu_baseline(seconds_budget=max(2.0, 60.0 / max(1, args.warmup + args.steps)))
        if i >= args.warmup:
            steps_dt.append(dt)
            steps_cells.append(cells)
    value = sum(steps_cells) / 1e9 / sum(steps_dt)
    base["value"] = value
    line = {"impl": "reference", "metric": "GCUPS", "value": value, "unit": "GCUPS", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * sum(steps_dt) / len(steps_dt), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": {"workload": CONFIG_NAME, "note": "CPU arm: the reference ships no CPU aligner; this is its own scalar "
                       "checking routine (src/cudasw4.cuh:2331-2392, built into oracle/_ref) or, without it, the oracle port, "
                       "on all host cores, bounded sample per step (see cpu_baseline.kind)"},
            "cpu_baseline": base,
            "e2e": {"value": value, "unit": "GCUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


C4_QUERIES = (0, 5, 9, 14, 19)
C4_SUBJECTS = 65_000_000
C4_RESIDUES = 17.0e9
C4_SEED = 4


def c4_leg(rank, local_rank, world, dev):
    """STRONG scaling on one fixed UniRef50-shaped database (see the module docstring). Returns the `c4` object on rank 0."""
    import numpy as np
    import torch
    import torch.distributed as dist
    import cudasw4_b200 as sw
    from cudasw4_b200 import dbformat, synth
    from cudasw4_b200.distributed import gather_topk
    from tests import oracle_lib  # the checker (CPU oracle); never on the measured path

    n_seqs = int(os.environ.get("SW4_BENCH_C4_SUBJECTS", C4_SUBJECTS))
    t0 = time.perf_counter()
    lengths = synth.config_c4_lengths(seed=C4_SEED, n=n_seqs, total=C4_RESIDUES * n_seqs / C4_SUBJECTS).astype(np.int32)
    queries = synth.load_queries()
    planted = {}
    for qi in C4_QUERIES:  # one exact copy of each query in the slot of a subject of the same length
        codes = dbformat.encode(queries[qi][1])
        gid = int(np.searchsorted(lengths, len(codes), side="left"))
        while gid in planted:
            gid += 1
        if gid < n_seqs and int(lengths[gid]) == len(codes):
            planted[gid] = codes
    eng = sw.CudaSW4(deviceIds=[local_rank], numTop=TOP_K, blosumType=62)
    eng.setShard(rank, world)
    eng.setPseudoDatabaseLengths(lengths, C4_SEED, planted)
    gen_s = time.perf_counter() - t0
    t0 = time.perf_counter()
    eng.prefetchDBToGpus()
    upload_s = time.perf_counter() - t0
    info = eng.dbInfo()
    total_residues = float(lengths.astype(np.int64).sum())
    oracle = oracle_lib.load()
    planted_by_len = {len(c): g for g, c in planted.items()}

    def sync():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()

    per_query, checked, sample_total, sum_cells, sum_s = [], True, 0, 0.0, 0.0
    single_results = []
    for qi in C4_QUERIES:
        q = queries[qi][1]
        qc = dbformat.encode(q)
        sync()
        res = eng.scan(q)
        single_results.append((res.scores, res.referenceIds))
        t = torch.tensor([res.stats.seconds], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        seconds = float(t.item())
        merged = gather_topk(res.scores, res.referenceIds, TOP_K, device=dev)
        # checks: (1) the planted copy is the best hit with the query's self score; (2) a sample of this rank's scores
        # (evenly spaced over its shard + its longest subjects) equals the CPU oracle on re-generated sequences
        ok = True
        if len(qc) in planted_by_len:
            self_score = int(oracle.scan(62, qc, dbformat.from_sequences([qc]), -11, -1)[0])
            ok &= merged[0] == (self_score, planted_by_len[len(qc)])
        scores, ids = eng.lastScanAllScores()
        n_local = len(ids)
        want = max(64, 3040 // world)
        pos = np.unique(np.concatenate([np.arange(0, n_local, max(1, n_local // want)), np.arange(max(0, n_local - 8), n_local)]))
        seqs = [planted[int(g)] if int(g) in planted else synth.pseudo_lengths_sequence(C4_SEED, int(g), int(lengths[g])) for g in ids[pos]]
        sample = dbformat.from_sequences(seqs, presorted=True)
        ok &= bool((oracle.scan(62, qc, sample, -11, -1, threads=host_threads()) == scores[pos]).all())
        flag = torch.tensor([1 if ok else 0, len(pos)], dtype=torch.int64, device=dev)
        if world > 1:
            both = [torch.zeros_like(flag) for _ in range(world)]
            dist.all_gather(both, flag)
            ok = all(int(b[0]) == 1 for b in both)
            n_sample = sum(int(b[1]) for b in both)
        else:
            n_sample = len(pos)
        checked &= ok
        sample_total = n_sample
        cells = total_residues * len(qc)
        sum_cells += cells
        sum_s += seconds
        per_query.append({"query": qi, "length": len(qc), "gcups": cells / 1e9 / seconds, "seconds": seconds,
                          "top1": list(merged[0]) if merged else None, "overflows": res.stats.numOverflows})
    # the same five queries through sw4_scan_many (several scans in flight): device-timed span of the call, max over ranks
    sync()
    many, total = eng.scanMany([queries[qi][1] for qi in C4_QUERIES])
    t = torch.tensor([total.seconds], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    batched_gcups = sum_cells / 1e9 / float(t.item())
    batched_same = all(m.scores == eng_res[0] and m.referenceIds == eng_res[1] for m, eng_res in zip(many, single_results))
    flag = torch.tensor([1 if batched_same else 0], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    checked &= bool(int(flag.item()))
    eng.close()
    if rank != 0:
        return None
    return {"gcups": sum_cells / 1e9 / sum_s, "batched_gcups": batched_gcups, "n_gpus": world, "scaling": "strong",
            "per_query": per_query, "checked": bool(checked),
            "check": f"planted copies of queries {list(C4_QUERIES)} found with their self scores; {sample_total} sampled subjects "
                     f"(all ranks) x 5 queries equal to the CPU oracle; sw4_scan_many lists equal to the single scans",
            "database": {"subjects": n_seqs, "residues": total_residues, "max_length": int(lengths[-1]),
                         "shard_subjects_rank0": int(info.shard_sequences), "shard_residues_rank0": int(info.shard_residues)},
            "generate_s": gen_s, "upload_s": upload_s, "queries": list(C4_QUERIES)}


def ref_gpu_leg(local_rank, ours_e2e_gcups, ours_value_gcups):
    """The reference's own align binary (oracle/_ref/align: unmodified sources built for sm_100a) on the same PseudoDB,
    same GPU, --dpx and default (half2) kernel types, as runpeakbenchmark.sh:27,44-50 runs it."""
    import re
    import tempfile
    from cudasw4_b200 import dbformat, synth
    binary = os.path.join(ROOT, "oracle", "_ref", "align")
    if not os.path.exists(binary):
        return {"unavailable": "oracle/_ref/align not built (needs /root/reference at build time)"}
    env = dict(os.environ)
    visible = env.get("CUDA_VISIBLE_DEVICES")
    env["CUDA_VISIBLE_DEVICES"] = visible.split(",")[local_rank] if visible else str(local_rank)
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        qfile = os.path.join(tmp, "allqueries.fasta")
        dbformat.write_fasta(qfile, synth.load_queries())
        for tag, extra in (("dpx", ["--dpx"]), ("half2", [])):
            args = [binary, "--query", qfile, "--pseudodb", str(N_SUBJECTS), str(SUBJECT_LEN), "--top", "0", "--verbose",
                    "--uploadFull", "--prefetchDBFile", "--mat", "blosum62"] + extra
            try:
                r = subprocess.run(args, cwd=tmp, env=env, capture_output=True, text=True, timeout=300)
            except subprocess.TimeoutExpired:
                out[tag + "_gcups"] = None
                continue
            tot = re.findall(r"Total time: ([0-9.e+-]+) s, ([0-9.e+-]+) GCUPS", r.stdout)
            per = re.findall(r"Scan time: ([0-9.e+-]+) s, ([0-9.e+-]+) GCUPS", r.stdout)
            out[tag + "_gcups"] = float(tot[-1][1]) if tot else None
            if per:  # aggregate of its per-query device-timed scans: sum(cells) / sum(scan seconds)
                secs = sum(float(p[0]) for p in per)
                out[tag + "_scan_gcups"] = N_SUBJECTS * SUBJECT_LEN * sum(len(q) for _, q in synth.load_queries()) / 1e9 / secs if secs > 0 else None
            if r.returncode != 0:
                out[tag + "_error"] = (r.stderr or r.stdout)[-200:]
    best = max([v for v in (out.get("dpx_gcups"), out.get("half2_gcups")) if v] or [0.0])
    best_scan = max([v for v in (out.get("dpx_scan_gcups"), out.get("half2_scan_gcups")) if v] or [0.0])
    out["ratio_vs_best"] = ours_e2e_gcups / best if best else None           # our end-to-end vs its "Total time" GCUPS
    out["ratio_vs_best_scan"] = ours_value_gcups / best_scan if best_scan else None  # device-timed scans on both sides
    out["command"] = "align --query allqueries.fasta --pseudodb 1000000 256 --top 0 --verbose --uploadFull --prefetchDBFile --mat blosum62 [--dpx]"
    return out


def dump_outputs(out_dir, merged):
    """What a caller of the timed path receives, from its last step: the merged top-k (score, global id) lists of the
    20 queries, as float64 (n_queries, TOP_K) arrays topk_scores.npy and topk_ids.npy (NaN pads a shorter list). The
    database and the queries are fixed, so two builds run with the same arguments can be compared array for array."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, col in (("topk_scores", 0), ("topk_ids", 1)):
        a = np.full((len(merged), TOP_K), np.nan)
        for qi, pairs in enumerate(merged):
            a[qi, :len(pairs)] = [p[col] for p in pairs]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-c4", action="store_true", help="skip the C4 strong-scaling leg")
    ap.add_argument("--no-ref-gpu", action="store_true", help="skip timing the reference's own GPU binary")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")  # one hardware queue per length-class stream
    import numpy as np
    import torch
    import torch.distributed as dist
    import cudasw4_b200 as sw
    from cudasw4_b200 import synth

    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local_rank))
    else:
        torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    queries = synth.load_queries()
    letters = [q for _, q in queries]
    total_q = sum(len(q) for q in letters)
    eng = sw.CudaSW4(deviceIds=[local_rank], numTop=TOP_K, blosumType=62)  # raises if libsw4b200.so / the GPU is missing
    eng.setShard(rank, world)
    eng.setPseudoDatabase(N_SUBJECTS * world, SUBJECT_LEN, 42)
    t0 = time.perf_counter()
    eng.prefetchDBToGpus()
    upload_s = time.perf_counter() - t0
    info = eng.dbInfo()
    shard_residues = int(info.shard_residues)

    from cudasw4_b200.distributed import gather_topk
    single = bool(os.environ.get("SW4_BENCH_SINGLE"))  # development switch: one sw4_scan per query instead of sw4_scan_many

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def one_step():
        """One pass of the hot path over the query batch: the 20 queries through sw4_scan_many (host letters in, top-k
        out). Returns (device-timed seconds of the call, launches, merged top-k list of every query)."""
        if single:
            dev_s, launches, results = 0.0, 0, []
            for q in letters:
                r = eng.scan(q)
                dev_s += r.stats.seconds
                launches += r.stats.kernelLaunches
                results.append(r)
        else:
            results, total = eng.scanMany(letters)
            dev_s, launches = total.seconds, total.kernelLaunches
        # the only exchange step: k (score, id) pairs per rank and query (NCCL all_gather), merged on every rank
        merged = [gather_topk(r.scores, r.referenceIds, TOP_K, device=dev) for r in results]
        return dev_s, launches, merged

    def kernel_step():
        """Same 20 queries one sw4_scan at a time: the score kernels of one query run alone, so their CUDA-event time
        (stats.kernel_seconds) is exclusive. Used for the roofline only."""
        ker_s = 0.0
        for q in letters:
            ker_s += eng.scan(q).stats.kernelSeconds
        return ker_s

    for _ in range(args.warmup):
        one_step()
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    wall0 = time.perf_counter()
    dev_s = 0.0
    launches = 0
    merged = None
    for _ in range(args.steps):
        d, l, merged = one_step()
        dev_s += d
        launches += l
    barrier()
    wall = time.perf_counter() - wall0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, merged)
    ker_s = 0.0
    for _ in range(args.steps):
        ker_s += kernel_step()
    clocks = sampler.stop()
    eng.close()

    # max over ranks; exact cell count = sum of the ranks' shard residues
    t = torch.tensor([dev_s, ker_s, wall], dtype=torch.float64, device=dev)
    lt = torch.tensor([launches, shard_residues], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(lt, op=dist.ReduceOp.SUM)
    dev_s, ker_s, wall = [float(x) for x in t.cpu()]
    launches, all_residues = int(lt[0].item()), int(lt[1].item())

    c4 = None
    if not args.no_c4 and os.environ.get("SW4_BENCH_C4", "1") != "0":
        try:
            c4 = c4_leg(rank, local_rank, world, dev)
        except Exception as exc:  # the headline line must still be printed
            c4 = {"error": f"{type(exc).__name__}: {exc}"[:300]}

    if rank == 0:
        cells_per_step = float(all_residues) * total_q
        cells = cells_per_step * args.steps
        value = cells / 1e9 / dev_s
        e2e = cells / 1e9 / wall
        kernel_gcups = cells / 1e9 / ker_s
        peaks, peak_src = _peaks()
        sm_hz = (clocks["sm_mhz"] or peaks.get("sm_max_mhz", 1965.0)) * 1e6
        # ALU(DPX)-pipe roofline: 3.5 ALU-pipe instructions per cell-pair (1 max3-relu, 2 add-max, 1/2 max3), pipe issues one
        # warp instruction per 2 clocks per scheduler (measured, tools/ubench/pipes.cu): 64 cells per 7 clocks per scheduler
        sms = torch.cuda.get_device_properties(dev).multi_processor_count
        peak_gcups = sms * 4 * 64 / 7.0 * sm_hz / 1e9 * world
        # HBM side (for the record): per scan the kernel streams the shard once, 1 byte per residue (u16 fused pair code)
        hbm_bytes = float(all_residues) * len(queries) * args.steps
        line = {
            "metric": "GCUPS", "value": value, "unit": "GCUPS", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dev_s / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "s16x2 (DPX) with exact s32 re-scoring", "data": "synthetic",
            "config": {"workload": CONFIG_NAME, "subjects_per_gpu": N_SUBJECTS, "subject_length": SUBJECT_LEN,
                       "queries": len(queries), "query_residues": total_q, "cells_per_step": cells_per_step,
                       "api": "20 sw4_scan calls per step" if single else "one sw4_scan_many call per step (20 queries, 3 in flight)",
                       "timing": "value: CUDA events inside libsw4b200.so on its own streams, first query's upload -> last "
                                 "result in pinned host memory, max over ranks; e2e: host wall clock around the same calls + "
                                 "the NCCL gather of the per-rank top-k",
                       "l2_note": "each scan streams 256 MB of database per GPU (> 126 MB L2) and scans alternate 20 different "
                                  "query profiles, so no timed iteration re-reads L2-resident inputs",
                       "db_upload_s": upload_s, "top1": merged[-1][0] if merged and merged[-1] else None},
            "clocks": clocks,
            "e2e": {"value": e2e, "unit": "GCUPS", "h2d_bytes_per_step": total_q + 441 * len(queries),
                    "d2h_bytes_per_step": len(queries) * (2 * TOP_K * 4 + 32)},
            "gpu_launches": launches,
            "roofline": {"bound": "int_dpx_pipe", "achieved": kernel_gcups, "peak": peak_gcups, "unit": "GCUPS",
                         "frac": kernel_gcups / peak_gcups,
                         "peak_model": f"{sms} SMs x 4 schedulers x 64 cells / 7 clk (3.5 DPX ALU-pipe ops per s16x2 cell-pair at "
                                       f"1 warp-inst / 2 clk, measured) x {sm_hz/1e6:.0f} MHz (nvidia-smi under load)",
                         "measured": "score kernels alone (CUDA events around them on the library's stream), the 20 queries "
                                     "scanned one at a time so that the intervals do not overlap, same number of steps",
                         "traffic": (_traffic() or {}).get("dram_bytes_read_plus_write_per_launch"),
                         "traffic_detail": _traffic(),
                         "hbm": {"achieved": hbm_bytes / 1e9 / ker_s, "peak": peaks.get("hbm_gbs"), "unit": "GB/s",
                                 "frac": hbm_bytes / 1e9 / ker_s / peaks.get("hbm_gbs", 6650.0), "peak_source": peak_src,
                                 "note": "database streaming only; the path is compute bound (1/len_query bytes per cell)"}},
        }
        if c4 is not None:
            line["c4"] = c4
        if world == 1 and not args.no_ref_gpu:
            try:
                line["ref_gpu"] = ref_gpu_leg(local_rank, e2e, value)
            except Exception as exc:
                line["ref_gpu"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"], _, _ = cpu_baseline()
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
