"""One-process-per-GPU deployment helpers: the only exchange step of a sharded scan.

Every rank scans its own shard (`CudaSW4.setShard(rank, world)`) and owns a sorted top-k list of (score, global id)
pairs; `gather_topk` all-gathers those k pairs per rank (k * 8 bytes, NCCL on GPUs, gloo in the CPU tests) and merges
them under the engine's total order (score descending, id ascending). This is what the reference does with three
device-to-device copies into GPU 0 plus a thrust sort (reference src/cudasw4.cuh:1415-1458); there is no collective
on the compute path.

`gather_score_statistics` does the same for E-values: it all-reduces every rank's score histogram of one query and fits
the sum, so every rank gets the statistics of the whole database.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.distributed as dist


def merge_topk(lists, k: int):
    """lists: iterable of (scores, ids) per shard. Returns the k best (score, id) pairs, ties by ascending id."""
    pairs = []
    for scores, ids in lists:
        pairs.extend((int(s), int(i)) for s, i in zip(scores, ids) if int(i) >= 0)
    pairs.sort(key=lambda t: (-t[0], t[1]))
    return pairs[:k]


def gather_topk(scores, ids, k: int, device=None, group=None):
    """All ranks call this with their local top-k (shorter lists are padded). Every rank returns the merged list."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    if world == 1:
        return merge_topk([(scores, ids)], k)
    device = device or torch.device("cpu")
    mine = torch.full((2 * k,), -1, dtype=torch.int32, device=device)
    n = min(k, len(scores))
    mine[:n] = torch.as_tensor(list(scores[:n]), dtype=torch.int32, device=device)
    mine[k:k + n] = torch.as_tensor(list(ids[:n]), dtype=torch.int32, device=device)
    out = torch.empty(world * 2 * k, dtype=torch.int32, device=device)  # flat: gloo and nccl both accept this shape
    dist.all_gather_into_tensor(out, mine, group=group)
    rows = out.view(world, 2 * k).cpu().tolist()
    return merge_topk([(r[:k], r[k:]) for r in rows], k)


def gather_score_statistics(sw4, query_index: int, query_length: int, device=None, group=None):
    """All ranks call this after a scan with score statistics enabled (CudaSW4.setScoreStatistics). The int64 histograms
    of query `query_index` are summed over the ranks (gloo or NCCL) and fitted (cudasw4_b200.fit_score_statistics), so
    every rank returns the same lambda and K, bit for bit, as one handle over the whole database would."""
    from . import fit_score_statistics

    counts, lensums = sw4.lastScoreHistogram(query_index)
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        both = torch.from_numpy(np.concatenate([counts, lensums])).to(device or torch.device("cpu"))
        dist.all_reduce(both, op=dist.ReduceOp.SUM, group=group)
        both = both.cpu().numpy()
        counts, lensums = both[:len(counts)], both[len(counts):]
    return fit_score_statistics(counts, lensums, query_length)


def shard_of(global_id: int, world: int, block: int = 256) -> int:
    """Which shard scans subject `global_id` (interleaved blocks of 256 consecutive subjects of the sorted database,
    cudasw4_b200/csrc/engine.cu: assignShards)."""
    return (global_id // block) % world
