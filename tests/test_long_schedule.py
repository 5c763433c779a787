"""CPU check of the CTA-wide array kernels' schedule (cudasw4_b200/csrc/kernels_s16_long.cuh, kernels_s32_long.cuh).

The kernels have no spin waits: every cross-warp hand-over relies on the CTA barrier taken every kLongBatch steps. This
test replays the schedule arithmetic (who writes / reads which FIFO slot, border row and ring slot at which step) for
every array width the engine can pick and checks that each read is separated from its write by a barrier, and that no
slot is overwritten before its last reader is past a barrier. Constants are parsed from the kernel header, the shape
rule (W, P, S from the query length) is restated from engine.cu / s16_long_ring_slots."""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _constants():
    src = open(os.path.join(ROOT, "cudasw4_b200", "csrc", "kernels_s16_long.cuh")).read()
    get = lambda name: int(re.search(r"constexpr int %s = (\d+);" % name, src).group(1))
    return {k: get(k) for k in ("kLongLag", "kLongFifoRows", "kLongBatch", "kLongMaxWarps")}


def _shape(q, c):
    """engine.cu: P = round_up(q + 32, 16); W = largest power of two <= kLongMaxWarps with kLongLag * W + 64 <= P."""
    P = (q + 32 + 15) // 16 * 16
    W = c["kLongMaxWarps"]
    while W > 1 and c["kLongLag"] * W + 64 > P:
        W //= 2
    S = (c["kLongLag"] * W + 16 + 31) // 32 * 32
    return W, P, S


def _barrier_between(t_write, t_read, batch):
    """A barrier is taken before every step that is a multiple of `batch`: is there one with t_write < b <= t_read?"""
    b = (t_write // batch + 1) * batch
    return b <= t_read


@pytest.mark.parametrize("q", [128, 129, 143, 144, 160, 255, 333, 415, 416, 567, 767, 768, 800, 1000, 5478, 35000])
def test_hand_over_and_ring_are_barrier_separated(q):
    c = _constants()
    lag, fifo, batch = c["kLongLag"], c["kLongFifoRows"], c["kLongBatch"]
    W, P, S = _shape(q, c)
    assert W >= 2 and P % batch == 0 and P >= q + 32 and P >= lag * W + 64 and S >= lag * W + 16 and S % 32 == 0
    assert lag == 32 + batch, "a warp trails its predecessor by its 32 lanes plus one batch"
    rows = sorted(set(list(range(0, min(q, 200))) + list(range(max(0, q - 200), q))))
    for w in range(1, W):  # shared-memory FIFO between warp w-1 (lane 31 writes) and warp w (lane 0 reads)
        for r in rows:
            t_w = r + lag * (w - 1) + 31
            t_r = r + lag * w
            assert _barrier_between(t_w, t_r, batch), (w, r)
            # the slot's next writer: row r + fifo of this period, or the first row of the next period with the same slot
            nxt = [t_w + fifo] if r + fifo < q else []
            r2 = r % fifo
            nxt.append(P + r2 + lag * (w - 1) + 31)
            assert all(_barrier_between(t_r, t, batch) for t in nxt), (w, r)
    for r in rows:  # global border: warp W-1 (period k) -> cp.async prefetch one batch ahead -> warp 0 (period k+1)
        t_w = r + lag * (W - 1) + 31
        t_use = P + r
        t_issue = t_use // batch * batch - batch          # issued at the start of the previous batch ...
        t_done = t_issue + batch                          # ... and waited for at the next barrier
        assert _barrier_between(t_w, t_issue, batch) and t_done <= t_use, r
        # the FIFO slot the prefetch lands in was last read for row r - fifo, or for the previous period's last row with
        # the same slot; the copy is issued right after a barrier, so "read before t_issue" is enough
        prev_reads = [P + r - fifo] if r >= fifo else [rho for rho in range(r % fifo, q, fifo)][-1:]
        assert all(t < t_issue for t in prev_reads), r
    # ring: slot (tau mod S) is filled during the batch before tau's batch (issued right after a barrier, waited for at
    # the next one), read by the lanes until tau + lag (W - 1) + 31, and refilled for tau + S one ring turn later
    last_skew = lag * (W - 1) + 31
    for tau in range(0, 3 * S):
        t_fill_issue = tau // batch * batch - batch
        assert t_fill_issue + batch <= tau
        t_refill_issue = (tau + S) // batch * batch - batch
        assert tau + last_skew < t_refill_issue, (tau, S, W)
    # descriptor table: written by warp 0 at k P, read by warp w at k P + lag w, rewritten at (k + 2) P
    for w in range(1, W):
        assert _barrier_between(0, lag * w, batch) and 2 * P > lag * w + batch


def _constants2():
    src = open(os.path.join(ROOT, "cudasw4_b200", "csrc", "kernels_s16_long2.cuh")).read()
    get = lambda name: int(re.search(r"constexpr int %s = (\d+);" % name, src).group(1))
    c = {k: get(k) for k in ("kLag2", "kFifo2", "kLong2Warps", "kLong2MaxW")}
    c["ring"] = lambda W: (2 * c["kLag2"] * W + 16 + 31) // 32 * 32   # s16_long2_ring_slots (query rows)
    return c


def _shape2(q, c):
    """s16_long2_warps: P (steps) = round_up(ceil(q/2) + 32, 16); W = largest power of two <= kLong2MaxW with
    kLag2 * W + 16 <= P."""
    P = ((q + 1) // 2 + 32 + 15) // 16 * 16
    W = c["kLong2MaxW"]
    while W > 1 and c["kLag2"] * W + 16 > P:
        W //= 2
    return W, P


def _long2_queries():
    """Query lengths on both sides of every W transition of the two-row array, and up to 35,000."""
    c = _constants2()
    qs, prev = {300, 1000, 5478, 20001, 35000}, None
    for q in range(1, 2000):
        W = _shape2(q, c)[0]
        if prev is not None and W != prev and prev >= 2:
            qs.update((q - 1, q, q + 1))
        prev = W
    return sorted(q for q in qs if _shape2(q, c)[0] >= 2)


@pytest.mark.parametrize("q", _long2_queries())
def test_long2_hand_over_and_ring_are_barrier_separated(q):
    """kernels_s16_long2.cuh: every lane takes two query rows per step; warp w of an array trails warp w-1 by kLag2
    steps and lane l of a warp trails lane l-1 by one step, so lane l of warp w is at step (t - kLag2 w - l) mod P at
    time t. CTA barriers come before every step t that is a multiple of 8. The 16 / W arrays of a CTA run in phase on
    one ring with their own FIFOs, descriptors and border rows."""
    c = _constants2()
    lag, fifo, batch = c["kLag2"], c["kFifo2"], 8
    W, P = _shape2(q, c)
    S = c["ring"](W)
    q_steps = (q + 1) // 2
    assert W in (2, 4, 8) and P % 16 == 0 and P >= q_steps + 32 and P >= lag * W + 16 and S >= 2 * lag * W + 16 and S % 32 == 0
    assert lag == 32 + batch, "a warp trails its predecessor by its 32 lanes plus one batch"
    assert fifo & (fifo - 1) == 0 and fifo >= batch, "FIFO entries are addressed with & (kFifo2 - 1) in whole batches"
    assert c["kLong2Warps"] % W == 0 and c["kLong2MaxW"] <= c["kLong2Warps"]
    steps = sorted(set(range(min(P, 160))) | set(range(max(0, P - 160), P)))

    def write_time(w, p, k=0):   # lane 31 of warp w writes its right border of step p (every step of a period)
        return k * P + p + lag * w + 31

    for w in range(1, W):
        for p in steps:
            if p >= q_steps:
                continue                   # lane 0 takes the boundary column at gap steps: the entry is not read
            t_w, t_r = write_time(w - 1, p), p + lag * w
            assert _barrier_between(t_w, t_r, batch), (W, w, p)
            # the entry (p mod fifo) is rewritten for step p + fifo, or in the next period for the first step with that
            # entry; whichever comes first must follow the read by a barrier
            nxt = [write_time(w - 1, p2, 1) for p2 in range(p % fifo, P, fifo)][:1]
            if p + fifo < P:
                nxt.append(write_time(w - 1, p + fifo))
            assert all(_barrier_between(t_r, t, batch) for t in nxt), (W, w, p)
    for p in steps:
        # global border: warp W-1 of period k writes entry p; warp 0's lanes 0..7 fetch entries e..e+7 with cp.async at
        # the barrier one batch before lane 0 of warp 0 uses them (period k+1), and wait for them at the next barrier
        if p >= q_steps:
            continue
        t_use = P + p
        t_issue = t_use // batch * batch - batch
        assert _barrier_between(write_time(W - 1, p), t_issue, batch) and t_issue + batch <= t_use, (W, p)
        assert write_time(W - 1, p, 1) > t_issue + batch   # the next period's rewrite comes after the copy landed
        # the FIFO entry the copy lands in was last read for step p - fifo (same period) or for the previous period's
        # last real step with the same entry: both before the barrier the copy is issued after
        prev = [P + p - fifo] if p >= fifo else [rho for rho in range(p % fifo, q_steps, fifo)][-1:]
        assert all(t < t_issue for t in prev), (W, p)
    # ring: S query rows = S / 2 steps; the rows of time tau are filled in the batch before tau's batch, read by the lanes
    # until tau + lag (W - 1) + 31, and refilled for tau + S / 2 one ring turn later
    last_skew = lag * (W - 1) + 31
    for tau in range(0, 3 * S):
        t_fill_issue = tau // batch * batch - batch
        assert t_fill_issue + batch <= tau
        t_refill_issue = (tau + S // 2) // batch * batch - batch
        assert tau + last_skew < t_refill_issue, (tau, S, W)
    # a batch reads 16 consecutive ring rows from a lane's slot at the batch start; the 16-row mirror behind the ring's
    # end covers the wrap (S is a multiple of 16, so the slot at a batch start is even and at most S - 2)
    assert S % 16 == 0 and (S - 2) + 15 < S + 16
    # descriptors: written by warp 0 at the restart at k P, read by warp w at k P + lag w, rewritten at (k + 2) P
    for w in range(1, W):
        assert _barrier_between(0, lag * w, batch) and lag * w < 2 * P - batch
    # per-CTA resources of the 16 / W arrays: FIFO inputs by warp index in the CTA (the last warp of an array writes the
    # global border, never the next array's first FIFO), descriptor tables of 2 W entries, one border row array each
    arrays = c["kLong2Warps"] // W
    desc = [(a * 2 * W, a * 2 * W + 2 * W) for a in range(arrays)]
    assert desc[-1][1] <= 2 * c["kLong2Warps"] and all(desc[i][1] <= desc[i + 1][0] for i in range(arrays - 1))
    fifo_out = {a * W + w + 1 for a in range(arrays) for w in range(W - 1)}
    assert fifo_out.isdisjoint({a * W for a in range(arrays)}) and max(fifo_out) < c["kLong2Warps"]


def test_long2_kernel_text_matches_the_replay():
    """The expressions the long2 replay above restates."""
    src = open(os.path.join(ROOT, "cudasw4_b200", "csrc", "kernels_s16_long2.cuh")).read()
    for expr in (
        "const int skew = kLag2 * w + lane;",
        "int p = skew == 0 ? 0 : P - skew;",
        "int xs = skew == 0 ? 0 : S - 2 * skew;",
        "const int pRestart = lane == 0 ? 0 : P - lane;",
        "if (e + lane < qSteps) cp_async16(fifoIn + ((e + lane) & (kFifo2 - 1)) * 16, border + e + lane);",
        "const uint32_t inBase = fifoIn + (p0 & (kFifo2 - 8)) * 16;",
        "const uint32_t outA = fifoOut + (p31 & (kFifo2 - 1)) * 16, out7 = fifoOut + (e7 & (kFifo2 - 1)) * 16;",
        "if (lastWarp) *(i < 7 ? bA + i : b7) = make_uint4(HlastA, ElastA, Hp[R - 1], ElastB);",
        "if (take && i < nReal) {",
        "static_for<8>(",
        "volatile int4* slot = desc + (periodIndex & 1) * W + i;",
        "+ arr * 2 * W;",
        "uint4* border = prm.border + (size_t)(blockIdx.x * (kLong2Warps / W) + arr) * prm.borderStride;",
        "static inline int s16_long2_ring_slots(int warps) { return (2 * kLag2 * warps + 16 + 31) / 32 * 32; }",
        "const int p0 = ((qlen + 1) / 2 + 32 + 15) / 16 * 16;",
        "while (w > 1 && kLag2 * w + 16 > p0) w >>= 1;",
    ):
        assert expr in src, expr


def test_engine_and_kernel_agree_on_the_shape_rule():
    eng = open(os.path.join(ROOT, "cudasw4_b200", "csrc", "engine.cu")).read()
    assert "(qlen + 32 + 15) / 16 * 16" in eng and "kLongLag * longWarps + 64 > p0" in eng
    hdr = open(os.path.join(ROOT, "cudasw4_b200", "csrc", "kernels_s16_long.cuh")).read()
    assert "(kLongLag * warps + 16 + 31) / 32 * 32" in hdr
