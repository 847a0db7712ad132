"""Which access path, head outcome and compiled form the chunk-step kernels take — TEST INFRASTRUCTURE, no tests.

``abr_step_kernel`` and ``abr_rollout_kernel`` (abr_step.cu) find the segment a download ends in through a per-trace
bucket index, staged in shared memory or read from global memory, with a branch-free ``head_fast`` and a general
``head_any`` behind it; the fused episode guesses the next step's head ahead of time.  None of that changes a result,
so a bit-exact comparison alone cannot show which of those paths a test went through.  This module restates, in
numpy and from the source:

* ``trace_tables``: the tables of ``abr_trace_table_kernel`` (C, M, scale, the index rows), ``cell_of`` bit for bit;
* ``head_outcome``: what the head of a step does, from the pre-step state the oracle exposes and the chunk size;
* ``speculation``: what became of the fused episode's guess of each next head (FIXED / RANDOM run-ahead loop);
* ``step_form`` / ``step_grid`` / ``step_paths``: ``launch_step``'s form and output type, persistent grid,
  shared-memory buffer and per-tile staging;
  ``rollout_form`` / ``rollout_paths``: ``launch_rollout_form`` (with ``uniform_util`` and the output type) and the
  fused block's ``use_smem``;
* ``reset_fmod`` / ``advance_fmod`` / ``pow2_inverse_exact``: the ``fmod`` branches of ``reset_seg_phase`` /
  ``advance_trace`` and ``pow2_inverse``;
* ``stats_fused`` / ``stats_stage1``: the two reduction trees of SPEC §6, bit for bit;
* ``STEP_CASES`` and ``reachable_cells``: the cases of ``test_gpu_step_forms.py`` and the cells they must reach
  (``reachable_cells`` lists the few it leaves out, and why).

``test_step_forms_ledger.py`` checks, on the CPU, that the sources still contain what this restatement relies on and
that the cases reach every reachable cell.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

# constants of abr_step.cu / abr_common.cuh (the ledger checks them against the sources)
K_TILE = 128
K_STEP_TILES = 8
K_TILE_BLOCKS_PER_SM = 7
K_PREFETCH_MIN_BYTES = 192 << 20
K_PF_DIST = 2                      # ABR_STEP_PF_DIST
K_ROLLOUT_BLOCK = 64
K_SMEM_OPT_IN_LIMIT = 200 * 1024
K_IDX_MAX_T = 65535
K_STATS_GROUP = 32
K_STATS_BLOCK = 256
K_STATS_SESSIONS_PER_BLOCK = 1024
K_WRAP_GUARD = 1 << 20
B200_SMS = 148
NUM_ACC = 11
ROUND = 6755399441055744.0         # 1.5 * 2^52: cell_of's rounding constant

FIXED, RANDOM, BBA, RATE, BOLA = 0, 1, 2, 3, 4   # abr_b200.h ABR_POLICY_*


def cum_stride(T_max):
    return (T_max + 8 + 3) & ~3


def idx_cells(T):
    return 2 * T if T <= K_IDX_MAX_T else 0


def idx_stride(T_max):
    return (2 * T_max + 2 + 7) & ~7 if T_max <= K_IDX_MAX_T else 0


def cum_smem_doubles(T_max):
    return cum_stride(T_max) + 2


def cell_of(x, scale, M):
    """min(low word of x * scale + 1.5 * 2^52, M - 1): two separately rounded fp64 operations, as the kernel's
    dmul / dadd."""
    y = np.asarray(x, np.float64) * np.float64(scale) + np.float64(ROUND)
    lo = (np.atleast_1d(y).view(np.uint64) & np.uint64(0xffffffff)).astype(np.int64)
    return np.minimum(lo, M - 1)


# ---------------------------------------------------------------------------------------------------------------------
# trace tables (abr_trace_table_kernel)
# ---------------------------------------------------------------------------------------------------------------------
@dataclass
class Tables:
    C: np.ndarray       # [n_traces][cum_stride]: C[0..T], +inf behind
    P: np.ndarray       # [n_traces] C[T]
    scale: np.ndarray   # [n_traces]
    T: np.ndarray       # [n_traces]
    M: np.ndarray       # [n_traces] index cells, 0 = no index
    I: np.ndarray       # [n_traces]
    ok: np.ndarray      # [n_traces]
    idx: list           # [n_traces] the index row idx[0..M] (int64), None when M == 0
    T_max: int


def trace_tables(bw, tl, ti, payload, T_max=None):
    bw = np.asarray(bw, np.float64)
    n_tr = bw.shape[0]
    T_max = bw.shape[1] if T_max is None else T_max
    cs = cum_stride(T_max)
    C = np.full((n_tr, cs), np.inf)
    P, scale, Ms, oks, idx = np.zeros(n_tr), np.zeros(n_tr), np.zeros(n_tr, np.int64), np.zeros(n_tr, bool), []
    for t in range(n_tr):
        T, I = int(tl[t]), float(ti[t])
        c = np.add.accumulate((bw[t, :T] * payload) * I)       # left to right, one rounding per addition
        C[t, 0] = 0.0
        C[t, 1:T + 1] = c
        mincap = np.min(C[t, 1:T + 1] - C[t, :T])
        P[t] = c[-1]
        ok = bool(c[-1] > 0.0 and c[-1] < np.inf and mincap > 0.0)
        M = idx_cells(T) if idx_stride(T_max) > 0 else 0
        s = 0.0
        if M > 0 and ok:
            with np.errstate(over="ignore", divide="ignore"):
                s = float(np.float64(M) / np.float64(c[-1]))
            if not (s > 0.0 and s < np.inf):
                M = 0
        else:
            M = 0
        scale[t], Ms[t], oks[t] = s, M, ok
        if M > 0:
            cells = cell_of(C[t, 1:T], s, M)                  # interior boundaries C[1..T-1], non-decreasing
            idx.append(np.searchsorted(cells, np.arange(M + 1), side="left").astype(np.int64))
        else:
            idx.append(None)
    return Tables(C, P, scale, np.asarray(tl, np.int64), Ms, np.asarray(ti, np.float64), oks, idx, T_max)


# ---------------------------------------------------------------------------------------------------------------------
# head of a step
# ---------------------------------------------------------------------------------------------------------------------
# "fast": head_fast settled it (staged: <= 3 candidates and <= 1 wrap; global: the eight-entry window);
# head_any: "guard" (the 2^20-period safety net), "noidx_linear" / "noidx_bisect" (M = 0, T <= 9 / T >= 10),
# "wraps" (>= 2 whole periods), "bisect" (> 8 candidates in the cell), "cands" (candidates past the fast window)
OUTCOMES = ("fast", "cands", "bisect", "wraps", "noidx_linear", "noidx_bisect", "guard")


def fast_ok(tab, tr, raw, smem):
    """head_fast's success for sessions on traces tr (all with M > 0) and download ends raw; smem: staged variant."""
    tr = np.asarray(tr, np.int64)
    raw = np.asarray(raw, np.float64)
    smem = np.broadcast_to(np.asarray(smem, bool), raw.shape)
    P = tab.P[tr]
    w = raw >= P
    t = np.where(w, raw - P, raw)
    ok = np.zeros(raw.shape, bool)
    for k in np.unique(tr):
        m = tr == k
        b = cell_of(t[m], tab.scale[k], int(tab.M[k]))
        j0 = tab.idx[k][b]
        C = tab.C[k]
        tk = t[m]
        # staged: C[j0+1..j0+3] <= t counted, then t < C[j+1]
        j = j0 + (C[j0 + 1] <= tk) + (C[j0 + 2] <= tk) + (C[j0 + 3] <= tk)
        ok_s = tk < C[j + 1]
        # global: the aligned window C[q0 .. q0+7], 1 <= count <= 7
        q0 = j0 & ~3
        n_le = sum((C[q0 + i] <= tk).astype(np.int64) for i in range(8))
        ok_g = (n_le >= 1) & (n_le <= 7)
        ok[m] = np.where(smem[m], ok_s, ok_g) & (tk < P[m])
    return ok


def head_outcome(tab, tr, raw, smem):
    """OUTCOMES entry of every session's head (arrays over sessions)."""
    tr = np.asarray(tr, np.int64)
    raw = np.asarray(raw, np.float64)
    smem = np.broadcast_to(np.asarray(smem, bool), raw.shape)
    P, M, T = tab.P[tr], tab.M[tr], tab.T[tr]
    periods = raw / P
    assert not np.any(np.abs(periods - K_WRAP_GUARD) < 0.01 * K_WRAP_GUARD), "too close to the safety net to classify"
    out = np.full(raw.shape, "", dtype=object)
    out[periods > K_WRAP_GUARD] = "guard"
    noidx = (out == "") & (M == 0)
    out[noidx & (T - 1 <= 8)] = "noidx_linear"
    out[noidx & (T - 1 > 8)] = "noidx_bisect"
    rest = np.flatnonzero(out == "")
    if rest.size:
        ok = fast_ok(tab, tr[rest], raw[rest], smem[rest])
        out[rest[ok]] = "fast"
        rest = rest[~ok]
    for s in rest:
        target = raw[s] - P[s] if raw[s] >= P[s] else raw[s]
        if target >= P[s]:
            out[s] = "wraps"
            continue
        k = tr[s]
        b = int(cell_of(target, tab.scale[k], int(tab.M[k]))[0])
        out[s] = "bisect" if tab.idx[k][b + 1] - tab.idx[k][b] > 8 else "cands"
    return out


# ---------------------------------------------------------------------------------------------------------------------
# run-ahead speculation of the fused episode (FIXED / RANDOM, not live)
# ---------------------------------------------------------------------------------------------------------------------
SPECULATION = ("used", "slept", "missed", "warp_slept", "no_index")


def speculation(tab, tr, smem, pos_after, size_next, slept):
    """[steps - 1][N] SPECULATION entry of the guess made in iteration t (the head of step t + 1), t < steps - 1.

    pos_after[t]: the position after step t (the target of its head when it did not sleep); size_next[t]: the chunk
    size of step t + 1; slept[t]: step t slept (moved the position).  calm is warp-uniform: the lanes of a warp are 32
    consecutive sessions of a 64-session block (the last warp only has its valid sessions)."""
    steps1, N = np.asarray(pos_after).shape
    tr = np.asarray(tr, np.int64)
    smem = np.asarray(smem, bool)
    can = smem | (tab.M[tr] > 0)
    out = np.full((steps1, N), "", dtype=object)
    warp = np.arange(N) // 32
    for t in range(steps1):
        if t == 0:
            calm = np.ones(N, bool)
        else:
            any_moved = np.zeros(warp[-1] + 1, bool)
            np.logical_or.at(any_moved, warp, slept[t - 1])
            calm = ~any_moved[warp]
        o = out[t]
        o[~can] = "no_index"
        o[can & ~calm] = "warp_slept"
        o[can & calm & slept[t]] = "slept"
        rest = np.flatnonzero(can & calm & ~slept[t])
        if rest.size:
            ok = np.zeros(rest.size, bool)
            with_idx = tab.M[tr[rest]] > 0
            r = rest[with_idx]
            ok[with_idx] = fast_ok(tab, tr[r], pos_after[t][r] + size_next[t][r], smem[r])
            o[rest[ok]] = "used"
            o[rest[~ok]] = "missed"
    return out


# ---------------------------------------------------------------------------------------------------------------------
# dispatch
# ---------------------------------------------------------------------------------------------------------------------
def step_form(live=0, track_history=0, track_acc=0, auto_reset=1, has_core=True, policy=False, ot="f64"):
    """launch_step's kernel abr_step_kernel<FAST, LIVE, POL, OT> as (form, OT): form "POL" (step_policy, double
    outputs only), "LIVE", "FAST" or "GEN"; OT "f64" or "f32" (the fp32-output mode)."""
    if policy:
        assert ot == "f64"
        return ("POL", ot)
    if live:
        return ("LIVE", ot)
    return ("FAST" if has_core and not track_history and not track_acc and auto_reset else "GEN", ot)


def step_grid(n, sms=B200_SMS):
    """(tiles_per_block, grid) of launch_step's persistent grid."""
    total = (n + K_TILE - 1) // K_TILE
    tpb = max((total + sms * K_TILE_BLOCKS_PER_SM - 1) // (sms * K_TILE_BLOCKS_PER_SM), K_STEP_TILES)
    return tpb, (total + tpb - 1) // tpb


def step_smem_doubles(T_max):
    sd = cum_smem_doubles(T_max)
    nbytes = sd * 8 + idx_stride(T_max) * 2
    return 0 if nbytes > K_SMEM_OPT_IN_LIMIT or idx_stride(T_max) == 0 else sd


def step_prefetch(n, sms=B200_SMS):
    """The L2 bulk prefetch runs: the batch streams from HBM and a block has a tile K_PF_DIST ahead."""
    tpb, _ = step_grid(n, sms)
    return n * 121 >= K_PREFETCH_MIN_BYTES and tpb > K_PF_DIST


@dataclass
class StepPaths:
    smem: np.ndarray                      # [N] the session's head reads the staged rows
    restages: np.ndarray                  # [grid] stagings per block (parity of the k-th: k mod 2)
    straddle: int = 0                     # sessions of a mixed tile on the staged trace (shared-memory path)
    mixed_tiles: int = 0                  # tiles whose first and last session differ in trace
    mixed_per_block: np.ndarray = None    # [grid]
    partial_last_tile: bool = False
    partial_last_block: bool = False


def step_paths(trace_id, T_max, sms=B200_SMS):
    """The per-tile staging of abr_step_kernel for the sessions' traces (environment order)."""
    tid = np.asarray(trace_id, np.int64)
    n = tid.size
    tpb, grid = step_grid(n, sms)
    smem = np.zeros(n, bool)
    restages = np.zeros(grid, np.int64)
    mixed = np.zeros(grid, np.int64)
    straddle = 0
    staging = step_smem_doubles(T_max) != 0
    for blk in range(grid):
        staged = -1
        for k in range(tpb):
            t0 = (blk * tpb + k) * K_TILE
            if t0 >= n:
                break
            t1 = min(t0 + K_TILE, n)
            first, last = tid[t0], tid[t1 - 1]
            mixed[blk] += first != last
            if not staging:
                continue
            if first == last and first != staged:
                staged = first
                restages[blk] += 1
            on = tid[t0:t1] == staged
            smem[t0:t1] = on
            if first != last:
                straddle += int(on.sum())
    total = (n + K_TILE - 1) // K_TILE
    return StepPaths(smem, restages, straddle, int(mixed.sum()), mixed, n % K_TILE != 0, total % tpb != 0)


def rollout_form(policy, live=0, track_history=0, auto_reset=1, has_core=True, actions=False, none=False,
                 uniform_util=True, ot="f64"):
    """(POLICY, FAST, NOOUT, LIVE, UNI, OT) of launch_rollout_form, or None for a call it rejects.  NOOUT stores no
    output, so an fp32 call runs its double instantiation."""
    ahead = policy in (FIXED, RANDOM)
    if live:
        return (policy, False, False, True, False, ot)
    plain = not track_history and auto_reset
    fast = plain and has_core and not actions
    none = plain and none
    if policy == RATE:
        return None if (fast or none) else (policy, False, False, False, False, ot)
    uni = bool(uniform_util)
    if fast:
        return (policy, True, False, False, ahead and uni, ot)
    if none:
        return (policy, True, True, False, ahead and uni, "f64")
    return (policy, False, False, False, False, ot)


def rollout_smem_bytes(T_max, V, A):
    sd = cum_smem_doubles(T_max)
    nbytes = (sd + 2 * V * A) * 8 + idx_stride(T_max) * 2
    return 0 if nbytes > K_SMEM_OPT_IN_LIMIT or idx_stride(T_max) == 0 else nbytes


def rollout_paths(tab, trace_id, V, A):
    """[N] use_smem of each session's 64-session block."""
    tid = np.asarray(trace_id, np.int64)
    n = tid.size
    out = np.zeros(n, bool)
    if rollout_smem_bytes(tab.T_max, V, A) == 0:
        return out
    for b0 in range(0, n, K_ROLLOUT_BLOCK):
        blk = tid[b0:b0 + K_ROLLOUT_BLOCK]
        out[b0:b0 + K_ROLLOUT_BLOCK] = bool(np.all(blk == blk[0]) and tab.M[blk[0]] > 0)
    return out


# ---------------------------------------------------------------------------------------------------------------------
# position edges
# ---------------------------------------------------------------------------------------------------------------------
def pow2_inverse_exact(d):
    """pow2_inverse(d) != 0: d is a power of two in [2^-500, 2^500]."""
    bits = int(np.float64(d).view(np.uint64))
    hi, lo = bits >> 32, bits & 0xffffffff
    e = (hi >> 20) & 0x7ff
    return lo == 0 and (hi & 0x800fffff) == 0 and 523 <= e <= 1523


def reset_fmod(off, I):
    """reset_seg_phase takes the fmod branch: floor(off / I) is not in [0, 2^31)."""
    n = np.floor(np.asarray(off, np.float64) / np.asarray(I, np.float64))
    return ~((n >= 0.0) & (n < 2147483648.0))


def advance_fmod(dt, I):
    """advance_trace takes the fmod branch (up to the phase carried in, < 1 segment): dt / I >= 2147480000."""
    return np.asarray(dt, np.float64) / np.asarray(I, np.float64) >= 2147480000.0


# ---------------------------------------------------------------------------------------------------------------------
# statistics (SPEC §6): the two reduction trees
# ---------------------------------------------------------------------------------------------------------------------
def _shfl_tree(x):
    """Lane 0 of the shuffle tree over the 32 columns x[..., 0:32] (x[l] += x[l + d], d = 16, 8, 4, 2, 1)."""
    x = x.copy()
    for d in (16, 8, 4, 2, 1):
        x[..., :d] = x[..., :d] + x[..., d:2 * d]
    return x[..., 0]


def _pad(acc, width):
    n = acc.shape[1]
    m = -(-max(n, 1) // width) * width
    out = np.zeros((acc.shape[0], m))
    out[:, :n] = acc
    return out


def _groups_and_final(partials):
    """stats_group_sum over every group, then stats_final_sum; partials [n_partials][NUM_ACC]."""
    n_p = partials.shape[0]
    n_groups = -(-n_p // K_STATS_GROUP)
    p = np.zeros((n_groups * K_STATS_GROUP, NUM_ACC))
    p[:n_p] = partials
    p = p.reshape(n_groups, 4, 8, NUM_ACC)
    s = p[:, :, 0]
    for k in range(1, 8):
        s = s + p[:, :, k]
    group = ((s[:, 0] + s[:, 1]) + s[:, 2]) + s[:, 3]                 # [n_groups][NUM_ACC]
    rounds = -(-n_groups // 32)
    g = np.zeros((rounds * 32, NUM_ACC))
    g[:n_groups] = group
    q = np.zeros((4, NUM_ACC))
    for r in range(rounds):
        for k in range(8):
            q = q + g[r * 32 + 4 * k: r * 32 + 4 * k + 4]          # thread q adds group r*32 + q + 4k
    return ((q[0] + q[1]) + q[2]) + q[3]


def stats_fused(acc):
    """env.stats() after a fused episode: 64-session block partials (two warp trees, then warp 0 + warp 1)."""
    a = _pad(np.asarray(acc, np.float64), K_ROLLOUT_BLOCK)
    blocks = a.reshape(NUM_ACC, -1, 2, 32)
    w = _shfl_tree(blocks)                                          # [NUM_ACC][blocks][2]
    partials = (w[..., 0] + w[..., 1]).T
    return _groups_and_final(partials)


def stats_stage1(acc):
    """env.stats() otherwise: abr_stats_stage1 over 1 024-session blocks (256 strided thread sums, then block_sum)."""
    a = _pad(np.asarray(acc, np.float64), K_STATS_SESSIONS_PER_BLOCK)
    blocks = a.reshape(NUM_ACC, -1, K_STATS_SESSIONS_PER_BLOCK // K_STATS_BLOCK, K_STATS_BLOCK)
    x = np.zeros(blocks.shape[:2] + (K_STATS_BLOCK,))
    for r in range(blocks.shape[2]):                                # thread t: sessions t, t + 256, ... in order
        x = x + blocks[:, :, r]
    warps = _shfl_tree(x.reshape(x.shape[:2] + (K_STATS_BLOCK // 32, 32)))   # [NUM_ACC][blocks][8]
    lane = np.zeros(warps.shape[:2] + (32,))
    lane[..., :K_STATS_BLOCK // 32] = warps
    partials = _shfl_tree(lane).T
    return _groups_and_final(partials)


# ---------------------------------------------------------------------------------------------------------------------
# worlds, layouts and the case table of test_gpu_step_forms.py
# ---------------------------------------------------------------------------------------------------------------------
LADDER = (300.0, 750.0, 1200.0, 1850.0, 2850.0, 4300.0)
SHORT_TRACES = (1, 5, 9, 10, 200, 2048)         # next to one long trace in the long-trace worlds


def make_world(name):
    """(bitrates, sizes, bw, trace_len, trace_interval) of a named world (deterministic)."""
    from abrsimulator_b200 import synth
    bitrates, sizes = synth.make_video(24, ladder=LADDER, seed=3)
    rng = np.random.default_rng(17)
    if name.startswith("long"):
        # one trace of T_max segments and the short ones; T_max > 65 535 leaves the whole environment without index
        T_max = int(name[4:])
        tl = np.array((T_max,) + SHORT_TRACES, np.int32)
        bw = synth.make_traces(len(tl), T_max, seed=5)[0]
        return bitrates, sizes, bw, tl, np.ones(len(tl))
    if name == "mixed":
        # 0: log-uniform 1e-3 .. 10 Mbit/s (cells with 4+ and 9+ boundaries), 1: one segment of 0.5 Mbit/s (downloads
        # wrap the period several times), 2: a plain trace, 3: a run of 60 near-empty segments (one cell holds all 60
        # boundaries), 4: five segments
        T = 300
        bw = np.zeros((5, T))
        bw[0] = np.exp(rng.uniform(np.log(1e-3), np.log(10.0), T))
        bw[1, 0] = 0.5
        bw[2] = synth.make_traces(1, T, seed=9)[0][0]
        bw[3, :260] = np.r_[np.full(100, 5.0), np.full(60, 1e-4), np.full(100, 5.0)]
        bw[4, :5] = (1.0, 3.0, 0.5, 2.0, 1.5)
        return bitrates, sizes, bw, np.array([T, 1, T, 260, 5], np.int32), np.array([1.0, 1.0, 0.5, 2.0, 1.0])
    if name == "mixedv":
        # the mixed world with a bitrate ladder scaled per chunk: the utility rows differ, uniform_util = 0
        bitrates, sizes, bw, tl, ti = make_world("mixed")
        return np.ascontiguousarray(bitrates * np.linspace(0.8, 1.2, len(bitrates))[:, None]), sizes, bw, tl, ti
    if name == "guard":
        # a period of 1.9e-7 Mbit: every download runs past 2^20 periods (the safety net); and a plain trace
        bw = np.zeros((2, 100))
        bw[0, :2] = 1e-7
        bw[1] = synth.make_traces(1, 100, seed=4)[0][0]
        return bitrates, sizes, bw, np.array([2, 100], np.int32), np.array([1.0, 1.0])
    if name == "edges":
        # segments of 2^-31 s and 1e-9 s at 1e9 Mbit/s (a sleep or a live wait of seconds crosses > 2^31 segments), a
        # plain trace of 1 s segments and one of 0.3 s
        bw = np.zeros((4, 100))
        bw[0, :50] = bw[1, :50] = 1e9
        bw[2] = synth.make_traces(1, 100, seed=6)[0][0]
        bw[3] = synth.make_traces(1, 100, seed=7)[0][0]
        return bitrates, sizes, bw, np.array([50, 50, 100, 100], np.int32), np.array([2.0 ** -31, 1e-9, 1.0, 0.3])
    if name == "bign":
        bw, tl, ti = synth.make_traces(16, 300, seed=8)
        return bitrates, sizes, bw, tl, ti
    raise KeyError(name)


def make_layout(case, tl, ti, sms=B200_SMS):
    """(trace_id, start_offset) of the case's sessions, in environment order.

    "grouped": runs of 128 sessions per trace (one tile of the per-step kernel, two blocks of the fused one), then
    three tiles of random traces, then a partial tile.  "bign": runs of two tiles per trace (a restage every other
    tile), in every full block one tile of random traces and one tile whose first 60 sessions are on the trace
    staged before it (they straddle onto it), and a partial last tile and block.  Offsets: uniform over 1.5 periods; the
    edges world adds offsets of >= 2^31 segments."""
    rng = np.random.default_rng(case.seed)
    N, n_tr = case.N, len(tl)
    if case.layout == "grouped":
        tid = (np.arange(N) // K_TILE) % n_tr
        lo = 2 * n_tr * K_TILE
        tid[lo:lo + 3 * K_TILE] = rng.integers(0, n_tr, 3 * K_TILE)
    else:
        tid = (np.arange(N) // (2 * K_TILE)) % n_tr
        tpb, grid = step_grid(N, sms)
        for b in range(grid):
            t5, t10 = (b * tpb + 5) * K_TILE, (b * tpb + 10) * K_TILE
            tid[t5:t5 + K_TILE] = rng.integers(0, n_tr, K_TILE)[:max(0, min(K_TILE, N - t5))]
            if t10 + K_TILE <= N:
                tid[t10:t10 + 60] = tid[t10 - 1]
    tid = tid.astype(np.int32)
    off = rng.uniform(0, 1.5, N) * (tl * ti)[tid]
    if case.world == "edges":
        big = rng.random(N) < 0.3
        off[big] = rng.uniform(2.2, 3.0, big.sum()) * 2.0 ** 31 * ti[tid[big]]
    return tid, off


@dataclass(frozen=True)
class StepCase:
    """One run of a chunk-step kernel against the oracle.  kernel: "step" (per-step calls with random actions),
    "policy" (abr_env_step_policy, greedy, on random logits), "fused" (one episode of `policy`), "run" / "run_host"
    (the fused reset + episode + cost + statistics of abr_env_run / abr_env_run_host), "lookahead" (per-step calls,
    then abr_env_lookahead_decide with horizon H).  params: environment parameters; want: the fused episode's outputs
    ("core" = the six of the FAST forms, "core+" = with the actions, "none"); dtype: "f64", or "f32" for the
    fp32-output mode; reaches: the cells the case claims, checked against its own data on the GPU."""
    name: str
    world: str
    kernel: str
    N: int
    steps: int
    reaches: frozenset
    policy: int = FIXED
    params: tuple = ()
    want: str = "core"
    layout: str = "grouped"
    H: int = 2
    seed: int = 1
    dtype: str = "f64"

    @property
    def kw(self):
        return dict(self.params)

    @property
    def uniform_util(self):
        return self.world != "mixedv"

    def form(self):
        p = self.kw
        live, th, ar = p.get("live", 0), p.get("track_history", 0), p.get("auto_reset", 1)
        if self.kernel in ("step", "lookahead"):
            return step_form(live, th, p.get("track_acc", 0), ar, ot=self.dtype)
        if self.kernel == "policy":
            return step_form(policy=True)
        if self.kernel == "run":          # the six outputs of the FAST forms
            return rollout_form(self.policy, live, th, ar, True, False, False, self.uniform_util)
        if self.kernel == "run_host":     # the reward trajectory only
            return rollout_form(self.policy, live, th, ar, False, False, False, self.uniform_util)
        return rollout_form(self.policy, live, th, ar, self.want.startswith("core"), self.want == "core+",
                            self.want == "none", self.uniform_util, self.dtype)

    def cost(self):
        """Oracle session-steps (the lookahead's tree: A^H leaves of H steps per session)."""
        base = self.N * self.steps * (2 if self.kernel in ("fused", "run", "run_host") else 1)
        return base + (self.N * len(LADDER) ** self.H * self.H if self.kernel == "lookahead" else 0)


def head(kernel, path, outcome):
    return ("head", kernel, path, outcome)


def spec(path, outcome):
    return ("spec", path, outcome)


def fused_form_cells(form, paths=("smem", "global")):
    return {("fused", form, p) for p in paths}


def step_form_cells(form, paths=("smem", "global")):
    return {("step", form, p) for p in paths}


def _fs(*cells):
    return frozenset(cells)


def _with(c, cells):
    return StepCase(**{**c.__dict__, "reaches": frozenset(cells)})


def _cases():
    cases = []
    GEN_STEP = (("track_acc", 1), ("track_history", 1), ("max_buffer", 20.0))
    CAP = (("max_buffer", 20.0),)
    LIVE = (("live", 1), ("start_up_length", 8.0))
    # long traces next to short ones: every kernel, at the last T_max with an index and at two without
    for T_max in (65535, 65536, 70000):
        w = f"long{T_max}"
        n = 7 * 2 * K_TILE + 3 * K_TILE + 37
        ix = T_max <= K_IDX_MAX_T
        heads = {"fast"} if ix else {"noidx_linear", "noidx_bisect"}
        c = StepCase(f"{w}-step", w, "step", n, 12, frozenset(), params=GEN_STEP)
        cases.append(_with(c, {head("step", "global", o) for o in heads} | step_form_cells(c.form(), ("global",))))
        for pol, want in ((FIXED, "core"), (RANDOM, "none"), (BBA, "core+"), (BOLA, "core")):
            c = StepCase(f"{w}-fused-p{pol}-{want}", w, "fused", n, 12, frozenset(), policy=pol, want=want, params=CAP)
            r = {head("fused", "global", o) for o in heads} | fused_form_cells(c.form(), ("global",))
            if pol in (FIXED, RANDOM) and not ix:
                r.add(spec("global", "no_index"))
            cases.append(_with(c, r))
        cases.append(StepCase(f"{w}-lookahead", w, "lookahead", n, 6,
                              _fs(*[head("lookahead", "global", o) for o in heads]), params=CAP))
    # the head outcomes and the speculation outcomes on both paths, every form of both kernels
    N = 5 * 2 * K_TILE + 3 * K_TILE + 37
    any_heads = ("fast", "cands", "bisect", "wraps")
    for tag, params in (("gen", GEN_STEP), ("fast", CAP)):
        for dtype in ("f64", "f32"):
            c = StepCase(f"mixed-step-{tag}-{dtype}", "mixed", "step", N, 30, frozenset(), params=params, dtype=dtype)
            cases.append(_with(c, {head("step", p, o) for p in ("smem", "global") for o in any_heads}
                               | step_form_cells(c.form())))
    c = StepCase("mixed-step-policy", "mixed", "policy", N, 30, frozenset(), params=CAP)
    cases.append(_with(c, {head("step", p, o) for p in ("smem", "global") for o in any_heads}
                       | step_form_cells(c.form())))
    cases.append(StepCase("mixed-lookahead", "mixed", "lookahead", N, 9,
                          _fs(*[head("lookahead", "global", o) for o in any_heads]), params=CAP, H=2))
    # one fused case per form: every policy, output set, output type and live mode, on the one-ladder world and on
    # the world whose utility rows differ per chunk (the run-ahead loop without the carried utility)
    seen = set()
    for world in ("mixed", "mixedv"):
        for pol in (FIXED, RANDOM, BBA, BOLA, RATE):
            base = CAP + ((("track_history", 1),) if pol == RATE else ())
            for want, live in (("core", 0), ("core+", 0), ("none", 0), ("core", 1)):
                for dtype in ("f64",) if want == "none" else ("f64", "f32"):
                    params = base + (LIVE if live else ())
                    c = StepCase(f"{world}-fused-p{pol}-{want}{'-live' if live else ''}-{dtype}", world, "fused", N,
                                 30, frozenset(), policy=pol, want=want, params=params, seed=2 + pol, dtype=dtype)
                    f = c.form()
                    if f is None or f in seen:
                        continue
                    seen.add(f)
                    r = fused_form_cells(f)
                    if not live:
                        r |= {head("fused", p, o) for p in ("smem", "global") for o in any_heads}
                    if pol in (FIXED, RANDOM) and not live:
                        r |= {spec(p, o) for p in ("smem", "global") for o in ("used", "slept", "missed", "warp_slept")}
                    cases.append(_with(c, r))
    # the fused reset of abr_env_run (six outputs) and abr_env_run_host (host buffers, the reward trajectory)
    for kernel in ("run", "run_host"):
        for pol in (FIXED, BBA):
            c = StepCase(f"mixed-{kernel}-p{pol}", "mixed", kernel, N, 30, frozenset(), policy=pol, params=CAP,
                         seed=9 + pol)
            cases.append(_with(c, {("reset", kernel, "smem"), ("reset", kernel, "global")} | fused_form_cells(c.form())))
    # the safety net of the whole-period loop
    ng = 2 * 2 * K_TILE + 3 * K_TILE + 37
    cases.append(StepCase("guard-step", "guard", "step", ng, 3,
                          _fs(head("step", "smem", "guard"), head("step", "global", "guard")), params=CAP))
    # one step: the fused episode counts a session once however many of its steps hit the safety net
    cases.append(StepCase("guard-fused", "guard", "fused", ng, 1,
                          _fs(head("fused", "smem", "guard"), head("fused", "global", "guard")), params=CAP))
    cases.append(StepCase("guard-lookahead", "guard", "lookahead", ng, 1, _fs(head("lookahead", "global", "guard")),
                          params=CAP, H=1))
    # positions past 2^31 segments, exact and inexact reciprocals
    ne = 4 * 2 * K_TILE + 3 * K_TILE + 37
    for q in (3.0, 4.0):
        cases.append(StepCase(f"edges-step-q{q:g}", "edges", "step", ne, 8,
                              _fs(("edge", "reset_fmod"), ("edge", "sleep_fmod"), ("edge", "I_pow2"),
                                  ("edge", "I_inexact"), ("edge", "q_pow2" if q == 4.0 else "q_inexact")),
                              params=(("max_buffer", 20.0), ("sleep_quantum", q))))
        cases.append(StepCase(f"edges-fused-q{q:g}", "edges", "fused", ne, 8,
                              _fs(("edge", "reset_fmod"), ("edge", "sleep_fmod")), policy=RANDOM,
                              params=(("max_buffer", 20.0), ("sleep_quantum", q))))
    for dtype in ("f64", "f32"):
        c = StepCase(f"edges-step-live-{dtype}", "edges", "step", ne, 8, frozenset(), params=LIVE, dtype=dtype)
        cases.append(_with(c, {("edge", "live_fmod")} | step_form_cells(c.form())))
    # the per-step kernel's persistent grid beyond one tile per block and SM, streaming from HBM
    c = StepCase("bign-step", "bign", "step", (1 << 21) + 77, 2, frozenset(), layout="bign")
    cases.append(_with(c, {("dispatch", d) for d in DISPATCH} | step_form_cells(c.form())
                       | {head("step", "smem", "fast"), head("step", "global", "fast")}))
    return cases


DISPATCH = ("prefetch", "tiles_per_block>kStepTiles", "partial_tile", "partial_block", "parity0", "parity1",
            "straddle", "mixed_tile_per_block")
STEP_CASES = _cases()


def reachable_cells():
    """Every cell a legal call can reach, except these (each covered otherwise or out of reach):

    * heads in live mode: the pause gate moves the position before the head, and the oracle only exposes the state
      before the gate; a live step runs the same head<SMEM> as the others, whose cells are listed;
    * ("head", "step", "smem", "noidx_*"): the per-step kernel stages a trace without looking at M, so a staged
      trace without index is possible, but only when 2T / P overflows (a period capacity below ~1e-305), where every
      chunk size of a real ladder runs past 2^20 periods and takes the safety net first;
    * the fused episode's RATE policy has no FAST / NOOUT form (launch_rollout_form rejects those calls)."""
    cells = set()
    for kernel in ("step", "fused", "lookahead"):
        for o in OUTCOMES:
            cells.add(head(kernel, "global", o))
            if kernel != "lookahead" and not o.startswith("noidx"):   # use_smem needs M > 0 (see above for step)
                cells.add(head(kernel, "smem", o))
    for o in SPECULATION:
        cells.add(spec("global", o))
        if o != "no_index":
            cells.add(spec("smem", o))
    for pol in (FIXED, RANDOM, BBA, RATE, BOLA):
        for live in (0, 1):
            for th in (0, 1):
                for has_core, actions, none in ((True, False, False), (True, True, False), (False, False, True)):
                    for uni in (True, False):
                        for ot in ("f64", "f32"):
                            f = rollout_form(pol, live, th, 1, has_core, actions, none, uni, ot)
                            if f is not None:
                                cells |= fused_form_cells(f)
    for f in ("FAST", "GEN", "LIVE"):
        for ot in ("f64", "f32"):
            cells |= step_form_cells((f, ot))
    cells |= step_form_cells(("POL", "f64"))
    cells |= {("reset", k, p) for k in ("run", "run_host") for p in ("smem", "global")}
    cells |= {("edge", e) for e in ("reset_fmod", "sleep_fmod", "live_fmod", "I_pow2", "I_inexact", "q_pow2",
                                    "q_inexact")}
    cells |= {("dispatch", d) for d in DISPATCH}
    return cells
