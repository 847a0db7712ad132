"""CPU-only: the clairvoyant lookahead of SPEC §4.4 on the C environment oracle against the pure-Python restatement
(both in tests/lookahead_oracle.py), known answers and full-horizon optimality."""
import itertools

import numpy as np
import pytest

from oracle import oracle as orc
from oracle import step_oracle as so
from helpers import bits_equal, small_world
import lookahead_oracle as lo
from lookahead_oracle import lookahead


def decide(env, H, want_seq=False):
    out = lo.decide(env, H, want_seq)
    assert out[-1] == 0                                   # no lookahead step hits the safety net
    return out[:-1]


# ---- the C restatement against the pure-Python one, on random mid-episode states ----
CASES = [   # (A, H, params)
    (3, 3, dict()),
    (3, 2, dict(auto_reset=0, smooth_prev_ladder=1)),
    (6, 2, dict(utility_mode=1, max_buffer=9.0)),
    (3, 3, dict(auto_reset=0, utility_mode=1, smooth_prev_ladder=1, max_buffer=9.0, default_quality=-1)),
    (4, 3, dict(max_buffer=10.0, track_history=1, default_quality=2)),
]


@pytest.mark.parametrize("A,H,params", CASES, ids=[f"A{a}-H{h}-{i}" for i, (a, h, _) in enumerate(CASES)])
def test_c_oracle_equals_python_restatement(A, H, params):
    V, N = 7, 12
    ladder = [300.0, 750.0, 1200.0, 1850.0, 2850.0, 4300.0][:A] if A <= 6 else None
    bitrates, sizes, bw, tl, ti = small_world(n_traces=5, T=40, V=V, ladder=ladder, ragged=True)
    P = dict(orc.DEFAULTS, **params)
    env = orc.OracleEnv(bw, tl, ti, sizes, bitrates, N, **P)
    rng = np.random.default_rng(A * 10 + H)
    tid = rng.integers(0, 5, size=N).astype(np.int32)
    off = rng.uniform(0, 100, size=N)
    env.reset(tid, off)
    util = orc.utility_table(bitrates, P["utility_mode"], P["utility_scale"])
    py = [so.Session(bw[tid[s], :tl[tid[s]]], ti[tid[s]], sizes.tolist(), util.tolist(), P, off[s]) for s in range(N)]
    seen = dict(short=0, done=0, sleep=0, states=0)
    for t in range(V + 3):
        act, val, seq = decide(env, H, want_seq=True)
        for s in range(N):
            a, v, r = lookahead(py[s], H)
            assert (act[s], seq[s].tolist()) == (a, r), (t, s)
            assert bits_equal(val[s], v) == 0, (t, s, val[s], v)
            seen["short"] += 0 < V - py[s].chunk < H and not py[s].done
            seen["done"] += py[s].done
        seen["states"] += N
        a = rng.integers(0, A, size=N).astype(np.int32)
        o = env.step(a)
        for s in range(N):
            py[s].step(int(a[s]))
        seen["sleep"] += int((o["sleep"] > 0).sum())
    assert env.errors() == 0
    assert seen["short"] > 0                              # sessions near the end of the video: h < H
    if not P["auto_reset"]:
        assert seen["done"] > 0
    if P["max_buffer"] < 60.0:
        assert seen["sleep"] > 0                          # the sleep cap is reached on these states


# ---- known answers ----
LADDER = np.array([300.0, 750.0, 1200.0, 1850.0, 2850.0, 4300.0])


def one_session_env(bw, interval, bitrates, V, **params):
    br = np.tile(np.asarray(bitrates, np.float64), (V, 1))
    env = orc.OracleEnv(np.asarray(bw, np.float64)[None, :], [len(bw)], [interval], br * 4.0, br, 1, **params)
    env.reset(np.zeros(1, np.int32))
    return env


def test_ample_bandwidth_picks_the_top_quality():
    env = one_session_env(np.full(16, 1e7), 1.0, LADDER, 10, default_quality=-1, rtt=0.0)
    for H in (1, 3, 5):
        act, val, seq = decide(env, H, want_seq=True)
        assert act[0] == 5 and seq[0].tolist() == [5] * H
        assert val[0] > 0.0


def test_greedy_top_quality_rebuffers_two_chunks_later():
    """Utilities 1 and 3.  The trace opens with one 10 ms segment of 17 000 kbit and then crawls at 100 kbps: the top
    quality now (12 000 kbit) is the best single step, but then the chunk after next no longer fits the fast segment
    and stalls for ~22 s; three low chunks (12 000 kbit) all fit."""
    bw = np.full(8000, 100.0)
    bw[0] = 1.7e6
    kw = dict(default_quality=-1, rtt=0.0, payload=1.0, smooth_penalty=0.0)
    env = one_session_env(bw, 0.01, [1000.0, 3000.0], 6, **kw)
    act1, val1 = decide(env, 1)
    act3, val3, seq3 = decide(env, 3, want_seq=True)
    assert act1[0] == 1
    assert act3[0] == 0 and seq3[0].tolist() == [0, 0, 0]
    # greedy: top now, then the cheapest continuation, stalls at k + 2 and not before
    reb = [env.step([q])["rebuf"][0] for q in (1, 0, 0)]
    assert reb[1] == 0.0 and reb[2] > 20.0


def test_flat_ladder_ties_keep_index_zero():
    env = one_session_env(np.full(16, 3000.0), 1.0, [1000.0] * 4, 10)
    env.step([2])
    act, val, seq = decide(env, 4, want_seq=True)
    assert act[0] == 0 and seq[0].tolist() == [0, 0, 0, 0]


def test_nothing_left_to_plan():
    env = one_session_env(np.full(16, 3000.0), 1.0, LADDER, 3, auto_reset=0)
    for q in (1, 2, 3):
        env.step([q])
    assert env.field("done")[0] == 1
    act, val, seq = decide(env, 5, want_seq=True)
    assert act[0] == 0 and seq[0].tolist() == [-1] * 5
    assert val[0] == 0.0 and not np.signbit(val[0])


# ---- with H = V from a reset the decisions reach the best fixed sequence ----
def test_full_horizon_lookahead_reaches_the_best_fixed_sequence():
    V, A = 5, 3
    bitrates, sizes, bw, tl, ti = small_world(n_traces=3, T=30, V=V, ladder=[400.0, 1500.0, 4000.0], ragged=True)
    P = dict(max_buffer=12.0)
    seqs = np.array(list(itertools.product(range(A), repeat=V)), np.int32)     # 243 sequences, C order
    M = len(seqs)
    for tr, off in ((0, 3.7), (1, 41.0), (2, 0.0)):
        fixed = orc.OracleEnv(bw, tl, ti, sizes, bitrates, M, **P)
        fixed.reset(np.full(M, tr, np.int32), np.full(M, off))
        J = fixed.rollout(orc.POLICY_FIXED, V, actions=np.ascontiguousarray(seqs.T))["acc"][0]
        env = orc.OracleEnv(bw, tl, ti, sizes, bitrates, 1, **P)
        env.reset([tr], [off])
        act, val, seq = decide(env, V, want_seq=True)
        best = int(np.argmax(J))                         # the first maximum
        assert bits_equal(val[0], J.max()) == 0 and seq[0].tolist() == seqs[best].tolist()
        total = 0.0
        for _ in range(V):
            a, _ = decide(env, V)
            total = total + env.step(a)["reward"][0]
        assert total >= J.max() - 1e-12 * abs(J.max()) and (J <= total + 1e-12 * abs(J.max())).all()
        assert abs(total - J.max()) <= 1e-12 * abs(J.max())
