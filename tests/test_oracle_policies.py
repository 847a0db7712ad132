"""CPU-only: the RATE and BOLA policies of SPEC §4.2 / §4.3 in the C restatement (tests/policy_oracle.c), the
pure-Python restatement, and the C-ABI's parameter handling (no GPU needed)."""
import ctypes
import math

import numpy as np
import pytest

import policy_oracle as po
from policy_oracle import bola_action, bola_table, rb_action

LADDER = [300.0, 750.0, 1200.0, 1850.0, 2850.0, 4300.0]


def decide(policy, sizes, chunk, buffer, ring, hist_len, done=None, default_quality=1, **pp):
    return po.policy_decide(policy, np.atleast_2d(sizes), np.atleast_1d(chunk), np.atleast_1d(buffer),
                            np.atleast_2d(ring), np.atleast_1d(hist_len), done=done, default_quality=default_quality,
                            **pp)


# ---- rate-based, known answers ----
def test_rb_empty_ring_takes_the_default_quality():
    sizes = np.array([LADDER])
    ring = np.zeros((1, 5))
    assert decide(po.POLICY_RATE, sizes, 0, 0.0, ring, 0, default_quality=3)[0] == 3
    assert decide(po.POLICY_RATE, sizes, 0, 0.0, ring, 0, default_quality=-1)[0] == 0
    assert rb_action(LADDER, [], 3, 4.0) == 3 and rb_action(LADDER, [], -1, 4.0) == 0


def test_rb_a_size_equal_to_the_budget_fits():
    # samples 2 and 2 (powers of two: every operation exact): hm = 2, budget = (1 * 2) * 4 = 8
    sizes = np.array([[1.0, 8.0, 8.0 + 2.0 ** -49, 16.0]])
    ring = np.array([[2.0, 2.0, 0.0, 0.0, 0.0]])
    assert decide(po.POLICY_RATE, sizes, 0, 0.0, ring, 2)[0] == 1
    assert rb_action(sizes[0], [2.0, 2.0], 1, 4.0) == 1
    # safety 0.5 halves the budget to 4: only quality 0 fits
    assert decide(po.POLICY_RATE, sizes, 0, 0.0, ring, 2, rb_safety=0.5)[0] == 0


def test_rb_non_monotone_row_gives_the_largest_fitting_index():
    sizes = np.array([[5.0, 1.0, 9.0, 3.0, 20.0]])   # budget 4: indices 1 and 3 fit
    ring = np.array([[1.0, 1.0, 1.0, 1.0, 1.0]])
    assert decide(po.POLICY_RATE, sizes, 0, 0.0, ring, 7)[0] == 3
    sizes = np.array([[5.0, 6.0, 9.0]])              # nothing fits: 0
    assert decide(po.POLICY_RATE, sizes, 0, 0.0, ring, 7)[0] == 0


def test_rb_reads_the_n_most_recent_samples_of_the_ring():
    # K = 3, hist_len = 5: the newest sample is at slot 4 mod 3 = 1, the window is slots 2, 0, 1
    ring = np.array([[4.0, 4.0, 4.0]])
    sizes = np.array([[1.0, 15.9, 16.0, 16.1]])
    assert decide(po.POLICY_RATE, sizes, 0, 0.0, ring, 5)[0] == 2
    ring = np.array([[1.0, 1.0, 1000.0]])             # hm of (1000, 1, 1) = 3 / 2.001 -> budget ~6
    assert decide(po.POLICY_RATE, sizes, 0, 0.0, ring, 5)[0] == 0


# ---- BOLA, known answers ----
def test_bola_low_buffer_picks_the_lowest_quality():
    # the lowest quality's score (min_buffer - buffer) / size[0] is positive exactly below min_buffer; on a ladder
    # with a wide range (here top / bottom = 14.3) it is also the largest score for a low buffer
    sizes = np.array([LADDER, LADDER])
    for b in (0.0, 2.0, 4.0):
        assert decide(po.POLICY_BOLA, sizes, 1, b, np.zeros((1, 5)), 0)[0] == 0
    v, vmax = bola_table(sizes)
    gp = vmax / (30.0 / 10.0 - 1.0)
    Vp = 10.0 / gp
    s0 = lambda b: (Vp * (v[1][0] + gp) - b) / sizes[1][0]
    assert s0(9.99) > 0.0 and s0(10.01) < 0.0


def test_bola_at_and_above_target_buffer():
    # the highest quality's score crosses 0 at the target: just below it the top quality still has a positive score
    sizes = np.array([LADDER])
    assert decide(po.POLICY_BOLA, sizes, 0, 29.0, np.zeros((1, 5)), 0)[0] == len(LADDER) - 1


def test_bola_equal_scores_give_the_first_index_and_a_flat_ladder_gives_0():
    # a flat ladder: every v = 0 -> v_max = 0 -> 0 whatever the buffer
    flat = np.array([[2.0, 2.0, 2.0]])
    for b in (0.0, 20.0, 100.0):
        assert decide(po.POLICY_BOLA, flat, 0, b, np.zeros((1, 5)), 0)[0] == 0
    # duplicate sizes in a rising ladder: qualities 1 and 2 have the same score; the first one wins
    sizes = np.array([[1.0, 4.0, 4.0, 16.0]])
    v, vmax = bola_table(sizes)
    gp = vmax / (30.0 / 10.0 - 1.0)
    Vp = 10.0 / gp
    score = lambda a, b: (Vp * (v[0][a] + gp) - b) / sizes[0][a]
    b = 12.0                        # scores -2, 2, 2, 1.125: qualities 1 and 2 tie for the largest
    assert score(1, b) == score(2, b) and score(1, b) > max(score(0, b), score(3, b))
    assert decide(po.POLICY_BOLA, sizes, 0, b, np.zeros((1, 5)), 0)[0] == 1
    assert bola_action(sizes[0], v[0], vmax, b) == 1


def test_bola_mid_buffer_worked_by_hand():
    # sizes 1, e, e^2 (v = 0, 1, 2 up to the last bit of log), min 10, target 30:
    # gp = 2 / (3 - 1) = 1, Vp = 10.  Scores at b = 15: (10*1 - 15)/1 = -5, (10*2 - 15)/e = 1.84, (10*3 - 15)/e^2 = 2.03
    # -> quality 2; at b = 19: -9, 0.37, 1.49 -> 2; at b = 22: -12, -0.74, 1.08 -> 2; at b = 27: ..., 0.41 -> 2;
    # at b = 12: -2, 2.94, 2.44 -> quality 1
    e = math.e
    sizes = np.array([[1.0, e, e * e]])
    # and at b = 9: 1, 4.05, 2.84 -> 1; at b = 5: 5, 5.52, 3.38 -> 1 (on this narrow ladder the lowest quality loses
    # to quality 1 even below min_buffer)
    expect = {12.0: 1, 15.0: 2, 19.0: 2, 22.0: 2, 27.0: 2, 9.0: 1, 5.0: 1}
    for b, q in expect.items():
        assert decide(po.POLICY_BOLA, sizes, 0, b, np.zeros((1, 5)), 0)[0] == q, b
        v, vmax = bola_table(sizes)
        assert bola_action(sizes[0], v[0], vmax, b) == q


def test_done_sessions_answer_0_for_rate_and_bola_and_bba_is_unchanged():
    sizes = np.array([LADDER, LADDER])
    ring = np.full((2, 5), 5000.0)
    chunk = np.array([2, 2], np.int32)                # chunk == V: past the last chunk
    done = np.array([1, 1], np.uint8)
    buf = np.array([40.0, 3.0])
    for pol in (po.POLICY_RATE, po.POLICY_BOLA):
        assert decide(pol, sizes, chunk, buf, ring, [5, 5], done=done).tolist() == [0, 0]
    assert decide(po.POLICY_BBA, sizes, chunk, buf, ring, [5, 5], done=done).tolist() == [len(LADDER) - 1, 0]


# ---- the C oracle against the Python restatement on random states ----
@pytest.mark.parametrize("seed", range(3))
def test_c_oracle_equals_python_restatement_on_random_states(seed):
    rng = np.random.default_rng(seed)
    N, V, A, K = 4000, 7, 6, 5
    sizes = np.sort(rng.uniform(50.0, 20000.0, size=(V, A)), axis=1)
    sizes[1] = rng.uniform(50.0, 20000.0, size=A)            # a non-monotone row
    sizes[2, 3] = sizes[2, 2]                                 # a duplicate size: equal BOLA scores
    sizes[3] = 1000.0                                         # a flat row
    sizes[4, 2] = 4096.0                                      # = the budget of a ring of 1024s at safety 1
    chunk = rng.integers(0, V, size=N).astype(np.int32)
    buffer = rng.uniform(0.0, 60.0, size=N)
    buffer[::17] = 10.0
    buffer[::19] = 0.0
    hist_len = rng.integers(0, 3 * K, size=N).astype(np.int32)
    ring = rng.uniform(100.0, 8000.0, size=(N, K))
    ring[::11] = 1024.0                                      # exact harmonic mean: a budget of exactly 4096
    dq = int(rng.integers(-1, A))
    safety = float(rng.choice([1.0, 0.8, 1.25]))
    lo, hi = float(rng.choice([5.0, 10.0])), float(rng.choice([20.0, 30.0, 60.0]))
    got_rb = po.policy_decide(po.POLICY_RATE, sizes, chunk, buffer, ring, hist_len, default_quality=dq,
                              chunk_length=4.0, rb_safety=safety)
    got_bola = po.policy_decide(po.POLICY_BOLA, sizes, chunk, buffer, ring, hist_len, default_quality=dq,
                                chunk_length=4.0, bola_min_buffer=lo, bola_target_buffer=hi)
    v, vmax = bola_table(sizes.tolist())
    for s in range(N):
        L = int(hist_len[s])
        n = min(L, K)
        hist = [float(ring[s, (L - n + j) % K]) for j in range(n)]
        row = sizes[chunk[s]].tolist()
        assert got_rb[s] == rb_action(row, hist, dq, 4.0, safety), s
        assert got_bola[s] == bola_action(row, v[chunk[s]], vmax, float(buffer[s]), lo, hi), s
    # the states cover every branch
    assert (hist_len == 0).any() and len(set(got_rb.tolist())) > 2 and len(set(got_bola.tolist())) > 2


# ---- parameters ----
def test_policy_params_defaults_in_the_c_abi_and_the_oracle():
    from abrsimulator_b200 import _lib
    lib = _lib.load()
    pp = _lib.AbrPolicyParams()
    lib.abr_policy_params_default(ctypes.byref(pp))
    assert (pp.rb_safety, pp.bola_min_buffer, pp.bola_target_buffer) == (1.0, 10.0, 30.0)
    assert ctypes.sizeof(_lib.AbrPolicyParams) == 3 * 8
    assert po.DEFAULTS == dict(rb_safety=1.0, bola_min_buffer=10.0, bola_target_buffer=30.0)
    assert (_lib.POLICY_RATE, _lib.POLICY_BOLA) == (3, 4)


BAD = [dict(rb_safety=0.0), dict(rb_safety=-1.0), dict(rb_safety=float("inf")), dict(rb_safety=float("nan")),
       dict(bola_min_buffer=0.0), dict(bola_min_buffer=30.0, bola_target_buffer=30.0),
       dict(bola_min_buffer=40.0, bola_target_buffer=30.0), dict(bola_target_buffer=float("inf")),
       dict(bola_min_buffer=float("nan"))]


@pytest.mark.parametrize("bad", BAD, ids=lambda d: ",".join(f"{k}={v}" for k, v in d.items()))
def test_invalid_policy_params_are_rejected_without_a_device(bad):
    from abrsimulator_b200 import _lib
    lib = _lib.load()
    pp = _lib.AbrPolicyParams()
    lib.abr_policy_params_default(ctypes.byref(pp))
    for k, v in bad.items():
        setattr(pp, k, v)
    rc = lib.abr_env_set_policy_params(None, ctypes.byref(pp))
    assert rc == 1 and b"env is NULL" not in lib.abr_last_error(), lib.abr_last_error()
    # the oracle rejects the same values and keeps its parameters
    sizes = np.array([LADDER])
    e = po.PolicyEnv(np.ones((1, 4)), [4], [1.0], sizes, sizes, 1)
    assert not e.set_policy_params(**bad) and e.policy_params == po.DEFAULTS


def test_valid_policy_params_with_a_null_env_report_the_env():
    from abrsimulator_b200 import _lib
    lib = _lib.load()
    pp = _lib.AbrPolicyParams(1.1, 5.0, 20.0)
    assert lib.abr_env_set_policy_params(None, ctypes.byref(pp)) == 1 and b"env is NULL" in lib.abr_last_error()
    assert lib.abr_env_set_policy_params(None, None) == 1
    assert lib.abr_env_policy_decide(None, 3, None, None) == 1


def test_oracle_env_policy_params_change_the_decision():
    sizes = np.array([LADDER] * 4)
    e = po.PolicyEnv(np.full((1, 8), 3000.0), [8], [1.0], sizes, sizes, 2, track_history=1, default_quality=0)
    e.reset([0, 0], [0.0, 3.0])
    for _ in range(3):
        e.step([2, 2], want_next_sizes=False)
    a1 = e.policy_decide(po.POLICY_RATE)
    assert e.set_policy_params(rb_safety=0.25)
    a2 = e.policy_decide(po.POLICY_RATE)
    assert (a2 <= a1).all() and (a2 < a1).any()


@pytest.mark.parametrize("live", [False, True])
def test_stepwise_oracle_episode_equals_the_oracles_fused_episode(live):
    """PolicyEnv runs RATE / BOLA episodes as decide + step per chunk on the environment oracle; for BBA the same
    composition reproduces the oracle's own fused episode bit for bit (actions, trajectories, sums, state)."""
    from oracle import oracle as orc
    from helpers import small_world
    bitrates, sizes, bw, tl, ti = small_world(n_traces=6, T=120, V=20, ragged=True)
    N, steps = 300, 50
    P = dict(track_history=1, **(dict(live=1, start_up_length=8.0) if live else {}))
    a = po.PolicyEnv(bw, tl, ti, sizes, bitrates, N, **P)
    b = po.PolicyEnv(bw, tl, ti, sizes, bitrates, N, **P)
    rng = np.random.default_rng(4)
    tid, off = rng.integers(0, 6, size=N).astype(np.int32), rng.uniform(0, 300.0, size=N)
    speed = rng.choice([0.8, 1.0, 1.25], size=(20, N)) if live else None
    a.reset(tid, off)
    b.reset(tid, off)
    x = a.stepwise_rollout(po.POLICY_BBA, steps, speed=speed)
    y = b.rollout(orc.POLICY_BBA, steps, speed=speed)
    for k in ("delay", "sleep", "buffer", "rebuf", "reward", "latency", "acc"):
        assert np.array_equal(x[k].view(np.uint64), y[k].view(np.uint64)), k
    assert np.array_equal(x["actions"], y["actions"]) and np.array_equal(x["eov"], y["eov"])
    for f in ("seg", "chunk", "buffer", "pos", "hist_len", "bw_hist"):
        assert np.array_equal(a.field(f), b.field(f)), f
    assert len(np.unique(y["actions"])) >= 3 and y["eov"].sum() >= N
