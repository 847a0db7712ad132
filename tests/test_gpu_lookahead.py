"""GPU parity of the clairvoyant lookahead (SPEC §4.4, abr_env_lookahead_decide) against the CPU oracle
(tests/lookahead_oracle.py on oracle/abr_oracle.c), bit for bit, and against the step kernel itself.  Run with -m gpu."""
import ctypes as C
import itertools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from abrsimulator_b200 import _lib, synth
from abrsimulator_b200.datamodel import Chunk, NetworkInfo, QOEMetric
from abrsimulator_b200.env import BatchedABREnv
from abrsimulator_b200.simulator import LookaheadPolicy, Simulator
from oracle import oracle as orc
from helpers import bits_equal, small_world
import lookahead_oracle as lo

LADDERS = {3: (300.0, 1850.0, 4300.0), 6: synth.LADDER_KBPS}
INVALID, RANGE, STATE = 1, 3, 4


def world(ladder, A, n_traces=12, T=300, V=48):
    """'vbr': one bitrate ladder, per-chunk VBR sizes, equal trace lengths; 'ragged': a different ladder per chunk,
    ragged trace lengths and mixed segment durations (the worlds of test_gpu_policies.py)."""
    bitrates, sizes, bw, tl, ti = small_world(n_traces=n_traces, T=T, V=V, ladder=LADDERS[A],
                                              ragged=(ladder == "ragged"))
    if ladder == "ragged":
        scale = np.random.default_rng(8).uniform(0.6, 1.6, size=(V, 1))
        bitrates = np.ascontiguousarray(bitrates * scale)
        sizes = np.ascontiguousarray(sizes * scale)
    return bitrates, sizes, bw, tl, ti


def sessions(N, n_traces, layout, seed=21):
    """'smem': blocks of 64 consecutive sessions on one trace; 'global': interleaved traces."""
    rng = np.random.default_rng(seed)
    if layout == "smem":
        tid = ((np.arange(N) // 64) % n_traces).astype(np.int32)
    else:
        tid = rng.integers(0, n_traces, size=N).astype(np.int32)
    return tid, rng.uniform(0, 900.0, size=N)


def pair(N, A, ladder="vbr", n_traces=12, T=300, V=48, **params):
    bitrates, sizes, bw, tl, ti = world(ladder, A, n_traces, T, V)
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, **params)
    ref = orc.OracleEnv(bw, tl, ti, sizes, bitrates, N, **params)
    return env, ref


def check_decision(env, ref, H, back=lambda t: t.cpu().numpy()):
    act, val, seq = env.lookahead_decide(H, want_value=True, want_seq=True)
    e_act, e_val, e_seq, flagged = lo.decide(ref, H, want_seq=True)
    assert flagged == 0
    assert np.array_equal(back(act), e_act)
    assert bits_equal(back(val), e_val) == 0
    assert np.array_equal(back(seq.t()).T, e_seq)       # back() reorders the last axis: the sessions
    return e_act, e_val, e_seq


def random_steps(env, ref, n, A, rng):
    for _ in range(n):
        a = rng.integers(0, A, size=env.n).astype(np.int32)
        env.step(torch.from_numpy(a).cuda(), want_next_sizes=False)
        ref.step(a, want_next_sizes=False)


# 1. bit for bit against the oracle: shapes, layouts, worlds, states after 0, 17 and 46 steps
@pytest.mark.parametrize("layout", ["smem", "global"])
@pytest.mark.parametrize("ladder", ["vbr", "ragged"])
@pytest.mark.parametrize("A,H", list(itertools.product((3, 6), (1, 2, 5))))
def test_decision_matches_oracle(A, H, ladder, layout):
    N = 640
    env, ref = pair(N, A, ladder, max_buffer=30.0)
    tid, off = sessions(N, 12, layout)
    env.reset(tid, off)
    ref.reset(tid, off)
    rng = np.random.default_rng(A * 7 + H)
    acts = []
    for n in (0, 17, 29):                              # states after 0, 17 and 46 steps
        random_steps(env, ref, n, A, rng)
        e_act, _, e_seq = check_decision(env, ref, H)
        acts.append(e_act)
    assert (e_seq[:, :min(H, 2)] >= 0).all() and (e_seq[:, 2:] == -1).all()   # after 46 of 48 chunks two are left
    assert len(np.unique(np.concatenate(acts))) >= 2
    assert env.error_count() == 0 and ref.errors() == 0


@pytest.mark.parametrize("A,N", [(3, 300), (6, 48)])
def test_horizon_7_matches_oracle(A, N):
    env, ref = pair(N, A, "ragged")
    tid, off = sessions(N, 12, "global", seed=5)
    env.reset(tid, off)
    ref.reset(tid, off)
    random_steps(env, ref, 9, A, np.random.default_rng(1))
    check_decision(env, ref, 7)


def test_done_sessions_and_the_end_of_the_video_without_auto_reset():
    N, A, V = 500, 6, 12
    env, ref = pair(N, A, "ragged", V=V, auto_reset=0, smooth_prev_ladder=1, utility_mode=1, max_buffer=20.0)
    tid, off = sessions(N, 12, "global", seed=8)
    env.reset(tid, off)
    ref.reset(tid, off)
    rng = np.random.default_rng(2)
    for t in range(V + 1):
        _, e_val, e_seq = check_decision(env, ref, 3)
        random_steps(env, ref, 1, A, rng)
    assert (e_seq == -1).all() and (e_val == 0.0).all()
    assert env.error_count() == 0


def test_trace_sorted_order_equals_the_callers_order():
    N, A = 3000, 6
    env, ref = pair(N, A, "ragged", n_traces=37, T=96)
    tid = (np.arange(N) % 37).astype(np.int32)
    off = np.random.default_rng(3).uniform(0, 150.0, size=N)
    env.reset(tid, off, sort_by_trace=True)
    ref.reset(tid, off)
    check_decision(env, ref, 3, back=lambda t: env.to_caller_order(t).cpu().numpy())


# 2. the best sequence replayed through abr_env_step sums to the best value, bit for bit
@pytest.mark.parametrize("ladder", ["vbr", "ragged"])
def test_best_sequence_replayed_by_the_step_kernel_gives_the_best_value(ladder):
    N, A, H = 2048, 6, 5
    env, _ = pair(N, A, ladder, max_buffer=30.0)
    twin, _ = pair(N, A, ladder, max_buffer=30.0)
    tid, off = sessions(N, 12, "smem")
    rng = np.random.default_rng(4)
    for e in (env, twin):
        e.reset(tid, off)
    for n in (0, 17, 29):
        for _ in range(n):
            a = torch.from_numpy(rng.integers(0, A, size=N).astype(np.int32)).cuda()
            env.step(a, want_next_sizes=False)
            twin.step(a, want_next_sizes=False)
        _, val, seq = env.lookahead_decide(H, want_value=True, want_seq=True)
        h = int((seq[0] >= 0).sum().item())
        assert h == min(H, 48 - int(env.state("chunk")[0].item())) and (seq[:, :h] >= 0).all()
        total = torch.zeros(N, dtype=torch.float64, device="cuda")
        states = {f: twin.state(f).clone() for f in ("seg", "chunk", "last_q", "phase", "pos", "buffer")}
        for d in range(h):
            total = total + twin.step(seq[:, d].contiguous(), want_next_sizes=False).reward
        assert bits_equal(total.cpu().numpy(), val.cpu().numpy()) == 0
        for f, t in states.items():                    # back to the decision's state for the next round
            twin.state(f).copy_(t)


# 3. the decision changes nothing
def test_decision_has_no_side_effects():
    N, A = 1500, 6
    P = dict(track_history=1, track_acc=1, hist_k=4)
    a, _ = pair(N, A, "ragged", **P)
    b, _ = pair(N, A, "ragged", **P)
    tid, off = sessions(N, 12, "global")
    rng = np.random.default_rng(6)
    for e in (a, b):
        e.reset(tid, off, sort_by_trace=True)
    steps = torch.from_numpy(rng.integers(0, A, size=(7, N)).astype(np.int32)).cuda()
    for e in (a, b):
        for t in range(7):
            e.step(steps[t], want_next_sizes=False)
    names = list(_lib.FIELDS)
    before = {f: a.state(f).clone() for f in names}
    err = a.error_count()
    a.lookahead_decide(5, want_value=True, want_seq=True)
    a.lookahead_decide(2)
    for f in names:
        assert torch.equal(a.state(f).view(torch.uint8), before[f].view(torch.uint8)), f
    assert a.error_count() == err == 0
    logits = torch.from_numpy(np.random.default_rng(7).normal(size=(N, A)).astype(np.float32)).cuda()
    act_a = torch.empty(N, dtype=torch.int32, device="cuda")
    act_b = torch.empty(N, dtype=torch.int32, device="cuda")
    for t in range(3):
        a.step_policy(logits, sample=True, seed=11, action_out=act_a)
        b.step_policy(logits, sample=True, seed=11, action_out=act_b)
        assert torch.equal(act_a, act_b), t
        a.lookahead_decide(3)
    for f in names:
        assert torch.equal(a.state(f), b.state(f)), f


# 4. episodes
def test_episode_equals_the_oracle_decide_and_step():
    N, A, H, V = 4096, 3, 5, 48
    P = dict(track_acc=1, max_buffer=30.0)
    env, ref = pair(N, A, "vbr", **P)
    twin, _ = pair(N, A, "vbr", **P)
    tid, off = sessions(N, 12, "smem")
    for e in (env, twin, ref):
        e.reset(tid, off)
    acc = np.zeros((orc.NUM_ACC, N))
    for t in range(V):
        act = env.lookahead_decide(H)
        e_act, _, _ = lo.decide(ref, H)
        assert np.array_equal(act.cpu().numpy(), e_act), t
        r = env.step(act, want_next_sizes=False)
        o = ref.step(e_act, want_next_sizes=False, acc=acc)
        for kg, kc in (("delay", "delay"), ("sleep", "sleep"), ("buffer", "buffer"), ("rebuffer", "rebuf"),
                       ("reward", "reward")):
            assert bits_equal(getattr(r, kg).cpu().numpy(), o[kc]) == 0, (t, kg)
    assert bits_equal(env.session_acc().cpu().numpy(), acc) == 0
    twin.lookahead_episode(V, H)
    assert torch.equal(twin.session_acc(), env.session_acc())
    for f in ("seg", "chunk", "last_q", "phase", "pos", "buffer"):
        assert torch.equal(twin.state(f), env.state(f)), f
    assert env.error_count() == 0 and ref.errors() == 0


def test_full_horizon_lookahead_reaches_the_best_fixed_sequence():
    V, A = 5, 3
    seqs = np.array(list(itertools.product(range(A), repeat=V)), np.int32)     # 243 sequences, C order
    M = len(seqs)
    bitrates, sizes, bw, tl, ti = world("ragged", A, n_traces=3, T=30, V=V)
    P = dict(max_buffer=12.0, track_acc=1)
    for tr, off in ((0, 3.7), (1, 41.0), (2, 0.0)):
        fixed = BatchedABREnv(bw, sizes, bitrates, M, trace_len=tl, trace_interval=ti, **P)
        fixed.reset(np.full(M, tr, np.int32), np.full(M, off))
        fixed.rollout("fixed", V, actions=np.ascontiguousarray(seqs.T), want=())
        J = fixed.session_acc()[0].cpu().numpy()
        env = BatchedABREnv(bw, sizes, bitrates, 1, trace_len=tl, trace_interval=ti, **P)
        env.reset(np.array([tr], np.int32), np.array([off]))
        act, val, seq = env.lookahead_decide(V, want_value=True, want_seq=True)
        assert bits_equal(val.cpu().numpy(), J.max()) == 0
        assert seq[0].tolist() == seqs[int(np.argmax(J))].tolist()
        env.lookahead_episode(V, V)
        total = float(env.session_acc()[0, 0])
        assert total >= J.max() - 1e-12 * abs(J.max()) and abs(total - J.max()) <= 1e-12 * abs(J.max())


# 5. full size, once
def test_full_size_65536_sessions():
    N, A, H = 65536, 6, 5
    bitrates, sizes = synth.make_video(48)
    bw, tl, ti = synth.make_traces(1024, 2048)
    tid, off = synth.make_sessions(N, 1024, 2048, group=1)
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti)
    env.reset(tid, off, sort_by_trace=True)
    act, val, seq = env.lookahead_decide(H, want_value=True, want_seq=True)
    back = lambda t: env.to_caller_order(t).cpu().numpy()
    pick = np.arange(0, N, N // 2048)
    ref = orc.OracleEnv(bw, tl, ti, sizes, bitrates, len(pick))
    ref.reset(tid[pick], off[pick])
    e_act, e_val, e_seq, _ = lo.decide(ref, H, want_seq=True)
    assert np.array_equal(back(act)[pick], e_act)
    assert bits_equal(back(val)[pick], e_val) == 0
    assert np.array_equal(back(seq.t()).T[pick], e_seq)
    assert env.error_count() == 0


# 6. errors
def _decide(lib, h, horizon, act):
    rc = lib.abr_env_lookahead_decide(h, C.c_int(horizon), act, None, None, None)
    return rc, ("" if rc == 0 else lib.abr_last_error().decode())


def expect(got, code, text=""):
    rc, msg = got
    assert rc == code and text in msg, (rc, msg, code, text)


def test_errors():
    lib = _lib.load()
    bitrates, sizes, bw, tl, ti = small_world(n_traces=4, T=64, V=10)
    env = BatchedABREnv(bw, sizes, bitrates, 8, trace_len=tl, trace_interval=ti)
    live = BatchedABREnv(bw, sizes, bitrates, 8, trace_len=tl, trace_interval=ti, live=1, start_up_length=8.0)
    act = C.c_void_p(torch.zeros(8, dtype=torch.int32, device="cuda").data_ptr())
    expect(_decide(lib, None, 3, act), INVALID, "env is NULL")
    expect(_decide(lib, env._h, 3, act), STATE, "abr_env_reset has not been called")
    expect(_decide(lib, live._h, 3, act), STATE, "abr_env_reset has not been called")    # not reset before live
    live.reset(np.zeros(0, np.int32))
    expect(_decide(lib, live._h, 0, None), STATE, "not available in live mode")         # live before empty batch
    live.reset(np.zeros(4, np.int32))
    expect(_decide(lib, live._h, 3, act), STATE, "not available in live mode")
    expect(_decide(lib, live._h, 9, None), STATE, "not available in live mode")         # live before the rest
    env.reset(np.zeros(0, np.int32))
    expect(_decide(lib, env._h, 0, None), 0)                                            # empty batch: a no-op
    env.reset(np.zeros(4, np.int32))
    expect(_decide(lib, env._h, 3, None), INVALID, "action is NULL")
    expect(_decide(lib, env._h, 0, None), INVALID, "action is NULL")                    # NULL action before horizon
    for bad in (0, -1, 9):
        expect(_decide(lib, env._h, bad, act), RANGE, "horizon must be in [1, 8]")
    expect(_decide(lib, env._h, 8, act), RANGE, "2^20")                                 # 6^8 > 2^20
    expect(_decide(lib, env._h, 7, act), 0)                                             # 6^7 <= 2^20
    with pytest.raises(_lib.AbrError) as ei:
        env.lookahead_decide(8)
    assert ei.value.code == RANGE and "2^20" in str(ei.value)
    assert env.error_count() == 0
    sim = Simulator(LookaheadPolicy(3), None)
    sim.set_qoe_metric(QOEMetric(4.3, 1.0, 2.0, 0.1))
    sim.set_network_info(1.0, list(bw[0]))
    sim.set_mpd(4.0, 24.0, 8.0, [Chunk(list(b / 1000.0)) for b in bitrates])
    with pytest.raises(ValueError, match="SPEC §7"):
        sim.run_batch(4)


# 7. the Simulator marker
def test_simulator_marker_equals_the_env_episode():
    bitrates, sizes, bw, tl, ti = small_world(n_traces=2, T=200, V=30)
    qoe = QOEMetric(4.3, 0.5, 2.0, 0.1)
    sim = Simulator(LookaheadPolicy(3), None)
    sim.set_qoe_metric(qoe)
    nets = [NetworkInfo(1.0, list(bw[0])), NetworkInfo(0.5, list(bw[1][:60]))]
    sim.set_network_info(1.0, nets)
    sim.set_mpd(4.0, 24.0, None, [Chunk(list(b / 1000.0)) for b in bitrates])
    n = 128
    costs = sim.run_batch(n)
    P = dict(chunk_length=4.0, max_buffer=24.0, rebuf_penalty=4.3, smooth_penalty=0.5, utility_scale=1.0, rtt=0.0,
             payload=1.0, sleep_quantum=0.01, smooth_prev_ladder=1, latency_tick=0.01, default_quality=-1, auto_reset=0,
             track_acc=1)
    bw2 = np.ones((2, 200)); bw2[0] = bw[0]; bw2[1, :60] = bw[1][:60]
    tl2, ti2 = np.array([200, 60], np.int32), np.array([1.0, 0.5])
    env = BatchedABREnv(bw2, bitrates / 1000.0 * 4.0, bitrates / 1000.0, n, trace_len=tl2, trace_interval=ti2, **P)
    tid = ((np.arange(n) * 2) // n).astype(np.int32)
    env.reset(tid)
    env.lookahead_episode(30, 3)
    acc = env.session_acc().cpu().numpy()
    assert bits_equal(costs, 4.3 * acc[1] + 0.5 * acc[3]) == 0
    assert (acc[6] == 30).all() and env.error_count() == 0
