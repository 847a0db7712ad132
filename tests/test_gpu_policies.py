"""GPU parity of the RATE and BOLA policies (SPEC §4.2, §4.3) — in the fused episode and as the batched per-step
decision abr_env_policy_decide — against the CPU oracle (tests/policy_oracle.py on oracle/abr_oracle.c), bit for bit.
Run with -m gpu."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from abrsimulator_b200 import _lib, synth
from abrsimulator_b200.datamodel import Chunk, NetworkInfo, QOEMetric
from abrsimulator_b200.env import BatchedABREnv
from abrsimulator_b200.simulator import BolaPolicy, RateBasedPolicy, Simulator
from oracle import oracle as orc
from helpers import assert_close, bits_equal, small_world
import policy_oracle as po

POLICIES = ["rate", "bola"]
PID = dict(rate=po.POLICY_RATE, bola=po.POLICY_BOLA, bba=po.POLICY_BBA)
TRAJ = (("delay", "delay"), ("sleep", "sleep"), ("buffer", "buffer"), ("rebuffer", "rebuf"), ("reward", "reward"))
LIVE = dict(live=1, start_up_length=8.0, startup_penalty=2.0, latency_penalty=0.1)


def world(ladder, n_traces=12, T=300, V=48):
    """'vbr': one bitrate ladder, per-chunk VBR sizes, equal trace lengths; 'ragged': a different ladder per chunk,
    ragged trace lengths and mixed segment durations."""
    bitrates, sizes, bw, tl, ti = small_world(n_traces=n_traces, T=T, V=V, ragged=(ladder == "ragged"))
    if ladder == "ragged":
        scale = np.random.default_rng(8).uniform(0.6, 1.6, size=(V, 1))
        bitrates = np.ascontiguousarray(bitrates * scale)
        sizes = np.ascontiguousarray(sizes * scale)
    return bitrates, sizes, bw, tl, ti


def sessions(N, n_traces, layout, seed=21):
    """'smem': blocks of 64 consecutive sessions on one trace (shared-memory path); 'global': interleaved traces."""
    rng = np.random.default_rng(seed)
    if layout == "smem":
        tid = ((np.arange(N) // 64) % n_traces).astype(np.int32)
    else:
        tid = rng.integers(0, n_traces, size=N).astype(np.int32)
    return tid, rng.uniform(0, 900.0, size=N)


def pair(N, params, ladder="vbr", n_traces=12, T=300, V=48, policy_params=None):
    bitrates, sizes, bw, tl, ti = world(ladder, n_traces, T, V)
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, **params)
    ref = po.PolicyEnv(bw, tl, ti, sizes, bitrates, N, **params)
    if policy_params:
        env.set_policy_params(**policy_params)
        assert ref.set_policy_params(**policy_params)
    return env, ref


def ring_valid(ring_sn, hist_len, K):
    """[N][K] ring -> the min(hist_len, K) most recent samples of each session, oldest first (NaN-padded)."""
    out = np.full_like(ring_sn, np.nan)
    for s in range(ring_sn.shape[0]):
        L = int(hist_len[s])
        n = min(L, K)
        for j in range(n):
            out[s, j] = ring_sn[s, (L - n + j) % K]
    return out


def check_all_state(env, ref):
    for f in ("seg", "chunk", "last_q", "trace_id", "hist_len"):
        assert np.array_equal(env.state(f).cpu().numpy(), ref.field(f)), f
    for f in ("phase", "pos", "buffer"):
        assert bits_equal(env.state(f).cpu().numpy(), ref.field(f)) == 0, f
    if env.params.track_history:
        hl = ref.field("hist_len")
        a = ring_valid(env.state("bw_hist").cpu().numpy().T.copy(), hl, env.K)
        b = ring_valid(ref.field("bw_hist"), hl, env.K)
        assert np.array_equal(np.isnan(a), np.isnan(b)) and bits_equal(np.nan_to_num(a), np.nan_to_num(b)) == 0


def check_episode(env, ref, got, exp, N, steps):
    assert np.array_equal(got["actions"].cpu().numpy(), exp["actions"])
    for kg, kc in TRAJ:
        assert_close(got[kg].cpu().numpy(), exp[kc], kg)
    assert np.array_equal(got["end_of_video"].cpu().numpy(), exp["eov"])
    assert_close(env.session_acc().cpu().numpy(), exp["acc"], "acc")
    check_all_state(env, ref)
    np.testing.assert_allclose(env.stats().cpu().numpy(), orc.stats_from_acc(exp["acc"]), rtol=1e-9)
    assert env.error_count() == 0 and ref.errors() == 0


# 1. the fused episode over two end-of-video resets
@pytest.mark.parametrize("layout", ["smem", "global"])
@pytest.mark.parametrize("ladder", ["vbr", "ragged"])
@pytest.mark.parametrize("policy", POLICIES)
def test_fused_rollout_matches_oracle_over_two_resets(policy, ladder, layout):
    N, steps = 4096, 100
    env, ref = pair(N, dict(track_history=1), ladder)
    tid, off = sessions(N, 12, layout)
    env.reset(tid, off)
    ref.reset(tid, off)
    got = env.rollout(policy, steps, seed=3)
    exp = ref.rollout(PID[policy], steps, seed=3)
    check_episode(env, ref, got, exp, N, steps)
    eov = exp["eov"]
    assert eov[47].all() and eov[95].all() and int(eov.sum()) == 2 * N
    acts = exp["actions"]
    assert len(np.unique(acts)) >= 3                         # the policy actually adapts
    if policy == "rate":                                     # after each reset the ring is empty: default quality
        assert (acts[0] == 1).all() and (acts[48] == 1).all() and (acts[96] == 1).all()


# 2. episodes split into calls
@pytest.mark.parametrize("policy", POLICIES)
def test_split_rollout_equals_one_rollout(policy):
    N = 1000
    env_a, _ = pair(N, dict(track_history=1), "ragged")
    env_b, _ = pair(N, dict(track_history=1), "ragged")
    tid, off = sessions(N, 12, "global")
    env_a.reset(tid, off)
    env_b.reset(tid, off)
    whole = env_a.rollout(policy, 48)
    h1 = env_b.rollout(policy, 24)
    h2 = env_b.rollout(policy, 24)
    for k in whole:
        assert torch.equal(whole[k], torch.cat([h1[k], h2[k]])), k
    for f in ("seg", "chunk", "last_q", "phase", "pos", "buffer", "hist_len", "bw_hist"):
        assert torch.equal(env_a.state(f), env_b.state(f)), f
    # each launch adds its own per-session sum into the accumulators: two partial sums round differently from one
    a, b = env_a.state("acc").cpu().numpy(), env_b.state("acc").cpu().numpy()
    np.testing.assert_allclose(b, a, rtol=1e-12, atol=1e-12)
    assert np.array_equal(a[6:8], b[6:8])                    # step and episode counts are exact


# 3. whole runs: device-resident and host buffers (pinned and pageable)
@pytest.mark.parametrize("policy", POLICIES)
def test_run_and_run_host_equal_reset_and_rollout(policy):
    N, steps = 3000, 60
    P = dict(track_history=1)
    env_a, _ = pair(N, P, policy_params=dict(rb_safety=0.9, bola_min_buffer=8.0, bola_target_buffer=40.0))
    env_b, _ = pair(N, P, policy_params=dict(rb_safety=0.9, bola_min_buffer=8.0, bola_target_buffer=40.0))
    tid, off = sessions(N, 12, "smem")
    env_a.reset(tid, off)
    exp = env_a.rollout(policy, steps, seed=9)
    acc = env_a.session_acc().cpu().numpy()
    cost = env_a.qoe_cost().cpu().numpy()
    stats = env_a.stats().cpu().numpy()
    out, c2, s2 = env_b.run(policy, steps, tid, off, seed=9, want=("reward", "buffer", "end_of_video", "actions"))
    for k in out:
        assert torch.equal(out[k], exp[k]), k
    assert bits_equal(c2.cpu().numpy(), cost) == 0 and bits_equal(env_b.session_acc().cpu().numpy(), acc) == 0
    np.testing.assert_allclose(s2.cpu().numpy(), stats, rtol=1e-12)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    for host_in in (lambda a: a, pin):
        h = env_b.run_host(policy, steps, host_in(tid), host_in(off), seed=9, want_qoe_cost=True,
                           want_reward_traj=True)
        assert bits_equal(np.asarray(h["acc"]), acc) == 0
        assert bits_equal(np.asarray(h["qoe_cost"]), cost) == 0
        assert bits_equal(np.asarray(h["reward"]), exp["reward"].cpu().numpy()) == 0
        np.testing.assert_allclose(np.asarray(h["stats"]), stats, rtol=1e-12)
    assert env_b.error_count() == 0


# 4. fp32-output mode
@pytest.mark.parametrize("policy", POLICIES)
def test_fp32_outputs_are_the_fp64_outputs_rounded_once(policy):
    N, steps = 2000, 60
    env_a, _ = pair(N, dict(track_history=1))
    env_b, _ = pair(N, dict(track_history=1))
    tid, off = sessions(N, 12, "smem")
    env_a.reset(tid, off)
    env_b.reset(tid, off)
    g64 = env_a.rollout(policy, steps)
    g32 = env_b.rollout(policy, steps, dtype=torch.float32)
    for k in g64:
        if k in ("actions", "end_of_video"):
            assert torch.equal(g64[k], g32[k]), k
        else:
            assert g32[k].dtype == torch.float32 and torch.equal(g64[k].float(), g32[k]), k
    for f in ("phase", "pos", "buffer", "bw_hist", "acc"):
        assert torch.equal(env_a.state(f), env_b.state(f)), f


# 5. live mode with a per-chunk speed table
@pytest.mark.parametrize("policy", POLICIES)
def test_fused_live_episode_matches_oracle(policy):
    N, steps, V = 64 * 9 + 21, 75, 30
    P = dict(LIVE, track_history=1)
    env, ref = pair(N, P, "ragged", n_traces=5, V=V)
    tid, off = sessions(N, 5, "smem")
    tid[64 * 4:64 * 6] = np.random.default_rng(2).integers(0, 5, size=128)     # two mixed blocks -> global path
    speed = np.random.default_rng(31).choice([0.75, 1.0, 1.0, 1.25, 1.5], size=(V, N))
    env.reset(tid, off)
    ref.reset(tid, off)
    want = ("delay", "sleep", "buffer", "rebuffer", "reward", "latency", "end_of_video", "actions")
    got = env.rollout(policy, steps, speed=speed, want=want)
    exp = ref.rollout(PID[policy], steps, speed=speed)
    check_episode(env, ref, got, exp, N, steps)
    assert_close(got["latency"].cpu().numpy(), exp["latency"], "latency")
    for f in ("t_now", "play_time", "play_len"):
        assert bits_equal(env.state(f).cpu().numpy(), ref.field(f)) == 0, f
    assert len(np.unique(exp["actions"])) >= 3


# 6. the per-step decision
@pytest.mark.parametrize("live", [False, True])
@pytest.mark.parametrize("policy", POLICIES + ["bba"])
def test_policy_decide_then_step_equals_the_fused_episode(policy, live):
    N, steps = 1500, 70
    P = dict(track_history=1, track_acc=1, **(LIVE if live else {}))
    env_a, ref = pair(N, P, "ragged")
    env_b, _ = pair(N, P, "ragged")
    tid, off = sessions(N, 12, "global")
    speed = np.random.default_rng(5).choice([0.8, 1.0, 1.25], size=(48, N)) if live else None
    for e in (env_a, env_b, ref):
        e.reset(tid, off)
    want = ("delay", "sleep", "buffer", "rebuffer", "reward", "end_of_video", "actions")
    whole = env_a.rollout(policy, steps, speed=speed, want=want)
    act = torch.empty(N, dtype=torch.int32, device="cuda")
    for t in range(steps):
        env_b.policy_decide(policy, out=act)
        exp_act = ref.policy_decide(PID[policy])
        assert np.array_equal(act.cpu().numpy(), exp_act), t
        assert torch.equal(act, whole["actions"][t]), t
        r = env_b.step(act, want_next_sizes=False, speed=speed)
        ref.step(exp_act, want_next_sizes=False, speed=speed)
        assert torch.equal(r.reward, whole["reward"][t]) and torch.equal(r.buffer, whole["buffer"][t]), t
        assert torch.equal(r.delay, whole["delay"][t]) and torch.equal(r.end_of_video, whole["end_of_video"][t]), t
    for f in ("seg", "chunk", "last_q", "phase", "pos", "buffer", "hist_len", "bw_hist", "acc"):
        assert torch.equal(env_a.state(f), env_b.state(f)), f
    check_all_state(env_b, ref)
    assert env_a.error_count() == 0 and env_b.error_count() == 0


@pytest.mark.parametrize("policy", POLICIES + ["bba"])
def test_policy_decide_on_crafted_states(policy):
    """Ties between BOLA scores, budgets that equal a size exactly, empty and wrapped rings, done sessions."""
    V, A, K, N = 3, 5, 4, 512
    sizes = np.array([[1.0, 2.0, 4.0, 4.0, 8.0],          # duplicate size: equal scores
                      [0.5, 3.0, 2.0, 6.0, 5.0],          # non-monotone
                      [1.0, 1.5, 2.25, 3.375, 5.0625]])
    bitrates = sizes / 4.0
    rng = np.random.default_rng(17)
    P = dict(track_history=1, hist_k=K, auto_reset=0, default_quality=2, chunk_length=4.0)
    env = BatchedABREnv(np.ones((1, 16)), sizes, bitrates, N, **P)
    env.reset(np.zeros(N, np.int32))
    chunk = rng.integers(0, V + 1, size=N).astype(np.int32)          # V: done
    done = (chunk == V).astype(np.uint8)
    buffer = rng.choice([0.0, 5.0, 9.5, 10.0, 12.0, 20.0, 29.0, 35.0, rng.uniform(0, 60)], size=N)
    hist_len = rng.integers(0, 3 * K, size=N).astype(np.int32)
    ring = rng.choice([0.25, 0.5, 1.0, 2.0, 0.375], size=(N, K))     # exact harmonic means -> budgets on sizes
    dev = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a)).to("cuda", dt)
    env.state("chunk").copy_(dev(chunk, torch.int32))
    env.state("done").copy_(dev(done, torch.uint8))
    env.state("buffer").copy_(dev(buffer, torch.float64))
    env.state("hist_len").copy_(dev(hist_len, torch.int32))
    env.state("bw_hist").copy_(dev(ring.T, torch.float64))
    for pp in (dict(), dict(rb_safety=0.5, bola_min_buffer=5.0, bola_target_buffer=20.0)):
        if pp:
            env.set_policy_params(**pp)
        got = env.policy_decide(policy).cpu().numpy()
        exp = po.policy_decide(PID[policy], sizes, chunk, buffer, ring, hist_len, done=done, default_quality=2,
                               chunk_length=4.0, **pp)
        assert np.array_equal(got, exp)
        if policy != "bba":
            assert (got[done == 1] == 0).all()
    assert len(np.unique(got)) >= 3


# 7. trace-sorted session order
@pytest.mark.parametrize("policy", POLICIES)
def test_trace_sorted_order_equals_the_callers_order(policy):
    N, steps = 3000, 60
    env_a, _ = pair(N, dict(track_history=1), "ragged", n_traces=37, T=96)
    env_b, _ = pair(N, dict(track_history=1), "ragged", n_traces=37, T=96)
    tid = (np.arange(N) % 37).astype(np.int32)
    off = np.random.default_rng(3).uniform(0, 150.0, size=N)
    env_a.reset(tid, off, session_base=500)
    env_b.reset(tid, off, session_base=500, sort_by_trace=True)
    out_a = env_a.rollout(policy, steps)
    out_b = env_b.rollout(policy, steps)
    for k in out_a:
        assert torch.equal(out_a[k], env_b.to_caller_order(out_b[k])), k
    for f in ("seg", "chunk", "last_q", "phase", "pos", "buffer", "hist_len"):
        assert torch.equal(env_a.state(f), env_b.to_caller_order(env_b.state(f))), f
    assert torch.equal(env_a.state("acc"), env_b.to_caller_order(env_b.state("acc")))
    a1 = env_a.policy_decide(policy)
    assert torch.equal(a1, env_b.to_caller_order(env_b.policy_decide(policy)))


# 8. the Simulator markers
@pytest.mark.parametrize("live", [False, True])
@pytest.mark.parametrize("marker", ["rate", "bola"])
def test_simulator_markers_equal_the_env_path(marker, live):
    bitrates, sizes, bw, tl, ti = small_world(n_traces=2, T=200, V=30)
    ctrl = RateBasedPolicy(0.85) if marker == "rate" else BolaPolicy(6.0, 24.0)
    qoe = QOEMetric(4.3, 0.5, 2.0, 0.1)
    sim = Simulator(ctrl, None)
    sim.set_qoe_metric(qoe)
    nets = [NetworkInfo(1.0, list(bw[0])), NetworkInfo(0.5, list(bw[1][:60]))]
    sim.set_network_info(1.0, nets)
    sim.set_mpd(4.0, 24.0, 8.0 if live else None, [Chunk(list(b / 1000.0)) for b in bitrates])
    n = 128
    costs = sim.run_batch(n)
    P = dict(chunk_length=4.0, max_buffer=24.0, rebuf_penalty=4.3, smooth_penalty=0.5, utility_scale=1.0, rtt=0.0,
             payload=1.0, sleep_quantum=0.01, smooth_prev_ladder=1, latency_tick=0.01, default_quality=-1, auto_reset=0)
    if live:
        P.update(LIVE, track_acc=1)
    if marker == "rate":
        P.update(track_history=1)
    pp = dict(rb_safety=0.85) if marker == "rate" else dict(bola_min_buffer=6.0, bola_target_buffer=24.0)
    bw2 = np.ones((2, 200)); bw2[0] = bw[0]; bw2[1, :60] = bw[1][:60]
    tl2, ti2 = np.array([200, 60], np.int32), np.array([1.0, 0.5])
    env = BatchedABREnv(bw2, bitrates / 1000.0 * 4.0, bitrates / 1000.0, n, trace_len=tl2, trace_interval=ti2, **P)
    env.set_policy_params(**pp)
    tid = ((np.arange(n) * 2) // n).astype(np.int32)
    if live:
        env.reset(tid)
        env.rollout(marker, 30, want=())
        want = env.qoe_cost().cpu().numpy()
    else:
        want = env.run_host(marker, 30, tid, want_qoe_cost=True)["qoe_cost"]
    assert bits_equal(costs, want) == 0
    ref = po.PolicyEnv(bw2, tl2, ti2, bitrates / 1000.0 * 4.0, bitrates / 1000.0, n, **P)
    assert ref.set_policy_params(**pp)
    ref.reset(tid)
    a = ref.rollout(PID[marker], 30)["acc"]
    exp = 4.3 * a[1] + 0.5 * a[3]
    if live:
        exp = exp + 2.0 * a[8] + 0.1 * a[9] / (0.01 * a[10])
    np.testing.assert_allclose(costs, exp, rtol=1e-12)


# 9. errors
def test_errors():
    bitrates, sizes, bw, tl, ti = small_world(n_traces=4, T=64, V=10)
    N = 256
    tid = np.zeros(N, np.int32)
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti)     # track_history = 0
    env.reset(tid)
    act = torch.empty(N, dtype=torch.int32, device="cuda")
    calls = [lambda: env.rollout("rate", 5), lambda: env.rollout("rate", 5, dtype=torch.float32),
             lambda: env.run("rate", 5, tid), lambda: env.run("rate", 0, tid), lambda: env.run_host("rate", 5, tid),
             lambda: env.policy_decide("rate", out=act)]
    for c in calls:
        with pytest.raises(_lib.AbrError) as ei:
            c()
        assert ei.value.code == 4 and "track_history" in str(ei.value)
    env.reset(tid)
    env.rollout("bola", 5)                               # BOLA needs no history
    zero = sizes.copy()
    zero[3, 0] = 0.0
    envz = BatchedABREnv(bw, zero, bitrates, N, trace_len=tl, trace_interval=ti, track_history=1)   # creates fine
    envz.reset(tid)
    envz.rollout("rate", 5)
    for c in (lambda: envz.rollout("bola", 5), lambda: envz.run_host("bola", 5, tid),
              lambda: envz.run("bola", 5, tid), lambda: envz.policy_decide("bola", out=act)):
        with pytest.raises(_lib.AbrError) as ei:
            c()
        assert ei.value.code == 1 and "positive chunk sizes" in str(ei.value)
    envz.reset(tid)
    for bad in (5, -1):
        with pytest.raises(_lib.AbrError) as ei:
            envz.rollout(bad, 5)
        assert ei.value.code == 1
    for bad in ("fixed", "random", 5, 0):
        with pytest.raises(_lib.AbrError) as ei:
            envz.policy_decide(bad, out=act)
        assert ei.value.code == 1
    for bad in (dict(rb_safety=0.0), dict(bola_min_buffer=30.0), dict(bola_target_buffer=float("nan"))):
        with pytest.raises(_lib.AbrError) as ei:
            env.set_policy_params(**bad)
        assert ei.value.code == 1
    assert env.error_count() == 0 and envz.error_count() == 0


# 10. full size
@pytest.mark.parametrize("policy", POLICIES)
def test_full_size_sorted_by_trace_bit_exact_65536x48(policy):
    N, steps = 65536, 48
    bitrates, sizes = synth.make_video(48)
    bw, tl, ti = synth.make_traces(1024, 2048)
    tid, off = synth.make_sessions(N, 1024, 2048, group=1)
    P = dict(track_history=1)
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, **P)
    env.reset(tid, off, sort_by_trace=True)
    out = env.rollout(policy, steps)
    perm = env.perm.cpu().numpy()
    ref = po.PolicyEnv(bw, tl, ti, sizes, bitrates, N, **P)
    ref.reset(tid, off)
    exp = ref.rollout(PID[policy], steps)
    back = lambda t: env.to_caller_order(t).cpu().numpy()
    assert np.array_equal(back(out["actions"]), exp["actions"])
    for kg, kc in TRAJ:
        assert bits_equal(back(out[kg]), exp[kc]) == 0, kg
    assert np.array_equal(back(out["end_of_video"]), exp["eov"])
    assert bits_equal(back(env.session_acc()), exp["acc"]) == 0
    assert np.array_equal(back(env.state("chunk")), ref.field("chunk"))
    assert bits_equal(back(env.state("buffer")), ref.field("buffer")) == 0
    assert sorted(perm.tolist()) == list(range(N))
    assert env.error_count() == 0
