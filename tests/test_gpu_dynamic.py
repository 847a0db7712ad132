"""GPU parity of the DYNAMIC policy (SPEC §4.6) — in the fused episode and as the batched per-step decision
abr_env_policy_decide — against the CPU oracle (tests/dynamic_oracle.py on oracle/abr_oracle.c), bit for bit.  The
traces alternate high and low bandwidth phases, and every case checks in its own oracle run that the rule switches
both ways (rate -> BOLA and BOLA -> rate inside an episode).  Run with -m gpu."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from abrsimulator_b200 import _lib, synth
from abrsimulator_b200.datamodel import Chunk, NetworkInfo, QOEMetric
from abrsimulator_b200.env import BatchedABREnv
from abrsimulator_b200.simulator import DynamicPolicy, Simulator
from oracle import oracle as orc
from helpers import assert_close, bits_equal, small_world
import dynamic_oracle as do

DYN = do.POLICY_DYNAMIC
TRAJ = (("delay", "delay"), ("sleep", "sleep"), ("buffer", "buffer"), ("rebuffer", "rebuf"), ("reward", "reward"))
LIVE = dict(live=1, start_up_length=8.0, startup_penalty=2.0, latency_penalty=0.1)
STATE = ("seg", "chunk", "last_q", "trace_id", "hist_len", "dyn_mode")


def phased(bw, seed=77):
    """Alternating high (x4) and low (x0.12) phases of 40..90 segments: the buffer climbs past switch_on in the high
    phases and drains below switch_off in the low ones."""
    rng = np.random.default_rng(seed)
    n, T = bw.shape
    t = np.arange(T)
    period = rng.integers(40, 90, size=(n, 1))
    shift = rng.integers(0, 90, size=(n, 1))
    return np.ascontiguousarray(bw * np.where(((t + shift) // period) % 2 == 0, 4.0, 0.12))


def world(ladder="vbr", n_traces=12, T=300, V=48):
    bitrates, sizes, bw, tl, ti = small_world(n_traces=n_traces, T=T, V=V, ragged=(ladder == "ragged"))
    if ladder == "ragged":
        scale = np.random.default_rng(8).uniform(0.6, 1.6, size=(V, 1))
        bitrates = np.ascontiguousarray(bitrates * scale)
        sizes = np.ascontiguousarray(sizes * scale)
    return bitrates, sizes, phased(bw), tl, ti


def sessions(N, n_traces, layout, seed=21):
    """'smem': blocks of 64 consecutive sessions on one trace (shared-memory path); 'global': interleaved traces."""
    rng = np.random.default_rng(seed)
    if layout == "smem":
        tid = ((np.arange(N) // 64) % n_traces).astype(np.int32)
    else:
        tid = rng.integers(0, n_traces, size=N).astype(np.int32)
    return tid, rng.uniform(0, 900.0, size=N)


def make(N, params, ladder="vbr", n_traces=12, T=300, V=48, n_env=1, policy_params=None, dynamic_params=None):
    """n_env device environments and one oracle over the same world, with the same parameters installed."""
    bitrates, sizes, bw, tl, ti = world(ladder, n_traces, T, V)
    envs = [BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, **params) for _ in range(n_env)]
    ref = do.DynamicEnv(bw, tl, ti, sizes, bitrates, N, **params)
    for e in envs:
        if policy_params:
            e.set_policy_params(**policy_params)
        if dynamic_params:
            e.set_dynamic_params(**dynamic_params)
    if policy_params:
        assert ref.set_policy_params(**policy_params)
    if dynamic_params:
        assert ref.set_dynamic_params(**dynamic_params)
    return envs, ref


def assert_switches(ref):
    up, down = ref.switches()
    assert up > 0 and down > 0, (up, down)


def ring_valid(ring_sn, hist_len, K):
    out = np.full_like(ring_sn, np.nan)
    for s in range(ring_sn.shape[0]):
        L = int(hist_len[s])
        n = min(L, K)
        for j in range(n):
            out[s, j] = ring_sn[s, (L - n + j) % K]
    return out


def check_state(env, ref):
    for f in STATE:
        got = env.state(f).cpu().numpy()
        assert np.array_equal(got, ref.dyn_mode if f == "dyn_mode" else ref.field(f)), f
    for f in ("phase", "pos", "buffer"):
        assert bits_equal(env.state(f).cpu().numpy(), ref.field(f)) == 0, f
    hl = ref.field("hist_len")
    a = ring_valid(env.state("bw_hist").cpu().numpy().T.copy(), hl, env.K)
    b = ring_valid(ref.field("bw_hist"), hl, env.K)
    assert np.array_equal(np.isnan(a), np.isnan(b)) and bits_equal(np.nan_to_num(a), np.nan_to_num(b)) == 0


def check_episode(env, ref, got, exp):
    assert np.array_equal(got["actions"].cpu().numpy(), exp["actions"])
    for kg, kc in TRAJ:
        assert_close(got[kg].cpu().numpy(), exp[kc], kg)
    assert np.array_equal(got["end_of_video"].cpu().numpy(), exp["eov"])
    assert_close(env.session_acc().cpu().numpy(), exp["acc"], "acc")
    check_state(env, ref)
    np.testing.assert_allclose(env.stats().cpu().numpy(), orc.stats_from_acc(exp["acc"]), rtol=1e-9)
    assert env.error_count() == 0 and ref.errors() == 0


# 1. the fused episode on both trace paths, over end-of-video resets (auto_reset 1) or past the end (auto_reset 0)
@pytest.mark.parametrize("auto_reset", [1, 0])
@pytest.mark.parametrize("layout", ["smem", "global"])
def test_fused_episode_matches_oracle(layout, auto_reset):
    N, steps = 4096, 100
    (env,), ref = make(N, dict(track_history=1, auto_reset=auto_reset))
    tid, off = sessions(N, 12, layout)
    env.reset(tid, off)
    ref.reset(tid, off)
    got = env.rollout("dynamic", steps, seed=3)
    exp = ref.rollout(DYN, steps)
    check_episode(env, ref, got, exp)
    assert_switches(ref)
    eov = exp["eov"]
    assert eov[47].all()
    if auto_reset:
        assert eov[95].all() and int(eov.sum()) == 2 * N
        assert (exp["actions"][48] == 1).all() and (exp["actions"][96] == 1).all()   # rate rule, empty ring
    else:
        assert (exp["actions"][48:] == 0).all()                                      # inert steps
    assert len(np.unique(exp["actions"])) >= 4


# 2. an episode split into calls: the rule carries over in dyn_mode
def test_split_episode_equals_one_episode():
    N = 1000
    (env_a, env_b), ref = make(N, dict(track_history=1), "ragged", n_env=2)
    tid, off = sessions(N, 12, "global")
    for e in (env_a, env_b, ref):
        e.reset(tid, off)
    whole = env_a.rollout("dynamic", 48)
    h1 = env_b.rollout("dynamic", 24)
    mid = env_b.state("dyn_mode").clone()
    h2 = env_b.rollout("dynamic", 24)
    for k in whole:
        assert torch.equal(whole[k], torch.cat([h1[k], h2[k]])), k
    for f in ("seg", "chunk", "last_q", "phase", "pos", "buffer", "hist_len", "bw_hist", "dyn_mode"):
        assert torch.equal(env_a.state(f), env_b.state(f)), f
    a, b = env_a.state("acc").cpu().numpy(), env_b.state("acc").cpu().numpy()
    np.testing.assert_allclose(b, a, rtol=1e-12, atol=1e-12)
    assert np.array_equal(a[6:8], b[6:8])
    exp = ref.rollout(DYN, 48)
    assert np.array_equal(whole["actions"].cpu().numpy(), exp["actions"])
    assert np.array_equal(mid.cpu().numpy(), ref.decisions[23][2])
    check_state(env_b, ref)
    assert_switches(ref)
    assert (mid == 1).any() and (mid == 0).any()


# 3. whole runs: device-resident and host buffers (pinned and pageable)
def test_run_and_run_host_equal_reset_and_rollout():
    N, steps = 3000, 60
    P = dict(track_history=1)
    pp, dp = dict(rb_safety=0.9, bola_min_buffer=8.0, bola_target_buffer=40.0), dict(switch_on_buffer=15.0,
                                                                                   switch_off_buffer=4.0)
    (env_a, env_b), ref = make(N, P, n_env=2, policy_params=pp, dynamic_params=dp)
    tid, off = sessions(N, 12, "smem")
    env_a.reset(tid, off)
    exp = env_a.rollout("dynamic", steps, seed=9)
    acc = env_a.session_acc().cpu().numpy()
    cost = env_a.qoe_cost().cpu().numpy()
    stats = env_a.stats().cpu().numpy()
    mode = env_a.state("dyn_mode").clone()
    out, c2, s2 = env_b.run("dynamic", steps, tid, off, seed=9, want=("reward", "buffer", "end_of_video", "actions"))
    for k in out:
        assert torch.equal(out[k], exp[k]), k
    assert bits_equal(c2.cpu().numpy(), cost) == 0 and bits_equal(env_b.session_acc().cpu().numpy(), acc) == 0
    np.testing.assert_allclose(s2.cpu().numpy(), stats, rtol=1e-12)
    assert torch.equal(env_b.state("dyn_mode"), mode)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    for host_in in (lambda a: a, pin):
        h = env_b.run_host("dynamic", steps, host_in(tid), host_in(off), seed=9, want_qoe_cost=True,
                           want_reward_traj=True)
        assert bits_equal(np.asarray(h["acc"]), acc) == 0
        assert bits_equal(np.asarray(h["qoe_cost"]), cost) == 0
        assert bits_equal(np.asarray(h["reward"]), exp["reward"].cpu().numpy()) == 0
        np.testing.assert_allclose(np.asarray(h["stats"]), stats, rtol=1e-12)
        assert torch.equal(env_b.state("dyn_mode"), mode)
    assert env_b.error_count() == 0
    ref.reset(tid, off)
    r = ref.rollout(DYN, steps)
    assert np.array_equal(exp["actions"].cpu().numpy(), r["actions"]) and bits_equal(acc, r["acc"]) == 0
    assert np.array_equal(mode.cpu().numpy(), ref.dyn_mode)
    assert_switches(ref)


# 4. fp32-output mode
def test_fp32_outputs_are_the_fp64_outputs_rounded_once():
    N, steps = 2000, 60
    (env_a, env_b), ref = make(N, dict(track_history=1), n_env=2)
    tid, off = sessions(N, 12, "smem")
    for e in (env_a, env_b, ref):
        e.reset(tid, off)
    g64 = env_a.rollout("dynamic", steps)
    g32 = env_b.rollout("dynamic", steps, dtype=torch.float32)
    for k in g64:
        if k in ("actions", "end_of_video"):
            assert torch.equal(g64[k], g32[k]), k
        else:
            assert g32[k].dtype == torch.float32 and torch.equal(g64[k].float(), g32[k]), k
    for f in ("phase", "pos", "buffer", "bw_hist", "acc", "dyn_mode"):
        assert torch.equal(env_a.state(f), env_b.state(f)), f
    exp = ref.rollout(DYN, steps)
    check_episode(env_a, ref, g64, exp)
    assert_switches(ref)


# 5. live mode with a per-chunk speed table
def _live_case(dtype):
    N, steps, V = 64 * 9 + 21, 75, 30
    P = dict(LIVE, track_history=1)
    (env,), ref = make(N, P, "ragged", n_traces=5, V=V)
    tid, off = sessions(N, 5, "smem")
    tid[64 * 4:64 * 6] = np.random.default_rng(2).integers(0, 5, size=128)     # two mixed blocks -> global path
    speed = np.random.default_rng(31).choice([0.75, 1.0, 1.0, 1.25, 1.5], size=(V, N))
    env.reset(tid, off)
    ref.reset(tid, off)
    want = ("delay", "sleep", "buffer", "rebuffer", "reward", "latency", "end_of_video", "actions")
    got = env.rollout("dynamic", steps, speed=speed, want=want, dtype=dtype)
    exp = ref.rollout(DYN, steps, speed=speed)
    assert_switches(ref)
    return env, ref, got, exp


def test_fused_live_episode_matches_oracle():
    env, ref, got, exp = _live_case(torch.float64)
    check_episode(env, ref, got, exp)
    assert_close(got["latency"].cpu().numpy(), exp["latency"], "latency")
    for f in ("t_now", "play_time", "play_len"):
        assert bits_equal(env.state(f).cpu().numpy(), ref.field(f)) == 0, f


def test_fused_live_episode_with_fp32_outputs():
    env, ref, got, exp = _live_case(torch.float32)
    assert np.array_equal(got["actions"].cpu().numpy(), exp["actions"])
    for kg, kc in TRAJ + (("latency", "latency"),):
        assert got[kg].dtype == torch.float32
        assert np.array_equal(got[kg].cpu().numpy(), exp[kc].astype(np.float32)), kg
    assert bits_equal(env.session_acc().cpu().numpy(), exp["acc"]) == 0
    check_state(env, ref)


# 6. the per-step decision
@pytest.mark.parametrize("live", [False, True])
def test_policy_decide_then_step_equals_the_fused_episode(live):
    N, steps = 1500, 70
    P = dict(track_history=1, track_acc=1, **(LIVE if live else {}))
    (env_a, env_b), ref = make(N, P, "ragged", n_env=2)
    tid, off = sessions(N, 12, "global")
    speed = np.random.default_rng(5).choice([0.8, 1.0, 1.25], size=(48, N)) if live else None
    for e in (env_a, env_b, ref):
        e.reset(tid, off)
    want = ("delay", "sleep", "buffer", "rebuffer", "reward", "end_of_video", "actions")
    whole = env_a.rollout("dynamic", steps, speed=speed, want=want)
    act = torch.empty(N, dtype=torch.int32, device="cuda")
    for t in range(steps):
        env_b.policy_decide("dynamic", out=act)
        exp_act = ref.policy_decide(DYN)
        assert np.array_equal(act.cpu().numpy(), exp_act), t
        assert np.array_equal(env_b.state("dyn_mode").cpu().numpy(), ref.dyn_mode), t
        assert torch.equal(act, whole["actions"][t]), t
        again = env_b.policy_decide("dynamic")                       # a repeated decision changes nothing
        assert torch.equal(again, act) and np.array_equal(env_b.state("dyn_mode").cpu().numpy(), ref.dyn_mode), t
        r = env_b.step(act, want_next_sizes=False, speed=speed)
        ref.step(exp_act, want_next_sizes=False, speed=speed)
        assert torch.equal(r.reward, whole["reward"][t]) and torch.equal(r.buffer, whole["buffer"][t]), t
        assert torch.equal(r.delay, whole["delay"][t]) and torch.equal(r.end_of_video, whole["end_of_video"][t]), t
    for f in ("seg", "chunk", "last_q", "phase", "pos", "buffer", "hist_len", "bw_hist", "acc", "dyn_mode"):
        assert torch.equal(env_a.state(f), env_b.state(f)), f
    check_state(env_b, ref)
    assert_switches(ref)
    assert env_a.error_count() == 0 and env_b.error_count() == 0


# 7. trace-sorted session order
def test_trace_sorted_order_equals_the_callers_order():
    N, steps = 3000, 60
    (env_a, env_b), ref = make(N, dict(track_history=1), "ragged", n_traces=37, T=96, n_env=2)
    tid = (np.arange(N) % 37).astype(np.int32)
    off = np.random.default_rng(3).uniform(0, 150.0, size=N)
    env_a.reset(tid, off, session_base=500)
    env_b.reset(tid, off, session_base=500, sort_by_trace=True)
    ref.reset(tid, off)
    out_a = env_a.rollout("dynamic", steps)
    out_b = env_b.rollout("dynamic", steps)
    for k in out_a:
        assert torch.equal(out_a[k], env_b.to_caller_order(out_b[k])), k
    for f in ("seg", "chunk", "last_q", "phase", "pos", "buffer", "hist_len", "dyn_mode"):
        assert torch.equal(env_a.state(f), env_b.to_caller_order(env_b.state(f))), f
    assert torch.equal(env_a.state("acc"), env_b.to_caller_order(env_b.state("acc")))
    a1 = env_a.policy_decide("dynamic")
    assert torch.equal(a1, env_b.to_caller_order(env_b.policy_decide("dynamic")))
    assert torch.equal(env_a.state("dyn_mode"), env_b.to_caller_order(env_b.state("dyn_mode")))
    exp = ref.rollout(DYN, steps)
    assert np.array_equal(out_a["actions"].cpu().numpy(), exp["actions"])
    assert_switches(ref)


# 8. the Simulator marker
@pytest.mark.parametrize("live", [False, True])
def test_simulator_marker_equals_the_env_path(live):
    bitrates, sizes, bw, tl, ti = small_world(n_traces=2, T=200, V=30)
    bw = phased(bw, seed=5)
    ctrl = DynamicPolicy(10.0, 5.0, 0.85, 6.0, 24.0)
    qoe = QOEMetric(4.3, 0.5, 2.0, 0.1)
    sim = Simulator(ctrl, None)
    sim.set_qoe_metric(qoe)
    nets = [NetworkInfo(1.0, list(bw[0])), NetworkInfo(0.5, list(bw[1][:60]))]
    sim.set_network_info(1.0, nets)
    sim.set_mpd(4.0, 24.0, 8.0 if live else None, [Chunk(list(b / 1000.0)) for b in bitrates])
    n = 128
    costs = sim.run_batch(n)
    P = dict(chunk_length=4.0, max_buffer=24.0, rebuf_penalty=4.3, smooth_penalty=0.5, utility_scale=1.0, rtt=0.0,
             payload=1.0, sleep_quantum=0.01, smooth_prev_ladder=1, latency_tick=0.01, default_quality=-1, auto_reset=0,
             track_history=1)
    if live:
        P.update(LIVE, track_acc=1)
    pp = dict(rb_safety=0.85, bola_min_buffer=6.0, bola_target_buffer=24.0)
    dp = dict(switch_on_buffer=10.0, switch_off_buffer=5.0)
    bw2 = np.ones((2, 200)); bw2[0] = bw[0]; bw2[1, :60] = bw[1][:60]
    tl2, ti2 = np.array([200, 60], np.int32), np.array([1.0, 0.5])
    env = BatchedABREnv(bw2, bitrates / 1000.0 * 4.0, bitrates / 1000.0, n, trace_len=tl2, trace_interval=ti2, **P)
    env.set_policy_params(**pp)
    env.set_dynamic_params(**dp)
    tid = ((np.arange(n) * 2) // n).astype(np.int32)
    off = None
    if live:
        env.reset(tid)
        env.rollout("dynamic", 30, want=())
        want = env.qoe_cost().cpu().numpy()
    else:
        want = env.run_host("dynamic", 30, tid, want_qoe_cost=True)["qoe_cost"]
    assert bits_equal(costs, want) == 0
    ref = do.DynamicEnv(bw2, tl2, ti2, bitrates / 1000.0 * 4.0, bitrates / 1000.0, n, **P)
    assert ref.set_policy_params(**pp) and ref.set_dynamic_params(**dp)
    ref.reset(tid, off)
    a = ref.rollout(DYN, 30)["acc"]
    exp = 4.3 * a[1] + 0.5 * a[3]
    if live:
        exp = exp + 2.0 * a[8] + 0.1 * a[9] / (0.01 * a[10])
    np.testing.assert_allclose(costs, exp, rtol=1e-12)
    assert_switches(ref)


# 9. errors, and their order
def test_errors():
    bitrates, sizes, bw, tl, ti = world("vbr", n_traces=4, T=64, V=10)
    N = 256
    tid = np.zeros(N, np.int32)
    act = torch.empty(N, dtype=torch.int32, device="cuda")
    zero = sizes.copy()
    zero[3, 0] = 0.0

    def expect(code, text, calls):
        for c in calls:
            with pytest.raises(_lib.AbrError) as ei:
                c()
            assert ei.value.code == code and text in str(ei.value), str(ei.value)

    def calls(e, pol="dynamic"):
        return [lambda: e.rollout(pol, 5), lambda: e.rollout(pol, 5, dtype=torch.float32),
                lambda: e.run(pol, 5, tid), lambda: e.run(pol, 0, tid), lambda: e.run_host(pol, 5, tid),
                lambda: e.policy_decide(pol, out=act)]

    plain = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti)        # track_history = 0
    plain.reset(tid)
    expect(4, "ABR_POLICY_DYNAMIC needs the throughput history", calls(plain))
    expect(4, "dyn_mode needs track_history = 1", [lambda: plain.state("dyn_mode")])
    both = BatchedABREnv(bw, zero, bitrates, N, trace_len=tl, trace_interval=ti)          # no history, a zero size
    both.reset(tid)
    expect(4, "track_history", calls(both))                                               # the history first
    envz = BatchedABREnv(bw, zero, bitrates, N, trace_len=tl, trace_interval=ti, track_history=1)
    envz.reset(tid)
    expect(1, "positive chunk sizes", calls(envz))
    envz.rollout("rate", 5)                                                               # RATE still runs there
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, track_history=1)
    env.reset(tid)
    assert (env.state("dyn_mode") == 0).all()                                             # zero at creation
    before = env.policy_decide("dynamic").clone()
    for bad in (dict(switch_on_buffer=float("nan")), dict(switch_off_buffer=float("inf")),
                dict(switch_on_buffer=6.0), dict(switch_on_buffer=3.0), dict(switch_off_buffer=-1.0)):
        expect(1, "switch_off_buffer < switch_on_buffer", [lambda: env.set_dynamic_params(**bad)])
    assert torch.equal(env.policy_decide("dynamic"), before)                              # nothing changed
    for bad in (6, -1):
        expect(1, f"unknown policy {bad}", calls(env, bad)[:5])
        expect(1, f"abr_env_policy_decide takes ABR_POLICY_BBA, _RATE or _BOLA (got {bad}), or ABR_POLICY_DYNAMIC",
               [lambda: env.policy_decide(bad, out=act)])
    assert env.error_count() == 0 and envz.error_count() == 0
    # every error case above still had data in which the rule switches both ways
    ref = do.DynamicEnv(bw, tl, ti, sizes, bitrates, N, track_history=1)
    ref.reset(np.arange(N, dtype=np.int32) % 4, np.random.default_rng(1).uniform(0, 60.0, size=N))
    ref.rollout(DYN, 30)
    assert_switches(ref)


# 10. full size
def test_full_size_sorted_by_trace_bit_exact_65536x48():
    N, steps = 65536, 48
    bitrates, sizes = synth.make_video(48)
    bw, tl, ti = synth.make_traces(1024, 2048)
    bw = phased(bw)
    tid, off = synth.make_sessions(N, 1024, 2048, group=1)
    P = dict(track_history=1)
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, **P)
    env.reset(tid, off, sort_by_trace=True)
    out = env.rollout("dynamic", steps)
    perm = env.perm.cpu().numpy()
    ref = do.DynamicEnv(bw, tl, ti, sizes, bitrates, N, **P)
    ref.reset(tid, off)
    exp = ref.rollout(DYN, steps)
    back = lambda t: env.to_caller_order(t).cpu().numpy()
    assert np.array_equal(back(out["actions"]), exp["actions"])
    for kg, kc in TRAJ:
        assert bits_equal(back(out[kg]), exp[kc]) == 0, kg
    assert np.array_equal(back(out["end_of_video"]), exp["eov"])
    assert bits_equal(back(env.session_acc()), exp["acc"]) == 0
    assert np.array_equal(back(env.state("chunk")), ref.field("chunk"))
    assert bits_equal(back(env.state("buffer")), ref.field("buffer")) == 0
    assert np.array_equal(back(env.state("dyn_mode")), ref.dyn_mode)
    assert sorted(perm.tolist()) == list(range(N))
    assert env.error_count() == 0
    assert_switches(ref)
