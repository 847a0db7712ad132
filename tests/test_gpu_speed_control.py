"""GPU parity of the catch-up speed control of live mode (SPEC §7.2) — in the per-step live step, the fused live
episode of every built-in policy, abr_env_run / abr_env_run_host and the Simulator façade — against the CPU oracle
(tests/speed_oracle.py on oracle/abr_oracle.c), bit for bit.  The traces alternate high and low bandwidth phases, and
every case checks in its own oracle run that the controller sped up, slowed down and held a speed-up back with the
buffer guard.  Run with -m gpu."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from abrsimulator_b200 import _lib
from abrsimulator_b200.datamodel import Chunk, NetworkInfo, QOEMetric
from abrsimulator_b200.env import BatchedABREnv
from abrsimulator_b200.simulator import BufferBasedPolicy, CatchupSpeedController, Simulator
from abrsimulator_b200.mpc import MPCBitrateController
from oracle import oracle as orc
from helpers import assert_close, bits_equal, small_world
import speed_oracle as sp
from test_gpu_dynamic import phased, sessions

POLICIES = dict(fixed=0, random=1, bba=2, rate=3, bola=4, dynamic=5)
TRAJ = (("delay", "delay"), ("sleep", "sleep"), ("buffer", "buffer"), ("rebuffer", "rebuf"), ("reward", "reward"),
        ("latency", "latency"))
LIVE = dict(live=1, start_up_length=8.0, max_buffer=20.0, startup_penalty=2.0, latency_penalty=0.1, track_history=1,
            track_acc=1)
CTL = dict(target_latency=14.0, max_drift=0.5, gain=2.5, dead_band=0.02, min_buffer=6.0)
STATE = ("seg", "chunk", "last_q", "trace_id", "hist_len", "play_id", "started", "done")
FSTATE = ("phase", "pos", "buffer", "t_now", "play_time", "play_len")


def world(n_traces=12, T=300, V=48):
    bitrates, sizes, bw, tl, ti = small_world(n_traces=n_traces, T=T, V=V)
    return bitrates, sizes, phased(bw), tl, ti


def make(N, params=None, n_env=1, ctl=CTL, **w):
    """n_env device environments and one oracle over the same world, with the controller installed on all."""
    P = dict(LIVE, **(params or {}))
    bitrates, sizes, bw, tl, ti = world(**w)
    envs = [BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, **P) for _ in range(n_env)]
    ref = sp.SpeedEnv(bw, tl, ti, sizes, bitrates, N, **{k: v for k, v in P.items() if k != "track_acc"})
    if ctl is not None:
        for e in envs:
            e.set_speed_control(**ctl)
        ref.set_speed_control(**ctl)
    return envs, ref


def covered(ref):
    up, down, guard = ref.counts()
    assert up > 0 and down > 0 and guard > 0, (up, down, guard)


def check_state(env, ref, order=None):
    back = (lambda t: t) if order is None else order
    for f in STATE:
        assert np.array_equal(back(env.state(f)).cpu().numpy(), ref.field(f)), f
    for f in FSTATE:
        assert bits_equal(back(env.state(f)).cpu().numpy(), ref.field(f)) == 0, f
    assert bits_equal(back(env.state("play_speed")).cpu().numpy(), ref.play_speed) == 0


def check_traj(got, exp, f32=False):
    for kg, kc in TRAJ:
        if kg in got:
            want = exp[kc].astype(np.float32) if f32 else exp[kc]
            assert bits_equal(got[kg].cpu().numpy().astype(np.float64), want.astype(np.float64)) == 0, kg
    if "end_of_video" in got:
        assert np.array_equal(got["end_of_video"].cpu().numpy(), exp["eov"])


# 1. the per-step live step, fp64 and fp32 outputs, both trace paths, auto_reset 0 and 1
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("layout", ["smem", "global"])
@pytest.mark.parametrize("auto_reset", [1, 0])
def test_per_step_live_matches_oracle(dtype, layout, auto_reset):
    N, steps = 3000, 60
    (env,), ref = make(N, dict(auto_reset=auto_reset))
    tid, off = sessions(N, 12, layout)
    env.reset(tid, off)
    ref.reset(tid, off)
    rng = np.random.default_rng(3)
    acc = np.zeros((orc.NUM_ACC, N))
    f32 = dtype == torch.float32
    for t in range(steps):
        a = rng.integers(0, 6, size=N).astype(np.int32)
        r = env.step(a, want_throughput=True, dtype=dtype)
        o = ref.step(a, acc=acc)
        for kg, kc in (("delay", "delay"), ("sleep", "sleep"), ("buffer", "buffer"), ("rebuffer", "rebuf"),
                       ("reward", "reward"), ("latency", "latency"), ("throughput", "throughput")):
            want = o[kc].astype(np.float32).astype(np.float64) if f32 else o[kc]
            assert bits_equal(getattr(r, kg).cpu().numpy().astype(np.float64), want) == 0, (t, kg)
        assert np.array_equal(r.end_of_video.cpu().numpy(), o["eov"])
        want_ns = o["next_sizes"].astype(np.float32) if f32 else o["next_sizes"]
        assert bits_equal(r.next_sizes.cpu().numpy().astype(np.float64), want_ns.astype(np.float64)) == 0
    check_state(env, ref)
    assert_close(env.session_acc().cpu().numpy(), acc, "acc")
    assert env.error_count() == 0 and ref.errors() == 0
    covered(ref)


# 2. the fused live episode of every built-in policy, fp64 and fp32 outputs
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("policy", list(POLICIES))
def test_fused_live_episode_matches_oracle(policy, dtype):
    N, steps = 2048, 60
    (env,), ref = make(N, dict(auto_reset=1 if dtype == torch.float64 else 0))
    tid, off = sessions(N, 12, "smem" if policy in ("bba", "rate") else "global")
    env.reset(tid, off)
    ref.reset(tid, off)
    actions = np.random.default_rng(5).integers(0, 6, size=(steps, N)).astype(np.int32) if policy == "fixed" else None
    want = ("delay", "sleep", "buffer", "rebuffer", "reward", "latency", "end_of_video", "actions")
    got = env.rollout(policy, steps, seed=7, actions=actions, want=want, dtype=dtype)
    exp = ref.rollout(POLICIES[policy], steps, seed=7, actions=actions)
    assert np.array_equal(got["actions"].cpu().numpy(), exp["actions"])
    check_traj(got, exp, f32=dtype == torch.float32)
    assert_close(env.session_acc().cpu().numpy(), exp["acc"], "acc")
    check_state(env, ref)
    np.testing.assert_allclose(env.stats().cpu().numpy(), orc.stats_from_acc(exp["acc"]), rtol=1e-9)
    assert env.error_count() == 0 and ref.errors() == 0
    covered(ref)


# 3. split episodes: the decision of the chunk being played carries from one call to the next
@pytest.mark.parametrize("policy", ["bba", "dynamic"])
def test_split_episode_equals_one_episode(policy):
    N = 2048
    (env_a, env_b), ref = make(N, n_env=2)
    tid, off = sessions(N, 12, "global")
    for e in (env_a, env_b, ref):
        e.reset(tid, off)
    one = env_a.rollout(policy, 48, seed=3)
    two = [env_b.rollout(policy, 24, seed=3) for _ in range(2)]
    for k in one:
        assert torch.equal(one[k], torch.cat([two[0][k], two[1][k]])), k
    for f in STATE + FSTATE + ("play_speed",):
        assert torch.equal(env_a.state(f), env_b.state(f)), f
    ref.rollout(POLICIES[policy], 48, seed=3)
    check_state(env_a, ref)
    covered(ref)


# 4. whole runs: abr_env_run and abr_env_run_host start fresh (the first piece of every session decides)
def test_run_and_run_host_equal_reset_and_rollout():
    N, steps = 3000, 48
    (env_a, env_b), ref = make(N, n_env=2)
    tid, off = sessions(N, 12, "smem")
    env_a.reset(tid, off)
    exp = env_a.rollout("bba", steps)
    acc = env_a.session_acc().cpu().numpy()
    cost = env_a.qoe_cost().cpu().numpy()
    speed = env_a.state("play_speed").clone()
    out, c2, _ = env_b.run("bba", steps, tid, off, want=("reward", "buffer", "end_of_video"))
    for k in out:
        assert torch.equal(out[k], exp[k]), k
    assert bits_equal(c2.cpu().numpy(), cost) == 0 and bits_equal(env_b.session_acc().cpu().numpy(), acc) == 0
    assert torch.equal(env_b.state("play_speed"), speed)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    for host_in in (lambda a: a, pin):
        h = env_b.run_host("bba", steps, host_in(tid), host_in(off), want_qoe_cost=True, want_reward_traj=True)
        assert bits_equal(np.asarray(h["acc"]), acc) == 0 and bits_equal(np.asarray(h["qoe_cost"]), cost) == 0
        assert bits_equal(np.asarray(h["reward"]), exp["reward"].cpu().numpy()) == 0
        assert torch.equal(env_b.state("play_speed"), speed)
    ref.reset(tid, off)
    r = ref.rollout(orc.POLICY_BBA, steps)
    assert bits_equal(acc, r["acc"]) == 0 and bits_equal(speed.cpu().numpy(), ref.play_speed) == 0
    covered(ref)


# 5. session order: sorted by trace against the caller's order, play_speed kept in environment order
def test_sorted_and_installed_orders_equal_the_callers_order():
    N, steps = 3000, 48
    (env_a, env_b, env_c), ref = make(N, n_env=3, n_traces=37, T=96)
    tid = (np.arange(N) % 37).astype(np.int32)
    off = np.random.default_rng(3).uniform(0, 150.0, size=N)
    env_a.reset(tid, off)
    env_b.reset(tid, off, sort_by_trace=True)
    perm = np.random.default_rng(4).permutation(N).astype(np.int32)
    env_c.set_order(perm)
    env_c.reset(tid[perm], off[perm])                          # inputs in environment order under an installed order
    ref.reset(tid, off)
    out_a = env_a.rollout("bba", steps)
    out_b = env_b.rollout("bba", steps)
    out_c = env_c.rollout("bba", steps)
    for k in out_a:
        assert torch.equal(out_a[k], env_b.to_caller_order(out_b[k])), k
        assert torch.equal(out_a[k], env_c.to_caller_order(out_c[k])), k
    for e in (env_b, env_c):   # per-step too
        a = torch.from_numpy(np.random.default_rng(9).integers(0, 6, size=N).astype(np.int32)).cuda()
        e.step(e.to_env_order(a))
    env_a.step(torch.from_numpy(np.random.default_rng(9).integers(0, 6, size=N).astype(np.int32)).cuda())
    for f in STATE + FSTATE + ("play_speed",):
        assert torch.equal(env_a.state(f), env_b.to_caller_order(env_b.state(f))), f
        assert torch.equal(env_a.state(f), env_c.to_caller_order(env_c.state(f))), f
    ref.rollout(orc.POLICY_BBA, steps)
    ref.step(np.random.default_rng(9).integers(0, 6, size=N).astype(np.int32))
    check_state(env_a, ref)
    covered(ref)


# 6. installing and removing the controller in the middle of an episode (SPEC §7.2)
def test_install_and_remove_mid_episode():
    N = 3000
    (env,), ref = make(N, ctl=None)
    tid, off = sessions(N, 12, "global")
    env.reset(tid, off)
    ref.reset(tid, off)
    rng = np.random.default_rng(6)
    table = rng.choice([0.8, 1.0, 1.25], size=(env.V, N))
    for t in range(48):
        if t == 10:
            env.set_speed_control(**CTL)
            ref.set_speed_control(**CTL)
        if t == 30:
            env.set_speed_control(None)
            ref.set_speed_control(None)
        a = rng.integers(0, 6, size=N).astype(np.int32)
        v = table if t >= 30 and t % 2 else None
        r = env.step(a, speed=None if v is None else torch.from_numpy(v).cuda())
        o = ref.step(a, speed=v)
        for kg, kc in TRAJ:
            assert bits_equal(getattr(r, kg).cpu().numpy(), o[kc]) == 0, (t, kg)
    check_state(env, ref)
    assert env.error_count() == 0
    covered(ref)


# 7. identities: an endless dead band is the live step without a table; a logged episode replays through the table
def test_an_endless_dead_band_is_the_live_step_without_a_table():
    N = 4096
    (env_a, env_b), _ = make(N, n_env=2, ctl=None)
    env_a.set_speed_control(dead_band=1e300)
    tid, off = sessions(N, 12, "smem")
    for e in (env_a, env_b):
        e.reset(tid, off)
    x, y = env_a.rollout("rate", 30), env_b.rollout("rate", 30)
    for k in x:
        assert torch.equal(x[k], y[k]), k
    a = torch.from_numpy(np.random.default_rng(1).integers(0, 6, size=N).astype(np.int32)).cuda()
    for _ in range(20):
        r, s = env_a.step(a), env_b.step(a)
        for k in ("delay", "sleep", "buffer", "rebuffer", "reward", "latency"):
            assert torch.equal(getattr(r, k), getattr(s, k)), k
    for f in STATE + FSTATE + ("acc",):
        assert torch.equal(env_a.state(f), env_b.state(f)), f


@pytest.mark.parametrize("auto_reset,steps", [(0, 60), (1, 48)])
def test_the_logged_decisions_replay_through_the_table(auto_reset, steps):
    N = 4096
    (env_ctl, env_tab), ref = make(N, dict(auto_reset=auto_reset), n_env=2)
    env_tab.set_speed_control(None)
    log = ref.start_log()
    tid, off = sessions(N, 12, "global")
    for e in (env_ctl, env_tab, ref):
        e.reset(tid, off)
    actions = np.random.default_rng(auto_reset).integers(0, 6, size=(steps, N)).astype(np.int32)
    for t in range(steps):
        ref.step(actions[t])
    covered(ref)
    table = torch.from_numpy(log).cuda()
    for t in range(steps):
        a = torch.from_numpy(actions[t]).cuda()
        r, s = env_ctl.step(a), env_tab.step(a, speed=table)
        for k in ("delay", "sleep", "buffer", "rebuffer", "reward", "latency", "end_of_video"):
            assert torch.equal(getattr(r, k), getattr(s, k)), (t, k)
    for f in STATE + FSTATE + ("acc",):
        assert torch.equal(env_ctl.state(f), env_tab.state(f)), f
    check_state(env_ctl, ref)


# 8. the Simulator marker on the three live paths: MPC, the built-in policy markers, callback controllers
class _Cycle:
    def get_next_bitrate(self, chunk_id, previous_bitrates, previous_bandwidths, buffer_level):
        return chunk_id % 4


@pytest.mark.parametrize("path", ["mpc", "marker", "callback"])
def test_simulator_marker_equals_the_env_path(path):
    bitrates, sizes, bw, tl, ti = small_world(n_traces=2, T=200, V=30)
    bw = phased(bw, seed=5)
    ctrl = dict(mpc=MPCBitrateController(horizon=4, mode="robust"), marker=BufferBasedPolicy(4.0, 8.0), callback=_Cycle())[path]
    spd = CatchupSpeedController(10.0, 0.4, 2.0, 0.05, 5.0)
    qoe = QOEMetric(4.3, 0.5, 2.0, 0.1)
    nets = [NetworkInfo(1.0, list(bw[0])), NetworkInfo(0.5, list(bw[1][:60]))]
    costs = {}
    for s in (spd, None):
        sim = Simulator(ctrl, s)
        sim.set_qoe_metric(qoe)
        sim.set_network_info(1.0, nets)
        sim.set_mpd(4.0, 24.0, 8.0, [Chunk(list(b / 1000.0)) for b in bitrates])
        costs[s is None] = sim.run_batch(128)
    assert not np.array_equal(costs[False], costs[True])       # the controller changed the runs
    P = dict(chunk_length=4.0, max_buffer=24.0, rebuf_penalty=4.3, smooth_penalty=0.5, utility_scale=1.0, rtt=0.0,
             payload=1.0, sleep_quantum=0.01, smooth_prev_ladder=1, latency_tick=0.01, default_quality=-1, auto_reset=0,
             live=1, start_up_length=8.0, startup_penalty=2.0, latency_penalty=0.1, track_acc=1, track_history=1,
             bba_reservoir=4.0, bba_cushion=8.0)
    bw2 = np.ones((2, 200)); bw2[0] = bw[0]; bw2[1, :60] = bw[1][:60]
    tl2, ti2 = np.array([200, 60], np.int32), np.array([1.0, 0.5])
    n = 128
    env = BatchedABREnv(bw2, bitrates / 1000.0 * 4.0, bitrates / 1000.0, n, trace_len=tl2, trace_interval=ti2, **P)
    env.set_speed_control(**vars(spd))
    tid = ((np.arange(n) * 2) // n).astype(np.int32)
    env.reset(tid)
    if path == "mpc":
        for _ in range(30):
            env.step(env.mpc_decide(4, "robust"), want_next_sizes=False)
    elif path == "marker":
        env.rollout("bba", 30, want=())
    else:
        for k in range(30):
            env.step(np.full(n, k % 4, np.int32), want_next_sizes=False)
    assert bits_equal(costs[False], env.qoe_cost().cpu().numpy()) == 0
    if path == "marker":
        ref = sp.SpeedEnv(bw2, tl2, ti2, bitrates / 1000.0 * 4.0, bitrates / 1000.0, n,
                          **{k: v for k, v in P.items() if k != "track_acc"})
        ref.set_speed_control(**vars(spd))
        ref.reset(tid)
        a = ref.rollout(orc.POLICY_BBA, 30)["acc"]
        exp = 4.3 * a[1] + 0.5 * a[3] + 2.0 * a[8] + 0.1 * a[9] / (0.01 * a[10])
        np.testing.assert_allclose(costs[False], exp, rtol=1e-12)
        up, down, _ = ref.counts()
        assert up > 0 and down > 0


# 9. errors, and their order
def test_errors():
    bitrates, sizes, bw, tl, ti = world(n_traces=4, T=64, V=10)
    N = 256
    live = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, **LIVE)
    vod = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti)
    lib = live._lib
    bad = _lib.AbrSpeedParams()
    lib.abr_speed_params_default(bad)
    bad.max_drift = 1.0
    good = _lib.AbrSpeedParams()
    lib.abr_speed_params_default(good)
    # invalid parameters come first, then a NULL env, then live = 0
    assert lib.abr_env_set_speed_control(vod._h, bad) == 1 and b"max_drift" in lib.abr_last_error()
    assert lib.abr_env_set_speed_control(None, good) == 1 and b"env is NULL" in lib.abr_last_error()
    assert lib.abr_env_set_speed_control(vod._h, good) == 4 and b"live" in lib.abr_last_error()
    assert lib.abr_env_set_speed_control(vod._h, None) == 4
    with pytest.raises(_lib.AbrError):
        vod.set_speed_control()
    with pytest.raises(_lib.AbrError):
        live.set_speed_control(gain=0.0)
    with pytest.raises(TypeError):
        live.set_speed_control(gian=1.0)
    # play_speed exists on live environments only
    p = np.zeros(1, np.uintp)
    assert lib.abr_env_state_ptr(vod._h, 25, _lib._addr(p)) == 4
    assert lib.abr_env_state_ptr(live._h, 25, _lib._addr(p)) == 0 and p[0] != 0
    # a table together with the controller: the C-ABI after the reset check, before any device work; Python first
    tid = np.zeros(N, np.int32)
    live.set_speed_control(**CTL)
    act = torch.zeros(N, dtype=torch.int32, device="cuda")
    table = torch.ones(live.V, N, dtype=torch.float64, device="cuda")
    out = torch.empty(N, dtype=torch.float64, device="cuda")
    assert lib.abr_env_step_live(live._h, _lib._addr(act), _lib._addr(table), *[None] * 9, None) == 4   # not reset
    live.reset(tid)
    assert torch.count_nonzero(live.state("play_speed")) == 0   # zero at creation; a reset does not touch it
    before = live.state("t_now").clone()
    assert lib.abr_env_step_live(live._h, _lib._addr(act), _lib._addr(table), _lib._addr(out), *[None] * 8,
                                 None) == 1
    assert b"exclusive" in lib.abr_last_error()
    assert lib.abr_env_rollout_fused_live(live._h, 2, 0, 4, None, _lib._addr(table), *[None] * 8, None) == 1
    assert lib.abr_env_rollout_fused_f32(live._h, 2, 0, 4, None, _lib._addr(table), *[None] * 8, None) == 1
    assert lib.abr_env_step_f32(live._h, _lib._addr(act), _lib._addr(table), *[None] * 9, None) == 1
    assert torch.equal(live.state("t_now"), before)
    with pytest.raises(ValueError, match="exclusive"):
        live.step(act, speed=table)
    with pytest.raises(ValueError, match="exclusive"):
        live.rollout("bba", 4, speed=table)
    live.set_speed_control(None)
    live.step(act, speed=table)                                  # removed: the table plays again
    assert live.error_count() == 0


# 10. full size, sorted by trace
def test_full_size_65536x48_bit_exact():
    N, steps = 65536, 48
    (env,), ref = make(N, n_traces=64, T=300)
    tid = np.random.default_rng(2).integers(0, 64, size=N).astype(np.int32)
    off = np.random.default_rng(3).uniform(0, 300.0, size=N)
    env.reset(tid, off, sort_by_trace=True)
    ref.reset(tid, off)
    got = env.rollout("bba", steps, want=("delay", "buffer", "rebuffer", "reward", "latency", "actions"))
    exp = ref.rollout(orc.POLICY_BBA, steps)
    back = env.to_caller_order
    assert np.array_equal(back(got["actions"]).cpu().numpy(), exp["actions"])
    for kg, kc in (("delay", "delay"), ("buffer", "buffer"), ("rebuffer", "rebuf"), ("reward", "reward"),
                   ("latency", "latency")):
        assert bits_equal(back(got[kg]).cpu().numpy(), exp[kc]) == 0, kg
    assert_close(back(env.session_acc()).cpu().numpy(), exp["acc"], "acc")
    check_state(env, ref, order=back)
    covered(ref)
