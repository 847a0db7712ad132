"""GPU parity of the chunk-step kernels (per-step and fused episode), through the C-ABI — run with -m gpu.

Oracle: oracle/abr_oracle.c (SPEC.md restated; its live-mode dynamics pinned by the reference's own tick loop,
tests/golden/sim_ref_tick_golden.json — test_kernels_are_the_limit_of_the_references_own_tick_loop).
Bar: 1e-9 relative (BASELINE.json) — and, because both sides execute the same IEEE operations in the
same order without FMA contraction, bit-identical.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from abrsimulator_b200 import synth
from abrsimulator_b200.env import BatchedABREnv, StepResult
from abrsimulator_b200.datamodel import Chunk, NetworkInfo, QOEMetric
from abrsimulator_b200.simulator import Simulator, BufferBasedPolicy, RandomPolicy
from abrsimulator_b200.mpc import MPCBitrateController
from abrsimulator_b200 import _lib
from oracle import oracle as orc
from helpers import (small_world, assert_close, bits_equal, load_step_golden, speed_table, load_ref_tick_golden,
                     ref_tick_params, ref_tick_world, check_against_ref_tick)

STATE_I = ("seg", "chunk", "last_q", "trace_id")
STATE_F = ("phase", "pos", "buffer")


def make_pair(N, params=None, **world):
    params = params or {}
    bitrates, sizes, bw, tl, ti = small_world(**world)
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, **params)
    ref = orc.OracleEnv(bw, tl, ti, sizes, bitrates, N, **params)
    n_traces, T = bw.shape
    rng = np.random.default_rng(11)
    tid = rng.integers(0, n_traces, size=N).astype(np.int32)
    off = rng.uniform(0, T * float(np.max(ti)) * 1.5, size=N)
    off[:4] = [0.0, float(ti[tid[1]]), 1e-9, 3.0 * float(ti[tid[3]])]   # segment boundaries
    env.reset(tid, off)
    ref.reset(tid, off)
    return env, ref


def check_state(env, ref):
    for f in STATE_I:
        assert np.array_equal(env.state(f).cpu().numpy(), ref.field(f)), f
    for f in STATE_F:
        assert bits_equal(env.state(f).cpu().numpy(), ref.field(f)) == 0, f


@pytest.mark.parametrize("ragged", [False, True])
def test_step_matches_oracle_over_two_episodes(ragged):
    N, steps = 4096, 100                       # 48-chunk video: crosses two end-of-video resets
    env, ref = make_pair(N, dict(track_history=1), ragged=ragged)
    check_state(env, ref)
    rng = np.random.default_rng(3)
    for t in range(steps):
        a = rng.integers(0, env.A, size=N).astype(np.int32)
        got = env.step(a, want_throughput=True)
        exp = ref.step(a)
        assert_close(got.delay.cpu().numpy(), exp["delay"], f"delay@{t}")
        assert_close(got.sleep.cpu().numpy(), exp["sleep"], f"sleep@{t}")
        assert_close(got.buffer.cpu().numpy(), exp["buffer"], f"buffer@{t}")
        assert_close(got.rebuffer.cpu().numpy(), exp["rebuf"], f"rebuf@{t}")
        assert_close(got.reward.cpu().numpy(), exp["reward"], f"reward@{t}")
        assert_close(got.throughput.cpu().numpy(), exp["throughput"], f"thr@{t}")
        assert_close(got.next_sizes.cpu().numpy(), exp["next_sizes"], f"next_sizes@{t}")
        assert np.array_equal(got.end_of_video.cpu().numpy(), exp["eov"])
        if t in (47, 48, 95, 96):
            assert got.end_of_video.sum().item() == (N if t in (47, 95) else 0)
    check_state(env, ref)
    assert np.array_equal(env.state("hist_len").cpu().numpy(), ref.field("hist_len"))
    assert env.error_count() == 0 and ref.errors() == 0


def test_sleep_cap_and_rebuffer_paths_are_exercised():
    """Fast network + lowest bitrate fills the buffer past max_buffer (sleep); slow network rebuffers."""
    N = 512
    env, ref = make_pair(N, dict(max_buffer=12.0, sleep_quantum=0.5), n_traces=8, T=64)
    slept = rebuffered = 0
    for t in range(40):
        a = np.full(N, 0 if t < 20 else env.A - 1, np.int32)
        got = env.step(a)
        exp = ref.step(a)
        for k_g, k_c in (("delay", "delay"), ("sleep", "sleep"), ("buffer", "buffer"), ("rebuffer", "rebuf"),
                         ("reward", "reward")):
            assert_close(getattr(got, k_g).cpu().numpy(), exp[k_c], f"{k_g}@{t}")
        slept += int((exp["sleep"] > 0).sum())
        rebuffered += int((exp["rebuf"] > 0).sum())
        assert float(got.buffer.max()) <= 12.0 + 1e-12
    assert slept > 1000 and rebuffered > 100
    check_state(env, ref)


def test_no_auto_reset_sessions_become_inert():
    N = 256
    env, ref = make_pair(N, dict(auto_reset=0, track_acc=1), V=6)
    for t in range(9):
        a = np.full(N, t % env.A, np.int32)
        got = env.step(a)
        exp = ref.step(a)
        assert_close(got.reward.cpu().numpy(), exp["reward"], f"reward@{t}")
        assert_close(got.buffer.cpu().numpy(), exp["buffer"], f"buffer@{t}")
        assert_close(got.next_sizes.cpu().numpy(), exp["next_sizes"], f"next@{t}")
        assert np.array_equal(got.end_of_video.cpu().numpy(), exp["eov"])
        if t >= 6:
            assert float(got.delay.abs().sum()) == 0.0
    assert np.array_equal(env.state("done").cpu().numpy(), np.ones(N, np.uint8))
    acc = env.session_acc().cpu().numpy()
    assert np.all(acc[6] == 6.0) and np.all(acc[7] == 1.0)


@pytest.mark.parametrize("policy", ["random", "bba", "fixed"])
def test_fused_rollout_matches_oracle(policy):
    N, steps = 4096, 60
    env, ref = make_pair(N, dict(track_history=1), ragged=(policy == "bba"))
    acts = np.random.default_rng(9).integers(0, env.A, size=(steps, N)).astype(np.int32) if policy == "fixed" else None
    got = env.rollout(policy, steps, seed=0xDEADBEEFCAFE, actions=acts)
    pid = dict(random=orc.POLICY_RANDOM, bba=orc.POLICY_BBA, fixed=orc.POLICY_FIXED)[policy]
    exp = ref.rollout(pid, steps, seed=0xDEADBEEFCAFE, actions=acts)
    assert np.array_equal(got["actions"].cpu().numpy(), exp["actions"])
    for k_g, k_c in (("delay", "delay"), ("sleep", "sleep"), ("buffer", "buffer"), ("rebuffer", "rebuf"),
                     ("reward", "reward")):
        assert_close(got[k_g].cpu().numpy(), exp[k_c], k_g)
    assert np.array_equal(got["end_of_video"].cpu().numpy(), exp["eov"])
    assert_close(env.session_acc().cpu().numpy(), exp["acc"], "acc")
    check_state(env, ref)
    stats = env.stats().cpu().numpy()
    exp_stats = orc.stats_from_acc(exp["acc"])
    np.testing.assert_allclose(stats, exp_stats, rtol=1e-9)
    assert stats[6] == N * steps and stats[7] == N            # counts are exact
    assert env.error_count() == 0


@pytest.mark.parametrize("ragged", [False, True])
def test_fused_rollout_shared_memory_trace_path(ragged):
    """Blocks of 64 consecutive sessions on one trace take the shared-memory staged path; blocks with mixed
    traces (and the last, partial block) take the global path — both must match the oracle bit for bit."""
    N, steps = 64 * 40 + 17, 60
    bitrates, sizes, bw, tl, ti = small_world(n_traces=12, T=300, ragged=ragged)
    params = dict(track_history=1)
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, **params)
    ref = orc.OracleEnv(bw, tl, ti, sizes, bitrates, N, **params)
    rng = np.random.default_rng(21)
    tid = ((np.arange(N) // 64) % 12).astype(np.int32)
    tid[64 * 30:64 * 36] = rng.integers(0, 12, size=64 * 6)        # six mixed blocks -> global path
    off = rng.uniform(0, 900.0, size=N)
    env.reset(tid, off)
    ref.reset(tid, off)
    got = env.rollout("random", steps, seed=99)
    exp = ref.rollout(orc.POLICY_RANDOM, steps, seed=99)
    assert np.array_equal(got["actions"].cpu().numpy(), exp["actions"])
    for k_g, k_c in (("delay", "delay"), ("sleep", "sleep"), ("buffer", "buffer"), ("rebuffer", "rebuf"),
                     ("reward", "reward")):
        assert_close(got[k_g].cpu().numpy(), exp[k_c], k_g)
    assert_close(env.session_acc().cpu().numpy(), exp["acc"], "acc")
    check_state(env, ref)
    assert bits_equal(env.state("bw_hist").cpu().numpy().T[:, :], ref.field("bw_hist")) == 0
    assert env.error_count() == 0


@pytest.mark.parametrize("T", [6000, 30000])
def test_long_traces_take_the_opt_in_shared_memory_path_or_fall_back(T):
    """6 000 segments need 77 KB (fused) / 48 KB (per-step) of shared memory per block: the opt-in path;
    30 000 segments do not fit and run on the global path.  Both must match the oracle bit for bit."""
    N, steps = 256 * 3 + 40, 24
    bitrates, sizes, bw, tl, ti = small_world(n_traces=3, T=T, V=12)
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti)
    ref = orc.OracleEnv(bw, tl, ti, sizes, bitrates, N)
    tid = ((np.arange(N) // 256) % 3).astype(np.int32)
    off = np.random.default_rng(2).uniform(0, float(T), size=N)
    off[:8] = T - 1e-3                                   # downloads that run past the end of the trace period
    for fused in (True, False):
        env.reset(tid, off)
        ref.reset(tid, off)
        if fused:
            got = env.rollout("random", steps, seed=11)
            exp = ref.rollout(orc.POLICY_RANDOM, steps, seed=11)
            for k_g, k_c in (("delay", "delay"), ("sleep", "sleep"), ("buffer", "buffer"), ("rebuffer", "rebuf"),
                             ("reward", "reward")):
                assert_close(got[k_g].cpu().numpy(), exp[k_c], k_g)
        else:
            rng = np.random.default_rng(3)
            for t in range(steps):
                a = rng.integers(0, env.A, size=N).astype(np.int32)
                g, e = env.step(a), ref.step(a)
                assert_close(g.delay.cpu().numpy(), e["delay"], f"delay@{t}")
                assert_close(g.buffer.cpu().numpy(), e["buffer"], f"buffer@{t}")
                assert_close(g.reward.cpu().numpy(), e["reward"], f"reward@{t}")
        check_state(env, ref)
    assert env.error_count() == 0 and ref.errors() == 0


def test_fused_rollout_key_search_with_equal_keys():
    """The shared-memory path searches on the high words of the capacity table; a trace whose capacities are tiny
    next to its running total gives long runs of equal keys, which the exact 64-bit scan must settle."""
    N, steps = 64 * 6, 40
    bitrates, sizes, bw, tl, ti = small_world(n_traces=3, T=50)
    bw = bw.copy()
    bw[0, :] = 1e-2
    bw[0, 0] = 1e6                       # C[j] = 9.5e5 + j * 9.5e-3: one key for the whole trace
    bw[1, :] = 0.3
    bw[1, 7] = 4e4
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti)
    ref = orc.OracleEnv(bw, tl, ti, sizes, bitrates, N)
    tid = ((np.arange(N) // 64) % 3).astype(np.int32)
    off = np.random.default_rng(8).uniform(0, 200.0, size=N)
    env.reset(tid, off)
    ref.reset(tid, off)
    got = env.rollout("random", steps, seed=5)
    exp = ref.rollout(orc.POLICY_RANDOM, steps, seed=5)
    for k_g, k_c in (("delay", "delay"), ("sleep", "sleep"), ("buffer", "buffer"), ("rebuffer", "rebuf"),
                     ("reward", "reward")):
        assert_close(got[k_g].cpu().numpy(), exp[k_c], k_g)
    check_state(env, ref)
    assert env.error_count() == 0 and ref.errors() == 0


@pytest.mark.parametrize("ragged", [False, True])
@pytest.mark.parametrize("fast", [False, True])
def test_step_kernel_shared_memory_trace_path(ragged, fast):
    """Per-step kernel: a block walks consecutive tiles of 128 sessions; tiles on one trace use the staged
    capacity row (restaged when the trace changes between tiles), mixed tiles and the partial last tile included."""
    N, steps = 256 * 11 + 100, 30
    bitrates, sizes, bw, tl, ti = small_world(n_traces=9, T=400, ragged=ragged)
    params = dict(track_history=0 if fast else 1, track_acc=0 if fast else 1)
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, **params)
    ref = orc.OracleEnv(bw, tl, ti, sizes, bitrates, N, **params)
    rng = np.random.default_rng(5)
    tid = ((np.arange(N) // 512) % 9).astype(np.int32)             # two tiles per trace: a restage inside a block
    tid[256 * 5:256 * 6] = rng.integers(0, 9, size=256)            # one mixed tile -> global path, then staged again
    tid[256 * 8:256 * 9 + 7] = 3                                   # a trace change in the middle of a tile
    off = rng.uniform(0, 1200.0, size=N)
    env.reset(tid, off)
    ref.reset(tid, off)
    acc = np.zeros((orc.NUM_ACC, N))
    for t in range(steps):
        a = rng.integers(0, env.A, size=N).astype(np.int32)
        got = env.step(a)
        exp = ref.step(a, acc=acc)
        for k_g, k_c in (("delay", "delay"), ("sleep", "sleep"), ("buffer", "buffer"), ("rebuffer", "rebuf"),
                         ("reward", "reward")):
            assert_close(getattr(got, k_g).cpu().numpy(), exp[k_c], f"{k_g}@{t}")
        assert np.array_equal(got.end_of_video.cpu().numpy(), exp["eov"])
    check_state(env, ref)
    if not fast:
        assert_close(env.session_acc().cpu().numpy(), acc, "acc")
    assert env.error_count() == 0


@pytest.mark.parametrize("policy", ["random", "bba", "fixed"])
def test_fast_variant_of_the_fused_kernel(policy):
    """All six trajectory outputs, no action trace, no history, auto_reset on selects the kernel variant compiled
    without per-output null checks and inert bookkeeping (the bench shape): same results as the generic variant
    and as the oracle, over two episodes (crosses the end-of-video reset), on both trace paths."""
    N, steps = 64 * 20 + 9, 100
    bitrates, sizes, bw, tl, ti = small_world(n_traces=10, T=200)
    tid = ((np.arange(N) // 64) % 10).astype(np.int32)
    tid[64 * 12:64 * 15] = np.random.default_rng(2).integers(0, 10, size=64 * 3)     # mixed blocks: global path
    off = np.random.default_rng(3).uniform(0, 400.0, size=N)
    acts = np.random.default_rng(4).integers(0, 6, size=(steps, N)).astype(np.int32) if policy == "fixed" else None
    six = ("delay", "sleep", "buffer", "rebuffer", "reward", "end_of_video")
    outs = []
    for want in (six, six + ("actions",)):
        env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti)
        env.reset(tid, off)
        outs.append((env.rollout(policy, steps, seed=11, actions=acts, want=want), env.session_acc().clone(),
                     env.stats().clone(), {f: env.state(f).clone() for f in STATE_I + STATE_F}))
        assert env.error_count() == 0
    (fast, acc_f, st_f, state_f), (gen, acc_g, st_g, state_g) = outs
    for k in six:
        assert torch.equal(fast[k], gen[k]), k
    assert torch.equal(acc_f, acc_g) and torch.equal(st_f, st_g)
    for f in STATE_I + STATE_F:
        assert torch.equal(state_f[f], state_g[f]), f
    ref = orc.OracleEnv(bw, tl, ti, sizes, bitrates, N)
    ref.reset(tid, off)
    pid = dict(random=orc.POLICY_RANDOM, bba=orc.POLICY_BBA, fixed=orc.POLICY_FIXED)[policy]
    exp = ref.rollout(pid, steps, seed=11, actions=acts)
    for k_g, k_c in (("delay", "delay"), ("sleep", "sleep"), ("buffer", "buffer"), ("rebuffer", "rebuf"),
                     ("reward", "reward")):
        assert_close(fast[k_g].cpu().numpy(), exp[k_c], k_g)
    assert np.array_equal(fast["end_of_video"].cpu().numpy(), exp["eov"])
    assert_close(acc_f.cpu().numpy(), exp["acc"], "acc")


def test_fused_rollout_equals_stepwise():
    """Size-independent property: the fused episode is the per-step kernel applied `steps` times."""
    N, steps = 2048, 48
    env_a, _ = make_pair(N)
    env_b, _ = make_pair(N)
    got = env_a.rollout("random", steps, seed=5)
    acts = got["actions"]
    for t in range(steps):
        r = env_b.step(acts[t], want_next_sizes=False)
        assert torch.equal(r.reward, got["reward"][t]) and torch.equal(r.delay, got["delay"][t])
        assert torch.equal(r.buffer, got["buffer"][t])
    for f in STATE_I + STATE_F:
        assert torch.equal(env_a.state(f), env_b.state(f)), f


def test_sharded_random_rollout_equals_unsharded():
    """Sharding invariance (SPEC §4): two half shards draw the same actions and produce the same
    trajectories as one full run, and their statistics add up."""
    N, steps = 4096, 48
    bitrates, sizes, bw, tl, ti = small_world(n_traces=32, T=256)
    tid, off = synth.make_sessions(N, 32, 256)
    full = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti)
    full.reset(tid, off)
    ref = full.rollout("random", steps, seed=42, want=("reward", "actions"))
    parts = []
    stats = torch.zeros(_lib.NUM_STATS, dtype=torch.float64, device="cuda")
    for lo, hi in ((0, N // 2), (N // 2, N)):
        tid_s, off_s = synth.make_sessions(hi - lo, 32, 256, session_base=lo)
        assert np.array_equal(tid_s, tid[lo:hi]) and np.array_equal(off_s, off[lo:hi])
        e = BatchedABREnv(bw, sizes, bitrates, hi - lo, trace_len=tl, trace_interval=ti)
        e.reset(tid_s, off_s, session_base=lo)
        parts.append(e.rollout("random", steps, seed=42, want=("reward", "actions")))
        stats += e.stats()
    assert torch.equal(torch.cat([p["actions"] for p in parts], dim=1), ref["actions"])
    assert torch.equal(torch.cat([p["reward"] for p in parts], dim=1), ref["reward"])
    np.testing.assert_allclose(stats.cpu().numpy(), full.stats().cpu().numpy(), rtol=1e-12)


@pytest.mark.parametrize("mode", [0, 1])
def test_mpc_episode_matches_oracle(mode):
    """decide -> step loop over a whole video with the env-owned history ring and robust error state."""
    N, H = 192, 4
    params = dict(track_history=1, track_acc=1, hist_k=5)
    env, ref = make_pair(N, params, V=20, n_traces=8, T=64)
    for t in range(26):                         # crosses the end-of-video reset
        act, bj = env.mpc_decide(H, mode, want_score=True)
        act_ref, bj_ref = ref.mpc_decide(H, mode)
        assert np.array_equal(act.cpu().numpy(), act_ref), f"actions differ at chunk {t}"
        ok = ~np.isnan(bj_ref)
        assert bits_equal(bj.cpu().numpy()[ok], bj_ref[ok]) == 0
        got = env.step(act, want_next_sizes=False)
        exp = ref.step(act_ref, want_next_sizes=False)
        assert_close(got.reward.cpu().numpy(), exp["reward"], f"reward@{t}")
    check_state(env, ref)
    assert bits_equal(env.state("last_pred").cpu().numpy(), ref.field("last_pred")) == 0
    assert np.array_equal(env.state("err_len").cpu().numpy(), ref.field("err_len"))
    assert env.error_count() == 0 and ref.errors() == 0


def test_log_utility_mode_matches_oracle():
    """utility_mode = 1: U = ln(bitrate / top bitrate), the reference's log_bitrate_utility (mpc.py:99-102)."""
    N, steps = 1024, 30
    params = dict(utility_mode=1, track_history=1, rebuf_penalty=2.66, smooth_penalty=1.0)
    env, ref = make_pair(N, params, V=24)
    util_g = env.state("utility").cpu().numpy()
    bitr = small_world(V=24)[0]
    np.testing.assert_allclose(util_g, np.log(bitr / bitr[:, -1:]), rtol=1e-15, atol=0)
    assert np.all(util_g[:, -1] == 0.0) and np.all(util_g[:, 0] < 0.0)
    got = env.rollout("bba", steps)
    exp = ref.rollout(orc.POLICY_BBA, steps)
    assert np.array_equal(got["actions"].cpu().numpy(), exp["actions"])
    assert_close(got["reward"].cpu().numpy(), exp["reward"], "reward")
    for mode in (0, 1):
        act = env.mpc_decide(4, mode).cpu().numpy()
        act_ref, _ = ref.mpc_decide(4, mode)
        assert np.array_equal(act, act_ref)


LIVE = dict(live=1, start_up_length=8.0, max_buffer=16.0, latency_penalty=0.05, startup_penalty=1.0, track_acc=1)


@pytest.mark.parametrize("ragged", [False, True])
def test_live_mode_step_matches_oracle(ragged):
    """SPEC §7: live-edge gate, start-up latch, playback speed per played chunk as a second action, latency and its
    integral — over two videos."""
    N, steps = 2048, 70
    env, ref = make_pair(N, dict(LIVE, track_history=1), V=30, ragged=ragged)
    rng = np.random.default_rng(17)
    acc = np.zeros((orc.NUM_ACC, N))
    for t in range(steps):
        a = rng.integers(0, env.A, size=N).astype(np.int32)
        v = rng.choice([0.75, 1.0, 1.0, 1.25, 1.5], size=(30, N))      # the table may be rewritten between steps
        got = env.step(a, speed=v, want_throughput=True)
        exp = ref.step(a, speed=v, acc=acc)
        for k_g, k_c in (("delay", "delay"), ("sleep", "sleep"), ("buffer", "buffer"), ("rebuffer", "rebuf"),
                         ("reward", "reward"), ("latency", "latency"), ("throughput", "throughput")):
            assert_close(getattr(got, k_g).cpu().numpy(), exp[k_c], f"{k_g}@{t}")
        assert np.array_equal(got.end_of_video.cpu().numpy(), exp["eov"])
    check_state(env, ref)
    for f in ("t_now", "play_time", "play_len"):
        assert bits_equal(env.state(f).cpu().numpy(), ref.field(f)) == 0, f
    assert np.array_equal(env.state("started").cpu().numpy(), ref.field("started"))
    assert np.array_equal(env.state("play_id").cpu().numpy(), ref.field("play_id"))
    assert_close(env.session_acc().cpu().numpy(), acc, "acc")
    assert acc[8].min() > 0 and acc[9].min() > 0 and acc[10].min() > 0 and (acc[1] > 0).any()
    # session cost: rw*rebuf + vw*smooth + sw*startup + lw*average_latency, the reference's average_latency being the
    # latency integral over the playing time per tick and per second of content played (Simulator.py:83-86,179-180)
    want = 4.3 * acc[1] + 1.0 * acc[3] + 1.0 * acc[8] + 0.05 * (acc[9] / (0.01 * acc[10]))
    np.testing.assert_allclose(env.qoe_cost().cpu().numpy(), want, rtol=1e-12)
    assert env.error_count() == 0
    with pytest.raises(_lib.AbrError):
        BatchedABREnv(np.ones((1, 8)), np.ones((2, 3)), np.ones((2, 3)), 4, live=1, start_up_length=100.0)


@pytest.mark.parametrize("policy", ["random", "bba", "fixed"])
def test_fused_live_episode_matches_oracle(policy):
    """SPEC §7 in the fused episode: speed table [V][N], latency output, start-up / latency / played accumulators,
    sorted (shared-memory path) and mixed blocks; and the same episode step by step."""
    N, steps = 64 * 9 + 21, 75
    bitrates, sizes, bw, tl, ti = small_world(n_traces=5, T=300, V=30, ragged=(policy == "bba"))
    P = dict(LIVE, track_history=1)
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, **P)
    ref = orc.OracleEnv(bw, tl, ti, sizes, bitrates, N, **P)
    rng = np.random.default_rng(31)
    tid = ((np.arange(N) // 64) % 5).astype(np.int32)
    tid[64 * 4:64 * 6] = rng.integers(0, 5, size=128)            # two mixed blocks -> global path
    off = rng.uniform(0, 500.0, size=N)
    speed = rng.choice([0.75, 1.0, 1.0, 1.25, 1.5], size=(30, N))
    acts = rng.integers(0, env.A, size=(steps, N)).astype(np.int32) if policy == "fixed" else None
    pid = dict(random=orc.POLICY_RANDOM, bba=orc.POLICY_BBA, fixed=orc.POLICY_FIXED)[policy]
    env.reset(tid, off)
    ref.reset(tid, off)
    want = ("delay", "sleep", "buffer", "rebuffer", "reward", "latency", "end_of_video", "actions")
    got = env.rollout(policy, steps, seed=77, actions=acts, speed=speed, want=want)
    exp = ref.rollout(pid, steps, seed=77, actions=acts, speed=speed)
    assert np.array_equal(got["actions"].cpu().numpy(), exp["actions"])
    for k_g, k_c in (("delay", "delay"), ("sleep", "sleep"), ("buffer", "buffer"), ("rebuffer", "rebuf"),
                     ("reward", "reward"), ("latency", "latency")):
        assert_close(got[k_g].cpu().numpy(), exp[k_c], k_g)
    assert np.array_equal(got["end_of_video"].cpu().numpy(), exp["eov"])
    assert_close(env.session_acc().cpu().numpy(), exp["acc"], "acc")
    assert exp["acc"][8].min() > 0 and exp["acc"][9].min() > 0 and exp["acc"][10].min() > 0
    check_state(env, ref)
    for f in ("t_now", "play_time", "play_len"):
        assert bits_equal(env.state(f).cpu().numpy(), ref.field(f)) == 0, f
    assert np.array_equal(env.state("started").cpu().numpy(), ref.field("started"))
    assert np.array_equal(env.state("play_id").cpu().numpy(), ref.field("play_id"))
    # the same actions and speeds through the per-step kernel
    env.reset(tid, off)
    a_all = got["actions"]
    for t in range(steps):
        r = env.step(a_all[t], speed=speed)
        assert bits_equal(r.reward.cpu().numpy(), exp["reward"][t]) == 0, t
        assert bits_equal(r.latency.cpu().numpy(), exp["latency"][t]) == 0, t
    # statistics vector carries the three live sums
    st = env.stats().cpu().numpy()
    np.testing.assert_allclose(st[8:], [exp["acc"][8].sum(), exp["acc"][9].sum(), exp["acc"][10].sum()], rtol=1e-9)
    assert env.error_count() == 0
    # without a speed table every session plays at speed 1
    env.reset(tid, off)
    ref.reset(tid, off)
    g1 = env.rollout(policy, 12, seed=5, actions=None if acts is None else acts[:12], want=("reward", "latency"))
    e1 = ref.rollout(pid, 12, seed=5, actions=None if acts is None else acts[:12])
    assert_close(g1["latency"].cpu().numpy(), e1["latency"], "latency(speed 1)")


def test_simulator_facade_live_mode():
    """The reference's Simulator is a live simulator: MPD with start_up_length, speed controller, latency weight."""
    bitrates, sizes, bw, tl, ti = small_world(n_traces=1, T=200, V=20)

    class Speed:
        def __init__(self):
            self.n = 0

        def get_next_speed(self):
            self.n += 1
            return 1.25 if self.n > 10 else 1.0

    class Second:
        def get_next_bitrate(self, chunk_id, previous_bitrates, previous_bandwidths, buffer_level):
            return 1

    sp = Speed()
    sim = Simulator(Second(), sp)
    sim.set_qoe_metric(QOEMetric(4.3, 0.5, 2.0, 0.1))
    sim.set_network_info(1.0, list(bw[0]))
    sim.set_mpd(4.0, 16.0, 8.0, [Chunk(list(b / 1000.0)) for b in bitrates])
    cost = sim.run()
    assert sp.n == 20
    # the façade's defaults are the reference's environment: no RTT, no payload factor, own-ladder variance term
    P = dict(chunk_length=4.0, max_buffer=16.0, rebuf_penalty=4.3, smooth_penalty=0.5, utility_scale=1.0, rtt=0.0,
             payload=1.0, sleep_quantum=0.01, smooth_prev_ladder=1, latency_tick=0.01,
             default_quality=-1, auto_reset=0, live=1, start_up_length=8.0, startup_penalty=2.0, latency_penalty=0.1)
    ref = orc.OracleEnv(bw, tl, ti, bitrates / 1000.0 * 4.0, bitrates / 1000.0, 1, **P)
    ref.reset(np.zeros(1, np.int32))
    acc = np.zeros((orc.NUM_ACC, 1))
    table = np.array([1.25 if k >= 10 else 1.0 for k in range(20)])[:, None]     # speed of the k-th played chunk
    for k in range(20):
        ref.step(np.ones(1, np.int32), speed=table, acc=acc)
    want = 4.3 * acc[1, 0] + 0.5 * acc[3, 0] + 2.0 * acc[8, 0] + 0.1 * acc[9, 0] / (0.01 * acc[10, 0])
    assert cost == pytest.approx(want, rel=1e-12) and acc[8, 0] > 0 and acc[9, 0] > 0
    assert sim.last_run["startup"][0] == acc[8, 0]
    # built-in policy markers and the MPC controller also run in live mode
    for ctrl in (BufferBasedPolicy(), RandomPolicy(5), MPCBitrateController(horizon=3, mode="robust")):
        sim2 = Simulator(ctrl, None)
        sim2.set_qoe_metric(QOEMetric(4.3, 0.5, 2.0, 0.1))
        sim2.set_network_info(1.0, [NetworkInfo(1.0, list(bw[0])), NetworkInfo(0.5, list(bw[0][:60]))])
        sim2.set_mpd(4.0, 16.0, 8.0, [Chunk(list(b / 1000.0)) for b in bitrates])
        costs = sim2.run_batch(64)
        assert costs.shape == (64,) and np.all(np.isfinite(costs)) and np.all(costs > 0)
        if isinstance(ctrl, BufferBasedPolicy):     # one fused live episode: compare with the oracle's
            bw2 = np.ones((2, 200)); bw2[0] = bw[0]; bw2[1, :60] = bw[0][:60]
            ref2 = orc.OracleEnv(bw2, np.array([200, 60], np.int32), np.array([1.0, 0.5]), bitrates / 1000.0 * 4.0,
                                 bitrates / 1000.0, 64, **dict(P, smooth_penalty=0.5, bba_reservoir=ctrl.reservoir,
                                                               bba_cushion=ctrl.cushion))
            ref2.reset(((np.arange(64) * 2) // 64).astype(np.int32))
            a2 = ref2.rollout(orc.POLICY_BBA, 20)["acc"]
            np.testing.assert_allclose(costs, 4.3 * a2[1] + 0.5 * a2[3] + 2.0 * a2[8] + 0.1 * a2[9] / (0.01 * a2[10]),
                                       rtol=1e-12)


def test_run_host_path_matches_oracle():
    N, steps = 3000, 48
    bitrates, sizes, bw, tl, ti = small_world(n_traces=32, T=256)
    tid, off = synth.make_sessions(N, 32, 256)
    env = BatchedABREnv(bw, sizes, bitrates, 4096, trace_len=tl, trace_interval=ti)
    out = env.run_host("bba", steps, tid, off, want_reward_traj=True, want_qoe_cost=True)
    ref = orc.OracleEnv(bw, tl, ti, sizes, bitrates, N)
    ref.reset(tid, off)
    exp = ref.rollout(orc.POLICY_BBA, steps)
    assert_close(out["acc"], exp["acc"], "acc")
    assert_close(out["reward"], exp["reward"], "reward")
    np.testing.assert_allclose(out["stats"], orc.stats_from_acc(exp["acc"]), rtol=1e-9)
    # per-session QoE cost of Simulator.calculate_qoe (Simulator.py:83-86), computed on the device
    assert_close(out["qoe_cost"], 4.3 * exp["acc"][1] + 1.0 * exp["acc"][3], "qoe_cost")


def test_invalid_inputs_are_flagged_or_rejected():
    bitrates, sizes, bw, tl, ti = small_world(n_traces=4, T=32)
    env = BatchedABREnv(bw, sizes, bitrates, 64, trace_len=tl, trace_interval=ti)
    env.reset(np.zeros(64, np.int32))
    a = np.zeros(64, np.int32)
    a[5], a[9] = -1, 99
    env.step(a)
    assert env.error_count() == 2
    with pytest.raises(_lib.AbrError):
        env.reset(np.zeros(65, np.int32))                       # over capacity
    bad = bw.copy()
    bad[1, 3] = 0.0
    with pytest.raises(_lib.AbrError):
        BatchedABREnv(bad, sizes, bitrates, 8, trace_len=tl, trace_interval=ti)   # zero bandwidth (D14 analogue)
    with pytest.raises(_lib.AbrError):
        BatchedABREnv(bw, -sizes, bitrates, 8, trace_len=tl, trace_interval=ti)
    with pytest.raises(ValueError):
        env.step(np.zeros(3, np.int32))


def test_edge_shapes_empty_batch_single_chunk_video_and_widest_ladder():
    """Empty batch (legal no-op), a one-chunk video (end of video on every step), the widest supported ladder
    (A = 16, runtime-A MPC path) and the longest history ring (K = 64)."""
    bitrates, sizes, bw, tl, ti = small_world(n_traces=4, T=64)
    env = BatchedABREnv(bw, sizes, bitrates, 16, trace_len=tl, trace_interval=ti)
    with pytest.raises(_lib.AbrError):
        env.rollout("bba", 4)                                  # reset has not been called
    env.reset(np.zeros(0, np.int32))
    out = env.rollout("bba", 4)
    assert out["reward"].shape == (4, 0)
    assert env.step(np.zeros(0, np.int32)).reward.numel() == 0
    assert float(env.stats().abs().sum()) == 0.0 and env.mpc_decide(3, "robust").numel() == 0
    # one-chunk video
    env1, ref1 = make_pair(128, dict(track_acc=1), V=1)
    for t in range(3):
        a = np.full(128, t % 6, np.int32)
        got, exp = env1.step(a), ref1.step(a)
        assert_close(got.reward.cpu().numpy(), exp["reward"], "reward")
        assert bool((got.end_of_video == 1).all())
    assert np.all(env1.session_acc().cpu().numpy()[7] == 3.0)
    # A = 16, K = 64
    lad = tuple(float(x) for x in np.linspace(200, 8000, 16))
    params = dict(track_history=1, hist_k=64)
    env16, ref16 = make_pair(256, params, V=20, ladder=lad)
    for t in range(5):
        act = env16.mpc_decide(2, t % 2)
        act_ref, _ = ref16.mpc_decide(2, t % 2)
        assert np.array_equal(act.cpu().numpy(), act_ref)
        got, exp = env16.step(act, want_next_sizes=True), ref16.step(act_ref)
        assert_close(got.next_sizes.cpu().numpy(), exp["next_sizes"], "next_sizes")
    with pytest.raises(_lib.AbrError):
        env16.mpc_decide(8, 0)                                 # 16^8 sequences exceed the 2^31-1 index range
    with pytest.raises(_lib.AbrError):
        BatchedABREnv(bw, np.ones((4, 17)), np.ones((4, 17)), 8)                      # A > 16
    with pytest.raises(_lib.AbrError):
        BatchedABREnv(bw, sizes, bitrates, 8, trace_len=tl, trace_interval=ti, hist_k=65)


def test_calls_are_cuda_graph_capturable():
    """Device-pointer entry points never synchronise or allocate, so reset + fused episode + statistics can be
    captured into a CUDA graph and replayed with identical results."""
    import ctypes as C
    N, steps = 4096, 24
    bitrates, sizes, bw, tl, ti = small_world(n_traces=16, T=128)
    tid, off = synth.make_sessions(N, 16, 128, group=64)
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti)
    tid_d, off_d = torch.from_numpy(tid).cuda(), torch.from_numpy(off).cuda()
    out = {k: torch.empty(steps, N, dtype=torch.float64, device="cuda") for k in
           ("delay", "sleep", "buffer", "rebuffer", "reward")}
    out["end_of_video"] = torch.empty(steps, N, dtype=torch.uint8, device="cuda")
    stats = torch.empty(_lib.NUM_STATS, dtype=torch.float64, device="cuda")

    def one():
        env.reset(tid_d, off_d)
        env.rollout("bba", steps, out=out)
        _lib.check(env._lib.abr_stats_partial(env._h, C.c_void_p(stats.data_ptr()),
                                              C.c_void_p(torch.cuda.current_stream().cuda_stream)))

    one()
    torch.cuda.synchronize()
    ref_reward, ref_stats = out["reward"].clone(), stats.clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        one()
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        one()
    out["reward"].zero_()
    stats.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out["reward"], ref_reward) and torch.equal(stats, ref_stats)


@pytest.mark.parametrize("group", [64, 1])
def test_full_size_bit_exact_against_the_c_oracle_65536x48(group):
    """BASELINE configs[1] at its full size, every one of the 65 536 x 48 x 6 outputs, the final state and the
    per-session sums against oracle/abr_oracle.c: bit-identical.  group = 64: the benchmark's layout (every block
    follows one trace: shared-memory path); group = 1: trace = session mod n_traces (global path)."""
    N, steps = 65536, 48
    bitrates, sizes = synth.make_video(48)
    bw, tl, ti = synth.make_traces(1024, 2048)
    tid, off = synth.make_sessions(N, 1024, 2048, group=group)
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti)
    out, cost, stats = env.run("random", steps, tid, off, seed=20260101)
    ref = orc.OracleEnv(bw, tl, ti, sizes, bitrates, N)
    ref.reset(tid, off)
    exp = ref.rollout(orc.POLICY_RANDOM, steps, seed=20260101)
    for kg, kc in (("delay", "delay"), ("sleep", "sleep"), ("buffer", "buffer"), ("rebuffer", "rebuf"), ("reward", "reward")):
        assert bits_equal(out[kg].cpu().numpy(), exp[kc]) == 0, kg
    assert np.array_equal(out["end_of_video"].cpu().numpy(), exp["eov"])
    assert bits_equal(env.session_acc().cpu().numpy(), exp["acc"]) == 0
    check_state(env, ref)
    np.testing.assert_allclose(stats.cpu().numpy(), orc.stats_from_acc(exp["acc"]), rtol=1e-9)
    assert env.error_count() == 0


def test_full_size_properties_65536x48():
    """BASELINE config 2 at full size: properties that need no oracle."""
    N, steps = 65536, 48
    bitrates, sizes = synth.make_video(48)
    bw, tl, ti = synth.make_traces(1024, 2048)
    tid, off = synth.make_sessions(N, 1024, 2048, group=64)
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti)
    env.reset(tid, off)
    out = env.rollout("random", steps, seed=7)
    assert env.error_count() == 0
    d, sl, b, rb, rw, q = (out[k] for k in ("delay", "sleep", "buffer", "rebuffer", "reward", "actions"))
    assert bool((d > 0.08).all()) and bool((rb >= 0).all()) and bool((sl >= 0).all())
    assert float(b.max()) <= 60.0 and float(b.min()) >= 4.0 - 1e-12        # buffer in [L, max_buffer]
    assert bool((out["end_of_video"][-1] == 1).all()) and int(out["end_of_video"][:-1].sum()) == 0
    # buffer recursion: b_t = max(b_{t-1} - delay, 0) + L - sleep
    prev = torch.cat([torch.zeros(1, N, dtype=torch.float64, device="cuda"), b[:-1]])
    assert torch.equal(torch.clamp(prev - d, min=0.0) + 4.0 - sl, b)
    assert torch.equal(torch.clamp(d - prev, min=0.0), rb)
    # reward identity from the outputs
    U = torch.from_numpy(bitrates * 0.001).cuda()
    u = U[torch.arange(steps, device="cuda")[:, None].expand(-1, N), q.long()]
    last = torch.cat([torch.ones(1, N, dtype=torch.int64, device="cuda"), q[:-1].long()])
    up = U[torch.arange(steps, device="cuda")[:, None].expand(-1, N), last]
    assert torch.equal((u - 4.3 * rb) - 1.0 * (u - up).abs(), rw)
    # physics, independent of the capacity table: the bandwidth integral over every download interval is the chunk
    # size.  The trace clock of a session advances by (delay - rtt) + sleep per step; integrate the raw square wave
    # in extended precision for a sample of sessions.
    sample = np.arange(0, N, 97)
    dn, sn, qn = (x[:, sample].cpu().numpy() for x in (d, sl, q))
    ld = np.longdouble
    worst = 0.0
    for c, s_idx in enumerate(sample):
        rate = bw[tid[s_idx]].astype(ld) * ld(0.95)
        Ccum = np.concatenate([[ld(0)], np.cumsum(rate)])            # interval = 1 s
        P = Ccum[-1]

        def F(t):                                                    # data deliverable in [0, t)
            n, r = divmod(t, ld(2048))
            j = int(r)
            return n * P + Ccum[j] + rate[j] * (r - j)
        t0 = ld(off[s_idx])
        for t in range(steps):
            dl = ld(dn[t, c]) - ld(0.08)
            got = F(t0 + dl) - F(t0)
            want = ld(sizes[t, qn[t, c]])
            worst = max(worst, float(abs(got - want) / want))
            t0 = t0 + dl + ld(sn[t, c])
    assert worst < 1e-9, worst
    # determinism: a second run from the same reset is bit-identical
    env.reset(tid, off)
    out2 = env.rollout("random", steps, seed=7, want=("reward",))
    assert torch.equal(out2["reward"], rw)
    # random actions are uniform over the ladder
    hist = torch.bincount(q.flatten().long(), minlength=6).double() / q.numel()
    assert float((hist - 1 / 6).abs().max()) < 2e-3


def test_simulator_facade_run():
    """Simulator API (Simulator.py:45-93): setters + run() -> QoE cost rw*rebuffer + vw*sum|dbitrate|."""
    bitrates, sizes, bw, tl, ti = small_world(n_traces=1, T=200, V=30)
    sim = Simulator(BufferBasedPolicy(), None)
    sim.set_qoe_metric(QOEMetric(4.3, 0.001, 0, 0))
    sim.set_network_info(1.0, list(bw[0]))
    sim.set_mpd(4.0, 60.0, None, [Chunk(list(b / 1000.0)) for b in bitrates])   # sizes = bitrate * chunk_length; no start_up_length: on-demand
    cost = sim.run()
    # the façade's defaults are the reference's environment (no RTT, no payload factor, tick-sized pause quantum)
    P = dict(chunk_length=4.0, max_buffer=60.0, rebuf_penalty=4.3, smooth_penalty=0.001, utility_scale=1.0,
             default_quality=-1, auto_reset=0, rtt=0.0, payload=1.0, sleep_quantum=0.01, smooth_prev_ladder=1)
    ref = orc.OracleEnv(bw, tl, ti, bitrates / 1000.0 * 4.0, bitrates / 1000.0, 1, **P)
    ref.reset(np.zeros(1, np.int32))
    exp = ref.rollout(orc.POLICY_BBA, 30)
    want = 4.3 * exp["acc"][1, 0] + 0.001 * exp["acc"][3, 0]
    assert cost == pytest.approx(want, rel=1e-12)

    class Lowest:                                   # generic controller protocol (Simulator.py:155)
        def __init__(self):
            self.calls = []

        def get_next_bitrate(self, chunk_id, previous_bitrates, previous_bandwidths, buffer_level):
            self.calls.append((chunk_id, len(previous_bitrates), len(previous_bandwidths), buffer_level))
            return 0

    ctl = Lowest()
    sim2 = Simulator(ctl, None)
    sim2.set_qoe_metric(QOEMetric(4.3, 0.001, 0, 0))
    sim2.set_network_info(NetworkInfo(1.0, list(bw[0])).interval, list(bw[0]))
    sim2.set_mpd(4.0, 60.0, None, [Chunk(list(b / 1000.0)) for b in bitrates])
    cost2 = sim2.run()
    assert len(ctl.calls) == 30 and ctl.calls[5][:3] == (5, 5, 5)
    ref.reset(np.zeros(1, np.int32))
    exp2 = ref.rollout(orc.POLICY_FIXED, 30, actions=np.zeros((30, 1), np.int32))
    assert cost2 == pytest.approx(4.3 * exp2["acc"][1, 0] + 0.001 * exp2["acc"][3, 0], rel=1e-12)
    # many sessions with the random policy
    sim3 = Simulator(RandomPolicy(3), None)
    sim3.set_qoe_metric(QOEMetric(4.3, 1.0, 0, 0))
    sim3.set_network_info(1.0, [NetworkInfo(1.0, list(bw[0])), NetworkInfo(0.5, list(bw[0][:50]))])
    sim3.set_mpd(4.0, 60.0, None, [Chunk(list(b / 1000.0)) for b in bitrates])
    costs = sim3.run_batch(100)
    assert costs.shape == (100,) and np.all(np.isfinite(costs)) and np.all(costs >= 0)


@pytest.mark.parametrize("case", load_step_golden(), ids=lambda c: c["name"])
def test_kernels_reproduce_the_step_spec_fixture(case):
    """Committed fixture (tests/golden/step_spec_golden.json): per-step kernel bit for bit, then — for the on-demand
    cases — the fused episode with the same action table."""
    N = len(case["trace_id"])
    P = dict(case["params"], track_acc=0)
    env = BatchedABREnv(case["bw"], case["sizes"], case["bitrates"], N, trace_len=case["tl"], trace_interval=case["ti"], **P)
    env.reset(case["trace_id"], case["start_offset"])
    live = bool(P.get("live"))
    for t, a in enumerate(case["actions"]):
        v = speed_table(case["speeds"], env.V, N)
        got = env.step(a, speed=v, want_throughput=True) if live else env.step(a, want_throughput=True)
        pairs = [("delay", "delay"), ("sleep", "sleep"), ("buffer", "buffer"), ("rebuffer", "rebuf"), ("reward", "reward"),
                 ("throughput", "throughput")] + ([("latency", "latency")] if live else [])
        for k_g, k_c in pairs:
            assert bits_equal(getattr(got, k_g).cpu().numpy(), case["outputs"][k_c][t]) == 0, (case["name"], t, k_g)
        assert np.array_equal(got.end_of_video.cpu().numpy(), case["eov"][t])
    assert np.array_equal(env.state("seg").cpu().numpy(), case["final"]["seg"])
    assert bits_equal(env.state("phase").cpu().numpy(), case["final"]["phase"]) == 0
    assert bits_equal(env.state("pos").cpu().numpy(), case["final"]["pos"]) == 0
    if live:
        assert np.array_equal(env.state("play_id").cpu().numpy(), case["final"]["play_id"])
        assert bits_equal(env.state("play_len").cpu().numpy(), case["final"]["play_len"]) == 0
        assert bits_equal(env.state("play_time").cpu().numpy(), case["final"]["play_time"]) == 0
    # the fused episode with the same action (and speed) table
    env.reset(case["trace_id"], case["start_offset"])
    want = ("delay", "sleep", "buffer", "rebuffer", "reward") + (("latency",) if live else ())
    tr = env.rollout("fixed", len(case["actions"]), actions=case["actions"], want=want,
                     speed=speed_table(case["speeds"], env.V, N) if live else None)
    for k_g in want:
        k_c = "rebuf" if k_g == "rebuffer" else k_g
        assert bits_equal(tr[k_g].cpu().numpy(), case["outputs"][k_c]) == 0, (case["name"], k_g)
    assert env.error_count() == 0


class _ScriptedAbr:
    """get_next_bitrate of the controller protocol (Simulator.py:155): a fixed action per chunk."""

    def __init__(self, actions):
        self.actions = list(actions)

    def get_next_bitrate(self, chunk_id, previous_bitrates, previous_bandwidths, buffer_level):
        return int(self.actions[chunk_id])


class _ScriptedSpeed:
    """get_next_speed (Simulator.py:177): the k-th call returns speeds[k mod len]."""

    def __init__(self, speeds):
        self.speeds, self.n = list(speeds), 0

    def get_next_speed(self):
        v = self.speeds[self.n % len(self.speeds)]
        self.n += 1
        return float(v)


def test_kernels_are_the_limit_of_the_references_own_tick_loop():
    """The reference-derived pin of the chunk-step path, on the CUDA side (see the test of the same name in
    tests/test_oracle_step.py): the 60 scripted live sessions that /root/reference/Simulator.py's own run() loop
    played (tests/golden/sim_ref_tick_golden.json), through (a) the per-step kernel, timer by timer and chunk by
    chunk, and (b) the drop-in ``Simulator`` façade with the reference's constructor / setters / controller protocol,
    whose ``run()`` must return the reference's QoE cost within the loop's discretisation."""
    doc = load_ref_tick_golden()
    worst = {"reference": {}, "reference_fine": {}}
    for sc in doc["cases"]:
        br, sizes, bw, speed = ref_tick_world(sc)
        V = sc["V"]
        for name, tick in (("reference", doc["dt"]), ("reference_fine", doc["dt_fine"])):
            env = BatchedABREnv(bw, sizes, br, 1, trace_interval=sc["interval"], track_acc=1, **ref_tick_params(sc, tick))
            env.reset([0], [0.0])
            t, reb, su, pt = np.zeros(V), np.zeros(V), np.zeros(V), np.zeros(V)
            for k in range(V):
                env.step([sc["actions"][k]], want_next_sizes=False, speed=speed)
                acc = env.session_acc().cpu().numpy()[:, 0]
                t[k], reb[k], su[k], pt[k] = env.state("t_now").item(), acc[1], acc[8], env.state("play_time").item()
            calls = int(env.state("play_id").item()) + (1 if env.state("play_len").item() > 0 else 0)
            dev = check_against_ref_tick(sc, name, tick, t, reb, su, pt, acc[3], acc[9], acc[10], calls)
            for k_, d in dev.items():
                worst[name][k_] = max(worst[name].get(k_, 0.0), float(d))
            assert env.error_count() == 0
            if name == "reference":
                # the drop-in façade: reference constructor, setters and controller protocol (Simulator.py:46-77,155,177)
                w = sc["weights"]
                spd = _ScriptedSpeed(sc["speeds"])
                sim = Simulator(_ScriptedAbr(sc["actions"]), spd)
                sim.set_qoe_metric(QOEMetric(*w))
                sim.set_network_info(sc["interval"], list(sc["bandwidths"]))
                sim.set_mpd(sc["chunk_length"], sc["max_buffer"], sc["start_up_length"], [Chunk(list(b)) for b in sc["bitrates"]])
                cost = sim.run()
                want = w[0] * acc[1] + w[1] * acc[3] + w[2] * acc[8] + w[3] * (acc[9] / (tick * acc[10]))
                assert cost == pytest.approx(want, rel=1e-12), sc["index"]       # same kernels, same numbers
                ref = sc["reference"]
                bound = (2 * V + 2) * tick
                tol = (w[0] + w[2]) * bound + w[3] * 0.01 * max(ref["final"]["average_latency"], 1.0) + 1e-9 * abs(ref["qoe"])
                assert abs(cost - ref["qoe"]) <= tol, (sc["index"], cost, ref["qoe"])
    for k_ in worst["reference"]:
        assert worst["reference_fine"][k_] <= worst["reference"][k_] / 4, (k_, worst)


@pytest.mark.parametrize("seed", range(6))
def test_randomized_worlds_match_oracle(seed):
    """Differential fuzz: 25 random worlds per seed — trace lengths 1..400, arbitrary (non power-of-two) intervals,
    bandwidths spanning six orders of magnitude, zero-size chunks, rtt 0, many-period downloads, ragged ladders —
    through the fused episode (sorted and shuffled sessions) and the per-step kernel."""
    rng = np.random.default_rng(1000 + seed)
    for w in range(25):
        n_traces = int(rng.integers(1, 6))
        T = int(rng.choice([1, 2, 3, 17, 64, 255, 400]))
        V = int(rng.integers(1, 14))
        A = int(rng.integers(1, 9))
        scale = 10.0 ** rng.uniform(-3, 3)
        bw = scale * 10.0 ** rng.uniform(-1.5, 1.5, size=(n_traces, T))
        tl = rng.integers(1, T + 1, size=n_traces).astype(np.int32)
        ti = rng.choice([0.25, 0.3, 0.5, 1.0, 1.7, 2.0], size=n_traces)
        bitrates = np.sort(rng.uniform(100.0, 5000.0, size=(V, A)), axis=1)
        sizes = bitrates / 1000.0 * 4.0 * rng.uniform(0.5, 1.5, size=(V, A)) * 10.0 ** rng.uniform(-1, 1)
        if rng.random() < 0.3:
            sizes[rng.integers(0, V), rng.integers(0, A)] = 0.0
        params = dict(rtt=float(rng.choice([0.0, 0.08])), payload=float(rng.choice([0.95, 1.0])),
                      max_buffer=float(rng.choice([8.0, 20.0, 60.0])), sleep_quantum=float(rng.choice([0.3, 0.5])),
                      default_quality=int(rng.integers(-1, A)), auto_reset=int(rng.integers(0, 2)))
        N = 64 * int(rng.integers(1, 5)) + int(rng.integers(0, 64))
        tid = np.sort(rng.integers(0, n_traces, size=N)).astype(np.int32)
        if w % 3 == 0:
            tid = rng.permutation(tid)
        off = rng.uniform(0, 3.0 * float(np.max(tl * ti)), size=N)
        steps = int(rng.integers(1, 2 * V + 3))
        env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, **params)
        ref = orc.OracleEnv(bw, tl, ti, sizes, bitrates, N, **params)
        tag = f"seed {seed} world {w}"
        env.reset(tid, off)
        ref.reset(tid, off)
        got = env.rollout("random", steps, seed=w)
        exp = ref.rollout(orc.POLICY_RANDOM, steps, seed=w)
        for k_g, k_c in (("delay", "delay"), ("sleep", "sleep"), ("buffer", "buffer"), ("rebuffer", "rebuf"),
                         ("reward", "reward")):
            assert bits_equal(got[k_g].cpu().numpy(), exp[k_c]) == 0, (tag, "fused", k_g)
        assert np.array_equal(got["end_of_video"].cpu().numpy(), exp["eov"]), tag
        check_state(env, ref)
        for t in range(min(steps, 6)):
            a = rng.integers(0, A, size=N).astype(np.int32)
            g, e = env.step(a), ref.step(a)
            for k_g, k_c in (("delay", "delay"), ("buffer", "buffer"), ("rebuffer", "rebuf"), ("reward", "reward")):
                assert bits_equal(getattr(g, k_g).cpu().numpy(), e[k_c]) == 0, (tag, "step", t, k_g)
        check_state(env, ref)
        # a download that needs more than 2^20 trace periods trips the same guard on both sides (SPEC §3.1)
        assert (env.error_count() == 0) == (ref.errors() == 0), tag


# ---- optional fp32-output mode (BASELINE.json: "1e-5 for an optional fp32 mode") ----
# The arithmetic and the state stay fp64, so the bar is tighter than 1e-5: every output equals the oracle's fp64 value
# rounded once to float (bit-identical to numpy's float64 -> float32 conversion), and the state matches bit for bit.
F32_RTOL = 1e-5


def _check_f32(got, exp, name):
    got = got.cpu().numpy()
    assert got.dtype == np.float32, name
    np.testing.assert_allclose(got.astype(np.float64), exp, rtol=F32_RTOL, atol=1e-30, err_msg=name)
    assert np.array_equal(got.view(np.uint32), exp.astype(np.float32).view(np.uint32)), f"{name}: not the rounded fp64 value"


@pytest.mark.parametrize("ragged", [False, True])
def test_step_f32_outputs_are_rounded_fp64(ragged):
    N, steps = 2048, 60
    env, ref = make_pair(N, dict(track_history=1, track_acc=1), ragged=ragged)
    rng = np.random.default_rng(5)
    acc = np.zeros((orc.NUM_ACC, N))
    for t in range(steps):
        a = rng.integers(0, env.A, size=N).astype(np.int32)
        got = env.step(a, want_throughput=True, dtype=torch.float32)
        exp = ref.step(a, acc=acc)
        for k_g, k_c in (("delay", "delay"), ("sleep", "sleep"), ("buffer", "buffer"), ("rebuffer", "rebuf"),
                         ("reward", "reward"), ("throughput", "throughput"), ("next_sizes", "next_sizes")):
            _check_f32(getattr(got, k_g), exp[k_c], f"{k_g}@{t}")
        assert np.array_equal(got.end_of_video.cpu().numpy(), exp["eov"])
    check_state(env, ref)                                  # fp64 state: no drift
    assert_close(env.session_acc().cpu().numpy(), acc, "acc")


def test_step_f32_fast_path():
    """Default parameters (no history, no accumulators): the specialised per-step kernel."""
    N = 4096
    env, ref = make_pair(N)
    rng = np.random.default_rng(6)
    for t in range(50):
        a = rng.integers(0, env.A, size=N).astype(np.int32)
        got = env.step(a, want_next_sizes=False, dtype=torch.float32)
        exp = ref.step(a)
        for k_g, k_c in (("delay", "delay"), ("sleep", "sleep"), ("buffer", "buffer"), ("rebuffer", "rebuf"),
                         ("reward", "reward")):
            _check_f32(getattr(got, k_g), exp[k_c], f"{k_g}@{t}")
        assert np.array_equal(got.end_of_video.cpu().numpy(), exp["eov"])
    check_state(env, ref)


@pytest.mark.parametrize("policy", ["random", "bba", "fixed"])
def test_fused_rollout_f32(policy):
    N, steps = 4096, 60
    env, ref = make_pair(N, ragged=(policy == "bba"))
    acts = np.random.default_rng(9).integers(0, env.A, size=(steps, N)).astype(np.int32) if policy == "fixed" else None
    want = ("delay", "sleep", "buffer", "rebuffer", "reward", "end_of_video") + (("actions",) if policy == "bba" else ())
    got = env.rollout(policy, steps, seed=77, actions=acts, want=want, dtype=torch.float32)
    pid = dict(random=orc.POLICY_RANDOM, bba=orc.POLICY_BBA, fixed=orc.POLICY_FIXED)[policy]
    exp = ref.rollout(pid, steps, seed=77, actions=acts)
    for k_g, k_c in (("delay", "delay"), ("sleep", "sleep"), ("buffer", "buffer"), ("rebuffer", "rebuf"),
                     ("reward", "reward")):
        _check_f32(got[k_g], exp[k_c], k_g)
    assert np.array_equal(got["end_of_video"].cpu().numpy(), exp["eov"])
    if "actions" in got:
        assert np.array_equal(got["actions"].cpu().numpy(), exp["actions"])
    check_state(env, ref)
    assert_close(env.session_acc().cpu().numpy(), exp["acc"], "acc")      # accumulators stay fp64
    np.testing.assert_allclose(env.stats().cpu().numpy(), orc.stats_from_acc(exp["acc"]), rtol=1e-12)


def test_f32_rejects_mixed_output_dtypes():
    env, _ = make_pair(64)
    out = dict(delay=torch.empty(4, 64, dtype=torch.float32, device=env.device),
               reward=torch.empty(4, 64, dtype=torch.float64, device=env.device))
    with pytest.raises(TypeError):
        env.rollout("random", 4, out=out)
    with pytest.raises(TypeError):
        env.step(np.zeros(64, np.int32), dtype=torch.float16)


def test_run_host_zero_copy_equals_staged_copies():
    """Page-locked host buffers are read and written by the kernels directly (device alias under unified addressing);
    pageable ones go through staged copies.  Both give the same bytes, mixed combinations included."""
    N, steps = 5000, 48
    bitrates, sizes, bw, tl, ti = small_world(n_traces=32, T=256)
    tid, off = synth.make_sessions(N, 32, 256)
    env = BatchedABREnv(bw, sizes, bitrates, 8192, trace_len=tl, trace_interval=ti)
    pageable = env.run_host("random", steps, tid, off, seed=5, want_qoe_cost=True)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()
    tid_p, off_p = pin(tid.astype(np.int32)), pin(off.astype(np.float64))
    assert tid_p.dtype == np.int32 and off_p.dtype == np.float64
    out = dict(qoe_cost=pin(np.full(N, np.nan)), stats=pin(np.full(_lib.NUM_STATS, np.nan)))
    pinned = env.run_host("random", steps, tid_p, off_p, seed=5, out=out)
    assert out["qoe_cost"] is pinned["qoe_cost"]
    for k in ("acc", "stats", "qoe_cost"):
        assert bits_equal(pinned[k], pageable[k]) == 0, k
    mixed = env.run_host("random", steps, tid_p, off, seed=5, out=dict(qoe_cost=pin(np.full(N, np.nan))))   # pinned ids, pageable offsets
    for k in ("acc", "stats", "qoe_cost"):
        assert bits_equal(mixed[k], pageable[k]) == 0, k
    # interior pointers of page-locked allocations (slices) alias correctly too
    big_t, big_o, big_c = pin(np.zeros(N + 11, np.int32)), pin(np.zeros(N + 5)), pin(np.full(N + 3, np.nan))
    big_t[11:] = tid
    big_o[5:] = off
    inner = env.run_host("random", steps, big_t[11:], big_o[5:], seed=5, out=dict(qoe_cost=big_c[3:]))
    for k in ("acc", "stats", "qoe_cost"):
        assert bits_equal(inner[k], pageable[k]) == 0, k
    assert np.isnan(big_c[:3]).all()
    none_off = env.run_host("random", steps, tid_p, None, seed=5, out=dict(stats=pin(np.full(_lib.NUM_STATS, np.nan))))
    ref = orc.OracleEnv(bw, tl, ti, sizes, bitrates, N)
    ref.reset(tid, None)
    exp = ref.rollout(orc.POLICY_RANDOM, steps, seed=5)
    assert_close(none_off["acc"], exp["acc"], "acc")
    np.testing.assert_allclose(none_off["stats"], orc.stats_from_acc(exp["acc"]), rtol=1e-9)


ALL_FIELDS = ("seg", "chunk", "last_q", "trace_id", "hist_len", "done", "err_len", "phase", "pos", "buffer", "last_pred",
              "t_now", "play_time", "started")


@pytest.mark.parametrize("params", [dict(), dict(track_history=1), dict(auto_reset=0), dict(live=1, start_up_length=8.0),
                                    dict(live=1, track_history=1, auto_reset=0)])
@pytest.mark.parametrize("policy", ["random", "bba"])
def test_run_host_fused_reset_equals_reset_then_rollout(params, policy):
    """abr_env_run_host resets the sessions inside the episode kernel; every state array, the accumulators, the
    statistics, the session cost and the error count must equal abr_env_reset followed by abr_env_rollout_fused —
    also when the environment held another, longer run before (stale state must not leak through)."""
    N, steps = 3000, 57                      # V = 48: crosses an end of video
    bitrates, sizes, bw, tl, ti = small_world(n_traces=32, T=256, ragged=True)
    tid, off = synth.make_sessions(N, 32, 256)
    tid = tid.astype(np.int32)
    tid[7], tid[100] = -3, 32                # invalid traces: flagged and replaced by trace 0 (SPEC §2)
    env_a = BatchedABREnv(bw, sizes, bitrates, 4096, trace_len=tl, trace_interval=ti, **params)
    env_b = BatchedABREnv(bw, sizes, bitrates, 4096, trace_len=tl, trace_interval=ti, **params)
    for env in (env_a, env_b):               # dirty both environments with an unrelated run
        env.reset((np.arange(4096) % 32).astype(np.int32), np.linspace(0.0, 300.0, 4096))
        env.rollout("random", 31, seed=99, want=())
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()
    for host in (lambda a: a, pin):          # staged copies, then zero-copy
        e0 = env_a.error_count()
        out = env_a.run_host(policy, steps, host(tid), host(off), seed=3, want_qoe_cost=True,
                             out=dict(qoe_cost=host(np.full(N, np.nan))))
        err_a = env_a.error_count() - e0
        e0 = env_b.error_count()
        env_b.reset(tid, off)
        env_b.rollout(policy, steps, seed=3, want=())
        err_b = env_b.error_count() - e0
        assert err_a == err_b == 2
        for f in ALL_FIELDS:
            a, b = env_a.state(f).cpu().numpy()[:N], env_b.state(f).cpu().numpy()[:N]
            assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), f
        assert bits_equal(out["acc"], env_b.session_acc().cpu().numpy()) == 0
        assert bits_equal(out["stats"], env_b.stats().cpu().numpy()) == 0
        assert bits_equal(out["qoe_cost"], env_b.qoe_cost().cpu().numpy()) == 0
    if params.get("track_history"):
        assert bits_equal(env_a.state("bw_hist").cpu().numpy(), env_b.state("bw_hist").cpu().numpy()) == 0


@pytest.mark.parametrize("policy", ["random", "bba", "fixed"])
def test_env_run_equals_reset_rollout_cost_stats(policy):
    """abr_env_run (one launch) against the four separate calls and against the oracle."""
    N, steps = 4000, 50
    bitrates, sizes, bw, tl, ti = small_world(n_traces=32, T=256)
    tid, off = synth.make_sessions(N, 32, 256, group=64)
    acts = np.random.default_rng(4).integers(0, 6, size=(steps, N)).astype(np.int32) if policy == "fixed" else None
    env_a = BatchedABREnv(bw, sizes, bitrates, 4096, trace_len=tl, trace_interval=ti)
    env_b = BatchedABREnv(bw, sizes, bitrates, 4096, trace_len=tl, trace_interval=ti)
    env_a.reset((np.arange(4096) % 32).astype(np.int32))
    env_a.rollout("bba", 20, want=())                       # stale state and accumulators
    out, cost, stats = env_a.run(policy, steps, tid, off, seed=21, session_base=1000, actions=acts)
    env_b.reset(tid, off, session_base=1000)
    exp = env_b.rollout(policy, steps, seed=21, actions=acts)
    for k in out:
        assert torch.equal(out[k], exp[k]), k
    assert torch.equal(cost, env_b.qoe_cost()) and torch.equal(stats, env_b.stats())
    for f in ALL_FIELDS:
        assert torch.equal(env_a.state(f)[:N], env_b.state(f)[:N]), f
    assert torch.equal(env_a.session_acc(), env_b.session_acc())
    ref = orc.OracleEnv(bw, tl, ti, sizes, bitrates, N)
    ref.reset(tid, off)
    pid = dict(random=orc.POLICY_RANDOM, bba=orc.POLICY_BBA, fixed=orc.POLICY_FIXED)[policy]
    o = ref.rollout(pid, steps, seed=21, session_base=1000, actions=acts)
    assert_close(out["reward"].cpu().numpy(), o["reward"], "reward")
    assert_close(out["delay"].cpu().numpy(), o["delay"], "delay")
    assert_close(cost.cpu().numpy(), 4.3 * o["acc"][1] + 1.0 * o["acc"][3], "qoe_cost")
    # empty run: a plain reset
    out0, cost0, stats0 = env_a.run(policy, 0, tid, off, actions=None if acts is None else acts[:0])
    assert float(cost0.abs().sum()) == 0.0 and float(stats0.abs().sum()) == 0.0
    assert np.array_equal(env_a.state("chunk").cpu().numpy()[:N], np.zeros(N, np.int32))


@pytest.mark.parametrize("N", [1, 63, 64, 65, 2049, 70001])
def test_statistics_inside_the_episode_kernel_for_awkward_batch_sizes(N):
    """abr_env_run with a statistics buffer reduces the statistics inside the episode kernel (block partials summed per
    group of 32 blocks by the group's last block, the groups by the last group): one block, a partial group, several
    groups (70 001 sessions = 1 094 blocks = 35 groups), repeated launches (the counters return to zero) — always the
    bits that abr_stats_partial produces afterwards from the same partials, and the oracle's sums."""
    steps = 20
    bitrates, sizes, bw, tl, ti = small_world(n_traces=32, T=128)
    tid, off = synth.make_sessions(N, 32, 128, group=64)
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti)
    for seed in (3, 4, 3):
        out, cost, stats = env.run("random", steps, tid, off, seed=seed)
        assert torch.equal(stats, env.stats()), seed          # the separate two-stage reduction: same order, same bits
        acc = env.session_acc().cpu().numpy()
        np.testing.assert_allclose(stats.cpu().numpy(), acc.sum(axis=1), rtol=1e-12)
        assert stats[6].item() == N * steps
    ref = orc.OracleEnv(bw, tl, ti, sizes, bitrates, N)
    ref.reset(tid, off)
    o = ref.rollout(orc.POLICY_RANDOM, steps, seed=3)
    np.testing.assert_allclose(stats.cpu().numpy(), orc.stats_from_acc(o["acc"]), rtol=1e-9)


def test_prepared_host_run_equals_run_host():
    N, steps = 2000, 48
    bitrates, sizes, bw, tl, ti = small_world(n_traces=16, T=128)
    tid, off = synth.make_sessions(N, 16, 128)
    env = BatchedABREnv(bw, sizes, bitrates, 2048, trace_len=tl, trace_interval=ti)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    tid_p, off_p = pin(tid.astype(np.int32)), pin(off)
    plan = env.prepare_run_host("random", steps, tid_p, off_p, seed=1, want_qoe_cost=True,
                                out=dict(qoe_cost=pin(np.zeros(N)), stats=pin(np.zeros(_lib.NUM_STATS))))
    for seed in (1, 2, 1):
        got = plan(seed=seed)
        exp = env.run_host("random", steps, tid, off, seed=seed, want_qoe_cost=True)
        assert bits_equal(got["acc"], exp["acc"]) == 0
        assert bits_equal(got["qoe_cost"].numpy(), exp["qoe_cost"]) == 0
        assert bits_equal(got["stats"].numpy(), exp["stats"]) == 0
    off_p += 3.0                                   # new inputs go into the prepared buffers in place
    got = plan()
    exp = env.run_host("random", steps, tid, off + 3.0, seed=1, want_qoe_cost=True)
    assert bits_equal(got["qoe_cost"].numpy(), exp["qoe_cost"]) == 0
    assert env.n == N


def test_trace_sorted_order_is_bit_identical_to_the_callers_order():
    """Sessions given interleaved over the traces (trace = session mod n_traces): an environment that keeps them sorted
    by trace (abr_sort_by_trace + abr_env_set_order) returns, mapped back through the order, exactly what the
    unsorted environment returns — fused random episode (the policy is keyed by the caller's index), per-step kernel,
    state and statistics."""
    N, steps = 3000, 30
    bitrates, sizes, bw, tl, ti = small_world(n_traces=37, T=96, ragged=True)
    tid = (np.arange(N) % 37).astype(np.int32)
    off = np.random.default_rng(3).uniform(0, 150.0, size=N)
    env_a = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, max_buffer=20.0)
    env_b = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, max_buffer=20.0)
    env_a.reset(tid, off, session_base=500)
    env_b.reset(tid, off, session_base=500, sort_by_trace=True)
    perm = env_b.perm.cpu().numpy()
    assert sorted(perm.tolist()) == list(range(N))
    assert np.all(np.diff(tid[perm]) >= 0)                              # sorted by trace ...
    same = np.diff(tid[perm]) == 0
    assert np.all(np.diff(perm)[same] > 0)                              # ... and stable within a trace
    out_a = env_a.rollout("random", steps, seed=11)
    out_b = env_b.rollout("random", steps, seed=11)
    for k in out_a:
        assert torch.equal(out_a[k], env_b.to_caller_order(out_b[k])), k
    acts = torch.from_numpy(np.random.default_rng(4).integers(0, bitrates.shape[1], size=(5, N)).astype(np.int32)).cuda()
    for t in range(5):
        ra = env_a.step(acts[t])
        rb = env_b.step(env_b.to_env_order(acts[t]).contiguous())
        for f in ("delay", "sleep", "buffer", "rebuffer", "reward", "end_of_video", "next_sizes"):
            xa, xb = getattr(ra, f), getattr(rb, f)
            if xb.dim() == 2:
                xb = env_b.to_caller_order(xb.t().contiguous()).t()
            else:
                xb = env_b.to_caller_order(xb)
            assert torch.equal(xa, xb), (t, f)
    for f in ("seg", "chunk", "last_q", "phase", "pos", "buffer"):
        assert torch.equal(env_a.state(f), env_b.to_caller_order(env_b.state(f))), f
    np.testing.assert_allclose(env_a.stats().cpu().numpy(), env_b.stats().cpu().numpy(), rtol=1e-12)
    assert env_a.error_count() == 0 and env_b.error_count() == 0
    # a batch of another size needs a new order
    with pytest.raises(_lib.AbrError):
        env_b.reset(tid[:100], off[:100])
    env_b.set_order(None)
    env_b.reset(tid[:100], off[:100])


@pytest.mark.parametrize("N,n_traces,T", [(70001, 1024, 8), (5000, 13000, 4), (1, 3, 16), (33, 1, 16)])
def test_reset_sorted_is_the_stable_sort_by_trace(N, n_traces, T):
    """abr_env_reset_sorted (counting sort by trace + gather + reset in one call; CUB's radix sort for the shapes the
    counting sort does not take: here more than 11 264 traces) installs the order abr_sort_by_trace computes — the
    stable sort — and resets every session exactly like abr_env_reset on the reordered inputs."""
    bitrates, sizes, bw, tl, ti = small_world(n_traces=n_traces, T=T)
    rng = np.random.default_rng(N)
    tid = rng.integers(0, n_traces, size=N).astype(np.int32)
    off = rng.uniform(0, 3.0 * T, size=N)
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti)
    env.reset(tid, off, sort_by_trace=True)
    perm = env.perm.cpu().numpy()
    assert np.array_equal(perm, np.argsort(tid, kind="stable").astype(np.int32))
    assert np.array_equal(perm, env.sort_by_trace(tid).cpu().numpy())
    ref = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti)
    ref.reset(tid[perm], off[perm])
    for f in STATE_I + STATE_F:
        assert torch.equal(env.state(f), ref.state(f)), f
    assert env.error_count() == 0
    env.reset(tid, None, sort_by_trace=True)                 # no start offsets
    assert float(env.state("phase").abs().sum()) == 0.0 and int(env.state("seg").abs().sum()) == 0


# ---- SPEC §4.1: policy-in-the-loop step (abr_env_step_policy) ----
def _philox4x32_10(c, k):
    """Philox4x32-10 on uint32 numpy arrays: counter words c[0..3], key words k[0..1] (SPEC §4)."""
    M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
    c = [np.asarray(x, np.uint64) for x in c]
    k0, k1 = np.uint64(k[0]), np.uint64(k[1])
    mask = np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0, p1 = c[0] * np.uint64(M0), c[2] * np.uint64(M1)
        c = [((p1 >> np.uint64(32)) ^ c[1] ^ k0) & mask, p1 & mask, ((p0 >> np.uint64(32)) ^ c[3] ^ k1) & mask, p0 & mask]
        k0, k1 = (k0 + np.uint64(W0)) & mask, (k1 + np.uint64(W1)) & mask
    return c


def _perturbed_logits(logits, seed, draw, session_base=0):
    """logits[a] - ln(-ln(u_a)) of SPEC §4.1 in float32 (numpy's logf; the device's differs in the last bits)."""
    N, A = logits.shape
    g = np.arange(N, dtype=np.uint64) + np.uint64(session_base)
    out = np.empty((N, A), np.float32)
    for b in range((A + 3) // 4):
        w = _philox4x32_10([g & np.uint64(0xFFFFFFFF), g >> np.uint64(32), np.full(N, draw, np.uint64), np.full(N, b, np.uint64)],
                           [seed & 0xFFFFFFFF, seed >> 32])
        for k in range(4):
            a = 4 * b + k
            if a < A:
                u = ((w[k] >> np.uint64(9)).astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -23)
                out[:, a] = logits[:, a] - np.log(-np.log(u)).astype(np.float32)
    return out


def test_step_policy_greedy_equals_step_with_argmax_and_writes_the_observation():
    N = 3000
    env_a, _ = make_pair(N, dict(track_history=0))
    env_b, _ = make_pair(N, dict(track_history=0))
    A = env_a.A
    rng = np.random.default_rng(5)
    scales = (0.1, 1e-3, 0.25, 1e-6)
    obs = torch.zeros(4 + A, N, dtype=torch.float32, device="cuda")
    act = torch.zeros(N, dtype=torch.int32, device="cuda")
    total = torch.zeros(N, dtype=torch.float64, device="cuda")
    total_b = np.zeros(N)
    for t in range(60):                          # crosses an end of video
        lg = rng.normal(size=(N, A)).astype(np.float32)
        lg[::7, 2] = lg[::7, 4] = lg[::7].max(axis=1)        # exact ties: the first arg max wins
        lg[5] = np.nan                                         # all NaN: action 0
        logits = torch.from_numpy(lg).cuda()
        res = StepResult(*[torch.empty(N, dtype=torch.float64, device="cuda") for _ in range(5)], None,
                         torch.empty(N, dtype=torch.uint8, device="cuda"), None)
        env_a.step_policy(logits, sample=False, obs=obs, action_out=act, reward_sum=total, out=res, obs_scales=scales)
        exp_act = np.where(np.isnan(lg).all(axis=1), 0, np.nanargmax(np.where(np.isnan(lg), -np.inf, lg), axis=1)).astype(np.int32)
        assert np.array_equal(act.cpu().numpy(), exp_act)
        ref = env_b.step(exp_act, want_throughput=True)
        for name in ("delay", "sleep", "buffer", "rebuffer", "reward"):
            assert torch.equal(getattr(res, name), getattr(ref, name)), (t, name)
        assert torch.equal(res.end_of_video, ref.end_of_video)
        for f in STATE_I + STATE_F:
            assert torch.equal(env_a.state(f)[:N], env_b.state(f)[:N]), f
        total_b += ref.reward.cpu().numpy()
        o = obs.cpu().numpy()
        f32 = lambda x: np.asarray(x, np.float64).astype(np.float32)
        assert np.array_equal(o[0], f32(ref.buffer.cpu().numpy() * scales[0]))
        assert np.array_equal(o[1], f32(ref.throughput.cpu().numpy() * scales[1]))
        assert np.array_equal(o[2], f32(ref.delay.cpu().numpy() * scales[2]))
        assert np.array_equal(o[3], f32(exp_act.astype(np.float64) / A))
        assert np.array_equal(o[4:], f32(ref.next_sizes.cpu().numpy().T * scales[3]))
    assert bits_equal(total.cpu().numpy(), total_b) == 0


def test_step_policy_sampling_is_gumbel_max_over_philox_noise():
    N = 8192
    env, _ = make_pair(N, dict(track_history=0))
    A = env.A
    rng = np.random.default_rng(9)
    lg = rng.normal(scale=2.0, size=(N, A)).astype(np.float32)
    logits = torch.from_numpy(lg).cuda()
    act = torch.zeros(N, dtype=torch.int32, device="cuda")
    seed = 0x1234_5678_9ABC
    draws = []
    for draw in range(3):                        # the draw counter advances with every sampled call
        env.step_policy(logits, sample=True, seed=seed, action_out=act)
        a = act.cpu().numpy()
        draws.append(a.copy())
        z = _perturbed_logits(lg, seed, draw)
        # the device's logf may differ from numpy's in the last bits: the drawn action is an arg max up to that
        assert np.all(z[np.arange(N), a] >= z.max(axis=1) - 1e-5), draw
        assert np.mean(a == z.argmax(axis=1)) > 0.999
    assert not np.array_equal(draws[0], draws[1]) and not np.array_equal(draws[1], draws[2])
    # reset zeroes the counter: the same seed replays the same draws
    tid = env.state("trace_id")[:N].clone()
    env.reset(tid, None)
    env.step_policy(logits, sample=True, seed=seed, action_out=act)
    assert np.array_equal(act.cpu().numpy(), draws[0])
    # the draws follow softmax(logits): chi-square over sessions sharing one row of logits
    row = np.array([0.5, -1.0, 2.0, 0.0, 1.0, -0.5], np.float32)[:A]
    logits = torch.from_numpy(np.repeat(row[None, :], N, 0).copy()).cuda()
    counts = np.zeros(A)
    for _ in range(8):
        env.step_policy(logits, sample=True, seed=77, action_out=act)
        counts += np.bincount(act.cpu().numpy(), minlength=A)
    p = np.exp(row - row.max()); p /= p.sum()
    chi2 = ((counts - counts.sum() * p) ** 2 / (counts.sum() * p)).sum()
    assert chi2 < 30.0, (chi2, counts, p)        # 5 degrees of freedom: P(chi2 > 30) ~ 1e-5
    with pytest.raises(TypeError):
        env.step_policy(logits.double())


def _fuzz_fast_worlds(seed, n_worlds):
    """Random worlds through the FAST forms of the fused episode (abr_env_run: all six outputs, no action trace, reset and
    statistics inside the kernel) — the kernels the benchmark runs — for the three policies, with one ladder for all
    chunks (utility carried across steps) or one per chunk, sessions sorted by trace, shuffled, or sorted by the
    environment.  Every output, the state, the per-session sums and the costs bit-identical to the C oracle."""
    rng = np.random.default_rng(7000 + seed)
    for w in range(n_worlds):
        n_traces = int(rng.integers(1, 6))
        T = int(rng.choice([1, 2, 3, 17, 64, 255, 400]))
        V = int(rng.integers(1, 14))
        A = int(rng.integers(1, 9))
        scale = 10.0 ** rng.uniform(-2, 2)
        bw = scale * 10.0 ** rng.uniform(-1.2, 1.2, size=(n_traces, T))
        tl = rng.integers(1, T + 1, size=n_traces).astype(np.int32)
        ti = rng.choice([0.25, 0.3, 0.5, 1.0, 1.7, 2.0], size=n_traces)
        if rng.random() < 0.5:      # one ladder for the whole video
            bitrates = np.tile(np.sort(rng.uniform(100.0, 5000.0, size=A)), (V, 1))
        else:
            bitrates = np.sort(rng.uniform(100.0, 5000.0, size=(V, A)), axis=1)
        sizes = bitrates / 1000.0 * 4.0 * rng.uniform(0.5, 1.5, size=(V, A)) * 10.0 ** rng.uniform(-1, 1)
        params = dict(rtt=float(rng.choice([0.0, 0.08])), payload=float(rng.choice([0.95, 1.0])),
                      max_buffer=float(rng.choice([8.0, 20.0, 60.0])), sleep_quantum=float(rng.choice([0.3, 0.5])),
                      default_quality=int(rng.integers(-1, A)), smooth_prev_ladder=int(rng.integers(0, 2)),
                      utility_mode=int(rng.integers(0, 2)))
        N = 64 * int(rng.integers(1, 5)) + int(rng.integers(0, 64))
        tid = np.sort(rng.integers(0, n_traces, size=N)).astype(np.int32)
        layout = w % 3
        if layout:
            tid = rng.permutation(tid)
        off = rng.uniform(0, 3.0 * float(np.max(tl * ti)), size=N)
        steps = int(rng.integers(1, 2 * V + 3))
        policy = ("random", "bba", "fixed")[int(rng.integers(0, 3))]
        acts = rng.integers(0, A, size=(steps, N)).astype(np.int32) if policy == "fixed" else None
        env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, **params)
        ref = orc.OracleEnv(bw, tl, ti, sizes, bitrates, N, **params)
        tag = f"seed {seed} world {w} {policy} layout {layout}"
        ref.reset(tid, off)
        pid = dict(random=orc.POLICY_RANDOM, bba=orc.POLICY_BBA, fixed=orc.POLICY_FIXED)[policy]
        exp = ref.rollout(pid, steps, seed=w, session_base=17, actions=acts)
        if layout == 2:             # the environment sorts the shuffled sessions by trace; results mapped back
            env.reset(tid, off, session_base=17, sort_by_trace=True)
            got = env.rollout(policy, steps, seed=w, actions=None if acts is None else env.to_env_order(torch.from_numpy(acts)).contiguous(),
                              want=("delay", "sleep", "buffer", "rebuffer", "reward", "end_of_video"))
            got = {k: env.to_caller_order(x) for k, x in got.items()}
            acc = env.to_caller_order(env.session_acc())
        else:
            got, cost, stats = env.run(policy, steps, tid, off, seed=w, session_base=17, actions=acts)
            acc = env.session_acc()
            assert torch.equal(stats, env.stats()), tag
            np.testing.assert_allclose(stats.cpu().numpy(), orc.stats_from_acc(exp["acc"]), rtol=1e-9, atol=1e-300, err_msg=tag)
            assert bits_equal(cost.cpu().numpy(), params_cost(exp["acc"])) == 0, tag
            check_state(env, ref)
        for k_g, k_c in (("delay", "delay"), ("sleep", "sleep"), ("buffer", "buffer"), ("rebuffer", "rebuf"),
                         ("reward", "reward")):
            assert bits_equal(got[k_g].cpu().numpy(), exp[k_c]) == 0, (tag, k_g)
        assert np.array_equal(got["end_of_video"].cpu().numpy(), exp["eov"]), tag
        assert bits_equal(acc.cpu().numpy(), exp["acc"]) == 0, tag
        assert (env.error_count() == 0) == (ref.errors() == 0), tag


def params_cost(acc, rw=4.3, vw=1.0):
    """Simulator.calculate_qoe from the per-session sums (default weights): rw * sum(rebuffer) + vw * sum(smooth)."""
    return rw * acc[1] + vw * acc[3]


@pytest.mark.parametrize("seed", range(4))
def test_randomized_worlds_fast_kernels_match_oracle(seed):
    _fuzz_fast_worlds(seed, 20)
