"""GPU parity of per-session policy parameters (SPEC §4.7) — in the fused episode, abr_env_run / _host and the batched
per-step decision — against the C oracle (tests/session_params_oracle.py on oracle/abr_oracle.c), bit for bit, and
the identities the contract states: uniform parameters equal no installation, a one-launch sweep equals one
environment-wide environment per point, the parameters follow the caller's index under a sorted reset, removal
restores the old bits.  Run with -m gpu."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from abrsimulator_b200 import _lib
from abrsimulator_b200.env import BatchedABREnv
from oracle import oracle as orc
from helpers import assert_close, bits_equal, small_world
import dynamic_oracle as do
import policy_oracle as po
import session_params_oracle as so

POLICIES = {"bba": po.POLICY_BBA, "rate": po.POLICY_RATE, "bola": po.POLICY_BOLA, "dynamic": do.POLICY_DYNAMIC}
TRAJ = (("delay", "delay"), ("sleep", "sleep"), ("buffer", "buffer"), ("rebuffer", "rebuf"), ("reward", "reward"))
LIVE = dict(live=1, start_up_length=8.0, startup_penalty=2.0, latency_penalty=0.1)
WANT = ("delay", "sleep", "buffer", "rebuffer", "reward", "end_of_video", "actions")
ERR_INVALID, ERR_RANGE, ERR_STATE = 1, 3, 4          # abr_b200.h


def world(n_traces=12, T=300, V=48):
    bitrates, sizes, bw, tl, ti = small_world(n_traces=n_traces, T=T, V=V)
    rng = np.random.default_rng(77)
    t = np.arange(T)
    period = rng.integers(40, 90, size=(n_traces, 1))
    bw = np.ascontiguousarray(bw * np.where((t // period) % 2 == 0, 4.0, 0.12))   # high / low phases: DYNAMIC switches
    return bitrates, sizes, bw, tl, ti


def sessions(N, n_traces, layout, seed=21):
    """'smem': blocks of 64 consecutive sessions on one trace (shared-memory path); 'global': interleaved traces."""
    rng = np.random.default_rng(seed)
    if layout == "smem":
        tid = ((np.arange(N) // 64) % n_traces).astype(np.int32)
    else:
        tid = rng.integers(0, n_traces, size=N).astype(np.int32)
    return tid, rng.uniform(0, 900.0, size=N)


def knobs(N, seed=5, degenerate=False):
    """All-distinct parameters of N sessions; with `degenerate`, some near-degenerate ones as well."""
    rng = np.random.default_rng(seed)
    mn = rng.uniform(2.0, 20.0, N)
    on = rng.uniform(2.0, 25.0, N)
    k = dict(bba_reservoir=rng.uniform(-2.0, 15.0, N), bba_cushion=rng.uniform(0.5, 30.0, N),
             rb_safety=rng.uniform(0.3, 1.5, N), bola_min_buffer=mn, bola_target_buffer=mn + rng.uniform(0.5, 40.0, N),
             switch_on_buffer=on, switch_off_buffer=on * rng.uniform(0.0, 0.95, N))
    if degenerate:
        s = rng.choice(N, 4 * (N // 16), replace=False).reshape(4, -1)
        k["bba_cushion"][s[0]] = 1e-9                                          # a tiny cushion
        k["bola_target_buffer"][s[1]] = np.nextafter(k["bola_min_buffer"][s[1]], np.inf)   # min ~ target
        k["switch_off_buffer"][s[2]] = np.nextafter(k["switch_on_buffer"][s[2]], 0.0)     # off ~ on
        k["rb_safety"][s[3]] = 1e-300
    return k


def make(N, params, n_env=1):
    bitrates, sizes, bw, tl, ti = world()
    envs = [BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, **params) for _ in range(n_env)]
    ref = so.SessionParamsEnv(bw, tl, ti, sizes, bitrates, N, **params)
    return envs, ref


def check_episode(env, ref, got, exp, dtype="f64"):
    assert np.array_equal(got["actions"].cpu().numpy(), exp["actions"])
    for kg, kc in TRAJ:
        g = got[kg].cpu().numpy()
        if dtype == "f32":
            assert np.array_equal(g, exp[kc].astype(np.float32)), kg
        else:
            assert_close(g, exp[kc], kg)
    if "latency" in got:
        e = exp["latency"].astype(np.float32) if dtype == "f32" else exp["latency"]
        assert bits_equal(got["latency"].cpu().numpy(), e) == 0
    assert np.array_equal(got["end_of_video"].cpu().numpy(), exp["eov"])
    assert_close(env.session_acc().cpu().numpy(), exp["acc"], "acc")
    for f in ("seg", "chunk", "last_q", "trace_id", "hist_len"):
        assert np.array_equal(env.state(f).cpu().numpy(), ref.field(f)), f
    for f in ("phase", "pos", "buffer"):
        assert bits_equal(env.state(f).cpu().numpy(), ref.field(f)) == 0, f
    if env.params.track_history:
        assert np.array_equal(env.state("dyn_mode").cpu().numpy(), ref.dyn_mode)
    np.testing.assert_allclose(env.stats().cpu().numpy(), orc.stats_from_acc(exp["acc"]), rtol=1e-9)
    assert env.error_count() == 0 and ref.errors() == 0


def env_params(policy, live, auto_reset=1):
    p = dict(track_history=1 if policy in ("rate", "dynamic") else 0, auto_reset=auto_reset)
    if live:
        p.update(LIVE)
    return p


# 1. the form matrix: every per-session episode form (policy x live 0/1 x fp64/fp32) on both trace paths, auto_reset
#    0/1, against the oracle; live 2 (the speed controller) in test 6
@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("live", [0, 1])
@pytest.mark.parametrize("auto_reset", [1, 0])
@pytest.mark.parametrize("layout", ["smem", "global"])
@pytest.mark.parametrize("policy", list(POLICIES))
def test_session_episode_matches_oracle(policy, layout, auto_reset, live, dtype):
    N, steps = 1000, 60
    (env,), ref = make(N, env_params(policy, live, auto_reset))
    k = knobs(N, degenerate=True)
    env.reset(*sessions(N, 12, layout))
    ref.reset(*sessions(N, 12, layout))
    env.set_session_policy_params(**k)
    assert ref.set_session_params(**k)
    want = WANT + (("latency",) if live else ())
    got = env.rollout(policy, steps, want=want, dtype=torch.float32 if dtype == "f32" else torch.float64)
    exp = ref.rollout(POLICIES[policy], steps)
    check_episode(env, ref, got, exp, dtype)
    assert len(np.unique(exp["actions"])) >= 3
    if policy == "dynamic":
        up, down = ref.switches()
        assert up > 0 and down > 0


# 2. the four decision forms, and decide + step equals one episode step
@pytest.mark.parametrize("policy", list(POLICIES))
def test_decide_matches_oracle_and_decide_plus_step_is_the_episode(policy):
    N, steps = 3000, 30
    params = env_params(policy, 0)
    (env, env_b), ref = make(N, params, n_env=2)
    k = knobs(N, seed=8, degenerate=True)
    tid, off = sessions(N, 12, "global")
    for e in (env, env_b, ref):
        e.reset(tid, off)
    env.set_session_policy_params(**k)
    env_b.set_session_policy_params(**k)
    assert ref.set_session_params(**k)
    acts = []
    for t in range(steps):
        a = env.policy_decide(policy)
        assert np.array_equal(a.cpu().numpy(), ref.policy_decide(POLICIES[policy])), t
        acts.append(a.clone())
        env.step(a)
        ref.step(a.cpu().numpy(), want_next_sizes=False)
    got = env_b.rollout(policy, steps)
    assert np.array_equal(got["actions"].cpu().numpy(), torch.stack(acts).cpu().numpy())
    assert bits_equal(env.state("buffer").cpu().numpy(), env_b.state("buffer").cpu().numpy()) == 0


# 3. split episodes carry the state (DYNAMIC's rule in dyn_mode)
@pytest.mark.parametrize("policy", list(POLICIES))
def test_split_episode_equals_one_episode(policy):
    N = 700
    (a, b), _ = make(N, env_params(policy, 0), n_env=2)
    k = knobs(N, seed=3)
    tid, off = sessions(N, 12, "global")
    for e in (a, b):
        e.reset(tid, off)
        e.set_session_policy_params(**k)
    x = a.rollout(policy, 48)
    y1, y2 = b.rollout(policy, 24), b.rollout(policy, 24)
    for key in WANT:
        assert torch.equal(x[key], torch.cat([y1[key], y2[key]])), key
    for f in ("seg", "chunk", "last_q", "phase", "pos", "buffer", "hist_len") + (("dyn_mode",) if policy == "dynamic" else ()):
        assert torch.equal(a.state(f), b.state(f)), f
    # the accumulators add one sum per call: equal to rounding, the counts exactly
    acc_a, acc_b = a.session_acc().cpu().numpy(), b.session_acc().cpu().numpy()
    np.testing.assert_allclose(acc_b, acc_a, rtol=1e-12, atol=1e-12)
    assert np.array_equal(acc_a[6:8], acc_b[6:8])


# 4. run / run_host (pinned and pageable) equal reset + rollout
@pytest.mark.parametrize("policy", ["bba", "dynamic"])
def test_run_and_run_host_equal_reset_and_rollout(policy):
    N, steps = 900, 40
    (a, b, c), _ = make(N, env_params(policy, 0), n_env=3)
    k = knobs(N, seed=4)
    tid, off = sessions(N, 12, "smem")
    a.reset(tid, off)
    for e in (a, b, c):
        e.set_session_policy_params(n=N, **k)
    ref = a.rollout(policy, steps)
    out, cost, stats = b.run(policy, steps, torch.as_tensor(tid, device="cuda"), torch.as_tensor(off, device="cuda"),
                             qoe_cost=torch.empty(N, dtype=torch.float64, device="cuda"),
                             stats=torch.empty(_lib.NUM_STATS, dtype=torch.float64, device="cuda"))
    for key in ("delay", "sleep", "buffer", "rebuffer", "reward", "end_of_video"):
        assert torch.equal(out[key], ref[key]), key
    assert torch.equal(b.session_acc(), a.session_acc())
    for pinned in (False, True):
        t = torch.as_tensor(tid)
        o = torch.as_tensor(off)
        if pinned:
            t, o = t.pin_memory(), o.pin_memory()
        h = c.run_host(policy, steps, t, o, want_reward_traj=True)
        assert np.array_equal(h["reward"], ref["reward"].cpu().numpy())
        assert np.array_equal(h["acc"], a.session_acc().cpu().numpy())


# 5. identities: uniform = none; a partition into G configurations = G environment-wide environments; removal
@pytest.mark.parametrize("live", [0, 1, 2])
@pytest.mark.parametrize("policy", list(POLICIES))
def test_sweep_equals_environment_wide_runs(policy, live):
    N, G, steps = 1024, 4, 48
    params = env_params(policy, live)
    envs, _ = make(N, params, n_env=2)
    sweep, plain = envs
    if live == 2:
        for e in envs:
            e.set_speed_control()
    grid = [dict(bba_reservoir=3.0 + g, bba_cushion=6.0 + 4 * g, rb_safety=0.6 + 0.2 * g, bola_min_buffer=4.0 + 2 * g,
                 bola_target_buffer=20.0 + 6 * g, switch_on_buffer=8.0 + 3 * g, switch_off_buffer=3.0 + g)
            for g in range(G)]
    tid, off = sessions(N, 12, "global", seed=7)
    group = np.arange(N) % G
    fields = {f: np.array([grid[g][f] for g in group]) for f in so.FIELDS}
    sweep.reset(tid, off)
    sweep.set_session_policy_params(**fields)
    got = sweep.rollout(policy, steps)
    sweep.reset(tid, off)
    got32 = sweep.rollout(policy, steps, dtype=torch.float32)   # the fp32-output form: the fp64 outputs rounded once
    for key in ("delay", "sleep", "buffer", "rebuffer", "reward"):
        assert torch.equal(got32[key], got[key].float()), key
    bitrates, sizes, bw, tl, ti = world()
    for g in range(G):
        m = group == g
        kw = dict(params, bba_reservoir=grid[g]["bba_reservoir"], bba_cushion=grid[g]["bba_cushion"])
        e = BatchedABREnv(bw, sizes, bitrates, int(m.sum()), trace_len=tl, trace_interval=ti, **kw)
        if live == 2:
            e.set_speed_control()
        e.set_policy_params(**{f: grid[g][f] for f in ("rb_safety", "bola_min_buffer", "bola_target_buffer")})
        e.set_dynamic_params(**{f: grid[g][f] for f in ("switch_on_buffer", "switch_off_buffer")})
        e.reset(tid[m], off[m])
        exp = e.rollout(policy, steps)
        for key in WANT:
            assert torch.equal(got[key][:, torch.as_tensor(m, device="cuda")], exp[key]), (g, key)
    # uniform arrays of the environment-wide values give the environment-wide bits; so does removal
    plain.reset(tid, off)
    base = plain.rollout(policy, steps)
    wide = so.env_wide(plain.params)
    plain.reset(tid, off)
    plain.set_session_policy_params(**{f: np.full(N, wide[j]) for j, f in enumerate(so.FIELDS)})
    uni = plain.rollout(policy, steps)
    plain.set_session_policy_params(None)
    plain.reset(tid, off)
    again = plain.rollout(policy, steps)
    for key in WANT:
        assert torch.equal(uni[key], base[key]) and torch.equal(again[key], base[key]), key


# 6. sorted reset: the parameters follow the caller's index
@pytest.mark.parametrize("policy", ["bola", "dynamic"])
def test_sorted_environment_keys_parameters_by_caller_index(policy):
    N, steps = 1500, 40
    (a, b), ref = make(N, env_params(policy, 0), n_env=2)
    k = knobs(N, seed=11)
    tid, off = sessions(N, 12, "global", seed=9)
    a.reset(tid, off)
    b.reset(tid, off, sort_by_trace=True)
    for e in (a, b):
        e.set_session_policy_params(**k)
    x = a.rollout(policy, steps)
    y = b.rollout(policy, steps)
    for key in WANT:
        assert torch.equal(y[key], x[key][:, b.perm.long()]), key   # position p holds caller index perm[p]
    # the oracle run in environment order with the table mapped through perm
    ref.reset(tid[b.perm.cpu().numpy()], off[b.perm.cpu().numpy()])
    assert ref.set_session_params(**k)
    ref.perm = b.perm.cpu().numpy()
    exp = ref.rollout(POLICIES[policy], steps)
    assert np.array_equal(y["actions"].cpu().numpy(), exp["actions"])


# 7. FIXED / RANDOM ignore the parameters
def test_fixed_and_random_are_unaffected():
    N = 800
    (a, b), _ = make(N, dict(track_history=1), n_env=2)
    tid, off = sessions(N, 12, "smem")
    a.reset(tid, off)
    b.reset(tid, off)
    b.set_session_policy_params(**knobs(N))
    assert torch.equal(a.rollout("random", 30, seed=5)["reward"], b.rollout("random", 30, seed=5)["reward"])
    acts = torch.randint(0, a.A, (30, N), dtype=torch.int32, device="cuda")
    assert torch.equal(a.rollout("fixed", 30, actions=acts)["reward"], b.rollout("fixed", 30, actions=acts)["reward"])


# 8. errors, their order, and the previous installation left intact
BAD = [("bba_reservoir", np.nan), ("bba_reservoir", np.inf), ("bba_cushion", 0.0), ("bba_cushion", -1.0),
       ("bba_cushion", np.nan), ("rb_safety", 0.0), ("rb_safety", -np.inf), ("bola_min_buffer", 0.0),
       ("bola_min_buffer", np.nan), ("bola_target_buffer", 5.0), ("bola_target_buffer", np.inf),
       ("switch_on_buffer", np.nan), ("switch_off_buffer", -0.5), ("switch_off_buffer", 30.0),
       ("switch_off_buffer", np.inf)]


@pytest.mark.parametrize("field,value", BAD, ids=[f"{f}={v}" for f, v in BAD])
def test_invalid_values_name_the_session_and_field_and_keep_the_installation(field, value):
    N = 300
    (env,), _ = make(N, dict(track_history=1))
    tid, off = sessions(N, 12, "global")
    env.reset(tid, off)
    k = knobs(N, seed=2)
    k["bola_min_buffer"][:] = 10.0
    k["bola_target_buffer"][:] = 30.0
    k["switch_on_buffer"][:] = 12.0
    k["switch_off_buffer"][:] = 6.0
    env.set_session_policy_params(**k)
    before = env.session_policy_params()
    bad = {f: v.copy() for f, v in k.items()}
    bad[field][[137, 200]] = value
    x = so.fill(N, so.env_wide(env.params), **bad)
    assert so.first_invalid(x) == (137, so.FIELDS.index(field)) == so.first_invalid_py(x)
    with pytest.raises(_lib.AbrError) as e:
        env.set_session_policy_params(**bad)
    assert e.value.code == ERR_INVALID and f"session 137: {field}" in str(e.value)
    after = env.session_policy_params()
    for f in so.FIELDS:
        assert torch.equal(before[f], after[f]), f
    assert np.array_equal(after["bba_cushion"].cpu().numpy(), k["bba_cushion"])


def test_state_errors_and_getter():
    N = 256
    (env,), _ = make(N, dict(track_history=1))
    tid, off = sessions(N, 12, "global")
    env.reset(tid, off)
    assert env.session_policy_params() is None
    env.set_session_policy_params(rb_safety=np.linspace(0.5, 1.0, N))
    got = env.session_policy_params()
    wide = so.env_wide(env.params)
    for j, f in enumerate(so.FIELDS):
        exp = np.linspace(0.5, 1.0, N) if f == "rb_safety" else np.full(N, wide[j])
        assert np.array_equal(got[f].cpu().numpy(), exp), f
    for call in (lambda: env.set_policy_params(rb_safety=0.9), lambda: env.set_dynamic_params(switch_on_buffer=9.0)):
        with pytest.raises(_lib.AbrError) as e:
            call()
        assert e.value.code == ERR_STATE
    env.reset(tid[:100], off[:100])
    for call in (lambda: env.rollout("bola", 4), lambda: env.policy_decide("rate")):
        with pytest.raises(_lib.AbrError) as e:
            call()
        assert e.value.code == ERR_STATE
    env.rollout("random", 4)                      # FIXED / RANDOM do not check the count
    with pytest.raises(_lib.AbrError) as e:
        env.run("bba", 4, torch.as_tensor(tid[:50], device="cuda"))
    assert e.value.code == ERR_STATE
    with pytest.raises(_lib.AbrError) as e:
        env.set_session_policy_params(n=N + 10 ** 6, rb_safety=np.ones(N + 10 ** 6))
    assert e.value.code == ERR_RANGE
    env.set_session_policy_params(None)
    env.set_policy_params(rb_safety=0.9)
    env.rollout("bola", 4)


# 9. a graph captured with parameters installed replays with the values installed at replay time
def test_cuda_graph_replays_with_reinstalled_values():
    N, steps = 1024, 24
    (env, ref_env), _ = make(N, dict(track_history=1), n_env=2)
    tid, off = sessions(N, 12, "smem")
    k1, k2 = knobs(N, seed=1), knobs(N, seed=2)
    env.reset(tid, off)
    env.set_session_policy_params(**k1)
    out = {key: torch.empty(steps, N, dtype=torch.int32 if key == "actions" else
                            torch.uint8 if key == "end_of_video" else torch.float64, device="cuda") for key in WANT}
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        env.rollout("dynamic", steps, out=out)      # warm-up
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        env.rollout("dynamic", steps, out=out)
    env.reset(tid, off)
    env.set_session_policy_params(**k2)
    g.replay()
    torch.cuda.synchronize()
    ref_env.reset(tid, off)
    ref_env.set_session_policy_params(**k2)
    exp = ref_env.rollout("dynamic", steps)
    for key in WANT:
        assert torch.equal(out[key], exp[key]), key


# 10. the benchmark's size
@pytest.mark.parametrize("policy", list(POLICIES))
def test_full_size(policy):
    N, steps = 65536, 48
    G = 64
    params = env_params(policy, 0)
    (a, b), _ = make(N, params, n_env=2)
    tid, off = sessions(N, 12, "smem")
    group = np.arange(N) // (N // G)
    vals = dict(bba_reservoir=2.0 + 0.2 * group, bba_cushion=4.0 + 0.5 * group, rb_safety=0.5 + 0.01 * group,
                bola_min_buffer=3.0 + 0.2 * group, bola_target_buffer=25.0 + 0.5 * group,
                switch_on_buffer=9.0 + 0.1 * group, switch_off_buffer=4.0 + 0.05 * group)
    a.reset(tid, off)
    a.set_session_policy_params(**vals)
    got = a.rollout(policy, steps)
    # spot-check four points against environment-wide environments
    bitrates, sizes, bw, tl, ti = world()
    for g in (0, 21, 42, 63):
        m = group == g
        kw = dict(params, bba_reservoir=float(vals["bba_reservoir"][m][0]), bba_cushion=float(vals["bba_cushion"][m][0]))
        e = BatchedABREnv(bw, sizes, bitrates, int(m.sum()), trace_len=tl, trace_interval=ti, **kw)
        e.set_policy_params(**{f: float(vals[f][m][0]) for f in ("rb_safety", "bola_min_buffer", "bola_target_buffer")})
        e.set_dynamic_params(**{f: float(vals[f][m][0]) for f in ("switch_on_buffer", "switch_off_buffer")})
        e.reset(tid[m], off[m])
        exp = e.rollout(policy, steps)
        for key in WANT:
            assert torch.equal(got[key][:, torch.as_tensor(m, device="cuda")], exp[key]), (g, key)
    assert a.error_count() == 0


def test_example_check():
    import subprocess
    import sys
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "examples", "policy_sweep.py"), "--check"],
                       capture_output=True, text=True, cwd=root, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
