"""GPU parity of shared bottleneck links (SPEC §9, abr_env_run_shared) against the pure-Python oracle
(tests/shared_link_oracle.py), bit for bit, and the identities the contract states: G = 1 is abr_env_run, two
session_base shards are one run, the nullable outputs do not change any bit.  Run with -m gpu."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from abrsimulator_b200 import _lib, synth
from abrsimulator_b200.env import BatchedABREnv
from helpers import assert_close, small_world
import shared_link_oracle as sl

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
IDS = {"fixed": sl.FIXED, "random": sl.RANDOM, "bba": sl.BBA, "rate": sl.RATE, "bola": sl.BOLA, "dynamic": sl.DYNAMIC}
MIXED = ["bola", "rate", "bba", "dynamic", "random", "fixed"]
WANT = ("delay", "sleep", "buffer", "rebuffer", "reward", "end_of_video", "actions", "request_time")
TRAJ = (("delay", "delay"), ("sleep", "sleep"), ("buffer", "buffer"), ("rebuffer", "rebuf"), ("reward", "reward"),
        ("request_time", "request_time"))
STATE = ("seg", "phase", "pos", "chunk", "last_q", "buffer", "done", "hist_len", "trace_id")
ERR_INVALID, ERR_RANGE, ERR_STATE = 1, 3, 4          # abr_b200.h


def make(T=64, n_traces=6, V=6, cap=512, ragged=True, zero_sizes=False, **params):
    bitrates, sizes, bw, tl, ti = small_world(n_traces=n_traces, T=T, V=V, seed=T, ragged=ragged)
    if zero_sizes:
        sizes = sizes.copy()
        sizes[::2, 0] = 0.0
    kw = dict(track_history=1, max_buffer=20.0)   # a small buffer cap: the players sleep and join the link again
    kw.update(params)
    env = BatchedABREnv(bw, sizes, bitrates, cap, trace_len=tl, trace_interval=ti, **kw)
    return env, sl.world_of_env(env, bw, tl, ti, sizes)


def joins(N, rng):
    """Join delays on a 0.5 s grid: many exact ties, between players and with the link's events."""
    return rng.integers(0, 8, size=N) * 0.5


def run_both(env, w, steps, G, n_links, policy, seed=3, knobs=None, join=True, session_base=0, rng_seed=0, mixed=MIXED):
    rng = np.random.default_rng(rng_seed)
    N = n_links * G
    tid = rng.integers(0, len(w.bw), size=n_links).astype(np.int32)
    off = rng.uniform(0.0, 50.0, size=n_links)
    jd = joins(N, rng) if join else None
    actions = rng.integers(0, env.A, size=(steps, N)).astype(np.int32)
    pp = None
    if policy == "mixed":
        pp = [mixed[p % len(mixed)] for p in range(G)]
        pol = "bba"
    else:
        pol = policy
    if knobs is not None:
        env.set_session_policy_params(n=N, **knobs)
    out, link, cost, stats = env.run_shared(pol, steps, tid, G, link_offset=off, join_delay=jd, player_policy=pp,
                                            seed=seed, session_base=session_base, actions=actions, want=WANT)
    x = None if knobs is None else np.stack([np.asarray(knobs[f]) if f in knobs else np.full(N, w.wide[j])
                                             for j, f in enumerate(_lib.SESSION_PARAM_FIELDS)])
    ref = sl.run_shared(w, steps, G, tid, off, jd, IDS[pol], None if pp is None else [IDS[p] for p in pp], seed,
                        session_base, actions, knobs=x)
    return out, link, cost, stats, ref


def check(env, out, link, cost, stats, ref):
    for k_gpu, k_ref in TRAJ:
        assert_close(out[k_gpu].cpu().numpy(), ref[k_ref], k_gpu)
    assert np.array_equal(out["end_of_video"].cpu().numpy(), ref["eov"])
    assert np.array_equal(out["actions"].cpu().numpy(), ref["actions"])
    for k in ("time", "capacity", "delivered"):
        assert_close(link[k].cpu().numpy(), ref["link_" + k], "link_" + k)
    assert_close(env.session_acc().cpu().numpy(), ref["acc"], "acc")
    assert_close(cost.cpu().numpy(), ref["qoe_cost"], "qoe_cost")
    assert_close(env.qoe_cost().cpu().numpy(), ref["qoe_cost"], "qoe_cost()")
    assert torch.equal(stats, env.stats())
    for k in STATE:
        assert np.array_equal(env.state(k).cpu().numpy(), ref["state"][k]), k
    assert env.error_count() == ref["errors"]


def knob_set(N, rng):
    mn = rng.uniform(4.0, 12.0, N)
    on = rng.uniform(6.0, 16.0, N)
    return dict(bba_reservoir=rng.uniform(0.0, 8.0, N), rb_safety=rng.uniform(0.5, 1.3, N), bola_min_buffer=mn,
                bola_target_buffer=mn + rng.uniform(2.0, 20.0, N), switch_on_buffer=on,
                switch_off_buffer=on * rng.uniform(0.1, 0.9, N))


@pytest.mark.parametrize("policy", ["fixed", "random", "bba", "rate", "bola", "dynamic", "mixed"])
@pytest.mark.parametrize("G", [1, 2, 3, 8, 32])
def test_kernel_matches_oracle(G, policy):
    """5 links (not a multiple of the block's 4), ragged short traces that wrap inside a download, join ties, steps > V;
    auto_reset and the per-session knobs alternate with G."""
    env, w = make(auto_reset=G % 2)
    kn = knob_set(5 * G, np.random.default_rng(G)) if G in (3, 8, 32) and policy not in ("fixed", "random") else None
    out, link, cost, stats, ref = run_both(env, w, 14, G, 5, policy, knobs=kn, rng_seed=G)
    check(env, out, link, cost, stats, ref)


@pytest.mark.parametrize("layout", ["smem", "global", "noindex"])
def test_both_trace_paths(layout):
    """smem: rows staged per warp; global: rows too large to stage (20 000 segments); noindex: a trace longer than
    65 535 segments, which has no bucket index."""
    T = {"smem": 200, "global": 20000, "noindex": 70000}[layout]
    env, w = make(T=T, n_traces=2, ragged=False)
    out, link, cost, stats, ref = run_both(env, w, 12, 4, 3, "mixed", rng_seed=7)
    check(env, out, link, cost, stats, ref)


@pytest.mark.parametrize("policy", ["fixed", "bba", "rate", "mixed0"])
def test_zero_size_chunks(policy):
    env, w = make(zero_sizes=True)
    # mixed0: the policies that accept a zero size, mixed
    out, link, cost, stats, ref = run_both(env, w, 10, 4, 3, "mixed" if policy == "mixed0" else policy, rng_seed=11,
                                           mixed=["fixed", "rate", "bba", "random"])
    check(env, out, link, cost, stats, ref)


def test_bad_join_delays_and_trace_ids_are_counted_as_the_oracle_counts_them():
    env, w = make()
    tid = np.array([0, 99, 1], np.int32)
    jd = np.array([0.0, -1.0, np.nan, np.inf, 0.5, 0.5], np.float64)
    out, link, cost, stats = env.run_shared("bba", 6, tid, 2, join_delay=jd, want=WANT)
    ref = sl.run_shared(w, 6, 2, tid, None, jd, sl.BBA)
    check(env, out, link, cost, stats, ref)
    assert ref["errors"] == 3 + 2


@pytest.mark.parametrize("policy", ["fixed", "random", "bba", "rate", "bola", "dynamic"])
def test_one_player_per_link_is_abr_env_run_at_the_bench_size(policy):
    N, steps = 65536, 48
    bitrates, sizes = synth.make_video(48)
    bw, tl, ti = synth.make_traces(1024, 2048)
    tid, off = synth.make_sessions(N, 1024, 2048)
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, track_history=1)
    actions = torch.randint(0, env.A, (steps, N), dtype=torch.int32, device=env.device)
    want = ("delay", "sleep", "buffer", "rebuffer", "reward", "end_of_video", "actions")
    a, cost_a, _ = env.run(policy, steps, tid, off, seed=5, actions=actions, want=want)
    acc_a, stats_a = env.session_acc().clone(), env.stats()
    st_a = {k: env.state(k).clone() for k in STATE + (("dyn_mode",) if policy == "dynamic" else ())}
    errors = env.error_count()
    b, link, cost_b, stats_b = env.run_shared(policy, steps, tid, 1, link_offset=off, seed=5, actions=actions,
                                              want=want)
    for k in want:
        assert torch.equal(a[k], b[k]), k
    assert torch.equal(cost_a, cost_b) and torch.equal(acc_a, env.session_acc())
    # the statistics are abr_stats_partial's tree over the accumulators; abr_env_run's come from its episode's block
    # partials: the same sums in another order
    assert torch.equal(stats_b, env.stats())
    assert torch.allclose(stats_a, stats_b, rtol=1e-12, atol=0) and torch.equal(stats_a[6:8], stats_b[6:8])
    for k, t in st_a.items():
        assert torch.equal(t, env.state(k)), k
    assert env.error_count() == 2 * errors


def test_two_session_base_shards_are_one_run():
    env, w = make(cap=1024)
    G, L, steps = 4, 12, 10
    rng = np.random.default_rng(2)
    tid = rng.integers(0, 6, size=L).astype(np.int32)
    off = rng.uniform(0, 40, size=L)
    jd = joins(L * G, rng)
    full = env.run_shared("random", steps, tid, G, off, jd, seed=9, session_base=100, want=WANT)
    full = [dict((k, v.clone()) for k, v in d.items()) if isinstance(d, dict) else d.clone() for d in full]
    h = L // 2
    parts = [env.run_shared("random", steps, tid[s], G, off[s], jd[s.start * G:s.stop * G], seed=9,
                            session_base=100 + s.start * G, want=WANT) for s in (slice(0, h), slice(h, L))]
    for k in WANT:
        assert torch.equal(full[0][k], torch.cat([parts[0][0][k], parts[1][0][k]], 1)), k
    for k in full[1]:
        assert torch.equal(full[1][k], torch.cat([parts[0][1][k], parts[1][1][k]])), k
    assert torch.equal(full[2], torch.cat([parts[0][2], parts[1][2]]))


def test_every_subset_of_outputs_gives_the_same_bits():
    env, w = make()
    G, L, steps = 3, 5, 9
    rng = np.random.default_rng(4)
    tid = rng.integers(0, 6, size=L).astype(np.int32)
    jd = joins(L * G, rng)
    pp = ["bola", "rate", "dynamic"]
    base = env.run_shared("bba", steps, tid, G, join_delay=jd, player_policy=pp, want=WANT)
    base = [dict((k, v.clone()) for k, v in d.items()) if isinstance(d, dict) else d.clone() for d in base]
    acc, state = env.session_acc().clone(), {k: env.state(k).clone() for k in STATE}
    for sub in [(), ("delay",), ("reward", "request_time"), ("end_of_video", "actions", "sleep"), ("buffer", "rebuffer")]:
        for link_want in [(), ("delivered",), ("time", "capacity")]:
            o, l, c, s = env.run_shared("bba", steps, tid, G, join_delay=jd, player_policy=pp, want=sub,
                                        link_want=link_want, qoe_cost=False if "delay" in sub else None,
                                        stats=False if sub == () else None)
            for k in sub:
                assert torch.equal(o[k], base[0][k]), (sub, k)
            for k in link_want:
                assert torch.equal(l[k], base[1][k]), (link_want, k)
            if c is not None:
                assert torch.equal(c, base[2])
            if s is not None:
                assert torch.equal(s, base[3])
            assert torch.equal(env.session_acc(), acc)
            for k in STATE:
                assert torch.equal(env.state(k), state[k]), k


def test_argument_checks_in_order():
    env, w = make(cap=64)
    lib = env._lib
    tid = torch.zeros(4, dtype=torch.int32, device=env.device)
    o = _lib.AbrSharedOutputs()
    call = lambda e=env._h, pol=2, pp=None, steps=4, G=4, t=tid.data_ptr(), n_links=4, actions=None: \
        lib.abr_env_run_shared(e, pol, pp, 0, steps, G, t, None, None, n_links, 0, actions, o, None, None, None)
    assert call(t=None) == ERR_INVALID
    assert call(G=0) == ERR_RANGE and call(G=33) == ERR_RANGE and call(n_links=17) == ERR_RANGE
    assert call(steps=-1) == ERR_RANGE and call(n_links=-1) == ERR_RANGE
    assert call(pol=9) == ERR_INVALID and call(pol=0) == ERR_INVALID     # unknown; FIXED without actions
    pp = np.array([2, 3, 4, 7], np.int32)
    assert call(pp=pp.ctypes.data) == ERR_INVALID                        # slot 3
    env.set_session_policy_params(n=8, rb_safety=np.ones(8))
    assert call() == ERR_STATE and call(pol=1) == 0                      # 16 sessions against 8; RANDOM ignores them
    assert call(G=16, n_links=17) == ERR_RANGE                           # the range before the count
    env.set_session_policy_params(None)
    env.set_order(torch.arange(16, dtype=torch.int32, device=env.device))
    assert call(G=0) == ERR_STATE and b"order" in lib.abr_last_error()   # the order before the range
    env.set_order(None)
    no_hist, _ = make(cap=64, track_history=0)
    assert no_hist._lib.abr_env_run_shared(no_hist._h, 3, None, 0, 4, 4, tid.data_ptr(), None, None, 4, 0, None, o,
                                           None, None, None) == ERR_STATE
    zero, _ = make(cap=64, zero_sizes=True)
    assert zero._lib.abr_env_run_shared(zero._h, 4, None, 0, 4, 4, tid.data_ptr(), None, None, 4, 0, None, o, None,
                                        None, None) == ERR_INVALID
    live, _ = make(cap=64, live=1)
    assert live._lib.abr_env_run_shared(live._h, 2, None, 0, 4, 0, None, None, None, 4, 0, None, o, None, None,
                                        None) == ERR_INVALID                          # NULL trace ids first
    assert live._lib.abr_env_run_shared(live._h, 2, None, 0, 4, 0, tid.data_ptr(), None, None, 4, 0, None, o, None,
                                        None, None) == ERR_STATE                      # live before the range


def test_the_example_check_passes():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "examples", "shared_link.py"), "--check", "--links", "256"],
                       capture_output=True, text=True, cwd=ROOT, timeout=1200)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "check: ok" in r.stdout
