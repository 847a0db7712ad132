"""Every entry point under an installed session order.  Run with -m gpu.

Two environments get the same sessions, interleaved over the traces (trace = session mod n_traces, with a few invalid
ids): A keeps the caller's order, B sorts them by trace (``reset(..., sort_by_trace=True)``).  B gets its per-session
inputs through ``to_env_order`` and its results go back through ``to_caller_order``; the two must be bit-identical,
and so must the state, the accumulators and the error counts.  The statistics vector sums over environment positions,
so A and B add the same numbers in different orders: its counts must be equal, its sums within SPEC §6's 1e-9
relative.

Entry points covered here that the other order tests do not: ``step_f32``, ``step_live`` with a [V][N] speed table,
``step_policy`` (greedy and sampled: Gumbel draws keyed by ``session_base + perm[p]``, the [F][N] observation,
``action_out``, ``reward_sum``), the fused live and fp32 episodes, ``run``, ``run_host`` (pinned and pageable),
``mpc_decide`` (ref and robust: the K-major history ring, ``last_pred``, the error ring), ``throughput_history`` and
``qoe_cost``.  A two-shard emulation on one GPU checks that a shard sorted on its own keys its draws by the global
caller index.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from abrsimulator_b200 import _lib
from abrsimulator_b200.env import BatchedABREnv, StepResult
from helpers import small_world

N, N_TRACES, STEPS, BASE = 3000, 37, 24, 500
STATE = ("seg", "chunk", "last_q", "trace_id", "phase", "pos", "buffer", "done", "hist_len", "err_len", "t_now",
         "play_time", "started", "play_id", "play_len")
LIVE = dict(live=1, start_up_length=8.0, max_buffer=16.0, latency_penalty=0.05, startup_penalty=1.0, track_acc=1)
HIST = dict(track_history=1, track_acc=1)
COUNTS = (6, 7)                       # steps and sessions finished: exact; the other entries are sums


def sessions(n=N):
    tid = (np.arange(n) % N_TRACES).astype(np.int32)
    tid[5::97] = -1                   # invalid ids: one error each at every reset, trace 0 like the sort
    tid[11::89] = N_TRACES
    off = np.random.default_rng(3).uniform(0, 150.0, size=n)
    return tid, off


class Side:
    """One environment and the maps between the caller's order and its own."""

    def __init__(self, sort, params, n=N, base=BASE, tid=None, off=None):
        bitrates, sizes, bw, tl, ti = small_world(n_traces=N_TRACES, T=96, V=24, ragged=True)
        self.A, self.V = bitrates.shape[1], bitrates.shape[0]
        self.env = BatchedABREnv(bw, sizes, bitrates, n, trace_len=tl, trace_interval=ti, **params)
        if tid is None:
            tid, off = sessions(n)
        self.tid, self.off = tid, off
        self.env.reset(tid, off, session_base=base, sort_by_trace=sort)
        self.perm = self.env.perm.cpu().numpy().astype(np.int64) if sort else None

    def inp(self, x):
        """[..., N] caller order -> environment order (device, contiguous)."""
        x = torch.as_tensor(x).cuda()
        return self.env.to_env_order(x).contiguous()

    def inp_rows(self, x):
        """[N, ...] caller order -> environment order."""
        return self.inp(torch.as_tensor(x).cuda().t()).t().contiguous()

    def out(self, x):
        """Environment order -> caller order, always a copy (state views and reused buffers change later)."""
        return self.env.to_caller_order(x).clone()

    def out_rows(self, x):
        return self.out(x.t().contiguous()).t()

    def host_inp(self, x):
        return np.ascontiguousarray(x if self.perm is None else np.asarray(x)[..., self.perm])

    def host_out(self, x):
        if self.perm is None:
            return np.asarray(x)
        inv = np.empty_like(self.perm)
        inv[self.perm] = np.arange(self.perm.size)
        return np.asarray(x)[..., inv]


def rng_tensor(shape, seed, lo, hi, dtype):
    g = np.random.default_rng(seed)
    if dtype == torch.int32:
        return torch.from_numpy(g.integers(lo, hi, size=shape).astype(np.int32))
    return torch.from_numpy(g.uniform(lo, hi, size=shape)).to(dtype)


# ---- the entry points: each returns {name: caller-order tensor or array} ----
def step_results(s, r, rows=("next_sizes",)):
    return {f: (s.out_rows(x) if f in rows else s.out(x)) for f, x in r._asdict().items() if x is not None}


def ep_step_f32(s):
    got = {}
    acts = rng_tensor((6, N), 4, 0, s.A, torch.int32)
    for t in range(6):
        r = s.env.step(s.inp(acts[t]), want_throughput=True, dtype=torch.float32)
        got.update({f"{k}{t}": v for k, v in step_results(s, r).items()})
    return got


def ep_step_live(s):
    got = {}
    acts = rng_tensor((6, N), 5, 0, s.A, torch.int32)
    speed = rng_tensor((s.V, N), 6, 0.5, 2.0, torch.float64)             # [V][N]: per session and content chunk
    for t in range(6):
        r = s.env.step(s.inp(acts[t]), want_throughput=True, speed=s.inp(speed))
        got.update({f"{k}{t}": v for k, v in step_results(s, r).items()})
    return got


def ep_step_policy(sample):
    def run(s):
        got = {}
        F = 4 + s.A
        obs = torch.empty(F * N, dtype=torch.float32, device="cuda")
        act = torch.empty(N, dtype=torch.int32, device="cuda")
        rsum = torch.zeros(N, dtype=torch.float64, device="cuda")
        out = StepResult(*[torch.empty(N, dtype=torch.float64, device="cuda") for _ in range(5)], None,
                         torch.empty(N, dtype=torch.uint8, device="cuda"), None)
        for t in range(5):
            logits = rng_tensor((N, s.A), 10 + t, -2.0, 2.0, torch.float32)
            logits[::7, 1] = float("nan")                                  # NaN scores never win
            s.env.step_policy(s.inp_rows(logits), sample=sample, seed=99, obs=obs, action_out=act, reward_sum=rsum,
                              out=out, obs_scales=(0.1, 1e-3, 0.5, 1e-6))
            got[f"obs{t}"] = s.out(obs.view(F, N))
            got[f"action{t}"] = s.out(act)
            got.update({f"{k}{t}": v for k, v in step_results(s, out).items()})
        got["reward_sum"] = s.out(rsum)
        return got
    return run


def ep_fused_live(s):
    speed = rng_tensor((s.V, N), 7, 0.5, 2.0, torch.float64)
    want = ("delay", "sleep", "buffer", "rebuffer", "reward", "latency", "end_of_video", "actions")
    out = s.env.rollout("random", STEPS, seed=13, speed=s.inp(speed), want=want)
    return {k: s.out(v) for k, v in out.items()}


def ep_fused_f32(s):
    out = s.env.rollout("random", STEPS, seed=17, dtype=torch.float32)
    got = {k: s.out(v) for k, v in out.items()}
    acts = rng_tensor((STEPS, N), 8, 0, s.A, torch.int32)
    out = s.env.rollout("fixed", STEPS, actions=s.inp(acts), dtype=torch.float32)
    got.update({"fixed_" + k: s.out(v) for k, v in out.items()})
    return got


def ep_run(s):
    want = ("delay", "sleep", "buffer", "rebuffer", "reward", "end_of_video", "actions")
    out, cost, stats = s.env.run("random", STEPS, s.inp(s.tid), s.inp(s.off), seed=21, session_base=BASE, want=want)
    got = {k: s.out(v) for k, v in out.items()}
    got["qoe_cost"] = s.out(cost)
    got["stats_counts"] = stats[list(COUNTS)]
    acts = rng_tensor((STEPS, N), 9, 0, s.A, torch.int32)
    out, cost, _ = s.env.run("fixed", STEPS, s.inp(s.tid), None, session_base=BASE, actions=s.inp(acts), want=want)
    got.update({"fixed_" + k: s.out(v) for k, v in out.items()})
    got["fixed_qoe_cost"] = s.out(cost)
    return got


def ep_run_host(pinned):
    def run(s):
        pin = (lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()) if pinned else np.ascontiguousarray
        out = dict(qoe_cost=pin(np.zeros(N)), stats=pin(np.zeros(_lib.NUM_STATS)))
        res = s.env.run_host("random", STEPS, pin(s.host_inp(s.tid)), pin(s.host_inp(s.off)), seed=23,
                             session_base=BASE, want_reward_traj=True, want_qoe_cost=True, out=out)
        as_np = lambda x: x.numpy() if isinstance(x, torch.Tensor) else x
        got = {k: torch.from_numpy(np.ascontiguousarray(s.host_out(as_np(res[k])))) for k in ("acc", "reward", "qoe_cost")}
        got["stats_counts"] = torch.from_numpy(as_np(res["stats"])[list(COUNTS)].copy())
        acts = rng_tensor((STEPS, N), 12, 0, s.A, torch.int32).numpy()
        res = s.env.run_host("fixed", STEPS, pin(s.host_inp(s.tid)), None, session_base=BASE,
                             actions=pin(s.host_inp(acts)), want_reward_traj=True)
        got["fixed_reward"] = torch.from_numpy(np.ascontiguousarray(s.host_out(res["reward"])))
        return got
    return run


def ep_mpc(mode):
    def run(s):
        got = {}
        acts = rng_tensor((4, N), 14, 0, s.A, torch.int32)
        for t in range(4):                                                # fill part of the ring first
            s.env.step(s.inp(acts[t]))
        for t in range(8):                                                # then MPC in the loop: the ring wraps
            a, j = s.env.mpc_decide(horizon=3, mode=mode, want_score=True)
            got[f"action{t}"], got[f"score{t}"] = s.out(a), s.out(j)
            s.env.step(a)
            got[f"last_pred{t}"] = s.out(s.env.state("last_pred"))
            got[f"err_ring{t}"] = s.out(s.env.state("err_ring"))
            got[f"bw_hist{t}"] = s.out(s.env.state("bw_hist"))
        return got
    return run


def ep_throughput_history(s):
    got = {}
    acts = rng_tensor((9, N), 15, 0, s.A, torch.int32)
    for t in range(9):                                                    # K = 5: before and after the ring wraps
        s.env.step(s.inp(acts[t]))
        x, n = s.env.throughput_history()
        got[f"x{t}"], got[f"n{t}"] = s.out_rows(x), s.out(n)
    return got


def ep_qoe_cost(s):
    got = {}
    acts = rng_tensor((STEPS, N), 16, 0, s.A, torch.int32)
    for t in range(STEPS):
        s.env.step(s.inp(acts[t]))
        if t % 8 == 7:
            got[f"cost{t}"] = s.out(s.env.qoe_cost())
    return got


ENTRY_POINTS = [
    ("step_f32", dict(), ep_step_f32),
    ("step_f32_hist", HIST, ep_step_f32),
    ("step_live_speed_table", LIVE, ep_step_live),
    ("step_policy_greedy", dict(track_acc=1), ep_step_policy(False)),
    ("step_policy_sampled", dict(track_acc=1), ep_step_policy(True)),
    ("fused_live", LIVE, ep_fused_live),
    ("fused_f32", dict(), ep_fused_f32),
    ("fused_f32_hist", HIST, ep_fused_f32),
    ("run", dict(track_acc=1), ep_run),
    ("run_host_pinned", dict(track_acc=1), ep_run_host(True)),
    ("run_host_pageable", dict(track_acc=1), ep_run_host(False)),
    ("mpc_decide_ref", HIST, ep_mpc("ref")),
    ("mpc_decide_robust", HIST, ep_mpc("robust")),
    ("throughput_history", HIST, ep_throughput_history),
    ("qoe_cost", dict(track_acc=1), ep_qoe_cost),
    ("qoe_cost_live", LIVE, ep_qoe_cost),
]


def bits(x):
    x = x.detach().cpu() if isinstance(x, torch.Tensor) else torch.from_numpy(np.asarray(x))
    if x.dtype == torch.float64:
        return x.contiguous().view(torch.int64)
    if x.dtype == torch.float32:
        return x.contiguous().view(torch.int32)
    return x


def assert_same(got_a, got_b):
    assert got_a.keys() == got_b.keys()
    for k in got_a:
        a, b = bits(got_a[k]), bits(got_b[k])
        assert a.shape == b.shape and a.dtype == b.dtype, k
        nd = int((a != b).sum())
        assert nd == 0, f"{k}: {nd} of {a.numel()} values differ"


def assert_same_env(a, b):
    for f in STATE:
        assert torch.equal(bits(a.env.state(f)), bits(b.out(b.env.state(f)))), f
    assert torch.equal(bits(a.env.session_acc()), bits(b.out(b.env.session_acc())))
    assert a.env.error_count() == b.env.error_count() > 0
    sa, sb = a.env.stats().cpu().numpy(), b.env.stats().cpu().numpy()
    assert np.array_equal(sa[list(COUNTS)], sb[list(COUNTS)])
    np.testing.assert_allclose(sb, sa, rtol=1e-9, atol=0)     # summed over environment positions: another order


@pytest.mark.parametrize("params,entry", [(p, e) for _, p, e in ENTRY_POINTS], ids=[n for n, _, _ in ENTRY_POINTS])
def test_sorted_environment_is_bit_identical_to_the_callers_order(params, entry):
    a, b = Side(False, params), Side(True, params)
    tid = a.tid
    bucket = np.where((tid < 0) | (tid >= N_TRACES), 0, tid)
    assert np.array_equal(b.perm, np.argsort(bucket, kind="stable"))
    assert_same(entry(a), entry(b))
    assert_same_env(a, b)


# ---- two shards on one GPU: session_base 0 and N/2, each sorted on its own ----
def shards():
    tid, off = sessions()
    h = N // 2
    full = Side(False, dict(track_acc=1), base=0, tid=tid, off=off)
    parts = [Side(True, dict(track_acc=1), n=h, base=0, tid=tid[:h], off=off[:h]),
             Side(True, dict(track_acc=1), n=N - h, base=h, tid=tid[h:], off=off[h:])]
    return full, parts, h


def test_two_sorted_shards_equal_one_environment_fused_random():
    full, parts, h = shards()
    want = full.env.rollout("random", STEPS, seed=31)
    got = [p.env.rollout("random", STEPS, seed=31) for p in parts]
    for k in want:
        cat = torch.cat([parts[0].out(got[0][k]), parts[1].out(got[1][k])], dim=-1)
        assert torch.equal(bits(want[k]), bits(cat)), k
    acc = torch.cat([parts[0].out(parts[0].env.session_acc()), parts[1].out(parts[1].env.session_acc())], dim=-1)
    assert torch.equal(bits(full.env.session_acc()), bits(acc))


def test_two_sorted_shards_equal_one_environment_sampled_step_policy():
    full, parts, h = shards()
    A = full.A
    for t in range(6):
        logits = rng_tensor((N, A), 40 + t, -1.0, 1.0, torch.float32)
        obs = full.env.step_policy(logits.cuda(), sample=True, seed=5,
                                   obs=torch.empty((4 + A) * N, dtype=torch.float32, device="cuda"),
                                   action_out=torch.empty(N, dtype=torch.int32, device="cuda"))
        want = obs.view(4 + A, N).clone()
        cat = []
        for p, rows in zip(parts, (slice(0, h), slice(h, N))):
            n = p.env.n
            o = p.env.step_policy(p.inp_rows(logits[rows]), sample=True, seed=5,
                                  obs=torch.empty((4 + A) * n, dtype=torch.float32, device="cuda"))
            cat.append(p.out(o.view(4 + A, n)))
        assert torch.equal(bits(want), bits(torch.cat(cat, dim=-1))), t
    for f in ("last_q", "buffer", "chunk", "seg", "phase"):
        st = torch.cat([parts[0].out(parts[0].env.state(f)), parts[1].out(parts[1].env.state(f))])
        assert torch.equal(bits(full.env.state(f)), bits(st)), f
