"""MPC over caller-supplied throughput scenarios (SPEC §5.7) on the device, bit for bit against the C restatement in
tests/mpc_scen_oracle.py.  Run with -m gpu.

Every compiled form and path of the scenario kernel (the ledger in test_capi_mpc_scen.py proves that SCEN_CASES reach
them all), the identities with mpc_decide_pred, no side effects under every session layout, input errors, episodes
with a torch sampler (eager and replayed from a CUDA graph), the C-ABI's error codes, and the example.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from abrsimulator_b200 import _lib
from abrsimulator_b200.env import BatchedABREnv
from oracle import oracle as orc
from helpers import bits_equal, small_world
import mpc_scen_oracle as ms
import search_forms as sf

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEQ_STATE = ("seg", "chunk", "last_q", "trace_id", "hist_len", "done", "err_len", "phase", "pos", "buffer", "bw_hist",
             "last_pred", "err_ring", "acc")
OBJ_NAME = {ms.MEAN: "mean", ms.WORST: "worst"}


def _case_env(case, seed):
    """An environment whose sessions hold the case's states (tiled), and the numpy inputs."""
    b, kw = sf.mpc_inputs(case.robust_case(), seed)
    n, T, K, H = case.n, case.tile, case.K, case.H
    rng = np.random.default_rng(2000 + seed)
    N = case.N
    env = BatchedABREnv(np.full((1, 8), 3.0), b["sizes"], b["bitrates"], N, auto_reset=case.auto_reset,
                        default_quality=0, **kw)
    env.reset(np.zeros(N, np.int32))
    done = np.zeros(n, np.uint8)
    if not case.auto_reset:
        done[len(case.hs)::5] = 1          # the first session of every horizon stays live
    if case.ties:   # dyadic throughputs and weights: every quantity exact, twin rungs tie bit for bit
        pred = rng.choice([0.25, 0.5, 1.0, 2.0], size=(n, K, H))
        w = rng.choice([0.0, 0.25, 0.5, 1.0], size=(n, K)) if case.weighted else None
    else:           # a log-uniform level per session (every rung is chosen), scenarios within a factor of 2 of it
        level = np.exp(rng.uniform(np.log(0.1), np.log(8.0), size=(n, 1, 1)))
        pred = level * np.exp(rng.uniform(-0.7, 0.7, size=(n, K, H)))
        w = rng.uniform(0.0, 3.0, size=(n, K)) * (rng.random((n, K)) < 0.7) if case.weighted else None
    if w is not None:
        w[:, 0] += 0.25
    tile = lambda x: np.ascontiguousarray(np.tile(x, (T,) + (1,) * (x.ndim - 1)))
    env.state("chunk").copy_(torch.as_tensor(tile(b["chunk"])))
    env.state("last_q").copy_(torch.as_tensor(tile(b["prev_q"])))
    env.state("buffer").copy_(torch.as_tensor(tile(b["buffer"])))
    env.state("done").copy_(torch.as_tensor(tile(done)))
    return env, b, kw, done, pred, w, tile


def twin_above(bitrates, chunk, a):
    """Rung a + 1 of the chunk is a twin of rung a (same bitrate, and in the tie worlds the same size)."""
    return a + 1 < bitrates.shape[1] and bitrates[chunk, a] == bitrates[chunk, a + 1]


@pytest.mark.parametrize("case", ms.SCEN_CASES, ids=[c.id for c in ms.SCEN_CASES])
def test_every_form_matches_the_oracle(case):
    seed = ms.SCEN_CASES.index(case)
    env, b, kw, done, pred, w, tile = _case_env(case, seed)
    exp = ms.decide_scen_c(b["sizes"], b["bitrates"], b["chunk"], b["prev_q"], b["buffer"], pred, case.H,
                           kw["chunk_length"], kw["max_buffer"], case.vw, case.rw, case.objective, w,
                           done=None if case.auto_reset else done)
    live = np.flatnonzero(done == 0) if not case.auto_reset else np.arange(case.n)
    h_got = (exp["best_seq"][live] >= 0).sum(axis=1)
    assert exp["n_errors"] == 0 and sorted(set(h_got.tolist())) == sorted(case.hs)
    assert case.A == 1 or case.rw == 0.0 or len(np.unique(exp["action"][live])) >= 2   # rw = 0: the top rung
    if case.ties:   # optima tied with the twin-rung sequence, in another prefix (step 0) and among a thread's leaves
        twin_at = lambda i: [s for s in live if exp["best_seq"][s, i] >= 0 and
                             twin_above(b["bitrates"], b["chunk"][s] + i, exp["best_seq"][s, i])]
        assert twin_at(0) and any(twin_at(h - 1) for h in case.hs)
    P = torch.as_tensor(tile(pred), device=env.device)
    W = None if w is None else torch.as_tensor(tile(w), device=env.device)
    for exhaustive in (bool(case.flags), not case.flags):     # pruned and exhaustive: identical
        act, bj, seq = env.mpc_decide_scen(P, case.H, weights=W, objective=OBJ_NAME[case.objective], want_score=True,
                                           want_seq=True, exhaustive=exhaustive)
        act, bj, seq = act.cpu().numpy(), bj.cpu().numpy(), seq.cpu().numpy()
        assert np.array_equal(act, tile(exp["action"])), exhaustive
        assert np.array_equal(seq, tile(exp["best_seq"])), exhaustive
        assert bits_equal(bj, tile(exp["best_J"])) == 0, exhaustive
    assert env.error_count() == 0


def _played_env(N=300, K=5, steps=9, seed=0, **params):
    bitrates, sizes, bw, tl, ti = small_world(n_traces=16, T=128, V=48, seed=seed, ragged=True)
    kw = dict(track_history=1, hist_k=K, max_buffer=30.0)
    kw.update(params)
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, **kw)
    rng = np.random.default_rng(seed)
    env.reset(rng.integers(0, 16, size=N).astype(np.int32), rng.uniform(0, 100, size=N))
    env.rollout("random", steps, seed=seed + 1, want=())
    return env, (bitrates, sizes, bw, tl, ti), kw


@pytest.mark.parametrize("H,exhaustive", [(1, False), (3, False), (5, False), (5, True), (7, False)])
def test_identities_with_the_prediction_decision(H, exhaustive):
    """K = 1 (no weights, either objective; MEAN with w = 1) and K identical rows under WORST: mpc_decide_pred on the
    row, bit for bit."""
    N = 2048 if H < 7 else 64
    env, _, _ = _played_env(N=N, K=6, steps=11 if H != 7 else 43)
    rng = np.random.default_rng(H)
    row = torch.as_tensor(rng.uniform(0.3, 6.0, size=(N, H)), device=env.device)
    ref = env.mpc_decide_pred(row, H, want_score=True, want_seq=True, exhaustive=exhaustive)
    ones = torch.ones(N, 1, dtype=torch.float64, device=env.device)
    for scen, obj, w in ((row[:, None], "mean", None), (row[:, None], "worst", None), (row[:, None], "mean", ones),
                         (row[:, None].expand(N, 5, H), "worst", None)):
        got = env.mpc_decide_scen(scen, H, weights=w, objective=obj, want_score=True, want_seq=True,
                                  exhaustive=exhaustive)
        assert torch.equal(got[0], ref[0]) and torch.equal(got[2], ref[2]), obj
        assert bits_equal(got[1].cpu().numpy(), ref[1].cpu().numpy()) == 0, obj
    assert len(torch.unique(ref[0])) >= 2


def _state_bytes(env):
    return {f: env.state(f).clone() for f in SEQ_STATE}


@pytest.mark.parametrize("variant", ["history", "no_history", "live", "sorted"])
def test_no_state_changes_and_environment_order(variant):
    params = dict(no_history=dict(track_history=0), live=dict(live=1), history={}, sorted={})[variant]
    env, world, kw = _played_env(N=257, K=5, steps=7, seed=3, track_acc=1, **params)
    H, K = 4, 6
    if variant == "sorted":
        tid = env.state("trace_id").cpu().numpy()
        env.reset(tid, sort_by_trace=True)
        env.rollout("random", 6, seed=9, want=())
        assert env.perm is not None and not torch.equal(env.perm.cpu(), torch.arange(257, dtype=torch.int32))
    rng = np.random.default_rng(5)
    pred = rng.uniform(0.3, 6.0, size=(257, K, H))
    w = rng.uniform(0.0, 1.0, size=(257, K))
    p = env.params
    util = orc.utility_table(world[0], p.utility_mode, p.utility_scale)
    perm = env.perm.long().cpu().numpy() if variant == "sorted" else np.arange(257)
    for obj, ww in (("mean", w), ("worst", None)):
        # the caller's tables are per session; the rows passed are in environment order (position p holds session
        # perm[p]), and the results are mapped back through perm
        rows = lambda x: torch.as_tensor(np.ascontiguousarray(x[perm]), device=env.device)
        before = _state_bytes(env)
        e0 = env.error_count()
        act, bj, seq = env.mpc_decide_scen(rows(pred), H, weights=None if ww is None else rows(ww), objective=obj,
                                           want_score=True, want_seq=True)
        torch.cuda.synchronize()
        for f, t in before.items():
            assert torch.equal(env.state(f).view(torch.uint8), t.view(torch.uint8)), f
        assert env.error_count() == e0
        exp = ms.decide_scen_c(world[1], util, env.state("chunk").cpu().numpy(), env.state("last_q").cpu().numpy(),
                               env.state("buffer").cpu().numpy(), pred[perm], H, p.chunk_length, p.max_buffer,
                               p.smooth_penalty, p.rebuf_penalty, ms.OBJECTIVES[obj], None if ww is None else ww[perm])
        got_a, got_s = np.empty(257, np.int32), np.empty((257, H), np.int32)
        got_a[perm], got_s[perm] = act.cpu().numpy(), seq.cpu().numpy()
        want_a, want_s = np.empty(257, np.int32), np.empty((257, H), np.int32)
        want_a[perm], want_s[perm] = exp["action"], exp["best_seq"]
        assert np.array_equal(got_a, want_a) and np.array_equal(got_s, want_s)
        assert bits_equal(bj.cpu().numpy(), exp["best_J"]) == 0


def test_input_errors_are_counted_once_per_session():
    env, _, _ = _played_env(N=10, K=5, steps=2, seed=6)
    H, K = 5, 3
    assert int(env.state("chunk").max()) + H <= 48
    dev = env.device
    pred = torch.full((10, K, H), 2.0, dtype=torch.float64, device=dev)
    pred[1, 0, 0], pred[2, 1, 4], pred[3, 2, 2] = 0.0, float("nan"), float("inf")
    pred[4, 0, 1], pred[4, 2, 3] = -1.0, -2.0                 # two bad entries, one error
    w = torch.ones(10, K, dtype=torch.float64, device=dev)
    w[5, 1], w[6] = -0.5, 0.0
    w[7, 0] = float("nan")
    for obj, ww, bad in (("mean", w, [1, 2, 3, 4, 5, 6, 7]), ("worst", None, [1, 2, 3, 4])):
        e0 = env.error_count()
        a, bj = env.mpc_decide_scen(pred, H, weights=ww, objective=obj, want_score=True)
        good = [s for s in range(10) if s not in bad]
        assert (a[bad] == -1).all() and (a[good] >= 0).all() and torch.isnan(bj[bad]).all(), obj
        assert env.error_count() == e0 + len(bad), obj
    # NaN past the truncated horizon is not read
    env.state("chunk").fill_(45)                               # h = 3 of 5
    p2 = torch.full((10, K, H), 2.0, dtype=torch.float64, device=dev)
    p2[:, :, 3:] = float("nan")
    e0 = env.error_count()
    a = env.mpc_decide_scen(p2, H)
    assert (a >= 0).all() and env.error_count() == e0


def test_error_codes_and_precedence():
    lib = _lib.load()
    env, _, _ = _played_env(N=8, K=5, steps=2)
    dev = env.device
    act = torch.empty(8, dtype=torch.int32, device=dev)
    pred = torch.full((8, 4, 5), 2.0, dtype=torch.float64, device=dev)
    wt = torch.ones(8, 4, dtype=torch.float64, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    A = lambda t: None if t is None else t.data_ptr()

    def call(e, H=5, K=4, obj=0, flags=0, p=pred, w=None, a=act):
        rc = lib.abr_env_mpc_decide_scen(e, H, K, obj, flags, A(p), A(w), A(a), None, None, st)
        return rc, lib.abr_last_error().decode()

    everything_wrong = dict(H=99, K=77, obj=5, flags=3, p=None, w=wt, a=None)
    rc, msg = call(None, **everything_wrong)
    assert rc == 1 and "env is NULL" in msg
    fresh = BatchedABREnv(np.full((1, 8), 3.0), np.ones((4, 3)), np.ones((4, 3)), 4)
    rc, msg = call(fresh._h, **everything_wrong)
    assert rc == 4 and "reset" in msg
    fresh.reset(np.zeros(0, np.int32))
    assert call(fresh._h, **everything_wrong)[0] == 0                        # empty batch: no-op
    rc, msg = call(env._h, **everything_wrong)
    assert rc == 1 and "action is NULL" in msg
    rc, msg = call(env._h, **dict(everything_wrong, a=act))
    assert rc == 1 and "pred is NULL" in msg
    rc, msg = call(env._h, H=99, K=77, obj=5, flags=3, w=wt)
    assert rc == 1 and "objective" in msg
    rc, msg = call(env._h, H=99, K=77, obj=1, flags=3, w=wt)
    assert rc == 1 and "weights" in msg
    rc, msg = call(env._h, H=99, K=77, obj=1, flags=3)
    assert rc == 1 and "flags" in msg
    for flags in (_lib.MPC_TRUNCATE, _lib.MPC_EMPTY_DEFAULT, _lib.MPC_PRED_SES, _lib.MPC_MODE_EXHAUSTIVE):
        assert call(env._h, H=99, K=77, flags=flags)[0] == 1
    for H in (0, 9, 99):
        rc, msg = call(env._h, H=H, K=77)
        assert rc == 3 and "horizon" in msg
    big = BatchedABREnv(np.full((1, 8), 3.0), np.ones((40, 16)), np.ones((40, 16)), 4)
    big.reset(np.zeros(4, np.int32))
    rc, msg = call(big._h, H=8, K=77)
    assert rc == 3 and "2^31" in msg
    for K in (0, 17, -1):
        rc, msg = call(env._h, K=K)
        assert rc == 3 and "n_scen" in msg
    assert call(env._h, K=4, flags=_lib.MPC_EXHAUSTIVE, w=wt)[0] == 0
    assert call(env._h, K=4, obj=1)[0] == 0
    # the Python layer
    with pytest.raises(ValueError):
        env.mpc_decide_scen(pred[:, :, :4], 5)
    with pytest.raises(ValueError):
        env.mpc_decide_scen(pred, 5, weights=wt[:, :3])
    with pytest.raises(ValueError):
        env.mpc_decide_scen(pred, 5, objective="median")
    with pytest.raises(TypeError):
        env.mpc_decide_scen(pred.cpu(), 5)
    with pytest.raises(_lib.AbrError):
        env.mpc_decide_scen(torch.full((8, 17, 5), 2.0, dtype=torch.float64, device=dev), 5)
    a32 = env.mpc_decide_scen(pred.float(), 5)
    assert torch.equal(a32, env.mpc_decide_scen(pred, 5))
    flat = pred[:, :, 0].contiguous()
    assert torch.equal(env.mpc_decide_scen(flat, 5), env.mpc_decide_scen(pred, 5))


class FlatSampler:
    """Deterministic torch sampler: the last K throughput samples as flat scenarios, weight 1/n, missing samples a
    placeholder with weight 0, and one fallback scenario without history.  Device ops only."""

    def __init__(self, fallback=3.0):
        self.fallback = fallback

    def __call__(self, env):
        x, n = env.throughput_history()
        have = ~torch.isnan(x)
        scen = torch.where(have, x, torch.full_like(x, self.fallback))
        w = have.to(torch.float64) / n.clamp(min=1).to(torch.float64)[:, None]
        w[:, 0] = torch.where(n > 0, w[:, 0], torch.ones_like(w[:, 0]))
        return scen, w


def _sampler_reference(ref, fallback=3.0):
    hl, ring, K = ref.field("hist_len"), ref.field("bw_hist"), ref.K
    N = len(hl)
    scen = np.full((N, K), fallback)
    w = np.zeros((N, K))
    for s in range(N):
        m = min(hl[s], K)
        start = 0 if hl[s] <= K else hl[s] % K
        for j in range(m):
            scen[s, j] = ring[s, (start + j) % K]
            w[s, j] = 1.0 / m
        if m == 0:
            w[s, 0] = 1.0
    return scen, w


@pytest.mark.parametrize("auto_reset,objective", [(1, "mean"), (0, "worst")])
def test_episode_with_a_torch_sampler_matches_the_oracle(auto_reset, objective):
    N, steps, H = 193, 48, 5
    bitrates, sizes, bw, tl, ti = small_world(n_traces=16, T=128, V=20, seed=4, ragged=True)
    kw = dict(track_history=1, hist_k=5, max_buffer=30.0, auto_reset=auto_reset, track_acc=1)
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, **kw)
    rng = np.random.default_rng(11)
    tid, off = rng.integers(0, 16, size=N).astype(np.int32), rng.uniform(0, 100, size=N)
    env.reset(tid, off)
    ref = orc.OracleEnv(bw, tl, ti, sizes, bitrates, N, **dict(orc.DEFAULTS, **{k: v for k, v in kw.items()
                                                                                if k != "track_acc"}))
    ref.reset(tid, off)
    acc = np.zeros((orc.NUM_ACC, N))
    obj = ms.OBJECTIVES[objective]
    for _ in range(steps):
        scen, w = _sampler_reference(ref)
        pred = np.repeat(scen[:, :, None], H, axis=2)
        r = ms.env_decide_scen(ref, pred, H, obj, w if obj == ms.MEAN else None)
        assert r["n_errors"] == 0
        ref.step(r["action"], acc=acc)
    sampler = FlatSampler()
    smp = sampler if objective == "mean" else (lambda e: sampler(e)[0])
    env.mpc_episode_scen(steps, smp, H, objective=objective)
    assert bits_equal(env.session_acc().cpu().numpy(), acc) == 0
    assert env.error_count() == 0 and (acc[0] != 0).all()

    # one chunk captured in a CUDA graph and replayed equals the eager run
    env2 = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, **kw)
    env2.reset(tid, off)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        env2.mpc_episode_scen(1, smp, H, objective=objective)       # warm-up chunk
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        env2.mpc_episode_scen(1, smp, H, objective=objective)
    for _ in range(steps - 1):
        g.replay()
    torch.cuda.synchronize()
    assert bits_equal(env2.session_acc().cpu().numpy(), acc) == 0


def scen_smem_bytes(A, H, K, wps):
    """Dynamic shared memory of a launch (launch_mpc_scen: scen_slot_doubles per session slot, plus the scratch)."""
    return 8 * ((4 // wps) * (H * A + K * H * A + A * A + K + 2 * A + 8) + 2 * K * 128)


@pytest.mark.parametrize("H,tile,wps", [(3, 1, 1), (7, 1, 4), (7, 400, 1)])
def test_sixteen_scenarios_past_the_default_shared_memory(H, tile, wps):
    """K = 16 with A = 16: 69 KB at H = 3 with a warp per session, 50 KB at H = 7 with a block per session, and 104 KB
    at H = 7 with a warp per session (the largest legal shape), all past the 48 KB default."""
    rng = np.random.default_rng(21 + H)
    V, A, K, n = 12, 16, 16, 6
    N = n * tile
    assert ms.scen_form(A, H, 1, N, ms.MEAN, 0, 1.0, 4.3)[0][0] == wps
    assert scen_smem_bytes(A, H, K, wps) > 48 * 1024
    lad = np.sort(rng.uniform(0.2, 5.0, size=A))
    bitrates = np.tile(lad, (V, 1))
    sizes = bitrates * 4.0 * rng.uniform(0.8, 1.2, size=(V, A))
    env = BatchedABREnv(np.full((1, 8), 3.0), sizes, bitrates, N, max_buffer=30.0)
    env.reset(np.zeros(N, np.int32))
    chunk = np.array([0, 3, 5, 8, 10, 11] if H == 3 else [8, 9, 10, 11, 8, 10], np.int32)   # h <= 4 at H = 7
    prev_q = rng.integers(-1, A, size=n).astype(np.int32)
    tiled = lambda x: np.ascontiguousarray(np.tile(x, (tile,) + (1,) * (x.ndim - 1)))
    env.state("chunk").copy_(torch.as_tensor(tiled(chunk)))
    env.state("last_q").copy_(torch.as_tensor(tiled(prev_q)))
    buf = env.state("buffer").cpu().numpy()[:n]
    pred = np.exp(rng.uniform(np.log(0.5), np.log(30.0), size=(n, K, H)))
    p = env.params
    util = orc.utility_table(bitrates, p.utility_mode, p.utility_scale)
    for obj in ("mean", "worst"):
        for exhaustive in (False, True):
            act, bj, seq = env.mpc_decide_scen(torch.as_tensor(tiled(pred), device=env.device), H, objective=obj,
                                               want_score=True, want_seq=True, exhaustive=exhaustive)
            exp = ms.decide_scen_c(sizes, util, chunk, prev_q, buf, pred, H, p.chunk_length, p.max_buffer,
                                   p.smooth_penalty, p.rebuf_penalty, ms.OBJECTIVES[obj])
            assert np.array_equal(act.cpu().numpy(), tiled(exp["action"]))
            assert np.array_equal(seq.cpu().numpy(), tiled(exp["best_seq"]))
            assert bits_equal(bj.cpu().numpy(), tiled(exp["best_J"])) == 0
    assert env.error_count() == 0


def test_no_finite_aggregate_gives_sequence_zero():
    """A subnormal throughput is valid, but sizes / p overflows to inf: every sequence then rebuffers forever.  With
    rw > 0 every Q is -inf; with rw = 0, or MEAN with weight 0 on that scenario, every Q is NaN.  SPEC §5.7: sequence 0,
    best_j = +inf, as the C oracle restates."""
    for rw in (4.3, 0.0):
        env, world, _ = _played_env(N=12, K=5, steps=3, seed=7, rebuf_penalty=rw)
        H, K = 4, 2
        pred = np.full((12, K, H), 2.0)
        pred[:, 0, 1] = 1e-310
        p = env.params
        util = orc.utility_table(world[0], p.utility_mode, p.utility_scale)
        st = [env.state(f).cpu().numpy() for f in ("chunk", "last_q", "buffer")]
        for obj, w in (("worst", None), ("mean", None), ("mean", np.tile([0.0, 1.0], (12, 1)))):
            exp = ms.decide_scen_c(world[1], util, *st, pred, H, p.chunk_length, p.max_buffer, p.smooth_penalty, rw,
                                   ms.OBJECTIVES[obj], w)
            assert (exp["action"] == 0).all() and (exp["best_J"] == np.inf).all() and exp["n_errors"] == 0
            for exhaustive in (False, True):
                act, bj, seq = env.mpc_decide_scen(torch.as_tensor(pred, device=env.device), H,
                                                   weights=None if w is None else torch.as_tensor(w, device=env.device),
                                                   objective=obj, want_score=True, want_seq=True, exhaustive=exhaustive)
                assert np.array_equal(act.cpu().numpy(), exp["action"]) and np.array_equal(seq.cpu().numpy(),
                                                                                         exp["best_seq"])
                assert bits_equal(bj.cpu().numpy(), exp["best_J"]) == 0
        assert env.error_count() == 0


def test_the_draw_counter_is_not_advanced():
    """Sampled policy steps after a decision draw what they draw without it: the decision leaves the counter alone."""
    a, _, _ = _played_env(N=64, K=5, steps=3, seed=9)
    b, _, _ = _played_env(N=64, K=5, steps=3, seed=9)
    logits = torch.zeros(64, a.A, dtype=torch.float32, device=a.device)
    a.step_policy(logits, sample=True, seed=5)
    b.step_policy(logits, sample=True, seed=5)
    pred = torch.full((64, 3, 4), 2.0, dtype=torch.float64, device=a.device)
    a.mpc_decide_scen(pred, 4)
    a.mpc_decide_scen(pred, 4, objective="worst", exhaustive=True)
    acts = []
    for _ in range(3):
        a.step_policy(logits, sample=True, seed=5)
        b.step_policy(logits, sample=True, seed=5)
        assert torch.equal(a.state("last_q"), b.state("last_q")) and torch.equal(a.state("buffer"), b.state("buffer"))
        acts.append(a.state("last_q")[:64].clone())
    assert not torch.equal(acts[0], acts[1])        # the sampled actions vary from step to step


def test_example_runs():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "examples", "mpc_scenarios.py"), "--sessions", "512",
                        "--steps", "12", "--check"], capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
    for name in ("robust MPC", "scenario MPC, mean", "scenario MPC, worst", "lookahead"):
        assert name in r.stdout, r.stdout
    assert "graph replay matches the eager run bit for bit" in r.stdout, r.stdout
