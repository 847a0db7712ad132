"""MPC over caller-supplied throughput predictions (SPEC §5.6) on the device, bit for bit against the C restatement in
tests/mpc_pred_oracle.py.  Run with -m gpu.

Every compiled form of the caller-prediction kernels (the ledger in test_capi_mpc_pred.py proves that PRED_CASES reach
them all), the identity with the robust decision, no side effects, episodes with a torch predictor (eager and replayed
from a CUDA graph), the C-ABI's error codes, and a full-size call.
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
from abrsimulator_b200.mpc import decide_batch
from oracle import oracle as orc
from helpers import bits_equal, small_world
import mpc_pred_oracle as mp
import search_forms as sf

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEQ_STATE = ("seg", "chunk", "last_q", "trace_id", "hist_len", "done", "err_len", "phase", "pos", "buffer", "bw_hist",
             "last_pred", "err_ring", "acc")


def _case_env(case, seed):
    """An environment whose sessions hold the case's states (tiled), and the numpy inputs."""
    b, kw = sf.mpc_inputs(case.robust_case(), seed)
    V, n, T = sf.MPC_V, case.n, case.tile
    rng = np.random.default_rng(1000 + seed)
    N = case.N
    env = BatchedABREnv(np.full((1, 8), 3.0), b["sizes"], b["bitrates"], N, auto_reset=case.auto_reset,
                        default_quality=0, **kw)
    env.reset(np.zeros(N, np.int32))
    done = np.zeros(n, np.uint8)
    if not case.auto_reset:
        done[len(case.hs)::5] = 1          # the first session of every horizon stays live
    pred = np.exp(rng.uniform(np.log(0.1), np.log(8.0), size=(n, case.H)))   # log-uniform: every rung is chosen
    tile = lambda x: np.ascontiguousarray(np.tile(x, (T,) + (1,) * (x.ndim - 1)))
    env.state("chunk").copy_(torch.as_tensor(tile(b["chunk"])))
    env.state("last_q").copy_(torch.as_tensor(tile(b["prev_q"])))
    env.state("buffer").copy_(torch.as_tensor(tile(b["buffer"])))
    env.state("done").copy_(torch.as_tensor(tile(done)))
    return env, b, kw, done, pred, tile


@pytest.mark.parametrize("case", mp.PRED_CASES, ids=[c.id for c in mp.PRED_CASES])
def test_every_form_matches_the_oracle(case):
    seed = mp.PRED_CASES.index(case)
    env, b, kw, done, pred, tile = _case_env(case, seed)
    exp = mp.decide_pred_c(b["sizes"], b["bitrates"], b["chunk"], b["prev_q"], b["buffer"], pred, case.H,
                           kw["chunk_length"], kw["max_buffer"], case.vw, case.rw,
                           done=None if case.auto_reset else done)
    live = np.flatnonzero(done == 0) if not case.auto_reset else np.arange(case.n)
    h_got = (exp["best_seq"][live] >= 0).sum(axis=1)
    assert exp["n_errors"] == 0 and sorted(set(h_got.tolist())) == sorted(case.hs)
    assert case.A == 1 or len(np.unique(exp["action"][live])) >= 2
    P = torch.as_tensor(tile(pred), device=env.device)
    for exhaustive in (bool(case.flags), not case.flags):     # pruned and exhaustive: identical
        act, bj, seq = env.mpc_decide_pred(P, case.H, want_score=True, want_seq=True, exhaustive=exhaustive)
        act, bj, seq = act.cpu().numpy(), bj.cpu().numpy(), seq.cpu().numpy()
        assert np.array_equal(act, tile(exp["action"])), exhaustive
        assert np.array_equal(seq, tile(exp["best_seq"])), exhaustive
        assert bits_equal(bj, tile(exp["best_J"])) == 0, exhaustive
    assert env.error_count() == 0


def _played_env(N=300, K=5, steps=9, seed=0, **params):
    """An environment after `steps` random-policy steps, so that every session has history and robust state."""
    bitrates, sizes, bw, tl, ti = small_world(n_traces=16, T=128, V=48, seed=seed, ragged=True)
    kw = dict(track_history=1, hist_k=K, max_buffer=30.0)
    kw.update(params)
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, **kw)
    rng = np.random.default_rng(seed)
    env.reset(rng.integers(0, 16, size=N).astype(np.int32), rng.uniform(0, 100, size=N))
    env.rollout("random", steps, seed=seed + 1, want=())
    return env, (bitrates, sizes, bw, tl, ti), kw


@pytest.mark.parametrize("H,exhaustive", [(1, False), (3, False), (5, False), (5, True), (7, False)])
def test_robust_predictions_reproduce_the_robust_decision(H, exhaustive):
    """pred[s][i] = c_s, the robust prediction of the state: the robust decision, bit for bit."""
    N = 2048 if H < 7 else 64
    env, _, _ = _played_env(N=N, K=6, steps=11 if H != 7 else 43)
    assert int(env.state("hist_len").min()) >= 1
    ring = env.state("bw_hist").t().contiguous()
    out = decide_batch(env.state("sizes"), env.state("utility"), env.state("chunk").clone(),
                       env.state("last_q").clone(), env.state("buffer").clone(), ring, env.state("hist_len").clone(), H,
                       mode="robust", flags=_lib.MPC_EXHAUSTIVE if exhaustive else 0, params=env.params,
                       last_pred=env.state("last_pred").clone(), err_ring=env.state("err_ring").t().contiguous(),
                       err_len=env.state("err_len").clone())
    c = out["preds"][:, 0].contiguous()
    act, bj, seq = env.mpc_decide_pred(c, H, want_score=True, want_seq=True, exhaustive=exhaustive)
    assert torch.equal(act, out["action"]) and torch.equal(seq, out["best_seq"])
    assert bits_equal(bj.cpu().numpy(), out["best_j"].cpu().numpy()) == 0
    assert len(torch.unique(act)) >= 2
    if H == 7:
        assert int((seq >= 0).sum(1).min()) < H        # sessions near the end of the video
    a2, bj2 = env.mpc_decide(H, mode="robust", want_score=True, exhaustive=exhaustive)
    assert torch.equal(a2, act) and bits_equal(bj2.cpu().numpy(), bj.cpu().numpy()) == 0


def _state_bytes(env):
    return {f: env.state(f).clone() for f in SEQ_STATE}


@pytest.mark.parametrize("variant", ["history", "no_history", "live", "sorted"])
def test_no_state_changes_and_environment_order(variant):
    params = dict(no_history=dict(track_history=0), live=dict(live=1), history={}, sorted={})[variant]
    env, world, kw = _played_env(N=257, K=5, steps=7, seed=3, **params)
    H = 4
    if variant == "sorted":
        tid = env.state("trace_id").cpu().numpy()
        env.reset(tid, sort_by_trace=True)
        env.rollout("random", 6, seed=9, want=())
        assert env.perm is not None and not torch.equal(env.perm.cpu(), torch.arange(257, dtype=torch.int32))
    rng = np.random.default_rng(5)
    pred = rng.uniform(0.3, 6.0, size=(257, H))
    before = _state_bytes(env)
    e0 = env.error_count()
    act, bj, seq = env.mpc_decide_pred(torch.as_tensor(pred, device=env.device), H, want_score=True, want_seq=True)
    torch.cuda.synchronize()
    for f, t in before.items():
        assert torch.equal(env.state(f).view(torch.uint8), t.view(torch.uint8)), f
    assert env.error_count() == e0
    p = env.params
    util = orc.utility_table(world[0], p.utility_mode, p.utility_scale)
    exp = mp.decide_pred_c(world[1], util, env.state("chunk").cpu().numpy(), env.state("last_q").cpu().numpy(),
                           env.state("buffer").cpu().numpy(), pred, H, p.chunk_length, p.max_buffer, p.smooth_penalty,
                           p.rebuf_penalty)
    assert np.array_equal(act.cpu().numpy(), exp["action"]) and np.array_equal(seq.cpu().numpy(), exp["best_seq"])
    assert bits_equal(bj.cpu().numpy(), exp["best_J"]) == 0
    if variant == "no_history":
        with pytest.raises(ValueError):
            env.throughput_history()


def test_throughput_history_is_the_ring_oldest_first():
    env, _, _ = _played_env(N=40, K=5, steps=13, seed=2)
    x, n = env.throughput_history()
    ring, hl = env.state("bw_hist").cpu().numpy(), env.state("hist_len").cpu().numpy()
    K = env.K
    for s in range(40):
        m = min(hl[s], K)
        start = 0 if hl[s] <= K else hl[s] % K
        want = [ring[(start + j) % K, s] for j in range(m)]
        assert n[s] == m and x[s, :m].cpu().tolist() == want and torch.isnan(x[s, m:]).all()


STEP_SCALE = [1.0, 0.75, 1.25, 0.5, 1.0]


class LastSamplePredictor:
    """Deterministic torch predictor: the newest throughput sample, scaled per step (3.0 before the first sample).
    Device ops only, so that a chunk can be captured in a CUDA graph."""

    def __init__(self, device):
        self.scale = torch.tensor(STEP_SCALE, dtype=torch.float64, device=device)

    def __call__(self, env):
        x, n = env.throughput_history()
        last = x.gather(1, (n.long() - 1).clamp(min=0)[:, None])[:, 0]
        last = torch.where(n > 0, last, torch.full_like(last, 3.0))
        return last[:, None] * self.scale


@pytest.mark.parametrize("auto_reset", [1, 0])
def test_episode_with_a_torch_predictor_matches_the_oracle(auto_reset):
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
    for _ in range(steps):
        hl, ring = ref.field("hist_len"), ref.field("bw_hist")
        last = np.array([ring[s, (hl[s] - 1) % ref.K] if hl[s] > 0 else 3.0 for s in range(N)])
        pred = last[:, None] * np.array(STEP_SCALE)
        r = mp.env_decide_pred(ref, pred, H)
        assert r["n_errors"] == 0
        ref.step(r["action"], acc=acc)
    predictor = LastSamplePredictor(env.device)
    env.mpc_episode_pred(steps, predictor, H)
    got = env.session_acc().cpu().numpy()
    assert bits_equal(got, acc) == 0
    assert env.error_count() == 0 and (acc[0] != 0).all()

    # one chunk captured in a CUDA graph and replayed equals the eager run
    env2 = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, **kw)
    env2.reset(tid, off)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        env2.mpc_episode_pred(1, predictor, H)       # warm-up chunk (allocations, first launches)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        env2.mpc_episode_pred(1, predictor, H)
    for _ in range(steps - 1):
        g.replay()
    torch.cuda.synchronize()
    assert bits_equal(env2.session_acc().cpu().numpy(), acc) == 0


def test_error_codes_and_precedence():
    lib = _lib.load()
    env, _, _ = _played_env(N=8, K=5, steps=2)
    dev = env.device
    act = torch.empty(8, dtype=torch.int32, device=dev)
    pred = torch.full((8, 5), 2.0, dtype=torch.float64, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    A = lambda t: None if t is None else t.data_ptr()

    def call(e, H=5, flags=0, p=pred, a=act):
        rc = lib.abr_env_mpc_decide_pred(e, H, flags, A(p), A(a), None, None, st)
        return rc, lib.abr_last_error().decode()

    rc, msg = call(None, H=99, flags=3, p=None, a=None)
    assert rc == 1 and "env is NULL" in msg
    fresh = BatchedABREnv(np.full((1, 8), 3.0), np.ones((4, 3)), np.ones((4, 3)), 4)
    rc, msg = call(fresh._h, H=99, flags=3, p=None, a=None)
    assert rc == 4 and "reset" in msg
    fresh.reset(np.zeros(0, np.int32))
    assert call(fresh._h, H=99, flags=3, p=None, a=None)[0] == 0            # empty batch: no-op
    rc, msg = call(env._h, H=99, flags=3, p=None, a=None)
    assert rc == 1 and "action is NULL" in msg
    rc, msg = call(env._h, H=99, flags=3, p=None)
    assert rc == 1 and "pred is NULL" in msg
    rc, msg = call(env._h, H=99, flags=3)
    assert rc == 1 and "flags" in msg
    for flags in (_lib.MPC_TRUNCATE, _lib.MPC_EMPTY_DEFAULT, _lib.MPC_PRED_SES, _lib.MPC_MODE_EXHAUSTIVE):
        assert call(env._h, H=99, flags=flags)[0] == 1
    for H in (0, 9, 99):
        rc, msg = call(env._h, H=H)
        assert rc == 3 and "horizon" in msg
    assert call(env._h, H=5, flags=_lib.MPC_EXHAUSTIVE)[0] == 0
    big = BatchedABREnv(np.full((1, 8), 3.0), np.ones((40, 16)), np.ones((40, 16)), 4)
    big.reset(np.zeros(4, np.int32))
    rc, msg = call(big._h, H=8)
    assert rc == 3 and "2^31" in msg
    # invalid predictions: action -1, the session counted once
    e0 = env.error_count()
    bad = pred.clone()
    bad[1, 0], bad[3, 4], bad[5, 2] = 0.0, float("nan"), -float("inf")
    a = env.mpc_decide_pred(bad, 5)
    assert (a[[1, 3, 5]] == -1).all() and (a[[0, 2, 4, 6, 7]] >= 0).all()
    assert env.error_count() == e0 + 3
    with pytest.raises(ValueError):
        env.mpc_decide_pred(pred[:, :4], 5)
    with pytest.raises(TypeError):
        env.mpc_decide_pred(pred.cpu(), 5)
    a32 = env.mpc_decide_pred(pred.float(), 5)
    assert torch.equal(a32, env.mpc_decide_pred(pred, 5))
    assert torch.equal(env.mpc_decide_pred(pred[:, 0].contiguous(), 5), env.mpc_decide_pred(pred, 5))


def test_full_size_call_on_a_strided_sample():
    N, H = 131072, 5
    env, world, _ = _played_env(N=N, K=5, steps=6, seed=8)
    rng = np.random.default_rng(8)
    pred = rng.uniform(0.3, 6.0, size=(N, H))
    act, bj, seq = env.mpc_decide_pred(torch.as_tensor(pred, device=env.device), H, want_score=True, want_seq=True)
    idx = np.arange(0, N, 61)
    p = env.params
    util = orc.utility_table(world[0], p.utility_mode, p.utility_scale)
    exp = mp.decide_pred_c(world[1], util, env.state("chunk").cpu().numpy()[idx], env.state("last_q").cpu().numpy()[idx],
                           env.state("buffer").cpu().numpy()[idx], pred[idx], H, p.chunk_length, p.max_buffer,
                           p.smooth_penalty, p.rebuf_penalty)
    assert np.array_equal(act.cpu().numpy()[idx], exp["action"])
    assert np.array_equal(seq.cpu().numpy()[idx], exp["best_seq"])
    assert bits_equal(bj.cpu().numpy()[idx], exp["best_J"]) == 0
    assert len(np.unique(exp["action"])) >= 3


def test_example_runs():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "examples", "mpc_predictor.py"), "--sessions", "512",
                        "--steps", "12", "--graph"], capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "robust MPC" in r.stdout and "lookahead" in r.stdout
