"""GPU: the windowed observation of the policy-in-the-loop step (SPEC §4.5), bit for bit — run with -m gpu.

Against the numpy restatement on top of the C oracle (tests/obs_window_oracle.py) after every step; against
``step_policy`` on a twin environment for everything but the observation; ``observe_window``; installed session
orders; CUDA-graph replay; the C-ABI's checks in their order; and the example's two paths.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from abrsimulator_b200 import _lib
from abrsimulator_b200.env import BatchedABREnv, StepResult
from oracle import oracle as orc
import obs_window_oracle as wo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STATE = ("seg", "chunk", "last_q", "trace_id", "phase", "pos", "buffer", "done", "hist_len", "bw_hist", "acc",
         "last_pred", "err_len")
SCALES = (0.5, 0.1, 1e-3, 0.25, 1e-2)


def u32(x):
    return np.ascontiguousarray(x, np.float32).view(np.uint32)


def one_hot(actions, A):
    a = torch.as_tensor(actions, device="cuda").long()
    return torch.nn.functional.one_hot(a, A).float().contiguous()


def pair(N, A, V=48, seed=0, **params):
    bitrates, sizes, bw, tl, ti = wo.world(A, V=V, seed=seed)
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, **params)
    ref = orc.OracleEnv(bw, tl, ti, sizes, bitrates, N, **params)
    tid, off = wo.sessions(N, bw.shape[0], bw.shape[1], seed=11 + seed)
    return env, ref, tid, off


def twins(N, A, V=20, **params):
    bitrates, sizes, bw, tl, ti = wo.world(A, V=V)
    tid, off = wo.sessions(N, bw.shape[0], bw.shape[1])
    envs = [BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, **params) for _ in range(2)]
    for e in envs:
        e.reset(tid, off)
    return envs, tid, off


@pytest.mark.parametrize("W, A, N, V, auto_reset, hist, acc, dq", wo.CASES,
                         ids=[f"W{c[0]}-A{c[1]}-N{c[2]}-V{c[3]}-ar{c[4]}-h{c[5]}-acc{c[6]}" for c in wo.CASES])
def test_every_step_matches_the_restatement(W, A, N, V, auto_reset, hist, acc, dq):
    params = dict(auto_reset=auto_reset, track_history=hist, track_acc=acc, default_quality=dq)
    env, ref, tid, off = pair(N, A, V=V, **params)
    env.reset(tid, off)
    ref.reset(tid, off)
    w = wo.WindowObs(ref, W, SCALES)
    obs = env.observe_window(W, SCALES)
    assert np.array_equal(u32(obs.cpu().numpy()), u32(w.observe()))
    acts = wo.action_table(wo.STEPS, N, A)
    for t in range(wo.STEPS):
        env.step_policy_window(one_hot(acts[t], A), obs, sample=False, scales=SCALES)
        w.step(acts[t])
        got = obs.cpu().numpy()
        bad = np.nonzero((u32(got) != u32(w.obs)).any(axis=1))[0]
        assert bad.size == 0, f"step {t}: rows {bad.tolist()} differ"
    assert env.error_count() == 0 and ref.errors() == 0
    for f in ("chunk", "last_q", "buffer"):
        assert np.array_equal(env.state(f).cpu().numpy(), ref.field(f)), f


@pytest.mark.parametrize("sample", [False, True])
@pytest.mark.parametrize("auto_reset", [0, 1])
def test_everything_but_the_observation_is_step_policy(sample, auto_reset):
    N, W = 3000, 8
    (ea, eb), _, _ = twins(N, 6, auto_reset=auto_reset, track_history=1, track_acc=1)
    A, dev = ea.A, ea.device
    rng = np.random.default_rng(21)
    obs_w = ea.observe_window(W, SCALES)
    obs_1 = torch.zeros(4 + A, N, dtype=torch.float32, device=dev)
    bufs = [(torch.zeros(N, dtype=torch.int32, device=dev), torch.zeros(N, dtype=torch.float64, device=dev),
             StepResult(*[torch.empty(N, dtype=torch.float64, device=dev) for _ in range(5)], None,
                        torch.empty(N, dtype=torch.uint8, device=dev), None)) for _ in range(2)]
    n_rolled = 0
    for t in range(64):
        lg = rng.normal(size=(N, A)).astype(np.float32)
        lg[::9] = np.nan                                     # all NaN: action 0
        logits = torch.from_numpy(lg).to(dev)
        inert = eb.state("done").cpu().numpy() != 0
        (act_a, sum_a, res_a), (act_b, sum_b, res_b) = bufs
        ea.step_policy_window(logits, obs_w, sample=sample, seed=0xABCDEF12345, scales=SCALES, action_out=act_a,
                              reward_sum=sum_a, out=res_a)
        eb.step_policy(logits, sample=sample, seed=0xABCDEF12345, obs=obs_1, action_out=act_b, reward_sum=sum_b,
                       out=res_b, obs_scales=SCALES[1:])
        assert torch.equal(act_a, act_b) and torch.equal(sum_a, sum_b), t
        for name in ("delay", "sleep", "buffer", "rebuffer", "reward", "end_of_video"):
            assert torch.equal(getattr(res_a, name), getattr(res_b, name)), (t, name)
        for f in STATE:
            assert torch.equal(ea.state(f), eb.state(f)), (t, f)
        # the newest window entries are rows 1 and 2 of the §4.1 observation, where the step rolled the windows
        o_w, o_1 = obs_w.cpu().numpy(), obs_1.cpu().numpy()
        rolled = ~inert & ~((res_a.end_of_video.cpu().numpy() != 0) & bool(auto_reset))
        assert np.array_equal(u32(o_w[3 + W - 1, rolled]), u32(o_1[1, rolled]))
        assert np.array_equal(u32(o_w[3 + 2 * W - 1, rolled]), u32(o_1[2, rolled]))
        assert np.array_equal(u32(o_w[3 + 2 * W:]), u32(o_1[4:]))
        n_rolled += int(rolled.sum())
    assert n_rolled >= 19 * N         # every session's steps before its end of video
    assert ea.error_count() == eb.error_count() == 0
    if not auto_reset:
        assert ea.state("done").all()


def test_observe_window_after_resets_and_mid_episode():
    N, W, A = 3000, 8, 6
    env, ref, tid, off = pair(N, A, track_history=1)
    util = orc.utility_table(ref.bitrates, env.params.utility_mode, env.params.utility_scale)

    def expected():
        head, nxt = wo.state_rows(util, ref.sizes, *[env.state(f).cpu().numpy() for f in ("chunk", "last_q", "buffer")],
                                  env.state("done").cpu().numpy() != 0, SCALES)
        return np.concatenate([head, np.zeros((2 * W, N), np.float32), nxt])

    env.reset(tid, off)
    obs = env.observe_window(W, SCALES)
    assert np.array_equal(u32(obs.cpu().numpy()), u32(expected()))
    acts = wo.action_table(10, N, A)
    for t in range(10):
        env.step_policy_window(one_hot(acts[t], A), obs, sample=False, scales=SCALES)
    stepped = obs.cpu().numpy()
    again = env.observe_window(W, SCALES, obs=obs)             # the windows restart, the other rows stay
    assert again is obs
    o = obs.cpu().numpy()
    assert np.array_equal(u32(o), u32(expected()))
    assert np.array_equal(u32(o[:3]), u32(stepped[:3])) and np.array_equal(u32(o[3 + 2 * W:]), u32(stepped[3 + 2 * W:]))
    assert stepped[3:3 + 2 * W].all() and not o[3:3 + 2 * W].any()
    # sorted reset: columns in environment order
    sorted_env, _, _, _ = pair(N, A, track_history=1)
    sorted_env.reset(tid, off, sort_by_trace=True)
    perm = sorted_env.perm.long().cpu().numpy()
    assert not np.array_equal(perm, np.arange(N))
    env.reset(tid, off)
    plain = env.observe_window(W, SCALES).cpu().numpy()
    assert np.array_equal(u32(sorted_env.observe_window(W, SCALES).cpu().numpy()), u32(plain[:, perm]))


def test_a_sorted_and_an_unsorted_environment_agree_through_perm():
    N, W, A = 5000, 8, 6
    bitrates, sizes, bw, tl, ti = wo.world(A, V=20)
    tid, off = wo.sessions(N, bw.shape[0], bw.shape[1])
    mk = lambda: BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, auto_reset=0, track_history=1)
    plain, srt = mk(), mk()
    plain.reset(tid, off, session_base=1000)
    srt.reset(tid, off, session_base=1000, sort_by_trace=True)
    perm = srt.perm.long()
    o_p, o_s = plain.observe_window(W, SCALES), srt.observe_window(W, SCALES)
    rng = np.random.default_rng(4)
    for t in range(30):
        logits = torch.from_numpy(rng.normal(size=(N, A)).astype(np.float32)).cuda()
        plain.step_policy_window(logits, o_p, sample=t % 2 == 0, seed=99, scales=SCALES)
        srt.step_policy_window(logits[perm].contiguous(), o_s, sample=t % 2 == 0, seed=99, scales=SCALES)
        assert torch.equal(o_s, o_p[:, perm]), t
    assert plain.error_count() == srt.error_count() == 0


def test_a_captured_chunk_replayed_48_times_equals_the_eager_loop():
    N, W = 4096, 8
    (eg, ee), _, _ = twins(N, 6, V=20, track_history=1, track_acc=1)
    A, dev = eg.A, eg.device
    logits = torch.from_numpy(np.random.default_rng(8).normal(size=(N, A)).astype(np.float32)).to(dev)
    runs = []
    for e in (eg, ee):
        runs.append(dict(obs=e.observe_window(W, SCALES), act=torch.zeros(N, dtype=torch.int32, device=dev),
                         total=torch.zeros(N, dtype=torch.float64, device=dev)))
    chunk = lambda e, r: e.step_policy_window(logits, r["obs"], sample=True, seed=7, scales=SCALES,
                                              action_out=r["act"], reward_sum=r["total"])
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        chunk(eg, runs[0])
    for _ in range(48):
        g.replay()
        chunk(ee, runs[1])
    torch.cuda.synchronize()
    for k in ("obs", "act", "total"):
        assert torch.equal(runs[0][k], runs[1][k]), k
    for f in STATE:
        assert torch.equal(eg.state(f), ee.state(f)), f


def test_c_abi_checks_in_order():
    lib = _lib.load()
    N, A, W = 8, 6, 4
    (env, _), tid, off = twins(N, A)
    dev = env.device
    st = torch.cuda.current_stream().cuda_stream
    logits = torch.zeros(N, A, dtype=torch.float32, device=dev)
    obs = torch.zeros(3 + 2 * W + A, N, dtype=torch.float32, device=dev)
    spec = _lib.AbrObsWindowSpec(W, 1, 1, 1, 1, 1)
    bad = _lib.AbrObsWindowSpec(0, 1, 1, 1, 1, 1)
    P = lambda t: None if t is None else t.data_ptr()

    def step(h, lg=logits, sp=spec, ob=obs):
        rc = lib.abr_env_step_policy_window(h, P(lg), 0, 0, sp, P(ob), *[None] * 8, st)
        return rc, lib.abr_last_error().decode()

    def observe(h, sp=spec, ob=obs):
        rc = lib.abr_env_observe_window(h, sp, P(ob), st)
        return rc, lib.abr_last_error().decode()

    for call in (step, observe):
        kw = dict(lg=None) if call is step else {}
        rc, msg = call(None, sp=None, ob=None, **kw)
        assert rc == 1 and "env is NULL" in msg
        fresh = BatchedABREnv(np.full((1, 8), 3.0), np.ones((4, A)), np.ones((4, A)), 4)
        rc, msg = call(fresh._h, sp=None, ob=None, **kw)
        assert rc == 4 and "reset" in msg
        live = BatchedABREnv(np.full((1, 8), 3.0), np.ones((4, A)), np.ones((4, A)), 4, live=1)
        live.reset(np.zeros(4, np.int32))
        rc, msg = call(live._h, sp=None, ob=None, **kw)
        assert rc == 4 and "live mode" in msg
        fresh.reset(np.zeros(0, np.int32))
        assert call(fresh._h, sp=bad, ob=None, **kw)[0] == 0          # empty batch: no-op
        if call is step:
            rc, msg = call(env._h, lg=None, sp=None, ob=None)
            assert rc == 1 and "logits is NULL" in msg
        rc, msg = call(env._h, sp=None, ob=None)
        assert rc == 1 and "spec is NULL" in msg
        rc, msg = call(env._h, sp=bad, ob=None)
        assert rc == 1 and "obs is NULL" in msg
        for w in (0, -1, 33):
            rc, msg = call(env._h, sp=_lib.AbrObsWindowSpec(w, 1, 1, 1, 1, 1))
            assert rc == 3 and "window" in msg
        assert call(env._h)[0] == 0
    for w in (1, 32):
        o = env.observe_window(w)
        env.step_policy_window(logits, o, sample=False)
    with pytest.raises(TypeError):
        env.step_policy_window(logits, obs[:-1])
    with pytest.raises(TypeError):
        env.step_policy_window(logits, obs.double())
    with pytest.raises(TypeError):
        env.step_policy_window(logits.double(), obs)
    with pytest.raises(ValueError):
        env.observe_window(33)
    assert env.error_count() == 0


def test_the_example_fused_path_equals_its_torch_glue_path():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "examples", "pensieve_harness.py"), "--check",
                        "--sessions", "4099", "--chunks", "20"], capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "fused == torch-glue" in r.stdout
