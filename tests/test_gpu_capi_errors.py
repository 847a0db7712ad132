"""Error codes and messages of the C-ABI entry points, one fault at a time, the precedence of paired faults, and the
kernel launches a whole run issues.  Every argument is passed as an explicit ctypes value, so the calls mean the same
with or without declared signatures.  Run with -m gpu."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from abrsimulator_b200 import _lib
from abrsimulator_b200.env import BatchedABREnv
from helpers import small_world

I, LL, U64, D = C.c_int, C.c_longlong, C.c_uint64, C.c_double
INVALID, RANGE, STATE = 1, 3, 4
FIXED, RANDOM, BBA, RATE, BOLA = 0, 1, 2, 3, 4
CAP = 8
BIG_STEPS = 2 ** 31 - 1          # with 3 sessions: steps * N > 2^32 - 1
OK = (0, "")


def P(x):
    """A buffer's address as c_void_p (None stays NULL): device tensors, host tensors and numpy arrays."""
    if x is None:
        return None
    return C.c_void_p(x.data_ptr() if isinstance(x, torch.Tensor) else x.ctypes.data)


def rc_of(fn, *args):
    """(return code, the thread's last error message when the code is not 0)."""
    rc = fn(*args)
    return rc, ("" if rc == 0 else _lib.load().abr_last_error().decode())


def expect(got, code, text=""):
    rc, msg = got
    assert rc == code and text in msg, (rc, msg, code, text)


def make_env(**params):
    bitrates, sizes, bw, tl, ti = small_world(n_traces=4, T=64, V=10)
    if params.pop("zero_size", False):
        sizes = sizes.copy()
        sizes[3, 0] = 0.0
    return BatchedABREnv(bw, sizes, bitrates, CAP, trace_len=tl, trace_interval=ti, **params)


def reset(env, n):
    env.reset(np.zeros(n, np.int32))


@pytest.fixture(scope="module")
def lib():
    return _lib.load()


@pytest.fixture
def dev():
    z = lambda dt: torch.zeros(CAP, dtype=dt, device="cuda")
    return dict(act=z(torch.int32), f64=z(torch.float64), logits=torch.zeros(CAP * 6, dtype=torch.float32, device="cuda"))


# ---- per-step entry points ----
def _step_calls(lib):
    """abr_env_step, _live and _f32 as f(handle, action)."""
    return (lambda h, a: rc_of(lib.abr_env_step, h, a, *[None] * 8, None),
            lambda h, a: rc_of(lib.abr_env_step_live, h, a, *[None] * 10, None),
            lambda h, a: rc_of(lib.abr_env_step_f32, h, a, *[None] * 10, None))


def test_step_entry_points(lib, dev):
    env = make_env()
    act = P(dev["act"])
    for step in _step_calls(lib):
        expect(step(None, act), INVALID, "env is NULL")
        expect(step(env._h, act), STATE, "abr_env_reset has not been called")
        expect(step(env._h, None), STATE, "abr_env_reset has not been called")      # not reset before NULL action
    reset(env, 0)
    for step in _step_calls(lib):
        expect(step(env._h, None), *OK)                                            # empty batch: a no-op
    reset(env, 4)
    for step in _step_calls(lib):
        expect(step(env._h, None), INVALID, "action is NULL")


def _step_policy(lib, h, logits):
    return rc_of(lib.abr_env_step_policy, h, logits, I(0), U64(0), *[None] * 10, None)


def test_step_policy(lib, dev):
    env, live = make_env(), make_env(live=1, start_up_length=8.0)
    logits = P(dev["logits"])
    expect(_step_policy(lib, None, logits), INVALID, "env is NULL")
    expect(_step_policy(lib, env._h, logits), STATE, "abr_env_reset has not been called")
    expect(_step_policy(lib, live._h, logits), STATE, "abr_env_reset has not been called")   # not reset before live
    reset(live, 0)
    expect(_step_policy(lib, live._h, None), STATE, "not available in live mode")          # live before empty batch
    reset(live, 4)
    expect(_step_policy(lib, live._h, logits), STATE, "not available in live mode")
    reset(env, 0)
    expect(_step_policy(lib, env._h, None), *OK)
    reset(env, 4)
    expect(_step_policy(lib, env._h, None), INVALID, "logits is NULL")


# ---- fused episode ----
def _rollouts(lib):
    """abr_env_rollout_fused, _live and _f32 as f(handle, policy, steps, actions_in, speed, latency)."""
    return (lambda h, pol, steps, a_in, speed=None, lat=None:
            rc_of(lib.abr_env_rollout_fused, h, I(pol), U64(1), I(steps), a_in, *[None] * 7, None),
            lambda h, pol, steps, a_in, speed=None, lat=None:
            rc_of(lib.abr_env_rollout_fused_live, h, I(pol), U64(1), I(steps), a_in, speed, *[None] * 5, lat, None,
                  None, None),
            lambda h, pol, steps, a_in, speed=None, lat=None:
            rc_of(lib.abr_env_rollout_fused_f32, h, I(pol), U64(1), I(steps), a_in, speed, *[None] * 5, lat, None,
                  None, None))


def test_rollout_entry_points(lib, dev):
    buf = P(dev["f64"])
    for i, roll in enumerate(_rollouts(lib)):
        plain, zero = make_env(), make_env(zero_size=True, track_history=1)
        expect(roll(None, BBA, 1, None), INVALID, "env is NULL")
        expect(roll(plain._h, BBA, 1, None), STATE, "abr_env_reset has not been called")
        expect(roll(plain._h, 99, -1, None), STATE, "abr_env_reset has not been called")
        reset(plain, 0)
        expect(roll(plain._h, 99, -1, None), *OK)                     # an empty batch comes before every other check
        reset(plain, 3)
        expect(roll(plain._h, BBA, -1, None), RANGE, "steps must be >= 0")
        expect(roll(plain._h, 99, -1, None), RANGE, "steps must be >= 0")          # steps before the policy
        expect(roll(plain._h, 99, 1, None), INVALID, "unknown policy 99")
        expect(roll(plain._h, -1, 1, None), INVALID, "unknown policy -1")
        expect(roll(plain._h, RATE, 1, None), STATE, "track_history")
        expect(roll(plain._h, FIXED, 1, None), INVALID, "ABR_POLICY_FIXED needs d_actions_in")
        expect(roll(plain._h, RANDOM, BIG_STEPS, None), RANGE, "exceeds 2^32 - 1")
        expect(roll(plain._h, RATE, BIG_STEPS, None), STATE, "track_history")     # the policy before the size
        reset(zero, 3)
        expect(roll(zero._h, BOLA, 1, None), INVALID, "BOLA needs positive chunk sizes")
        expect(roll(zero._h, FIXED, 1, None), INVALID, "ABR_POLICY_FIXED needs d_actions_in")
        if i == 0:
            continue
        for kw in (dict(speed=buf), dict(lat=buf)):                   # live outputs on an on-demand environment
            expect(roll(plain._h, BBA, 1, None, **kw), STATE, "speed / latency belong to live mode")
            expect(roll(plain._h, FIXED, 1, None, **kw), INVALID, "ABR_POLICY_FIXED needs d_actions_in")
            expect(roll(plain._h, BBA, BIG_STEPS, None, **kw), STATE, "speed / latency belong to live mode")


# ---- whole runs ----
def _run(lib, h, policy, steps, tid, n, actions=None, cost=None, stats=None, off=None):
    return rc_of(lib.abr_env_run, h, I(policy), U64(3), I(steps), tid, off, I(n), LL(0), actions, *[None] * 7, cost,
                 stats, None)


def _run_host(lib, h, policy, steps, tid, n, actions=None, acc=None, stats=None, reward=None, cost=None, off=None):
    return rc_of(lib.abr_env_run_host, h, I(policy), U64(3), I(steps), tid, off, I(n), LL(0), actions, acc, stats,
                 reward, cost, None)


def test_run(lib, dev):
    plain, hist, zero = make_env(), make_env(track_history=1), make_env(zero_size=True, track_history=1)
    tid = P(torch.zeros(CAP + 1, dtype=torch.int32, device="cuda"))
    h = plain._h
    expect(_run(lib, None, BBA, 1, tid, 4), INVALID, "env or trace_id is NULL")
    expect(_run(lib, h, BBA, 1, None, 4), INVALID, "env or trace_id is NULL")
    expect(_run(lib, h, BBA, 1, None, 0), *OK)
    for n in (CAP + 1, -1):
        expect(_run(lib, h, BBA, 1, tid, n), RANGE, f"n_sessions {n} exceeds capacity {CAP}")
    expect(_run(lib, h, BBA, -1, tid, 4), RANGE, "steps must be >= 0")
    expect(_run(lib, h, BBA, -1, tid, CAP + 1), RANGE, "exceeds capacity")          # capacity before steps
    expect(_run(lib, h, BBA, -1, None, 4), INVALID, "env or trace_id is NULL")
    expect(_run(lib, h, 99, 1, tid, 4), INVALID, "unknown policy 99")
    expect(_run(lib, h, 99, -1, tid, 4), RANGE, "steps must be >= 0")
    expect(_run(lib, h, RATE, 1, tid, 4), STATE, "track_history")
    expect(_run(lib, zero._h, BOLA, 1, tid, 4), INVALID, "BOLA needs positive chunk sizes")
    expect(_run(lib, h, FIXED, 1, tid, 4), INVALID, "ABR_POLICY_FIXED needs d_actions_in")
    expect(_run(lib, h, FIXED, 0, tid, 4), *OK)                   # only an episode that runs needs the actions
    expect(_run(lib, h, FIXED, 1, tid, 0), *OK)
    expect(_run(lib, h, RANDOM, BIG_STEPS, tid, 3), RANGE, "exceeds 2^32 - 1")
    hist.set_order(torch.arange(4, dtype=torch.int32, device="cuda"))
    expect(_run(lib, hist._h, BBA, 1, tid, 5), STATE, "the installed session order has 4 entries, the batch 5")
    expect(_run(lib, hist._h, FIXED, 1, tid, 5), INVALID, "ABR_POLICY_FIXED needs d_actions_in")   # before the order
    expect(_run(lib, hist._h, BBA, -1, tid, 5), RANGE, "steps must be >= 0")
    expect(_run(lib, hist._h, BBA, 1, tid, CAP + 1), RANGE, "exceeds capacity")
    expect(_run(lib, hist._h, BBA, 1, tid, 4), *OK)


def test_run_host(lib):
    plain, hist, zero = make_env(), make_env(track_history=1), make_env(zero_size=True, track_history=1)
    tid = P(np.zeros(CAP + 1, np.int32))
    h = plain._h
    expect(_run_host(lib, None, BBA, 1, tid, 4), INVALID, "env is NULL")
    expect(_run_host(lib, None, BBA, -1, tid, 4), INVALID, "env is NULL")
    expect(_run_host(lib, h, BBA, -1, tid, 4), RANGE, "steps must be >= 0")
    expect(_run_host(lib, h, BBA, -1, None, 4), RANGE, "steps must be >= 0")        # steps before the trace ids
    expect(_run_host(lib, h, BBA, -1, tid, CAP + 1), RANGE, "steps must be >= 0")   # and before the capacity
    expect(_run_host(lib, h, BBA, 1, None, 4), INVALID, "env or trace_id is NULL")
    expect(_run_host(lib, h, BBA, 1, None, 0), *OK)
    for n in (CAP + 1, -1):
        expect(_run_host(lib, h, BBA, 1, tid, n), RANGE, f"n_sessions {n} exceeds capacity {CAP}")
    expect(_run_host(lib, h, BBA, 1, None, CAP + 1), INVALID, "env or trace_id is NULL")
    expect(_run_host(lib, h, 99, 1, tid, 4), INVALID, "unknown policy 99")
    expect(_run_host(lib, h, 99, 1, tid, CAP + 1), RANGE, "exceeds capacity")
    expect(_run_host(lib, h, RATE, 1, tid, 4), STATE, "track_history")
    expect(_run_host(lib, zero._h, BOLA, 1, tid, 4), INVALID, "BOLA needs positive chunk sizes")
    for steps, n in ((1, 4), (0, 4), (1, 0)):             # FIXED needs its actions even when no episode runs
        expect(_run_host(lib, h, FIXED, steps, tid, n), INVALID, "ABR_POLICY_FIXED needs h_actions_in")
    expect(_run_host(lib, h, RANDOM, BIG_STEPS, tid, 3), RANGE, "exceeds 2^32 - 1")
    hist.set_order(torch.arange(4, dtype=torch.int32, device="cuda"))
    expect(_run_host(lib, hist._h, BBA, 1, tid, 5), STATE, "the installed session order has 4 entries, the batch 5")
    expect(_run_host(lib, hist._h, FIXED, 1, tid, 5), INVALID, "ABR_POLICY_FIXED needs h_actions_in")
    expect(_run_host(lib, hist._h, BBA, 1, tid, 4), *OK)


def _launches(call):
    before = _lib.launch_count()
    expect(call(), *OK)
    return _lib.launch_count() - before


def test_whole_run_launch_counts(lib):
    """Fused (sessions and steps): one episode launch.  Unfused (no steps): reset + cost + the two statistics stages.
    run_host adds one cost launch when the cost buffer is pageable, and none when it is page-locked (zero-copy)."""
    env = make_env()
    n = 6
    tid_d = torch.zeros(n, dtype=torch.int32, device="cuda")
    cost_d, stats_d = torch.zeros(n, dtype=torch.float64, device="cuda"), torch.zeros(11, dtype=torch.float64, device="cuda")
    assert _launches(lambda: _run(lib, env._h, BBA, 5, P(tid_d), n, cost=P(cost_d), stats=P(stats_d))) == 1
    assert _launches(lambda: _run(lib, env._h, BBA, 0, P(tid_d), n, cost=P(cost_d), stats=P(stats_d))) == 4
    assert _launches(lambda: _run(lib, env._h, BBA, 5, P(tid_d), 0, cost=P(cost_d), stats=P(stats_d))) == 0
    for pinned in (False, True):
        host = lambda shape, dt: torch.zeros(shape, dtype=dt, pin_memory=pinned).numpy()
        tid, cost, stats, acc = host(n, torch.int32), host(n, torch.float64), host(11, torch.float64), host((11, n), torch.float64)
        fused = _launches(lambda: _run_host(lib, env._h, BBA, 5, P(tid), n, acc=P(acc), stats=P(stats), cost=P(cost)))
        assert fused == (1 if pinned else 2), (pinned, fused)
        assert _launches(lambda: _run_host(lib, env._h, BBA, 0, P(tid), n, acc=P(acc), stats=P(stats), cost=P(cost))) == 4
        reward = host((5, n), torch.float64)
        assert _launches(lambda: _run_host(lib, env._h, BBA, 5, P(tid), n, reward=P(reward))) == 1
    torch.cuda.synchronize()


# ---- per-step decisions ----
def test_policy_decide(lib, dev):
    plain, hist, zero = make_env(), make_env(track_history=1), make_env(zero_size=True, track_history=1)
    act = P(dev["act"])
    call = lambda env, pol, a=act: rc_of(lib.abr_env_policy_decide, None if env is None else env._h, I(pol), a, None)
    expect(call(None, BBA), INVALID, "env is NULL")
    for bad in (FIXED, RANDOM, 99):
        expect(call(plain, bad), INVALID, f"abr_env_policy_decide takes ABR_POLICY_BBA, _RATE or _BOLA (got {bad})")
    expect(call(plain, RATE), STATE, "track_history")                # the policy before the reset state
    expect(call(zero, BOLA), INVALID, "BOLA needs positive chunk sizes")
    expect(call(hist, RATE), STATE, "abr_env_reset has not been called")
    reset(hist, 0)
    expect(call(hist, RATE, None), *OK)
    expect(call(hist, FIXED, None), INVALID, "abr_env_policy_decide takes")
    reset(hist, 4)
    expect(call(hist, BOLA, None), INVALID, "action is NULL")
    expect(call(hist, RATE), *OK)


def test_env_mpc_decide(lib, dev):
    plain, hist = make_env(), make_env(track_history=1)
    act = P(dev["act"])
    call = lambda env, H, mode, a=act: rc_of(lib.abr_env_mpc_decide, None if env is None else env._h, I(H), I(mode),
                                             a, None, None)
    expect(call(None, 5, 1), INVALID, "env is NULL")
    expect(call(hist, 5, 1), STATE, "abr_env_reset has not been called")
    reset(hist, 0)
    expect(call(hist, 0, 7, None), *OK)
    reset(hist, 4)
    reset(plain, 4)
    expect(call(hist, 5, 1, None), INVALID, "action is NULL")
    expect(call(hist, 0, 7, None), INVALID, "action is NULL")
    expect(call(hist, 5, 7), INVALID, "unknown MPC mode 7")
    expect(call(hist, 5, 0x100 | 7), INVALID, "unknown MPC mode 7")
    expect(call(plain, 5, 1), STATE, "needs the throughput history")
    expect(call(plain, 5, 7), INVALID, "unknown MPC mode")                           # mode before history
    for H in (0, 9):
        expect(call(hist, H, 1), RANGE, f"horizon must be in [1, 8] (got {H})")
    expect(call(plain, 9, 1), STATE, "needs the throughput history")                # history before the horizon
    expect(call(hist, 5, 0x100 | 1), *OK)


# ---- standalone MPC ----
N_MPC, K_MPC, V_MPC, A_MPC = 4, 5, 10, 6


def _mpc_inputs(host, A=A_MPC):
    """Valid inputs of one standalone decision: device tensors, or host numpy arrays (tables then sizes/bitrates)."""
    rng = np.random.default_rng(3)
    sizes = rng.uniform(1.0, 2.0, (V_MPC, A)) * np.arange(1, A + 1)
    second = np.tile(np.arange(1, A + 1) * 300.0, (V_MPC, 1))
    arrays = dict(sizes=sizes, second=second, chunk=np.zeros(N_MPC, np.int32), prev_q=np.zeros(N_MPC, np.int32),
                  buffer=np.full(N_MPC, 10.0), bw_hist=rng.uniform(1.0, 3.0, (N_MPC, K_MPC)),
                  hist_len=np.full(N_MPC, K_MPC, np.int32), last_pred=np.zeros(N_MPC), err_ring=np.zeros((N_MPC, K_MPC)),
                  err_len=np.zeros(N_MPC, np.int32), action=np.zeros(N_MPC, np.int32), startup_delay=np.zeros(N_MPC),
                  errors=np.zeros(1, np.int32))
    if not host:
        arrays = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in arrays.items()}
    return arrays


def _mpc_call(lib, host, startup, x, params, V=V_MPC, A=A_MPC, N=N_MPC, K=K_MPC, H=3, mode=1, flags=0, n_ts=1,
              ts_step=0.0, robust=("last_pred", "err_ring", "err_len"), drop=()):
    """One standalone decision; `drop` names the pointers passed as NULL, `robust` the robust-state arrays given."""
    p = lambda k: None if k in drop else P(x[k])
    r = lambda k: p(k) if k in robust else None
    head = (p("sizes"), p("second"), I(V), I(A), None if "params" in drop else C.byref(params), I(N), p("chunk"),
            p("prev_q"), p("buffer"), p("bw_hist"), p("hist_len"), I(K), r("last_pred"), r("err_ring"), r("err_len"),
            I(H), I(mode), I(flags))
    tail = (None, None, None, p("errors"))
    stream = () if host else (None,)
    if startup:
        fn = lib.abr_mpc_decide_startup_host if host else lib.abr_mpc_decide_startup
        return rc_of(fn, *head, None, I(n_ts), D(ts_step), p("action"), p("startup_delay"), *tail, *stream)
    fn = lib.abr_mpc_decide_host if host else lib.abr_mpc_decide
    return rc_of(fn, *head, p("action"), *tail, *stream)


@pytest.mark.parametrize("startup", [False, True])
def test_standalone_mpc_device(lib, startup):
    x, x16 = _mpc_inputs(False), _mpc_inputs(False, A=16)
    params = _lib.default_params()
    call = lambda **kw: _mpc_call(lib, False, startup, x, params, **kw)
    expect(call(), *OK)
    expect(call(N=0), *OK)
    for k in ("sizes", "second", "chunk", "prev_q", "buffer", "bw_hist", "hist_len", "action"):
        expect(call(drop=(k,)), INVALID, "a required pointer is NULL")
    expect(call(drop=("params",)), INVALID, "params is NULL")
    expect(call(drop=("params", "chunk")), INVALID, "a required pointer is NULL")
    expect(call(N=-1), RANGE, "N must be >= 0 and V >= 1")
    expect(call(V=0), RANGE, "N must be >= 0 and V >= 1")
    expect(call(drop=("params",), N=-1), INVALID, "params is NULL")
    expect(call(K=0), RANGE, "K must be >= 1")
    expect(call(N=-1, K=0), RANGE, "N must be >= 0")
    expect(call(mode=2), INVALID, "unknown MPC mode 2")
    expect(call(K=0, mode=2), RANGE, "K must be >= 1")
    expect(call(flags=4, mode=1), INVALID, "ABR_MPC_PRED_SES")
    expect(call(flags=4, mode=0), *OK)
    expect(call(mode=2, flags=4), INVALID, "unknown MPC mode 2")
    for given in (("last_pred",), ("err_ring", "err_len"), ("last_pred", "err_len")):
        expect(call(robust=given), INVALID, "last_pred, err_ring and err_len must be given together")
    expect(call(robust=()), *OK)
    expect(call(robust=("last_pred",), flags=4), INVALID, "ABR_MPC_PRED_SES")
    for H in (0, 9):
        expect(call(H=H), RANGE, f"horizon must be in [1, 8] (got {H})")
    expect(call(H=9, mode=2), INVALID, "unknown MPC mode")                         # the mode before the shape
    expect(call(H=9, robust=("last_pred",)), INVALID, "must be given together")
    for A in (0, 17):
        expect(call(A=A), RANGE, "A must be in [1, 16]")
    expect(_mpc_call(lib, False, startup, x16, params, A=16, H=8), RANGE, "exceed the 2^31-1 index range")
    expect(call(H=0, A=17), RANGE, "horizon must be in [1, 8]")
    if not startup:
        return
    expect(call(drop=("startup_delay",)), INVALID, "startup_delay is NULL")
    expect(call(drop=("startup_delay", "action", "params")), INVALID, "startup_delay is NULL")
    for n_ts in (0, 4097):
        expect(call(n_ts=n_ts), RANGE, f"n_ts must be in [1, 4096] (got {n_ts})")
    expect(call(n_ts=4, ts_step=0.0), RANGE, "ts_step must be finite and > 0")
    expect(call(n_ts=4, ts_step=float("inf")), RANGE, "ts_step must be finite and > 0")
    expect(call(n_ts=1, ts_step=0.0), *OK)
    expect(call(n_ts=4, ts_step=0.5), *OK)
    expect(call(n_ts=0, robust=("last_pred",)), INVALID, "must be given together")
    expect(call(n_ts=0, H=9), RANGE, "n_ts must be in")                            # n_ts before the shape
    bad = _lib.default_params(startup_penalty=float("inf"))
    expect(_mpc_call(lib, False, True, x, bad, n_ts=4, ts_step=0.5), INVALID, "startup_penalty must be finite")
    expect(_mpc_call(lib, False, True, x, bad, n_ts=1), *OK)
    expect(_mpc_call(lib, False, True, x, bad, n_ts=4, ts_step=0.0), RANGE, "ts_step must be finite and > 0")
    expect(_mpc_call(lib, False, True, x, bad, n_ts=4, ts_step=0.5, H=9), INVALID, "startup_penalty must be finite")


@pytest.mark.parametrize("startup", [False, True])
def test_standalone_mpc_host(lib, startup):
    x, x16 = _mpc_inputs(True), _mpc_inputs(True, A=16)
    params = _lib.default_params()
    call = lambda **kw: _mpc_call(lib, True, startup, x, params, **kw)
    expect(call(), *OK)
    expect(call(N=0), *OK)
    for k in ("chunk", "prev_q", "buffer", "bw_hist", "hist_len", "action"):
        expect(call(drop=(k,)), INVALID, "a required pointer is NULL")
    for k in ("sizes", "second"):
        expect(call(drop=(k,)), INVALID, "sizes/bitrates is NULL")
    expect(call(drop=("sizes", "action")), INVALID, "a required pointer is NULL")    # pointers before the tables
    for V, A in ((0, A_MPC), (V_MPC, 0), (V_MPC, 17)):
        expect(call(V=V, A=A), RANGE, f"need V >= 1 and 1 <= A <= 16 (got V={V} A={A})")
    nan = dict(x, sizes=x["sizes"].copy())
    nan["sizes"][2, 1] = np.nan
    expect(_mpc_call(lib, True, startup, nan, params), INVALID, "sizes[13] = nan is not finite and >= 0")
    expect(call(drop=("params",)), INVALID, "params is NULL")
    expect(call(drop=("params",), A=17), RANGE, "need V >= 1 and 1 <= A <= 16")      # the tables before the params
    expect(call(N=-1), RANGE, "N must be >= 0 and K >= 1")
    expect(call(K=0), RANGE, "N must be >= 0 and K >= 1")
    expect(call(drop=("params",), K=0), INVALID, "params is NULL")
    for H in (0, 9):
        expect(call(H=H), RANGE, f"horizon must be in [1, 8] (got {H})")
    expect(call(K=0, H=9), RANGE, "N must be >= 0 and K >= 1")                       # N, K before the shape
    expect(_mpc_call(lib, True, startup, x16, params, A=16, H=8), RANGE, "exceed the 2^31-1 index range")
    expect(call(mode=2), INVALID, "unknown MPC mode 2")
    expect(call(mode=2, H=9), RANGE, "horizon must be in [1, 8]")                    # the shape before the mode
    expect(call(flags=4, mode=1), INVALID, "ABR_MPC_PRED_SES")
    expect(call(mode=2, flags=4), INVALID, "unknown MPC mode 2")
    for given in (("last_pred",), ("err_ring", "err_len"), ()):   # a partial robust state is taken as none
        expect(call(robust=given), *OK)
    if not startup:
        return
    expect(call(drop=("startup_delay",)), INVALID, "startup_delay is NULL")
    expect(call(drop=("startup_delay", "chunk", "sizes")), INVALID, "startup_delay is NULL")
    for n_ts in (0, 4097):
        expect(call(n_ts=n_ts), RANGE, f"n_ts must be in [1, 4096] (got {n_ts})")
    expect(call(n_ts=4, ts_step=-1.0), RANGE, "ts_step must be finite and > 0")
    expect(call(n_ts=4, ts_step=0.5), *OK)
    expect(call(n_ts=0, H=9), RANGE, "horizon must be in [1, 8]")                    # the shape before n_ts
    expect(call(n_ts=0, mode=2), INVALID, "unknown MPC mode")                        # the mode before n_ts
    bad = _lib.default_params(startup_penalty=float("inf"))
    expect(_mpc_call(lib, True, True, x, bad, n_ts=4, ts_step=0.5), INVALID, "startup_penalty must be finite")


def test_score_host(lib):
    x = _mpc_inputs(True)
    params = _lib.default_params()
    hist = np.array([1.0, 2.0, 1.5])
    seqs = np.zeros((2, 3), np.int32)
    scores = np.zeros(2)

    def call(V=V_MPC, A=A_MPC, chunk=0, prev_q=0, h=hist, n_hist=3, H=3, mode=1, s=seqs, M=2, drop=()):
        p = lambda k, a: None if k in drop else P(a)
        return rc_of(lib.abr_mpc_score_host, p("sizes", x["sizes"]), p("second", x["second"]), I(V), I(A),
                     None if "params" in drop else C.byref(params), I(chunk), I(prev_q), D(10.0), p("hist", h),
                     I(n_hist), I(H), I(mode), D(0.0), p("seqs", s), I(M), p("scores", scores))

    expect(call(), *OK)
    for k in ("hist", "seqs", "scores"):
        expect(call(drop=(k,)), INVALID, "a required pointer is NULL")
    expect(call(drop=("sizes",)), INVALID, "sizes/bitrates is NULL")
    expect(call(drop=("sizes", "hist")), INVALID, "a required pointer is NULL")
    expect(call(A=17), RANGE, "need V >= 1 and 1 <= A <= 16")
    expect(call(drop=("params",)), INVALID, "params is NULL")
    expect(call(drop=("params",), V=0), RANGE, "need V >= 1")
    expect(call(H=9), RANGE, "horizon must be in [1, 8]")
    expect(call(drop=("params",), H=9), INVALID, "params is NULL")
    expect(call(mode=2), INVALID, "unknown MPC mode 2")
    expect(call(mode=2, H=9), RANGE, "horizon must be in [1, 8]")
    expect(call(M=-1), RANGE, "M must be >= 0")
    expect(call(M=-1, mode=2), INVALID, "unknown MPC mode 2")
    expect(call(n_hist=0), RANGE, "empty throughput history")
    expect(call(h=np.array([1.0, 0.0, 1.5])), RANGE, "zero throughput sample")
    expect(call(chunk=8), RANGE, "chunk_idx + horizon exceeds the video")
    expect(call(prev_q=A_MPC), RANGE, "prev_q out of range")
    expect(call(s=np.full((2, 3), A_MPC, np.int32)), RANGE, "sequence entry 0 out of range")


# ---- resets ----
def test_reset_entry_points(lib):
    env = make_env()
    tid = P(torch.zeros(CAP + 1, dtype=torch.int32, device="cuda"))
    htid = P(np.zeros(CAP + 1, np.int32))
    calls = (lambda h, t, n: rc_of(lib.abr_env_reset, h, t, None, I(n), LL(0), None),
             lambda h, t, n: rc_of(lib.abr_env_reset_sorted, h, t, None, I(n), LL(0), None))
    for call in calls:
        expect(call(None, tid, 4), INVALID, "env or trace_id is NULL")
        expect(call(env._h, None, 4), INVALID, "env or trace_id is NULL")
        expect(call(env._h, tid, CAP + 1), RANGE, "exceeds capacity")
        expect(call(env._h, None, CAP + 1), INVALID, "env or trace_id is NULL")
        expect(call(env._h, tid, 4), *OK)
    expect(rc_of(lib.abr_env_reset_host, env._h, htid, None, I(CAP + 1), LL(0), None), RANGE, "exceeds capacity")
    env.set_order(torch.arange(4, dtype=torch.int32, device="cuda"))
    expect(calls[0](env._h, tid, 5), STATE, "the installed session order has 4 entries, the batch 5")
    expect(calls[0](env._h, tid, CAP + 1), RANGE, "exceeds capacity")
    expect(calls[1](env._h, tid, 5), *OK)                         # installs its own order
    expect(rc_of(lib.abr_env_reset_host, env._h, htid, None, I(4), LL(0), None), STATE, "the installed session order")
    torch.cuda.synchronize()
