"""CPU-only: the catch-up speed control of live mode (SPEC §7.2) — known answers of the rule, the C restatement against
the pure-Python one on random live sessions, the dead-band and replay identities on the oracle, parameter validation
and its order, and include/abr_b200_speed.h against its ctypes table."""
import math
import os
import re

import numpy as np
import pytest

from abrsimulator_b200 import _build, _lib
from oracle import oracle as orc
from helpers import small_world, bits_equal
from test_capi_signatures import ROOT, c_kind, ctypes_kind
import speed_oracle as sp

STATE = ("seg", "chunk", "last_q", "phase", "pos", "buffer", "t_now", "play_time", "play_len", "play_id", "started",
         "done", "hist_len")


def both(tc, pt, b, **kw):
    """The rule from both restatements, which must agree bit for bit."""
    v, w = sp.rule(tc, pt, b, **kw), sp.rule_c(tc, pt, b, **kw)
    assert bits_equal(np.array([v]), np.array([w])) == 0, (tc, pt, b, kw)
    return v


# ---- known answers ----
def test_inside_the_dead_band_the_speed_is_1():
    assert both(20.0, 8.0 - 0.02, 10.0) == 1.0                  # e = +0.02 = dead_band
    assert both(20.0, 8.0 + 0.02, 10.0) == 1.0                  # e = -0.02
    assert both(20.0, 8.0 - 0.03, 10.0) > 1.0                   # just outside


def test_above_and_below_the_target():
    assert both(20.0, 7.0, 10.0) == 1.0 + 0.5 * (2.5 / 3.5)     # e = +1: y = 2.5
    assert both(20.0, 10.0, 10.0) == 1.0 + 0.5 * (-5.0 / 6.0)   # e = -2: y = -5
    assert both(5.0, 1.0, 10.0, target_latency=4.0, gain=1.0, max_drift=0.25, dead_band=0.0) == 1.0
    assert both(5.0, 0.0, 10.0, target_latency=4.0, gain=1.0, max_drift=0.25) == 1.0 + 0.25 * 0.5


def test_the_buffer_guard_holds_a_speed_up_at_1_but_not_a_slow_down():
    assert both(20.0, 7.0, 6.0 - 1e-9) == 1.0
    assert both(20.0, 7.0, 6.0) > 1.0                           # b < min_buffer, strict
    assert both(20.0, 10.0, 0.5) < 1.0                          # slowing down is always allowed
    assert both(20.0, 7.0, 0.0, min_buffer=0.0) > 1.0


@pytest.mark.parametrize("e", [1e3, 1e6, 1e12, -1e3, -1e6, -1e12])
def test_large_errors_stay_strictly_inside_the_range(e):
    v = both(e + 12.0, 0.0, 100.0)
    assert 0.5 < v < 1.5
    assert (v > 1.0) == (e > 0)


def test_an_undecided_chunk_is_decided_where_it_is_in_its_middle():
    """play_speed = 0 (no decision stored): the controller installed while a chunk is half played decides at once."""
    bitrates, sizes, bw, tl, ti = small_world(n_traces=2, T=40, V=10, seed=3)
    P = dict(orc.DEFAULTS, live=1, start_up_length=4.0, max_buffer=16.0)
    env = sp.SpeedEnv(bw, tl, ti, sizes, bitrates, 1, **P)
    env.reset(np.array([0], np.int32), np.array([3.0]))
    util = orc.utility_table(bitrates, 0, P["utility_scale"])
    py = sp.SpeedSession(bw[0, :tl[0]], ti[0], sizes.tolist(), util.tolist(), P, 3.0)
    t = 0
    while not (env.field("play_len")[0] > 0.0):
        env.step([0])
        py.step(0)
        t += 1
        assert t < 10
    assert env.play_speed[0] == 0.0
    env.set_speed_control(target_latency=0.0, min_buffer=0.0)
    py.control = dict(sp.DEFAULTS, target_latency=0.0, min_buffer=0.0)
    c, r = env.step([1]), py.step(1)
    for k in ("delay", "buffer", "rebuf", "reward", "latency"):
        assert c[k][0] == r[k], k
    assert env.play_speed[0] == py.play_speed and py.decisions[0] > 1.0   # the first decision: mid-chunk, latency > 0


# ---- C restatement against Python ----
def dip_and_surge_world(seed, n_traces=8, T=60, V=48):
    """Traces with deep dips (stalls, latency above the target) and surges (full buffers, latency below it)."""
    bitrates, sizes, bw, tl, ti = small_world(n_traces=n_traces, T=T, V=V, seed=seed, ragged=True)
    rng = np.random.default_rng(seed)
    for t in range(n_traces):
        for _ in range(3):
            a = int(rng.integers(0, T - 8))
            bw[t, a:a + int(rng.integers(2, 8))] *= rng.choice([0.05, 0.2, 4.0, 10.0])
    return bitrates, sizes, bw, tl, ti


def live_params(**kw):
    return dict(orc.DEFAULTS, live=1, start_up_length=8.0, max_buffer=20.0, latency_penalty=0.05, **kw)


@pytest.mark.parametrize("auto_reset,prev_ladder", [(0, 0), (0, 1), (1, 0), (1, 1)])
def test_c_restatement_equals_python_on_random_live_sessions(auto_reset, prev_ladder):
    N, steps = 500, 48
    seed = 11 + 2 * auto_reset + prev_ladder
    bitrates, sizes, bw, tl, ti = dip_and_surge_world(seed)
    P = live_params(auto_reset=auto_reset, smooth_prev_ladder=prev_ladder, track_history=1)
    ctl = dict(target_latency=[14.0, 18.0, 16.0, 20.0][2 * auto_reset + prev_ladder], gain=2.5, max_drift=0.5,
               dead_band=0.02, min_buffer=[6.0, 4.0, 8.0, 5.0][2 * auto_reset + prev_ladder])
    env = sp.SpeedEnv(bw, tl, ti, sizes, bitrates, N, **P)
    env.set_speed_control(**ctl)
    rng = np.random.default_rng(seed)
    tid = rng.integers(0, bw.shape[0], size=N).astype(np.int32)
    off = rng.uniform(0, 60, size=N)
    env.reset(tid, off)
    util = orc.utility_table(bitrates, 0, P["utility_scale"])
    py = [sp.SpeedSession(bw[tid[s], :tl[tid[s]]], ti[tid[s]], sizes.tolist(), util.tolist(), P, off[s]) for s in range(N)]
    for p in py:
        p.control = dict(ctl)
    for t in range(steps):
        a = rng.integers(0, sizes.shape[1], size=N).astype(np.int32)
        c = env.step(a)
        for s in range(N):
            r = py[s].step(int(a[s]))
            for k in ("delay", "sleep", "buffer", "rebuf", "reward", "latency", "throughput"):
                assert c[k][s] == r[k], (t, s, k)
            assert c["eov"][s] == r["eov"]
    for name, attr in (("t_now", "t_now"), ("play_time", "play_time"), ("play_len", "play_len"), ("buffer", "buffer")):
        assert bits_equal(env.field(name), np.array([getattr(p, attr) for p in py])) == 0, name
    assert np.array_equal(env.field("play_id"), [p.play_id for p in py])
    assert bits_equal(env.play_speed, np.array([p.play_speed for p in py])) == 0
    up, down, guard = env.counts()
    assert up > 0 and down > 0 and guard > 0, env.counts()
    assert up + down > 0.3 * sum(len(p.decisions) for p in py)
    assert env.errors() == 0


def test_with_the_controller_off_the_restated_step_is_the_oracles():
    """tests/speed_oracle.c restates the oracle's step: with no controller, with and without a table, bit for bit."""
    N, steps = 64, 60
    bitrates, sizes, bw, tl, ti = dip_and_surge_world(5)
    P = live_params(auto_reset=1)
    a_env, b_env = sp.SpeedEnv(bw, tl, ti, sizes, bitrates, N, **P), orc.OracleEnv(bw, tl, ti, sizes, bitrates, N, **P)
    rng = np.random.default_rng(2)
    tid, off = rng.integers(0, 8, size=N).astype(np.int32), rng.uniform(0, 60, size=N)
    a_env.reset(tid, off)
    b_env.reset(tid, off)
    for t in range(steps):
        a = rng.integers(0, 6, size=N).astype(np.int32)
        v = rng.choice([0.75, 1.0, 1.5], size=(sizes.shape[0], N)) if t % 2 else None
        x, y = a_env.step(a, speed=v), b_env.step(a, speed=v)
        for k in ("delay", "sleep", "buffer", "rebuf", "reward", "latency", "throughput", "eov"):
            assert bits_equal(x[k], y[k]) == 0, (t, k)
    for f in STATE:
        assert bits_equal(a_env.field(f), b_env.field(f)) == 0, f


# ---- identities ----
@pytest.mark.parametrize("policy", [orc.POLICY_RANDOM, orc.POLICY_BBA, 3, 4, 5])
def test_an_endless_dead_band_is_the_live_step_without_a_table(policy):
    N, steps = 128, 48
    bitrates, sizes, bw, tl, ti = dip_and_surge_world(7)
    P = live_params(auto_reset=1, track_history=1)
    a_env, b_env = sp.SpeedEnv(bw, tl, ti, sizes, bitrates, N, **P), sp.SpeedEnv(bw, tl, ti, sizes, bitrates, N, **P)
    a_env.set_speed_control(dead_band=1e300)
    rng = np.random.default_rng(4)
    tid, off = rng.integers(0, 8, size=N).astype(np.int32), rng.uniform(0, 60, size=N)
    a_env.reset(tid, off)
    b_env.reset(tid, off)
    x, y = a_env.rollout(policy, steps, seed=3), b_env.rollout(policy, steps, seed=3)
    for k in x:
        assert bits_equal(x[k], y[k]) == 0, k
    for f in STATE:
        assert bits_equal(a_env.field(f), b_env.field(f)) == 0, f
    assert np.all(a_env.play_speed[a_env.field("play_id") > 0] == 1.0)


@pytest.mark.parametrize("auto_reset,steps", [(0, 60), (1, 40)])
def test_replaying_the_logged_decisions_through_the_table_reproduces_the_episode(auto_reset, steps):
    N = 256
    bitrates, sizes, bw, tl, ti = dip_and_surge_world(9, V=40)
    P = live_params(auto_reset=auto_reset)
    ctl, ref = sp.SpeedEnv(bw, tl, ti, sizes, bitrates, N, **P), orc.OracleEnv(bw, tl, ti, sizes, bitrates, N, **P)
    ctl.set_speed_control(target_latency=16.0)
    log = ctl.start_log()
    rng = np.random.default_rng(auto_reset)
    tid, off = rng.integers(0, 8, size=N).astype(np.int32), rng.uniform(0, 60, size=N)
    actions = rng.integers(0, 6, size=(steps, N)).astype(np.int32)
    ctl.reset(tid, off)
    x = ctl.rollout(orc.POLICY_FIXED, steps, actions=actions)
    ref.reset(tid, off)
    y = ref.rollout(orc.POLICY_FIXED, steps, actions=actions, speed=log)
    for k in x:
        assert bits_equal(x[k], y[k]) == 0, k
    for f in STATE:
        assert bits_equal(ctl.field(f), ref.field(f)) == 0, f
    up, down, guard = ctl.counts()
    assert up > 0 and down > 0 and guard > 0


# ---- parameters ----
BAD = [dict(target_latency=-1.0), dict(max_drift=0.0), dict(max_drift=1.0), dict(max_drift=-0.5), dict(gain=0.0),
       dict(gain=-1.0), dict(dead_band=-0.01), dict(min_buffer=-1.0), dict(target_latency=math.inf),
       dict(gain=math.nan), dict(dead_band=math.inf), dict(min_buffer=math.nan), dict(max_drift=math.nan)]


@pytest.mark.parametrize("bad", BAD)
def test_invalid_params_are_rejected_before_the_env_is_looked_at(bad):
    assert sp.params_invalid(**bad)
    lib = _lib.load()
    p = _lib.AbrSpeedParams()
    lib.abr_speed_params_default(p)
    for k, v in bad.items():
        setattr(p, k, v)
    assert lib.abr_env_set_speed_control(None, p) == 1
    assert b"speed control parameters" in lib.abr_last_error() or b"need target_latency" in lib.abr_last_error()


def test_defaults_and_edge_values_are_valid_and_a_null_env_comes_next():
    lib = _lib.load()
    p = _lib.AbrSpeedParams()
    lib.abr_speed_params_default(p)
    assert {k: getattr(p, k) for k in sp.NAMES} == sp.DEFAULTS
    assert not sp.params_invalid()
    assert not sp.params_invalid(target_latency=0.0, dead_band=0.0, min_buffer=0.0, max_drift=1e-9, gain=1e-9)
    assert lib.abr_env_set_speed_control(None, p) == 1 and b"env is NULL" in lib.abr_last_error()
    assert lib.abr_env_set_speed_control(None, None) == 1 and b"env is NULL" in lib.abr_last_error()


# ---- the companion header ----
def header_text():
    with open(os.path.join(ROOT, "include", "abr_b200_speed.h")) as f:
        return f.read()


def test_the_companion_header_matches_its_ctypes_table():
    text = re.sub(r"/\*.*?\*/", " ", header_text(), flags=re.S)
    text = "\n".join(line for line in text.splitlines() if not line.lstrip().startswith("#"))
    decls = []
    for ret, name, params in re.findall(r"([A-Za-z_][\w \t\n*]*?)\b(abr_\w+)\s*\(([^()]*)\)\s*;", text):
        decls.append((name, ret.split()[-1], [re.sub(r"\w+$", "", x.strip()).strip() for x in params.split(",")]))
    assert [d[0] for d in decls] == list(_lib.SPEED_SIGNATURES)
    others = (set(_lib.SIGNATURES) | set(_lib.EXTRA_SIGNATURES) | set(_lib.MPC_PRED_SIGNATURES) |
              set(_lib.OBS_SIGNATURES) | set(_lib.MPC_SCEN_SIGNATURES) | set(_lib.DYNAMIC_SIGNATURES))
    assert not set(_lib.SPEED_SIGNATURES) & others
    def kind(c):   # c_kind, with this header's own struct
        if "AbrSpeedParams" in c and c.count("*") == 1:
            return ("ptr", "AbrSpeedParams")
        return c_kind(c)
    for name, ret, params in decls:
        restype, argtypes = _lib.SPEED_SIGNATURES[name]
        assert [ctypes_kind(t) for t in argtypes] == [kind(c) for c in params], name
        assert ctypes_kind(restype) == kind(ret), name
    fields = re.search(r"typedef struct AbrSpeedParams \{\s*double ([^;]*);", header_text()).group(1)
    assert tuple(f.strip() for f in fields.split(",")) == sp.NAMES == tuple(n for n, _ in _lib.AbrSpeedParams._fields_)


def test_the_field_id_the_table_and_the_build_agree():
    assert int(re.search(r"#define\s+ABR_F_PLAY_SPEED\s+(\d+)", header_text()).group(1)) == \
        _lib.SPEED_FIELDS["play_speed"][0]
    assert _lib.SPEED_FIELDS == dict(play_speed=(25, "float64")) and "play_speed" not in _lib.FIELDS
    lib = _lib.load()
    for name, (restype, argtypes) in _lib.SPEED_SIGNATURES.items():
        fn = getattr(lib, name)
        assert fn.restype is restype and list(fn.argtypes) == argtypes, name
    assert os.path.normpath(os.path.join(ROOT, "include", "abr_b200_speed.h")) in [os.path.normpath(h) for h in _build.HEADERS]


def test_the_controller_forms_are_dispatched_without_respelling_the_table_forms():
    with open(os.path.join(ROOT, "abrsimulator_b200", "csrc", "abr_step.cu")) as f:
        src = " ".join(f.read().split())
    assert "else if (live && v.spd.on) e = go(abr_step_kernel<false, 2, 0, OT>);" in src
    assert "if (live == 2) return go(abr_rollout_kernel<P, false, false, 2, false, OT>, o);" in src
    assert "const int live = v.p.live == 0 ? 0 : (v.spd.on ? 2 : 1);" in src
