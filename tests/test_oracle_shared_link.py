"""CPU-only: the shared-link oracle (SPEC §9) against the single-session step oracle at G = 1, its symmetries, known
answers on constant traces, the header against its ctypes table, and the argument checks that need no device."""
import math
import os
import re

import numpy as np
import pytest

from abrsimulator_b200 import _lib
from helpers import small_world
from test_capi_signatures import ctypes_kind
import session_params_oracle as spo
import shared_link_oracle as sl
from oracle import step_oracle as so

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
POLICIES = (sl.FIXED, sl.RANDOM, sl.BBA, sl.RATE, sl.BOLA, sl.DYNAMIC)
P0 = dict(chunk_length=4.0, max_buffer=60.0, rtt=0.08, payload=0.95, sleep_quantum=0.5, rebuf_penalty=4.3,
          smooth_penalty=1.0, default_quality=1, auto_reset=1, hist_k=5, track_history=1, smooth_prev_ladder=0,
          start_up_length=0.0)
WIDE = [5.0, 10.0, 1.0, 10.0, 30.0, 12.0, 6.0]


def world(V=6, T=40, n_traces=4, seed=0, **kw):
    bitrates, sizes, bw, tl, ti = small_world(n_traces=n_traces, T=T, V=V, seed=seed, ragged=True)
    return sl.World(bw, tl, ti, sizes, bitrates * 0.001, dict(P0, **kw), WIDE)


def session_loop(w, steps, tr, off, policy, seed=0, g=0, actions=None):
    """SPEC §3+§4 for one session: step_oracle.Session with the policy oracles' decision before every step."""
    P, K = w.P, w.P["hist_k"]
    s = so.Session(w.bw[tr][:w.tl[tr]], w.ti[tr], w.sizes, w.util, P, start_offset=off, table=w.table(tr))
    mode, out = 0, []
    for k in range(steps):
        if policy == sl.FIXED:
            q = int(actions[k])
        elif policy == sl.RANDOM:
            q = sl.random_action(seed, g, k, w.A)
        elif policy == sl.BBA:
            q = spo.session_action(sl.BBA, w.sizes[0], None, 0.0, None, s.buffer, s.chunk, 0, P["default_quality"],
                                   P["chunk_length"], w.wide)[0]
        elif s.done:
            q = 0
        else:
            c = s.chunk
            q, m = spo.session_action(policy, w.sizes[c], w.v[c], w.v_max, s.history[-K:], s.buffer, c, mode,
                                      P["default_quality"], P["chunk_length"], w.wide)
            mode = m if policy == sl.DYNAMIC else mode
        o = s.step(q)
        o["actions"] = q
        out.append(o)
    return s, out


@pytest.mark.parametrize("auto_reset", [0, 1])
@pytest.mark.parametrize("policy", POLICIES)
def test_one_player_per_link_is_the_single_session_episode(policy, auto_reset):
    w = world(auto_reset=auto_reset)
    steps, n_links = 15, 4                     # steps > V: end of video, auto_reset or the inert steps
    tid = [0, 1, 2, 3]
    off = [0.0, 3.25, 17.5, 1.0]
    rng = np.random.default_rng(policy)
    actions = rng.integers(0, w.A, size=(steps, n_links)).astype(np.int32)
    r = sl.run_shared(w, steps, 1, tid, off, policy=policy, seed=11, session_base=5, actions=actions)
    for l in range(n_links):
        s, out = session_loop(w, steps, tid[l], off[l], policy, seed=11, g=5 + l, actions=actions[:, l])
        for key, rk in (("delay", "delay"), ("sleep", "sleep"), ("buffer", "buffer"), ("rebuf", "rebuf"),
                        ("reward", "reward"), ("eov", "eov"), ("actions", "actions")):
            exp = np.array([o[key] for o in out], r[rk].dtype)
            assert np.array_equal(r[rk][:, l], exp), (key, l)
        st = r["state"]
        assert (st["seg"][l], st["phase"][l], st["pos"][l]) == (s.seg, s.phi, s.pos)
        assert (st["chunk"][l], st["buffer"][l], st["done"][l]) == (s.chunk, s.buffer, int(s.done))
        live = [o for o in out if not o["inert"]]
        assert r["acc"][0, l] == sum_lr(o["reward"] for o in live) and r["acc"][6, l] == len(live)
        # the link's clock is the sum of the delays without the RTT and the sleeps (RTT takes no link time)
        assert r["link_time"][l] == pytest.approx(sum((o["delay"] - w.P["rtt"]) + o["sleep"] for o in live), rel=1e-12)
    assert r["errors"] == 0


def sum_lr(xs):
    s = 0.0
    for x in xs:
        s = s + x
    return s


@pytest.mark.parametrize("policy", POLICIES)
def test_players_with_identical_slots_and_joins_get_identical_trajectories(policy):
    w = world(seed=1)
    G, steps = 4, 12
    actions = np.repeat(np.random.default_rng(3).integers(0, w.A, size=(steps, 1)), 2 * G, 1).astype(np.int32)
    r = sl.run_shared(w, steps, G, [1, 2], [2.0, 0.0], join_delay=[1.5] * 2 * G, policy=policy, seed=3,
                      actions=actions)
    for key in ("delay", "sleep", "buffer", "rebuf", "reward", "request_time"):
        for l in range(2):
            blk = r[key][:, l * G:(l + 1) * G]
            if policy == sl.RANDOM:      # draws are keyed by the session: only the first download is the same
                continue
            assert np.array_equal(blk, np.repeat(blk[:, :1], G, 1)), (key, l)
    assert (r["request_time"][0] == 1.5).all()


def test_permuting_the_slots_of_a_link_permutes_its_outputs():
    w = world(seed=2, V=8)
    G, steps = 5, 14
    pols = [sl.BOLA, sl.RATE, sl.BBA, sl.DYNAMIC, sl.FIXED]
    join = np.array([0.0, 3.0, 3.0, 0.5, 7.25])
    rng = np.random.default_rng(9)
    actions = rng.integers(0, w.A, size=(steps, G)).astype(np.int32)
    knobs = spo.fill(G, WIDE, bba_reservoir=rng.uniform(2, 8, G), rb_safety=rng.uniform(0.5, 1.2, G))
    base = sl.run_shared(w, steps, G, [3], [4.0], join_delay=join, player_policy=pols, actions=actions, knobs=knobs)
    perm = [3, 0, 4, 1, 2]
    r = sl.run_shared(w, steps, G, [3], [4.0], join_delay=join[perm], player_policy=[pols[p] for p in perm],
                      actions=actions[:, perm], knobs=knobs[:, perm])
    for key in ("delay", "sleep", "buffer", "rebuf", "reward", "request_time", "actions", "eov"):
        assert np.array_equal(r[key], base[key][:, perm]), key
    for key in ("acc", "qoe_cost"):
        assert np.array_equal(r[key], base[key][..., perm]), key
    for key in ("chunk", "buffer", "pos", "phase", "seg"):
        assert np.array_equal(r["state"][key], base["state"][key][perm]), key
    for key in ("link_time", "link_capacity"):
        assert np.array_equal(r[key], base[key]), key
    assert r["link_delivered"][0] == pytest.approx(base["link_delivered"][0], rel=1e-15)   # only the summation order


def constant_world(bw=1000.0, T=8, V=6, **kw):
    sizes = np.tile(np.array([[1000.0, 2500.0, 4000.0, 6000.0]]), (V, 1))
    return sl.World(np.full((1, T), bw), [T], [1.0], sizes, sizes * 0.001, dict(P0, **kw), WIDE)


def test_two_players_requesting_together_each_see_half_the_bandwidth():
    w = constant_world()
    actions = np.full((3, 2), 2, np.int32)
    r = sl.run_shared(w, 3, 2, [0], policy=sl.FIXED, actions=actions)
    exp = 2 * 4000.0 / (1000.0 * 0.95) + 0.08
    assert r["delay"][0] == pytest.approx([exp, exp], rel=1e-12)


@pytest.mark.parametrize("G", [1, 2, 3, 7])
def test_a_busy_link_delivers_the_capacity_it_traverses(G):
    w = world(seed=4, max_buffer=1e9)     # no sleep: from the first request on, some download is always active
    rng = np.random.default_rng(G)
    actions = rng.integers(0, w.A, size=(10, 2 * G)).astype(np.int32)
    r = sl.run_shared(w, 10, G, [0, 3], [0.0, 5.5], policy=sl.FIXED, actions=actions)
    np.testing.assert_allclose(r["link_delivered"], r["link_capacity"], rtol=1e-12)
    np.testing.assert_allclose(r["link_delivered"], actions_sizes(w, actions, G), rtol=1e-15)


def actions_sizes(w, actions, G):
    steps, N = actions.shape
    tot = np.zeros(N // G)
    for i in range(N):
        for k in range(steps):
            tot[i // G] += w.sizes[k % w.V][actions[k, i]]
    return tot


def test_staggered_join_known_answer():
    # payload 1: 1000 units/s.  A requests 4000 at t = 0, B the same at t = 1.  A is alone for 1 s (1000 units), then
    # both share: A's last 3000 take 6 s (t = 7), by then B has 3000 and takes 1 s more at the full rate (t = 8).
    w = constant_world(payload=1.0, rtt=0.0)
    actions = np.full((1, 2), 2, np.int32)
    r = sl.run_shared(w, 1, 2, [0], join_delay=[0.0, 1.0], policy=sl.FIXED, actions=actions)
    assert r["request_time"][0].tolist() == [0.0, 1.0]
    assert r["delay"][0] == pytest.approx([7.0, 7.0], rel=1e-12)
    assert r["link_time"][0] == pytest.approx(8.0, rel=1e-12)
    assert r["link_capacity"][0] == pytest.approx(8000.0, rel=1e-12)
    assert r["link_delivered"][0] == 8000.0
    assert r["rebuf"][0].tolist() == r["delay"][0].tolist()       # an empty buffer stalls for the whole download


def test_exact_ties_and_short_traces_that_wrap_inside_a_download():
    w = world(seed=5, T=3, n_traces=2)
    G = 4
    r = sl.run_shared(w, 20, G, [0, 1], join_delay=[0.0, 2.0, 2.0, 0.0] * 2, player_policy=[sl.BOLA, sl.RATE] * 2)
    assert r["errors"] == 0
    assert (np.diff(r["request_time"], axis=0) >= 0).all()
    assert (r["delay"] > 0).all()


def test_bad_join_delays_and_trace_ids_count_once_per_player_and_join_at_zero():
    w = world(seed=6)
    r = sl.run_shared(w, 3, 2, [99, 0], join_delay=[-1.0, math.nan, math.inf, 0.0], policy=sl.BBA)
    assert r["request_time"][0].tolist() == [0.0, 0.0, 0.0, 0.0]
    assert r["errors"] == 2 + 1 + 1 + 1      # trace id 99 for both players of link 0; the three bad delays
    assert r["state"]["trace_id"].tolist() == [0, 0, 0, 0]


# ---- the C-ABI without a device ----
def header_text():
    with open(os.path.join(ROOT, "include", "abr_b200_shared.h")) as f:
        return f.read()


def test_the_header_matches_its_ctypes_table():
    text = re.sub(r"/\*.*?\*/", " ", header_text(), flags=re.S)
    text = "\n".join(line for line in text.splitlines() if not line.lstrip().startswith("#"))
    decls = re.findall(r"([A-Za-z_][\w \t\n*]*?)\b(abr_\w+)\s*\(([^()]*)\)\s*;", text)
    assert [d[1] for d in decls] == list(_lib.SHARED_SIGNATURES)

    def kind(c):
        c = " ".join(c.replace("*", " * ").split())
        if "*" in c:
            base = c.replace("const", "").replace("*", "").split()[0]
            return ("ptr", base if base == "AbrSharedOutputs" else None)
        return {"int": "i32", "void": "void", "uint64_t": "u64", "long long": "i64"}[c]
    for ret, name, params in decls:
        restype, argtypes = _lib.SHARED_SIGNATURES[name]
        types = [re.sub(r"\w+$", "", p.strip()).strip() for p in params.split(",")]
        assert [ctypes_kind(t) for t in argtypes] == [kind(t) for t in types], name
        assert ctypes_kind(restype) == kind(ret.split()[-1]), name
    fields = re.search(r"typedef struct AbrSharedOutputs \{(.*?)\} AbrSharedOutputs;", text + header_text(), re.S).group(1)
    assert re.findall(r"\*\s*(d_\w+)", fields) == [f for f, _ in _lib.AbrSharedOutputs._fields_]


def test_the_build_tracks_the_header_and_the_library_carries_the_table():
    from abrsimulator_b200 import _build
    assert any(h.endswith("abr_b200_shared.h") for h in _build.HEADERS)
    assert "abr_shared.cu" in _build.SOURCES
    lib = _lib.load()
    for name, (restype, argtypes) in _lib.SHARED_SIGNATURES.items():
        fn = getattr(lib, name)
        assert fn.restype is restype and list(fn.argtypes) == argtypes, name


def test_a_null_env_fails_first_without_a_device():
    lib = _lib.load()
    rc = lib.abr_env_run_shared(None, 2, None, 0, 4, 40, None, None, None, 1, 0, None, None, None, None, None)
    assert rc == 1 and b"NULL" in lib.abr_last_error()


def test_jain_index():
    pytest.importorskip("torch")
    from abrsimulator_b200.env import jain_index
    j = jain_index(np.array([[1.0, 1.0, 1.0, 1.0], [4.0, 0.0, 0.0, 0.0], [1.0, 3.0, 1.0, 3.0]]))
    assert j.tolist() == [1.0, 0.25, 0.8]
