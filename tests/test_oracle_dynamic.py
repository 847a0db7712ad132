"""CPU-only: the DYNAMIC policy of SPEC §4.6 in the C restatement (tests/dynamic_oracle.c) and the pure-Python one,
its known answers and identities on the environment oracle, the C-ABI's parameter handling, include/abr_b200_dynamic.h
against the ctypes table _lib.DYNAMIC_SIGNATURES, and the ledger of the kernel forms a DYNAMIC call takes."""
import ctypes
import os
import re

import numpy as np
import pytest

import dynamic_oracle as do
import policy_oracle as po
from abrsimulator_b200 import _lib
from helpers import small_world
from test_capi_signatures import ROOT, ctypes_kind

LADDER = [300.0, 750.0, 1200.0, 1850.0, 2850.0, 4300.0]
ON, OFF = 12.0, 6.0


def decide(sizes, chunk, buffer, mode, ring=None, hist_len=0, done=None, **kw):
    """One-session (or few-session) DYNAMIC decisions; ring defaults to five samples of 2000."""
    chunk, buffer, mode = np.atleast_1d(chunk), np.atleast_1d(buffer), np.atleast_1d(mode)
    N = len(buffer)
    ring = np.full((N, 5), 2000.0) if ring is None else np.atleast_2d(ring)
    hist_len = np.broadcast_to(np.atleast_1d(hist_len), (N,))
    return do.dynamic_decide(np.atleast_2d(sizes), chunk, buffer, ring, hist_len, mode, done=done, **kw)


def rate_and_bola(sizes, chunk, buffer, ring, hist_len, **kw):
    pp = {k: v for k, v in kw.items() if k in po.DEFAULTS}
    r = po.policy_decide(po.POLICY_RATE, sizes, chunk, buffer, ring, hist_len, **pp)
    b = po.policy_decide(po.POLICY_BOLA, sizes, chunk, buffer, ring, hist_len, **pp)
    return r, b


# ---- known answers ----
def test_a_rising_buffer_switches_to_bola_at_the_first_buffer_above_switch_on():
    sizes = np.array([LADDER] * 8)
    mode = np.zeros(1, np.uint8)
    path = [0.0, 4.0, 8.0, 11.999, ON, np.nextafter(ON, np.inf), 20.0, 35.0]
    modes = []
    for k, b in enumerate(path):
        a, mode = decide(sizes, k, b, mode)
        modes.append(int(mode[0]))
        r, bo = rate_and_bola(sizes, [k], [b], np.full((1, 5), 2000.0), [0])
        assert a[0] == (bo[0] if mode[0] else r[0]), k
    assert modes == [0, 0, 0, 0, 0, 1, 1, 1]               # 12 itself does not switch: strict >


def test_between_the_thresholds_the_mode_holds_from_either_side():
    sizes = np.array([LADDER] * 4)
    for b in (np.nextafter(OFF, np.inf), 7.0, 9.0, 11.0, ON):
        for m in (0, 1):
            _, m2 = decide(sizes, 2, b, [m])
            assert m2[0] == m, (b, m)


def test_bola_hands_back_at_a_buffer_at_or_below_switch_off():
    sizes = np.array([LADDER] * 4)
    for b in (OFF, 5.0, 0.0):
        a, m = decide(sizes, 3, b, [1])
        r, _ = rate_and_bola(sizes, [3], [b], np.full((1, 5), 2000.0), [0])
        assert m[0] == 0 and a[0] == r[0], b
    _, m = decide(sizes, 3, np.nextafter(OFF, np.inf), [1])
    assert m[0] == 1


def test_the_first_decision_of_an_episode_ignores_the_stored_mode():
    sizes = np.array([LADDER] * 4)
    ring = np.full((1, 5), 900.0)
    for b in (0.0, 8.0, ON):                               # chunk 0 after any reset has b = 0; 8 and 12 pin the rule
        a, m = decide(sizes, 0, b, [1], ring=ring, hist_len=3)
        r, _ = rate_and_bola(sizes, [0], [b], ring, [3])
        assert m[0] == 0 and a[0] == r[0], b
    _, m = decide(sizes, 1, 8.0, [1], ring=ring, hist_len=3)
    assert m[0] == 1                                      # the same state past chunk 0 keeps BOLA


def test_done_sessions_answer_0_and_keep_their_mode():
    sizes = np.array([LADDER] * 2)
    a, m = decide(sizes, [2, 2], [40.0, 1.0], [0, 1], done=np.array([1, 1], np.uint8))
    assert a.tolist() == [0, 0] and m.tolist() == [0, 1]


# ---- the C oracle against the Python restatement ----
@pytest.mark.parametrize("seed", range(3))
def test_c_oracle_equals_python_restatement_on_random_states(seed):
    rng = np.random.default_rng(seed)
    N, V, A, K = 4000, 7, 6, 5
    sizes = np.sort(rng.uniform(50.0, 20000.0, size=(V, A)), axis=1)
    sizes[1] = rng.uniform(50.0, 20000.0, size=A)
    sizes[2, 3] = sizes[2, 2]
    sizes[3] = 1000.0
    on, off = [(12.0, 6.0), (20.0, 0.0), (8.0, 7.5)][seed]
    chunk = rng.integers(0, V + 1, size=N).astype(np.int32)          # V: done
    chunk[::13] = 0
    done = (chunk == V).astype(np.uint8)
    buffer = rng.uniform(0.0, 40.0, size=N)
    buffer[::7] = on                                                 # exactly on each threshold
    buffer[3::7] = off
    buffer[5::11] = np.nextafter(on, np.inf)
    mode = rng.integers(0, 2, size=N).astype(np.uint8)
    hist_len = rng.integers(0, 3 * K, size=N).astype(np.int32)
    ring = rng.uniform(100.0, 8000.0, size=(N, K))
    dq = int(rng.integers(-1, A))
    pp = dict(rb_safety=float(rng.choice([1.0, 0.8])), bola_min_buffer=float(rng.choice([5.0, 10.0])),
              bola_target_buffer=float(rng.choice([20.0, 30.0])))
    act, m = do.dynamic_decide(sizes, np.minimum(chunk, V - 1), buffer, ring, hist_len, mode, done=done,
                               default_quality=dq, chunk_length=4.0, switch_on_buffer=on, switch_off_buffer=off, **pp)
    v, vmax = po.bola_table(sizes.tolist())
    for s in range(N):
        if done[s]:
            assert act[s] == 0 and m[s] == mode[s], s
            continue
        L = int(hist_len[s])
        n = min(L, K)
        hist = [float(ring[s, (L - n + j) % K]) for j in range(n)]
        k = int(chunk[s])
        q, mm = do.dynamic_action(sizes[k].tolist(), v[k], vmax, hist, float(buffer[s]), k, int(mode[s]), dq, 4.0,
                                  on, off, **pp)
        assert (act[s], m[s]) == (q, mm), s
    live = done == 0
    # the states reach every branch: both modes in and out, both switches, chunk 0 with a stored BOLA mode
    for mi in (0, 1):
        for mo in (0, 1):
            assert ((mode == mi) & (m == mo) & live & (chunk > 0)).any(), (mi, mo)
    assert ((chunk == 0) & (mode == 1) & live).any() and (buffer == on).any() and (buffer == off).any()


def test_two_decisions_without_a_step_agree():
    rng = np.random.default_rng(9)
    N, V, A, K = 3000, 5, 6, 5
    sizes = np.sort(rng.uniform(100.0, 9000.0, size=(V, A)), axis=1)
    chunk = rng.integers(0, V, size=N).astype(np.int32)
    buffer = rng.choice([0.0, OFF, 7.0, ON, 13.0, 30.0], size=N)
    mode = rng.integers(0, 2, size=N).astype(np.uint8)
    hist_len = rng.integers(0, 8, size=N).astype(np.int32)
    ring = rng.uniform(100.0, 8000.0, size=(N, K))
    a1, m1 = do.dynamic_decide(sizes, chunk, buffer, ring, hist_len, mode)
    a2, m2 = do.dynamic_decide(sizes, chunk, buffer, ring, hist_len, m1)
    assert np.array_equal(a1, a2) and np.array_equal(m1, m2)
    assert (m1 != mode).any()


# ---- identities on the environment oracle ----
def _pair(N=300, V=20, **P):
    bitrates, sizes, bw, tl, ti = small_world(n_traces=6, T=120, V=V, ragged=True)
    mk = lambda: do.DynamicEnv(bw, tl, ti, sizes, bitrates, N, track_history=1, **P)
    rng = np.random.default_rng(4)
    tid, off = rng.integers(0, 6, size=N).astype(np.int32), rng.uniform(0, 300.0, size=N)
    a, b = mk(), mk()
    a.reset(tid, off)
    b.reset(tid, off)
    return a, b


def test_an_unreachable_switch_on_is_the_rate_episode_bit_for_bit():
    a, b = _pair()
    assert a.set_dynamic_params(switch_on_buffer=1e300)
    x = a.rollout(do.POLICY_DYNAMIC, 50)
    y = b.rollout(po.POLICY_RATE, 50)
    for k in ("delay", "sleep", "buffer", "rebuf", "reward", "latency", "acc"):
        assert np.array_equal(x[k].view(np.uint64), y[k].view(np.uint64)), k
    assert np.array_equal(x["actions"], y["actions"]) and np.array_equal(x["eov"], y["eov"])
    assert (a.dyn_mode == 0).all() and y["eov"].sum() >= 300


@pytest.mark.parametrize("params", [dict(), dict(rb_safety=0.8, bola_min_buffer=6.0, bola_target_buffer=40.0)])
def test_the_smallest_switch_on_is_rate_at_chunk_0_and_bola_after(params):
    """off = 0, on = 5e-324: the pre-step buffer after any download is > 0 (on demand, buffer >= L after a step)."""
    a, _ = _pair()
    assert a.set_dynamic_params(switch_on_buffer=5e-324, switch_off_buffer=0.0)
    if params:
        assert a.set_policy_params(**params)
    saw_reset = False
    for t in range(50):
        chunk = a.field("chunk")
        r = a.policy_decide(po.POLICY_RATE)
        b = a.policy_decide(po.POLICY_BOLA)
        q = a.policy_decide(do.POLICY_DYNAMIC)
        assert np.array_equal(q, np.where(chunk == 0, r, b)), t
        assert np.array_equal(a.dyn_mode, (chunk != 0).astype(np.uint8)), t
        saw_reset |= bool((chunk == 0).any() and t > 0)
        a.step(q, want_next_sizes=False)
    assert saw_reset


def test_the_oracle_episode_switches_both_ways():
    a, _ = _pair(N=400, V=40)
    a.rollout(do.POLICY_DYNAMIC, 80)
    up, down = a.switches()
    assert up > 0 and down > 0


# ---- parameters ----
BAD = [dict(switch_on_buffer=float("nan")), dict(switch_off_buffer=float("nan")), dict(switch_on_buffer=float("inf")),
       dict(switch_off_buffer=float("-inf")), dict(switch_on_buffer=6.0), dict(switch_on_buffer=5.0),
       dict(switch_off_buffer=-1.0), dict(switch_off_buffer=-0.5, switch_on_buffer=0.0)]


@pytest.mark.parametrize("bad", BAD, ids=lambda d: ",".join(f"{k}={v}" for k, v in d.items()))
def test_invalid_dynamic_params_are_rejected_without_a_device(bad):
    lib = _lib.load()
    dp = _lib.AbrDynamicParams()
    lib.abr_dynamic_params_default(ctypes.byref(dp))
    for k, v in bad.items():
        setattr(dp, k, v)
    assert lib.abr_env_set_dynamic_params(None, ctypes.byref(dp)) == 1
    assert b"switch_off_buffer < switch_on_buffer" in lib.abr_last_error(), lib.abr_last_error()
    assert do.params_invalid(**bad)
    sizes = np.array([LADDER])
    e = do.DynamicEnv(np.ones((1, 4)), [4], [1.0], sizes, sizes, 1)
    assert not e.set_dynamic_params(**bad) and e.dynamic_params == do.DEFAULTS


def test_defaults_size_and_valid_params_with_a_null_env():
    lib = _lib.load()
    dp = _lib.AbrDynamicParams()
    lib.abr_dynamic_params_default(ctypes.byref(dp))
    assert (dp.switch_on_buffer, dp.switch_off_buffer) == (12.0, 6.0) and do.DEFAULTS == dict(switch_on_buffer=12.0,
                                                                                            switch_off_buffer=6.0)
    assert ctypes.sizeof(_lib.AbrDynamicParams) == 16
    for on, off in ((12.0, 6.0), (5e-324, 0.0), (1e300, 0.0)):
        assert not do.params_invalid(switch_on_buffer=on, switch_off_buffer=off)
        assert lib.abr_env_set_dynamic_params(None, ctypes.byref(_lib.AbrDynamicParams(on, off))) == 1
        assert b"env is NULL" in lib.abr_last_error()
    assert lib.abr_env_set_dynamic_params(None, None) == 1 and b"NULL" in lib.abr_last_error()
    assert lib.abr_env_policy_decide(None, do.POLICY_DYNAMIC, None, None) == 1
    assert b"env is NULL" in lib.abr_last_error()


# ---- include/abr_b200_dynamic.h against the binding ----
def header_text():
    with open(os.path.join(ROOT, "include", "abr_b200_dynamic.h")) as f:
        return f.read()


def test_the_companion_header_matches_its_ctypes_table():
    text = re.sub(r"/\*.*?\*/", " ", header_text(), flags=re.S)
    text = "\n".join(line for line in text.splitlines() if not line.lstrip().startswith("#"))
    decls = re.findall(r"([A-Za-z_][\w \t\n*]*?)\b(abr_\w+)\s*\(([^()]*)\)\s*;", text)
    assert [d[1] for d in decls] == list(_lib.DYNAMIC_SIGNATURES)
    others = (set(_lib.SIGNATURES) | set(_lib.EXTRA_SIGNATURES) | set(_lib.MPC_PRED_SIGNATURES) |
              set(_lib.OBS_SIGNATURES) | set(_lib.MPC_SCEN_SIGNATURES))
    assert not set(_lib.DYNAMIC_SIGNATURES) & others

    def kind(c):
        c = " ".join(c.replace("*", " * ").split())
        if "*" in c:
            base = c.replace("const", "").replace("*", "").split()[0]
            return ("ptr", base if base == "AbrDynamicParams" else None)
        return {"int": "i32", "void": "void"}[c]
    for ret, name, params in decls:
        restype, argtypes = _lib.DYNAMIC_SIGNATURES[name]
        types = [re.sub(r"\w+$", "", p.strip()).strip() for p in params.split(",")]
        assert [ctypes_kind(t) for t in argtypes] == [kind(t) for t in types], name
        assert ctypes_kind(restype) == kind(ret.split()[-1]), name


def test_the_header_constants_match_the_binding():
    defs = {k: int(v) for k, v in re.findall(r"#define\s+(ABR_\w+)\s+(\d+)", header_text())}
    assert defs == dict(ABR_POLICY_DYNAMIC=_lib.POLICY_DYNAMIC, ABR_F_DYN_MODE=_lib.FIELDS["dyn_mode"][0])
    assert _lib.POLICY_DYNAMIC == do.POLICY_DYNAMIC == 5 and _lib.FIELDS["dyn_mode"] == (24, "uint8")
    fields = re.search(r"typedef struct AbrDynamicParams \{(.*?)\} AbrDynamicParams;", header_text(), re.S).group(1)
    assert fields.split() == ["double", "switch_on_buffer,", "switch_off_buffer;"]
    assert [f for f, _ in _lib.AbrDynamicParams._fields_] == ["switch_on_buffer", "switch_off_buffer"]


def test_the_loaded_library_carries_the_table_and_the_build_tracks_the_header():
    from abrsimulator_b200 import _build
    lib = _lib.load()
    for name, (restype, argtypes) in _lib.DYNAMIC_SIGNATURES.items():
        fn = getattr(lib, name)
        assert fn.restype is restype and list(fn.argtypes) == argtypes, name
    assert any(h.endswith("abr_b200_dynamic.h") for h in _build.HEADERS)


# ---- the forms ledger ----
def dynamic_form(call, live=False, dtype="f64"):
    """The kernel instantiation a DYNAMIC call takes, as launch_rollout_form / launch_policy_decide choose it: the
    episode takes RATE's forms (it reads the history ring, so the FAST / NOOUT forms never apply), the general form or
    the live form, with fp64 or fp32 outputs; the decision takes its own kernel.
    abr_rollout_kernel<POLICY, FAST, NOOUT, LIVE, UNI, OT>."""
    if call == "decide":
        return "abr_policy_decide_kernel<5>"
    ot = "double" if dtype == "f64" else "float"
    return f"abr_rollout_kernel<5, false, false, {'true' if live else 'false'}, false, {ot}>"


FORMS = {dynamic_form("episode", live, dt) for live in (False, True) for dt in ("f64", "f32")} | {dynamic_form("decide")}

# The cases of tests/test_gpu_dynamic.py and the forms their DYNAMIC calls reach.
GPU_CASES = {
    "test_fused_episode_matches_oracle": {dynamic_form("episode")},
    "test_split_episode_equals_one_episode": {dynamic_form("episode")},
    "test_run_and_run_host_equal_reset_and_rollout": {dynamic_form("episode")},
    "test_fp32_outputs_are_the_fp64_outputs_rounded_once": {dynamic_form("episode"), dynamic_form("episode", False, "f32")},
    "test_fused_live_episode_matches_oracle": {dynamic_form("episode", True)},
    "test_fused_live_episode_with_fp32_outputs": {dynamic_form("episode", True, "f32")},
    "test_policy_decide_then_step_equals_the_fused_episode": {dynamic_form("decide"), dynamic_form("episode"),
                                                              dynamic_form("episode", True)},
}


def test_the_gpu_cases_reach_every_form():
    assert set().union(*GPU_CASES.values()) == FORMS and len(FORMS) == 5
    with open(os.path.join(ROOT, "tests", "test_gpu_dynamic.py")) as f:
        src = f.read()
    for name in GPU_CASES:
        assert re.search(rf"^def {name}\(", src, re.M), name


def test_the_restated_dispatch_matches_the_source_of_one_decision_kernel():
    with open(os.path.join(ROOT, "abrsimulator_b200", "csrc", "abr_step.cu")) as f:
        src = " ".join(f.read().split())
    assert "if constexpr (P == ABR_POLICY_RATE || P == ABR_POLICY_DYNAMIC) { if (fast || none) return cudaErrorInvalidValue; " \
           "return go(abr_rollout_kernel<P, false, false, false, false, OT>, o);" in src
    assert "if (live) return go(abr_rollout_kernel<P, false, false, true, false, OT>, o);" in src
    assert "case ABR_POLICY_DYNAMIC: e = launch_rollout_form<ABR_POLICY_DYNAMIC>(go, o, o_none, live, fast, none, uni);" in src
    assert "case ABR_POLICY_DYNAMIC: launch_decide_form<ABR_POLICY_DYNAMIC>(v, d_action, st); break;" in src
    assert "else abr_policy_decide_kernel<P><<<grid, kStepBlock, 0, st>>>(v, d_action);" in src
    # the episode's forms exist for fp64 and fp32 outputs: launch_rollout is instantiated for both
    assert "template cudaError_t launch_rollout<double>(" in src and "template cudaError_t launch_rollout<float>(" in src
