"""CPU only: per-session policy parameters (SPEC §4.7).  The C restatement against the pure-Python one, its identities
against the environment-wide oracles, the device derivation of BOLA's (Vp, gp), the header against its ctypes table,
the checks a call makes without a device, and the dispatch of the new kernel forms against the GPU case table."""
import ctypes
import os
import re

import numpy as np
import pytest

from abrsimulator_b200 import _lib
from helpers import small_world
from test_capi_signatures import ctypes_kind
import dynamic_oracle as do
import policy_oracle as po
import session_params_oracle as so

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
POLICIES = (po.POLICY_BBA, po.POLICY_RATE, po.POLICY_BOLA, do.POLICY_DYNAMIC)


def random_state(N, seed, V=20, A=6, K=5):
    rng = np.random.default_rng(seed)
    _, sizes, _, _, _ = small_world(n_traces=2, T=16, V=V)
    chunk = rng.integers(0, V, N).astype(np.int32)
    chunk[rng.random(N) < 0.1] = 0
    buffer = rng.uniform(0.0, 45.0, N)
    ring = rng.uniform(0.1, 8.0, (N, K))
    hist_len = rng.integers(0, 12, N).astype(np.int32)
    mode = rng.integers(0, 2, N).astype(np.uint8)
    done = (rng.random(N) < 0.05).astype(np.uint8)
    return sizes, chunk, buffer, ring, hist_len, mode, done


def random_knobs(N, seed, vmax_zero=False):
    rng = np.random.default_rng(seed)
    mn = rng.uniform(0.5, 20.0, N)
    on = rng.uniform(0.5, 25.0, N)
    x = np.stack([rng.uniform(-5.0, 20.0, N), rng.uniform(1e-9, 30.0, N), rng.uniform(0.2, 1.6, N), mn,
                  mn + rng.uniform(0.0, 40.0, N), on, on * rng.uniform(0.0, 1.0, N)])
    s = rng.choice(N, 4 * (N // 10), replace=False).reshape(4, -1)
    x[1, s[0]] = 1e-12                                      # a tiny cushion
    x[4, s[1]] = np.nextafter(x[3, s[1]], np.inf)           # min ~ target
    x[6, s[2]] = np.nextafter(x[5, s[2]], 0.0)              # off ~ on
    x[2, s[3]] = 1e-300
    assert so.first_invalid(x) is None
    return x


@pytest.mark.parametrize("policy", POLICIES)
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_c_oracle_equals_python_restatement(policy, seed):
    N = 1500
    sizes, chunk, buffer, ring, hist_len, mode, done = random_state(N, seed)
    x = random_knobs(N, seed + 10)
    act, m = so.sp_decide(policy, sizes, x, chunk, buffer, ring, hist_len, mode, done=done)
    v, vmax = po.bola_table(sizes)
    for s in range(N):
        if done[s] and policy != po.POLICY_BBA:
            assert act[s] == 0 and m[s] == mode[s]
            continue
        n = min(int(hist_len[s]), ring.shape[1])
        hist = [ring[s, (hist_len[s] - n + j) % ring.shape[1]] for j in range(n)]
        a, mm = so.session_action(policy, list(sizes[chunk[s]]), v[chunk[s]], vmax, hist, float(buffer[s]),
                                  int(chunk[s]), int(mode[s]), 1, 4.0, [float(y) for y in x[:, s]])
        assert (act[s], m[s]) == (a, mm), s


def test_flat_ladders_answer_0_under_bola():
    """v_max = 0 (every ladder flat): BOLA answers 0 whatever the knobs; gp = 0 and Vp = inf are derived as the host
    derives them."""
    N = 50
    sizes = np.full((6, 4), 2.0)
    x = random_knobs(N, 3)
    rng = np.random.default_rng(3)
    act, _ = so.sp_decide(po.POLICY_BOLA, sizes, x, rng.integers(0, 6, N), rng.uniform(0, 40, N),
                          rng.uniform(1, 3, (N, 5)), np.full(N, 3), np.zeros(N))
    assert (act == 0).all()
    Vp, gp = so.bola_derive(0.0, 10.0, 30.0)
    assert gp == 0.0 and Vp == np.inf


@pytest.mark.parametrize("policy", POLICIES)
def test_uniform_knobs_are_the_environment_wide_oracle(policy):
    N = 2000
    sizes, chunk, buffer, ring, hist_len, mode, done = random_state(N, 7)
    pp = dict(rb_safety=0.8, bola_min_buffer=6.0, bola_target_buffer=40.0)
    dp = dict(switch_on_buffer=9.0, switch_off_buffer=4.0)
    wide = [4.0, 12.0, pp["rb_safety"], pp["bola_min_buffer"], pp["bola_target_buffer"], dp["switch_on_buffer"],
            dp["switch_off_buffer"]]
    x = np.repeat(np.array(wide)[:, None], N, axis=1)
    got, m = so.sp_decide(policy, sizes, x, chunk, buffer, ring, hist_len, mode, done=done)
    if policy == do.POLICY_DYNAMIC:
        exp, me = do.dynamic_decide(sizes, chunk, buffer, ring, hist_len, mode, done=done, **pp, **dp)
        assert np.array_equal(m, me)
    else:
        exp = po.policy_decide(policy, sizes, chunk, buffer, ring, hist_len, done=done, bba_reservoir=4.0,
                               bba_cushion=12.0, **pp)
    assert np.array_equal(got, exp)


@pytest.mark.parametrize("policy", POLICIES)
def test_a_partition_is_g_environment_wide_episodes(policy):
    """G configurations over one batch of oracle sessions equal G environment-wide oracle runs, session for session."""
    bitrates, sizes, bw, tl, ti = small_world(n_traces=6, T=120, V=20)
    N, G, steps = 240, 3, 30
    rng = np.random.default_rng(4)
    tid, off = rng.integers(0, 6, N).astype(np.int32), rng.uniform(0, 300.0, N)
    grid = [dict(bba_reservoir=3.0 + g, bba_cushion=6.0 + 5 * g, rb_safety=0.6 + 0.25 * g, bola_min_buffer=5.0 + 3 * g,
                 bola_target_buffer=20.0 + 8 * g, switch_on_buffer=8.0 + 4 * g, switch_off_buffer=2.0 + 2 * g)
            for g in range(G)]
    group = np.arange(N) % G
    sweep = so.SessionParamsEnv(bw, tl, ti, sizes, bitrates, N, track_history=1)
    sweep.reset(tid, off)
    assert sweep.set_session_params(**{f: np.array([grid[g][f] for g in group]) for f in so.FIELDS})
    got = sweep.rollout(policy, steps)
    for g in range(G):
        msk = group == g
        e = do.DynamicEnv(bw, tl, ti, sizes, bitrates, int(msk.sum()), track_history=1,
                          bba_reservoir=grid[g]["bba_reservoir"], bba_cushion=grid[g]["bba_cushion"])
        assert e.set_policy_params(**{f: grid[g][f] for f in ("rb_safety", "bola_min_buffer", "bola_target_buffer")})
        assert e.set_dynamic_params(**{f: grid[g][f] for f in ("switch_on_buffer", "switch_off_buffer")})
        e.reset(tid[msk], off[msk])
        exp = e.stepwise_rollout(policy, steps)
        for k in ("actions", "delay", "buffer", "reward"):
            assert np.array_equal(np.ascontiguousarray(got[k][:, msk]).view(np.uint8), exp[k].view(np.uint8)), (g, k)


def test_device_derivation_is_install_policy_params():
    """gp = v_max / (target / min - 1.0), Vp = min / gp: fp64, two divisions and a subtraction, no FMA; numpy
    restates it element-wise and the C oracle derives the environment-wide pair with the same operations."""
    rng = np.random.default_rng(5)
    mn = rng.uniform(1e-3, 50.0, 5000)
    tg = mn + rng.uniform(1e-9, 60.0, 5000)
    for vmax in (0.0, 0.5, float(np.log(4300 / 300))):
        with np.errstate(divide="ignore"):
            gp = vmax / (tg / mn - 1.0)
            Vp = mn / gp
        for s in range(0, 5000, 97):
            assert so.bola_derive(vmax, mn[s], tg[s]) == (Vp[s], gp[s])


def test_validation_order_c_and_python_agree():
    rng = np.random.default_rng(6)
    base = np.array([5.0, 10.0, 1.0, 10.0, 30.0, 12.0, 6.0])
    bad_values = [np.nan, np.inf, -np.inf, 0.0, -1.0, 1e300]
    for _ in range(400):
        x = np.repeat(base[:, None], 8, axis=1)
        for _ in range(rng.integers(1, 4)):
            x[rng.integers(0, 7), rng.integers(0, 8)] = bad_values[rng.integers(0, len(bad_values))]
        assert so.first_invalid(x) == so.first_invalid_py(x)


# ---- the C-ABI without a device ----
def test_null_env_and_bad_n_are_reported_without_a_device():
    lib = _lib.load()
    sp = _lib.AbrSessionPolicyParams()
    assert lib.abr_env_set_session_policy_params(None, ctypes.byref(sp), 4, None) == 1
    assert b"env is NULL" in lib.abr_last_error()
    assert lib.abr_env_set_session_policy_params(None, None, 0, None) == 1
    assert lib.abr_env_get_session_policy_params(None, None, 4, None) == 1


def header_text():
    with open(os.path.join(ROOT, "include", "abr_b200_session_params.h")) as f:
        return f.read()


def test_the_header_matches_its_ctypes_table():
    text = re.sub(r"/\*.*?\*/", " ", header_text(), flags=re.S)
    text = "\n".join(line for line in text.splitlines() if not line.lstrip().startswith("#"))
    decls = re.findall(r"([A-Za-z_][\w \t\n*]*?)\b(abr_\w+)\s*\(([^()]*)\)\s*;", text)
    assert [d[1] for d in decls] == list(_lib.SESSION_PARAMS_SIGNATURES)

    def kind(c):
        c = " ".join(c.replace("*", " * ").split())
        if "*" in c:
            base = c.replace("const", "").replace("*", "").split()[0]
            return ("ptr", base if base == "AbrSessionPolicyParams" else None)
        return {"int": "i32", "void": "void"}[c]
    for ret, name, params in decls:
        restype, argtypes = _lib.SESSION_PARAMS_SIGNATURES[name]
        types = [re.sub(r"\w+$", "", p.strip()).strip() for p in params.split(",")]
        assert [ctypes_kind(t) for t in argtypes] == [kind(t) for t in types], name
        assert ctypes_kind(restype) == kind(ret.split()[-1]), name
    fields = re.search(r"typedef struct AbrSessionPolicyParams \{(.*?)\} AbrSessionPolicyParams;", header_text(),
                       re.S).group(1)
    names = re.findall(r"\*(d_\w+)", fields)
    assert names == [f for f, _ in _lib.AbrSessionPolicyParams._fields_] == ["d_" + f for f in so.FIELDS]
    assert tuple(_lib.SESSION_PARAM_FIELDS) == so.FIELDS


def test_the_build_tracks_the_header_and_the_library_carries_the_table():
    from abrsimulator_b200 import _build
    assert any(h.endswith("abr_b200_session_params.h") for h in _build.HEADERS)
    lib = _lib.load()
    for name, (restype, argtypes) in _lib.SESSION_PARAMS_SIGNATURES.items():
        fn = getattr(lib, name)
        assert fn.restype is restype and list(fn.argtypes) == argtypes, name


# ---- the forms ledger ----
NAMES = {po.POLICY_BBA: "BBA", po.POLICY_RATE: "RATE", po.POLICY_BOLA: "BOLA", do.POLICY_DYNAMIC: "DYNAMIC"}
EPISODE_FORMS = {(p, live, ot) for p in NAMES for live in (0, 1, 2) for ot in ("double", "float")}
DECIDE_FORMS = set(NAMES)


def test_the_dispatch_names_exactly_the_per_session_forms():
    with open(os.path.join(ROOT, "abrsimulator_b200", "csrc", "abr_step.cu")) as f:
        src = " ".join(f.read().split())
    # the episode: one per-session form per live mode, for each of the four policies, instantiated for both output types
    assert ("constexpr int PS = P | kPolicySession; if (live == 2) return go(abr_rollout_kernel<PS, false, false, 2, "
            "false, OT>, o); if (live == 1) return go(abr_rollout_kernel<PS, false, false, 1, false, OT>, o); "
            "return go(abr_rollout_kernel<PS, false, false, 0, false, OT>, o);") in src
    pols = re.findall(r"if \(v\.sp\.on && policy == ABR_POLICY_(\w+)\) e = launch_rollout_session_form<ABR_POLICY_(\w+)>",
                      src)
    assert sorted(a for a, b in pols if a == b) == sorted(NAMES.values())
    assert "template cudaError_t launch_rollout<double>(" in src and "template cudaError_t launch_rollout<float>(" in src
    # the decision: the per-session form of each of the four policies while the knobs are installed
    assert ("if (v.sp.on) abr_policy_decide_kernel<P | kPolicySession><<<grid, kStepBlock, 0, st>>>(v, d_action); "
            "else abr_policy_decide_kernel<P><<<grid, kStepBlock, 0, st>>>(v, d_action);") in src
    dec = re.findall(r"case ABR_POLICY_(\w+): launch_decide_form<ABR_POLICY_(\w+)>\(v, d_action, st\);", src)
    assert sorted(a for a, b in dec if a == b) == sorted(NAMES.values())
    assert len(EPISODE_FORMS) == 24 and len(DECIDE_FORMS) == 4


def test_the_gpu_cases_cover_every_form():
    """test_gpu_session_params.py: the oracle matrix takes every policy x live 0/1 x fp64/fp32 form on both trace
    paths; live 2 (the speed controller) runs in the sweep identity for every policy (its fp32 form through the
    same template, checked by the matrix's fp32 legs); the decision test takes the four decision forms."""
    with open(os.path.join(ROOT, "tests", "test_gpu_session_params.py")) as f:
        src = f.read()
    assert '@pytest.mark.parametrize("dtype", ["f64", "f32"])' in src
    assert '@pytest.mark.parametrize("live", [0, 1])' in src and '@pytest.mark.parametrize("live", [0, 1, 2])' in src
    assert '@pytest.mark.parametrize("layout", ["smem", "global"])' in src
    assert "def test_decide_matches_oracle_and_decide_plus_step_is_the_episode(policy)" in src
