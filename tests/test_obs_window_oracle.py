"""CPU-only: the numpy restatement of the windowed observation (SPEC §4.5, tests/obs_window_oracle.py) on known
answers, include/abr_b200_obs.h against the ctypes table _lib.OBS_SIGNATURES, and the checks of both entry points
that need no device."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from abrsimulator_b200 import _lib
from oracle import oracle as orc
from test_capi_signatures import ROOT, ctypes_kind
import obs_window_oracle as wo


def make(W, A=6, V=48, N=64, scales=(1.0,) * 5, **params):
    bitrates, sizes, bw, tl, ti = wo.world(A, V=V)
    ref = orc.OracleEnv(bw, tl, ti, sizes, bitrates, N, **params)
    tid, off = wo.sessions(N, bw.shape[0], bw.shape[1])
    ref.reset(tid, off)
    w = wo.WindowObs(ref, W, scales)
    w.observe()
    return w


def test_first_observation_is_the_reset_state_with_empty_windows():
    w = make(8, default_quality=2, scales=(0.5, 0.1, 1e-3, 0.25, 1e-2))
    ref, o = w.ref, w.obs
    _, _, _, wt, wd, sz = wo.rows(ref.A, 8)
    assert np.array_equal(o[0], np.full(ref.N, wo.f32(w.util[0, 2] * 0.5)))
    assert not o[1].any() and np.array_equal(o[2], np.ones(ref.N, np.float32))
    assert not o[wt].any() and not o[wd].any()
    assert np.array_equal(o[sz], np.repeat(wo.f32(ref.sizes[0] * 1e-2)[:, None], ref.N, 1))


def test_window_of_one_is_the_last_sample():
    w = make(1, track_history=1)
    acts = wo.action_table(10, w.ref.N, w.ref.A)
    for t in range(10):
        out = w.step(acts[t])
        assert np.array_equal(w.obs[3], wo.f32(out["throughput"]))
        assert np.array_equal(w.obs[4], wo.f32(out["delay"]))
        assert np.array_equal(w.obs[0], wo.f32(w.util[w.ref.field("chunk") - 1, acts[t]]))


def test_newest_entries_equal_the_rows_of_the_4_1_observation():
    """The last window entries are row 1 and row 2 of the SPEC §4.1 observation at the same scales; the older ones
    are the earlier steps' entries, oldest first."""
    scales = (1.0, 1.0, 1e-3, 0.25, 1.0)
    w = make(8, scales=scales)
    acts = wo.action_table(12, w.ref.N, w.ref.A)
    hist_t, hist_d = [], []
    for t in range(12):
        out = w.step(acts[t])
        hist_t.append(wo.f32(out["throughput"] * scales[2]))
        hist_d.append(wo.f32(out["delay"] * scales[3]))
        k = min(t + 1, 8)
        assert np.array_equal(w.obs[3 + 8 - k:3 + 8], np.stack(hist_t[-k:]))
        assert np.array_equal(w.obs[3 + 16 - k:3 + 16], np.stack(hist_d[-k:]))
        assert not w.obs[3:3 + 8 - k].any() and not w.obs[3 + 8:3 + 16 - k].any()


@pytest.mark.parametrize("auto_reset", [1, 0])
def test_three_chunk_video_never_fills_a_window_of_eight(auto_reset):
    w = make(8, V=3, auto_reset=auto_reset)
    ref, N = w.ref, w.ref.N
    acts = wo.action_table(7, N, ref.A)
    for t in range(7):
        before = w.obs.copy()
        out = w.step(acts[t])
        k = t % 3 + 1 if auto_reset else min(t + 1, 3)
        if auto_reset and t % 3 == 2:           # the end of the video: the column is the new episode's first one
            assert np.array_equal(out["eov"], np.ones(N, np.uint8))
            assert not w.obs[3:19].any()
            assert np.array_equal(w.obs[2], np.ones(N, np.float32)) and not w.obs[1].any()
            continue
        assert not w.obs[3:3 + 8 - k].any() and w.obs[3 + 8 - k:11].all()
        assert not w.obs[11:19 - k].any() and w.obs[19 - k:19].all()
        if not auto_reset and t >= 3:           # inert: the windows are neither read nor written
            assert np.array_equal(w.obs[3:19], before[3:19])
            assert not w.obs[2].any() and not w.obs[19:].any()
        assert np.array_equal(w.obs[2], wo.f32((3.0 - ref.field("chunk")) / 3.0))


def test_products_are_rounded_once():
    """The restatement rounds the fp64 product once (fp32(x * s), not fp32(x) * fp32(s))."""
    w = make(8, scales=(1 / 3, 1 / 7, 1 / 11, 1 / 13, 1 / 17))
    out = w.step(wo.action_table(1, w.ref.N, w.ref.A)[0])
    assert np.array_equal(w.obs[10], (out["throughput"] * (1 / 11)).astype(np.float32))
    assert np.array_equal(w.obs[1], (w.ref.field("buffer") * (1 / 7)).astype(np.float32))


def test_negative_default_quality_gives_a_zero_utility_row():
    w = make(4, default_quality=-1)
    assert not w.obs[0].any()
    w.step(np.zeros(w.ref.N, np.int32))
    assert np.array_equal(w.obs[0], np.full(w.ref.N, wo.f32(w.util[0, 0])))


def test_case_table_covers_the_issue_grid():
    cases = wo.CASES
    assert {c[0] for c in cases} == {1, 8, 32} and {c[1] for c in cases} == {1, 6, 10}
    assert {c[2] for c in cases} == {1, 127, 3000, 2 ** 21 + 77}
    assert {c[4] for c in cases} == {0, 1} and {c[5] for c in cases} == {0, 1} and {c[6] for c in cases} == {0, 1}
    assert all(wo.STEPS > c[3] for c in cases) and wo.STEPS >= 60


# ---- the C-ABI ----
def header_declarations():
    with open(os.path.join(ROOT, "include", "abr_b200_obs.h")) as f:
        text = re.sub(r"/\*.*?\*/", " ", f.read(), flags=re.S)
    text = "\n".join(line for line in text.splitlines() if not line.lstrip().startswith("#"))
    struct = re.search(r"typedef struct AbrObsWindowSpec \{(.*?)\} AbrObsWindowSpec;", text, flags=re.S).group(1)
    decls = []
    for ret, name, params in re.findall(r"([A-Za-z_][\w \t\n*]*?)\b(abr_\w+)\s*\(([^()]*)\)\s*;", text):
        types = [re.sub(r"\w+$", "", p.strip()).strip() for p in params.split(",")]
        decls.append((name, ret.split()[-1], types))
    return struct, decls


def c_kind(t):
    t = " ".join(t.replace("*", " * ").split())
    if "*" in t:
        base = t.replace("const", "").replace("*", "").split()
        return ("ptr", base[0] if base and base[0] in ("AbrObsWindowSpec",) else None)
    return {"int": "i32", "int32_t": "i32", "uint64_t": "u64", "double": "f64", "void": "void"}[t]


def test_the_companion_header_matches_its_ctypes_table():
    struct, decls = header_declarations()
    assert [d[0] for d in decls] == list(_lib.OBS_SIGNATURES) == ["abr_env_step_policy_window", "abr_env_observe_window"]
    assert not set(_lib.OBS_SIGNATURES) & (set(_lib.SIGNATURES) | set(_lib.EXTRA_SIGNATURES) |
                                           set(_lib.MPC_PRED_SIGNATURES))
    for name, ret, params in decls:
        restype, argtypes = _lib.OBS_SIGNATURES[name]
        assert [ctypes_kind(t) for t in argtypes] == [c_kind(c) for c in params], name
        assert ctypes_kind(restype) == c_kind(ret), name
    fields = []
    for decl in filter(str.strip, struct.split(";")):
        typ, names = decl.split(None, 1)
        fields += [(n.strip(), typ) for n in names.split(",")]
    assert fields == [("window", "int32_t")] + [(n, "double") for n in (
        "util_scale", "buffer_scale", "throughput_scale", "delay_scale", "size_scale")]
    assert [(n, t) for n, t in _lib.AbrObsWindowSpec._fields_] == [("window", C.c_int32)] + [
        (n, C.c_double) for n, _ in fields[1:]]


def test_the_loaded_library_carries_the_table():
    lib = _lib.load()
    for name, (restype, argtypes) in _lib.OBS_SIGNATURES.items():
        fn = getattr(lib, name)
        assert fn.restype is restype and list(fn.argtypes) == argtypes, name


def test_a_null_env_is_reported_before_anything_else():
    lib = _lib.load()
    bad = _lib.AbrObsWindowSpec(99, 1, 1, 1, 1, 1)
    assert lib.abr_env_step_policy_window(None, None, 1, 7, bad, *[None] * 10) == 1
    assert b"env is NULL" in lib.abr_last_error()
    assert lib.abr_env_observe_window(None, None, None, None) == 1
    assert b"env is NULL" in lib.abr_last_error()


def test_the_build_tracks_the_header():
    from abrsimulator_b200 import _build
    assert any(h.endswith("abr_b200_obs.h") for h in _build.HEADERS)
