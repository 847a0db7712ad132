"""CPU-only: include/abr_b200_mpc_scen.h against the ctypes table _lib.MPC_SCEN_SIGNATURES, the check of
abr_env_mpc_decide_scen (SPEC §5.7) that needs no device, and the ledger that the GPU case table of
test_gpu_mpc_scen.py reaches every compiled form and path of the scenario MPC kernel."""
import os
import re

from abrsimulator_b200 import _lib
from test_capi_signatures import ROOT, c_kind, ctypes_kind
import mpc_scen_oracle as ms


def header_text():
    with open(os.path.join(ROOT, "include", "abr_b200_mpc_scen.h")) as f:
        return f.read()


def header_declarations():
    """[(name, return type, [parameter types])] of the abr_* functions of the companion header, in order."""
    text = re.sub(r"/\*.*?\*/", " ", header_text(), flags=re.S)
    text = "\n".join(line for line in text.splitlines() if not line.lstrip().startswith("#"))
    decls = []
    for ret, name, params in re.findall(r"([A-Za-z_][\w \t\n*]*?)\b(abr_\w+)\s*\(([^()]*)\)\s*;", text):
        types = [re.sub(r"\w+$", "", p.strip()).strip() for p in params.split(",")]
        decls.append((name, ret.split()[-1], types))
    return decls


def test_the_companion_header_matches_its_ctypes_table():
    decls = header_declarations()
    assert [d[0] for d in decls] == list(_lib.MPC_SCEN_SIGNATURES) == ["abr_env_mpc_decide_scen"]
    others = (set(_lib.SIGNATURES) | set(_lib.EXTRA_SIGNATURES) | set(_lib.MPC_PRED_SIGNATURES) |
              set(_lib.OBS_SIGNATURES))
    assert not set(_lib.MPC_SCEN_SIGNATURES) & others
    for name, ret, params in decls:
        restype, argtypes = _lib.MPC_SCEN_SIGNATURES[name]
        assert [ctypes_kind(t) for t in argtypes] == [c_kind(c) for c in params], name
        assert ctypes_kind(restype) == c_kind(ret), name


def test_the_header_constants_match_the_binding():
    defs = dict(re.findall(r"#define\s+(ABR_MPC_SCEN_\w+)\s+(\d+)", header_text()))
    assert {k: int(v) for k, v in defs.items()} == dict(ABR_MPC_SCEN_MEAN=_lib.MPC_SCEN_MEAN,
                                                        ABR_MPC_SCEN_WORST=_lib.MPC_SCEN_WORST,
                                                        ABR_MPC_SCEN_MAX=_lib.MPC_SCEN_MAX)
    assert (ms.MEAN, ms.WORST, ms.K_MAX_SCEN) == (_lib.MPC_SCEN_MEAN, _lib.MPC_SCEN_WORST, _lib.MPC_SCEN_MAX)


def test_the_loaded_library_carries_the_table():
    lib = _lib.load()
    for name, (restype, argtypes) in _lib.MPC_SCEN_SIGNATURES.items():
        fn = getattr(lib, name)
        assert fn.restype is restype and list(fn.argtypes) == argtypes, name


def test_a_null_env_is_reported_before_anything_else():
    lib = _lib.load()
    assert lib.abr_env_mpc_decide_scen(None, 99, 77, 5, 3, None, None, None, None, None, None) == 1
    assert b"env is NULL" in lib.abr_last_error()


def test_the_build_tracks_the_header():
    from abrsimulator_b200 import _build
    assert any(h.endswith("abr_b200_mpc_scen.h") for h in _build.HEADERS)


def test_the_restated_dispatch_matches_the_source():
    """The constants and expressions scen_form restates, as abr_mpc_scen.cu spells them."""
    with open(os.path.join(ROOT, "abrsimulator_b200", "csrc", "abr_mpc_scen.cu")) as f:
        src = f.read()
    launcher = src[src.index("cudaError_t launch_mpc_scen("):]
    launcher = launcher[:launcher.index("\n}\n")]
    assert "const int wps = (a.N >= (long long)sms * 16 || combos < 32 * 36 * 4) ? 1 : kScenWarpsPerBlock;" in launcher
    assert "if (blocks > (long long)sms * 64) blocks = (long long)sms * 64;" in launcher
    assert ("const bool prune = !(a.flags & ABR_MPC_EXHAUSTIVE) && a.p.smooth_penalty >= 0.0 && "
            "a.p.rebuf_penalty >= 0.0;") in launcher
    assert re.findall(r"case (\d+): e = run_mpc_scen_wps<\1>", launcher) == [str(a) for a in ms.COMPILED_A]
    assert "default: e = run_mpc_scen_wps<0>" in launcher
    assert "constexpr int kScenWarpsPerBlock = 4;" in src
    search = src[src.index("__device__ __forceinline__ SearchOut scen_search("):]
    assert "const int P = h >= 2 ? h - 2 : 0;" in search and "if (h == 1) {" in search


def test_the_gpu_cases_reach_every_form_of_the_scenario_kernel():
    want = ms.reachable_scen_cells()
    got = set().union(*(c.cells() for c in ms.SCEN_CASES))
    assert not want - got, sorted(want - got)
    # every compiled ladder size and both session layouts, both objectives, pruned and exhaustive (A = 2 never gets
    # a block per session: 2^8 sequences are fewer than the threshold)
    assert {(c[0], c[1], c[3], c[4]) for c in want} == {(w, at, o, m) for w in (1, 4) for at in (0, 2, 3, 4, 5, 6, 8)
                                                        for o in (ms.MEAN, ms.WORST) for m in ("prune", "enum")
                                                        if (w, at) != (4, 2)}
    assert {c[2] for c in got} == set(ms.PATHS)
    assert any(c.N > 4 * 64 * ms.B200_SMS for c in ms.SCEN_CASES)     # a block slot serves several sessions


def test_removing_a_sole_case_breaks_the_ledger():
    want = ms.reachable_scen_cells()
    for i, c in enumerate(ms.SCEN_CASES):
        rest = set().union(*(d.cells() for j, d in enumerate(ms.SCEN_CASES) if j != i))
        if c.cells() - rest:
            assert want - rest
            return
    raise AssertionError("no case is the only one to reach a cell")


def test_ties_and_zero_penalties_reach_both_layouts_and_objectives():
    """Cases in the tie worlds (exact ties between a sequence and its twin-rung copy, in another prefix and among one
    thread's leaves) and with smooth_penalty = 0 or rebuf_penalty = 0 under branch and bound; every case also runs
    exhaustively on the device.  The GPU test asserts that the ties are there."""
    ties = {(c.cells().pop()[0], c.objective) for c in ms.SCEN_CASES if c.ties}
    assert ties == {(w, o) for w in (1, 4) for o in (ms.MEAN, ms.WORST)}
    assert all(not c.flags and c.vw >= 0 and c.rw >= 0 for c in ms.SCEN_CASES if c.ties)
    for zero in ("vw", "rw"):
        got = {(c.cells().pop()[0], c.objective) for c in ms.SCEN_CASES
               if getattr(c, zero) == 0.0 and not c.flags and c.vw >= 0}
        assert got == {(w, o) for w in (1, 4) for o in (ms.MEAN, ms.WORST)}, zero
