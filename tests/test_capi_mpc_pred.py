"""CPU-only: include/abr_b200_mpc_pred.h against the ctypes table _lib.MPC_PRED_SIGNATURES, the check of
abr_env_mpc_decide_pred (SPEC §5.6) that needs no device, and the ledger that the GPU case table of
test_gpu_mpc_pred.py reaches every compiled form of the caller-prediction MPC kernels."""
import os
import re

from abrsimulator_b200 import _lib
from test_capi_signatures import ROOT, c_kind, ctypes_kind
import search_forms as sf
from mpc_pred_oracle import PRED_CASES


def header_declarations():
    """[(name, return type, [parameter types])] of the abr_* functions of the companion header, in order."""
    with open(os.path.join(ROOT, "include", "abr_b200_mpc_pred.h")) as f:
        text = re.sub(r"/\*.*?\*/", " ", f.read(), flags=re.S)
    text = "\n".join(line for line in text.splitlines() if not line.lstrip().startswith("#"))
    decls = []
    for ret, name, params in re.findall(r"([A-Za-z_][\w \t\n*]*?)\b(abr_\w+)\s*\(([^()]*)\)\s*;", text):
        types = [re.sub(r"\w+$", "", p.strip()).strip() for p in params.split(",")]
        decls.append((name, ret.split()[-1], types))
    return decls


def test_the_companion_header_matches_its_ctypes_table():
    decls = header_declarations()
    assert [d[0] for d in decls] == list(_lib.MPC_PRED_SIGNATURES) == ["abr_env_mpc_decide_pred"]
    assert not set(_lib.MPC_PRED_SIGNATURES) & (set(_lib.SIGNATURES) | set(_lib.EXTRA_SIGNATURES))
    for name, ret, params in decls:
        restype, argtypes = _lib.MPC_PRED_SIGNATURES[name]
        assert [ctypes_kind(t) for t in argtypes] == [c_kind(c) for c in params], name
        assert ctypes_kind(restype) == c_kind(ret), name


def test_the_loaded_library_carries_the_table():
    lib = _lib.load()
    for name, (restype, argtypes) in _lib.MPC_PRED_SIGNATURES.items():
        fn = getattr(lib, name)
        assert fn.restype is restype and list(fn.argtypes) == argtypes, name


def test_a_null_env_is_reported_before_anything_else():
    lib = _lib.load()
    assert lib.abr_env_mpc_decide_pred(None, 99, 77, None, None, None, None, None) == 1
    assert b"env is NULL" in lib.abr_last_error()


def test_the_build_tracks_the_header():
    from abrsimulator_b200 import _build
    assert any(h.endswith("abr_b200_mpc_pred.h") for h in _build.HEADERS)


def reachable_pred_cells(sms=sf.B200_SMS):
    """Every (wps, AT, path, search mode, vw1) cell a legal abr_env_mpc_decide_pred call reaches: mode 1 with flags
    0 or ABR_MPC_EXHAUSTIVE, every h <= H, N on both sides of the warp-per-session threshold."""
    cells = set()
    for A, H in sf.legal_mpc_shapes():
        for N in (1, 16 * sms - 1, 16 * sms):
            for flags in (0, sf.MPC_EXHAUSTIVE):
                for vw, rw in ((1.0, 4.3), (0.6, 4.3), (-0.5, 4.3)):
                    for h in range(1, H + 1):
                        cells.add(sf.mpc_form(A, H, h, N, 1, flags, vw, rw, sms)[0])
    return cells


def case_cells(case, sms=sf.B200_SMS):
    return {sf.mpc_form(case.A, case.H, h, case.N, 1, case.flags, case.vw, case.rw, sms)[0] for h in case.hs}


def test_the_gpu_cases_reach_every_form_of_the_prediction_kernels():
    want = reachable_pred_cells()
    got = set().union(*(case_cells(c) for c in PRED_CASES))
    assert not want - got, sorted(want - got)
    # every compiled ladder size and both session layouts, pruned and exhaustive (A = 2 never gets a block per
    # session: 2^8 sequences are fewer than the threshold)
    assert {(c[0], c[1], c[3]) for c in want} == {(w, at, m) for w in (1, 4) for at in (0, 2, 3, 4, 5, 6, 8)
                                                  for m in ("prune", "enum") if (w, at) != (4, 2)}
    assert {c[2] for c in got} == set(sf.PATHS)


def test_removing_a_sole_case_breaks_the_ledger():
    want = reachable_pred_cells()
    for i, c in enumerate(PRED_CASES):
        rest = set().union(*(case_cells(d) for j, d in enumerate(PRED_CASES) if j != i))
        if case_cells(c) - rest:
            assert want - rest
            return
    raise AssertionError("no case is the only one to reach a cell")
