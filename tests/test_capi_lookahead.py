"""CPU-only: include/abr_b200_lookahead.h against the ctypes table _lib.EXTRA_SIGNATURES, and the checks of
abr_env_lookahead_decide (SPEC §4.4) that need no device."""
import os
import re

from abrsimulator_b200 import _lib
from test_capi_signatures import ROOT, c_kind, ctypes_kind


def lookahead_header_declarations():
    """[(name, return type, [parameter types])] of the abr_* functions of the companion header, in order."""
    with open(os.path.join(ROOT, "include", "abr_b200_lookahead.h")) as f:
        text = re.sub(r"/\*.*?\*/", " ", f.read(), flags=re.S)
    text = "\n".join(line for line in text.splitlines() if not line.lstrip().startswith("#"))
    decls = []
    for ret, name, params in re.findall(r"([A-Za-z_][\w \t\n*]*?)\b(abr_\w+)\s*\(([^()]*)\)\s*;", text):
        types = [re.sub(r"\w+$", "", p.strip()).strip() for p in params.split(",")]
        decls.append((name, ret.split()[-1], types))
    return decls


def test_the_companion_header_matches_its_ctypes_table():
    decls = lookahead_header_declarations()
    assert [d[0] for d in decls] == list(_lib.EXTRA_SIGNATURES) == ["abr_env_lookahead_decide"]
    assert not set(_lib.EXTRA_SIGNATURES) & set(_lib.SIGNATURES)
    for name, ret, params in decls:
        restype, argtypes = _lib.EXTRA_SIGNATURES[name]
        assert [ctypes_kind(t) for t in argtypes] == [c_kind(c) for c in params], name
        assert ctypes_kind(restype) == c_kind(ret), name


def test_the_loaded_library_carries_the_companion_table():
    lib = _lib.load()
    for name, (restype, argtypes) in _lib.EXTRA_SIGNATURES.items():
        fn = getattr(lib, name)
        assert fn.restype is restype and list(fn.argtypes) == argtypes, name


def test_a_null_env_is_reported_before_anything_else():
    lib = _lib.load()
    assert lib.abr_env_lookahead_decide(None, 99, None, None, None, None) == 1
    assert b"env is NULL" in lib.abr_last_error()
