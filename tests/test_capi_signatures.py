"""CPU-only: the ctypes signature table of abrsimulator_b200._lib against include/abr_b200.h, and that declared
signatures turn wrong arguments into Python errors instead of undefined behaviour."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from abrsimulator_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STRUCTS = ("AbrParams", "AbrPolicyParams", "AbrObsSpec")


def header_declarations():
    """[(name, return type, [parameter types])] of every abr_* function in the header, in order."""
    with open(os.path.join(ROOT, "include", "abr_b200.h")) as f:
        text = f.read()
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    text = re.sub(r"//[^\n]*", " ", text)
    text = "\n".join(line for line in text.splitlines() if not line.lstrip().startswith("#"))
    decls = []
    for ret, name, params in re.findall(r"([A-Za-z_][\w \t\n*]*?)\b(abr_\w+)\s*\(([^()]*)\)\s*;", text):
        ret = " ".join(ret.split()[-2:]) if ret.split()[-2:-1] in (["const"], ["long"]) else ret.split()[-1]
        types = [] if params.strip() in ("", "void") else [re.sub(r"\w+$", "", p.strip()).strip() for p in params.split(",")]
        decls.append((name, ret.replace(" *", "*"), types))
    return decls


def c_kind(t):
    """pointer (with the struct it points to, if any), i32, i64, u64, f64 or void of a C type."""
    t = " ".join(t.replace("*", " * ").split())
    if "*" in t:
        base = t.replace("const", "").replace("*", "").split()
        return ("ptr", base[0] if base and base[0] in STRUCTS and t.count("*") == 1 else None)
    return {"int": "i32", "int32_t": "i32", "long long": "i64", "uint64_t": "u64", "double": "f64", "void": "void"}[t]


def ctypes_kind(t):
    if t is None:
        return "void"
    if issubclass(t, C._Pointer):
        return ("ptr", t._type_.__name__)
    if t in (C.c_void_p, C.c_char_p):
        return ("ptr", None)
    return {C.c_int: "i32", C.c_longlong: "i64", C.c_uint64: "u64", C.c_double: "f64"}[t]


DECLS = header_declarations()


def test_the_header_declares_every_symbol_of_the_table_in_its_order():
    assert len(DECLS) == 37
    assert [d[0] for d in DECLS] == list(_lib.SIGNATURES) == list(_lib.SYMBOLS)


@pytest.mark.parametrize("name, ret, params", DECLS, ids=[d[0] for d in DECLS])
def test_signature_matches_the_header(name, ret, params):
    restype, argtypes = _lib.SIGNATURES[name]
    assert len(argtypes) == len(params), (name, argtypes, params)
    for i, (c, t) in enumerate(zip(params, argtypes)):
        assert ctypes_kind(t) == c_kind(c), (name, i, c, t)
    assert ctypes_kind(restype) == c_kind(ret), (name, ret, restype)


def test_the_loaded_library_carries_the_table():
    lib = _lib.load()
    for name, (restype, argtypes) in _lib.SIGNATURES.items():
        fn = getattr(lib, name)
        assert fn.restype is restype and list(fn.argtypes) == argtypes, name


def test_wrong_arguments_raise_before_the_call():
    lib = _lib.load()
    assert lib.abr_sort_by_trace(None, 0, 1, None, None) == 0          # an empty sort needs no device
    assert lib.abr_sort_by_trace(None, -1, 1, None, None) == 3
    assert b"n_sessions must be >= 0" in lib.abr_last_error()
    with pytest.raises(C.ArgumentError):
        lib.abr_sort_by_trace(None, C.c_longlong(0), 1, None, None)     # a 64-bit value for an int
    with pytest.raises(C.ArgumentError):
        lib.abr_sort_by_trace(None, 0.0, 1, None, None)
    with pytest.raises(C.ArgumentError):
        lib.abr_sort_by_trace(np.zeros(4, np.int32), 0, 1, None, None)  # a buffer instead of its address
    with pytest.raises(TypeError):
        lib.abr_sort_by_trace(None, 0, 1, None)                         # one argument short
    with pytest.raises(C.ArgumentError):
        lib.abr_params_default(_lib.AbrPolicyParams())                  # the wrong struct
    with pytest.raises(C.ArgumentError):
        lib.abr_env_set_policy_params(None, C.c_int(1))
    p = _lib.AbrParams()
    lib.abr_params_default(p)                                           # a struct passes by reference
    assert p.chunk_length == 4.0 and p.hist_k == 5
