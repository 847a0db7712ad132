"""Oracle of per-session policy parameters (SPEC §4.7) — TEST INFRASTRUCTURE.

Two restatements: ``tests/session_params_oracle.c`` (scalar C on top of ``tests/dynamic_oracle.c`` and
``tests/policy_oracle.c``, included unchanged, compiled here into a temporary directory) and the pure-Python
``session_action`` on top of ``policy_oracle`` / ``dynamic_oracle``.  ``SessionParamsEnv`` keeps a [7][N] table of
knobs next to the environment oracle, keyed by the caller's index of each session, and runs the built-in policies'
episodes as a decision plus the oracle's own step per chunk.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import dynamic_oracle as do
import policy_oracle as po

FIELDS = ("bba_reservoir", "bba_cushion", "rb_safety", "bola_min_buffer", "bola_target_buffer", "switch_on_buffer",
          "switch_off_buffer")
BUILTIN = (po.POLICY_BBA, po.POLICY_RATE, po.POLICY_BOLA, do.POLICY_DYNAMIC)
_HERE = os.path.dirname(os.path.abspath(__file__))
_SRCS = [os.path.join(_HERE, f) for f in ("session_params_oracle.c", "dynamic_oracle.c", "policy_oracle.c")]
_lib = None


def lib():
    """The compiled C restatement (built once per version of the sources, outside the repository tree)."""
    global _lib
    if _lib is None:
        h = hashlib.sha256()
        for f in _SRCS:
            h.update(open(f, "rb").read())
        d = os.path.join(tempfile.gettempdir(), f"abr_session_params_oracle_{os.getuid()}")
        os.makedirs(d, exist_ok=True)
        so = os.path.join(d, f"libsession_params_oracle_{h.hexdigest()[:16]}.so")
        if not os.path.exists(so):
            tmp = f"{so}.{os.getpid()}"
            subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC", "-o", tmp,
                                   _SRCS[0], "-lm"])
            os.replace(tmp, so)
        _lib = C.CDLL(so)
        _lib.sp_first_invalid.argtypes = [C.c_void_p, C.c_int, C.c_int]
        _lib.sp_bola_derive.argtypes = [C.c_double, C.c_double, C.c_double, C.c_void_p, C.c_void_p]
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def env_wide(params, policy_params=None, dynamic_params=None):
    """The seven environment-wide values in field order (AbrParams' bba_*, then the setters' current values)."""
    pp = dict(po.DEFAULTS, **(policy_params or {}))
    dp = dict(do.DEFAULTS, **(dynamic_params or {}))
    return [float(params.bba_reservoir), float(params.bba_cushion), pp["rb_safety"], pp["bola_min_buffer"],
            pp["bola_target_buffer"], dp["switch_on_buffer"], dp["switch_off_buffer"]]


def fill(n, wide, **fields):
    """[7][n] table: the given arrays, the environment-wide value for the others."""
    x = np.empty((7, n))
    for f, name in enumerate(FIELDS):
        x[f] = np.asarray(fields[name], np.float64) if name in fields else wide[f]
    return x


def first_invalid(x):
    """(session, field) of the smallest failing session and its first failing field, or None (C restatement)."""
    x = np.ascontiguousarray(x, np.float64)
    n = x.shape[1]
    for s in range(n):
        f = lib().sp_first_invalid(_p(x), n, s)
        if f >= 0:
            return s, f
    return None


def first_invalid_py(x):
    """Pure-Python restatement of first_invalid."""
    fin = np.isfinite
    for s in range(x.shape[1]):
        r, c, rb, mn, tg, on, off = x[:, s]
        checks = (fin(r), fin(c) and c > 0, fin(rb) and rb > 0, fin(mn) and mn > 0, fin(tg) and mn < tg, fin(on),
                  fin(off) and off >= 0 and off < on)
        for f, ok in enumerate(checks):
            if not ok:
                return s, f
    return None


def bola_derive(vmax, mn, tg):
    Vp, gp = C.c_double(), C.c_double()
    lib().sp_bola_derive(vmax, mn, tg, C.byref(Vp), C.byref(gp))
    return Vp.value, gp.value


def sp_decide(policy, sizes, x, chunk, buffer, bw_hist, hist_len, mode, done=None, default_quality=1,
              chunk_length=4.0):
    """The C rule for N sessions with knobs x [7][N]; returns (actions, new modes)."""
    sizes = np.ascontiguousarray(sizes, np.float64)
    V, A = sizes.shape
    x = np.ascontiguousarray(x, np.float64)
    chunk, hist_len = (np.ascontiguousarray(a, np.int32) for a in (chunk, hist_len))
    buffer, bw_hist = (np.ascontiguousarray(a, np.float64) for a in (buffer, bw_hist))
    m = np.array(mode, np.uint8, copy=True)
    N, K = bw_hist.shape
    d = None if done is None else np.ascontiguousarray(done, np.uint8)
    act = np.empty(N, np.int32)
    D = C.c_double
    lib().sp_decide(_p(sizes), C.c_int(V), C.c_int(A), C.c_int(default_quality), D(chunk_length), _p(x), C.c_int(N),
                    C.c_int(policy), _p(chunk), _p(buffer), _p(d), _p(bw_hist), _p(hist_len), C.c_int(K), _p(m),
                    _p(act))
    return act, m


def session_action(policy, size_row, v_row, v_max, history, buffer, chunk, prev_mode, default_quality, chunk_length,
                   knobs):
    """(action, mode) of one session that is not done, knobs = its seven values (pure Python)."""
    r, c, rb, mn, tg, on, off = knobs
    if policy == po.POLICY_BBA:
        A = len(size_row)
        if buffer < r:
            return 0, prev_mode
        if buffer >= r + c:
            return A - 1, prev_mode
        return min(int(np.floor(((A - 1) * (buffer - r)) / c)), A - 1), prev_mode
    if policy == do.POLICY_DYNAMIC:
        return do.dynamic_action(size_row, v_row, v_max, history, buffer, chunk, prev_mode, default_quality,
                                 chunk_length, on, off, rb, mn, tg)
    if policy == po.POLICY_RATE:
        return po.rb_action(size_row, history, default_quality, chunk_length, rb), prev_mode
    return po.bola_action(size_row, v_row, v_max, buffer, mn, tg), prev_mode


class SessionParamsEnv(do.DynamicEnv):
    """``DynamicEnv`` with per-session knobs: ``set_session_params`` installs a [7][N] table in caller order (``perm``
    maps environment positions to caller indices when the sessions are kept in another order)."""

    def __init__(self, *args, **kw):
        super().__init__(*args, **kw)
        self.knobs = None
        self.perm = None

    def set_session_params(self, **fields):
        x = fill(self.N, env_wide(self.params, self.policy_params, self.dynamic_params), **fields)
        if first_invalid(x) is not None:
            return False
        self.knobs = x
        return True

    def policy_decide(self, policy):
        if self.knobs is None or policy not in BUILTIN:
            return super().policy_decide(policy)
        p = self.params
        x = self.knobs if self.perm is None else self.knobs[:, self.perm]
        act, self.dyn_mode = sp_decide(policy, self.sizes, x, self.field("chunk"), self.field("buffer"),
                                       self.field("bw_hist").reshape(self.N, self.K), self.field("hist_len"),
                                       self.dyn_mode, done=self.field("done"), default_quality=p.default_quality,
                                       chunk_length=p.chunk_length)
        if policy == do.POLICY_DYNAMIC:
            self.decisions.append((self.field("chunk"), self.field("done"), self.dyn_mode.copy()))
        return act

    def rollout(self, policy, steps, seed=0, session_base=0, actions=None, want_traj=True, speed=None):
        if self.knobs is None or policy not in BUILTIN:
            return super().rollout(policy, steps, seed, session_base, actions, want_traj, speed)
        return self.stepwise_rollout(policy, steps, speed)
