"""Oracle of the catch-up speed control of live mode (SPEC §7.2) — TEST INFRASTRUCTURE.

Two restatements: ``tests/speed_oracle.c`` (the environment oracle ``oracle/abr_oracle.c`` included as it is, with the
controller's decision where a speed is read; no FMA contraction, compiled here into a temporary directory) and the
pure-Python ``SpeedSession`` on top of ``oracle/step_oracle.py``'s ``Session`` playback model.  ``SpeedEnv`` runs the
C restatement on the state of a ``dynamic_oracle.DynamicEnv``, so that every built-in policy has an episode under the
controller: FIXED, RANDOM and BBA as the C episode, RATE, BOLA and DYNAMIC as decide + step per chunk.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import dynamic_oracle as do
from oracle import oracle as orc
from oracle import step_oracle as so

NAMES = ("target_latency", "max_drift", "gain", "dead_band", "min_buffer")
DEFAULTS = dict(target_latency=12.0, max_drift=0.5, gain=2.5, dead_band=0.02, min_buffer=6.0)
_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "speed_oracle.c")
_lib = None


def lib():
    """The compiled C restatement (built once per version of both sources, outside the repository tree)."""
    global _lib
    if _lib is None:
        h = hashlib.sha256()
        for f in (_SRC, os.path.join(_HERE, "..", "oracle", "abr_oracle.c"), os.path.join(_HERE, "..", "oracle", "abr_oracle.h")):
            h.update(open(f, "rb").read())
        d = os.path.join(tempfile.gettempdir(), f"abr_speed_oracle_{os.getuid()}")
        os.makedirs(d, exist_ok=True)
        so_path = os.path.join(d, f"libspeed_oracle_{h.hexdigest()[:16]}.so")
        if not os.path.exists(so_path):
            tmp = f"{so_path}.{os.getpid()}"
            subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC", "-o", tmp,
                                   _SRC, "-lm"])
            os.replace(tmp, so_path)
        _lib = C.CDLL(so_path)
        _lib.spd_create.restype = C.c_void_p
        _lib.spd_create.argtypes = [C.c_int]
        _lib.spd_destroy.argtypes = [C.c_void_p]
        _lib.spd_set.argtypes = [C.c_void_p, C.c_void_p]
        _lib.spd_set_log.argtypes = [C.c_void_p, C.c_void_p]
        _lib.spd_play_speed.restype = C.c_void_p
        _lib.spd_counts.restype = C.c_void_p
        _lib.spd_counts.argtypes = [C.c_void_p]
        _lib.spd_play_speed.argtypes = [C.c_void_p]
        _lib.spd_params_invalid.argtypes = [C.c_void_p]
        _lib.spd_rule.restype = C.c_double
        _lib.spd_rule.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_double]
    return _lib


def _vec(params):
    p = dict(DEFAULTS, **params)
    return np.array([float(p[k]) for k in NAMES])


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def params_invalid(**params):
    return bool(lib().spd_params_invalid(_p(_vec(params))))


def rule_c(tc, play_time, buffer, **params):
    """The C rule: the speed of a chunk that starts to play at wall clock tc with play_time played and the buffer."""
    return lib().spd_rule(_p(_vec(params)), tc, play_time, buffer)


# ---- pure-Python restatement ----
def rule(tc, play_time, buffer, target_latency=12.0, max_drift=0.5, gain=2.5, dead_band=0.02, min_buffer=6.0):
    """SPEC §7.2, in its order of operations."""
    e = (tc - play_time) - target_latency
    if abs(e) <= dead_band:
        v = 1.0
    else:
        y = gain * e
        v = 1.0 + max_drift * (y / (1.0 + abs(y)))
    if v > 1.0 and buffer < min_buffer:
        v = 1.0
    return v


class SpeedSession(so.Session):
    """``Session`` with the controller: ``control`` (a dict of the five parameters, or None for the table / 1.0) and
    ``play_speed`` (the stored decision, 0 at creation).  The playback model calls ``_speed_of`` at the top of every
    loop iteration of play_wall / play_content; the controller decides there when chunk play_id has not played yet."""

    def __init__(self, *args, **kw):
        super().__init__(*args, **kw)
        self.control = None
        self.play_speed = 0.0
        self.decisions = []
        self._acc = None

    def _play_wall(self, dt, acc):
        self._acc = acc
        return super()._play_wall(dt, acc)

    def _play_content(self, x, acc):
        self._acc = acc
        return super()._play_content(x, acc)

    def _speed_of(self, k):
        if self.control is None:
            return super()._speed_of(k)
        if self.play_len == 0.0 or not (self.play_speed > 0.0):
            self.play_speed = rule(self._acc["tc"], self.play_time, self.buffer, **self.control)
            self.decisions.append(self.play_speed)
        return self.play_speed


class SpeedEnv(do.DynamicEnv):
    """The environment oracle under the controller of SPEC §7.2 (``set_speed_control``), with every built-in policy.
    ``play_speed`` is the per-session decision; ``log`` ([V, N], or None) receives every decision at
    [min(play_id, V - 1), s]."""

    def __init__(self, *args, **kw):
        super().__init__(*args, **kw)
        self._c = C.c_void_p(lib().spd_create(self.N))
        self.log = None

    def __del__(self):
        try:
            if self._c:
                lib().spd_destroy(self._c)
                self._c = None
        except Exception:
            pass
        super().__del__()

    def set_speed_control(self, params=(), **kw):
        """``set_speed_control(**params)`` installs (defaults for omitted fields), ``set_speed_control(None)`` removes."""
        self._params = None if params is None else _vec(kw)
        lib().spd_set(self._c, _p(self._params))

    def start_log(self, fill=1.0):
        self.log = np.full((self.V, self.N), fill)
        lib().spd_set_log(self._c, _p(self.log))
        return self.log

    def counts(self):
        """(decisions above 1, below 1, held at 1 by the buffer guard) since the environment was created."""
        ptr = lib().spd_counts(self._c)
        return tuple(int(x) for x in np.frombuffer((C.c_int64 * 3).from_address(ptr), dtype=np.int64))

    @property
    def play_speed(self):
        ptr = lib().spd_play_speed(self._c)
        return np.frombuffer((C.c_double * self.N).from_address(ptr), dtype=np.float64).copy()

    def step(self, action, want_next_sizes=True, speed=None, acc=None):
        N, A = self.N, self.A
        a = np.ascontiguousarray(action, dtype=np.int32)
        v = None if speed is None else np.ascontiguousarray(speed, dtype=np.float64)
        out = dict(delay=np.empty(N), sleep=np.empty(N), buffer=np.empty(N), rebuf=np.empty(N),
                   reward=np.empty(N), latency=np.empty(N), eov=np.empty(N, np.uint8), throughput=np.empty(N),
                   next_sizes=np.empty((N, A)) if want_next_sizes else None)
        lib().spd_env_step_live(self._h, self._c, _p(a), _p(v), _p(out["delay"]), _p(out["sleep"]), _p(out["buffer"]),
                                _p(out["rebuf"]), _p(out["reward"]), _p(out["latency"]), _p(out["next_sizes"]),
                                _p(out["eov"]), _p(out["throughput"]), _p(acc))
        return out

    def rollout(self, policy, steps, seed=0, session_base=0, actions=None, want_traj=True, speed=None):
        if policy not in (orc.POLICY_FIXED, orc.POLICY_RANDOM, orc.POLICY_BBA):
            return self.stepwise_rollout(policy, steps, speed)
        N = self.N
        a_in = None if actions is None else np.ascontiguousarray(actions, dtype=np.int32)
        v = None if speed is None else np.ascontiguousarray(speed, dtype=np.float64)
        tr = dict(acc=np.empty((orc.NUM_ACC, N)))
        if want_traj:
            for k in ("delay", "sleep", "buffer", "rebuf", "reward", "latency"):
                tr[k] = np.empty((steps, N))
            tr["eov"] = np.empty((steps, N), np.uint8)
            tr["actions"] = np.empty((steps, N), np.int32)
        lib().spd_env_rollout_live(self._h, self._c, C.c_int(policy), C.c_uint64(seed), C.c_int64(session_base),
                                   C.c_int(steps), _p(a_in), _p(v), _p(tr.get("delay")), _p(tr.get("sleep")),
                                   _p(tr.get("buffer")), _p(tr.get("rebuf")), _p(tr.get("reward")),
                                   _p(tr.get("latency")), _p(tr.get("eov")), _p(tr.get("actions")), _p(tr["acc"]))
        return tr

