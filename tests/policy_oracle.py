"""Oracle of the RATE and BOLA policies (SPEC §4.2, §4.3) — TEST INFRASTRUCTURE.

Two restatements of the rules: ``tests/policy_oracle.c`` (scalar C, no FMA contraction, compiled here into a temporary
directory) and the pure-Python functions ``rb_action`` / ``bola_table`` / ``bola_action``.  ``PolicyEnv`` runs the
policies on the environment oracle (``oracle/abr_oracle.c``): each fused-episode step is the policy's decision on the
oracle's state followed by the oracle's own step, which is what SPEC §3+§4 define an episode to be.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import math
import os
import subprocess
import tempfile

import numpy as np

from oracle import oracle as orc

POLICY_BBA, POLICY_RATE, POLICY_BOLA = 2, 3, 4
DEFAULTS = dict(rb_safety=1.0, bola_min_buffer=10.0, bola_target_buffer=30.0)
_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "policy_oracle.c")
_lib = None


def lib():
    """The compiled C restatement (built once per source version, outside the repository tree)."""
    global _lib
    if _lib is None:
        src = open(_SRC, "rb").read()
        d = os.path.join(tempfile.gettempdir(), f"abr_policy_oracle_{os.getuid()}")
        os.makedirs(d, exist_ok=True)
        so = os.path.join(d, f"libpolicy_oracle_{hashlib.sha256(src).hexdigest()[:16]}.so")
        if not os.path.exists(so):
            tmp = f"{so}.{os.getpid()}"
            subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC", "-o", tmp,
                                   _SRC, "-lm"])
            os.replace(tmp, so)
        _lib = C.CDLL(so)
        _lib.pol_params_invalid.argtypes = [C.c_double] * 3
    return _lib


def params_invalid(**pp):
    p = dict(DEFAULTS, **pp)
    return bool(lib().pol_params_invalid(p["rb_safety"], p["bola_min_buffer"], p["bola_target_buffer"]))


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def policy_decide(policy, sizes, chunk, buffer, bw_hist, hist_len, done=None, default_quality=1, chunk_length=4.0,
                  bba_reservoir=5.0, bba_cushion=10.0, **pp):
    """The C rules on caller-given states: bw_hist [N][K] rings (newest sample at slot (hist_len - 1) mod K)."""
    p = dict(DEFAULTS, **pp)
    sizes = np.ascontiguousarray(sizes, dtype=np.float64)
    V, A = sizes.shape
    chunk, hist_len = (np.ascontiguousarray(x, dtype=np.int32) for x in (chunk, hist_len))
    buffer, bw_hist = (np.ascontiguousarray(x, dtype=np.float64) for x in (buffer, bw_hist))
    N, K = bw_hist.shape
    d = None if done is None else np.ascontiguousarray(done, dtype=np.uint8)
    act = np.empty(N, np.int32)
    D = C.c_double
    lib().pol_decide(_p(sizes), C.c_int(V), C.c_int(A), C.c_int(default_quality), D(chunk_length), D(bba_reservoir),
                     D(bba_cushion), D(p["rb_safety"]), D(p["bola_min_buffer"]), D(p["bola_target_buffer"]), C.c_int(N),
                     C.c_int(policy), _p(chunk), _p(buffer), _p(d), _p(bw_hist), _p(hist_len), C.c_int(K), _p(act))
    return act


class PolicyEnv(orc.OracleEnv):
    """The environment oracle with the RATE and BOLA policies: ``set_policy_params``, ``policy_decide`` and a
    ``rollout`` that accepts them (the other policies are the environment oracle's own episode)."""

    def __init__(self, *args, **kw):
        super().__init__(*args, **kw)
        self.policy_params = dict(DEFAULTS)

    def set_policy_params(self, **kw):
        """False (and nothing changes) when the values are invalid."""
        if params_invalid(**dict(self.policy_params, **kw)):
            return False
        self.policy_params.update(kw)
        return True

    def policy_decide(self, policy):
        p = self.params
        return policy_decide(policy, self.sizes, self.field("chunk"), self.field("buffer"),
                             self.field("bw_hist").reshape(self.N, self.K), self.field("hist_len"),
                             done=self.field("done"), default_quality=p.default_quality, chunk_length=p.chunk_length,
                             bba_reservoir=p.bba_reservoir, bba_cushion=p.bba_cushion, **self.policy_params)

    def rollout(self, policy, steps, seed=0, session_base=0, actions=None, want_traj=True, speed=None):
        if policy not in (POLICY_RATE, POLICY_BOLA):
            return super().rollout(policy, steps, seed, session_base, actions, want_traj, speed)
        return self.stepwise_rollout(policy, steps, speed)

    def stepwise_rollout(self, policy, steps, speed=None):
        """A fused episode of a state-dependent policy (BBA, RATE, BOLA) as decide + step per chunk."""
        N = self.N
        tr = dict(acc=np.zeros((orc.NUM_ACC, N)))     # the steps add into it left to right, as the episode sums
        keys = ("delay", "sleep", "buffer", "rebuf", "reward", "latency")
        for k in keys:
            tr[k] = np.empty((steps, N))
        tr["eov"] = np.empty((steps, N), np.uint8)
        tr["actions"] = np.empty((steps, N), np.int32)
        for t in range(steps):
            a = self.policy_decide(policy)
            o = self.step(a, want_next_sizes=False, speed=speed, acc=tr["acc"])
            for k in keys:
                tr[k][t] = o[k]
            tr["eov"][t] = o["eov"]
            tr["actions"][t] = a
        return tr


# ---- pure-Python restatement ----
def rb_action(size_row, history, default_quality, chunk_length, rb_safety=1.0):
    """SPEC §4.2: ``history`` = the min(hist_len, K) most recent throughput samples, oldest first."""
    A = len(size_row)
    if len(history) == 0:
        return min(max(default_quality, 0), A - 1)
    S = 0.0
    for x in history:
        S = S + 1.0 / x
    budget = (rb_safety * (len(history) / S)) * chunk_length
    q = 0
    for a in range(A):
        if size_row[a] <= budget:
            q = a
    return q


def bola_table(sizes):
    """SPEC §4.3: v[k][a] = log(sizes[k][a] / sizes[k][0]) and v_max."""
    v = [[math.log(row[a] / row[0]) for a in range(len(row))] for row in sizes]
    return v, max(max(r) for r in v)


def bola_action(size_row, v_row, v_max, buffer, min_buffer=10.0, target_buffer=30.0):
    """SPEC §4.3 on the pre-step buffer: the first quality of the largest (Vp·(v + gp) − buffer) / size."""
    if v_max <= 0.0:
        return 0
    gp = v_max / (target_buffer / min_buffer - 1.0)
    Vp = min_buffer / gp
    q, best = 0, 0.0
    for a in range(len(size_row)):
        sc = (Vp * (v_row[a] + gp) - buffer) / size_row[a]
        if a == 0 or sc > best:
            q, best = a, sc
    return q
