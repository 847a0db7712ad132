"""Oracle of the DYNAMIC policy (SPEC §4.6) — TEST INFRASTRUCTURE.

Two restatements of the rule: ``tests/dynamic_oracle.c`` (scalar C on top of ``tests/policy_oracle.c``'s rate and BOLA
rules, no FMA contraction, compiled here into a temporary directory) and the pure-Python ``dynamic_action`` on top of
``policy_oracle.rb_action`` / ``bola_action``.  ``DynamicEnv`` keeps the per-session mode next to the environment
oracle and runs the policy's episode as a decision plus the oracle's own step per chunk, which is what SPEC §3+§4
define an episode to be.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import policy_oracle as po

POLICY_DYNAMIC = 5
DEFAULTS = dict(switch_on_buffer=12.0, switch_off_buffer=6.0)
_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "dynamic_oracle.c")
_lib = None


def lib():
    """The compiled C restatement (built once per version of both sources, outside the repository tree)."""
    global _lib
    if _lib is None:
        h = hashlib.sha256()
        for f in (_SRC, os.path.join(_HERE, "policy_oracle.c")):
            h.update(open(f, "rb").read())
        d = os.path.join(tempfile.gettempdir(), f"abr_dynamic_oracle_{os.getuid()}")
        os.makedirs(d, exist_ok=True)
        so = os.path.join(d, f"libdynamic_oracle_{h.hexdigest()[:16]}.so")
        if not os.path.exists(so):
            tmp = f"{so}.{os.getpid()}"
            subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC", "-o", tmp,
                                   _SRC, "-lm"])
            os.replace(tmp, so)
        _lib = C.CDLL(so)
        _lib.dyn_params_invalid.argtypes = [C.c_double] * 2
    return _lib


def params_invalid(**dp):
    p = dict(DEFAULTS, **dp)
    return bool(lib().dyn_params_invalid(p["switch_on_buffer"], p["switch_off_buffer"]))


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def dynamic_decide(sizes, chunk, buffer, bw_hist, hist_len, mode, done=None, default_quality=1, chunk_length=4.0,
                   **params):
    """The C rule on caller-given states: bw_hist [N][K] rings (newest sample at slot (hist_len - 1) mod K), mode [N]
    the rule each session's last decision left.  Returns (actions, the new modes); the inputs are not changed."""
    p = dict(po.DEFAULTS, **DEFAULTS)
    p.update(params)
    sizes = np.ascontiguousarray(sizes, dtype=np.float64)
    V, A = sizes.shape
    chunk, hist_len = (np.ascontiguousarray(x, dtype=np.int32) for x in (chunk, hist_len))
    buffer, bw_hist = (np.ascontiguousarray(x, dtype=np.float64) for x in (buffer, bw_hist))
    m = np.array(mode, dtype=np.uint8, copy=True)
    N, K = bw_hist.shape
    d = None if done is None else np.ascontiguousarray(done, dtype=np.uint8)
    act = np.empty(N, np.int32)
    D = C.c_double
    lib().dyn_decide(_p(sizes), C.c_int(V), C.c_int(A), C.c_int(default_quality), D(chunk_length), D(p["rb_safety"]),
                     D(p["bola_min_buffer"]), D(p["bola_target_buffer"]), D(p["switch_on_buffer"]),
                     D(p["switch_off_buffer"]), C.c_int(N), _p(chunk), _p(buffer), _p(d), _p(bw_hist), _p(hist_len),
                     C.c_int(K), _p(m), _p(act))
    return act, m


# ---- pure-Python restatement ----
def dynamic_mode(chunk, buffer, prev_mode, switch_on_buffer=12.0, switch_off_buffer=6.0):
    """SPEC §4.6: the rule of this decision (1 = BOLA, 0 = rate) on the pre-step buffer."""
    prev = 0 if chunk == 0 else prev_mode
    return 1 if buffer > (switch_off_buffer if prev else switch_on_buffer) else 0


def dynamic_action(size_row, v_row, v_max, history, buffer, chunk, prev_mode, default_quality, chunk_length,
                   switch_on_buffer=12.0, switch_off_buffer=6.0, rb_safety=1.0, bola_min_buffer=10.0,
                   bola_target_buffer=30.0):
    """(action, mode) of a session that is not done; ``history`` as for ``policy_oracle.rb_action``."""
    m = dynamic_mode(chunk, buffer, prev_mode, switch_on_buffer, switch_off_buffer)
    if m:
        return po.bola_action(size_row, v_row, v_max, buffer, bola_min_buffer, bola_target_buffer), m
    return po.rb_action(size_row, history, default_quality, chunk_length, rb_safety), m


class DynamicEnv(po.PolicyEnv):
    """``PolicyEnv`` with the DYNAMIC policy: the per-session mode (zero at creation, written only by DYNAMIC
    decisions), ``set_dynamic_params``, and a ``policy_decide`` / ``rollout`` that accept it.  ``decisions`` records
    (chunk, done, mode after the decision) of every DYNAMIC decision, so that a test can see the rule switch."""

    def __init__(self, *args, **kw):
        super().__init__(*args, **kw)
        self.dynamic_params = dict(DEFAULTS)
        self.dyn_mode = np.zeros(self.N, np.uint8)
        self.decisions = []

    def set_dynamic_params(self, **kw):
        """False (and nothing changes) when the values are invalid."""
        if params_invalid(**dict(self.dynamic_params, **kw)):
            return False
        self.dynamic_params.update(kw)
        return True

    def policy_decide(self, policy):
        if policy != POLICY_DYNAMIC:
            return super().policy_decide(policy)
        p = self.params
        chunk, done = self.field("chunk"), self.field("done")
        act, self.dyn_mode = dynamic_decide(
            self.sizes, chunk, self.field("buffer"), self.field("bw_hist").reshape(self.N, self.K),
            self.field("hist_len"), self.dyn_mode, done=done, default_quality=p.default_quality,
            chunk_length=p.chunk_length, **self.policy_params, **self.dynamic_params)
        self.decisions.append((chunk, done, self.dyn_mode.copy()))
        return act

    def switches(self):
        """(rate -> BOLA, BOLA -> rate) switches between consecutive DYNAMIC decisions of a session inside an
        episode (neither decision on a done session, the later one past chunk 0)."""
        if len(self.decisions) < 2:
            return 0, 0
        ch, dn, m = (np.array([d[k] for d in self.decisions]) for k in range(3))
        inside = (dn[:-1] == 0) & (dn[1:] == 0) & (ch[1:] > 0)
        return (int(((m[:-1] == 0) & (m[1:] == 1) & inside).sum()), int(((m[:-1] == 1) & (m[1:] == 0) & inside).sum()))

    def rollout(self, policy, steps, seed=0, session_base=0, actions=None, want_traj=True, speed=None):
        if policy != POLICY_DYNAMIC:
            return super().rollout(policy, steps, seed, session_base, actions, want_traj, speed)
        return self.stepwise_rollout(policy, steps, speed)
