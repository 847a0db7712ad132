"""Oracle of the clairvoyant lookahead (SPEC §4.4) — TEST INFRASTRUCTURE.  Two restatements:

* ``decide(env, H)`` on the C environment oracle (``oracle/abr_oracle.c``): for every session, A^h copies of its state
  (every field the oracle exposes, the K ring slots included) in a fresh oracle environment, one per sequence in C
  order, run through the oracle's FIXED episode for h steps; the episode's reward sum (left to right from +0) is J.
  The original environment is only read.
* ``lookahead(sess, H)`` on the pure-Python ``oracle/step_oracle.Session``: ``copy.deepcopy`` per sequence.
"""
from __future__ import annotations

import copy
import ctypes as C
import itertools

import numpy as np

from oracle import oracle as orc

# the state fields of orc_env_field: (id, dtype, per-session width; 0 = the ring capacity K)
_FIELDS = dict(seg=(0, np.int32, 1), chunk=(1, np.int32, 1), last_q=(2, np.int32, 1), trace_id=(3, np.int32, 1),
               hist_len=(4, np.int32, 1), done=(5, np.uint8, 1), err_len=(6, np.int32, 1), started=(7, np.uint8, 1),
               play_id=(8, np.int32, 1), phase=(10, np.float64, 1), buffer=(11, np.float64, 1),
               bw_hist=(12, np.float64, 0), last_pred=(13, np.float64, 1), err_ring=(14, np.float64, 0),
               t_now=(16, np.float64, 1), play_time=(17, np.float64, 1), pos=(18, np.float64, 1),
               play_len=(19, np.float64, 1))
_BATCH = 1 << 19     # session copies per oracle environment


def _params(env):
    return {name: getattr(env.params, name) for name, _ in orc.OrcParams._fields_}


def _put(env, name, values):
    fid, dt, _ = _FIELDS[name]
    a = np.ascontiguousarray(values, dtype=dt)
    C.memmove(orc.lib().orc_env_field(env._h, C.c_int(fid)), a.ctypes.data, a.nbytes)


def _sums(env, state, idx, h):
    """J[len(idx)][A^h] of the sessions idx, and whether an oracle step hit the safety net."""
    A = env.A
    M = A ** h
    seqs = np.array(list(itertools.product(range(A), repeat=h)), np.int32)    # C order, a_0 slowest
    clone = orc.OracleEnv(env.trace_bw, env.trace_len, env.trace_interval, env.sizes, env.bitrates, len(idx) * M,
                          **_params(env))
    for name, v in state.items():
        _put(clone, name, np.repeat(v[idx], M, axis=0))
    acts = np.ascontiguousarray(np.tile(seqs, (len(idx), 1)).T)                 # [h][sessions * M]
    J = clone.rollout(orc.POLICY_FIXED, h, actions=acts, want_traj=False)["acc"][0].reshape(len(idx), M)
    return J, clone.errors() > 0


def decide(env, H, want_seq=False):
    """(action, best_value[, best_seq]) of SPEC §4.4 for every session of the oracle environment ``env``, and the
    number of sessions whose lookahead steps hit the safety net of §3.1 (what the decision adds to the error count)."""
    N, A, V = env.N, env.A, env.V
    state = {name: env.field(name) for name in _FIELDS}
    h_of = np.where(state["done"] != 0, 0, np.minimum(H, V - state["chunk"]))
    act = np.zeros(N, np.int32)
    val = np.zeros(N)
    seq = np.full((N, H), -1, np.int32)
    flagged = 0
    for h in range(1, H + 1):
        sel = np.flatnonzero(h_of == h)
        step = max(1, _BATCH // A ** h)
        for b in range(0, len(sel), step):
            idx = sel[b:b + step]
            J, hit = _sums(env, state, idx, h)
            if hit:          # attribute the safety net to sessions: one at a time
                flagged += sum(_sums(env, state, idx[k:k + 1], h)[1] for k in range(len(idx)))
            best = np.argmax(J, axis=1)                                     # the first maximum
            val[idx] = J[np.arange(len(idx)), best]
            digits = np.array(list(itertools.product(range(A), repeat=h)), np.int32)[best]
            seq[idx, :h] = digits
            act[idx] = digits[:, 0]
    return (act, val, seq, flagged) if want_seq else (act, val, flagged)


def _clone(sess):
    """A deep copy of the session's state; the read-only tables (trace, capacity table, ladders) are shared."""
    memo = {id(x): x for x in (sess.bw, sess.rate, sess.C, sess.sizes, sess.util, sess.P)}
    return copy.deepcopy(sess, memo)


def lookahead(sess, H):
    """(action, best_value, best_seq) of SPEC §4.4 for one ``step_oracle.Session``; ``sess`` is left as it is."""
    h = 0 if sess.done else min(H, sess.V - sess.chunk)
    if h == 0:
        return 0, 0.0, [-1] * H
    best, best_R = 0.0, None
    for R in itertools.product(range(sess.A), repeat=h):   # C order, a_0 slowest
        s = _clone(sess)
        J = 0.0
        for q in R:
            J = J + s.step(q)["reward"]
        if best_R is None or J > best:
            best, best_R = J, R
    return best_R[0], best, list(best_R) + [-1] * (H - h)
