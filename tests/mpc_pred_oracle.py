"""Oracle of MPC over caller-supplied throughput predictions (SPEC §5.6) — TEST INFRASTRUCTURE.

Two restatements of the contract: ``tests/mpc_pred_oracle.c`` (scalar C, no FMA contraction, compiled here into a
temporary directory), bound as ``decide_pred_c``, and the pure-Python ``objective_pred`` / ``decide_pred``.  The
objective is SPEC §5.2's (``oracle/mpc_oracle.py`` ``objective_robust``) with the step-i download time divided by the
caller's p_i instead of one robust prediction c.  ``env_decide_pred`` runs the C restatement on the state of an
environment oracle (``oracle/abr_oracle.c``), so that decide + ``OracleEnv.step`` is the reference of an episode.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import itertools
import math
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "mpc_pred_oracle.c")
_lib = None


def lib():
    """The compiled C restatement (built once per source version, outside the repository tree)."""
    global _lib
    if _lib is None:
        src = open(_SRC, "rb").read()
        d = os.path.join(tempfile.gettempdir(), f"abr_mpc_pred_oracle_{os.getuid()}")
        os.makedirs(d, exist_ok=True)
        so = os.path.join(d, f"libmpc_pred_oracle_{hashlib.sha256(src).hexdigest()[:16]}.so")
        if not os.path.exists(so):
            tmp = f"{so}.{os.getpid()}"
            subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC", "-o", tmp,
                                   _SRC, "-lm"])
            os.replace(tmp, so)
        _lib = C.CDLL(so)
        _lib.orc_mpc_decide_pred.restype = C.c_int
        _lib.orc_mpc_decide_pred.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int] + [C.c_double] * 4 + \
            [C.c_int] + [C.c_void_p] * 5 + [C.c_int] + [C.c_void_p] * 3
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data


def decide_pred_c(sizes, util, chunk, prev_q, buffer, pred, H, chunk_length, max_buffer, vw, rw, done=None):
    """orc_mpc_decide_pred over N sessions: dict(action, best_J, best_seq, n_errors)."""
    sizes, util = (np.ascontiguousarray(x, dtype=np.float64) for x in (sizes, util))
    V, A = sizes.shape
    chunk, prev_q = (np.ascontiguousarray(x, dtype=np.int32) for x in (chunk, prev_q))
    buffer = np.ascontiguousarray(buffer, dtype=np.float64)
    pred = np.ascontiguousarray(pred, dtype=np.float64).reshape(len(chunk), H)
    dn = None if done is None else np.ascontiguousarray(done, dtype=np.uint8)
    N = len(chunk)
    act, bj, seq = np.empty(N, np.int32), np.empty(N), np.empty((N, H), np.int32)
    nerr = lib().orc_mpc_decide_pred(_p(sizes), _p(util), V, A, chunk_length, max_buffer, vw, rw, N, _p(chunk),
                                     _p(prev_q), _p(buffer), _p(dn), _p(pred), H, _p(act), _p(bj), _p(seq))
    return dict(action=act, best_J=bj, best_seq=seq, n_errors=nerr)


def env_decide_pred(env, pred, H):
    """decide_pred_c on the state of an ``oracle.OracleEnv`` (done sessions only without auto_reset, as the kernel
    reads them)."""
    p = env.params
    done = None if p.auto_reset else env.field("done")
    return decide_pred_c(env.sizes, util_of(env), env.field("chunk"), env.field("last_q"), env.field("buffer"), pred, H,
                         p.chunk_length, p.max_buffer, p.smooth_penalty, p.rebuf_penalty, done=done)


def util_of(env):
    from oracle import oracle as orc
    return orc.utility_table(env.bitrates, env.params.utility_mode, env.params.utility_scale)


def _max0(x):
    return x if x > 0 else 0.0


def objective_pred(R, k, prev_q, buffer_level, preds, U, sizes, chunk_length, max_buffer, vw, rw):
    """J of SPEC §5.6 for the sequence R: SPEC §5.2's objective with step i's download time sizes / preds[i]."""
    h = len(R)
    seq = [prev_q] + [int(r) for r in R]
    vq = 0.0
    qv = 0.0
    rt = 0.0
    b = buffer_level
    for i in range(h):
        a, ap = seq[i + 1], seq[i]
        vq = vq + U[k + i][a]
        if ap >= 0:
            qv = qv + abs(U[k + i][a] - U[k + i][ap])
        dl = sizes[k + i][a] / preds[i]
        rt = rt + _max0(dl - b)
        if i != h - 1:
            t = _max0(b - dl)
            w = _max0(t + chunk_length - max_buffer)
            b = _max0(t + chunk_length - w)
    return -((vq - vw * qv) - rw * rt)


def decide_pred(k, prev_q, buffer_level, preds, H, U, sizes, chunk_length, max_buffer, vw, rw, done=False):
    """SPEC §5.6 for one session.  Returns dict(action, best_seq, best_J, error): best_seq holds the h chosen
    actions; an input error has action -1."""
    A, V = len(U[0]), len(U)
    if done:
        return dict(action=0, best_seq=[], best_J=math.nan, error=False)
    if k < 0 or prev_q >= A:
        return dict(action=-1, best_seq=[], best_J=math.nan, error=True)
    h = min(H, V - k)
    if h <= 0:
        return dict(action=0, best_seq=[], best_J=math.nan, error=False)
    p = [float(x) for x in preds[:h]]
    if any(not (x > 0) or math.isinf(x) for x in p):
        return dict(action=-1, best_seq=[], best_J=math.nan, error=True)
    best_j, best_seq = None, None
    for R in itertools.product(range(A), repeat=h):
        j = objective_pred(R, k, prev_q, buffer_level, p, U, sizes, chunk_length, max_buffer, vw, rw)
        if best_j is None or j < best_j:
            best_j, best_seq = j, R
    return dict(action=int(best_seq[0]), best_seq=list(best_seq), best_J=best_j, error=False)


# ---- the GPU case table (test_gpu_mpc_pred.py; test_capi_mpc_pred.py proves it reaches every compiled form) ----
MPC_EXHAUSTIVE = 8


class PredCase:
    """abr_env_mpc_decide_pred over the sessions of search_forms.mpc_inputs for the shape (A, H, hs, n, tile), with
    per-step predictions drawn per session, `flags` 0 or ABR_MPC_EXHAUSTIVE, and every other case without auto_reset
    (a tenth of its sessions done)."""

    def __init__(self, A, H, hs, n, tile, flags, vw, auto_reset, rw=4.3):
        self.A, self.H, self.hs, self.n, self.tile = A, H, tuple(hs), n, tile
        self.flags, self.vw, self.rw, self.auto_reset = flags, vw, rw, auto_reset

    @property
    def N(self):
        return self.n * self.tile

    def robust_case(self):
        import search_forms as sf
        return sf.MpcCase(self.A, self.H, "robust", self.vw, self.hs, self.n, tile=self.tile, rw=self.rw)

    @property
    def id(self):
        return (f"A{self.A}H{self.H}-h{'.'.join(map(str, self.hs))}-n{self.n}x{self.tile}-"
                f"{'exh' if self.flags else 'bb'}-vw{self.vw:g}-reset{self.auto_reset}")


def _pred_cases():
    import search_forms as sf
    variants = [(0, 1.0), (0, 0.6), (MPC_EXHAUSTIVE, 1.0), (0, -0.5)]   # prune, prune, enum, enum (negative penalty)
    cases = []
    for i, (A, H, hs, n, tile) in enumerate(sf.SHAPES):
        for j, (flags, vw) in enumerate(variants):
            cases.append(PredCase(A, H, hs, n, tile, flags, vw, auto_reset=(i + j) % 2))
    # a block slot serves several sessions in turn
    cases.append(PredCase(3, 5, (1, 2, 4, 5), 24, 1600, 0, 1.0, auto_reset=0))
    return cases


PRED_CASES = _pred_cases()
