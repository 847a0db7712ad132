"""Oracle of MPC over caller-supplied throughput scenarios (SPEC §5.7) — TEST INFRASTRUCTURE.

Two restatements of the contract: ``tests/mpc_scen_oracle.c`` (scalar C, no FMA contraction, compiled here into a
temporary directory), bound as ``decide_scen_c``, and the pure-Python ``objective_scen`` / ``decide_scen``.  Each
scenario's value is SPEC §5.6's objective for that scenario's prediction row; the aggregate is the weighted mean
(left to right, starting from w_0 q_0) or the minimum.  ``env_decide_scen`` runs the C restatement on the state of an
environment oracle (``oracle/abr_oracle.c``), so that decide + ``OracleEnv.step`` is the reference of an episode.

The second half restates the dispatch of ``abr_mpc_scen_kernel`` (``scen_form``, ``reachable_scen_cells``) and holds
the GPU case table, ``SCEN_CASES``; ``test_capi_mpc_scen.py`` proves that the cases reach every cell.
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

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "mpc_scen_oracle.c")
_lib = None
MEAN, WORST = 0, 1
OBJECTIVES = dict(mean=MEAN, worst=WORST)


def lib():
    """The compiled C restatement (built once per source version, outside the repository tree)."""
    global _lib
    if _lib is None:
        src = open(_SRC, "rb").read()
        d = os.path.join(tempfile.gettempdir(), f"abr_mpc_scen_oracle_{os.getuid()}")
        os.makedirs(d, exist_ok=True)
        so = os.path.join(d, f"libmpc_scen_oracle_{hashlib.sha256(src).hexdigest()[:16]}.so")
        if not os.path.exists(so):
            tmp = f"{so}.{os.getpid()}"
            subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC", "-o", tmp,
                                   _SRC, "-lm"])
            os.replace(tmp, so)
        _lib = C.CDLL(so)
        _lib.orc_mpc_decide_scen.restype = C.c_int
        _lib.orc_mpc_decide_scen.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int] + [C.c_double] * 4 + \
            [C.c_int] + [C.c_void_p] * 6 + [C.c_int] * 3 + [C.c_void_p] * 3
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data


def decide_scen_c(sizes, util, chunk, prev_q, buffer, pred, H, chunk_length, max_buffer, vw, rw, objective=MEAN,
                  weight=None, done=None):
    """orc_mpc_decide_scen over N sessions; pred [N, K, H], weight [N, K] or None: dict(action, best_J, best_seq,
    n_errors)."""
    sizes, util = (np.ascontiguousarray(x, dtype=np.float64) for x in (sizes, util))
    V, A = sizes.shape
    chunk, prev_q = (np.ascontiguousarray(x, dtype=np.int32) for x in (chunk, prev_q))
    buffer = np.ascontiguousarray(buffer, dtype=np.float64)
    N = len(chunk)
    pred = np.ascontiguousarray(pred, dtype=np.float64).reshape(N, -1, H)
    K = pred.shape[1]
    w = None if weight is None else np.ascontiguousarray(weight, dtype=np.float64).reshape(N, K)
    dn = None if done is None else np.ascontiguousarray(done, dtype=np.uint8)
    act, bj, seq = np.empty(N, np.int32), np.empty(N), np.empty((N, H), np.int32)
    nerr = lib().orc_mpc_decide_scen(_p(sizes), _p(util), V, A, chunk_length, max_buffer, vw, rw, N, _p(chunk),
                                     _p(prev_q), _p(buffer), _p(dn), _p(pred), _p(w), K, H, objective, _p(act),
                                     _p(bj), _p(seq))
    return dict(action=act, best_J=bj, best_seq=seq, n_errors=nerr)


def util_of(env):
    from oracle import oracle as orc
    return orc.utility_table(env.bitrates, env.params.utility_mode, env.params.utility_scale)


def env_decide_scen(env, pred, H, objective=MEAN, weight=None):
    """decide_scen_c on the state of an ``oracle.OracleEnv`` (done sessions only without auto_reset, as the kernel
    reads them)."""
    p = env.params
    done = None if p.auto_reset else env.field("done")
    return decide_scen_c(env.sizes, util_of(env), env.field("chunk"), env.field("last_q"), env.field("buffer"), pred,
                         H, p.chunk_length, p.max_buffer, p.smooth_penalty, p.rebuf_penalty, objective, weight, done)


def _max0(x):
    return x if x > 0 else 0.0


def objective_scen(R, k, prev_q, buffer_level, preds, U, sizes, chunk_length, max_buffer, vw, rw, objective=MEAN,
                   weights=None):
    """J of SPEC §5.7 for the sequence R: preds [K][h], weights [K] (MEAN; None: 1/K each)."""
    h, K = len(R), len(preds)
    seq = [prev_q] + [int(r) for r in R]
    Q = None
    for c in range(K):
        vq = qv = rt = 0.0
        b = buffer_level
        for i in range(h):
            a, ap = seq[i + 1], seq[i]
            vq = vq + U[k + i][a]
            if ap >= 0:
                qv = qv + abs(U[k + i][a] - U[k + i][ap])
            dl = sizes[k + i][a] / preds[c][i]
            rt = rt + _max0(dl - b)
            if i != h - 1:
                t = _max0(b - dl)
                w = _max0(t + chunk_length - max_buffer)
                b = _max0(t + chunk_length - w)
        q = (vq - vw * qv) - rw * rt
        if objective == MEAN:
            wc = weights[c] if weights is not None else 1.0 / K
            Q = wc * q if c == 0 else Q + wc * q
        else:
            Q = q if c == 0 or q < Q else Q
    return -Q


def decide_scen(k, prev_q, buffer_level, preds, H, U, sizes, chunk_length, max_buffer, vw, rw, objective=MEAN,
                weights=None, done=False):
    """SPEC §5.7 for one session; preds [K][H].  Returns dict(action, best_seq, best_J, error)."""
    A, V = len(U[0]), len(U)
    if done:
        return dict(action=0, best_seq=[], best_J=math.nan, error=False)
    if k < 0 or prev_q >= A:
        return dict(action=-1, best_seq=[], best_J=math.nan, error=True)
    h = min(H, V - k)
    if h <= 0:
        return dict(action=0, best_seq=[], best_J=math.nan, error=False)
    p = [[float(x) for x in row[:h]] for row in preds]
    bad = any(not (x > 0) or math.isinf(x) for row in p for x in row)
    if objective == MEAN and weights is not None:
        w = [float(x) for x in weights]
        bad = bad or any(not (x >= 0) or math.isinf(x) for x in w) or all(x == 0 for x in w)
    if bad:
        return dict(action=-1, best_seq=[], best_J=math.nan, error=True)
    # the first minimum of J in C order, a NaN J never chosen; none below +inf: sequence 0, best_J = +inf
    best_j, best_seq = math.inf, (0,) * h
    for R in itertools.product(range(A), repeat=h):
        j = objective_scen(R, k, prev_q, buffer_level, p, U, sizes, chunk_length, max_buffer, vw, rw, objective,
                           weights)
        if j < best_j:
            best_j, best_seq = j, R
    return dict(action=int(best_seq[0]), best_seq=list(best_seq), best_J=best_j, error=False)


# ---- the dispatch of abr_mpc_scen_kernel (abr_mpc_scen.cu: launch_mpc_scen, scen_search) ----
MPC_EXHAUSTIVE = 8
B200_SMS = 148
K_MAX_A, K_MAX_H, K_MAX_SCEN = 16, 8, 16
K_MPC_WARPS_PER_BLOCK = 4
WPS_COMBOS = 32 * 36 * 4
COMPILED_A = (2, 3, 4, 5, 6, 8)
PATHS = ("h1", "root", "prefix")   # h == 1; h == 2 (one prefix: the root); h >= 3 (A^(h-2) prefixes)


def scen_form(A, H, h, N, objective, flags, vw, rw, sms=B200_SMS):
    """(cell, stride): cell = (wps, AT, path, objective, search mode "prune" / "enum", smooth_penalty == 1).  Restates
    launch_mpc_scen (`wps`, `blocks` capped at `sms * 64`, `prune`, the `switch (a.A)`) and the path choice of
    scen_search.  The kernel has no specialisation for smooth_penalty == 1 (vw * qv is exact at vw = 1); the axis is
    kept so that both sides are checked."""
    assert 1 <= h <= H <= K_MAX_H and 1 <= A <= K_MAX_A
    wps = 1 if (N >= 16 * sms or A ** H < WPS_COMBOS) else K_MPC_WARPS_PER_BLOCK
    spb = K_MPC_WARPS_PER_BLOCK // wps
    stride = (N + spb - 1) // spb > 64 * sms
    AT = A if A in COMPILED_A else 0
    prune = not (flags & MPC_EXHAUSTIVE) and vw >= 0.0 and rw >= 0.0
    path = PATHS[min(h, 3) - 1]
    return (wps, AT, path, objective, "prune" if prune else "enum", vw == 1.0), stride


def legal_shapes():
    return [(A, H) for A in range(1, K_MAX_A + 1) for H in range(1, K_MAX_H + 1) if A ** H <= 2 ** 31 - 1]


def reachable_scen_cells(sms=B200_SMS):
    """Every cell a legal call reaches: every shape, every h <= H, N on both sides of the warp-per-session threshold,
    both objectives, flags 0 or ABR_MPC_EXHAUSTIVE, both sides of smooth_penalty == 1 and a negative penalty."""
    cells = set()
    for A, H in legal_shapes():
        for N in (1, 16 * sms - 1, 16 * sms):
            for obj in (MEAN, WORST):
                for flags in (0, MPC_EXHAUSTIVE):
                    for vw, rw in ((1.0, 4.3), (0.6, 4.3), (-0.5, 4.3)):
                        for h in range(1, H + 1):
                            cells.add(scen_form(A, H, h, N, obj, flags, vw, rw, sms)[0])
    return cells


class ScenCase:
    """abr_env_mpc_decide_scen over `n` distinct sessions tiled `tile` times, with the horizons `hs` (round robin),
    K scenarios per session, the objective, `flags`, the penalties, weights (MEAN: None or drawn, some zero) and
    auto_reset (without it a fifth of the sessions are done).  `ties`: the tie worlds of search_forms.mpc_inputs (twin
    rungs, dyadic sizes and buffers) with dyadic scenario rows and weights, so that optima tie exactly with the same
    sequence through a twin rung: in another prefix when the twin is at step 0, in the same thread's leaves when it is
    at the last step."""

    def __init__(self, A, H, hs, n, tile, objective, flags, vw, K, weighted, auto_reset, rw=4.3, ties=False):
        self.A, self.H, self.hs, self.n, self.tile = A, H, tuple(hs), n, tile
        self.objective, self.flags, self.vw, self.rw = objective, flags, vw, rw
        self.K, self.weighted, self.auto_reset, self.ties = K, weighted, auto_reset, ties

    @property
    def N(self):
        return self.n * self.tile

    def cells(self, sms=B200_SMS):
        return {scen_form(self.A, self.H, h, self.N, self.objective, self.flags, self.vw, self.rw, sms)[0]
                for h in self.hs}

    def robust_case(self):
        import search_forms as sf
        return sf.MpcCase(self.A, self.H, "robust", self.vw, self.hs, self.n, tile=self.tile, rw=self.rw,
                          ties=self.ties)

    @property
    def id(self):
        obj = "mean" if self.objective == MEAN else "worst"
        return (f"A{self.A}H{self.H}-h{'.'.join(map(str, self.hs))}-n{self.n}x{self.tile}-{obj}K{self.K}"
                f"{'w' if self.weighted else ''}-{'exh' if self.flags else 'bb'}-vw{self.vw:g}"
                f"{'' if self.rw == 4.3 else f'rw{self.rw:g}'}{'-ties' if self.ties else ''}-reset{self.auto_reset}")


def _scen_cases():
    import search_forms as sf
    variants = [(MEAN, 0, 1.0), (MEAN, 0, 0.6), (MEAN, MPC_EXHAUSTIVE, 1.0), (MEAN, 0, -0.5),
                (WORST, 0, 1.0), (WORST, 0, 0.6), (WORST, MPC_EXHAUSTIVE, 1.0), (WORST, 0, -0.5)]
    ks = (1, 3, 16, 4, 2, 8, 5)
    cases = []
    for i, (A, H, _, n, tile) in enumerate(sf.SHAPES):
        hs = sorted({1, min(2, H), min(3, H), H})
        for j, (obj, flags, vw) in enumerate(variants):
            K = ks[(i + j) % len(ks)]
            # the large enumerations run with few scenarios, so that the oracle stays quick
            if A ** H * K > 2 ** 20:
                K = max(1, 2 ** 20 // A ** H)
            cases.append(ScenCase(A, H, hs, n, tile, obj, flags, vw, K, weighted=obj == MEAN and j % 2 == 0,
                                  auto_reset=(i + j) % 2))
    # a block slot serves several sessions in turn
    cases.append(ScenCase(3, 5, (1, 2, 4, 5), 24, 1600, MEAN, 0, 1.0, 4, weighted=True, auto_reset=0))
    cases.append(ScenCase(3, 5, (1, 2, 4, 5), 24, 1600, WORST, 0, 1.0, 4, weighted=False, auto_reset=1))
    # exact ties (the strict '>' per thread and the (value, index) reductions) and zero penalties under branch and
    # bound, on both session layouts and both objectives; each case also runs exhaustively
    for A, H, hs, n, tile in ((6, 4, (2, 3, 4), 24, 1), (6, 5, (3, 4, 5), 16, 16), (4, 7, (4, 5, 6), 24, 8)):
        for j, obj in enumerate((MEAN, WORST)):
            for vw, rw in ((1.0, 1.0), (0.0, 1.0), (0.5, 0.0)):
                cases.append(ScenCase(A, H, hs, n, tile, obj, 0, vw, 4 if obj == MEAN else 3,
                                      weighted=j == 0 and vw != 1.0, auto_reset=1, rw=rw, ties=True))
    for obj in (MEAN, WORST):   # both penalties zero, continuous ladder
        cases.append(ScenCase(6, 4, (1, 2, 4), 12, 1, obj, 0, 0.0, 5, weighted=obj == MEAN, auto_reset=0, rw=0.0))
    return cases


SCEN_CASES = _scen_cases()
