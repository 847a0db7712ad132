"""Which compiled form and path of the two search kernels a decision takes — TEST INFRASTRUCTURE, no tests.

``abr_mpc_kernel`` (abr_mpc.cu) has 42 instantiations ``<WPS, AT, CLAMP, PRUNE>``, and inside each one a session takes
one of four search paths chosen from its own truncated horizon h, with a ``VW1`` specialisation on top;
``abr_lookahead_kernel`` (abr_step.cu) lays out 32 / A sessions per warp and has a FAST form.  ``mpc_form`` and
``lookahead_form`` restate those choices in Python, ``reachable_mpc_cells`` enumerates every cell a legal call can
reach, and ``MPC_CASES`` / ``LOOKAHEAD_CASES`` are the cases of ``test_gpu_search_forms.py`` that reach them.
``test_search_forms_ledger.py`` checks, on the CPU, that the kernel sources still contain what the restatement relies
on and that the cases reach every reachable cell.
"""
from __future__ import annotations

from dataclasses import dataclass

# constants of abr_mpc.cu / abr_step.cu (the ledger checks them against the sources)
K_MAX_H = 8
K_MAX_A = 16
K_MPC_WARPS_PER_BLOCK = 4
K_PREFIX_CACHE = 64
K_MAX_LIVE_PREFIX = 256
K_MAX_LIVE_ROW = 1536
WPS_COMBOS = 32 * 36 * 4          # below this many sequences a session never gets a whole block
COMPILED_A = (2, 3, 4, 5, 6, 8)   # ladder sizes with their own instantiation; every other A runs the AT = 0 form
K_LOOKAHEAD_BLOCK = 128
LOOKAHEAD_MAX_COMBOS = 1 << 20
B200_SMS = 148

MPC_TRUNCATE, MPC_EXHAUSTIVE = 1, 8    # abr_b200.h
# the ways a caller selects the MPC search: (mode, flags); "robust" with a negative penalty is a sixth way in, but it
# selects the same kernel as "robust_exh"
MODES = dict(ref=(0, 0), ref_trunc=(0, MPC_TRUNCATE), robust=(1, 0), robust_exh=(1, MPC_EXHAUSTIVE))
PATHS = ("h1", "plain", "cache", "compact")


def mpc_form(A, H, h, N, mode, flags, vw, rw, sms=B200_SMS):
    """(cell, stride) of a session with truncated horizon h >= 1 in a call over N sessions.

    cell = (wps, AT, path, search_mode, vw1): warps per session, compiled ladder size (0 = runtime A), the search path
    the session takes, the kernel's (CLAMP, PRUNE) pair as "ref" / "enum" / "prune", and smooth_penalty == 1.0.
    stride: a block slot serves more than one session (the grid-stride loop of abr_mpc_kernel).

    Restates launch_mpc (abr_mpc.cu: `wps`, `blocks` capped at `sms * 64`, `prune`, the `switch (a.A)`) and the
    per-session choice in abr_mpc_kernel (`if (h == 1)`, the `compact` predicate, `use_cache` in search)."""
    assert 1 <= h <= H <= K_MAX_H and 1 <= A <= K_MAX_A
    wps = 1 if (N >= 16 * sms or A ** H < WPS_COMBOS) else K_MPC_WARPS_PER_BLOCK
    spb = K_MPC_WARPS_PER_BLOCK // wps
    stride = (N + spb - 1) // spb > 64 * sms
    AT = A if A in COMPILED_A else 0
    clamp = mode == 1
    prune = clamp and not (flags & MPC_EXHAUSTIVE) and vw >= 0.0 and rw >= 0.0
    search_mode = "prune" if prune else "enum" if clamp else "ref"
    if h == 1:
        path = "h1"
    else:
        n_pre = A ** (h - 2)                      # prefixes of depth h - 2
        n_par = n_pre // A if h >= 4 else 0       # their parents (search: P >= 2)
        compact = prune and h >= 4 and n_pre // A <= K_PREFIX_CACHE and n_pre <= K_MAX_LIVE_PREFIX and \
            n_pre * A <= K_MAX_LIVE_ROW
        use_cache = h >= 4 and n_par <= K_PREFIX_CACHE
        path = "compact" if compact else "cache" if use_cache else "plain"
    return (wps, AT, path, search_mode, vw == 1.0), stride


def lookahead_form(A, auto_reset):
    """(sessions per warp, idle lanes, FAST) of abr_lookahead_kernel: `per_warp = 32 / A`, FAST = auto_reset."""
    return 32 // A, 32 % A != 0, bool(auto_reset)


def legal_mpc_shapes():
    """(A, H) with 1 <= A <= 16, 1 <= H <= 8 and A^H <= 2^31 - 1 (check_mpc_shape in abr_capi.cu)."""
    return [(A, H) for A in range(1, K_MAX_A + 1) for H in range(1, K_MAX_H + 1) if A ** H <= 2 ** 31 - 1]


def reachable_mpc_cells(sms=B200_SMS):
    """Every cell a legal standalone or environment call can reach: all shapes, every h <= H (h == H only for mode 0
    without ABR_MPC_TRUNCATE), N on both sides of the warp-per-session threshold, every way to select the search, both
    sides of smooth_penalty == 1."""
    cells = set()
    for A, H in legal_mpc_shapes():
        cells |= reachable_mpc_cells_of(A, H, sms)
    return cells


def reachable_mpc_cells_of(A, H, sms=B200_SMS):
    cells = set()
    for N in (1, 16 * sms - 1, 16 * sms):
        for name, (mode, flags) in MODES.items():
            for vw, rw in ((1.0, 4.3), (0.6, 4.3), (-0.5, 4.3), (1.0, -2.0)):
                for h in range(1, H + 1):
                    if name == "ref" and h != H:
                        continue
                    cells.add(mpc_form(A, H, h, N, mode, flags, vw, rw, sms)[0])
    return cells


@dataclass(frozen=True)
class MpcCase:
    """One call of the standalone decision: `n` distinct sessions, repeated `tile` times (copy c of session s sits at
    c * n + s), their truncated horizons taken round robin from `hs` (h == H: a random chunk with k + H <= V; h < H:
    chunk V - h).  `ties`: worlds in which many sessions have exactly tied optima across different live prefixes
    (mpc_inputs).  `K`: ring capacity."""
    A: int
    H: int
    mode: str
    vw: float
    hs: tuple
    n: int
    tile: int = 1
    rw: float = 4.3
    K: int = 6
    ties: bool = False

    @property
    def N(self):
        return self.n * self.tile

    @property
    def mode_flags(self):
        return MODES[self.mode]

    def forms(self, sms=B200_SMS):
        """{h: (cell, stride)} of the case's searched sessions."""
        mode, flags = self.mode_flags
        return {h: mpc_form(self.A, self.H, h, self.N, mode, flags, self.vw, self.rw, sms) for h in self.hs}

    def slot_step(self, sms=B200_SMS):
        """How far apart the sessions that one block slot serves in turn lie: gridDim.x * sessions per block."""
        (wps, *_), _ = next(iter(self.forms(sms).values()))
        spb = K_MPC_WARPS_PER_BLOCK // wps
        return min(-(-self.N // spb), 64 * sms) * spb

    @property
    def id(self):
        """The cell first (shared by every h of the case: wps, AT, search mode, VW1; then the path of each h), then
        the inputs."""
        forms = self.forms()
        (wps, AT, _, search_mode, vw1), stride = forms[self.hs[0]]
        paths = ".".join(f"h{h}={forms[h][0][2]}" for h in self.hs)
        cell = f"wps{wps}-AT{AT}-{search_mode}-vw1{'on' if vw1 else 'off'}-{paths}" + ("-stride" if stride else "")
        pen = f"vw{self.vw:g}" + ("" if self.rw == 4.3 else f"rw{self.rw:g}")
        extra = (f"-K{self.K}" if self.K != 6 else "") + ("-ties" if self.ties else "") + \
            (f"-x{self.tile}" if self.tile > 1 else "")
        return f"{cell}-A{self.A}H{self.H}-{self.mode}-{pen}-n{self.n}{extra}"

    def cost(self):
        """Σ over distinct sessions of A^h·h: what the oracle enumerates."""
        per_h = [sum(1 for i in range(self.n) if self.hs[i % len(self.hs)] == h) for h in self.hs]
        return sum(c * self.A ** h * h for c, h in zip(per_h, self.hs))


# the ways to select the search, with both sides of smooth_penalty == 1: ref (mode 0, truncating), enum (robust with
# ABR_MPC_EXHAUSTIVE, or with a negative penalty) and prune (robust), each with VW1 on and off
VARIANTS = (
    dict(mode="ref_trunc", vw=1.0), dict(mode="ref_trunc", vw=0.6),
    dict(mode="robust", vw=1.0), dict(mode="robust", vw=0.6),
    dict(mode="robust_exh", vw=1.0), dict(mode="robust", vw=-0.5),
)

# (A, H, hs, n, tile): for every compiled ladder size, a warp-per-session shape (A^H < 4608, or tiled past 16 * SMs
# sessions) and a block-per-session shape (A^H >= 4608, few sessions), with horizons that reach every path the shape has
SHAPES = (
    # warp per session
    (1, 8, (1, 2, 3, 4, 8), 10, 1),
    (2, 8, (1, 2, 3, 4, 8), 20, 1),
    (3, 7, (1, 2, 4, 6, 7), 20, 1),
    (4, 6, (1, 2, 4, 6), 16, 1),         # h = 6: 64 parents = kPrefixCache, 256 prefixes = kMaxLivePrefix
    (5, 5, (1, 3, 4, 5), 16, 1),
    (6, 4, (1, 2, 4), 12, 1),
    (8, 4, (1, 2, 4), 12, 1),
    (8, 5, (1, 3, 5), 12, 200),          # h = 5: parent cache, not compactable (branch and bound with the cache)
    (7, 4, (1, 2, 4), 12, 1),
    (7, 5, (1, 3, 5), 12, 200),
    (16, 3, (1, 2, 3), 12, 1),
    (16, 4, (1, 2, 4), 6, 400),
    # block per session
    (3, 8, (1, 3, 5, 8), 16, 1),
    (4, 7, (1, 3, 6, 7), 16, 1),
    (5, 6, (1, 2, 5, 6), 16, 1),
    (6, 5, (1, 3, 5), 12, 1),
    (8, 5, (1, 3, 4, 5), 16, 1),
    (7, 5, (1, 2, 4, 5), 16, 1),
    (11, 4, (1, 3, 4), 12, 1),           # h = 4: 1 331 rows, the largest compactable shape
    (12, 4, (2, 4), 8, 1),               # h = 4: 1 728 rows > kMaxLiveRow, falls back to the cached search
    (16, 4, (1, 2, 4), 12, 1),
)

MPC_CASES = [MpcCase(A, H, hs=hs, n=n, tile=tile, **v) for A, H, hs, n, tile in SHAPES for v in VARIANTS] + [
    # a block slot serves several sessions (N > 4 * 64 * SMs with one warp per session), with every path in turn
    # (the n distinct sessions do not divide the slot step, so each slot's next session is another distinct one)
    MpcCase(3, 5, "ref_trunc", 1.0, (1, 2, 4, 5), 24, tile=1600),
    MpcCase(3, 5, "robust", 1.0, (1, 2, 4, 5), 24, tile=1600),
    MpcCase(7, 4, "robust", 0.6, (1, 3, 4), 24, tile=1600),
    # exact ties in the compacted search of a whole block per session: the live lists fill in atomic order, so the
    # first minimum rests on the (value, index) compare; dyadic penalties keep every term exact
    MpcCase(6, 5, "robust", 1.0, (4, 5), 16, tile=16, rw=1.0, ties=True),
    MpcCase(6, 5, "robust", 2.0, (4, 5), 16, tile=16, rw=1.0, ties=True),
    MpcCase(4, 7, "robust", 1.0, (4, 5, 6), 24, tile=8, rw=1.0, ties=True),
    MpcCase(4, 7, "robust", 0.5, (4, 5, 6), 24, tile=8, rw=1.0, ties=True),
    MpcCase(11, 4, "robust", 1.0, (4,), 12, tile=16, rw=1.0, ties=True),
    # throughput histories of more than 32 samples: the second round of the predictor's 32-lane loop
    MpcCase(6, 4, "ref", 1.0, (4,), 24, K=64),
    MpcCase(6, 4, "robust", 1.0, (1, 2, 4), 24, K=64),
    MpcCase(7, 5, "ref", 0.6, (5,), 16, K=40),
    MpcCase(7, 5, "robust", 1.0, (1, 4, 5), 24, K=40),
    MpcCase(5, 3, "robust", 1.0, (3,), 24, tile=200, K=64),
]


MPC_V = 48    # chunks of the standalone cases' videos


def mpc_inputs(case, seed):
    """The case's distinct sessions: worlds of test_gpu_mpc._random_batch, chunks that give the listed horizons, some
    sessions without a previous chunk, and robust error state.  Mode 0 charges the rebuffering of every chunk against
    its utility without the robust mode's clamp, so its chunks are short and light enough that the best rung depends
    on the session's predicted throughput.

    `ties`: the ladder is on a 0.25 grid with most rungs present twice (equal bitrate and size), sizes = bitrates,
    one-second chunks and buffers on the 0.25 grid; the throughput samples and error state give a robust prediction of
    exactly 1 or 2.  Every quantity is then a short dyadic fraction and exact, and an optimum through a doubled rung
    ties with the same sequence through its twin, in another live prefix."""
    import numpy as np
    rng = np.random.default_rng(seed)
    A, H, n, K, V = case.A, case.H, case.n, case.K, MPC_V
    ref = case.mode_flags[0] == 0
    if case.ties:
        vals = np.sort(rng.choice(np.arange(1, 40) * 0.25, size=(A + 1) // 2, replace=False))
        bitrates = np.tile(np.sort(np.concatenate([vals, vals[:A // 2]])), (V, 1))
        sizes = bitrates.copy()
    else:
        lad = np.sort(rng.uniform(0.2, 5.0, size=A))
        bitrates = np.tile(lad, (V, 1)) * rng.uniform(0.9, 1.1, size=(V, 1))
        sizes = bitrates * (0.35 if ref else 4.0) * rng.uniform(0.8, 1.2, size=(V, A))
    h_of = np.array([case.hs[i % len(case.hs)] for i in range(n)])
    chunk = np.where(h_of == H, rng.integers(0, V - H + 1, size=n), V - h_of).astype(np.int32)
    prev_q = rng.integers(-1, A, size=n).astype(np.int32)
    b = dict(sizes=np.ascontiguousarray(sizes), bitrates=np.ascontiguousarray(bitrates), chunk=chunk, prev_q=prev_q,
             buffer=np.round(rng.uniform(0, 40, size=n), 9), bw_hist=np.round(rng.uniform(0.2, 6.0, size=(n, K)), 9),
             hist_len=rng.integers(1, 2 * K + 1, size=n).astype(np.int32), h=h_of)
    b["last_pred"] = np.where(rng.random(n) < 0.8, rng.uniform(0.2, 6.0, n), 0.0)
    b["err_ring"] = rng.uniform(0, 0.5, size=(n, K))
    b["err_len"] = rng.integers(0, 2 * K, size=n).astype(np.int32)
    if case.ties:
        x = rng.choice([1.0, 2.0], size=n)                         # every sample x: harmonic mean x
        b["bw_hist"] = np.ascontiguousarray(np.repeat(x[:, None], K, axis=1))
        b["err_ring"] = np.ascontiguousarray(np.repeat(x[:, None] - 1.0, K, axis=1))   # x / (1 + max error) = 1 ...
        b["last_pred"] = x * rng.choice([0.0, 1.0], size=n)        # ... the new error |x - x| / x = 0 changes nothing
        b["buffer"] = np.round(rng.uniform(0, 12, size=n) * 4) / 4
    kw = dict(chunk_length=1.0 if case.ties else 0.25 if ref else 4.0, max_buffer=30.0, hist_k=K,
              smooth_penalty=case.vw, rebuf_penalty=case.rw, utility_scale=1.0)
    return b, kw


def mpc_expected(case, b, kw):
    """orc.mpc_decide on the distinct sessions.  Mode 0 has no truncation in the oracle: the sessions of each h are
    decided with horizon h (what ABR_MPC_TRUNCATE does), their rows padded with -1."""
    import numpy as np
    from oracle import oracle as orc
    mode, _ = case.mode_flags
    n, H = case.n, case.H
    util = orc.utility_table(b["bitrates"], 0, 1.0)
    p = orc.make_params(**kw)
    st = (b["last_pred"].copy(), b["err_ring"].copy(), b["err_len"].copy()) if mode == 1 else (None, None, None)
    groups = [(H, np.arange(n))] if mode == 1 else [(h, np.flatnonzero(b["h"] == h)) for h in case.hs]
    exp = dict(action=np.zeros(n, np.int32), best_J=np.zeros(n), best_seq=np.full((n, H), -1, np.int32),
               preds=np.zeros((n, H)), n_errors=0)
    for h, idx in groups:
        sub = lambda x: np.ascontiguousarray(x[idx])
        r = orc.mpc_decide(b["sizes"], util, sub(b["chunk"]), sub(b["prev_q"]), sub(b["buffer"]), sub(b["bw_hist"]),
                           sub(b["hist_len"]), h, mode, p, *st)
        exp["action"][idx] = r["action"]
        exp["best_J"][idx] = r["best_J"]
        exp["best_seq"][idx, :h] = r["best_seq"]
        exp["preds"][idx, :h] = r["preds"]
        exp["n_errors"] += r["n_errors"]
    return exp, util, st


def robust_values(case, b, kw, exp, s):
    """-J of every sequence of robust-mode session s, in C order: SPEC §5.2's objective (oracle/mpc_oracle.py
    objective_robust) at the oracle's prediction, vectorised over the sequences with the same operations in the same
    order."""
    import itertools
    import numpy as np
    A, h, k = case.A, int((exp["best_seq"][s] >= 0).sum()), int(b["chunk"][s])
    U = b["bitrates"]          # utility_table(bitrates, mode 0, scale 1)
    c, L, B, vw, rw = exp["preds"][s, 0], kw["chunk_length"], kw["max_buffer"], kw["smooth_penalty"], kw["rebuf_penalty"]
    seqs = np.array(list(itertools.product(range(A), repeat=h)))
    vq = qv = rt = np.zeros(len(seqs))
    buf = np.full(len(seqs), float(b["buffer"][s]))
    ap = np.full(len(seqs), int(b["prev_q"][s]))
    for i in range(h):
        a = seqs[:, i]
        u = U[k + i][a]
        vq = vq + u
        qv = np.where(ap >= 0, qv + np.abs(u - U[k + i][np.maximum(ap, 0)]), qv)
        dl = b["sizes"][k + i][a] / c
        rt = rt + np.maximum(dl - buf, 0.0)
        if i != h - 1:
            t = np.maximum(buf - dl, 0.0)
            w = np.maximum(t + L - B, 0.0)
            buf = np.maximum(t + L - w, 0.0)
        ap = a
    return (vq - vw * qv) - rw * rt


def prefix_ties(case, b, kw, exp):
    """Sessions whose optimum is tied, exactly, with a sequence in another depth-(h-2) prefix (another entry of the
    compacted search's live-prefix list).  Checks on the way that the restated values reproduce the oracle's optimum."""
    import numpy as np
    count = 0
    for s in range(case.n):
        q = robust_values(case, b, kw, exp, s)
        best = np.flatnonzero(q == q.max())
        h = int((exp["best_seq"][s] >= 0).sum())
        first = int(np.ravel_multi_index(tuple(exp["best_seq"][s, :h]), (case.A,) * h))
        assert -q.max() == exp["best_J"][s] and best[0] == first, s
        count += len(set((best // case.A ** 2).tolist())) > 1
    return count


@dataclass(frozen=True)
class LookaheadCase:
    """abr_env_lookahead_decide over `n` sessions of an A-rung ladder in a LOOKAHEAD_V-chunk video: one decision
    after each entry of `steps`, the number of random steps taken since the previous one."""
    A: int
    H: int
    auto_reset: int
    n: int
    steps: tuple = (9, 8)

    @property
    def id(self):
        return f"A{self.A}H{self.H}-reset{self.auto_reset}-n{self.n}"

    def cost(self):
        return self.n * self.A ** self.H * self.H * len(self.steps)


def _lookahead_cases():
    cases = []
    for auto_reset in (0, 1):
        for A in (1, 2, 5, 7, 11, 16):
            for H in (1, 3):
                per_block = (K_LOOKAHEAD_BLOCK // 32) * (32 // A)
                n = 2 * per_block + 1 + A if A ** H <= 512 else per_block + 3
                cases.append(LookaheadCase(A, H, auto_reset, n))
            if A <= 5:
                cases.append(LookaheadCase(A, 8, auto_reset, {1: 131, 2: 37, 5: 5}[A], steps=(7,)))
        cases.append(LookaheadCase(16, 5, auto_reset, 5, steps=(7,)))   # A^H = 2^20, the largest legal shape
    # sessions near the end of the video: truncated horizons (and, without auto_reset, done sessions)
    cases += [LookaheadCase(7, 3, 0, 77, steps=(17, 2, 1)), LookaheadCase(11, 3, 1, 29, steps=(17, 2, 1))]
    return cases


LOOKAHEAD_V = 20
LOOKAHEAD_CASES = _lookahead_cases()
