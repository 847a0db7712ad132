"""SPEC §4.5 restated in numpy on top of the C oracle's step: the windowed observation obs[3 + 2W + A][N].

``WindowObs`` keeps the caller's observation buffer next to an ``oracle.OracleEnv``.  ``observe()`` is
``abr_env_observe_window`` (both windows 0); ``step(actions)`` steps the oracle and updates the buffer as
``abr_env_step_policy_window`` does: a normal step moves both windows up one entry (fp32 values copied) and appends
thr * s_thr and delay * s_delay; a step that ends the video with auto_reset zeroes them; an inert step (a done
session, auto_reset = 0) leaves them.  Every other row is one fp64 operation rounded once to fp32, from the state after
the step.  Also: the world builder and the case table of the GPU tests.
"""
from __future__ import annotations

import numpy as np

from abrsimulator_b200 import synth
from oracle import oracle as orc


def f32(x):
    """fp64 values rounded once to fp32."""
    return np.asarray(x, np.float64).astype(np.float32)


def rows(A, W):
    """Row ranges of the observation: (utility, buffer, chunks left, throughput window, delay window, sizes)."""
    return 0, 1, 2, slice(3, 3 + W), slice(3 + W, 3 + 2 * W), slice(3 + 2 * W, 3 + 2 * W + A)


def state_rows(util, sizes, chunk, last_q, buffer, done, scales):
    """Rows 0-2 and the size rows of SPEC §4.5 from a state: ([3, N], [A, N]) float32."""
    V, A = sizes.shape
    s_util, s_buf, _, _, s_size = scales
    chunk = np.asarray(chunk, np.int64)
    last_q = np.asarray(last_q, np.int64)
    done = np.asarray(done, bool)
    k_prev = np.maximum(chunk - 1, 0)
    u = util[np.minimum(k_prev, V - 1), np.clip(last_q, 0, A - 1)]
    head = np.stack([np.where(last_q < 0, np.float32(0), f32(u * s_util)),
                     f32(np.asarray(buffer, np.float64) * s_buf),
                     f32((V - chunk).astype(np.float64) / V)])
    nxt = sizes[np.minimum(chunk, V - 1)].T * s_size          # [A, N]
    return head, np.where(done[None, :], np.float32(0), f32(nxt))


class WindowObs:
    """The windowed observation of an oracle environment (SPEC §4.5); ``obs`` is the [3 + 2W + A, N] buffer."""

    def __init__(self, ref: orc.OracleEnv, window, scales=(1.0,) * 5):
        self.ref, self.W, self.scales = ref, int(window), tuple(float(s) for s in scales)
        p = ref.params
        self.util = orc.utility_table(ref.bitrates, p.utility_mode, p.utility_scale)
        self.obs = np.zeros((3 + 2 * self.W + ref.A, ref.N), np.float32)

    def _state_rows(self):
        r = self.ref
        head, nxt = state_rows(self.util, r.sizes, r.field("chunk"), r.field("last_q"), r.field("buffer"),
                               r.field("done") != 0, self.scales)
        sz = rows(r.A, self.W)[5]
        self.obs[0:3] = head
        self.obs[sz] = nxt

    def observe(self):
        _, _, _, wt, wd, _ = rows(self.ref.A, self.W)
        self.obs[wt] = 0
        self.obs[wd] = 0
        self._state_rows()
        return self.obs

    def step(self, actions):
        """One oracle step with `actions`; returns the oracle's outputs.  ``self.obs`` is updated in place."""
        r, W = self.ref, self.W
        auto = bool(r.params.auto_reset)
        inert = np.zeros(r.N, bool) if auto else r.field("done") != 0
        out = r.step(actions)
        eov = out["eov"] != 0
        zero = eov & auto & ~inert
        roll = ~inert & ~zero
        _, _, _, wt, wd, _ = rows(r.A, W)
        for win, new in ((wt, f32(out["throughput"] * self.scales[2])), (wd, f32(out["delay"] * self.scales[3]))):
            block = self.obs[win]                                   # a view: [W, N]
            block[:W - 1, roll] = block[1:, roll].copy()
            block[W - 1, roll] = new[roll]
            block[:, zero] = 0
        self._state_rows()
        return out


def ladder(A):
    """A bitrate ladder of A rungs (kbit/s)."""
    base = np.array(synth.LADDER_KBPS + (6000.0, 8000.0, 10000.0, 12000.0), np.float64)
    return tuple(base[np.linspace(0, len(base) - 1, A).round().astype(int)] if A > 1 else base[:1])


def world(A, V=48, n_traces=16, T=128, seed=0):
    """(bitrates, sizes, bw, tl, ti): one ladder whose utility differs per chunk (so row 0's chunk index matters),
    ragged traces."""
    bitrates, sizes = synth.make_video(V, ladder=ladder(A), seed=seed)
    bitrates = np.ascontiguousarray(bitrates * (1.0 + 0.01 * np.arange(V))[:, None])
    bw, tl, ti = synth.make_traces(n_traces, T, seed=1234 + seed)
    rng = np.random.default_rng(seed + 5)
    tl = rng.integers(1, T + 1, size=n_traces).astype(np.int32)
    tl[-1] = T
    ti = rng.choice([0.5, 1.0, 2.0], size=n_traces)
    return bitrates, sizes, bw, tl, ti


def sessions(N, n_traces, T, seed=11):
    rng = np.random.default_rng(seed)
    tid = rng.integers(0, n_traces, size=N).astype(np.int32)
    off = rng.uniform(0, T * 2.0 * 1.5, size=N)
    return tid, off


def action_table(steps, N, A, seed=3):
    """The seeded greedy actions of the GPU tests: one-hot logits on this table."""
    return np.random.default_rng(seed).integers(0, A, size=(steps, N)).astype(np.int32)


# (W, A, N, V, auto_reset, track_history, track_acc, default_quality): every W in {1, 8, 32}, A in {1, 6, 10}, N in
# {1, 127, 3000, 2^21 + 77}, auto_reset 0 and 1, the two trackers on and off; V = 20 crosses three ends of video in
# 64 steps.  default_quality -1: row 0 is 0 until the first download.
CASES = (
    (1, 1, 1, 20, 1, 0, 0, 0),
    (8, 6, 127, 48, 0, 1, 1, 1),
    (32, 10, 3000, 20, 1, 1, 0, -1),
    (8, 10, 3000, 20, 0, 0, 1, 2),
    (32, 6, 127, 48, 0, 0, 0, 1),
    (1, 6, 3000, 20, 0, 1, 1, -1),
    (32, 1, 127, 20, 1, 1, 1, 0),
    (8, 6, 2 ** 21 + 77, 20, 1, 0, 0, 1),
    (8, 6, 2 ** 21 + 77, 48, 0, 1, 1, 1),
)
STEPS = 64
