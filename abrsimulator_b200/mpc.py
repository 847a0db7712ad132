"""MPC bitrate controller: host-side mirror of ``mpc.py:20-186`` over the CUDA decision kernel.

Same names, argument meaning and error behaviour as the reference's ``MPCBitrateController``:

* pull style (``mpc.py:181-186``): ``MPCBitrateController(player).next_bitrate()`` over a player exposing
  ``get_mpd() / get_qoe_metric() / get_next_chunk_info()`` (``mpc_test.py:39-50``);
* push style (the call ``Simulator.run`` makes, ``Simulator.py:155``):
  ``get_next_bitrate(chunk_id, previous_bitrates, previous_bandwidths, buffer_level)``;
* batched: ``decide_batch(...)`` over device tensors, and ``BatchedABREnv.mpc_decide``.

``mode="reference"`` reproduces the shipped arithmetic bit for bit (SPEC.md §5.1), including the growth
of ``previous_bandwidths`` by ``horizon`` entries per call (SURVEY.md D10) when ``strict_history=True``.
``mode="robust"`` is SPEC.md §5.2.  ``predictor="expsmoothing"`` (or ``predict_throughput(...,
method="expsmoothing")``) is the reference's second predictor (mpc.py:72-79, SPEC.md §5.4);
``next_bitrate_startup()`` is the start-up branch of the reference's pseudo-code (mpc.py:7-18, SPEC.md §5.3).
Every decision runs on the GPU; there is no CPU fallback.
"""
from __future__ import annotations

import itertools

import numpy as np

from . import _lib
from ._lib import MPC_REF, MPC_ROBUST, MPC_PRED_SES, _addr


class MPCBitrateController:
    """Drop-in for ``mpc.MPCBitrateController`` (mpc.py:20-59)."""

    def __init__(self, player=None, bitrate_utility=None, horizon=None, mode="reference", strict_history=True,
                 predictor="harmonic", **params):
        self.player = None
        self.mpd = None
        self.qoe = None
        if player:
            self.player = player
            self.mpd = player.get_mpd()
            self.qoe = player.get_qoe_metric()
        # like the reference (mpc.py:58, D9) the identity utility is always installed
        self.bitrate_utility = self.default_bitrate_utility
        self.horizon = 3 if horizon is None else horizon
        self.mode = MPC_ROBUST if mode in ("robust", MPC_ROBUST) else MPC_REF
        self.strict_history = strict_history
        if predictor not in ("harmonic", "expsmoothing"):
            raise ValueError("predictor must be 'harmonic' or 'expsmoothing' (mpc.py:69-93)")
        if predictor == "expsmoothing" and self.mode != MPC_REF:
            raise ValueError("the 'expsmoothing' predictor belongs to mode='reference'; the robust mode defines its own")
        self.predictor = predictor
        self.extra_params = dict(params)
        self.predicted_bandwidths = None
        # robust-mode predictor state (one session)
        self._last_pred = np.zeros(1)
        self._err_ring = None
        self._err_len = np.zeros(1, np.int32)
        self._tables_key = None
        self._tables = None

    # -- reference plumbing (mpc.py:61-67, with the missing `self` supplied) --
    def update_mpd(self):
        self.mpd = self.player.get_mpd()
        self._tables_key = None

    def update_qoe(self):
        self.qoe = self.player.get_qoe_metric()

    def default_bitrate_utility(self, bitrate):
        """Identity (mpc.py:95-97)."""
        return bitrate

    # -- tables / params --
    def _get_tables(self):
        key = (id(self.mpd), len(self.mpd.chunks))
        if self._tables_key != key:
            bitrates = np.array([list(c.bitrates) for c in self.mpd.chunks], dtype=np.float64)
            sizes = np.array([list(c.sizes) for c in self.mpd.chunks], dtype=np.float64)
            self._tables, self._tables_key = (np.ascontiguousarray(bitrates), np.ascontiguousarray(sizes)), key
        return self._tables

    def _params(self):
        kw = dict(chunk_length=float(self.mpd.chunk_length), max_buffer=float(self.mpd.max_buffer),
                  rebuf_penalty=float(self.qoe.rebuffer_weight), smooth_penalty=float(self.qoe.variance_weight),
                  utility_scale=1.0)
        kw.update(self.extra_params)
        return _lib.default_params(**kw)

    # -- one decision through the C-ABI with host buffers --
    def _decide(self, chunk, prev_q, history, buffer_level, horizon, ses=None, startup_grid=None):
        """``ses``: override of the predictor choice; ``startup_grid`` = (n_ts, ts_step): start-up phase (SPEC §5.3) —
        the returned tuple then carries the start-up delay as a fifth element."""
        lib = _lib.load()
        ses = (self.predictor == "expsmoothing") if ses is None else ses
        bitrates, sizes = self._get_tables()
        V, A = bitrates.shape
        hist = np.ascontiguousarray(list(history), dtype=np.float64)
        n = hist.size
        # the reference raises plain Python errors for these inputs (SURVEY.md D13, D14)
        if self.mode == MPC_REF:
            if n == 0:
                raise ZeroDivisionError("division by zero")            # mpc.py:90
            if np.any(hist == 0.0):
                raise ZeroDivisionError("float division by zero")       # mpc.py:88
            if chunk + horizon > V:
                raise IndexError("list index out of range")             # mpc.py:125-128
        p = self._params()
        K = max(n, int(p.hist_k), 1) if self.mode == MPC_REF else max(int(p.hist_k), 1)
        ring = np.zeros((1, K))
        if self.mode == MPC_REF:
            ring[0, :n] = hist
            hl = n
        else:   # ring semantics: the kernel takes the last K samples
            tail = hist[-K:]
            ring[0, :tail.size] = tail
            hl = tail.size
            if self._err_ring is None or self._err_ring.shape[1] != K:
                self._err_ring = np.zeros((1, K))
        act = np.empty(1, np.int32)
        bj = np.empty(1)
        seq = np.empty((1, horizon), np.int32)
        preds = np.empty((1, horizon))
        nerr = np.zeros(1, np.int32)
        robust = self.mode == MPC_ROBUST
        flags = MPC_PRED_SES if ses else 0
        # named: only their addresses are passed, so they must outlive the call
        chunk_a, prev_a = np.array([chunk], np.int32), np.array([prev_q], np.int32)
        buffer_a, hl_a = np.array([buffer_level], np.float64), np.array([hl], np.int32)
        head = (_addr(sizes), _addr(bitrates), V, A, p, 1, _addr(chunk_a), _addr(prev_a), _addr(buffer_a), _addr(ring),
                _addr(hl_a), K, _addr(self._last_pred) if robust else None, _addr(self._err_ring) if robust else None,
                _addr(self._err_len) if robust else None, horizon, self.mode, flags)
        ts = np.zeros(1)
        if startup_grid is None:
            _lib.check(lib.abr_mpc_decide_host(*head, _addr(act), _addr(bj), _addr(seq), _addr(preds), _addr(nerr)))
        else:
            n_ts, ts_step = startup_grid
            _lib.check(lib.abr_mpc_decide_startup_host(*head, None, int(n_ts), float(ts_step), _addr(act), _addr(ts),
                                                       _addr(bj), _addr(seq), _addr(preds), _addr(nerr)))
        if nerr[0] != 0 or act[0] < 0:
            raise ValueError("invalid MPC input (previous bitrate index out of range, or a non-positive prediction?)")
        if startup_grid is not None:
            return int(act[0]), seq[0].copy(), float(bj[0]), preds[0].copy(), float(ts[0])
        return int(act[0]), seq[0].copy(), float(bj[0]), preds[0].copy()

    # -- reference API --
    def predict_throughput(self, horizon, throughput_values, throughput_times=None, method="harmonic"):
        """``method="harmonic"`` (mpc.py:81-93): like the reference, the predictions are appended to
        ``throughput_values`` when ``strict_history`` is set (D10).  ``method="expsmoothing"`` (mpc.py:72-79): the flat
        forecast of simple exponential smoothing (alpha = 0.5, least-squares initial level — SPEC.md §5.4: the closed form
        of what the reference gets from statsmodels' ``SimpleExpSmoothing(data).fit(0.5).predict(...)``); returned as a
        numpy array like the reference's, the history is left alone."""
        if method not in ("harmonic", "expsmoothing"):
            raise ValueError(f"unknown prediction method {method!r} (mpc.py:69-93 knows 'harmonic' and 'expsmoothing')")
        if self.mpd is None:
            raise RuntimeError("predict_throughput needs a player (mpd) to run the kernel against")
        if method == "expsmoothing":
            vals = list(throughput_values)
            if len(vals) == 0:
                raise ValueError("zero-size array")              # what np / statsmodels raise for an empty series
            bitrates, _ = self._get_tables()
            saved_mode, self.mode = self.mode, MPC_REF
            try:
                hh = min(max(int(horizon), 1), bitrates.shape[0], 8)
                _, _, _, p = self._decide(0, 0, vals, 0.0, hh, ses=True)
            finally:
                self.mode = saved_mode
            return np.full(int(horizon), float(p[0]))            # flat forecast: every step is the last level
        bitrates, _ = self._get_tables()
        V = bitrates.shape[0]
        hist = list(throughput_values)
        if len(hist) == 0:
            raise ZeroDivisionError("division by zero")
        preds = []
        done = 0
        saved_mode = self.mode
        self.mode = MPC_REF
        try:
            while done < horizon:       # horizons longer than the video are predicted in slices
                hh = min(horizon - done, V, 8)
                _, _, _, p = self._decide(0, 0, hist, 0.0, hh)
                preds += [float(x) for x in p]
                hist += [float(x) for x in p]
                done += hh
        finally:
            self.mode = saved_mode
        if self.strict_history and isinstance(throughput_values, list):
            throughput_values.extend(preds)
        return preds

    def update_bandwidth_prediction(self):
        """mpc.py:164-169."""
        chunk_info = self.player.get_next_chunk_info()
        self.predicted_bandwidths = self.predict_throughput(self.horizon, chunk_info.previous_bandwidths)

    def optimize_qoe(self, chunk_info):
        """Best bitrate sequence as a float vector, like ``scipy.optimize.brute(finish=None)`` (mpc.py:171-179)."""
        hist = list(chunk_info.previous_bandwidths)
        if self.mode == MPC_REF and self.strict_history and self.predicted_bandwidths is not None:
            # the reference optimises with predictions made BEFORE they were appended to the list
            n_pred = len(self.predicted_bandwidths)
            if len(hist) >= n_pred and hist[-n_pred:] == list(self.predicted_bandwidths):
                hist = hist[:-n_pred]
        prev = getattr(chunk_info, "previous_bitrate", None)
        if prev is None:
            prev = chunk_info.previous_bitrates[-1]
        chunk = getattr(chunk_info, "chunk_number", None)
        if chunk is None:
            chunk = chunk_info.chunk_id
        _, seq, _, _ = self._decide(int(chunk), int(prev), hist, float(chunk_info.buffer_level), self.horizon)
        return seq.astype(np.float64)

    def next_bitrate(self):
        """mpc.py:181-186: predict, optimise, return ``int(result[0])`` — one kernel launch.  The predictions
        are appended to the player's ``previous_bandwidths`` afterwards, as the reference's predictor does (D10)."""
        chunk_info = self.player.get_next_chunk_info()
        prev = getattr(chunk_info, "previous_bitrate", None)
        if prev is None:
            prev = chunk_info.previous_bitrates[-1]
        chunk = getattr(chunk_info, "chunk_number", None)
        if chunk is None:
            chunk = chunk_info.chunk_id
        act, _, _, preds = self._decide(int(chunk), int(prev), list(chunk_info.previous_bandwidths),
                                        float(chunk_info.buffer_level), self.horizon)
        self.predicted_bandwidths = [float(x) for x in preds]
        if (self.mode == MPC_REF and self.predictor == "harmonic" and self.strict_history and
                isinstance(chunk_info.previous_bandwidths, list)):
            chunk_info.previous_bandwidths.extend(self.predicted_bandwidths)
        return act

    def next_bitrate_startup(self, n_ts=16, ts_step=0.5):
        """Start-up branch of the reference's pseudo-code (mpc.py:7-18: ``R[k], T_s = f_st(R[k-1], B[k], C_pred)`` —
        "start playback after T_s seconds"), which its code leaves as ``startup_delay = 0 #TODO`` (mpc.py:141):
        returns ``(bitrate, T_s)`` with ``T_s`` on the grid ``{0, ts_step, ..., (n_ts-1)*ts_step}`` (SPEC.md §5.3);
        ``startup_weight`` comes from the player's QoE metric (mpc.py:160)."""
        chunk_info = self.player.get_next_chunk_info()
        prev = getattr(chunk_info, "previous_bitrate", None)
        if prev is None:
            prev = chunk_info.previous_bitrates[-1]
        chunk = getattr(chunk_info, "chunk_number", None)
        if chunk is None:
            chunk = chunk_info.chunk_id
        saved = dict(self.extra_params)
        self.extra_params.setdefault("startup_penalty", float(getattr(self.qoe, "startup_weight", 0.0)))
        try:
            act, _, _, preds, ts = self._decide(int(chunk), int(prev), list(chunk_info.previous_bandwidths),
                                                float(chunk_info.buffer_level), self.horizon,
                                                startup_grid=(n_ts, ts_step))
        finally:
            self.extra_params = saved
        self.predicted_bandwidths = [float(x) for x in preds]
        harmonic = self.predictor == "harmonic"
        if self.mode == MPC_REF and harmonic and self.strict_history and isinstance(chunk_info.previous_bandwidths, list):
            chunk_info.previous_bandwidths.extend(self.predicted_bandwidths)
        return act, ts

    def get_next_bitrate(self, chunk_id, previous_bitrates, previous_bandwidths, buffer_level):
        """Push-style entry the environment calls (Simulator.py:155).  Never raises for an empty history
        or a horizon running past the video: returns the default quality / truncates instead."""
        V = len(self.mpd.chunks)
        prev = previous_bitrates[-1] if len(previous_bitrates) else int(self._params().default_quality)
        if len(previous_bandwidths) == 0:
            return int(self._params().default_quality)
        h = min(self.horizon, V - int(chunk_id))
        if h <= 0:
            return 0
        act, _, _, _ = self._decide(int(chunk_id), int(prev), list(previous_bandwidths), float(buffer_level), h)
        return act

    def objective(self, R_arg, chunk_info):
        """−QoE of one bitrate sequence (mpc.py:120-162), evaluated by the score kernel."""
        return float(self.objective_batch([list(R_arg)], chunk_info)[0])

    def objective_batch(self, sequences, chunk_info):
        lib = _lib.load()
        bitrates, sizes = self._get_tables()
        V, A = bitrates.shape
        seqs = np.ascontiguousarray(np.asarray(sequences, dtype=np.float64).astype(np.int32))   # int(r), mpc.py:122
        M, H = seqs.shape
        hist = list(chunk_info.previous_bandwidths)
        if self.predicted_bandwidths is not None and self.strict_history:
            n_pred = len(self.predicted_bandwidths)
            if len(hist) >= n_pred and hist[-n_pred:] == list(self.predicted_bandwidths):
                hist = hist[:-n_pred]
        hist = np.ascontiguousarray(hist, dtype=np.float64)
        if hist.size == 0 or np.any(hist == 0.0):
            raise ZeroDivisionError("division by zero")
        chunk = getattr(chunk_info, "chunk_number", None)
        if chunk is None:
            chunk = chunk_info.chunk_id
        if chunk + H > V:
            raise IndexError("list index out of range")
        prev = getattr(chunk_info, "previous_bitrate", None)
        if prev is None:
            prev = chunk_info.previous_bitrates[-1]
        scores = np.empty(M)
        p = self._params()
        _lib.check(lib.abr_mpc_score_host(_addr(sizes), _addr(bitrates), V, A, p, int(chunk), int(prev),
                                          float(chunk_info.buffer_level), _addr(hist), hist.size, H, self.mode, 0.0,
                                          _addr(seqs), M, _addr(scores)))
        return scores

    def score_grid(self, chunk_info):
        """All A^H scores in scipy.optimize.brute's C order (mpc.py:171-179)."""
        A = len(self.mpd.chunks[0].bitrates)
        seqs = list(itertools.product(range(A), repeat=self.horizon))
        return self.objective_batch(seqs, chunk_info)


def decide_batch(sizes, utility, chunk_idx, prev_q, buffer, bw_hist, hist_len, horizon, mode="reference", flags=0,
                 params=None, last_pred=None, err_ring=None, err_len=None, want=("best_j", "best_seq", "preds"),
                 startup=None, n_ts=1, ts_step=0.0):
    """Batched standalone decision over DEVICE tensors (``abr_mpc_decide`` / ``abr_mpc_decide_startup``).

    sizes/utility: [V, A] float64; chunk_idx/prev_q/hist_len: [N] int32; buffer: [N] float64;
    bw_hist: [N, K] float64 ring (SPEC §5).  Returns dict(action, best_j, best_seq, preds, errors).
    ``flags``: ``MPC_TRUNCATE | MPC_EMPTY_DEFAULT | MPC_PRED_SES``.  ``n_ts > 1``: start-up phase (SPEC §5.3) for the
    sessions with ``startup`` != 0 ([N] uint8, None = all); the result then carries ``startup_delay`` [N].
    """
    import torch
    from .env import _stream, _mode_id
    lib = _lib.load()
    V, A = sizes.shape
    N, K = bw_hist.shape
    dev = sizes.device
    p = params if params is not None else _lib.default_params()
    out = dict(action=torch.empty(N, dtype=torch.int32, device=dev),
               errors=torch.zeros(1, dtype=torch.int32, device=dev))
    if "best_j" in want:
        out["best_j"] = torch.empty(N, dtype=torch.float64, device=dev)
    if "best_seq" in want:
        out["best_seq"] = torch.empty(N, horizon, dtype=torch.int32, device=dev)
    if "preds" in want:
        out["preds"] = torch.empty(N, horizon, dtype=torch.float64, device=dev)
    for t in (sizes, utility, chunk_idx, prev_q, buffer, bw_hist, hist_len):
        if not t.is_contiguous():
            raise ValueError("tensors must be contiguous")
    head = (_addr(sizes), _addr(utility), V, A, p, N, _addr(chunk_idx), _addr(prev_q), _addr(buffer), _addr(bw_hist),
            _addr(hist_len), K, _addr(last_pred), _addr(err_ring), _addr(err_len), horizon, _mode_id(mode), flags)
    tail = (_addr(out.get("best_j")), _addr(out.get("best_seq")), _addr(out.get("preds")), _addr(out["errors"]), _stream())
    with torch.cuda.device(dev):
        if n_ts > 1:
            out["startup_delay"] = torch.empty(N, dtype=torch.float64, device=dev)
            if startup is not None and (startup.dtype != torch.uint8 or not startup.is_contiguous() or startup.numel() != N):
                raise ValueError("startup must be a contiguous uint8 tensor [N]")
            _lib.check(lib.abr_mpc_decide_startup(*head, _addr(startup), int(n_ts), float(ts_step), _addr(out["action"]),
                                                  _addr(out["startup_delay"]), *tail))
        else:
            _lib.check(lib.abr_mpc_decide(*head, _addr(out["action"]), *tail))
    return out
