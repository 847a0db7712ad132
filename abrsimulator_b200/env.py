"""Batched ABR environment: N independent streaming sessions stepped on one B200.

Host-side mirror of the reference's environment API (``Simulator.py:45-210``): construct from
bandwidth traces and per-bitrate chunk sizes, step with a bitrate index, get back download delay /
sleep / buffer / rebuffer / reward / next-chunk sizes / end-of-video.  All arithmetic happens in
the sm_100a kernels behind the C-ABI of ``include/abr_b200.h`` (semantics: SPEC.md); PyTorch is
used only for device memory and streams.  There is no CPU fallback.
"""
from __future__ import annotations

from collections import namedtuple

import numpy as np
import torch

from . import _lib
from ._lib import (AbrError, MPC_REF, MPC_ROBUST, NUM_ACC, NUM_STATS, POLICY_BBA, POLICY_BOLA,  # noqa: F401
                   POLICY_FIXED, POLICY_RANDOM, POLICY_RATE, _addr)
from .datamodel import MPD, NetworkInfo, QOEMetric, pack_traces

StepResult = namedtuple("StepResult", "delay sleep buffer rebuffer reward next_sizes end_of_video throughput latency",
                        defaults=(None,))

_POLICIES = {"fixed": POLICY_FIXED, "random": POLICY_RANDOM, "bba": POLICY_BBA, "buffer": POLICY_BBA,
             "rate": POLICY_RATE, "rb": POLICY_RATE, "bola": POLICY_BOLA}
_MODES = {"reference": MPC_REF, "ref": MPC_REF, "robust": MPC_ROBUST}


def _policy_id(policy):
    if isinstance(policy, str):
        return _POLICIES[policy]
    return int(policy)


def _mode_id(mode):
    if isinstance(mode, str):
        return _MODES[mode]
    return int(mode)


class _DevPtr:
    """Minimal __cuda_array_interface__ holder so torch can view library-owned device memory."""

    def __init__(self, ptr, shape, typestr, strides=None):
        self.__cuda_array_interface__ = dict(shape=tuple(shape), typestr=typestr, data=(int(ptr), False),
                                             version=3, strides=strides)


_TYPESTR = {"int32": "<i4", "uint8": "|u1", "float64": "<f8"}
_ITEMSIZE = {"int32": 4, "uint8": 1, "float64": 8}


def _stream():
    return torch.cuda.current_stream().cuda_stream


class _OnDevice:
    """``with torch.cuda.device(dev)`` that costs nothing when `dev` is already current (the usual one-process-per-GPU
    case): the per-call overhead of env.step matters when the kernel itself takes 25 us."""
    __slots__ = ("index", "prev")

    def __init__(self, device):
        self.index = device.index if device.index is not None else torch.cuda.current_device()
        self.prev = -1

    def __enter__(self):
        cur = torch.cuda.current_device()
        if cur != self.index:
            self.prev = cur
            torch.cuda.set_device(self.index)
        return self

    def __exit__(self, *exc):
        if self.prev >= 0:
            torch.cuda.set_device(self.prev)
            self.prev = -1
        return False


class HostRun:
    """A prepared ``abr_env_run_host`` call (``BatchedABREnv.prepare_run_host``).  ``run(seed=None)`` executes it on
    the stream that is current at that moment and returns the output dict; the input and output buffers are the ones
    given at preparation (kept alive here), so new inputs are written into them in place."""
    __slots__ = ("env", "args", "out", "keep", "fn", "n", "session_base")

    def __init__(self, env, args, out, keep):
        self.env, self.args, self.out, self.keep = env, args, out, keep
        self.fn = env._run_host
        self.n, self.session_base = args[6], int(args[7])

    def __call__(self, seed=None):
        a = self.args
        if seed is not None:
            a[2] = seed
        a[13] = torch.cuda.current_stream().cuda_stream
        env = self.env
        with env._on:
            rc = self.fn(*a)
        if rc:
            _lib.check(rc)
        env.n, env.session_base = self.n, self.session_base
        return self.out

    run = __call__


def _host(x, np_dtype, torch_dtype):
    """A contiguous host buffer of the given element type: CPU torch tensors and matching numpy arrays pass through."""
    if isinstance(x, torch.Tensor):
        if x.device.type != "cpu" or x.dtype != torch_dtype or not x.is_contiguous():
            raise TypeError(f"host tensors must be contiguous CPU {torch_dtype} (got {x.dtype} on {x.device})")
        return x
    return np.ascontiguousarray(x, dtype=np_dtype)


def _check_host_out(a, size, name):
    if a is None:
        return
    if isinstance(a, torch.Tensor):
        ok = a.device.type == "cpu" and a.dtype == torch.float64 and a.is_contiguous() and a.numel() == size
    else:
        ok = a.dtype == np.float64 and a.flags.c_contiguous and a.flags.writeable and a.size == size
    if not ok:
        raise TypeError(f"output {name!r} must be a contiguous host float64 buffer of {size} elements")


def _out_dtype(t, dtype):
    """float64 or float32: the dtype of a caller-given output tensor, else the requested one."""
    d = dtype if t is None else t.dtype
    if d not in (torch.float64, torch.float32):
        raise TypeError(f"outputs are float64 or float32 (got {d})")
    return d


def _float_rows(t, name, device):
    if not isinstance(t, torch.Tensor) or t.device != device or t.dtype not in (torch.float64, torch.float32):
        raise TypeError(f"{name} must be a float64 or float32 tensor on {device}")
    return t


class BatchedABREnv:
    """N sessions over shared trace / video tables.

    Parameters
    ----------
    trace_bw : [n_traces, T_max] float64 (host) — bandwidth per segment, same units as sizes/second
    trace_len : [n_traces] int (default: T_max for every trace)
    trace_interval : scalar or [n_traces] — segment duration in seconds (``NetworkInfo.interval``)
    sizes, bitrates : [V, A] float64 — per-chunk payload and ladder (``Chunk.sizes`` / ``Chunk.bitrates``)
    max_sessions : capacity of the SoA state
    **params : fields of ``AbrParams`` (chunk_length, max_buffer, rtt, payload, ...)
    """

    def __init__(self, trace_bw, sizes, bitrates, max_sessions, trace_len=None, trace_interval=1.0,
                 device=None, **params):
        if not torch.cuda.is_available():
            raise RuntimeError("BatchedABREnv needs a CUDA device (B200); there is no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self._on = _OnDevice(self.device)
        self._lib = _lib.load()
        self._run_host = self._lib.abr_env_run_host
        bw = np.ascontiguousarray(trace_bw, dtype=np.float64)
        if bw.ndim == 1:
            bw = bw[None, :]
        self.n_traces, self.T_max = bw.shape
        tl = np.full(self.n_traces, self.T_max, np.int32) if trace_len is None else \
            np.ascontiguousarray(trace_len, dtype=np.int32)
        ti = np.ascontiguousarray(np.broadcast_to(np.asarray(trace_interval, dtype=np.float64), (self.n_traces,)))
        sz = np.ascontiguousarray(sizes, dtype=np.float64)
        br = np.ascontiguousarray(bitrates, dtype=np.float64)
        if sz.shape != br.shape or sz.ndim != 2:
            raise ValueError("sizes and bitrates must both be [V, A]")
        self.V, self.A = sz.shape
        self.params = _lib.default_params(**params)
        self.K = int(self.params.hist_k)
        self.capacity = int(max_sessions)
        self.n = 0
        self.perm = None          # installed session order (set_order), environment position -> caller's index
        self._inv_perm = None
        self._h = None
        h = np.zeros(1, np.uintp)
        with self._on:
            _lib.check(self._lib.abr_env_create(_addr(bw), _addr(tl), _addr(ti), self.n_traces, self.T_max, _addr(sz),
                                                _addr(br), self.V, self.A, self.params, self.capacity, _addr(h)))
        self._h = int(h[0])
        self._stats = torch.empty(NUM_STATS, dtype=torch.float64, device=self.device)

    # -- construction from the reference's objects (Simulator.set_network_info / set_mpd / set_qoe_metric) --
    @classmethod
    def from_objects(cls, network_infos, mpd: MPD, qoe: QOEMetric = None, max_sessions=1, **params):
        if isinstance(network_infos, NetworkInfo):
            network_infos = [network_infos]
        bw, tl, ti = pack_traces(network_infos)
        bitrates, sizes = mpd.tables()
        kw = dict(chunk_length=float(mpd.chunk_length), max_buffer=float(mpd.max_buffer))
        if qoe is not None:
            kw.update(rebuf_penalty=float(qoe.rebuffer_weight), smooth_penalty=float(qoe.variance_weight))
        kw.update(params)
        return cls(bw, sizes, bitrates, max_sessions, trace_len=tl, trace_interval=ti, **kw)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.abr_env_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- helpers --
    def _dev(self, x, dtype):
        if isinstance(x, torch.Tensor):
            return x.to(device=self.device, dtype=dtype).contiguous()
        return torch.as_tensor(np.ascontiguousarray(x), dtype=dtype).to(self.device)

    def _empty(self, *shape, dtype=torch.float64):
        return torch.empty(*shape, dtype=dtype, device=self.device)

    def _speed_table(self, speed, n):
        """[V, N] float64 device table from a [V, N] table or a per-session vector [N]."""
        v = self._dev(speed, torch.float64)
        if v.dim() == 1 and v.numel() == n:
            v = v.unsqueeze(0).expand(self.V, n).contiguous()
        if v.numel() != self.V * n:
            raise ValueError(f"speed must be [V, N] = [{self.V}, {n}] (or [N]): the playback speed of each content chunk")
        return v

    # -- SPEC §2 --
    # -- session order (sessions are independent, so the environment may keep them sorted by trace) --
    def sort_by_trace(self, trace_id) -> torch.Tensor:
        """``perm`` (int32 [N], device): ``perm[p]`` = caller's index of the session that a trace-sorted environment
        keeps at position ``p`` (stable, deterministic; ``abr_sort_by_trace``)."""
        tid = self._dev(trace_id, torch.int32)
        perm = self._empty(tid.numel(), dtype=torch.int32)
        with self._on:
            _lib.check(self._lib.abr_sort_by_trace(_addr(tid), tid.numel(), self.n_traces, _addr(perm), _stream()))
        return perm

    def set_order(self, perm):
        """Install (``perm`` int32 [N]) or remove (None) the session order.  Afterwards every per-session array passed
        to or returned by this environment is in environment order: element ``p`` is the caller's session ``perm[p]``
        (``to_caller_order`` maps results back); the random policy stays keyed by the caller's index."""
        self.perm = None if perm is None else self._dev(perm, torch.int32)
        self._inv_perm = None
        with self._on:
            _lib.check(self._lib.abr_env_set_order(self._h, _addr(self.perm),
                                                   0 if self.perm is None else self.perm.numel(), _stream()))

    def to_env_order(self, x):
        """Caller-order array(s) [..., N] -> environment order (identity without an installed order)."""
        if self.perm is None:
            return x
        return torch.as_tensor(x).to(self.device).index_select(-1, self.perm.long())

    def to_caller_order(self, x):
        """Environment-order result [..., N] -> the caller's session order."""
        if self.perm is None:
            return x
        if self._inv_perm is None:
            self._inv_perm = torch.empty_like(self.perm, dtype=torch.int64)
            self._inv_perm[self.perm.long()] = torch.arange(self.perm.numel(), device=self.device)
        return x.index_select(-1, self._inv_perm)

    def reset(self, trace_id, start_offset=None, session_base=0, sort_by_trace=False):
        """SPEC §2.  ``sort_by_trace=True``: the sessions are given in the caller's order; the environment sorts them
        by trace (``sort_by_trace`` + ``set_order``) and keeps them in that order — see ``set_order``."""
        tid = self._dev(trace_id, torch.int32)
        off = None if start_offset is None else self._dev(start_offset, torch.float64)
        n = tid.numel()
        if off is not None and off.numel() != n:
            raise ValueError("start_offset must have one entry per session")
        if sort_by_trace:      # one call: counting sort by trace + gather of the inputs + reset (abr_env_reset_sorted)
            with self._on:
                _lib.check(self._lib.abr_env_reset_sorted(self._h, _addr(tid), _addr(off), n, session_base, _stream()))
            self.n = n
            self.session_base = int(session_base)
            self.perm, self._inv_perm = self.state("order"), None    # a view of the environment's own copy
            return
        with self._on:
            _lib.check(self._lib.abr_env_reset(self._h, _addr(tid), _addr(off), n, session_base, _stream()))
        self.n = n
        self.session_base = int(session_base)

    # -- SPEC §3 --
    def step(self, action, want_next_sizes=True, want_throughput=False, out=None, speed=None,
             want_latency=None, dtype=torch.float64) -> StepResult:
        """One chunk step for every session.  ``action``: int32 [N] on the device (or array-like).
        Live mode (``live=1``, SPEC §7): ``speed`` is the playback-speed table [V, N] — ``speed[k, s]`` is the speed
        at which session ``s`` plays content chunk ``k`` (the reference asks its speed controller once per played
        chunk, ``Simulator.py:176-177``); a vector [N] means one speed per session for every chunk; default 1.0.
        The result carries ``latency`` and ``sleep`` is the idle time before the download.
        ``dtype=torch.float32`` selects the optional fp32-output mode: the arithmetic and the state stay fp64, the
        outputs are rounded once to float (``abr_env_step_f32``)."""
        a = self._dev(action, torch.int32)
        if a.numel() != self.n:
            raise ValueError(f"action has {a.numel()} entries for {self.n} sessions")
        n = self.n
        live = bool(self.params.live)
        v = None
        if speed is not None:
            if not live:
                raise ValueError("speed is a live-mode action (create the environment with live=1)")
            v = self._speed_table(speed, n)
        if want_latency is None:
            want_latency = live
        if out is None:
            e = lambda *shape: self._empty(*shape, dtype=dtype)
            out = StepResult(e(n), e(n), e(n), e(n), e(n), e(n, self.A) if want_next_sizes else None,
                             self._empty(n, dtype=torch.uint8), e(n) if want_throughput else None,
                             e(n) if want_latency else None)
        fn = self._lib.abr_env_step_live if _out_dtype(out.delay, dtype) == torch.float64 else self._lib.abr_env_step_f32
        with self._on:
            _lib.check(fn(
                self._h, _addr(a), _addr(v), _addr(out.delay), _addr(out.sleep), _addr(out.buffer), _addr(out.rebuffer),
                _addr(out.reward), _addr(out.latency), _addr(out.next_sizes), _addr(out.end_of_video),
                _addr(out.throughput), _stream()))
        return out

    # -- SPEC §4.1: policy in the loop (RL harness) --
    def step_policy(self, logits, sample=True, seed=0, obs=None, action_out=None, reward_sum=None, out=None,
                    obs_scales=(1.0, 1.0, 1.0, 1.0)):
        """One chunk step with the action chosen inside the step kernel from the policy's ``logits`` (float32 [N, A] on
        the device): arg max, or with ``sample`` a draw from softmax(logits) (Gumbel-max, Philox noise keyed by the seed,
        the global session index and the environment's draw counter, which every sampled call advances and ``reset``
        zeroes).  The same kernel writes the next observation into ``obs`` (float32 [4 + A, N], feature-major: buffer,
        throughput, delay — each times its entry of ``obs_scales`` = (buffer, throughput, delay, size) — action / A,
        and the scaled sizes of the next chunk), the chosen action into ``action_out`` (int32 [N]) and adds the reward
        into ``reward_sum`` (float64 [N]).  ``out``: an optional StepResult whose delay / sleep / buffer / rebuffer /
        reward / end_of_video tensors receive the per-step outputs.  All arguments are used in place (graph-capturable);
        returns ``obs``."""
        n = self.n
        if logits.dtype != torch.float32 or logits.device != self.device or not logits.is_contiguous() or \
                logits.numel() != n * self.A:
            raise TypeError(f"logits must be a contiguous float32 [N, A] = [{n}, {self.A}] tensor on {self.device}")

        def chk(t, dtype, size, name):
            if t is not None and (t.dtype != dtype or t.device != self.device or not t.is_contiguous() or t.numel() != size):
                raise TypeError(f"{name} must be a contiguous {dtype} tensor of {size} elements on {self.device}")

        chk(obs, torch.float32, (4 + self.A) * n, "obs")
        chk(action_out, torch.int32, n, "action_out")
        chk(reward_sum, torch.float64, n, "reward_sum")
        spec = self._obs_spec = _lib.AbrObsSpec(*[float(x) for x in obs_scales])
        o = out
        for name in ("delay", "sleep", "buffer", "rebuffer", "reward") if o is not None else ():
            chk(getattr(o, name), torch.float64, n, name)
        if o is not None:
            chk(o.end_of_video, torch.uint8, n, "end_of_video")
        g = (lambda name: _addr(getattr(o, name))) if o is not None else (lambda name: None)
        with self._on:
            _lib.check(self._lib.abr_env_step_policy(
                self._h, _addr(logits), int(bool(sample)), int(seed), spec, _addr(obs),
                _addr(action_out), _addr(reward_sum), g("delay"), g("sleep"), g("buffer"), g("rebuffer"),
                g("reward"), g("end_of_video"), _stream()))
        return obs

    # -- SPEC §4.5: the windowed (Pensieve-style) observation --
    def _window_spec(self, window, scales):
        if not 1 <= int(window) <= 32:
            raise ValueError(f"window must be in [1, 32] (got {window})")
        if len(scales) != 5:
            raise ValueError("scales are (util, buffer, throughput, delay, size)")
        return _lib.AbrObsWindowSpec(int(window), *[float(x) for x in scales])

    def observe_window(self, window=8, scales=(1.0,) * 5, obs=None):
        """The windowed observation of the current state (float32 [3 + 2W + A, N], feature-major, W = ``window``) with
        both windows 0: the first observation of an episode, or a restart of the windows.  Rows: the last chunk's
        utility, the buffer, the chunks left / V, the last W throughputs, the last W download times (oldest first)
        and the next chunk's sizes, each times its entry of ``scales`` = (util, buffer, throughput, delay, size)
        (the chunks left are not scaled).  ``obs``: written in place when given."""
        spec = self._window_spec(window, scales)
        n, F = self.n, 3 + 2 * int(window) + self.A
        if obs is None:
            obs = self._empty(F, n, dtype=torch.float32)
        self._check_window_obs(obs, F, n)
        with self._on:
            _lib.check(self._lib.abr_env_observe_window(self._h, spec, _addr(obs), _stream()))
        return obs

    def _check_window_obs(self, obs, F, n):
        if obs.dtype != torch.float32 or obs.device != self.device or not obs.is_contiguous() or \
                tuple(obs.shape) != (F, n):
            raise TypeError(f"obs must be a contiguous float32 [3 + 2W + A, N] = [{F}, {n}] tensor on {self.device}")

    def step_policy_window(self, logits, obs, sample=True, seed=0, scales=(1.0,) * 5, action_out=None,
                           reward_sum=None, out=None):
        """``step_policy`` with the windowed observation of ``observe_window``: ``obs`` (float32 [3 + 2W + A, N],
        W = (rows - 3 - A) / 2) holds the two windows from one call to the next and is updated in place: each step
        moves them up one entry and appends its throughput and download time, a step that ends the video with
        auto_reset zeroes them, and an inert step (a done session, auto_reset=0) leaves them.  Action, per-step
        outputs, ``action_out``, ``reward_sum`` and the state are those of ``step_policy``.  All arguments are used in
        place (graph-capturable); returns ``obs``."""
        n = self.n
        if logits.dtype != torch.float32 or logits.device != self.device or not logits.is_contiguous() or \
                logits.numel() != n * self.A:
            raise TypeError(f"logits must be a contiguous float32 [N, A] = [{n}, {self.A}] tensor on {self.device}")
        if obs is None or obs.dim() != 2 or (obs.shape[0] - 3 - self.A) % 2 or obs.shape[0] < 5 + self.A:
            raise TypeError(f"obs must be a float32 [3 + 2W + A, N] tensor with W in [1, 32] (A = {self.A})")
        W = (obs.shape[0] - 3 - self.A) // 2
        spec = self._window_spec(W, scales)
        self._check_window_obs(obs, obs.shape[0], n)

        def chk(t, dtype, size, name):
            if t is not None and (t.dtype != dtype or t.device != self.device or not t.is_contiguous() or t.numel() != size):
                raise TypeError(f"{name} must be a contiguous {dtype} tensor of {size} elements on {self.device}")

        chk(action_out, torch.int32, n, "action_out")
        chk(reward_sum, torch.float64, n, "reward_sum")
        o = out
        for name in ("delay", "sleep", "buffer", "rebuffer", "reward") if o is not None else ():
            chk(getattr(o, name), torch.float64, n, name)
        if o is not None:
            chk(o.end_of_video, torch.uint8, n, "end_of_video")
        g = (lambda name: _addr(getattr(o, name))) if o is not None else (lambda name: None)
        with self._on:
            _lib.check(self._lib.abr_env_step_policy_window(
                self._h, _addr(logits), int(bool(sample)), int(seed), spec, _addr(obs),
                _addr(action_out), _addr(reward_sum), g("delay"), g("sleep"), g("buffer"), g("rebuffer"),
                g("reward"), g("end_of_video"), _stream()))
        return obs

    # -- SPEC §3+§4 --
    def rollout(self, policy, steps, seed=0, actions=None, want=("delay", "sleep", "buffer", "rebuffer", "reward",
                                                                "end_of_video", "actions"), out=None, speed=None,
                dtype=torch.float64):
        """`steps` chunk steps in one fused launch.  Returns a dict of [steps, N] device tensors.  In live mode
        (SPEC §7) ``speed`` is the playback-speed table [V, N] of ``step`` (default 1.0) and "latency" may be wanted.
        ``dtype=torch.float32``: fp32-output mode (fp64 arithmetic, outputs rounded once; 21 B instead of 41 B of
        trajectory per chunk-step)."""
        pid = _policy_id(policy)
        n = self.n
        a_in = None
        if pid == POLICY_FIXED:
            if actions is None:
                raise ValueError("policy 'fixed' needs an actions table [steps, N]")
            a_in = self._dev(actions, torch.int32)
            if a_in.numel() != steps * n:
                raise ValueError("actions must be [steps, N]")
        v = None
        if speed is not None:
            if not self.params.live:
                raise ValueError("speed is a live-mode action (create the environment with live=1)")
            v = self._speed_table(speed, n)
        if out is None:
            out = {}
            for k in want:
                dt = torch.uint8 if k == "end_of_video" else torch.int32 if k == "actions" else dtype
                out[k] = self._empty(steps, n, dtype=dt)
        fp = [t for k, t in out.items() if k not in ("end_of_video", "actions") and t is not None]
        f32 = _out_dtype(fp[0] if fp else None, dtype) == torch.float32
        if any(t.dtype != (torch.float32 if f32 else torch.float64) for t in fp):
            raise TypeError("all floating-point outputs must share one dtype (float64, or float32 for the fp32-output mode)")
        fn = self._lib.abr_env_rollout_fused_f32 if f32 else self._lib.abr_env_rollout_fused_live
        with self._on:
            _lib.check(fn(
                self._h, pid, seed, steps, _addr(a_in), _addr(v), _addr(out.get("delay")), _addr(out.get("sleep")),
                _addr(out.get("buffer")), _addr(out.get("rebuffer")), _addr(out.get("reward")), _addr(out.get("latency")),
                _addr(out.get("end_of_video")), _addr(out.get("actions")), _stream()))
        return out

    # -- SPEC §2+§3+§4+§6 in one launch --
    def run(self, policy, steps, trace_id, start_offset=None, seed=0, session_base=0, actions=None,
            want=("delay", "sleep", "buffer", "rebuffer", "reward", "end_of_video"), out=None, qoe_cost=None,
            stats=None):
        """One whole run, device-resident (``abr_env_run``): reset + `steps` chunk steps + per-session QoE cost +
        statistics in one kernel launch; the episode kernel resets the sessions itself and reduces the statistics.  ``trace_id`` / ``start_offset``: device tensors
        (or array-likes).  ``out``: dict of [steps, N] float64 device tensors as for ``rollout``; ``qoe_cost`` [N] and
        ``stats`` [NUM_STATS] are allocated when None (pass False to skip).  Returns (out, qoe_cost, stats)."""
        pid = _policy_id(policy)
        tid = self._dev(trace_id, torch.int32)
        n = tid.numel()
        off = None if start_offset is None else self._dev(start_offset, torch.float64)
        if off is not None and off.numel() != n:
            raise ValueError("start_offset must have one entry per session")
        a_in = None
        if pid == POLICY_FIXED:
            if actions is None:
                raise ValueError("policy 'fixed' needs an actions table [steps, N]")
            a_in = self._dev(actions, torch.int32)
            if a_in.numel() != steps * n:
                raise ValueError("actions must be [steps, N]")
        if out is None:
            out = {}
            for k in want:
                dt = torch.uint8 if k == "end_of_video" else torch.int32 if k == "actions" else torch.float64
                out[k] = self._empty(steps, n, dtype=dt)
        for k, t in out.items():
            if t is not None and k not in ("end_of_video", "actions") and t.dtype != torch.float64:
                raise TypeError("run() outputs are float64")
        qoe_cost = self._empty(n) if qoe_cost is None else (None if qoe_cost is False else qoe_cost)
        stats = self._empty(NUM_STATS) if stats is None else (None if stats is False else stats)
        g = out.get
        with self._on:
            _lib.check(self._lib.abr_env_run(
                self._h, pid, seed, steps, _addr(tid), _addr(off), n, session_base, _addr(a_in), _addr(g("delay")),
                _addr(g("sleep")), _addr(g("buffer")), _addr(g("rebuffer")), _addr(g("reward")),
                _addr(g("end_of_video")), _addr(g("actions")), _addr(qoe_cost), _addr(stats), _stream()))
        self.n = n
        self.session_base = int(session_base)
        return out, qoe_cost, stats

    # -- SPEC §4.2 / §4.3 --
    def set_policy_params(self, rb_safety=None, bola_min_buffer=None, bola_target_buffer=None):
        """Parameters of the "rate" and "bola" policies (SPEC §4.2, §4.3) for the following calls; arguments left at
        None keep their current value (defaults: 1.0, 10 s, 30 s).  Invalid values raise before anything changes."""
        cur = getattr(self, "_policy_params", None)
        if cur is None:
            cur = _lib.AbrPolicyParams()
            self._lib.abr_policy_params_default(cur)
        pp = _lib.AbrPolicyParams(cur.rb_safety if rb_safety is None else float(rb_safety),
                                  cur.bola_min_buffer if bola_min_buffer is None else float(bola_min_buffer),
                                  cur.bola_target_buffer if bola_target_buffer is None else float(bola_target_buffer))
        _lib.check(self._lib.abr_env_set_policy_params(self._h, pp))
        self._policy_params = pp

    def policy_decide(self, policy, out=None) -> torch.Tensor:
        """The action of a state-dependent built-in policy ("bba", "rate" or "bola") for every session, from the
        environment's own state (int32 [N] on the device); ``step`` with it is one step of the fused episode."""
        pid = _policy_id(policy)
        act = self._empty(self.n, dtype=torch.int32) if out is None else out
        if act.dtype != torch.int32 or act.device != self.device or not act.is_contiguous() or act.numel() != self.n:
            raise TypeError(f"out must be a contiguous int32 tensor of {self.n} elements on {self.device}")
        with self._on:
            _lib.check(self._lib.abr_env_policy_decide(self._h, pid, _addr(act), _stream()))
        return act

    # -- SPEC §5 --
    def mpc_decide(self, horizon=5, mode="robust", want_score=False, out=None, exhaustive=False):
        """MPC decision for every session (SPEC §5).  ``exhaustive``: evaluate all A^H sequences like the reference's
        ``scipy.optimize.brute`` instead of skipping the partial sequences whose bound already loses (robust mode's
        branch and bound; the decisions and objective values are identical either way)."""
        act = self._empty(self.n, dtype=torch.int32) if out is None else out
        bj = self._empty(self.n) if want_score else None
        mode_id = _mode_id(mode) | (_lib.MPC_MODE_EXHAUSTIVE if exhaustive else 0)
        with self._on:
            _lib.check(self._lib.abr_env_mpc_decide(self._h, horizon, mode_id, _addr(act), _addr(bj), _stream()))
        return (act, bj) if want_score else act

    def mpc_episode(self, steps, horizon=5, mode="robust", exhaustive=False):
        """decide -> step for `steps` chunks (needs track_history=1, track_acc=1 for statistics)."""
        act = self._empty(self.n, dtype=torch.int32)
        for _ in range(steps):
            self.mpc_decide(horizon, mode, out=act, exhaustive=exhaustive)
            with self._on:
                _lib.check(self._lib.abr_env_step(self._h, _addr(act), None, None, None, None, None, None, None, None,
                                                  _stream()))   # live mode: speed 1.0
        return act

    # -- SPEC §5.6 --
    def mpc_decide_pred(self, predictions, horizon=5, want_score=False, want_seq=False, out=None, exhaustive=False):
        """Robust MPC decision (SPEC §5.6) over the caller's throughput predictions instead of the built-in predictor:
        ``predictions`` is a device tensor [N] (one throughput for every step) or [N, horizon] (step i of session s at
        [s, i]), float64 or float32 (widened exactly), in environment order.  Only the first min(horizon, V - chunk)
        entries of a row are read; a session with one that is not finite and > 0 gets action -1 and counts as an
        error.  Reads no history ring (no track_history needed) and writes no state.  Returns the int32 [N] actions, or
        a tuple with the float64 [N] objective values J and / or the int32 [N, horizon] best sequences (-1 past the
        end of the video)."""
        act = self._empty(self.n, dtype=torch.int32) if out is None else out
        if act.dtype != torch.int32 or act.device != self.device or not act.is_contiguous() or act.numel() != self.n:
            raise TypeError(f"out must be a contiguous int32 tensor of {self.n} elements on {self.device}")
        p = predictions
        if not isinstance(p, torch.Tensor) or p.device != self.device or p.dtype not in (torch.float64, torch.float32):
            raise TypeError(f"predictions must be a float64 or float32 tensor on {self.device}")
        H = int(horizon)
        if p.dim() == 1 and p.shape[0] == self.n:
            p = p.unsqueeze(1).expand(self.n, H)
        if tuple(p.shape) != (self.n, H):
            raise ValueError(f"predictions must be [N] or [N, horizon] = [{self.n}, {H}] (got {tuple(p.shape)})")
        p = p.to(torch.float64).contiguous()
        bj = self._empty(self.n) if want_score else None
        seq = self._empty(self.n, H, dtype=torch.int32) if want_seq else None
        flags = _lib.MPC_EXHAUSTIVE if exhaustive else 0
        with self._on:
            _lib.check(self._lib.abr_env_mpc_decide_pred(self._h, H, flags, _addr(p), _addr(act), _addr(bj),
                                                         _addr(seq), _stream()))
        if not (want_score or want_seq):
            return act
        return (act,) + ((bj,) if want_score else ()) + ((seq,) if want_seq else ())

    def mpc_episode_pred(self, steps, predictor, horizon=5, exhaustive=False):
        """``predictor(env)`` -> mpc_decide_pred -> step for `steps` chunks (track_acc=1 for the per-session sums).
        ``predictor`` returns the [N] or [N, horizon] device predictions for the current state.  Nothing here
        synchronises with the host, so one chunk can be captured in a CUDA graph when the predictor allows it."""
        act = self._empty(self.n, dtype=torch.int32)
        for _ in range(steps):
            self.mpc_decide_pred(predictor(self), horizon, out=act, exhaustive=exhaustive)
            with self._on:
                _lib.check(self._lib.abr_env_step(self._h, _addr(act), None, None, None, None, None, None, None, None,
                                                  _stream()))   # live mode: speed 1.0
        return act

    # -- SPEC §5.7 --
    def mpc_decide_scen(self, scenarios, horizon=5, weights=None, objective="mean", want_score=False, want_seq=False,
                        out=None, exhaustive=False):
        """MPC decision (SPEC §5.7) over K caller-supplied throughput scenarios: the sequence whose SPEC §5.2
        objective values under the scenarios have the best weighted mean (``objective="mean"``) or the best worst case
        (``"worst"``).  ``scenarios`` is a device tensor [N, K, horizon] (scenario k of session s at [s, k]), or
        [N, K] for one throughput per scenario at every step, float64 or float32 (widened exactly), 1 <= K <= 16, in
        environment order.  ``weights`` [N, K] (mean only; None: 1/K each).  Only the first min(horizon, V - chunk)
        steps are read; a session with a throughput that is not finite and > 0, a weight that is not finite and >= 0,
        or only zero weights gets action -1 and counts as an error.  Reads no history ring and writes no state.
        Returns like ``mpc_decide_pred``."""
        act = self._empty(self.n, dtype=torch.int32) if out is None else out
        if act.dtype != torch.int32 or act.device != self.device or not act.is_contiguous() or act.numel() != self.n:
            raise TypeError(f"out must be a contiguous int32 tensor of {self.n} elements on {self.device}")
        objs = dict(mean=_lib.MPC_SCEN_MEAN, worst=_lib.MPC_SCEN_WORST)
        if objective not in objs:
            raise ValueError(f"objective must be 'mean' or 'worst' (got {objective!r})")
        H = int(horizon)
        p = _float_rows(scenarios, "scenarios", self.device)
        if p.dim() == 2 and p.shape[0] == self.n:
            p = p.unsqueeze(2).expand(self.n, p.shape[1], H)
        if p.dim() != 3 or p.shape[0] != self.n or p.shape[2] != H:
            raise ValueError(f"scenarios must be [N, K] or [N, K, horizon] with N = {self.n}, horizon = {H} "
                             f"(got {tuple(p.shape)})")
        K = p.shape[1]
        p = p.to(torch.float64).contiguous()
        w = None
        if weights is not None:
            w = _float_rows(weights, "weights", self.device)
            if tuple(w.shape) != (self.n, K):
                raise ValueError(f"weights must be [N, K] = [{self.n}, {K}] (got {tuple(w.shape)})")
            w = w.to(torch.float64).contiguous()
        bj = self._empty(self.n) if want_score else None
        seq = self._empty(self.n, H, dtype=torch.int32) if want_seq else None
        flags = _lib.MPC_EXHAUSTIVE if exhaustive else 0
        with self._on:
            _lib.check(self._lib.abr_env_mpc_decide_scen(self._h, H, K, objs[objective], flags, _addr(p), _addr(w),
                                                         _addr(act), _addr(bj), _addr(seq), _stream()))
        if not (want_score or want_seq):
            return act
        return (act,) + ((bj,) if want_score else ()) + ((seq,) if want_seq else ())

    def mpc_episode_scen(self, steps, sampler, horizon=5, objective="mean", exhaustive=False):
        """``sampler(env)`` -> mpc_decide_scen -> step for `steps` chunks (track_acc=1 for the per-session sums).
        ``sampler`` returns the scenarios ([N, K] or [N, K, horizon] on the device) or a pair (scenarios, weights)
        for the current state.  Nothing here synchronises with the host, so one chunk can be captured in a CUDA graph
        when the sampler allows it."""
        act = self._empty(self.n, dtype=torch.int32)
        for _ in range(steps):
            r = sampler(self)
            scen, w = r if isinstance(r, tuple) else (r, None)
            self.mpc_decide_scen(scen, horizon, weights=w, objective=objective, out=act, exhaustive=exhaustive)
            with self._on:
                _lib.check(self._lib.abr_env_step(self._h, _addr(act), None, None, None, None, None, None, None, None,
                                                  _stream()))   # live mode: speed 1.0
        return act

    def throughput_history(self):
        """The throughput samples of every session's history ring, for predictors: ``(x, n)`` with x float64 [N, K]
        oldest first and NaN past the n[s] = min(hist_len, K) samples a session has (int32 [N]).  Needs
        track_history=1.  Gathered on the device from the K-major ring, without a host synchronisation."""
        if not self.params.track_history:
            raise ValueError("throughput_history needs the throughput history: create the environment with "
                             "track_history=1")
        ring, hl = self.state("bw_hist"), self.state("hist_len")      # [K, N] slot-major, [N]
        K = self.K
        n = torch.clamp(hl, max=K)
        start = torch.where(hl <= K, torch.zeros_like(hl), hl % K)  # the oldest sample's slot once the ring wrapped
        j = torch.arange(K, device=self.device, dtype=hl.dtype)
        slot = (start[:, None] + j[None, :]) % K
        x = ring.t().gather(1, slot.long())
        return torch.where(j[None, :] < n[:, None], x, torch.full_like(x, float("nan"))), n

    # -- SPEC §4.4 --
    def lookahead_decide(self, horizon=5, want_value=False, want_seq=False, out=None):
        """Clairvoyant lookahead (SPEC §4.4): for every session, the first action of the bitrate sequence over the next
        min(horizon, V - chunk) chunks with the largest sum of the environment's own rewards against the session's
        actual future trace.  An upper reference that sees the future, not a deployable controller; the state does
        not change.  Returns the int32 [N] actions, or a tuple with the float64 [N] best values and / or the int32
        [N, horizon] best sequences (-1 past the end of the video).  Not available in live mode."""
        act = self._empty(self.n, dtype=torch.int32) if out is None else out
        if act.dtype != torch.int32 or act.device != self.device or not act.is_contiguous() or act.numel() != self.n:
            raise TypeError(f"out must be a contiguous int32 tensor of {self.n} elements on {self.device}")
        val = self._empty(self.n) if want_value else None
        seq = self._empty(self.n, int(horizon), dtype=torch.int32) if want_seq else None
        with self._on:
            _lib.check(self._lib.abr_env_lookahead_decide(self._h, horizon, _addr(act), _addr(val), _addr(seq),
                                                          _stream()))
        if not (want_value or want_seq):
            return act
        return (act,) + ((val,) if want_value else ()) + ((seq,) if want_seq else ())

    def lookahead_episode(self, steps, horizon=5):
        """lookahead_decide -> step for `steps` chunks (track_acc=1 for the per-session sums)."""
        act = self._empty(self.n, dtype=torch.int32)
        for _ in range(steps):
            self.lookahead_decide(horizon, out=act)
            with self._on:
                _lib.check(self._lib.abr_env_step(self._h, _addr(act), None, None, None, None, None, None, None, None,
                                                  _stream()))
        return act

    # -- SPEC §6 --
    def stats(self) -> torch.Tensor:
        """[Σreward, Σrebuffer, Σutility, Σsmooth, Σsleep, Σdelay, steps, episodes, Σstartup, Σlatency integral,
        Σcontent played] (the last three are live-mode sums, SPEC §7)."""
        out = torch.empty(NUM_STATS, dtype=torch.float64, device=self.device)
        with self._on:
            _lib.check(self._lib.abr_stats_partial(self._h, _addr(out), _stream()))
        return out

    def state(self, name) -> torch.Tensor:
        """Zero-copy view of a state field (library-owned device memory)."""
        fid, dt = _lib.FIELDS[name]
        p = np.zeros(1, np.uintp)
        _lib.check(self._lib.abr_env_state_ptr(self._h, fid, _addr(p)))
        cap = self.capacity
        if name in ("bw_hist", "err_ring"):
            shape = (self.K, cap)
        elif name == "acc":
            shape = (NUM_ACC, cap)
        elif name in ("sizes", "utility"):
            shape = (self.V, self.A)
        elif name == "trace_bw":
            shape = (self.n_traces, self.T_max)
        else:
            shape = (cap,)
        t = torch.as_tensor(_DevPtr(p[0], shape, _TYPESTR[dt]), device=self.device)
        if name in ("bw_hist", "err_ring", "acc"):
            return t[:, :self.n]
        if name in ("sizes", "utility", "trace_bw"):
            return t
        return t[:self.n]

    def session_acc(self) -> torch.Tensor:
        """[NUM_ACC, N] per-session sums (rows: reward, rebuffer, utility, smooth, sleep, delay, steps, episodes,
        startup, latency integral over the playing time, content played)."""
        return self.state("acc")

    def qoe_cost(self) -> torch.Tensor:
        """Per-session cost of ``Simulator.calculate_qoe`` (Simulator.py:83-86) from the accumulators, on the device."""
        out = self._empty(self.n)
        with self._on:
            _lib.check(self._lib.abr_env_qoe_cost(self._h, _addr(out), _stream()))
        return out

    def error_count(self) -> int:
        out = np.zeros(1, np.int64)
        with self._on:
            _lib.check(self._lib.abr_env_error_count(self._h, _addr(out), _stream()))
        return int(out[0])

    # -- host-buffer path (what Simulator.run() uses; e2e benchmark leg) --
    def run_host(self, policy, steps, trace_id, start_offset=None, seed=0, session_base=0, actions=None,
                 want_acc=True, want_stats=True, want_reward_traj=False, want_qoe_cost=False, out=None,
                 _prepare=False):
        """Reset + fused episode + statistics with HOST inputs and outputs: numpy arrays or CPU torch tensors
        (int32 / float64, contiguous).  Page-locked buffers (``tensor.pin_memory()``) are read and written by the
        kernels directly, pageable ones through staged copies.
        Returns dict(acc=[NUM_ACC,N], stats=[NUM_STATS], reward=[steps,N], qoe_cost=[N])."""
        pid = _policy_id(policy)
        tid = _host(trace_id, np.int32, torch.int32)
        n = tid.numel() if isinstance(tid, torch.Tensor) else tid.size
        off = None if start_offset is None else _host(start_offset, np.float64, torch.float64)
        a_in = None if actions is None else _host(actions, np.int32, torch.int32)
        size = lambda x: x.numel() if isinstance(x, torch.Tensor) else x.size
        if off is not None and size(off) != n:
            raise ValueError("start_offset must have one entry per session")
        if pid == POLICY_FIXED:
            if a_in is None:
                raise ValueError("policy 'fixed' needs an actions table [steps, N]")
            if size(a_in) != steps * n:
                raise ValueError("actions must be [steps, N]")
        out = {} if out is None else out
        if want_acc and "acc" not in out:
            out["acc"] = np.empty((NUM_ACC, n))
        if want_stats and "stats" not in out:
            out["stats"] = np.empty(NUM_STATS)
        if want_reward_traj and "reward" not in out:
            out["reward"] = np.empty((steps, n))
        if want_qoe_cost and "qoe_cost" not in out:
            out["qoe_cost"] = np.empty(n)
        g = out.get
        for k, size in (("acc", NUM_ACC * n), ("stats", NUM_STATS), ("reward", steps * n), ("qoe_cost", n)):
            _check_host_out(g(k), size, k)
        args = [self._h, pid, seed, steps, _addr(tid), _addr(off), n, session_base, _addr(a_in),
                _addr(g("acc")), _addr(g("stats")), _addr(g("reward")), _addr(g("qoe_cost")), None]
        if _prepare:
            return HostRun(self, args, out, (tid, off, a_in))
        args[13] = _stream()
        with self._on:
            rc = self._run_host(*args)
        if rc:
            _lib.check(rc)
        self.n = n
        self.session_base = int(session_base)
        return out

    def prepare_run_host(self, *args, **kw):
        """``run_host`` with the arguments validated and converted once: returns a ``HostRun``; calling it runs the
        episode on the same buffers (for callers that repeat a run, e.g. a sweep over seeds — the per-call cost of the
        Python façade drops from ~10 us to the ctypes call)."""
        return self.run_host(*args, _prepare=True, **kw)
