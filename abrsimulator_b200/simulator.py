"""``Simulator`` façade: the reference's environment API (``Simulator.py:45-210``) over the GPU kernels.

``Simulator(AbrController, SpeedController)``, ``set_qoe_metric``, ``set_network_info``, ``set_mpd`` and ``run()``
keep their reference signatures.  ``run()`` plays one session (or ``run_batch`` many) at chunk granularity
(SPEC.md §3) and returns the QoE *cost* of ``calculate_qoe`` (``Simulator.py:79-86``):
``rw·rebuffer_time + vw·Σ|Δbitrate| + sw·start_up_time + lw·average_latency``.  When the MPD carries a
``start_up_length`` (the reference's 5-argument ``MPD`` / ``set_mpd``) the session runs in live mode (SPEC.md §7:
live-edge availability gate, start-up latch, playback speed from the speed controller — asked once per *played*
chunk, ``Simulator.py:176-177`` — and the reference's ``average_latency``); with ``start_up_length=None`` it is the
on-demand environment of SPEC.md §3 and the last two terms are 0.

Defaults follow the reference, not the north-star constants of ``BatchedABREnv``: no RTT, no packet-payload factor
(``downloaded_size += bandwidth*dt``, ``Simulator.py:160``), a tick-sized (0.01 s, ``Simulator.py:133``) sleep
quantum, cost in bitrate units with each chunk's own ladder in the variance term (``Simulator.py:81-82``).  In live
mode the façade is the closed form of the reference's loop — ``tests/`` check it against that loop's own output
(``tests/golden/sim_ref_tick_golden.json``); keyword arguments of ``Simulator(...)`` override any of this
(e.g. ``Simulator(ctrl, None, rtt=0.08, payload=0.95, sleep_quantum=0.5)`` for the north-star environment).

Controllers
-----------
* any object with ``get_next_bitrate(chunk_id, previous_bitrates, previous_bandwidths, buffer_level) -> int``
  (the protocol ``Simulator.run`` calls, ``Simulator.py:155``) is driven chunk by chunk through the step kernel;
* the markers ``RandomPolicy(seed)`` / ``BufferBasedPolicy()`` / ``RateBasedPolicy()`` / ``BolaPolicy()`` /
  ``FixedPolicy(actions)`` and this package's ``MPCBitrateController`` run fully on the device (fused episode kernel,
  or decide+step kernels for MPC);
* ``LookaheadPolicy(horizon)`` is the clairvoyant reference of SPEC §4.4 (decide+step kernels, on-demand mode only).
"""
from __future__ import annotations

import numpy as np
import torch

from .datamodel import MPD, NetworkInfo, QOEMetric, load_mpd_file, load_network_trace
from .env import BatchedABREnv
from .mpc import MPCBitrateController
from ._lib import ACC_NAMES, MPC_ROBUST


class RandomPolicy:
    def __init__(self, seed=0):
        self.seed = int(seed)


class BufferBasedPolicy:
    def __init__(self, reservoir=5.0, cushion=10.0):
        self.reservoir, self.cushion = float(reservoir), float(cushion)


class RateBasedPolicy:
    """Rate-based bitrate choice (SPEC §4.2): the highest bitrate whose chunk fits ``safety`` times the harmonic mean of
    the last ``hist_k`` throughputs times the chunk length."""
    def __init__(self, safety=1.0):
        self.safety = float(safety)


class BolaPolicy:
    """BOLA (SPEC §4.3): the Lyapunov buffer rule with its (V, gamma*p) derived from the buffer range
    [min_buffer, target_buffer] in seconds."""
    def __init__(self, min_buffer=10.0, target_buffer=30.0):
        self.min_buffer, self.target_buffer = float(min_buffer), float(target_buffer)


class LookaheadPolicy:
    """Clairvoyant lookahead (SPEC §4.4): at every chunk, the first bitrate of the sequence over the next ``horizon``
    chunks with the largest sum of rewards against the session's actual future trace.  It sees the future: an upper
    reference to compare controllers against, not a controller a player could run.  Not available in live mode."""
    def __init__(self, horizon=5):
        self.horizon = int(horizon)


class FixedPolicy:
    def __init__(self, actions):
        self.actions = np.asarray(actions, dtype=np.int32)


class Simulator:
    def __init__(self, AbrController=None, SpeedController=None, **params):
        self.qoe_metric = None
        self.mpd = None
        self.network_info = None
        self.abr_controller = AbrController
        self.speed_controller = SpeedController      # get_next_speed() -> playback speed (live mode, Simulator.py:177)
        self.params = dict(params)
        self._env = None
        self.last_run = None

    # -- setters (Simulator.py:54-77) --
    def set_qoe_metric(self, qoe_metric):
        self.qoe_metric = qoe_metric
        self._env = None

    def set_network_info(self, interval, networktrace):
        """``networktrace``: path of a one-float-per-line file (Simulator.py:59-65), a sequence of
        bandwidths, a NetworkInfo, or a list of NetworkInfo (one trace per session group)."""
        if isinstance(networktrace, (str, bytes)):
            self.network_info = NetworkInfo(interval, load_network_trace(networktrace))
        elif isinstance(networktrace, NetworkInfo):
            self.network_info = networktrace
        elif len(networktrace) and isinstance(networktrace[0], NetworkInfo):
            self.network_info = list(networktrace)
        else:
            self.network_info = NetworkInfo(interval, list(networktrace))
        self._env = None

    def set_mpd(self, chunk_length, max_buffer, start_up_length, mpdfile):
        """``mpdfile``: path (one line of bitrates per chunk), or a list of ``Chunk``."""
        chunks = load_mpd_file(mpdfile) if isinstance(mpdfile, (str, bytes)) else list(mpdfile)
        self.mpd = MPD(len(chunks), chunk_length, max_buffer, start_up_length, chunks)
        self._env = None

    def get_mpd(self):
        return self.mpd

    def get_qoe_metric(self):
        return self.qoe_metric

    def calculate_qoe(self, rebuffer_time, previous_bitrates, start_up_time, average_latency):
        """Simulator.py:79-86 with the indexing repaired (D3): ladder of each chunk, consecutive indices."""
        q = self.qoe_metric
        variance = 0.0
        for i in range(0, len(previous_bitrates) - 1):
            variance += abs(self.mpd.chunks[i].bitrates[previous_bitrates[i]] -
                            self.mpd.chunks[i + 1].bitrates[previous_bitrates[i + 1]])
        return (q.rebuffer_weight * rebuffer_time + q.variance_weight * variance +
                q.startup_weight * start_up_time + getattr(q, "latency_weight", 0.0) * average_latency)

    # -- environment --
    _MARKERS = (RandomPolicy, BufferBasedPolicy, RateBasedPolicy, BolaPolicy, FixedPolicy)

    @staticmethod
    def _marker_policy(ctrl):
        """The fused-episode policy name of a built-in policy marker (None: buffer-based)."""
        return ("random" if isinstance(ctrl, RandomPolicy) else "fixed" if isinstance(ctrl, FixedPolicy) else
                "rate" if isinstance(ctrl, RateBasedPolicy) else "bola" if isinstance(ctrl, BolaPolicy) else "bba")

    def _marker_env(self, ctrl, n_sessions, **extra):
        """The environment of a built-in policy marker, with the marker's parameters installed."""
        if isinstance(ctrl, BufferBasedPolicy):
            extra.update(bba_reservoir=ctrl.reservoir, bba_cushion=ctrl.cushion)
        if isinstance(ctrl, RateBasedPolicy):
            extra.update(track_history=1)             # the rate-based rule reads the throughput history
        env = self._make_env(n_sessions, **extra)
        if isinstance(ctrl, RateBasedPolicy):
            env.set_policy_params(rb_safety=ctrl.safety)
        elif isinstance(ctrl, BolaPolicy):
            env.set_policy_params(bola_min_buffer=ctrl.min_buffer, bola_target_buffer=ctrl.target_buffer)
        return env

    def _make_env(self, n_sessions, **extra):
        if self.mpd is None or self.network_info is None or self.qoe_metric is None:
            raise RuntimeError("set_qoe_metric, set_network_info and set_mpd must be called before run()")
        # the reference's environment (see the module docstring): cost in bitrate units, first chunk free, no RTT, no
        # payload factor, continuous pause (one tick), variance over each chunk's own ladder
        kw = dict(utility_scale=1.0, default_quality=-1, auto_reset=0, rtt=0.0, payload=1.0, sleep_quantum=0.01,
                  latency_tick=0.01, smooth_prev_ladder=1)
        kw.update(self.params)
        kw.update(extra)
        return BatchedABREnv.from_objects(self.network_info, self.mpd, self.qoe_metric, max_sessions=n_sessions, **kw)

    def run(self):
        """One session over trace 0 from offset 0; returns the scalar QoE cost."""
        return float(self.run_batch(1)[0])

    def _live(self):
        return self.mpd is not None and self.mpd.start_up_length is not None and not self.params.get("force_vod", False)

    def run_batch(self, n_sessions, trace_id=None, start_offset=None, session_base=0):
        """``n_sessions`` independent sessions; returns a numpy vector of QoE costs (one per session)."""
        V = len(self.mpd.chunks)
        n_traces = len(self.network_info) if isinstance(self.network_info, list) else 1
        # default assignment: equal runs of consecutive sessions per trace (sessions sorted by trace take the
        # shared-memory path of the kernels, DESIGN.md §4)
        tid = ((np.arange(n_sessions, dtype=np.int64) * n_traces) // max(n_sessions, 1)).astype(np.int32) \
            if trace_id is None else np.asarray(trace_id, np.int32)
        ctrl = self.abr_controller
        q = self.qoe_metric
        if isinstance(ctrl, LookaheadPolicy) and self._live():
            raise ValueError("LookaheadPolicy is not available in live mode (SPEC §7): its objective has no playback "
                             "speeds and no latency term")
        if self._live():
            return self._run_live(n_sessions, tid, start_offset, session_base)
        if isinstance(ctrl, self._MARKERS) or ctrl is None:
            env = self._marker_env(ctrl, n_sessions)
            out = env.run_host(self._marker_policy(ctrl), V, tid, start_offset, seed=getattr(ctrl, "seed", 0),
                               session_base=session_base, actions=getattr(ctrl, "actions", None), want_qoe_cost=True)
            acc = out["acc"]
            self.last_run = dict(zip(ACC_NAMES, acc))
            return out["qoe_cost"]          # rw*rebuffer + vw*smooth, computed on the device
        elif isinstance(ctrl, MPCBitrateController):
            env = self._make_env(n_sessions, track_history=1, track_acc=1, **ctrl.extra_params)
            env.reset(tid, start_offset, session_base)
            env.mpc_episode(V, horizon=ctrl.horizon, mode="robust" if ctrl.mode == MPC_ROBUST else "reference")
            acc = env.session_acc().cpu().numpy()
        elif isinstance(ctrl, LookaheadPolicy):
            env = self._make_env(n_sessions, track_acc=1)
            env.reset(tid, start_offset, session_base)
            env.lookahead_episode(V, horizon=ctrl.horizon)
            acc = env.session_acc().cpu().numpy()
        else:
            acc = self._run_callback(self._make_env(n_sessions, track_acc=1), n_sessions, tid, start_offset)
        self.last_run = dict(zip(ACC_NAMES, acc))
        return q.rebuffer_weight * acc[1] + q.variance_weight * acc[3]

    def _run_live(self, n_sessions, tid, start_offset, session_base):
        """Live mode (SPEC §7): per-step kernel, one bitrate and one playback-speed decision per chunk."""
        q = self.qoe_metric
        ctrl = self.abr_controller
        extra = dict(live=1, start_up_length=float(self.mpd.start_up_length), startup_penalty=float(q.startup_weight),
                     latency_penalty=float(getattr(q, "latency_weight", 0.0)), track_acc=1)
        V = len(self.mpd.chunks)
        if isinstance(ctrl, MPCBitrateController):
            env = self._make_env(n_sessions, track_history=1, **extra, **ctrl.extra_params)
            env.reset(tid, start_offset, session_base)
            mode = "robust" if ctrl.mode == MPC_ROBUST else "reference"
            speed = self._speed_table(n_sessions, V)
            for _ in range(V):
                act = env.mpc_decide(ctrl.horizon, mode)
                env.step(act, want_next_sizes=False, speed=speed)
        elif isinstance(ctrl, self._MARKERS) or ctrl is None:
            # built-in policies: one fused live episode (abr_env_rollout_fused_live), speed table from the controller
            env = self._marker_env(ctrl, n_sessions, **extra)
            env.reset(tid, start_offset, session_base)
            speed = self._speed_table(n_sessions, V)
            env.rollout(self._marker_policy(ctrl), V, seed=getattr(ctrl, "seed", 0), actions=getattr(ctrl, "actions", None),
                        speed=speed, want=())
        else:
            env = self._make_env(n_sessions, **extra)
            self._run_callback(env, n_sessions, tid, start_offset, session_base)
        acc = env.session_acc().cpu().numpy()
        self.last_run = dict(zip(ACC_NAMES, acc))
        return env.qoe_cost().cpu().numpy()

    def _speed_table(self, n_sessions, V):
        """[V, N] playback speeds: ``get_next_speed()`` is called once per content chunk of every session, in playing
        order (the k-th call of a session's run is the speed of its k-th played chunk, Simulator.py:176-177).  The
        controller protocol takes no arguments, so its answers cannot depend on the session's state and may be
        drawn before the run."""
        if self.speed_controller is None:
            return None
        table = np.empty((V, n_sessions))
        for s in range(n_sessions):
            for k in range(V):
                table[k, s] = float(self.speed_controller.get_next_speed())
        return torch.from_numpy(table).to(self._device())

    @staticmethod
    def _device():
        return torch.device("cuda", torch.cuda.current_device())

    def _host_policy_actions(self, ctrl, k, n_sessions, buf, A, rng, session_base):
        """Built-in policy markers evaluated on the host (used in live mode, where the fused episode does not apply)."""
        if isinstance(ctrl, FixedPolicy):
            return np.ascontiguousarray(ctrl.actions.reshape(len(self.mpd.chunks), -1)[k], dtype=np.int32)
        if isinstance(ctrl, RandomPolicy):
            return rng.integers(0, A, size=n_sessions).astype(np.int32)
        r, c = ctrl.reservoir, ctrl.cushion          # BufferBasedPolicy / None
        qv = np.floor((A - 1) * (buf - r) / c)
        return np.clip(np.where(buf < r, 0, np.where(buf >= r + c, A - 1, qv)), 0, A - 1).astype(np.int32)

    def _run_callback(self, env, n_sessions, tid, start_offset, session_base=0):
        """One decision per session and chunk: the generic controller protocol ``get_next_bitrate(chunk_id,
        previous_bitrates, previous_bandwidths, buffer_level)`` (Simulator.py:155), or a built-in policy marker."""
        V = len(self.mpd.chunks)
        A = env.A
        ctrl = self.abr_controller if self.abr_controller is not None else BufferBasedPolicy()
        marker = isinstance(ctrl, (RandomPolicy, BufferBasedPolicy, FixedPolicy))
        live = bool(env.params.live)
        env.reset(tid, start_offset, session_base)
        speed = self._speed_table(n_sessions, V) if live else None
        prev_q = [[] for _ in range(n_sessions)]
        prev_bw = [[] for _ in range(n_sessions)]
        buf = np.zeros(n_sessions)
        rng = np.random.default_rng(getattr(ctrl, "seed", 0))
        for k in range(V):
            if marker:
                acts = self._host_policy_actions(ctrl, k, n_sessions, buf, A, rng, session_base)
            else:
                acts = np.array([ctrl.get_next_bitrate(k, prev_q[s], prev_bw[s], float(buf[s]))
                                 for s in range(n_sessions)], dtype=np.int32)
            r = env.step(torch.from_numpy(acts), want_next_sizes=False, want_throughput=True,
                         speed=speed)
            buf = r.buffer.cpu().numpy()
            if not marker:
                thr = r.throughput.cpu().numpy()
                for s in range(n_sessions):
                    prev_q[s].append(int(acts[s]))
                    prev_bw[s].append(float(thr[s]))
        return env.session_acc().cpu().numpy()
