#!/usr/bin/env python
"""bench.py — ABR chunk-steps/s (headline) and MPC decisions/s on N B200s, beside the CPU reference path.

Contract: ``python bench.py --gpus N --steps K --warmup W`` (under torchrun for N > 1) prints ONE JSON line on
rank 0.  A "step" is one pass of the hot path over one batch: reset + one fused 48-chunk episode of
``--sessions`` sessions per GPU (BASELINE.json configs[1]: random-policy chunk-step sweep, 65 536 sessions x 48
chunks on synthetic traces) + the statistics reduction.  Sessions shard across GPUs with no data-path
collective (weak scaling); the only collective is the final statistics all-gather.

``--impl reference`` times the reference's CPU path instead: the reference is pure Python and cannot travel to
the GPU box, so this runs the pure-Python port in ``oracle/`` (statement-level restatement, pinned to the
reference by tests/golden) on all host cores over a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import signal
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

V, A = 48, 6
N_TRACES, T_TRACE = 1024, 2048
SEED = 7
GROUP = 64                          # consecutive sessions per trace (one 64-thread block = one trace)
BYTES_PER_STEP = 5 * 8 + 1          # delay, sleep, buffer, rebuf, reward (f64) + end_of_video (u8)
BYTES_PER_SESSION = 40 + 36 + 176   # state load + state store + read-modify-write of the 11 accumulators, once per episode
# abr_env_run (reset fused into the episode kernel): 12 B of trace id + start offset in, the whole reset state out
# (36 B of position + 50 B that only a reset writes: trace_id, hist_len, last_pred, err_len, done, t_now, play_time,
# started, play_id, play_len) and the 11 accumulators written without being read
BYTES_PER_SESSION_RUN = 12 + 36 + 50 + 88


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--sessions", type=int, default=65536, help="sessions per GPU (configs[1])")
    ap.add_argument("--mpc-sessions", type=int, default=131072, help="MPC sessions per GPU (configs[2] / 8)")
    ap.add_argument("--mpc-strong-total", type=int, default=1 << 20,
                    help="configs[2] as written: a FIXED total of robust-MPC sessions sharded over the GPUs (strong "
                         "scaling), whole 48-chunk episode + the statistics all-reduce inside the timed region (0 = skip)")
    ap.add_argument("--mpc-horizon", type=int, default=5)
    ap.add_argument("--mpc-h7-sessions", type=int, default=2048, help="sessions per GPU of the horizon-7 leg (0 = skip)")
    ap.add_argument("--no-mpc", action="store_true")
    ap.add_argument("--no-step-form", action="store_true")
    ap.add_argument("--rl-sessions", type=int, default=1 << 19,
                    help="sessions per GPU of the RL-harness leg (configs[4] / 8; 0 = skip)")
    ap.add_argument("--step-sessions", type=int, default=1 << 22, help="sessions per GPU of the per-step-launch leg")
    ap.add_argument("--separate-reset", action="store_true",
                    help="timed step = abr_env_reset + abr_env_rollout_fused + statistics (three launches) instead of abr_env_run")
    ap.add_argument("--no-cpu-bind", action="store_true", help="do not restrict the rank to the CPU cores next to its GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU time budget of each cpu_baseline sample")
    ap.add_argument("--group", type=int, default=GROUP,
                    help="consecutive sessions per trace (default 64: every 64-thread block of the fused kernel follows "
                         "one trace and stages it in shared memory; 1 = trace = session mod n_traces, global path)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy: the [48][n] "
                         "trajectories of a fixed sample of the sessions and the statistics vector (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    globals()["GROUP"] = args.group
    return args


# ------------------------------------------------------------------------------------------------
# CPU legs (oracle port) — the only places bench.py executes oracle/
# ------------------------------------------------------------------------------------------------
def _py_step_worker(job):
    """Pure-Python port of the chunk step (oracle/step_oracle.py) over a block of sessions."""
    import numpy as np
    from abrsimulator_b200 import synth
    from oracle import oracle as orc, step_oracle as so
    lo, hi, budget_s = job
    bitrates, sizes = synth.make_video(V)
    bw, tl, ti = synth.make_traces(N_TRACES, T_TRACE)
    tid, off = synth.make_sessions(hi - lo, N_TRACES, T_TRACE, session_base=lo, group=GROUP)
    P = dict(orc.DEFAULTS)
    util = (bitrates * P["utility_scale"]).tolist()
    sz = sizes.tolist()
    t0 = time.perf_counter()
    done_steps = 0
    tot = 0.0
    tables = {}
    for s in range(hi - lo):
        tr = int(tid[s])
        if tr not in tables:    # per-trace capacity table, built once like the device does
            tables[tr] = (bw[tr].tolist(), so.capacity_table(bw[tr].tolist(), float(ti[tr]), P["payload"]))
        sess = so.Session(tables[tr][0], float(ti[tr]), sz, util, P, float(off[s]), table=tables[tr][1])
        g = lo + s
        for t in range(V):
            x16 = (orc.philox(g & 0xffffffff, g >> 32, t >> 3, 0, SEED, 0)[(t & 7) >> 1] >> (16 * (t & 1))) & 0xffff
            tot += sess.step((x16 * A) >> 16)["reward"]
        done_steps += V
        if time.perf_counter() - t0 > budget_s:
            break
    return done_steps, time.perf_counter() - t0, tot


def cpu_python_steps(n_procs, budget_s, sessions_per_proc=100000):
    import multiprocessing as mp
    jobs = [(i * sessions_per_proc, (i + 1) * sessions_per_proc, budget_s) for i in range(n_procs)]
    t0 = time.perf_counter()
    if n_procs == 1:
        res = [_py_step_worker(jobs[0])]
    else:
        with mp.get_context("spawn").Pool(n_procs) as pool:
            res = pool.map(_py_step_worker, jobs)
    wall = time.perf_counter() - t0
    steps = sum(r[0] for r in res)
    busy = max(r[1] for r in res)
    return steps / busy, steps, busy, wall


def cpu_c_oracle_steps(n_sessions=8192):
    import numpy as np
    from abrsimulator_b200 import synth
    from oracle import oracle as orc
    bitrates, sizes = synth.make_video(V)
    bw, tl, ti = synth.make_traces(N_TRACES, T_TRACE)
    tid, off = synth.make_sessions(n_sessions, N_TRACES, T_TRACE, group=GROUP)
    env = orc.OracleEnv(bw, tl, ti, sizes, bitrates, n_sessions)
    env.reset(tid, off)
    t0 = time.perf_counter()
    env.rollout(orc.POLICY_RANDOM, V, seed=SEED, want_traj=True)
    dt = time.perf_counter() - t0
    return n_sessions * V / dt, n_sessions, dt


def _py_mpc_worker(job):
    import numpy as np
    from abrsimulator_b200 import synth
    from oracle import mpc_oracle as mo
    idx0, count, H, budget_s = job
    bitrates, sizes = synth.make_video(V)
    util = (bitrates * 0.001).tolist()
    sz = sizes.tolist()
    rng = np.random.default_rng(1000 + idx0)
    t0 = time.perf_counter()
    n = 0
    for _ in range(count):
        st = mo.RobustState(5)
        hist = [float(x) for x in rng.uniform(0.2, 6.0, size=5)]
        mo.decide_robust(int(rng.integers(0, V - H)), int(rng.integers(0, A)), float(rng.uniform(0, 30)), hist, st, H,
                         util, sz, 4.0, 60.0, 1.0, 4.3)
        n += 1
        if time.perf_counter() - t0 > budget_s:
            break
    return n, time.perf_counter() - t0


def cpu_python_mpc(n_procs, H, budget_s):
    import multiprocessing as mp
    jobs = [(i, 100000, H, budget_s) for i in range(n_procs)]
    if n_procs == 1:
        res = [_py_mpc_worker(jobs[0])]
    else:
        with mp.get_context("spawn").Pool(n_procs) as pool:
            res = pool.map(_py_mpc_worker, jobs)
    n = sum(r[0] for r in res)
    busy = max(r[1] for r in res)
    return n / busy, n, busy


def run_reference(args):
    """--impl reference: the CPU path on all host cores, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    per_step_budget = max(1.0, min(6.0, 60.0 / max(1, args.steps + args.warmup)))
    rates = []
    for i in range(args.warmup + args.steps):
        rate, steps, busy, wall = cpu_python_steps(cores, per_step_budget)
        if i >= args.warmup:
            rates.append((rate, steps, busy))
    tot_steps = sum(r[1] for r in rates)
    tot_busy = sum(r[2] for r in rates)
    value = tot_steps / tot_busy
    sample = (f"pure-Python port of the chunk step (oracle/step_oracle.py; the reference's own loop does not run, "
              f"SURVEY D1-D6) on {cores} processes, ~{per_step_budget:.1f} s of sessions x 48 chunks per step, "
              f"{tot_steps} chunk-steps in total")
    line = dict(impl="reference", metric="chunk_steps_per_sec", value=value, unit="chunk-steps/s", n_gpus=args.gpus,
                steps=args.steps, warmup=args.warmup, ms_per_step=1e3 * tot_busy / max(1, args.steps),
                higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64", data="synthetic",
                config=workload_config(args),
                cpu_baseline=dict(value=value, unit="chunk-steps/s", cores=cores, kind="port", sample=sample),
                e2e=dict(value=value, unit="chunk-steps/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    if not args.no_mpc:
        r, n, busy = cpu_python_mpc(cores, args.mpc_horizon, min(10.0, args.cpu_seconds))
        line["mpc"] = dict(metric="mpc_decisions_per_sec", value=r, unit="decisions/s", horizon=args.mpc_horizon,
                           cores=cores, sample=f"{n} robust-MPC decisions (oracle/mpc_oracle.py port of mpc.py)")
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# same-run parity (BASELINE.md §4.3): the benchmarked configuration's own outputs against the C oracle, on a sample
# ------------------------------------------------------------------------------------------------
def parity_chunk_steps(out, tid_h, off_h, base, n_windows=4, window=512):
    """The trajectories the LAST timed step left in `out` ([V][N] device tensors) against oracle/abr_oracle.c run on
    `n_windows` windows of `window` consecutive sessions of this rank's shard (same traces, offsets, seed and global
    session indices).  Bit-exact is the bar (SPEC.md); the 1e-9 relative bar of BASELINE.json is reported beside it."""
    import numpy as np
    from abrsimulator_b200 import synth
    from oracle import oracle as orc
    N = tid_h.shape[0]
    window = min(window, N)
    starts = sorted({int(round(i * (N - window) / max(1, n_windows - 1))) for i in range(n_windows)})
    bitrates, sizes = synth.make_video(V)
    bw, tl, ti = synth.make_traces(N_TRACES, T_TRACE)
    keys = (("delay", "delay"), ("sleep", "sleep"), ("buffer", "buffer"), ("rebuffer", "rebuf"), ("reward", "reward"))
    values = differ = 0
    max_rel = 0.0
    eov_ok = True
    t0 = time.perf_counter()
    for k0 in starts:
        ref = orc.OracleEnv(bw, tl, ti, sizes, bitrates, window)
        ref.reset(tid_h[k0:k0 + window], off_h[k0:k0 + window])
        exp = ref.rollout(orc.POLICY_RANDOM, V, seed=SEED, session_base=base + k0)
        for kg, kc in keys:
            g = out[kg][:, k0:k0 + window].cpu().numpy()
            e = exp[kc]
            values += g.size
            differ += int((g.view(np.uint64) != e.view(np.uint64)).sum())
            max_rel = max(max_rel, float((np.abs(g - e) / np.maximum(np.abs(e), 1e-300)).max()))
        eov_ok = eov_ok and bool(np.array_equal(out["end_of_video"][:, k0:k0 + window].cpu().numpy(), exp["eov"]))
    return dict(checker="oracle/abr_oracle.c (SPEC.md restated; pinned to the reference's tick loop by tests/golden/sim_ref_tick_golden.json)",
                sessions_checked=len(starts) * window, chunk_steps_checked=len(starts) * window * V,
                values_checked=values, non_identical_values=differ, max_rel_err=max_rel, end_of_video_identical=eov_ok,
                bar="bit-identical (SPEC.md); BASELINE.json: 1e-9 relative", ok=bool(differ == 0 and eov_ok),
                seconds=time.perf_counter() - t0)


def parity_mpc(menv, H, act, sample=2048):
    """One robust-MPC launch at the benchmarked shape against the C oracle's exhaustive search on a strided sample of
    sessions: the state the kernel is about to read is snapshotted, the launch runs, and the chosen actions must be
    identical (SPEC §5.2: near-ties are resolved identically because nothing is reassociated)."""
    import numpy as np
    from oracle import oracle as orc
    M = menv.n
    idx = np.unique(np.linspace(0, M - 1, min(sample, M)).astype(np.int64))
    import torch
    ix = torch.from_numpy(idx).to(act.device)
    snap = {f: menv.state(f).index_select(-1, ix).cpu().numpy().copy()
            for f in ("chunk", "last_q", "buffer", "bw_hist", "hist_len", "last_pred", "err_ring", "err_len")}
    menv.mpc_decide(H, "robust", out=act)
    got = act.index_select(0, ix).cpu().numpy()
    p = orc.make_params(**{k: getattr(menv.params, k) for k in ("chunk_length", "max_buffer", "rebuf_penalty",
                                                               "smooth_penalty", "default_quality", "hist_k")})
    sizes = menv.state("sizes").cpu().numpy()
    util = menv.state("utility").cpu().numpy()
    t0 = time.perf_counter()
    lp = np.ascontiguousarray(snap["last_pred"])
    er = np.ascontiguousarray(snap["err_ring"].T)
    el = np.ascontiguousarray(snap["err_len"])
    exp = orc.mpc_decide(sizes, util, snap["chunk"], snap["last_q"], snap["buffer"], np.ascontiguousarray(snap["bw_hist"].T),
                         snap["hist_len"], H, 1, p, lp, er, el)
    bad = int((got != exp["action"]).sum())
    return dict(checker="oracle/abr_oracle.c exhaustive search (no prefix sharing)", decisions_checked=int(idx.size),
                sequences_per_decision=A ** H, disagreements=bad, ok=bool(bad == 0 and exp["n_errors"] == 0),
                seconds=time.perf_counter() - t0)


DUMP_SESSIONS = 16384               # sessions in the --dump-outputs sample: 48 x 16 384 x (5 x 8 + 4) B = 34.6 MB


def dump_outputs(path, out, stats):
    """--dump-outputs: what the last timed step handed back to its caller, as <path>/<name>.npy.  The five [48][N] fp64
    trajectories and end_of_video (as float32) are reduced to the same fixed, seeded sample of session columns (ascending
    order), so the files stay far below 64 MB at any --sessions; the statistics vector is written whole.  The inputs
    depend on the arguments only (seeded synthetic traces, video and sessions), so two builds run with the same
    arguments can be compared file by file.  Under torchrun rank 0 writes its own shard."""
    import numpy as np
    import torch
    N = out["reward"].shape[1]
    cols = np.sort(np.random.default_rng(SEED).choice(N, size=min(N, DUMP_SESSIONS), replace=False))
    ix = torch.from_numpy(cols).to(out["reward"].device)
    arrays = {k: out[k].index_select(1, ix).cpu().numpy() for k in ("delay", "sleep", "buffer", "rebuffer", "reward")}
    arrays["end_of_video"] = out["end_of_video"].index_select(1, ix).cpu().numpy().astype(np.float32)
    arrays["stats"] = stats.cpu().numpy()
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), a)


def workload_config(args):
    return dict(workload="configs[1]: random-policy chunk-step sweep, fused 48-chunk episodes",
                sessions_per_gpu=args.sessions, chunks=V, bitrates=A, n_traces=N_TRACES, trace_segments=T_TRACE,
                policy="random(philox)", sessions_per_trace=GROUP, outputs="delay,sleep,buffer,rebuffer,reward,end_of_video",
                l2="256 MiB buffer rewritten twice between timed steps (outside the timed intervals)",
                timing="one CUDA-event interval per step, all K steps enqueued back to back, one host wait at the end")


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc = None
        self.index = index
        self.t_load = None

    def mark_load(self):
        """Samples older than this moment (the poller is started early so that nvidia-smi's start-up, which holds
        driver locks for most of a second, is over before the timed region) are not counted."""
        import datetime
        self.t_load = datetime.datetime.now()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        import atexit
        atexit.register(self.proc.kill)                        # a run that fails before stop() leaves no poller behind

    def pause(self, on=True):
        """SIGSTOP / SIGCONT the poller: nvidia-smi queries take driver locks that the launch- and sync-latency
        bound host-buffer leg (90 us per call) would otherwise pay for."""
        if self.proc is not None:
            try:
                self.proc.send_signal(signal.SIGSTOP if on else signal.SIGCONT)
            except Exception:
                pass

    def stop(self):
        if self.proc is not None:
            self.pause(False)
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        import datetime
        for ln in out.strip().splitlines():
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f")
                if self.t_load is not None and ts < self.t_load:
                    continue
            except ValueError:
                pass
            f = f[1:]
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=max(mx) if mx else None,
                    samples=len(sm), reasons=sorted(reasons))


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from abrsimulator_b200 import synth, _lib
    from abrsimulator_b200.env import BatchedABREnv
    from abrsimulator_b200.distributed import allreduce_stats, max_over_ranks

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    from abrsimulator_b200.distributed import bind_to_gpu_cpus
    all_cpus = os.sched_getaffinity(0)
    cpus = None if args.no_cpu_bind else bind_to_gpu_cpus(local)   # cores of the NUMA node next to this rank's GPU
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                                        # early: see ClockSampler.mark_load

    N = args.sessions
    base = rank * N
    bitrates, sizes = synth.make_video(V)
    bw, tl, ti = synth.make_traces(N_TRACES, T_TRACE)
    tid_h, off_h = synth.make_sessions(N, N_TRACES, T_TRACE, session_base=base, group=GROUP)
    env = BatchedABREnv(bw, sizes, bitrates, max(N, args.mpc_sessions), trace_len=tl, trace_interval=ti)
    tid_d = torch.from_numpy(tid_h).to(dev)
    off_d = torch.from_numpy(off_h).to(dev)
    out = {k: torch.empty(V, N, dtype=torch.float64, device=dev) for k in ("delay", "sleep", "buffer", "rebuffer", "reward")}
    out["end_of_video"] = torch.empty(V, N, dtype=torch.uint8, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream()

    stats_buf = torch.empty(_lib.NUM_STATS, dtype=torch.float64, device=dev)

    def one_step(ev=None):
        if args.separate_reset:                                # three launches: reset, episode, statistics
            env.reset(tid_d, off_d, session_base=base)
            if ev:
                ev[0].record(stream)
            env.rollout("random", V, seed=SEED, out=out)
            if ev:
                ev[1].record(stream)
            return env.stats()
        # one launch: the episode kernel resets the sessions, and its last block reduces the statistics (abr_env_run with
        # a statistics buffer)
        if ev:
            ev[0].record(stream)
        env.run("random", V, tid_d, off_d, seed=SEED, session_base=base, out=out, qoe_cost=False, stats=stats_buf)
        if ev:
            ev[1].record(stream)
        return stats_buf

    for _ in range(max(3, args.warmup)):
        flush.fill_(1)
        stats = one_step()
    barrier()
    if rank == 0:
        sampler.mark_load()
    launches0 = _lib.launch_count()
    # The K timed steps are enqueued back to back — each behind two rewrites of the 256 MiB flush buffer (outside its
    # timed interval) — and the host waits once, at the end: it runs ahead of the GPU (a step takes the host ~60 us to
    # enqueue and the GPU ~200 us to execute with its flushes; a few flushes in front give it the head start), so every
    # interval between a step's two events is device time of that step and nothing else, also with eight ranks sharing
    # the host's cores.  Waiting for every step instead puts the host's launch path inside the interval as soon as
    # enqueueing the step takes longer than its flush.
    events = []
    barrier()
    wall0 = time.perf_counter()
    for _ in range(4):
        flush.fill_(3)
    for _ in range(args.steps):
        flush.fill_(1)                                         # evict L2 (outside the timed interval)
        flush.fill_(2)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        # A step of the default form is ONE launch, so the step's own two events are also the kernel's: a second
        # pair nested inside them only adds two event records (~2.7 us each on this stream) to the timed interval.
        # --separate-reset (three launches per step) keeps the inner pair around the episode kernel.
        k0, k1 = ((torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) if args.separate_reset
                  else (e0, e1))
        e0.record(stream)
        stats = one_step((k0, k1) if args.separate_reset else None)
        e1.record(stream)
        events.append((e0, e1, k0, k1))
    barrier()
    wall = time.perf_counter() - wall0
    if rank == 0 and args.dump_outputs:                        # before any later leg overwrites `out`
        dump_outputs(args.dump_outputs, out, stats)
    step_ms = [e0.elapsed_time(e1) for e0, e1, _, _ in events]
    kern_ms = [k0.elapsed_time(k1) for _, _, k0, k1 in events]
    launches = _lib.launch_count() - launches0
    total_ms = max_over_ranks(sum(step_ms), dev)
    kern_avg_ms = sum(kern_ms) / len(kern_ms)
    per_rank = None
    if world > 1:                                              # who is the slowest rank, and by how much
        mine = torch.tensor([sum(step_ms) / len(step_ms), kern_avg_ms], dtype=torch.float64, device=dev)
        allr = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        per_rank = dict(ms_per_step=[float(t[0]) for t in allr], kernel_ms=[float(t[1]) for t in allr])
    tot_stats = allreduce_stats(stats)                          # the one collective: final QoE statistics
    torch.cuda.synchronize()
    # ... and what it costs when it closes every step (BASELINE.json configs[2]: "final QoE all-reduce"): CUDA events
    # around the call on the launching stream, max over ranks.  88 bytes per rank: pure latency.
    collective = None
    if world > 1:
        cms = []
        for it in range(3 + 10):
            barrier()
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record(stream)
            allreduce_stats(stats)
            c1.record(stream)
            c1.synchronize()
            if it >= 3:
                cms.append(c0.elapsed_time(c1))
        cms.sort()
        collective = dict(op="all_gather of the per-rank statistics vector + rank-order sum (deterministic)",
                          bytes_per_rank=int(stats.numel() * 8), backend="nccl",
                          us=max_over_ranks(1e3 * cms[len(cms) // 2], dev),
                          step_with_collective_ms=total_ms / args.steps + max_over_ranks(cms[len(cms) // 2], dev),
                          note="not inside value / e2e (one reduction closes a run, not a step); "
                               "mpc.strong_scaling times it inside its region")
    chunk_steps = world * N * V * args.steps
    value = chunk_steps / (total_ms * 1e-3)
    errors = env.error_count()
    # every session of rank 0's shard: the C oracle replays the whole 65 536 x 48 batch in ~2 s
    parity = parity_chunk_steps(out, tid_h, off_h, base, n_windows=max(1, N // 4096), window=min(N, 4096)) if rank == 0 else None

    # ---- optional fp32-output mode (fp64 arithmetic and state; 5 x 4 + 1 B of trajectory per chunk-step) ----
    out32 = {k: torch.empty(V, N, dtype=torch.float32, device=dev) for k in ("delay", "sleep", "buffer", "rebuffer", "reward")}
    out32["end_of_video"] = out["end_of_video"]
    f32_ms = []
    for it in range(3 + 8):
        flush.fill_(1)
        env.reset(tid_d, off_d, session_base=base)
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record(stream)
        env.rollout("random", V, seed=SEED, out=out32)
        k1.record(stream)
        k1.synchronize()
        if it >= 3:
            f32_ms.append(k0.elapsed_time(k1))
    f32_kernel_ms = max_over_ranks(sum(f32_ms), dev) / len(f32_ms)
    f32_bytes = N * (V * (5 * 4 + 1) + BYTES_PER_SESSION)
    fp32_outputs = dict(kernel="abr_rollout_kernel<random, float>", kernel_ms=f32_kernel_ms,
                        chunk_steps_per_s=world * N * V / (f32_kernel_ms * 1e-3), bytes_per_chunk_step=21,
                        frac=f32_bytes / (f32_kernel_ms * 1e-3) / 1e9 / hbm_peak_gbs(),
                        max_rel_err_vs_f64=float(((out32["reward"].double() - out["reward"]).abs() /
                                                  out["reward"].abs().clamp_min(1e-300)).max()))
    del out32

    # ---- the other policy of configs[1]: buffer-based (the action depends on the state, so nothing is hoisted) ----
    bba_ms = []
    for it in range(3 + 8):
        flush.fill_(1)
        env.reset(tid_d, off_d, session_base=base)
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record(stream)
        env.rollout("bba", V, out=out)
        k1.record(stream)
        k1.synchronize()
        if it >= 3:
            bba_ms.append(k0.elapsed_time(k1))
    bba_kernel_ms = max_over_ranks(sum(bba_ms), dev) / len(bba_ms)
    bba = dict(kernel="abr_rollout_kernel<bba>", kernel_ms=bba_kernel_ms,
               chunk_steps_per_s=world * N * V / (bba_kernel_ms * 1e-3),
               frac=(N * (V * BYTES_PER_STEP + BYTES_PER_SESSION)) / (bba_kernel_ms * 1e-3) / 1e9 / hbm_peak_gbs())

    # ---- the same episode kernel with the session -> trace map of SURVEY.md §8(d), trace = session mod n_traces
    #      ("interleaved": no block follows one trace, every table probe is a scattered L2 read), and the same sessions with
    #      the environment keeping them sorted by trace (reset(sort_by_trace=True): abr_sort_by_trace + abr_env_set_order
    #      inside the timed call, outputs in environment order) ----
    fused_layouts = {}
    tid_i, off_i = synth.make_sessions(N, N_TRACES, T_TRACE, session_base=base, group=1)
    tid_id, off_id = torch.from_numpy(tid_i).to(dev), torch.from_numpy(off_i).to(dev)
    for name, sort in (("interleaved", False), ("interleaved_env_sorted", True)):
        ms_k, ms_all = [], []
        for it in range(3 + 8):
            flush.fill_(1)
            env.set_order(None)
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record(stream)
            env.reset(tid_id, off_id, session_base=base, sort_by_trace=sort)
            k0.record(stream)
            env.rollout("random", V, seed=SEED, out=out)
            k1.record(stream)
            a1.record(stream)
            a1.synchronize()
            if it >= 3:
                ms_k.append(k0.elapsed_time(k1))
                ms_all.append(a0.elapsed_time(a1))
        km = max_over_ranks(sum(ms_k), dev) / len(ms_k)
        am = max_over_ranks(sum(ms_all), dev) / len(ms_all)
        fused_layouts[name] = dict(kernel_ms=km, reset_plus_episode_ms=am,
                                   chunk_steps_per_s=world * N * V / (am * 1e-3),
                                   frac=(N * (V * BYTES_PER_STEP + BYTES_PER_SESSION)) / (km * 1e-3) / 1e9 / hbm_peak_gbs())
    env.set_order(None)
    env.reset(tid_d, off_d, session_base=base)

    # ---- e2e: the host-buffer call (Simulator.run semantics: per-session QoE sums + statistics to the host) ----
    # page-locked host tensors: the kernels pull the inputs and push the results over PCIe themselves (zero-copy)
    tid_p = torch.from_numpy(tid_h).pin_memory()
    off_p = torch.from_numpy(off_h).pin_memory()
    qoe_p = torch.empty(N, dtype=torch.float64).pin_memory()
    st_p = torch.empty(_lib.NUM_STATS, dtype=torch.float64).pin_memory()
    host_out = dict(qoe_cost=qoe_p, stats=st_p)
    if rank == 0:
        sampler.pause(True)
    # prepared call: arguments validated and converted once (a caller that repeats a run does the same)
    host_run = env.prepare_run_host("random", V, tid_p, off_p, seed=SEED, session_base=base, want_acc=False, out=host_out)
    for _ in range(10):
        host_run()
    # K calls per block, wall clock (the call synchronises), max over ranks; the median of five blocks is reported —
    # one block lasts ~2 ms, where a single scheduler hiccup of the host is 10 % of the figure
    blocks = []
    for _ in range(5):
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            host_run()
        torch.cuda.synchronize()
        blocks.append(max_over_ranks(time.perf_counter() - t0, dev))
    e2e_s = sorted(blocks)[len(blocks) // 2]
    if rank == 0:
        sampler.pause(False)
    e2e_value = chunk_steps / e2e_s
    h2d = N * 4 + N * 8
    d2h = N * 8 + _lib.NUM_STATS * 8

    # ---- e2e for a caller that wants the whole trajectory on the host (the north star's per-step outputs: delay, sleep,
    #      buffer, rebuffer, reward, end_of_video for every chunk): host inputs -> device, abr_env_run, 41 B per chunk-step
    #      back into pinned host buffers.  PCIe-bound by construction (129 MB per step). ----
    def traj_leg(dev_out, run):
        traj_p = {k: torch.empty(V, N, dtype=t.dtype).pin_memory() for k, t in dev_out.items()}
        traj_ms = []
        for it in range(2 + 5):
            barrier()
            t0 = time.perf_counter()
            tid_d.copy_(tid_p, non_blocking=True)
            off_d.copy_(off_p, non_blocking=True)
            run()
            for k in dev_out:
                traj_p[k].copy_(dev_out[k], non_blocking=True)
            torch.cuda.synchronize()
            if it >= 2:
                traj_ms.append(max_over_ranks(time.perf_counter() - t0, dev) * 1e3)
        traj_ms.sort()
        traj_bytes = sum(t.numel() * t.element_size() for t in traj_p.values())
        med = traj_ms[len(traj_ms) // 2]
        return dict(value=world * N * V / (med * 1e-3), unit="chunk-steps/s", ms_per_step=med, h2d_bytes_per_step=h2d,
                    d2h_bytes_per_step=traj_bytes, d2h_gb_per_s=traj_bytes / (med * 1e-3) / 1e9)

    e2e_traj = traj_leg(out, lambda: env.run("random", V, tid_d, off_d, seed=SEED, session_base=base, out=out,
                                             qoe_cost=False, stats=False))
    e2e_traj["call"] = "abr_env_run + device->host copies of all six [48][N] trajectories into pinned buffers"
    # the fp32-output mode is where the PCIe-bound caller gains: 21 instead of 41 bytes per chunk-step
    out32 = {k: torch.empty(V, N, dtype=torch.float32, device=dev) for k in ("delay", "sleep", "buffer", "rebuffer", "reward")}
    out32["end_of_video"] = out["end_of_video"]

    def run32():
        env.reset(tid_d, off_d, session_base=base)
        env.rollout("random", V, seed=SEED, out=out32)

    e2e_traj["fp32_outputs"] = traj_leg(out32, run32)
    e2e_traj["fp32_outputs"]["call"] = "abr_env_reset + abr_env_rollout_fused_f32 + device->host copies (fp64 arithmetic, outputs rounded once)"
    del out32

    # ---- MPC decisions/s (configs[2] sharded: robust MPC, horizon 5, 7 776 sequences per decision) ----
    mpc = None
    if not args.no_mpc:
        mpc = bench_mpc(args, env, dev, rank, world, base, barrier, max_over_ranks)

    step_form = None
    if not args.no_step_form:
        step_form = bench_step_form(args, dev, rank, world, barrier, max_over_ranks, hbm_peak_gbs())
    rl = None
    if not args.no_step_form and args.rl_sessions > 0:
        rl = bench_rl_harness(args, dev, rank, world, barrier, max_over_ranks)

    clocks = sampler.stop() if rank == 0 else None
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    per_session = BYTES_PER_SESSION if args.separate_reset else BYTES_PER_SESSION_RUN
    alg_bytes = N * V * BYTES_PER_STEP + N * per_session
    achieved = alg_bytes / (kern_avg_ms * 1e-3) / 1e9
    traffic = traffic_all = None
    try:
        traffic_all = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        traffic = traffic_all.get("abr_rollout_kernel")
    except Exception:
        pass
    line = dict(metric="chunk_steps_per_sec", value=value, unit="chunk-steps/s", n_gpus=world, steps=args.steps,
                warmup=max(3, args.warmup), ms_per_step=total_ms / args.steps, higher_is_better=True, scaling="weak",
                vs_baseline=None, dtype="f64", data="synthetic", config=workload_config(args),
                roofline=dict(kernel="abr_rollout_kernel<random>", bound="hbm", achieved=achieved, peak=hbm_peak,
                              unit="GB/s", frac=achieved / hbm_peak, traffic=traffic, peak_source=peak_src,
                              frac_of_nominal_8000_gbs=achieved / 8000.0,
                              algorithmic_bytes_per_launch=alg_bytes, kernel_ms=kern_avg_ms,
                              bytes_per_chunk_step=BYTES_PER_STEP, bytes_per_session=per_session,
                              launch="abr_env_rollout_fused after abr_env_reset" if args.separate_reset else
                                     "abr_env_run: reset and the final statistics reduction fused into the episode kernel "
                                     "(one launch per step)"),
                e2e=dict(value=e2e_value, unit="chunk-steps/s", h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h,
                         call="BatchedABREnv.prepare_run_host(...)() -> abr_env_run_host: reset + fused episode + statistics; the per-session QoE cost that "
                              "Simulator.run() returns ([N] doubles) and the statistics vector, written to pinned host buffers",
                         ms_per_step=1e3 * e2e_s / args.steps, timing="median of 5 blocks of K calls, wall clock, max over ranks",
                         blocks_ms_per_step=[1e3 * b / args.steps for b in blocks],
                         best_block_ms_per_step=1e3 * min(blocks) / args.steps,
                         host_cores=(f"{len(cpus)} cores next to the GPU (NVML affinity)" if cpus else "unbound"),
                         full_trajectory_to_host=e2e_traj),
                gpu_launches=int(launches), clocks=clocks, wall_s_timed_region=wall,
                qoe_stats=dict(zip(_lib.ACC_NAMES, [float(x) for x in tot_stats.cpu()])), flagged_sessions=errors,
                parity=parity)
    if mpc:
        line["mpc"] = mpc
    line["bba_policy"] = bba
    line["fused_kernel_layouts"] = dict(sorted_by_trace=dict(kernel_ms=kern_avg_ms, frac=achieved / hbm_peak,
                                                             note="the headline: 64 consecutive sessions per trace"),
                                        **fused_layouts)
    line["fp32_outputs"] = fp32_outputs
    if step_form:
        line["step_form"] = step_form
        # the per-step-launch kernel is the HBM-bound one (north star: >= 0.6 of peak); repeated at the top level
        line["roofline_step_kernel"] = dict(kernel="abr_step_kernel (one launch per chunk, 4 Mi sessions, state in HBM)",
                                            **step_form["roofline"], traffic=(traffic_all or {}).get("abr_step_kernel"),
                                            algorithmic_bytes_per_launch=step_form["sessions_per_gpu"] * step_form["bytes_per_session_step"],
                                            kernel_ms=step_form["ms_per_launch"])
    if rl:
        line["rl_harness"] = rl
    if per_rank is not None:
        line["per_rank"] = per_rank
    if collective is not None:
        line["collective"] = collective
    if world == 1 and not args.no_cpu_baseline:
        os.sched_setaffinity(0, all_cpus)
        line["cpu_baseline"] = cpu_baseline(args)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def hbm_peak_gbs():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        return 6650.0


def bench_step_form(args, dev, rank, world, barrier, max_over_ranks, hbm_peak):
    """Per-step-launch form (RL-harness shape, configs[4] per GPU): one abr_step_kernel launch per chunk over
    --step-sessions sessions with the SoA state in HBM; 121 algorithmic bytes per session-step.  Measured for two
    session layouts: sorted by trace (every 256-thread block follows one trace and stages its capacity row in shared
    memory) and interleaved (trace = session mod n_traces: every probe is a scattered global load)."""
    import torch
    from abrsimulator_b200 import synth
    from abrsimulator_b200.env import BatchedABREnv, StepResult
    M = args.step_sessions
    bitrates, sizes = synth.make_video(V)
    bw, tl, ti = synth.make_traces(N_TRACES, T_TRACE)
    env = BatchedABREnv(bw, sizes, bitrates, M, trace_len=tl, trace_interval=ti)
    g = torch.Generator(device=dev)
    g.manual_seed(1)
    acts = torch.randint(0, A, (8, M), dtype=torch.int32, device=dev, generator=g)
    out = StepResult(*[torch.empty(M, dtype=torch.float64, device=dev) for _ in range(5)], None,
                     torch.empty(M, dtype=torch.uint8, device=dev), None)
    stream = torch.cuda.current_stream()
    bytes_per = 40 + 4 + 36 + 41      # state read (seg, chunk, last_q, trace_id, phase, pos, buffer) + action, state write, outputs
    res = {}
    for name, group, sort in (("sorted_by_trace", max(256, M // N_TRACES), False), ("interleaved", 1, False),
                              ("interleaved_env_sorted", 1, True)):
        # interleaved: trace = session mod n_traces (SURVEY §8d), every probe of a lane a scattered L2 access;
        # interleaved_env_sorted: the same sessions, the environment keeps them sorted by trace (reset(sort_by_trace=True):
        # abr_sort_by_trace + abr_env_set_order, outside the timed region — the session->trace map is static) and all
        # per-session arrays are in environment order
        tid, off = synth.make_sessions(M, N_TRACES, T_TRACE, session_base=rank * M, group=group)
        env.set_order(None)
        env.reset(tid, off, session_base=rank * M, sort_by_trace=sort)
        for t in range(8):
            env.step(acts[t % 8], out=out)
        barrier()
        reps = 24
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for t in range(reps):
            env.step(acts[t % 8], out=out)
        e1.record(stream)
        e1.synchronize()
        ms = max_over_ranks(e0.elapsed_time(e1), dev) / reps
        achieved = M * bytes_per / (ms * 1e-3) / 1e9
        res[name] = dict(sessions_per_trace_run=group, ms_per_launch=ms,
                         session_steps_per_s=world * M / (ms * 1e-3),
                         roofline=dict(bound="hbm", achieved=achieved, peak=hbm_peak, unit="GB/s",
                                       frac=achieved / hbm_peak))
    # optional fp32-output mode on the trace-sorted layout: 5 x 4 + 1 B of outputs, state and arithmetic unchanged
    out32 = StepResult(*[torch.empty(M, dtype=torch.float32, device=dev) for _ in range(5)], None, out.end_of_video, None)
    tid, off = synth.make_sessions(M, N_TRACES, T_TRACE, session_base=rank * M, group=max(256, M // N_TRACES))
    env.set_order(None)
    env.reset(tid, off, session_base=rank * M)
    for t in range(8):
        env.step(acts[t % 8], out=out32)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for t in range(24):
        env.step(acts[t % 8], out=out32)
    e1.record(stream)
    e1.synchronize()
    ms32 = max_over_ranks(e0.elapsed_time(e1), dev) / 24
    bytes32 = 40 + 4 + 36 + 21
    res["sorted_by_trace_fp32_outputs"] = dict(ms_per_launch=ms32, session_steps_per_s=world * M / (ms32 * 1e-3),
                                               bytes_per_session_step=bytes32,
                                               roofline=dict(bound="hbm", achieved=M * bytes32 / (ms32 * 1e-3) / 1e9,
                                                             peak=hbm_peak, unit="GB/s",
                                                             frac=M * bytes32 / (ms32 * 1e-3) / 1e9 / hbm_peak))
    # the shape configs[4] names (4 Mi sessions over 8 GPUs = 524 288 per GPU): 63 MB of state + outputs per launch fit the
    # 126 MB L2, so a 256 MiB buffer is rewritten between the timed launches (outside the timed region)
    M4 = min(M, 1 << 19)
    cfg4 = None
    if M4 >= 1024:
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        env4 = BatchedABREnv(bw, sizes, bitrates, M4, trace_len=tl, trace_interval=ti)
        tid4, off4 = synth.make_sessions(M4, N_TRACES, T_TRACE, session_base=rank * M4, group=max(256, M4 // N_TRACES))
        env4.reset(tid4, off4, session_base=rank * M4)
        out4 = StepResult(*[torch.empty(M4, dtype=torch.float64, device=dev) for _ in range(5)], None,
                          torch.empty(M4, dtype=torch.uint8, device=dev), None)
        ms4 = []
        for t in range(4 + 12):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            env4.step(acts[t % 8][:M4], out=out4)
            e1.record(stream)
            e1.synchronize()
            if t >= 4:
                ms4.append(e0.elapsed_time(e1))
        m4 = max_over_ranks(sum(ms4), dev) / len(ms4)
        cfg4 = dict(sessions_per_gpu=M4, ms_per_launch=m4, session_steps_per_s=world * M4 / (m4 * 1e-3),
                    roofline=dict(bound="hbm", achieved=M4 * bytes_per / (m4 * 1e-3) / 1e9, peak=hbm_peak, unit="GB/s",
                                  frac=M4 * bytes_per / (m4 * 1e-3) / 1e9 / hbm_peak),
                    l2="256 MiB buffer rewritten between timed launches")
        del env4, flush
    best = res["sorted_by_trace"]
    return dict(kernel="abr_step_kernel", sessions_per_gpu=M, configs4_shape=cfg4, ms_per_launch=best["ms_per_launch"],
                session_steps_per_s=best["session_steps_per_s"], bytes_per_session_step=bytes_per,
                roofline=best["roofline"], layouts=res,
                note="4 Mi sessions per GPU (no config names this size: it is chosen so that 304 MB of SoA state + 172 MB "
                     "of outputs per launch exceed the 126 MB L2 and back-to-back launches measure HBM); configs4_shape is the "
                     "per-GPU shape of configs[4] with the L2 flushed between launches; headline = sessions sorted by trace "
                     "(shared-memory staged capacity rows)")


def bench_rl_harness(args, dev, rank, world, barrier, max_over_ranks):
    """RL rollout harness (configs[4] per GPU): a batched torch policy (MLP, fp32) <-> abr_env_step with every state
    tensor on the device, one 48-chunk episode of --rl-sessions sessions.  The policy kernels are torch's; the
    environment step, the observation inputs (throughput, next-chunk sizes) and the state are this library's."""
    import torch
    from abrsimulator_b200 import synth
    from abrsimulator_b200.env import BatchedABREnv
    from examples.rl_harness import Policy, GraphedEpisode
    M = args.rl_sessions
    bitrates, sizes = synth.make_video(V)
    bw, tl, ti = synth.make_traces(N_TRACES, T_TRACE)
    env = BatchedABREnv(bw, sizes, bitrates, M, trace_len=tl, trace_interval=ti)
    tid, off = synth.make_sessions(M, N_TRACES, T_TRACE, session_base=rank * M, group=max(256, M // N_TRACES))
    torch.manual_seed(0)
    torch.backends.cuda.matmul.allow_tf32 = True
    policy = Policy(4 + A, A).to(dev)
    stream = torch.cuda.current_stream()
    env.reset(tid, off, session_base=rank * M)
    res = {}
    for name, fused in (("fused", True), ("torch_glue", False)):
        env.reset(tid, off, session_base=rank * M)
        runner = GraphedEpisode(env, policy, fused=fused)
        runner.run(1)                                   # capture outside the timed episodes
        ms = []
        for ep in range(3):
            env.reset(tid, off, session_base=rank * M)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            total = runner.run(V)
            e1.record(stream)
            e1.synchronize()
            ms.append(max_over_ranks(e0.elapsed_time(e1), dev))
        best = min(ms[1:])
        res[name] = dict(ms_per_episode=best, env_steps_per_s=world * M * V / (best * 1e-3),
                         mean_episode_reward=float(total.mean().item()))
        del runner
    return dict(sessions_per_gpu=M, chunks=V, ms_per_episode=res["fused"]["ms_per_episode"],
                env_steps_per_s=res["fused"]["env_steps_per_s"], mean_episode_reward=res["fused"]["mean_episode_reward"],
                torch_glue=res["torch_glue"],
                note="policy forward (torch MLP, tf32) + abr_env_step_policy: Gumbel-max sampling, step, reward sum and the "
                     "fp32 feature-major observation in one library launch per chunk; one chunk captured into a CUDA graph "
                     "and replayed; state never leaves the device.  torch_glue: the same episode with the sampling and the "
                     "observation in eager PyTorch around abr_env_step (twelve more kernels per chunk)")


def bench_mpc(args, env, dev, rank, world, base, barrier, max_over_ranks):
    import torch
    from abrsimulator_b200 import synth, _lib
    from abrsimulator_b200.env import BatchedABREnv
    import ctypes as C
    H, M = args.mpc_horizon, args.mpc_sessions
    bitrates, sizes = synth.make_video(V)
    bw, tl, ti = synth.make_traces(N_TRACES, T_TRACE)
    menv = BatchedABREnv(bw, sizes, bitrates, M, trace_len=tl, trace_interval=ti, track_history=1, track_acc=1)
    tid, off = synth.make_sessions(M, N_TRACES, T_TRACE, session_base=rank * M, group=GROUP)
    menv.reset(tid, off, session_base=rank * M)
    menv.rollout("bba", 8, want=())                              # fill the throughput-history ring
    act = torch.empty(M, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream()
    for _ in range(3):
        menv.mpc_decide(H, "robust", out=act)
    barrier()
    reps = max(3, min(args.steps, 10))
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        menv.mpc_decide(H, "robust", out=act)
        e1.record(stream)
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    barrier()
    tot = max_over_ranks(sum(ms), dev)
    dec_per_s = world * M * reps / (tot * 1e-3)
    mpc_parity = parity_mpc(menv, H, act, sample=32768) if rank == 0 else None     # outside the timed launches
    # the same decisions by exhaustive enumeration (all A^H sequences, as scipy.optimize.brute does): the kernel the
    # FP64-issue roofline below is about; the default above is branch and bound with identical results
    act_x = torch.empty_like(act)
    for _ in range(2):
        menv.mpc_decide(H, "robust", out=act_x, exhaustive=True)
    ms_x = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        menv.mpc_decide(H, "robust", out=act_x, exhaustive=True)
        e1.record(stream)
        e1.synchronize()
        ms_x.append(e0.elapsed_time(e1))
    menv.mpc_decide(H, "robust", out=act)
    same_as_exhaustive = bool(torch.equal(act, act_x))
    exh_per_s = world * M * reps / (max_over_ranks(sum(ms_x), dev) * 1e-3)
    # reference-exact mode for comparison
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    menv.mpc_decide(H, "reference", out=act)
    e0.record(stream)
    menv.mpc_decide(H, "reference", out=act)
    e1.record(stream)
    e1.synchronize()
    ref_mode_rate = M / (e0.elapsed_time(e1) * 1e-3)
    # whole MPC episode (decide + step per chunk) for one video, with final statistics
    menv.reset(tid, off, session_base=rank * M)
    barrier()
    e0.record(stream)
    menv.mpc_episode(V, H, "robust")
    st = menv.stats()
    e1.record(stream)
    e1.synchronize()
    ep_ms = max_over_ranks(e0.elapsed_time(e1), dev)
    # configs[3]: horizon-7 stress (279 936 sequences per decision), 16 384 sessions over 8 GPUs = 2 048 per GPU;
    # too few sessions for a warp each, so the kernel gives every session a whole 128-thread block
    h7 = None
    if args.mpc_h7_sessions > 0:
        M7 = args.mpc_h7_sessions
        env7 = BatchedABREnv(bw, sizes, bitrates, M7, trace_len=tl, trace_interval=ti, track_history=1)
        tid7, off7 = synth.make_sessions(M7, N_TRACES, T_TRACE, session_base=rank * M7, group=GROUP)
        env7.reset(tid7, off7, session_base=rank * M7)
        env7.rollout("bba", 8, want=())
        act7 = torch.empty(M7, dtype=torch.int32, device=dev)
        env7.mpc_decide(7, "robust", out=act7)
        barrier()
        e0.record(stream)
        for _ in range(3):
            env7.mpc_decide(7, "robust", out=act7)
        e1.record(stream)
        e1.synchronize()
        ms7 = max_over_ranks(e0.elapsed_time(e1), dev) / 3
        h7 = dict(horizon=7, sequences_per_decision=A ** 7, sessions_per_gpu=M7, ms_per_launch=ms7,
                  decisions_per_s=world * M7 / (ms7 * 1e-3), sequences_per_s=world * M7 * A ** 7 / (ms7 * 1e-3))
    # configs[2] as BASELINE.json words it: "1M sessions sharded across 1/2/4/8 B200, final QoE all-reduce over NVLink" —
    # a fixed total (strong scaling).  Timed region, CUDA events on the launching stream, max over ranks: reset + 48 x
    # (decide + step) + statistics reduction + the all-gather of the per-rank statistics (the one collective).
    strong = None
    if args.mpc_strong_total > 0:
        from abrsimulator_b200.distributed import allreduce_stats, shard_range
        lo, hi = shard_range(args.mpc_strong_total, rank, world)
        Ms = hi - lo
        senv = menv if Ms <= M else BatchedABREnv(bw, sizes, bitrates, Ms, trace_len=tl, trace_interval=ti,
                                                  track_history=1, track_acc=1)
        tid_s, off_s = synth.make_sessions(Ms, N_TRACES, T_TRACE, session_base=lo, group=GROUP)
        tid_sd, off_sd = torch.from_numpy(tid_s).to(dev), torch.from_numpy(off_s).to(dev)
        coll_ms = []
        tot_ms = []
        for it in range(2):                                        # first pass warms up (NCCL communicator, allocator)
            barrier()
            e0.record(stream)
            senv.reset(tid_sd, off_sd, session_base=lo)
            senv.mpc_episode(V, H, "robust")
            st_s = senv.stats()
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record(stream)
            tot_s = allreduce_stats(st_s)
            c1.record(stream)
            e1.record(stream)
            e1.synchronize()
            tot_ms.append(max_over_ranks(e0.elapsed_time(e1), dev))
            coll_ms.append(max_over_ranks(c0.elapsed_time(c1), dev))
        strong = dict(workload="configs[2]: robust MPC, horizon 5, fixed total sharded over the GPUs, whole 48-chunk "
                               "episode + final statistics all-reduce", scaling="strong",
                      total_sessions=args.mpc_strong_total, sessions_per_gpu=Ms, chunks=V, ms=tot_ms[-1],
                      decisions_per_s=args.mpc_strong_total * V / (tot_ms[-1] * 1e-3),
                      collective=dict(op="all_gather of the per-rank statistics vector + rank-order sum (deterministic)",
                                      bytes_per_rank=int(st_s.numel() * 8), ms=coll_ms[-1], inside_timed_region=True,
                                      backend="nccl" if world > 1 else "none (one rank)"),
                      mean_reward_per_chunk=float(tot_s[0] / tot_s[6]), steps_total=float(tot_s[6]))
        if senv is not menv:
            del senv
    res = dict(metric="mpc_decisions_per_sec", value=dec_per_s, unit="decisions/s", horizon=H, mode="robust",
               search="branch and bound over the A^H sequences (exact: the decisions of the exhaustive enumeration, "
                      "checked in this run)",
               exhaustive=dict(decisions_per_s=exh_per_s, ms_per_launch=sum(ms_x) / len(ms_x),
                               identical_decisions=same_as_exhaustive),
               sequences_per_decision=A ** H, sessions_per_gpu=M, ms_per_launch=sum(ms) / len(ms),
               reference_exact_mode_decisions_per_s_per_gpu=ref_mode_rate,
               episode=dict(chunks=V, ms=ep_ms, decisions_per_s=world * M * V / (ep_ms * 1e-3),
                            mean_reward_per_chunk=float(st[0] / st[6])), horizon7=h7, parity=mpc_parity, strong_scaling=strong)
    if rank == 0:
        # drop-in controller latency: one next_bitrate() through abr_mpc_decide_host (mpc_test.py's scenario, horizon 5);
        # the reference's own mpc.py + scipy.optimize.brute: 0.14-0.19 s per A=6, H=5 decision, 26 ms at A=4 (SURVEY.md:199)
        from examples.mpc_dropin import reference_scenario
        from abrsimulator_b200.mpc import MPCBitrateController
        ctl = MPCBitrateController(reference_scenario()[0], horizon=H, strict_history=False)
        lat = []
        for it in range(60):
            t0 = time.perf_counter()
            ctl.next_bitrate()
            if it >= 10:
                lat.append((time.perf_counter() - t0) * 1e6)
        lat.sort()
        res["single_decision"] = dict(call="MPCBitrateController(player, horizon=5).next_bitrate() -> abr_mpc_decide_host "
                                           "(one host->device copy, one kernel, one device->host copy; no allocation)",
                                      median_us=lat[len(lat) // 2], p90_us=lat[int(len(lat) * 0.9)])
        lib = _lib.load()
        probe = {}
        for kind, name in ((0, "dadd"), (1, "dfma"), (2, "dadd_dmul_dsetp_mix")):
            g = C.c_double(0.0)
            t = C.c_float(0.0)
            _lib.check(lib.abr_fp64_probe(C.c_int(kind), C.c_int(4096), C.byref(g), C.byref(t), None))
            probe[name + "_gops"] = g.value
        # fp64-pipe thread-instructions the search executes per decision (DESIGN.md §5), counted from the SASS of the
        # inner loops: per prefix slot (rounded up to whole warps) one interior step (9) + A interior steps (9 each) +
        # A^2 leaves (7 arithmetic + 1 compare with smooth_penalty == 1), plus the parent-state cache fill
        # useful work only: the A^(H-2) = 216 real prefixes (the 8 idle lane-slots of the seventh warp-round are not
        # counted as achieved work)
        prefixes = A ** (H - 2)
        executed = prefixes * (9 + A * 9 + A * A * 8) + (A ** (H - 3) if H >= 3 else 0) * (H - 3) * 9
        naive = A ** H * (14 * (H - 1) + 13) + 4 * A * H
        peak = probe["dadd_gops"]
        res["roofline"] = dict(kernel="abr_mpc_kernel, exhaustive enumeration (ABR_MPC_EXHAUSTIVE)",
                               bound="fp64-issue", unit="Gop/s", peak=peak, peak_source="abr_fp64_probe (DADD chains, same run)",
                               probe=probe, executed_fp64_ops_per_decision=executed,
                               achieved=exh_per_s / world * executed / 1e9, frac=exh_per_s / world * executed / 1e9 / peak,
                               naive_equivalent_ops_per_decision=naive,
                               naive_equivalent_gops=dec_per_s / world * naive / 1e9,
                               note="the default search (branch and bound) executes about a third of these operations and is "
                                    "bound by the latency of its phases, not by FP64 issue")
    return res


def cpu_baseline(args):
    """The oracle port timed on this box's host cores, bounded sample (reported baseline, not the target)."""
    rate, steps, busy, _ = cpu_python_steps(1, args.cpu_seconds)
    c_rate, c_n, c_dt = cpu_c_oracle_steps()
    out = dict(value=rate, unit="chunk-steps/s", cores=1, kind="port",
               sample=f"pure-Python port (oracle/step_oracle.py) of the same random-policy workload: {steps} chunk-steps "
                      f"in {busy:.1f} s on 1 core of {os.cpu_count()}",
               c_oracle=dict(value=c_rate, unit="chunk-steps/s", cores=1,
                             sample=f"oracle/abr_oracle.c (gcc -O2), {c_n} sessions x 48 chunks in {c_dt:.2f} s"))
    if not args.no_mpc:
        r, n, b = cpu_python_mpc(1, args.mpc_horizon, args.cpu_seconds)
        out["mpc"] = dict(value=r, unit="decisions/s", cores=1,
                          sample=f"pure-Python port of mpc.py's search (oracle/mpc_oracle.py), {n} horizon-"
                                 f"{args.mpc_horizon} decisions in {b:.1f} s")
        try:    # the real thing cannot travel to the GPU box: the build-box record of oracle/time_reference_mpc.py
            rec = json.load(open(os.path.join(ROOT, "profiles", "ref_mpc_cpu_baseline.json")))
            out["mpc"]["reference_mpc_py_on_build_box"] = dict(
                decisions_per_s_one_core=rec["reference_mpc_py"]["one_core"]["decisions_per_s"],
                decisions_per_s_all_cores=rec["reference_mpc_py"]["all_cores"]["decisions_per_s"],
                cores=rec["cores"], impl=rec["reference_mpc_py"]["impl"], port_over_reference=rec["port_over_reference"],
                note="unmodified /root/reference/mpc.py + scipy.optimize.brute on the same inputs, measured in the build "
                     "container by oracle/time_reference_mpc.py (committed record profiles/ref_mpc_cpu_baseline.json)")
        except Exception:
            pass
    return out


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
