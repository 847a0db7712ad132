"""What per-session policy parameters (SPEC §4.7) cost, and what they save in a parameter sweep.

1. Overhead: the 65 536 x 48 episode on the bench world (synth video, 1 024 x 2 048 traces, 64 consecutive sessions
   per trace), six trajectory outputs, on one environment with track_history = 1, for BBA, RATE, BOLA and DYNAMIC,
   environment-wide against per-session parameters holding the same values.  The legs are interleaved launch by launch;
   every launch is preceded by a reset (untimed) and by overwriting a 256 MB buffer (the L2 holds 126 MB); CUDA events
   around each rollout.
2. Sweep: G = 64 points x 1 024 sessions.  Per-session: one launch of 65 536 sessions with the points installed.
   Environment-wide: 64 x (set_policy_params + reset + a 1 024-session launch) on one environment, as a sweep must run
   without per-session parameters.  Both end to end (host clock around the whole sweep, ending in a synchronise;
   per-session installation included), L2 overwritten once in front of each sweep.
3. Decision: policy_decide at 4 Mi sessions (state after eight steps of the rate policy), with and without per-session
   parameters, L2 overwritten in front of every launch.

usage: python profiles/time_session_params.py [launches=100] [out.json]"""
import json
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, ".")
from abrsimulator_b200 import synth
from abrsimulator_b200.env import BatchedABREnv

n_iter = int(sys.argv[1]) if len(sys.argv) > 1 else 100
out_path = sys.argv[2] if len(sys.argv) > 2 else None
assert torch.cuda.is_available(), "this measurement needs the GPU"
dev = torch.device("cuda", 0)
name = torch.cuda.get_device_name(0)
try:
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError):
    power = "unknown"

N, V, steps = 65536, 48, 48
bitrates, sizes = synth.make_video(V)
bw, tl, ti = synth.make_traces(1024, 2048)
tid, off = synth.make_sessions(N, 1024, 2048, group=64)
tid_d, off_d = torch.from_numpy(tid).to(dev), torch.from_numpy(off).to(dev)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, track_history=1)
WIDE = dict(bba_reservoir=5.0, bba_cushion=10.0, rb_safety=1.0, bola_min_buffer=10.0, bola_target_buffer=30.0,
            switch_on_buffer=12.0, switch_off_buffer=6.0)
same = {k: torch.full((N,), v, dtype=torch.float64, device=dev) for k, v in WIDE.items()}


def outputs():
    o = {k: torch.empty(steps, N, dtype=torch.float64, device=dev) for k in ("delay", "sleep", "buffer", "rebuffer", "reward")}
    o["end_of_video"] = torch.empty(steps, N, dtype=torch.uint8, device=dev)
    return o


def summary(us, work):
    us = sorted(us)
    mean = sum(us) / len(us)
    return dict(launches=len(us), mean_us=round(mean, 2), median_us=round(us[len(us) // 2], 2),
                p10_us=round(us[len(us) // 10], 2), p90_us=round(us[9 * len(us) // 10], 2),
                per_second=round(work / (mean * 1e-6), 0))


# ---- 1. overhead ----
pols = ["bba", "rate", "bola", "dynamic"]
legs = [(p, s) for p in pols for s in (False, True)]
outs = {leg: outputs() for leg in legs}
ev = {leg: [] for leg in legs}
for it in range(n_iter + 10):
    for leg in legs:
        pol, per_session = leg
        env.reset(tid_d, off_d)
        if per_session:
            env.set_session_policy_params(**same)
        flush.fill_(it & 0xff)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        env.rollout(pol, steps, seed=7, out=outs[leg])
        e1.record()
        if per_session:
            env.set_session_policy_params(None)
        if it >= 10:
            ev[leg].append((e0, e1))
torch.cuda.synchronize()
assert env.error_count() == 0
for pol in pols:   # identical values: identical bits
    for k in outs[(pol, False)]:
        assert torch.equal(outs[(pol, False)][k], outs[(pol, True)][k]), (pol, k)
result = dict(gpu=name, power_limit_and_max_sm_clock=power,
              episode=dict(sessions=N, steps=steps, layout="sorted by trace (64 sessions per trace)",
                           environment="track_history = 1 for every leg (the general kernel form)",
                           L2="256 MB overwritten before every launch", unit_per_second="chunk-steps/s",
                           outputs_identical_between_the_legs=True),
              rollout={})
for leg in legs:
    key = f"{leg[0]}_{'per_session' if leg[1] else 'environment_wide'}"
    result["rollout"][key] = summary([1e3 * a.elapsed_time(b) for a, b in ev[leg]], N * steps)
del env, outs

# ---- 2. sweep: 64 points x 1 024 sessions ----
G, P = 64, 1024
g = np.arange(G)
grid = dict(rb_safety=0.5 + 0.01 * g, bola_min_buffer=4.0 + 0.2 * g, bola_target_buffer=25.0 + 0.5 * g)
tid_p, off_p = synth.make_sessions(P, 1024, 2048, group=64)
tid_s, off_s = np.tile(tid_p, G), np.tile(off_p, G)
sweep_env = BatchedABREnv(bw, sizes, bitrates, G * P, trace_len=tl, trace_interval=ti, track_history=1)
point_env = BatchedABREnv(bw, sizes, bitrates, P, trace_len=tl, trace_interval=ti, track_history=1)
tid_sd, off_sd = torch.from_numpy(tid_s).to(dev), torch.from_numpy(off_s).to(dev)
tid_pd, off_pd = torch.from_numpy(tid_p).to(dev), torch.from_numpy(off_p).to(dev)
fields = {k: torch.from_numpy(np.repeat(v, P)).to(dev) for k, v in grid.items()}
o_sweep = {k: torch.empty(steps, G * P, dtype=torch.float64, device=dev) for k in ("reward",)}
o_point = {k: torch.empty(steps, P, dtype=torch.float64, device=dev) for k in ("reward",)}
res_sweep = {p: [] for p in ("rate", "bola", "dynamic")}
res_points = {p: [] for p in ("rate", "bola", "dynamic")}
n_sweep = max(10, n_iter // 5)
for it in range(n_sweep + 2):
    for pol in res_sweep:
        flush.fill_(it & 0xff)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sweep_env.reset(tid_sd, off_sd)
        sweep_env.set_session_policy_params(**fields)
        sweep_env.rollout(pol, steps, out=o_sweep)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        flush.fill_((it + 1) & 0xff)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        for j in range(G):
            point_env.set_policy_params(rb_safety=grid["rb_safety"][j], bola_min_buffer=grid["bola_min_buffer"][j],
                                        bola_target_buffer=grid["bola_target_buffer"][j])
            point_env.reset(tid_pd, off_pd)
            point_env.rollout(pol, steps, out=o_point)
        torch.cuda.synchronize()
        t3 = time.perf_counter()
        if it >= 2:
            res_sweep[pol].append(1e6 * (t1 - t0))
            res_points[pol].append(1e6 * (t3 - t2))
        if it == 0:   # the last point of both runs agrees bit for bit
            assert torch.equal(o_sweep["reward"][:, (G - 1) * P:], o_point["reward"]), pol
result["sweep"] = dict(points=G, sessions_per_point=P, steps=steps,
                       per_session="reset + set_session_policy_params + one 65 536-session launch",
                       environment_wide="64 x (set_policy_params + reset + a 1 024-session launch)",
                       timing="host clock around the whole sweep, ending in a synchronise", unit_per_second="chunk-steps/s")
for pol in res_sweep:
    a, b = summary(res_sweep[pol], G * P * steps), summary(res_points[pol], G * P * steps)
    result["sweep"][pol] = dict(per_session=a, environment_wide=b, speedup=round(b["mean_us"] / a["mean_us"], 2))
del sweep_env, point_env

# ---- 3. decision at 4 Mi sessions ----
Nd = 1 << 22
tid4, off4 = synth.make_sessions(Nd, 1024, 2048, group=64)
env4 = BatchedABREnv(bw, sizes, bitrates, Nd, trace_len=tl, trace_interval=ti, track_history=1)
env4.reset(torch.from_numpy(tid4).to(dev), torch.from_numpy(off4).to(dev))
env4.rollout("rate", 8, want=())
act = torch.empty(Nd, dtype=torch.int32, device=dev)
same4 = {k: torch.full((Nd,), v, dtype=torch.float64, device=dev) for k, v in WIDE.items()}
evd = {(p, s): [] for p in pols for s in (False, True)}
for it in range(n_iter + 10):
    for pol in pols:
        for per_session in (False, True):
            if per_session:
                env4.set_session_policy_params(**same4)
            flush.fill_(it & 0xff)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            env4.policy_decide(pol, out=act)
            e1.record()
            if per_session:
                env4.set_session_policy_params(None)
            if it >= 10:
                evd[(pol, per_session)].append((e0, e1))
torch.cuda.synchronize()
assert env4.error_count() == 0
result["decide"] = dict(sessions=Nd, state="after 8 steps of the rate policy", unit_per_second="decisions/s",
                        L2="256 MB overwritten before every launch")
for (pol, s), pairs in evd.items():
    result["decide"][f"{pol}_{'per_session' if s else 'environment_wide'}"] = summary(
        [1e3 * a.elapsed_time(b) for a, b in pairs], Nd)

line = json.dumps(result, indent=1)
print(line)
if out_path:
    with open(out_path, "w") as f:
        f.write(line + "\n")
