"""What the catch-up speed controller of live mode (SPEC §7.2) costs next to the [V][N] speed table, and what it does
to latency and rebuffering.

World: the bench world (synth video V = 48, 1 024 x 2 048 traces, sessions sorted by trace: 64 consecutive sessions per
trace) with live = 1, start_up_length = 8 s and latency_tick = 1 (so the latency accumulator over the content played
is the mean latency in seconds).  Every timed launch is preceded by overwriting a 256 MB buffer (the L2 holds 126 MB);
CUDA events around each launch; the three legs (no table, a constant [V][N] table of 1.0, the controller with its
defaults) are interleaved launch by launch so that they share the machine's noise.

* Episode: the fused live episode, 65 536 sessions x 48 chunks, policies ``bba`` and ``dynamic`` (track_history = 1),
  the six trajectory outputs and the latency requested; a reset (untimed) before every launch.
* Step: the per-step live step at 4 Mi sessions with a fixed action vector, state after eight steps.
* Effect (a result, not a timing): for target_latency in {8, 12, 16, 24} s against no control, the BBA episode of
  65 536 x 48 on the device gives the mean latency (sum of the latency integral / sum of content played) and the
  rebuffering per session; the shares of played chunks above, below and at 1 come from the CPU oracle of the
  controller (tests/speed_oracle.py, bit-identical to the kernels) on the first 4 096 sessions.

usage: python profiles/time_speed_control.py [launches=100] [out.json]"""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
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
P = dict(live=1, start_up_length=8.0, latency_tick=1.0, track_history=1)
bitrates, sizes = synth.make_video(V)
bw, tl, ti = synth.make_traces(1024, 2048)
tid, off = synth.make_sessions(N, 1024, 2048, group=64)
tid_d, off_d = torch.from_numpy(tid).to(dev), torch.from_numpy(off).to(dev)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
LEGS = ("none", "table_of_ones", "controller")


def summary(pairs, work):
    us = sorted(1e3 * a.elapsed_time(b) for a, b in pairs)
    mean = sum(us) / len(us)
    return dict(launches=len(us), mean_us=round(mean, 2), median_us=round(us[len(us) // 2], 2),
                p10_us=round(us[len(us) // 10], 2), p90_us=round(us[9 * len(us) // 10], 2),
                per_second=round(work / (mean * 1e-6), 0))


def set_leg(env, leg):
    if leg == "controller":
        env.set_speed_control()
    else:
        env.set_speed_control(None)


result = dict(gpu=name, power_limit_and_max_sm_clock=power,
              world=dict(video="synth V = 48", traces="1 024 x 2 048", layout="sorted by trace (64 sessions per trace)",
                         live="start_up_length = 8 s, latency_tick = 1", L2="256 MB overwritten before every launch",
                         controller="defaults: target_latency 12 s, max_drift 0.5, gain 2.5 /s, dead_band 0.02 s, "
                                    "min_buffer 6 s"))

# ---- fused live episode ----
env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, **P)
ones = torch.ones(V, N, dtype=torch.float64, device=dev)
out = {k: torch.empty(steps, N, dtype=torch.float64, device=dev)
       for k in ("delay", "sleep", "buffer", "rebuffer", "reward", "latency")}
out["end_of_video"] = torch.empty(steps, N, dtype=torch.uint8, device=dev)
result["episode"] = dict(sessions=N, steps=steps, unit_per_second="chunk-steps/s")
for pol in ("bba", "dynamic"):
    ev = {leg: [] for leg in LEGS}
    for it in range(n_iter + 5):
        for leg in LEGS:
            set_leg(env, leg)
            env.reset(tid_d, off_d)
            flush.fill_(it & 0xff)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            env.rollout(pol, steps, seed=7, out=out, speed=ones if leg == "table_of_ones" else None)
            e1.record()
            if it >= 5:
                ev[leg].append((e0, e1))
    torch.cuda.synchronize()
    result["episode"][pol] = {leg: summary(ev[leg], N * steps) for leg in LEGS}
assert env.error_count() == 0
del env, out, ones

# ---- per-step live step at 4 Mi sessions ----
Ns = 1 << 22
tid4, off4 = synth.make_sessions(Ns, 1024, 2048, group=64)
tid4_d, off4_d = torch.from_numpy(tid4).to(dev), torch.from_numpy(off4).to(dev)
env4 = BatchedABREnv(bw, sizes, bitrates, Ns, trace_len=tl, trace_interval=ti, **P)
act = torch.from_numpy((np.arange(Ns) % 6).astype(np.int32)).to(dev)
ones4 = torch.ones(V, Ns, dtype=torch.float64, device=dev)
env4.reset(tid4_d, off4_d)
res = env4.step(act)
ev = {leg: [] for leg in LEGS}
for it in range(n_iter + 5):
    for leg in LEGS:
        set_leg(env4, leg)
        env4.reset(tid4_d, off4_d)
        for _ in range(8):
            env4.step(act, out=res, speed=ones4 if leg == "table_of_ones" else None)
        flush.fill_(it & 0xff)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        env4.step(act, out=res, speed=ones4 if leg == "table_of_ones" else None)
        e1.record()
        if it >= 5:
            ev[leg].append((e0, e1))
torch.cuda.synchronize()
assert env4.error_count() == 0
result["step"] = dict(sessions=Ns, state="after 8 steps", unit_per_second="chunk-steps/s",
                      **{leg: summary(ev[leg], Ns) for leg in LEGS})
del env4, ones4, res

# ---- effect: latency, rebuffering and speeds ----
import speed_oracle as sp   # noqa: E402

n_orc = 4096
effect = []
for target in (None, 8.0, 12.0, 16.0, 24.0):
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, track_acc=1, **P)
    if target is not None:
        env.set_speed_control(target_latency=target)
    env.reset(tid_d, off_d)
    env.rollout("bba", steps, want=())
    acc = env.session_acc().double()
    row = dict(target_latency=target, mean_latency_s=round(float(acc[9].sum() / acc[10].sum()), 3),
               rebuffer_s_per_session=round(float(acc[1].mean()), 3))
    ref = sp.SpeedEnv(bw, tl, ti, sizes, bitrates, n_orc, **P)
    if target is not None:
        ref.set_speed_control(target_latency=target)
    log = ref.start_log(fill=np.nan)
    ref.reset(tid[:n_orc], off[:n_orc])
    ref.rollout(2, steps)
    x = log[~np.isnan(log)]
    if target is not None:
        assert np.array_equal(ref.play_speed, env.state("play_speed")[:n_orc].cpu().numpy()), "oracle and kernel differ"
        row.update(chunks_decided=int(x.size), share_above_1=round(float((x > 1.0).mean()), 4),
                   share_below_1=round(float((x < 1.0).mean()), 4), share_at_1=round(float((x == 1.0).mean()), 4))
    effect.append(row)
result["effect"] = dict(policy="bba", sessions=N, steps=steps, speed_shares="CPU oracle, first 4 096 sessions",
                        rows=effect)

line = json.dumps(result, indent=1)
print(line)
if out_path:
    with open(out_path, "w") as f:
        f.write(line + "\n")
