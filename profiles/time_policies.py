"""What the built-in policies cost in the fused episode, and what the batched per-step decision costs.

Episode: 65 536 sessions x 48 chunks on the bench world (synth video, 1 024 x 2 048 traces, sessions sorted by trace:
64 consecutive sessions per trace), the six trajectory outputs requested.  ``random``, ``bba`` and ``bola`` run on the
bench's environment (no history: the FAST kernel forms); ``rate`` needs the throughput history, so it runs on the same
world with track_history = 1 (the general form), next to ``bba`` on that environment, which isolates what the ring costs
from what the rule costs.  Every launch is preceded by a reset (untimed) and by overwriting a 256 MB buffer (the L2 holds
126 MB); CUDA events around each rollout; the policies are interleaved launch by launch so that they share the machine's
noise.  Decision: ``policy_decide`` for 4 Mi sessions (state after eight steps of the rate policy), L2 overwritten in
front of every launch.

usage: python profiles/time_policies.py [launches=200] [out.json]"""
import json
import subprocess
import sys

import torch

sys.path.insert(0, ".")
from abrsimulator_b200 import synth
from abrsimulator_b200.env import BatchedABREnv

n_iter = int(sys.argv[1]) if len(sys.argv) > 1 else 200
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
env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti)
env_h = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, track_history=1)


def outputs():
    o = {k: torch.empty(steps, N, dtype=torch.float64, device=dev) for k in ("delay", "sleep", "buffer", "rebuffer", "reward")}
    o["end_of_video"] = torch.empty(steps, N, dtype=torch.uint8, device=dev)
    return o


legs = [("random", env), ("bba", env), ("bola", env), ("bba", env_h), ("rate", env_h)]
outs = [outputs() for _ in legs]
ev = [[] for _ in legs]
for it in range(n_iter + 10):
    for j, (pol, e) in enumerate(legs):
        e.reset(tid_d, off_d)
        flush.fill_(it & 0xff)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        e.rollout(pol, steps, seed=7, out=outs[j])
        e1.record()
        if it >= 10:
            ev[j].append((e0, e1))
torch.cuda.synchronize()
assert env.error_count() == 0 and env_h.error_count() == 0


def summary(pairs, work):
    us = sorted(1e3 * a.elapsed_time(b) for a, b in pairs)
    mean = sum(us) / len(us)
    return dict(launches=len(us), mean_us=round(mean, 2), median_us=round(us[len(us) // 2], 2),
                p10_us=round(us[len(us) // 10], 2), p90_us=round(us[9 * len(us) // 10], 2),
                per_second=round(work / (mean * 1e-6), 0))


result = dict(gpu=name, power_limit_and_max_sm_clock=power,
              episode=dict(sessions=N, steps=steps, layout="sorted by trace (64 sessions per trace)",
                           L2="256 MB overwritten before every launch", unit_per_second="chunk-steps/s"),
              rollout={})
for j, (pol, e) in enumerate(legs):
    key = pol + ("_track_history" if e is env_h else "")
    result["rollout"][key] = summary(ev[j], N * steps)
del env, env_h, outs

# ---- batched decision at 4 Mi sessions ----
Nd = 1 << 22
tid4, off4 = synth.make_sessions(Nd, 1024, 2048, group=64)
env4 = BatchedABREnv(bw, sizes, bitrates, Nd, trace_len=tl, trace_interval=ti, track_history=1)
env4.reset(torch.from_numpy(tid4).to(dev), torch.from_numpy(off4).to(dev))
env4.rollout("rate", 8, want=())
act = torch.empty(Nd, dtype=torch.int32, device=dev)
dec = ["bba", "rate", "bola"]
evd = [[] for _ in dec]
for it in range(n_iter + 10):
    for j, pol in enumerate(dec):
        flush.fill_(it & 0xff)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        env4.policy_decide(pol, out=act)
        e1.record()
        if it >= 10:
            evd[j].append((e0, e1))
torch.cuda.synchronize()
assert env4.error_count() == 0
result["decide"] = dict(sessions=Nd, state="after 8 steps of the rate policy", unit_per_second="decisions/s",
                        L2="256 MB overwritten before every launch")
for j, pol in enumerate(dec):
    result["decide"][pol] = summary(evd[j], Nd)

line = json.dumps(result, indent=1)
print(line)
if out_path:
    with open(out_path, "w") as f:
        f.write(line + "\n")
