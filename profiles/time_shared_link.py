"""What a shared-link run (SPEC §9, abr_env_run_shared) costs, in downloads per second.

The bench world (synth video of 48 chunks, 1 024 x 2 048 traces), 65 536 players x 48 chunks, link l on trace
l mod 1 024, for G in {1, 2, 4, 8, 16, 32} players per link and the policies bba, bola, rate, dynamic and mixed
{bola, rate} (alternating slots); the six trajectory outputs, request_time and the three link outputs, the accumulators,
qoe_cost and the statistics.  Beside it, abr_env_run on the same 65 536 sessions, and the pure-Python oracle
(tests/shared_link_oracle.py) on one core, per download.  Every launch is preceded by overwriting a 256 MB buffer
(the L2 holds 126 MB); CUDA events around each call; the legs are interleaved launch by launch.

usage: python profiles/time_shared_link.py [launches=10] [out.json]"""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, ".")
sys.path.insert(0, "tests")
from abrsimulator_b200 import synth
from abrsimulator_b200.env import BatchedABREnv

n_iter = int(sys.argv[1]) if len(sys.argv) > 1 else 10
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
tid_run, off_run = synth.make_sessions(N, 1024, 2048)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, track_history=1)
WANT = ("delay", "sleep", "buffer", "rebuffer", "reward", "end_of_video", "request_time")


def summary(us, work):
    us = sorted(us)
    mean = sum(us) / len(us)
    return dict(launches=len(us), mean_us=round(mean, 1), median_us=round(us[len(us) // 2], 1),
                min_us=round(us[0], 1), max_us=round(us[-1], 1), downloads_per_second=round(work / (mean * 1e-6), 0))


def timed(fn):
    flush.fill_(1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e3


legs = []
for G in (1, 2, 4, 8, 16, 32):
    L = N // G
    tid = torch.from_numpy((np.arange(L) % 1024).astype(np.int32)).to(dev)
    off = torch.from_numpy(np.ascontiguousarray(off_run[:L])).to(dev)
    for pol in ("bba", "bola", "rate", "dynamic", "mixed"):
        pp = ["bola", "rate"] * (G // 2) if pol == "mixed" and G >= 2 else None
        if pol == "mixed" and G < 2:
            continue
        legs.append(((G, pol), lambda G=G, tid=tid, off=off, pol=pol, pp=pp: env.run_shared(
            "bba" if pp else pol, steps, tid, G, link_offset=off, player_policy=pp, want=WANT)))
tid_d, off_d = torch.from_numpy(tid_run).to(dev), torch.from_numpy(off_run).to(dev)
for pol in ("bba", "bola", "rate", "dynamic"):
    legs.append((("run", pol), lambda pol=pol: env.run(pol, steps, tid_d, off_d, want=WANT[:-1])))

times = {k: [] for k, _ in legs}
for it in range(n_iter + 2):
    for k, fn in legs:
        us = timed(fn)
        if it >= 2:
            times[k].append(us)

res = dict(card=name, power_limit_and_max_sm_clock=power, players=N, chunks=steps,
           l2="256 MB overwritten before every launch", shared={}, abr_env_run={})
for (a, pol), us in times.items():
    s = summary(us, N * steps)
    if a == "run":
        res["abr_env_run"][pol] = s
    else:
        res["shared"].setdefault(f"G={a}", {})[pol] = s

# the pure-Python oracle on one core: 16 links of 4 {bola, rate} players x 48 chunks
import shared_link_oracle as sl
w = sl.world_of_env(env, bw, tl, ti, sizes)
t0 = time.perf_counter()
sl.run_shared(w, steps, 4, list(range(16)), list(off_run[:16]), player_policy=[sl.BOLA, sl.RATE] * 2)
dt = time.perf_counter() - t0
res["python_oracle"] = dict(downloads=16 * 4 * steps, seconds=round(dt, 3),
                            us_per_download=round(dt / (16 * 4 * steps) * 1e6, 1))
print(json.dumps(res, indent=1))
if out_path:
    os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
