"""What the clairvoyant lookahead (SPEC §4.4, ``lookahead_decide``) costs, next to the fused BBA episode.

Bench world: synth video (V = 48, A = 6), 1 024 x 2 048 synthetic traces, sessions fresh from a reset (chunk 0, so every
decision plans the full horizon).  Decisions of 65 536 sessions for H = 3, 4, 5, with the sessions sorted by trace
(64 consecutive sessions per trace) and interleaved (one trace per session, in session order); H = 7 for 2 048
sorted sessions; one 48-chunk ``lookahead_episode`` (H = 5) of 16 384 sorted sessions; the fused ``bba`` episode of
65 536 sorted sessions x 48 chunks.  A 256 MB buffer (the L2 holds 126 MB) is overwritten in front of every timed
launch; CUDA events around each; two untimed launches of every shape first.  Lookahead steps/s counts every node of
the search tree: decisions x sum_{d=1..H} A^d / time.

usage: python profiles/time_lookahead.py [launches=20] [out.json]"""
import json
import subprocess
import sys

import torch

sys.path.insert(0, ".")
from abrsimulator_b200 import synth
from abrsimulator_b200.env import BatchedABREnv

n_iter = int(sys.argv[1]) if len(sys.argv) > 1 else 20
out_path = sys.argv[2] if len(sys.argv) > 2 else None
assert torch.cuda.is_available(), "this measurement needs the GPU"
dev = torch.device("cuda", 0)
name = torch.cuda.get_device_name(0)
try:
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError):
    power = "unknown"

V, A = 48, 6
bitrates, sizes = synth.make_video(V)
bw, tl, ti = synth.make_traces(1024, 2048)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)


def nodes(H):
    return sum(A ** d for d in range(1, H + 1))


def timed(fn, n, warm=2):
    """[us] of n launches of fn, each behind an L2 overwrite."""
    pairs = []
    for it in range(n + warm):
        flush.fill_(it & 0xff)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        if it >= warm:
            pairs.append((e0, e1))
    torch.cuda.synchronize()
    return sorted(1e3 * a.elapsed_time(b) for a, b in pairs)


def summary(us, decisions, H):
    mean = sum(us) / len(us)
    return dict(launches=len(us), mean_us=round(mean, 1), median_us=round(us[len(us) // 2], 1), min_us=round(us[0], 1),
                max_us=round(us[-1], 1), decisions_per_second=round(decisions / (mean * 1e-6), 0),
                lookahead_steps_per_second=round(decisions * nodes(H) / (mean * 1e-6), 0))


def make_env(N, group, **kw):
    tid, off = synth.make_sessions(N, 1024, 2048, group=group)
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, **kw)
    return env, torch.from_numpy(tid).to(dev), torch.from_numpy(off).to(dev)


result = dict(gpu=name, power_limit_and_max_sm_clock=power,
              world=dict(V=V, A=A, traces="1024 x 2048 synthetic", state="fresh from a reset (chunk 0)",
                         L2="256 MB overwritten before every launch"),
              decide={})

# ---- decisions at 65 536 sessions ----
N = 65536
for layout, group in (("sorted", 64), ("interleaved", 1)):
    env, tid, off = make_env(N, group)
    env.reset(tid, off)
    act = torch.empty(N, dtype=torch.int32, device=dev)
    for H in (3, 4, 5):
        us = timed(lambda: env.lookahead_decide(H, out=act), n_iter)
        result["decide"][f"{layout}_N{N}_H{H}"] = summary(us, N, H)
    assert env.error_count() == 0
    del env

# ---- H = 7 at 2 048 sessions ----
env, tid, off = make_env(2048, 64)
env.reset(tid, off)
act = torch.empty(2048, dtype=torch.int32, device=dev)
us = timed(lambda: env.lookahead_decide(7, out=act), max(3, n_iter // 4))
result["decide"]["sorted_N2048_H7"] = summary(us, 2048, 7)
del env

# ---- a 48-chunk lookahead episode at 16 384 sessions ----
Ne = 16384
env, tid, off = make_env(Ne, 64, track_acc=1)


def episode():
    env.reset(tid, off)
    env.lookahead_episode(V, 5)


us = timed(episode, max(3, n_iter // 4), warm=1)
mean = sum(us) / len(us)
result["episode"] = dict(sessions=Ne, chunks=V, horizon=5, launches=len(us), mean_ms=round(mean * 1e-3, 2),
                         min_ms=round(us[0] * 1e-3, 2), max_ms=round(us[-1] * 1e-3, 2),
                         chunk_steps_per_second=round(Ne * V / (mean * 1e-6), 0))
assert env.error_count() == 0
del env

# ---- the fused BBA episode, same run ----
env, tid, off = make_env(N, 64)


def bba():
    env.rollout("bba", V, seed=7, want=())


def bba_timed(n):
    pairs = []
    for it in range(n + 2):
        env.reset(tid, off)
        flush.fill_(it & 0xff)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        bba()
        e1.record()
        if it >= 2:
            pairs.append((e0, e1))
    torch.cuda.synchronize()
    return sorted(1e3 * a.elapsed_time(b) for a, b in pairs)


us = bba_timed(max(50, n_iter))
mean = sum(us) / len(us)
result["bba_episode"] = dict(sessions=N, chunks=V, outputs="none", launches=len(us), mean_us=round(mean, 2),
                             median_us=round(us[len(us) // 2], 2),
                             chunk_steps_per_second=round(N * V / (mean * 1e-6), 0))
best = max(v["lookahead_steps_per_second"] for v in result["decide"].values())
result["lookahead_steps_over_bba_chunk_steps"] = round(best / result["bba_episode"]["chunk_steps_per_second"], 3)

line = json.dumps(result, indent=1)
print(line)
if out_path:
    with open(out_path, "w") as f:
        f.write(line + "\n")
