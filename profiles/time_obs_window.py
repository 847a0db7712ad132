"""What the windowed observation (SPEC §4.5, ``step_policy_window``) costs next to the §4.1 step (``step_policy``).

Bench world: synth video (V = 48, A = 6), 1 024 x 2 048 synthetic traces, sessions sorted by trace (4 096 per trace),
W = 8.  Greedy steps (one launch each, no draw-counter bump) of 4 Mi sessions: ``step_policy`` writing its
[4 + A, N] observation, ``step_policy_window`` rolling its [3 + 2W + A, N] one, and the torch-glue path (``step_policy``
plus the same windowed observation built in eager PyTorch, as examples/pensieve_harness.py --torch-glue).  The
variants alternate launch by launch, a 256 MB buffer (the L2 holds 126 MB) is overwritten in front of every timed
launch, CUDA events around each, two untimed launches of each first.  Then graph-replayed 48-chunk episodes of
examples/pensieve_harness.py at 524 288 sessions, fused and torch-glue, alternating.

usage: python profiles/time_obs_window.py [launches=30] [out.json]"""
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, ".")
from abrsimulator_b200 import synth
from abrsimulator_b200.env import BatchedABREnv

sys.path.insert(0, os.path.join(".", "examples"))
import pensieve_harness as ph

n_iter = int(sys.argv[1]) if len(sys.argv) > 1 else 30
out_path = sys.argv[2] if len(sys.argv) > 2 else None
assert torch.cuda.is_available(), "this measurement needs the GPU"
dev = torch.device("cuda", 0)
name = torch.cuda.get_device_name(0)
try:
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError):
    power = "unknown"

V, A, W, N = 48, 6, 8, 4 << 20
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)


def obs_bytes(kind):
    """Observation bytes per session-step (written, read): §4.1 writes 4 (4 + A); §4.5 writes 4 (3 + 2W + A) and reads
    the 2 (W - 1) window entries it moves up.  The rest of the step (state, tables, logits) is the same for both."""
    if kind == "step_policy":
        return 4 * (4 + A), 0
    return 4 * (3 + 2 * W + A), 4 * 2 * (W - 1)


def timed(fns, n, warm=2):
    """[us] per function: n launches of each, alternating, each behind an L2 overwrite."""
    ev = [[] for _ in fns]
    for it in range(n + warm):
        for k, fn in enumerate(fns):
            flush.fill_((len(fns) * it + k) & 0xff)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            if it >= warm:
                ev[k].append((e0, e1))
    torch.cuda.synchronize()
    return [sorted(1e3 * a.elapsed_time(b) for a, b in p) for p in ev]


def summary(ts):
    return dict(median_us=round(ts[len(ts) // 2], 2), min_us=round(ts[0], 2), max_us=round(ts[-1], 2))


bitrates, sizes = synth.make_video(V)
bw, tl, ti = synth.make_traces(1024, 2048)
tid, off = synth.make_sessions(N, 1024, 2048, group=N // 1024)
envs = {}
for k in ("step_policy", "step_policy_window", "torch_glue"):
    envs[k] = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti)
    envs[k].reset(tid, off)
logits = torch.randn(N, A, device=dev)
obs41 = torch.zeros(4 + A, N, dtype=torch.float32, device=dev)
obs_w = envs["step_policy_window"].observe_window(W, ph.SCALES)
glue = ph.Buffers(envs["torch_glue"], W)
glue_actor = lambda obs: logits        # the glue path's own kernels, without an actor


def run_41():
    envs["step_policy"].step_policy(logits, sample=False, obs=obs41, obs_scales=ph.SCALES[1:])


def run_45():
    envs["step_policy_window"].step_policy_window(logits, obs_w, sample=False, scales=ph.SCALES)


def run_glue():
    ph.one_chunk(envs["torch_glue"], glue_actor, glue, sample=False, fused=False)


with torch.no_grad():
    t41, t45, tglue = timed([run_41, run_45, run_glue], n_iter)
assert torch.equal(obs_w, glue.obs), "the torch-glue observation differs from the kernel's"
steps = {}
for kind, ts in (("step_policy", t41), ("step_policy_window", t45), ("torch_glue", tglue)):
    w_b, r_b = obs_bytes("step_policy" if kind == "step_policy" else "window")
    steps[kind] = dict(summary(ts), ns_per_session_step=round(1e3 * ts[len(ts) // 2] / N, 4),
                       obs_bytes_written=w_b, obs_bytes_read=r_b)
steps["window_minus_step_policy_us"] = round(t45[len(t45) // 2] - t41[len(t41) // 2], 2)

# graph-replayed 48-chunk episodes of the example, fused and torch-glue, alternating
NE, CH = 524288, 48
world, (etid, eoff) = ph.make_world(NE, CH)
torch.manual_seed(0)
episode = {}
runners = {}
for kind in ("fused", "torch_glue"):
    env = ph.make_env(world, NE)
    env.reset(etid, eoff)
    actor = ph.Actor(W, env.A).to(dev)
    runners[kind] = (env, ph.GraphedEpisode(env, actor, W, fused=kind == "fused"))
    runners[kind][1].run(1)
ep_ts = {k: [] for k in runners}
for it in range(6):
    for kind, (env, r) in runners.items():
        env.reset(etid, eoff)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r.run(CH)
        e1.record()
        torch.cuda.synchronize()
        if it >= 1:
            ep_ts[kind].append(e0.elapsed_time(e1))
for kind, ts in ep_ts.items():
    ts.sort()
    episode[kind] = dict(median_ms=round(ts[len(ts) // 2], 3), min_ms=round(ts[0], 3), max_ms=round(ts[-1], 3))

result = dict(device=name, power_limit_and_max_sm_clock=power, sessions=N, A=A, W=W, launches=n_iter,
              l2="256 MB overwritten before every timed launch", step=steps,
              episode_48_chunks=dict(sessions=NE, window=W, graph_replayed=True, **episode))
line = json.dumps(result, indent=1)
print(line)
if out_path:
    os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
    with open(out_path, "w") as f:
        f.write(line + "\n")
