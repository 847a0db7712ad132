#!/usr/bin/env python
"""Pensieve-style RL harness: an actor with Pensieve's shape (Mao et al., SIGCOMM 2017) fed by the windowed
observation of the step kernel (`env.step_policy_window`, SPEC §4.5).

    python examples/pensieve_harness.py --sessions 524288 --chunks 48
    python examples/pensieve_harness.py --torch-glue          # the same observation rolled in PyTorch
    python examples/pensieve_harness.py --check --sessions 4099   # both paths, bit for bit

The observation is feature-major [3 + 2W + A, N]: the last chunk's utility, the buffer, the chunks left, the last W
throughputs, the last W download times and the next chunk's sizes.  The step kernel draws the action from the actor's
logits, steps the session, adds up the reward and rolls both windows in the caller's buffer (zeroed at an end of
video), so one library launch per chunk serves the whole state.  `--torch-glue` runs `env.step_policy` (SPEC §4.1)
and builds the same observation around it in eager PyTorch.  No host round trip happens inside the episode loop.
"""
from __future__ import annotations

import argparse
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from abrsimulator_b200 import synth                      # noqa: E402
from abrsimulator_b200.env import BatchedABREnv, StepResult   # noqa: E402

# (utility, buffer, throughput, delay, size): utility in Mbit/s, buffer / 10 s, throughput in Mbit/s, delay / 10 s,
# sizes in Mbit
SCALES = (1.0, 0.1, 1.0, 0.1, 1.0)
SEED = 0x5EED


class Actor(torch.nn.Module):
    """Pensieve's actor: one 1-D convolution over each window and over the next sizes, a linear layer over each of
    rows 0-2, one hidden layer over the concatenation and the logits."""

    def __init__(self, W, A, width=128, kernel=4):
        super().__init__()
        self.W, self.A = W, A
        k_w, k_a = min(kernel, W), min(kernel, A)
        self.scalars = torch.nn.ModuleList(torch.nn.Linear(1, width) for _ in range(3))
        self.conv_thr = torch.nn.Conv1d(1, width, k_w)
        self.conv_delay = torch.nn.Conv1d(1, width, k_w)
        self.conv_size = torch.nn.Conv1d(1, width, k_a)
        n_in = 3 * width + 2 * width * (W - k_w + 1) + width * (A - k_a + 1)
        self.hidden = torch.nn.Linear(n_in, width)
        self.out = torch.nn.Linear(width, A)

    def forward(self, obs):                     # obs [F, N] feature-major
        x = obs.t()
        W = self.W
        parts = [torch.relu(lin(x[:, j:j + 1])) for j, lin in enumerate(self.scalars)]
        for conv, rows in ((self.conv_thr, x[:, 3:3 + W]), (self.conv_delay, x[:, 3 + W:3 + 2 * W]),
                           (self.conv_size, x[:, 3 + 2 * W:])):
            parts.append(torch.relu(conv(rows.unsqueeze(1))).flatten(1))
        return self.out(torch.relu(self.hidden(torch.cat(parts, 1))))


class Buffers:
    """The in-place buffers of one episode loop (persistent, so that a chunk can be captured in a CUDA graph)."""

    def __init__(self, env, W):
        n, A, dev = env.n, env.A, env.device
        self.W = W
        self.obs = env.observe_window(W, SCALES)
        self.total = torch.zeros(n, dtype=torch.float64, device=dev)
        self.action = torch.zeros(n, dtype=torch.int32, device=dev)
        self.obs41 = torch.zeros(4 + A, n, dtype=torch.float32, device=dev)     # torch-glue only
        self.out = StepResult(*[torch.empty(n, dtype=torch.float64, device=dev) for _ in range(5)], None,
                              torch.empty(n, dtype=torch.uint8, device=dev), None)

    def restart(self, env):
        env.observe_window(self.W, SCALES, obs=self.obs)
        self.total.zero_()


def one_chunk(env, actor, b, sample=True, fused=True):
    """actor(obs) -> step -> next observation, on the device and in place."""
    logits = actor(b.obs)
    if fused:
        env.step_policy_window(logits, b.obs, sample=sample, seed=SEED, scales=SCALES, action_out=b.action,
                               reward_sum=b.total)
        return
    # SPEC §4.1 step, then the windowed observation rebuilt in PyTorch (the same fp64 products, rounded once)
    env.step_policy(logits, sample=sample, seed=SEED, obs=b.obs41, action_out=b.action, reward_sum=b.total, out=b.out,
                    obs_scales=SCALES[1:])
    W, V, obs = b.W, env.V, b.obs
    chunk, last_q = env.state("chunk").long(), env.state("last_q").long()
    util = env.state("utility")[(chunk - 1).clamp(min=0), last_q.clamp(min=0)]
    obs[0] = torch.where(last_q < 0, 0.0, util * SCALES[0]).float()
    obs[1] = (env.state("buffer") * SCALES[1]).float()
    obs[2] = ((V - chunk).double() / V).float()
    keep = (b.out.end_of_video == 0).float()          # an end of video (auto_reset) restarts the windows
    for lo, new in ((3, b.obs41[1]), (3 + W, b.obs41[2])):
        win = obs[lo:lo + W]
        win.copy_(torch.cat([win[1:], new[None]]) * keep)
    obs[3 + 2 * W:] = b.obs41[4:]


class GraphedEpisode:
    """One chunk captured into a CUDA graph once; an episode is `chunks` replays (call after ``env.reset``)."""

    def __init__(self, env, actor, W, sample=True, fused=True):
        self.env, self.actor, self.sample, self.fused = env, actor, sample, fused
        self.b = Buffers(env, W)
        self.graph = None

    def _capture(self):
        env = self.env
        snap = {f: env.state(f).clone() for f in ("seg", "chunk", "last_q", "phase", "pos", "buffer")}
        side = torch.cuda.Stream(device=env.device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):              # warm-up: allocator, cuDNN / cuBLAS plans
            one_chunk(env, self.actor, self.b, self.sample, self.fused)
        torch.cuda.current_stream().wait_stream(side)
        for f, t in snap.items():
            env.state(f).copy_(t)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            one_chunk(env, self.actor, self.b, self.sample, self.fused)

    def run(self, chunks):
        with torch.no_grad():
            if self.graph is None:
                self._capture()
            self.b.restart(self.env)
            for _ in range(chunks):
                self.graph.replay()
        return self.b.total


def make_world(sessions, chunks, seed=0):
    bitrates, sizes = synth.make_video(chunks, seed=seed)
    bw, tl, ti = synth.make_traces(1024, 2048)
    tid, off = synth.make_sessions(sessions, 1024, 2048, group=max(256, sessions // 1024))
    return (bw, sizes, bitrates, tl, ti), (tid, off)


def make_env(world, sessions):
    bw, sizes, bitrates, tl, ti = world
    return BatchedABREnv(bw, sizes, bitrates, sessions, trace_len=tl, trace_interval=ti)


def check(args, dev):
    """Both paths on twin environments with the same draws: observation, actions and rewards bit for bit."""
    world, (tid, off) = make_world(args.sessions, args.chunks)
    envs = [make_env(world, args.sessions) for _ in range(2)]
    actor = Actor(args.window, envs[0].A).to(dev)
    bufs = []
    for e in envs:
        e.reset(tid, off)
        bufs.append(Buffers(e, args.window))
    with torch.no_grad():
        for t in range(args.chunks + 5):          # crosses an end of video
            for e, b, fused in zip(envs, bufs, (True, False)):
                one_chunk(e, actor, b, fused=fused)
            for name in ("obs", "action", "total"):
                if not torch.equal(getattr(bufs[0], name), getattr(bufs[1], name)):
                    raise SystemExit(f"chunk {t}: {name} differs between the fused and the torch-glue path")
    print(f"fused == torch-glue: {args.sessions} sessions x {args.chunks + 5} chunks, window {args.window}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sessions", type=int, default=524288)
    ap.add_argument("--chunks", type=int, default=48)
    ap.add_argument("--window", type=int, default=8)
    ap.add_argument("--episodes", type=int, default=3)
    ap.add_argument("--torch-glue", action="store_true", help="step_policy + the windows rolled in PyTorch")
    ap.add_argument("--check", action="store_true", help="compare the two paths bit for bit")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    if args.check:
        return check(args, dev)
    world, (tid, off) = make_world(args.sessions, args.chunks)
    env = make_env(world, args.sessions)
    env.reset(tid, off)
    actor = Actor(args.window, env.A).to(dev)
    runner = GraphedEpisode(env, actor, args.window, fused=not args.torch_glue)
    for ep in range(args.episodes):
        env.reset(tid, off)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        total = runner.run(args.chunks)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        print(f"episode {ep}: {args.sessions} sessions x {args.chunks} chunks in {dt * 1e3:.1f} ms "
              f"({'torch-glue' if args.torch_glue else 'fused'}), mean episode reward {total.mean().item():.3f}")


if __name__ == "__main__":
    main()
