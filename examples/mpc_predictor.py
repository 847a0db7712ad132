#!/usr/bin/env python
"""Three MPCs on the same sessions: the built-in robust MPC, MPC over your own throughput predictor, and the
clairvoyant lookahead as the upper reference.

    python examples/mpc_predictor.py --sessions 65536 --steps 48 [--graph]

The predictor here is a torch EWMA over each session's throughput history (``env.throughput_history()``), discounted
by its own recent relative error, with one forecast per horizon step.  Any callable ``predictor(env) -> [N] or
[N, H]`` device tensor plugs in the same way, a torch model included: ``env.mpc_episode_pred`` calls it, then the
robust MPC search over its predictions (``abr_env_mpc_decide_pred``, SPEC §5.6), then the step.  ``--graph`` captures
one chunk (predictor, decision, step) in a CUDA graph and replays it for every chunk.  Prints the mean per-session
sum of rewards of each run.
"""
from __future__ import annotations

import argparse
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from abrsimulator_b200 import synth                      # noqa: E402
from abrsimulator_b200.env import BatchedABREnv           # noqa: E402


class EwmaPredictor:
    """Throughput forecast per horizon step from the history ring: an EWMA (weight `alpha` on the newer sample) of
    the samples, shrunk by the largest relative deviation of the last samples from it and by `decay` per step ahead.
    Device ops only: no host synchronisation, so it can be captured in a CUDA graph."""

    def __init__(self, env, horizon, alpha=0.4, decay=0.97, fallback=1.0):
        self.alpha, self.fallback = alpha, fallback
        self.steps = torch.tensor([decay ** i for i in range(horizon)], dtype=torch.float64, device=env.device)

    def __call__(self, env):
        x, n = env.throughput_history()              # [N, K] oldest first, NaN past n
        K = x.shape[1]
        valid = torch.arange(K, device=x.device)[None, :] < n[:, None]
        first = torch.where(n > 0, x[:, 0], torch.full_like(x[:, 0], self.fallback))
        s = first
        for j in range(1, K):
            s = torch.where(valid[:, j], self.alpha * x[:, j] + (1.0 - self.alpha) * s, s)
        dev = torch.where(valid, (x - s[:, None]).abs() / s[:, None], torch.zeros_like(x)).amax(dim=1)
        c = s / (1.0 + dev)
        return c[:, None] * self.steps[None, :]


def make_env(args, sessions):
    bitrates, sizes = synth.make_video(args.steps)
    bw, tl, ti = synth.make_traces(64, 256, seed=7)
    tid, off = synth.make_sessions(sessions, 64, 256, seed=11)
    env = BatchedABREnv(bw, sizes, bitrates, sessions, trace_len=tl, trace_interval=ti, track_history=1,
                        track_acc=1, hist_k=8)
    return env, tid, off


def run(args):
    env, tid, off = make_env(args, args.sessions)
    H = args.horizon
    results = {}

    env.reset(tid, off)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    env.mpc_episode(args.steps, H, mode="robust")
    torch.cuda.synchronize()
    results["robust MPC (built-in predictor)"] = (env.session_acc()[0].mean().item(), time.perf_counter() - t0)

    env.reset(tid, off)
    predictor = EwmaPredictor(env, H)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    if args.graph:
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):                   # first chunk eagerly: allocations and first launches
            env.mpc_episode_pred(1, predictor, H)
        torch.cuda.current_stream().wait_stream(s)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):                    # the second chunk is captured (and so runs on replay only)
            env.mpc_episode_pred(1, predictor, H)
        for _ in range(args.steps - 1):
            g.replay()
    else:
        env.mpc_episode_pred(args.steps, predictor, H)
    torch.cuda.synchronize()
    name = "MPC with a torch EWMA predictor" + (" (CUDA graph)" if args.graph else "")
    results[name] = (env.session_acc()[0].mean().item(), time.perf_counter() - t0)

    env.reset(tid, off)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    env.lookahead_episode(args.steps, H)
    torch.cuda.synchronize()
    results["clairvoyant lookahead (upper reference)"] = (env.session_acc()[0].mean().item(), time.perf_counter() - t0)
    assert env.error_count() == 0
    return results


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--sessions", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=48)
    ap.add_argument("--horizon", type=int, default=5)
    ap.add_argument("--graph", action="store_true", help="replay one captured chunk for the predictor's run")
    args = ap.parse_args()
    print(f"{args.sessions} sessions, {args.steps} chunks, horizon {args.horizon}, on {torch.cuda.get_device_name()}")
    for name, (reward, sec) in run(args).items():
        print(f"  {name:45s} mean per-session sum of rewards {reward:10.4f}   ({sec * 1e3:8.1f} ms)")


if __name__ == "__main__":
    main()
