#!/usr/bin/env python
"""Four MPCs on the same sessions: the built-in robust MPC, scenario MPC over an empirical throughput distribution
with the mean and with the worst-case objective, and the clairvoyant lookahead as the upper reference.

    python examples/mpc_scenarios.py --sessions 65536 --steps 48 [--graph] [--check]

The scenarios come from each session's throughput history (``env.throughput_history()``): each of the last K samples
is one flat future, weighted 1/n over the n samples the session has.  Missing samples repeat the newest one with
weight 0 (a valid throughput that changes neither the mean nor the minimum), and a session without history gets one
fallback scenario.  ``env.mpc_episode_scen`` calls the sampler, then the scenario search (``abr_env_mpc_decide_scen``,
SPEC §5.7), then the step.  ``--graph`` captures one chunk (sampler, decision, step) in a CUDA graph and replays it
for every chunk; ``--check`` runs both scenario MPCs eagerly and from a graph and requires identical per-session sums.
Prints the mean per-session sum of rewards of each run.
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


class EmpiricalSampler:
    """The last K throughput samples as K flat scenarios with weights 1/n.  Device ops only: no host
    synchronisation, so it can be captured in a CUDA graph."""

    def __init__(self, fallback=1.0):
        self.fallback = fallback

    def __call__(self, env):
        x, n = env.throughput_history()                   # [N, K] oldest first, NaN past n
        have = ~torch.isnan(x)
        newest = x.gather(1, (n.long() - 1).clamp(min=0)[:, None])
        newest = torch.where(n[:, None] > 0, newest, torch.full_like(newest, self.fallback))
        scen = torch.where(have, x, newest)
        w = have.to(torch.float64) / n.clamp(min=1).to(torch.float64)[:, None]
        w[:, 0] = torch.where(n > 0, w[:, 0], torch.ones_like(w[:, 0]))   # no history: the fallback, weight 1
        return scen, w


def make_env(args, sessions):
    bitrates, sizes = synth.make_video(args.steps)
    bw, tl, ti = synth.make_traces(64, 256, seed=7)
    tid, off = synth.make_sessions(sessions, 64, 256, seed=11)
    env = BatchedABREnv(bw, sizes, bitrates, sessions, trace_len=tl, trace_interval=ti, track_history=1,
                        track_acc=1, hist_k=args.scenarios)
    return env, tid, off


def scenario_episode(env, args, objective, graph):
    H, sampler = args.horizon, EmpiricalSampler()
    smp = sampler if objective == "mean" else (lambda e: sampler(e)[0])   # worst case: no weights
    if graph:
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):                        # first chunk eagerly: allocations and first launches
            env.mpc_episode_scen(1, smp, H, objective=objective)
        torch.cuda.current_stream().wait_stream(s)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):                         # the second chunk is captured (and so runs on replay only)
            env.mpc_episode_scen(1, smp, H, objective=objective)
        for _ in range(args.steps - 1):
            g.replay()
    else:
        env.mpc_episode_scen(args.steps, smp, H, objective=objective)


def run(args):
    env, tid, off = make_env(args, args.sessions)
    H = args.horizon
    results, sums = {}, {}

    def timed(name, fn):
        env.reset(tid, off)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        sums[name] = env.session_acc()[0].clone()
        results[name] = (sums[name].mean().item(), time.perf_counter() - t0)

    timed("robust MPC (built-in predictor)", lambda: env.mpc_episode(args.steps, H, mode="robust"))
    for objective in ("mean", "worst"):
        graphs = (False, True) if args.check else (args.graph,)
        for graph in graphs:
            name = f"scenario MPC, {objective} over {args.scenarios} samples" + (" (CUDA graph)" if graph else "")
            timed(name, lambda: scenario_episode(env, args, objective, graph))
        if args.check:
            a, b = (sums[n] for n in list(sums)[-2:])
            assert torch.equal(a.view(torch.int64), b.view(torch.int64)), f"{objective}: graph replay differs"
            print(f"  {objective}: graph replay matches the eager run bit for bit")
    timed("clairvoyant lookahead (upper reference)", lambda: env.lookahead_episode(args.steps, H))
    assert env.error_count() == 0
    return results


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--sessions", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=48)
    ap.add_argument("--horizon", type=int, default=5)
    ap.add_argument("--scenarios", type=int, default=8, help="history samples kept, one scenario each (<= 16)")
    ap.add_argument("--graph", action="store_true", help="replay one captured chunk for the scenario runs")
    ap.add_argument("--check", action="store_true", help="run the scenario MPCs eagerly and from a graph, compare")
    args = ap.parse_args()
    print(f"{args.sessions} sessions, {args.steps} chunks, horizon {args.horizon}, on {torch.cuda.get_device_name()}")
    for name, (reward, sec) in run(args).items():
        print(f"  {name:55s} mean per-session sum of rewards {reward:10.4f}   ({sec * 1e3:8.1f} ms)")


if __name__ == "__main__":
    main()
