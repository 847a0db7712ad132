#!/usr/bin/env python
"""An Oboe-style parameter sweep of the built-in policies in one fused launch per policy (SPEC §4.7).

    python examples/policy_sweep.py [--traces 256] [--copies 4] [--steps 48] [--check]

Every grid point (BOLA's (min, target) buffer range, BBA's (reservoir, cushion), the rate rule's safety factor) is
crossed with every trace of a ``synth.make_traces`` world, and each (point, trace) pair is one session with its own
parameters.  The generator draws one mean throughput level per trace, so the traces are binned by their mean into
network classes.  For each policy the example prints the mean QoE (per-session sum of rewards) of the default
configuration, of the best configuration over all traces and of the best configuration per class (Oboe's per-network
-state tuning).  ``--check`` runs four grid points as separate environment-wide environments and requires the sweep's
per-session outputs to equal them bit for bit.
"""
from __future__ import annotations

import argparse
import itertools
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from abrsimulator_b200 import synth                      # noqa: E402
from abrsimulator_b200.env import BatchedABREnv           # noqa: E402

DEFAULTS = dict(bba_reservoir=5.0, bba_cushion=10.0, rb_safety=1.0, bola_min_buffer=10.0, bola_target_buffer=30.0)
GRIDS = {
    "bba": [dict(bba_reservoir=r, bba_cushion=c) for r, c in itertools.product((2.0, 5.0, 8.0, 12.0), (5.0, 10.0, 20.0, 30.0))],
    "rate": [dict(rb_safety=s) for s in (0.5, 0.6, 0.7, 0.8, 0.9, 1.0, 1.1, 1.2)],
    "bola": [dict(bola_min_buffer=m, bola_target_buffer=t) for m, t in itertools.product((4.0, 8.0, 12.0, 16.0),
                                                                                          (20.0, 30.0, 45.0, 60.0))],
}
CLASSES = 4


def sweep(policy, grid, bw, tl, ti, sizes, bitrates, steps, copies):
    """The [points][traces * copies] per-session reward sums of one launch; session (g, t, c) has point g's values."""
    n_tr = bw.shape[0]
    per = n_tr * copies
    N = len(grid) * per
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti,
                        track_history=1 if policy == "rate" else 0)
    tid = np.tile(np.repeat(np.arange(n_tr, dtype=np.int32), copies), len(grid))
    off = np.tile(np.arange(per) % copies * 37.0, len(grid))
    env.reset(tid, off)
    fields = {f: np.repeat([p.get(f, DEFAULTS[f]) for p in grid], per) for f in grid[0]}
    env.set_session_policy_params(**fields)
    out = env.rollout(policy, steps)
    return env, out, env.session_acc()[0].view(len(grid), per).cpu().numpy(), tid, off


def environment_wide(policy, point, bw, tl, ti, sizes, bitrates, steps, tid, off):
    kw = dict(track_history=1 if policy == "rate" else 0)
    if "bba_reservoir" in point:
        kw.update(bba_reservoir=point["bba_reservoir"], bba_cushion=point["bba_cushion"])
    env = BatchedABREnv(bw, sizes, bitrates, len(tid), trace_len=tl, trace_interval=ti, **kw)
    pp = {f: v for f, v in point.items() if not f.startswith("bba")}
    if pp:
        env.set_policy_params(**pp)
    env.reset(tid, off)
    return env.rollout(policy, steps)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--traces", type=int, default=256)
    ap.add_argument("--copies", type=int, default=4)
    ap.add_argument("--steps", type=int, default=48)
    ap.add_argument("--check", action="store_true")
    a = ap.parse_args()
    bw, tl, ti = synth.make_traces(a.traces, 600, seed=11)
    bitrates, sizes = synth.make_video(48, seed=3)
    level = bw.mean(axis=1)
    cls = np.searchsorted(np.quantile(level, np.linspace(0, 1, CLASSES + 1)[1:-1]), level)   # class of each trace
    ok = True
    for policy, grid in GRIDS.items():
        env, out, qoe, tid, off = sweep(policy, grid, bw, tl, ti, sizes, bitrates, a.steps, a.copies)
        per_trace = qoe.reshape(len(grid), a.traces, a.copies).mean(axis=2)       # [points][traces]
        default = next(g for g, p in enumerate(grid) if all(p[f] == DEFAULTS[f] for f in p)) \
            if any(all(p[f] == DEFAULTS[f] for f in p) for p in grid) else None
        best = int(per_trace.mean(axis=1).argmax())
        per_class = [int(per_trace[:, cls == c].mean(axis=1).argmax()) for c in range(CLASSES)]
        oboe = np.mean([per_trace[per_class[c], cls == c].mean() * (cls == c).mean() for c in range(CLASSES)]) * CLASSES
        line = f"{policy:5s} {len(grid) * a.traces * a.copies} sessions, one launch:"
        if default is not None:
            line += f" default {per_trace[default].mean():8.3f}"
        line += f"  best global {per_trace[best].mean():8.3f} {grid[best]}  best per class {oboe:8.3f}"
        print(line)
        if a.check:
            per = a.traces * a.copies
            for g in sorted({0, len(grid) // 3, 2 * len(grid) // 3, len(grid) - 1}):
                sl = slice(g * per, (g + 1) * per)
                exp = environment_wide(policy, grid[g], bw, tl, ti, sizes, bitrates, a.steps, tid[sl], off[sl])
                for k, v in exp.items():
                    if not torch.equal(out[k][:, sl], v):
                        print(f"MISMATCH {policy} point {g} {k}")
                        ok = False
    if a.check:
        print("check:", "bit-identical to the environment-wide runs" if ok else "FAILED")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
