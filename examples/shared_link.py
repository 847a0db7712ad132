#!/usr/bin/env python
"""Players competing for one bottleneck (SPEC §9): fairness, efficiency and stability of the built-in policies.

    python examples/shared_link.py [--links 4096] [--steps 48] [--check]

Two scenarios, each one launch over ``--links`` links of a ``synth.make_traces`` world:

* four players per link, two BOLA and two rate-based, all starting at 0 s;
* two BOLA players per link, the second joining at 60 s, when the first has filled its buffer.

For each scenario the example prints, per policy slot, the mean utility per chunk, the rebuffering per player and the
bitrate switches per player; Jain's index of the players' mean utilities per link (mean over links); and the link
efficiency, the data delivered over the capacity the trace offered while the link was in use.  ``--check`` runs the
first eight links of each scenario through the pure-Python oracle of tests/shared_link_oracle.py and requires every
output to be bit-identical.
"""
from __future__ import annotations

import argparse
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from abrsimulator_b200 import synth                      # noqa: E402
from abrsimulator_b200.env import BatchedABREnv, jain_index   # noqa: E402

SCENARIOS = {
    "4 players: BOLA, BOLA, RATE, RATE": dict(player_policy=["bola", "bola", "rate", "rate"], join=[0.0] * 4),
    "2 BOLA players, the second joining at 60 s": dict(player_policy=["bola", "bola"], join=[0.0, 60.0]),
}


def run(env, sc, links, steps, n_traces, T):
    G = len(sc["player_policy"])
    tid = (np.arange(links) % n_traces).astype(np.int32)
    off = (np.arange(links) * 7.3) % T
    join = np.tile(np.asarray(sc["join"]), links)
    want = ("delay", "sleep", "buffer", "rebuffer", "reward", "end_of_video", "actions", "request_time")
    out, link, cost, stats = env.run_shared("bba", steps, tid, G, link_offset=off, join_delay=join,
                                            player_policy=sc["player_policy"], want=want)
    return tid, off, join, out, link


def report(name, env, sc, out, link, links, steps):
    G = len(sc["player_policy"])
    acc = env.session_acc().cpu().numpy().reshape(-1, links, G)   # [acc][link][slot]
    util = acc[2] / acc[6]                                          # mean utility per chunk
    act = out["actions"].cpu().numpy().reshape(steps, links, G)
    switches = (np.diff(act, axis=0) != 0).sum(0)                   # [link][slot]
    print(f"\n{name}  ({links} links x {G} players x {steps} chunks)")
    for p, pol in enumerate(sc["player_policy"]):
        print(f"  slot {p} {pol:>5}: utility {util[:, p].mean():6.3f} /chunk   rebuffer {acc[1][:, p].mean():7.2f} s"
              f"   switches {switches[:, p].mean():5.2f}")
    jain = jain_index(torch.from_numpy(util))
    eff = (link["delivered"] / link["capacity"]).cpu().numpy()
    print(f"  Jain's index of the mean utilities: {jain.mean().item():.4f}   link efficiency: {eff.mean():.4f}")


def check(env, sc, tid, off, join, out, link, steps, world, n_check=8):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import shared_link_oracle as sl
    G = len(sc["player_policy"])
    ids = {"bola": sl.BOLA, "rate": sl.RATE}
    ref = sl.run_shared(world, steps, G, tid[:n_check], off[:n_check], join[:n_check * G],
                        player_policy=[ids[p] for p in sc["player_policy"]])
    n = n_check * G
    ok = True
    for k_gpu, k_ref in (("delay", "delay"), ("sleep", "sleep"), ("buffer", "buffer"), ("rebuffer", "rebuf"),
                         ("reward", "reward"), ("request_time", "request_time"), ("actions", "actions"),
                         ("end_of_video", "eov")):
        ok &= bool(np.array_equal(out[k_gpu][:, :n].cpu().numpy(), ref[k_ref]))
    for k in ("time", "capacity", "delivered"):
        ok &= bool(np.array_equal(link[k][:n_check].cpu().numpy(), ref["link_" + k]))
    ok &= bool(np.array_equal(env.session_acc()[:, :n].cpu().numpy(), ref["acc"]))
    return ok


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--links", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=48)
    ap.add_argument("--traces", type=int, default=256)
    ap.add_argument("--check", action="store_true")
    a = ap.parse_args()
    T = 2048
    bitrates, sizes = synth.make_video(48)
    bw, tl, ti = synth.make_traces(a.traces, T)
    env = BatchedABREnv(bw, sizes, bitrates, a.links * 4, trace_len=tl, trace_interval=ti, track_history=1)
    ok = True
    for name, sc in SCENARIOS.items():
        tid, off, join, out, link = run(env, sc, a.links, a.steps, a.traces, T)
        report(name, env, sc, out, link, a.links, a.steps)
        if a.check:
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import shared_link_oracle as sl
            world = sl.world_of_env(env, bw, tl, ti, sizes)
            ok &= check(env, sc, tid, off, join, out, link, a.steps, world)
    if a.check:
        print("check:", "ok (bit-identical to the oracle)" if ok else "FAILED")
        sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
