"""What MPC over caller predictions (SPEC §5.6, ``mpc_decide_pred``) costs next to the robust MPC (``mpc_decide``).

Bench world: synth video (V = 48, A = 6), 1 024 x 2 048 synthetic traces, 64 consecutive sessions per trace, six BBA
chunks played so that every session has history and robust state.  ``mpc_decide_pred`` is fed the robust prediction c
of every session (the output ``preds`` of the standalone decision on a copy of the state, as an [N, H] float64
tensor), so both variants search the same tables.  Decisions of 131 072 sessions at H = 5, branch and bound and
exhaustive; 2 048 sessions at H = 7 (a block per session).  The two variants alternate launch by launch, a 256 MB
buffer (the L2 holds 126 MB) is overwritten in front of every timed launch, CUDA events around each, two untimed
launches of each first.  Then a 48-chunk episode of 16 384 sessions with the EWMA predictor of
examples/mpc_predictor.py, eager and replayed from a captured chunk, next to ``mpc_episode`` (robust).

usage: python profiles/time_mpc_pred.py [launches=30] [out.json]"""
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, ".")
from abrsimulator_b200 import _lib, synth
from abrsimulator_b200.env import BatchedABREnv
from abrsimulator_b200.mpc import decide_batch

sys.path.insert(0, os.path.join(".", "examples"))
from mpc_predictor import EwmaPredictor

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

V, A = 48, 6
bitrates, sizes = synth.make_video(V)
bw, tl, ti = synth.make_traces(1024, 2048)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)


def timed_pair(fa, fb, n, warm=2):
    """([us] of fa, [us] of fb): n launches of each, alternating, each behind an L2 overwrite."""
    pairs = ([], [])
    for it in range(n + warm):
        for k, fn in enumerate((fa, fb)):
            flush.fill_((2 * it + k) & 0xff)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            if it >= warm:
                pairs[k].append((e0, e1))
    torch.cuda.synchronize()
    return tuple(sorted(1e3 * a.elapsed_time(b) for a, b in p) for p in pairs)


def summary(us, decisions):
    mean = sum(us) / len(us)
    return dict(launches=len(us), mean_us=round(mean, 1), median_us=round(us[len(us) // 2], 1), min_us=round(us[0], 1),
                max_us=round(us[-1], 1), decisions_per_second=round(decisions / (mean * 1e-6), 0))


def played_env(N, **kw):
    tid, off = synth.make_sessions(N, 1024, 2048, group=64)
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, track_history=1, **kw)
    tid, off = torch.from_numpy(tid).to(dev), torch.from_numpy(off).to(dev)
    env.reset(tid, off)
    env.rollout("bba", 6, want=())
    return env, tid, off


def robust_c(env, H):
    """The robust prediction of every session, from the standalone decision on a copy of the state: [N, H]."""
    out = decide_batch(env.state("sizes"), env.state("utility"), env.state("chunk").clone(),
                       env.state("last_q").clone(), env.state("buffer").clone(), env.state("bw_hist").t().contiguous(),
                       env.state("hist_len").clone(), H, mode="robust", params=env.params,
                       last_pred=env.state("last_pred").clone(), err_ring=env.state("err_ring").t().contiguous(),
                       err_len=env.state("err_len").clone())
    return out["preds"][:, :1].expand(env.n, H).contiguous()


result = dict(gpu=name, power_limit_and_max_sm_clock=power,
              world=dict(V=V, A=A, traces="1024 x 2048 synthetic", state="6 BBA chunks after a reset",
                         L2="256 MB overwritten before every launch", order="the two variants alternate"),
              decide={})

for N, H, iters in ((131072, 5, n_iter), (2048, 7, max(4, n_iter // 3))):
    env, _, _ = played_env(N)
    pred = robust_c(env, H)
    act = torch.empty(N, dtype=torch.int32, device=dev)
    for exhaustive in (False, True):
        if H == 7 and exhaustive:
            continue
        rob, ext = timed_pair(lambda: env.mpc_decide(H, "robust", out=act, exhaustive=exhaustive),
                              lambda: env.mpc_decide_pred(pred, H, out=act, exhaustive=exhaustive), iters)
        key = f"N{N}_H{H}_{'exhaustive' if exhaustive else 'branch_and_bound'}"
        result["decide"][key] = dict(mpc_decide_robust=summary(rob, N), mpc_decide_pred=summary(ext, N))
        r = result["decide"][key]
        r["pred_over_robust_mean_time"] = round(r["mpc_decide_pred"]["mean_us"] / r["mpc_decide_robust"]["mean_us"], 3)
    assert env.error_count() == 0
    del env

# ---- 48-chunk episodes at 16 384 sessions ----
Ne, H = 16384, 5
env, tid, off = played_env(Ne, track_acc=1)
predictor = EwmaPredictor(env, H)


def robust_episode():
    env.reset(tid, off)
    env.mpc_episode(V, H, mode="robust")


def pred_episode():
    env.reset(tid, off)
    env.mpc_episode_pred(V, predictor, H)


env.reset(tid, off)
s = torch.cuda.Stream()
s.wait_stream(torch.cuda.current_stream())
with torch.cuda.stream(s):
    env.mpc_episode_pred(1, predictor, H)
torch.cuda.current_stream().wait_stream(s)
graph = torch.cuda.CUDAGraph()
with torch.cuda.graph(graph):
    env.mpc_episode_pred(1, predictor, H)


def graph_episode():
    env.reset(tid, off)
    for _ in range(V):
        graph.replay()


ep = {}
n_ep = max(3, n_iter // 6)
rob, eager = timed_pair(robust_episode, pred_episode, n_ep, warm=1)
_, replay = timed_pair(robust_episode, graph_episode, n_ep, warm=1)
for k, us in (("mpc_episode_robust", rob), ("mpc_episode_pred_ewma_eager", eager), ("mpc_episode_pred_ewma_graph", replay)):
    mean = sum(us) / len(us)
    ep[k] = dict(launches=len(us), mean_ms=round(mean * 1e-3, 3), min_ms=round(us[0] * 1e-3, 3),
                 max_ms=round(us[-1] * 1e-3, 3))
result["episode"] = dict(sessions=Ne, chunks=V, horizon=H, note="each includes the reset", **ep)
assert env.error_count() == 0

line = json.dumps(result, indent=1)
print(line)
if out_path:
    with open(out_path, "w") as f:
        f.write(line + "\n")
