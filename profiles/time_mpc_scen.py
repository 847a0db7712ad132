"""What MPC over throughput scenarios (SPEC §5.7, ``mpc_decide_scen``) costs next to MPC over one prediction row
(SPEC §5.6, ``mpc_decide_pred``).

Bench world: synth video (V = 48, A = 6), 1 024 x 2 048 synthetic traces, 64 consecutive sessions per trace, six BBA
chunks played.  Scenario k of session s is the session's robust prediction c times a factor drawn log-uniformly from
[0.5, 2] per (s, k, step), seeded; ``mpc_decide_pred`` gets scenario 0.  Decisions of 131 072 sessions at H = 5 for
K in {1, 4, 8, 16}, both objectives, branch and bound and exhaustive, each alternating launch by launch with
``mpc_decide_pred`` in the same search mode; 2 048 sessions at H = 7 (a block per session).  A 256 MB buffer (the L2
holds 126 MB) is overwritten in front of every timed launch, CUDA events around each, two untimed launches of each
first.  The FP64 roofline of the exhaustive runs counts the operations the search executes from the shapes
(``fp64_ops``) against ``abr_fp64_probe`` (DADD chains) in the same run.  Then a 48-chunk episode of 16 384 sessions
with the sampler of examples/mpc_scenarios.py (K = 8, mean), eager and replayed from a captured chunk, next to
``mpc_episode`` (robust).

usage: python profiles/time_mpc_scen.py [launches=20] [out.json]"""
import ctypes as C
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
from mpc_scenarios import EmpiricalSampler

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


def fp64_ops(A, h, K, objective):
    """FP64 operations the exhaustive search executes per decision of horizon h (scen_search): per prefix and
    scenario h-2 interior steps of 9; per (prefix, a4) 3 shared operations and 6 per scenario; per leaf 4 shared and
    1 compare, and per leaf and scenario 4 plus the aggregate (mean: multiply and add, worst: compare)."""
    agg = 2 if objective == "mean" else 1
    return A ** (h - 2) * K * (h - 2) * 9 + A ** (h - 1) * (3 + 6 * K) + A ** h * (5 + K * (4 + agg))


def played_env(N, **kw):
    tid, off = synth.make_sessions(N, 1024, 2048, group=64)
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, track_history=1, **kw)
    tid, off = torch.from_numpy(tid).to(dev), torch.from_numpy(off).to(dev)
    env.reset(tid, off)
    env.rollout("bba", 6, want=())
    return env, tid, off


def scenarios(env, H, K, seed):
    out = decide_batch(env.state("sizes"), env.state("utility"), env.state("chunk").clone(),
                       env.state("last_q").clone(), env.state("buffer").clone(), env.state("bw_hist").t().contiguous(),
                       env.state("hist_len").clone(), H, mode="robust", params=env.params,
                       last_pred=env.state("last_pred").clone(), err_ring=env.state("err_ring").t().contiguous(),
                       err_len=env.state("err_len").clone())
    c = out["preds"][:, :1]
    g = torch.Generator(device=dev).manual_seed(seed)
    f = torch.exp(torch.empty(env.n, K, H, dtype=torch.float64, device=dev).uniform_(-0.6931, 0.6931, generator=g))
    return (c[:, None, :] * f).contiguous()


lib = _lib.load()
probe = {}
for kind, pname in ((0, "dadd"), (1, "dfma")):
    g, t = C.c_double(0.0), C.c_float(0.0)
    _lib.check(lib.abr_fp64_probe(C.c_int(kind), C.c_int(4096), C.byref(g), C.byref(t), None))
    probe[pname + "_gops"] = round(g.value, 1)

result = dict(gpu=name, power_limit_and_max_sm_clock=power,
              world=dict(V=V, A=A, traces="1024 x 2048 synthetic", state="6 BBA chunks after a reset",
                         scenarios="robust c times log-uniform [0.5, 2] factors per (session, scenario, step)",
                         L2="256 MB overwritten before every launch",
                         order="each scenario call alternates with mpc_decide_pred on scenario 0"),
              fp64_probe=probe, decide={})

for N, H, Ks, iters in ((131072, 5, (1, 4, 8, 16), n_iter), (2048, 7, (4,), max(4, n_iter // 3))):
    env, _, _ = played_env(N)
    act = torch.empty(N, dtype=torch.int32, device=dev)
    for K in Ks:
        scen = scenarios(env, H, K, seed=K)
        row = scen[:, 0].contiguous()
        for objective in ("mean", "worst"):
            for exhaustive in (False, True):
                if H == 7 and exhaustive:
                    continue
                sc, pr = timed_pair(lambda: env.mpc_decide_scen(scen, H, objective=objective, out=act,
                                                                exhaustive=exhaustive),
                                    lambda: env.mpc_decide_pred(row, H, out=act, exhaustive=exhaustive), iters)
                key = f"N{N}_H{H}_K{K}_{objective}_{'exhaustive' if exhaustive else 'branch_and_bound'}"
                r = dict(mpc_decide_scen=summary(sc, N), mpc_decide_pred=summary(pr, N))
                r["scen_over_pred_mean_time"] = round(r["mpc_decide_scen"]["mean_us"] / r["mpc_decide_pred"]["mean_us"], 3)
                if exhaustive:
                    ops = fp64_ops(A, H, K, objective)
                    gops = ops * N / (r["mpc_decide_scen"]["mean_us"] * 1e-6) / 1e9
                    r["roofline"] = dict(fp64_ops_per_decision=ops, achieved_gops=round(gops, 1),
                                         fraction_of_dadd_probe=round(gops / probe["dadd_gops"], 3))
                result["decide"][key] = r
                print(key, r["mpc_decide_scen"]["mean_us"], r["mpc_decide_pred"]["mean_us"], flush=True)
    assert env.error_count() == 0
    del env

# ---- 48-chunk episodes at 16 384 sessions ----
Ne, H = 16384, 5
env, tid, off = played_env(Ne, track_acc=1, hist_k=8)
sampler = EmpiricalSampler()


def robust_episode():
    env.reset(tid, off)
    env.mpc_episode(V, H, mode="robust")


def scen_episode():
    env.reset(tid, off)
    env.mpc_episode_scen(V, sampler, H, objective="mean")


env.reset(tid, off)
s = torch.cuda.Stream()
s.wait_stream(torch.cuda.current_stream())
with torch.cuda.stream(s):
    env.mpc_episode_scen(1, sampler, H, objective="mean")
torch.cuda.current_stream().wait_stream(s)
graph = torch.cuda.CUDAGraph()
with torch.cuda.graph(graph):
    env.mpc_episode_scen(1, sampler, H, objective="mean")


def graph_episode():
    env.reset(tid, off)
    for _ in range(V):
        graph.replay()


ep = {}
n_ep = max(3, n_iter // 5)
rob, eager = timed_pair(robust_episode, scen_episode, n_ep, warm=1)
_, replay = timed_pair(robust_episode, graph_episode, n_ep, warm=1)
for k, us in (("mpc_episode_robust", rob), ("mpc_episode_scen_mean_K8_eager", eager),
              ("mpc_episode_scen_mean_K8_graph", replay)):
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
