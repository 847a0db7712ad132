"""The chunk-step kernels on every access path, head outcome, speculation outcome and compiled form that
``step_forms.py`` restates, bit for bit against the C oracle, and the statistics vector bit for bit against the
restated reduction trees.  Run with -m gpu.

Every case checks every output of every step (fp32 outputs: the oracle's value rounded once), the final state, the
accumulators, the per-session QoE cost, the statistics and the error count against ``oracle/abr_oracle.c``, and
asserts that the cells it is listed for occur in its own data.  The grid of the per-step kernel, and so its staging,
is restated for the SM count of the device the test runs on.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from abrsimulator_b200.env import BatchedABREnv, StepResult
from oracle import oracle as orc
from helpers import bits_equal
import lookahead_oracle as lo
import policy_oracle as po
import step_forms as sf

STATE_I = ("seg", "chunk", "last_q", "trace_id")
STATE_F = ("phase", "pos", "buffer")
OUT = (("delay", "delay"), ("sleep", "sleep"), ("buffer", "buffer"), ("rebuffer", "rebuf"), ("reward", "reward"))
WANT = dict(core=("delay", "sleep", "buffer", "rebuffer", "reward", "end_of_video"),
            none=())
WANT["core+"] = WANT["core"] + ("actions",)


def exact(got, exp, what):
    nd = bits_equal(np.asarray(got), np.asarray(exp))
    assert nd == 0, f"{what}: {nd} values differ"


def check_state(env, ref):
    for f in STATE_I:
        assert np.array_equal(env.state(f).cpu().numpy(), ref.field(f)), f
    for f in STATE_F:
        exact(env.state(f).cpu().numpy(), ref.field(f), f)


def session_cost(p, acc):
    """abr_qoe_cost_kernel's session_cost on the oracle's accumulators (same operations, same order)."""
    c = p.rebuf_penalty * acc[1] + p.smooth_penalty * acc[3]
    if p.live:
        c = c + p.startup_penalty * acc[8]
        with np.errstate(divide="ignore", invalid="ignore"):
            lat = np.where(acc[10] > 0.0, acc[9] / (p.latency_tick * acc[10]), 0.0)
        c = c + p.latency_penalty * lat
    return c


def observe_heads(case, tab, smem, pre_pos, pre_chunk, tid, actions, sizes):
    """Head outcomes of the steps that start at pre_pos / pre_chunk with `actions` ([steps][N] each)."""
    cells = set()
    kernel = dict(policy="step", run="fused", run_host="fused").get(case.kernel, case.kernel)
    for t in range(len(actions)):
        raw = pre_pos[t] + sizes[pre_chunk[t], actions[t]]
        out = sf.head_outcome(tab, tid, raw, smem)
        for path, m in (("smem", smem), ("global", ~smem)):
            cells |= {sf.head(kernel, path, o) for o in set(out[m].tolist())}
    return cells, out


@pytest.mark.parametrize("case", sf.STEP_CASES, ids=[c.name for c in sf.STEP_CASES])
def test_step_form_matches_oracle(case):
    sms = torch.cuda.get_device_properties(0).multi_processor_count   # launch_step sizes its grid from the device
    bitrates, sizes, bw, tl, ti = sf.make_world(case.world)
    N, p = case.N, case.kw
    tid, off = sf.make_layout(case, tl, ti, sms)
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, **p)
    ref = po.PolicyEnv(bw, tl, ti, sizes, bitrates, N, **p)
    env.reset(tid, off)
    ref.reset(tid, off)
    tab = sf.trace_tables(bw, tl, ti, ref.params.payload)
    live = bool(p.get("live", 0))
    f32 = case.dtype == "f32"
    dtype = torch.float32 if f32 else torch.float64
    as_out = (lambda x: np.asarray(x).astype(np.float32)) if f32 else (lambda x: x)   # an output is rounded once
    rng = np.random.default_rng(case.seed)
    seen = set()
    I_of = ti[tid]
    seen |= {("edge", "reset_fmod")} if sf.reset_fmod(off, I_of).any() else set()
    seen |= {("edge", "I_pow2" if sf.pow2_inverse_exact(x) else "I_inexact") for x in np.unique(I_of)}
    seen.add(("edge", "q_pow2" if sf.pow2_inverse_exact(ref.params.sleep_quantum) else "q_inexact"))
    pre_pos, pre_chunk, acts, sleeps = [], [], [], []
    expected_errors = 0          # what the kernels add to the error count beyond the oracle's per-step count

    def sleep_edges(sl):
        if sf.advance_fmod(sl, I_of).any():
            seen.add(("edge", "live_fmod" if live else "sleep_fmod"))

    if case.kernel in ("step", "policy", "lookahead"):
        paths = sf.step_paths(tid, tab.T_max, sms)
        smem = paths.smem
        form = case.form()
        seen |= {("step", form, "smem")} if smem.any() else set()
        seen |= {("step", form, "global")} if (~smem).any() else set()
        acc = np.zeros((orc.NUM_ACC, N))
        for t in range(case.steps):
            pre_pos.append(ref.field("pos")), pre_chunk.append(ref.field("chunk"))
            if case.kernel == "policy":    # greedy: the first arg max of the logits
                logits = rng.standard_normal((N, env.A)).astype(np.float32)
                a = np.argmax(logits, axis=1).astype(np.int32)
                e = lambda: torch.empty(N, dtype=torch.float64, device="cuda")
                got = StepResult(e(), e(), e(), e(), e(), None, torch.empty(N, dtype=torch.uint8, device="cuda"), None)
                act = torch.empty(N, dtype=torch.int32, device="cuda")
                env.step_policy(torch.from_numpy(logits).cuda(), sample=False, action_out=act, out=got)
                assert np.array_equal(act.cpu().numpy(), a), t
                keys = OUT
            else:
                a = rng.integers(0, env.A, size=N).astype(np.int32)
                got = env.step(a, want_throughput=True, dtype=dtype)
                keys = OUT + (("throughput", "throughput"), ("next_sizes", "next_sizes")) + \
                    ((("latency", "latency"),) if live else ())
            acts.append(a)
            exp = ref.step(a, acc=acc)
            for k_g, k_c in keys:
                assert getattr(got, k_g).dtype == (torch.float64 if case.kernel == "policy" else dtype)
                exact(getattr(got, k_g).cpu().numpy(), as_out(exp[k_c]), f"{k_g}@{t}")
            assert np.array_equal(got.end_of_video.cpu().numpy(), exp["eov"]), t
            sleep_edges(exp["sleep"])
        check_state(env, ref)
        if p.get("track_acc"):
            exact(env.session_acc().cpu().numpy(), acc, "acc")
            exact(env.qoe_cost().cpu().numpy(), session_cost(ref.params, acc), "qoe_cost")
            exact(env.stats().cpu().numpy(), sf.stats_stage1(acc), "stats")
        if case.layout == "bign":
            tpb, _ = sf.step_grid(N, sms)
            seen |= {("dispatch", "prefetch")} if sf.step_prefetch(N, sms) else set()
            seen |= {("dispatch", "tiles_per_block>kStepTiles")} if tpb > sf.K_STEP_TILES else set()
            seen |= {("dispatch", "partial_tile")} if paths.partial_last_tile else set()
            seen |= {("dispatch", "partial_block")} if paths.partial_last_block else set()
            seen |= {("dispatch", f"parity{k}") for k in (0, 1) if (paths.restages > k).any()}
            seen |= {("dispatch", "straddle")} if paths.straddle > 0 else set()
            seen |= {("dispatch", "mixed_tile_per_block")} if (paths.mixed_per_block[:-1] >= 1).all() else set()
        if case.kernel == "lookahead":
            smem = np.zeros(N, bool)
            act, val, seq = env.lookahead_decide(case.H, want_value=True, want_seq=True)
            e_act, e_val, e_seq, flagged = lo.decide(ref, case.H, want_seq=True)
            assert np.array_equal(act.cpu().numpy(), e_act)
            exact(val.cpu().numpy(), e_val, "best value")
            assert np.array_equal(seq.cpu().numpy(), e_seq)
            expected_errors = flagged   # SPEC §4.4: a session whose lookahead hits the safety net counts once
            # the first level of the tree: every first action from the decision's state
            pos, chunk = ref.field("pos"), ref.field("chunk")
            pre_pos = [pos] * env.A
            pre_chunk = [chunk] * env.A
            acts = [np.full(N, a, np.int32) for a in range(env.A)]
        if not live:
            cells, _ = observe_heads(case, tab, smem, pre_pos, pre_chunk, tid, acts, sizes)
            seen |= cells
    else:
        smem = sf.rollout_paths(tab, tid, env.V, env.A)
        form = case.form()
        seen |= {("fused", form, "smem")} if smem.any() else set()
        seen |= {("fused", form, "global")} if (~smem).any() else set()
        acts_in = rng.integers(0, env.A, size=(case.steps, N)).astype(np.int32) if case.policy == sf.FIXED else None
        seed = 0x5EED + case.seed
        exp = ref.rollout(case.policy, case.steps, seed=seed, actions=acts_in)
        if case.kernel == "fused":
            got = env.rollout(case.policy, case.steps, seed=seed, actions=acts_in, want=WANT[case.want], dtype=dtype)
            got = {k: v.cpu().numpy() for k, v in got.items()}
            exact(env.stats().cpu().numpy(), sf.stats_fused(exp["acc"]), "stats")
            exact(env.qoe_cost().cpu().numpy(), session_cost(ref.params, exp["acc"]), "qoe_cost")
        else:   # the fused reset: the kernel resets every session itself, then the episode, cost and statistics
            env.reset(np.zeros(N, np.int32))                   # a stale state for the fused reset to replace
            if case.kernel == "run":
                got, cost, stats = env.run(case.policy, case.steps, tid, off, seed=seed, actions=acts_in)
                got = {k: v.cpu().numpy() for k, v in got.items()}
                cost, stats = cost.cpu().numpy(), stats.cpu().numpy()
            else:
                res = env.run_host(case.policy, case.steps, tid, off, seed=seed, actions=acts_in,
                                   want_reward_traj=True, want_qoe_cost=True)
                got, cost, stats = dict(reward=res["reward"]), res["qoe_cost"], res["stats"]
                exact(res["acc"], exp["acc"], "acc (host)")
            exact(stats, sf.stats_fused(exp["acc"]), "stats")
            exact(cost, session_cost(ref.params, exp["acc"]), "qoe_cost")
            seen |= {("reset", case.kernel, path) for path, m in (("smem", smem), ("global", ~smem)) if m.any()}
        for k_g, k_c in OUT:
            if k_g in got:
                assert got[k_g].dtype == (np.float32 if f32 else np.float64), k_g
                exact(got[k_g], as_out(exp[k_c]), k_g)
        if "end_of_video" in got:
            assert np.array_equal(got["end_of_video"], exp["eov"])
        if "actions" in got:
            assert np.array_equal(got["actions"], exp["actions"])
        check_state(env, ref)
        exact(env.session_acc().cpu().numpy(), exp["acc"], "acc")
        sleep_edges(exp["sleep"])
        # replay the oracle's actions step by step for the pre-step states
        rep = orc.OracleEnv(bw, tl, ti, sizes, bitrates, N, **p)
        rep.reset(tid, off)
        for t in range(case.steps):
            pre_pos.append(rep.field("pos")), pre_chunk.append(rep.field("chunk"))
            o = rep.step(exp["actions"][t], want_next_sizes=False)
            sleeps.append(o["sleep"] > 0.0)
        acts = exp["actions"]
        if not live:
            cells, out = observe_heads(case, tab, smem, pre_pos, pre_chunk, tid, acts, sizes)
            seen |= cells
            if "guard" in out:
                # the fused episode counts a session once however many of its steps hit the safety net (one atomic
                # per session in rollout_session), the oracle once per step: equal here because the case runs one
                # step, which the restated count confirms
                assert case.steps == 1 and int((out == "guard").sum()) == ref.errors()
        if case.policy in (sf.FIXED, sf.RANDOM) and not live and case.steps > 1:
            sp = sf.speculation(tab, tid, smem, np.array(pre_pos[1:]),
                                sizes[np.array(pre_chunk[1:]), acts[1:]], np.array(sleeps[:-1]))
            for path, m in (("smem", smem), ("global", ~smem)):
                seen |= {sf.spec(path, o) for o in set(sp[:, m].ravel().tolist())}
    assert env.error_count() == ref.errors() + expected_errors
    missing = sorted(case.reaches - seen, key=str)
    assert not missing, missing


# ---- SPEC §6: the statistics vector, bit for bit, from both reduction trees ----
@pytest.mark.parametrize("N", [1, 63, 64, 65, 2049, 70001, (1 << 21) + 77])
def test_statistics_are_the_restated_reduction_trees(N):
    """After an episode (abr_env_run, the in-kernel reduction; rollout, the separate stage 2 over the episode's block
    partials) the statistics are the 64-session block tree; after per-step calls they are abr_stats_stage1's
    1 024-session tree.  Sessions on scattered traces, so that the partial sums are not round numbers."""
    bitrates, sizes, bw, tl, ti = sf.make_world("bign")
    rng = np.random.default_rng(N)
    tid = rng.integers(0, len(tl), N).astype(np.int32)
    off = rng.uniform(0, 300.0, N)
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, track_acc=1)
    _, _, stats = env.run("random", 6, tid, off, seed=7)
    acc = env.session_acc().cpu().numpy()
    exact(stats.cpu().numpy(), sf.stats_fused(acc), "run")
    exact(env.stats().cpu().numpy(), sf.stats_fused(acc), "stats after run")
    env.rollout("bba", 5, want=())
    acc = env.session_acc().cpu().numpy()
    exact(env.stats().cpu().numpy(), sf.stats_fused(acc), "stats after rollout")
    for _ in range(2):
        env.step(rng.integers(0, env.A, N).astype(np.int32), want_next_sizes=False)
    acc = env.session_acc().cpu().numpy()
    exact(env.stats().cpu().numpy(), sf.stats_stage1(acc), "stats after step")
    assert acc[6].min() == 13.0 and env.error_count() == 0
