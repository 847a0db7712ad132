"""The search kernels in every compiled form and search path they have, bit for bit against the C oracle.  Run with
-m gpu.

``search_forms.py`` restates which instantiation of ``abr_mpc_kernel`` (warps per session, compiled ladder size, robust
/ branch and bound, smooth_penalty == 1) and which per-session path (one level, plain, parent-state cache, compacted)
a decision takes, and lists cases that together reach every reachable combination; ``test_search_forms_ledger.py``
checks that on the CPU.  Here every case runs on the device against ``orc.mpc_decide``, and ``abr_lookahead_kernel``
runs at every lane layout (A = 1 ... 16) in both its forms against ``lookahead_oracle.decide``.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from abrsimulator_b200 import _lib
from abrsimulator_b200.env import BatchedABREnv
from abrsimulator_b200.mpc import decide_batch
from oracle import oracle as orc
from helpers import bits_equal, small_world
import lookahead_oracle as lo
import search_forms as sf

@pytest.mark.parametrize("case", sf.MPC_CASES, ids=[c.id for c in sf.MPC_CASES])
def test_mpc_form_matches_oracle(case):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert case.forms(sms) == case.forms(), "on this device the case leaves the cell it is listed for"
    if case.N > case.slot_step(sms):      # a slot's next session is another distinct session, not a copy
        assert case.slot_step(sms) % case.n != 0
    b, kw = sf.mpc_inputs(case, seed=sf.MPC_CASES.index(case))
    exp, util, st = sf.mpc_expected(case, b, kw)
    # non-degenerate: every listed horizon occurs, the decisions differ, and the ties cases do tie
    h_got = (exp["best_seq"] >= 0).sum(axis=1)
    assert exp["n_errors"] == 0 and sorted(set(h_got.tolist())) == sorted(case.hs)
    assert case.A == 1 or len(np.unique(exp["action"])) >= 2
    if case.ties:
        assert 2 * sf.prefix_ties(case, b, kw, exp) >= case.n
    mode, flags = case.mode_flags
    T, n = case.tile, case.n
    dev = torch.device("cuda")
    tile = lambda x: np.ascontiguousarray(np.tile(x, (T,) + (1,) * (x.ndim - 1)))
    t = lambda x, dt: torch.from_numpy(np.ascontiguousarray(x)).to(dev, dt)
    st_gpu = (None, None, None)
    if mode == 1:
        st_gpu = (t(tile(b["last_pred"]), torch.float64), t(tile(b["err_ring"]), torch.float64),
                  t(tile(b["err_len"]), torch.int32))
    got = decide_batch(t(b["sizes"], torch.float64), t(util, torch.float64), t(tile(b["chunk"]), torch.int32),
                       t(tile(b["prev_q"]), torch.int32), t(tile(b["buffer"]), torch.float64),
                       t(tile(b["bw_hist"]), torch.float64), t(tile(b["hist_len"]), torch.int32), case.H, mode, flags,
                       _lib.default_params(**kw), *st_gpu)
    torch.cuda.synchronize()
    per_copy = lambda x: x.cpu().numpy().reshape((T, n) + tuple(x.shape[1:]))
    assert int(got["errors"].item()) == 0
    act, seq, bj, preds = (per_copy(got[k]) for k in ("action", "best_seq", "best_j", "preds"))
    for c in range(T):          # every copy equals the oracle's decision of its original
        assert np.array_equal(act[c], exp["action"]), c
        assert np.array_equal(seq[c], exp["best_seq"]), c
        assert bits_equal(bj[c], exp["best_J"]) == 0, c
        if mode == 1:
            assert bits_equal(preds[c], exp["preds"]) == 0, c
        else:                   # mode 0 writes the predictions of the h chunks it looks at
            for h in case.hs:
                m = b["h"] == h
                assert bits_equal(preds[c][m, :h], exp["preds"][m, :h]) == 0, (c, h)
    if mode == 1:
        lp, er, el = (per_copy(x) for x in st_gpu)
        for c in range(T):
            assert bits_equal(lp[c], st[0]) == 0, c
            assert np.array_equal(el[c], st[2]), c
            for s in range(n):
                live = min(int(st[2][s]), case.K)
                assert bits_equal(er[c][s, :live], st[1][s, :live]) == 0, (c, s)


# ---- the environment's K-major history ring, more than 32 samples long and wrapped ----
@pytest.mark.parametrize("A", [16, 7])
def test_env_mpc_long_ring_matches_oracle(A):
    N, K, Vv = 96, 64, 100
    ladder = tuple(np.geomspace(200.0, 6000.0, A))
    bitrates, sizes, bw, tl, ti = small_world(n_traces=8, T=400, V=Vv, ladder=ladder)
    params = dict(track_history=1, hist_k=K, max_buffer=30.0)
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, **params)
    ref = orc.OracleEnv(bw, tl, ti, sizes, bitrates, N, **params)
    rng = np.random.default_rng(A)
    tid = rng.integers(0, 8, size=N).astype(np.int32)
    off = rng.uniform(0, 400.0, size=N)
    env.reset(tid, off)
    ref.reset(tid, off)

    def decide(H, mode):
        act, bj = env.mpc_decide(H, mode, want_score=True)
        e_act, e_bj = ref.mpc_decide(H, _lib.MPC_ROBUST if mode == "robust" else _lib.MPC_REF)
        assert np.array_equal(act.cpu().numpy(), e_act), (H, mode)
        ok = ~np.isnan(e_bj)
        assert bits_equal(bj.cpu().numpy()[ok], e_bj[ok]) == 0 and np.isnan(bj.cpu().numpy()[~ok]).all(), (H, mode)
        assert bits_equal(env.state("last_pred").cpu().numpy(), ref.field("last_pred")) == 0
        el = env.state("err_len").cpu().numpy()
        assert np.array_equal(el, ref.field("err_len"))
        er_g, er_c = env.state("err_ring").cpu().numpy().T, ref.field("err_ring")
        for s in range(N):
            live = min(int(el[s]), K)
            assert bits_equal(er_g[s, :live], er_c[s, :live]) == 0, s
        return e_act

    acts = []
    for t in range(72):                 # the error ring fills past 32, the throughput ring wraps past 64
        acts.append(decide(3, "robust"))
        a = rng.integers(0, A, size=N).astype(np.int32)
        env.step(torch.from_numpy(a).cuda(), want_next_sizes=False)
        ref.step(a, want_next_sizes=False)
    assert int(env.state("hist_len").min()) > K and int(env.state("err_len").min()) > 32
    for H in (3, 4):
        for mode in ("reference", "robust"):
            acts.append(decide(H, mode))
    for t in range(Vv - 72 + 3):        # decide -> step across the end of the video
        act = decide(4, "robust")
        env.step(torch.from_numpy(act).cuda(), want_next_sizes=False)
        ref.step(act, want_next_sizes=False)
        acts.append(act)
    assert int(env.state("chunk").max()) < 4
    assert len(np.unique(np.concatenate(acts))) >= 2
    assert env.error_count() == 0 and ref.errors() == 0


# ---- lookahead: every lane layout, both forms ----
def lookahead_ladder(A):
    """A ladder within the traces' 0.2-6 Mbit/s, so that the best first action varies from session to session."""
    return (1000.0,) if A == 1 else tuple(np.geomspace(150.0, 3500.0, A))


@pytest.mark.parametrize("case", sf.LOOKAHEAD_CASES, ids=[c.id for c in sf.LOOKAHEAD_CASES])
def test_lookahead_form_matches_oracle(case):
    A, H, N = case.A, case.H, case.n
    bitrates, sizes, bw, tl, ti = small_world(n_traces=8, T=200, V=sf.LOOKAHEAD_V, ladder=lookahead_ladder(A),
                                              ragged=True, seed=A)
    params = dict(auto_reset=case.auto_reset, max_buffer=30.0, default_quality=0)
    env = BatchedABREnv(bw, sizes, bitrates, N, trace_len=tl, trace_interval=ti, **params)
    ref = orc.OracleEnv(bw, tl, ti, sizes, bitrates, N, **params)
    rng = np.random.default_rng(100 * A + H)
    tid = rng.integers(0, 8, size=N).astype(np.int32)
    off = rng.uniform(0, 300.0, size=N)
    env.reset(tid, off)
    ref.reset(tid, off)
    acts, hs = [], set()
    for n_steps in case.steps:
        for _ in range(n_steps):
            a = rng.integers(0, A, size=N).astype(np.int32)
            env.step(torch.from_numpy(a).cuda(), want_next_sizes=False)
            ref.step(a, want_next_sizes=False)
        act, val, seq = env.lookahead_decide(H, want_value=True, want_seq=True)
        e_act, e_val, e_seq, flagged = lo.decide(ref, H, want_seq=True)
        assert flagged == 0
        assert np.array_equal(act.cpu().numpy(), e_act)
        assert bits_equal(val.cpu().numpy(), e_val) == 0
        assert np.array_equal(seq.cpu().numpy(), e_seq)
        acts.append(e_act)
        hs |= set((e_seq >= 0).sum(axis=1).tolist())
    assert A == 1 or len(np.unique(np.concatenate(acts))) >= 2
    assert max(hs) == H
    assert env.error_count() == 0 and ref.errors() == 0
