"""The session-order sort at every shape ``sort_forms.py`` restates, against the reference order.  Run with -m gpu.

For every case: ``reset(sort_by_trace=True)`` (``abr_env_reset_sorted``, the counting sort or the radix fallback)
installs exactly ``sort_forms.reference_order`` — the stable sort by trace, an invalid id sorting as trace 0 — and
``sort_by_trace`` (the radix sort on its own) returns the same order; every state field and the error count equal
those of ``abr_env_reset`` on the inputs put in that order, with start offsets and without.  One environment then
takes a sequence of calls whose path, run size and number of runs change, which checks that the histogram the
counting sort leaves behind is zero for the next call.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from abrsimulator_b200.env import BatchedABREnv
from helpers import small_world
import sort_forms as sf

STATE = ("seg", "chunk", "last_q", "trace_id", "phase", "pos", "buffer")
T = 4       # segments per trace: the sort reads no trace, so the tables are kept small


def world(n_traces):
    bitrates, sizes, bw, tl, ti = small_world(n_traces=n_traces, T=T, V=8)
    return bitrates, sizes, bw, tl, ti


def offsets(n, seed):
    return np.random.default_rng(seed).uniform(0, 3.0 * T, n)


def check_reset(env, ref, tid, off, want_errors):
    """env was reset sorted; ref gets the same sessions, put into the reference order by the caller, unsorted."""
    n_traces = env.n_traces
    perm = sf.reference_order(tid, n_traces)
    got = env.perm.cpu().numpy()
    assert np.array_equal(got, perm), f"installed order: {int((got != perm).sum())} of {perm.size} positions differ"
    e0 = ref.error_count()
    ref.reset(tid[perm], None if off is None else off[perm])
    for f in STATE:
        assert torch.equal(env.state(f), ref.state(f)), f
    assert ref.error_count() - e0 == want_errors
    return perm


def n_invalid(tid, n_traces):
    return int(((tid < 0) | (tid >= n_traces)).sum())


def sort_case(env, ref, tid, off, session_base=0):
    n_traces = env.n_traces
    e0 = env.error_count()
    env.reset(tid, off, session_base=session_base, sort_by_trace=True)
    bad = n_invalid(tid, n_traces)
    assert env.error_count() - e0 == bad            # one error per invalid id, at the reset only
    perm = check_reset(env, ref, tid, off, bad)
    assert env.session_base == session_base
    return perm


SMALL = [c for c in sf.SORT_CASES if not c.big]


@pytest.mark.parametrize("case", SMALL, ids=[c.name for c in SMALL])
def test_sorted_reset_installs_the_reference_order(case):
    sh = case.shape()
    bitrates, sizes, bw, tl, ti = world(case.n_traces)
    tid = case.ids()
    off = offsets(case.N, case.N) if case.offsets else None
    env = BatchedABREnv(bw, sizes, bitrates, case.N, trace_len=tl, trace_interval=ti)
    ref = BatchedABREnv(bw, sizes, bitrates, case.N, trace_len=tl, trace_interval=ti)
    perm = sort_case(env, ref, tid, off, session_base=7)
    sorted_by_radix = env.sort_by_trace(tid).cpu().numpy()
    assert np.array_equal(sorted_by_radix, perm), \
        f"abr_sort_by_trace: {int((sorted_by_radix != perm).sum())} of {perm.size} positions differ ({sh.path})"
    # the other half: without offsets when the case has them, with them when it has none
    sort_case(env, ref, tid, None if case.offsets else offsets(case.N, 1))
    assert env.error_count() == 2 * n_invalid(tid, case.n_traces)


def test_one_environment_through_changing_shapes():
    """SEQUENCE over 8 192 traces: S = 512 / 4 096, 4 to 196 runs, an empty batch, a histogram that grows; every call
    installs the reference order, so no cell of the histogram was left non-zero by the call before."""
    n_traces = sf.SEQUENCE_TRACES
    bitrates, sizes, bw, tl, ti = world(n_traces)
    cap = max(sf.SEQUENCE)
    env = BatchedABREnv(bw, sizes, bitrates, cap, trace_len=tl, trace_interval=ti)
    ref = BatchedABREnv(bw, sizes, bitrates, cap, trace_len=tl, trace_interval=ti)
    patterns = ("interleaved", "random", "reversed", "chunks", "invalid")
    for k, n in enumerate(sf.SEQUENCE):
        tid = sf.make_ids(patterns[k % len(patterns)], n, n_traces, seed=k)
        off = offsets(n, k) if k % 2 else None
        if n == 0:
            env.reset(tid, off, sort_by_trace=True)
            assert env.n == 0 and env.perm.numel() == 0
            continue
        sort_case(env, ref, tid, off, session_base=k)
        torch.cuda.synchronize()


def test_big_shapes_in_one_environment():
    """BIG_SEQUENCE over 11 264 traces in one environment: 23 * 2^20 sessions (the counting sort at S = 2^20, 48 KB of
    shared memory), 23 * 2^20 + 1 (the cells fallback: radix sort; invalid ids) and 100 000 (the counting sort again,
    on the histogram the first call left)."""
    n_traces = 11264
    bitrates, sizes, bw, tl, ti = world(n_traces)
    cap = max(sf.BIG_SEQUENCE)
    env = BatchedABREnv(bw, sizes, bitrates, cap, trace_len=tl, trace_interval=ti)
    ref = BatchedABREnv(bw, sizes, bitrates, cap, trace_len=tl, trace_interval=ti)
    big = {c.N: c for c in sf.SORT_CASES if c.big}
    for n in sf.BIG_SEQUENCE:
        c = big.get(n)
        tid = c.ids() if c else sf.make_ids("interleaved", n, n_traces)
        off = offsets(n, 3) if n == sf.BIG + 1 else None
        perm = sort_case(env, ref, tid, off)
        if c is not None and c.shape().path.startswith("radix"):
            assert np.array_equal(env.sort_by_trace(tid).cpu().numpy(), perm)
        del tid, off, perm
        torch.cuda.synchronize()


def test_sort_by_trace_on_two_streams_with_growing_scratch():
    """abr_sort_by_trace keeps one grow-only scratch buffer per host thread, ordered across streams by an event: a
    small sort, a larger one on another stream (the buffer grows), and a small one on the first stream again."""
    n_traces = 11265
    bitrates, sizes, bw, tl, ti = world(n_traces)
    env = BatchedABREnv(bw, sizes, bitrates, 1, trace_len=tl, trace_interval=ti)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    calls = ((s1, 1000, "invalid"), (s2, 300000, "reversed"), (s1, 5000, "random"), (s2, 300001, "invalid"))
    tids = [torch.from_numpy(sf.make_ids(p, n, n_traces, seed=n)).cuda() for _, n, p in calls]
    torch.cuda.synchronize()
    perms = []
    for (s, n, p), tid in zip(calls, tids):
        with torch.cuda.stream(s):
            perms.append(env.sort_by_trace(tid))
    torch.cuda.synchronize()
    for (s, n, p), tid, perm in zip(calls, tids, perms):
        want = sf.reference_order(tid.cpu().numpy(), n_traces)
        assert np.array_equal(perm.cpu().numpy(), want), (n, p)
