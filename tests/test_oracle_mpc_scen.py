"""CPU-only: MPC over caller-supplied throughput scenarios (SPEC §5.7).  The C restatement against the pure-Python
one (both in tests/mpc_scen_oracle.py) on random states, the identities with SPEC §5.6, and the input rules."""
import math

import numpy as np
import pytest

from helpers import bits_equal
import mpc_pred_oracle as mp
import mpc_scen_oracle as ms


def _world(rng, A, V):
    lad = np.sort(rng.uniform(0.2, 5.0, size=A))
    bitrates = np.tile(lad, (V, 1)) * rng.uniform(0.9, 1.1, size=(V, 1))
    sizes = bitrates * 4.0 * rng.uniform(0.8, 1.2, size=(V, A))
    return bitrates, sizes


def _states(rng, A, H, V, n, K):
    """n sessions: random chunks, a quarter within H of the end of the video, last_q = -1 for a fifth, K scenarios of
    per-step throughputs spread over a factor of 30."""
    chunk = np.where(rng.random(n) < 0.25, rng.integers(V - H, V + 1, size=n), rng.integers(0, V, size=n))
    prev_q = np.where(rng.random(n) < 0.2, -1, rng.integers(0, A, size=n))
    buffer = np.round(rng.uniform(0, 40, size=n), 9)
    pred = rng.uniform(0.2, 6.0, size=(n, K, H))
    return chunk.astype(np.int32), prev_q.astype(np.int32), buffer, pred


PENALTIES = [(1.0, 4.3), (0.6, 4.3), (2.5, 1.0), (0.0, 4.3), (1.0, 0.0), (0.0, 0.0)]
SHAPES = [(1, 4, 3), (2, 4, 5), (3, 3, 4), (4, 3, 2), (5, 2, 3), (6, 2, 1), (3, 1, 16)]   # (A, H, K)


@pytest.mark.parametrize("A,H,K", SHAPES, ids=[f"A{a}H{h}K{k}" for a, h, k in SHAPES])
@pytest.mark.parametrize("objective", ["mean", "worst"])
def test_c_restatement_equals_python_restatement(A, H, K, objective):
    V, n = 12, 60
    obj = ms.OBJECTIVES[objective]
    rng = np.random.default_rng(A * 100 + H * 10 + K + obj)
    seen = dict(short=0, past=0, noprev=0, states=0)
    for t, (vw, rw) in enumerate(PENALTIES):
        bitrates, sizes = _world(rng, A, V)
        chunk, prev_q, buffer, pred = _states(rng, A, H, V, n, K)
        w = None
        if obj == ms.MEAN and t % 2:
            w = rng.uniform(0, 2, size=(n, K)) * (rng.random((n, K)) < 0.8)
            w[:, 0] += 0.1
        L, B = 4.0, float(rng.choice([20.0, 60.0]))
        c = ms.decide_scen_c(sizes, bitrates, chunk, prev_q, buffer, pred, H, L, B, vw, rw, obj, w)
        assert c["n_errors"] == 0
        for s in range(n):
            py = ms.decide_scen(int(chunk[s]), int(prev_q[s]), float(buffer[s]), pred[s], H, bitrates.tolist(),
                                sizes.tolist(), L, B, vw, rw, obj, None if w is None else w[s])
            h = len(py["best_seq"])
            assert c["action"][s] == py["action"], s
            assert c["best_seq"][s].tolist() == py["best_seq"] + [-1] * (H - h), s
            assert bits_equal(c["best_J"][s], py["best_J"]) == 0, (s, c["best_J"][s], py["best_J"])
            seen["short"] += 0 < V - chunk[s] < H
            seen["past"] += chunk[s] >= V
            seen["noprev"] += prev_q[s] < 0
            seen["states"] += 1
    assert (seen["short"] or H == 1) and seen["past"] and seen["noprev"] and seen["states"] == 360


def _batch(seed, A=5, H=4, V=14, n=300):
    rng = np.random.default_rng(seed)
    bitrates, sizes = _world(rng, A, V)
    chunk, prev_q, buffer, pred = _states(rng, A, H, V, n, 1)
    return rng, bitrates, sizes, chunk, prev_q, buffer, pred[:, 0, :]


def _same(a, b, best_j=True):
    assert np.array_equal(a["action"], b["action"]) and np.array_equal(a["best_seq"], b["best_seq"])
    if best_j:
        assert bits_equal(a["best_J"], b["best_J"]) == 0


@pytest.mark.parametrize("vw,rw", [(1.0, 4.3), (0.6, 2.0)])
def test_one_scenario_is_the_prediction_decision(vw, rw):
    """K = 1: no weights and either objective, or MEAN with w = [1.0], decide as SPEC §5.6 on the same row."""
    _, bitrates, sizes, chunk, prev_q, buffer, row = _batch(1)
    H = row.shape[1]
    ref = mp.decide_pred_c(sizes, bitrates, chunk, prev_q, buffer, row, H, 4.0, 30.0, vw, rw)
    for obj, w in ((ms.MEAN, None), (ms.WORST, None), (ms.MEAN, np.ones((len(chunk), 1)))):
        got = ms.decide_scen_c(sizes, bitrates, chunk, prev_q, buffer, row[:, None, :], H, 4.0, 30.0, vw, rw, obj, w)
        _same(got, ref)


def test_identical_scenarios_under_worst_are_the_prediction_decision():
    _, bitrates, sizes, chunk, prev_q, buffer, row = _batch(2)
    H = row.shape[1]
    ref = mp.decide_pred_c(sizes, bitrates, chunk, prev_q, buffer, row, H, 4.0, 30.0, 1.0, 4.3)
    got = ms.decide_scen_c(sizes, bitrates, chunk, prev_q, buffer, np.repeat(row[:, None, :], 7, axis=1), H, 4.0, 30.0,
                           1.0, 4.3, ms.WORST)
    _same(got, ref)


def test_a_dominated_scenario_decides_the_worst_case():
    """Scenario 0 pointwise <= every other one.  With rw >= 0, buffer <= max_buffer and chunk_length <= max_buffer,
    every step of the rollout is monotone in fp64: the download time sizes / p falls as p grows; max0(x - b), the
    additions and t = max0(b - dl) are monotone; t + L <= B + L, and (t + L) - max0((t + L) - B) is either t + L or
    exactly B (Sterbenz: B <= t + L <= 2B).  So every rt_k >= rt_0, q_k <= q_0 fails only as q_k >= q_0, and WORST,
    which replaces Q only on a strict <, keeps q_0: the SPEC §5.6 decision on row 0, best_j included."""
    rng, bitrates, sizes, chunk, prev_q, buffer, row = _batch(3)
    H, N, B = row.shape[1], len(chunk), 40.0
    assert buffer.max() <= B
    others = row[:, None, :] * rng.uniform(1.0, 3.0, size=(N, 5, H))
    others[:, 2] = row                                  # a tie with scenario 0 is allowed
    pred = np.concatenate([row[:, None, :], others], axis=1)
    for vw, rw in ((1.0, 4.3), (0.0, 0.0), (0.6, 1.0)):
        ref = mp.decide_pred_c(sizes, bitrates, chunk, prev_q, buffer, row, H, 4.0, B, vw, rw)
        got = ms.decide_scen_c(sizes, bitrates, chunk, prev_q, buffer, pred, H, 4.0, B, vw, rw, ms.WORST)
        _same(got, ref)


def test_weights_scale_and_zero_weight_scenarios():
    rng, bitrates, sizes, chunk, prev_q, buffer, _ = _batch(4)
    N, K, H = len(chunk), 4, 4
    pred = rng.uniform(0.3, 6.0, size=(N, K, H))
    w = rng.uniform(0.1, 2.0, size=(N, K))
    base = ms.decide_scen_c(sizes, bitrates, chunk, prev_q, buffer, pred, H, 4.0, 30.0, 1.0, 4.3, ms.MEAN, w)
    for e in (-3, 5):
        got = ms.decide_scen_c(sizes, bitrates, chunk, prev_q, buffer, pred, H, 4.0, 30.0, 1.0, 4.3, ms.MEAN,
                               w * 2.0 ** e)
        _same(got, base, best_j=False)
        assert bits_equal(got["best_J"], base["best_J"] * 2.0 ** e) == 0
    extra = np.concatenate([pred, rng.uniform(0.01, 0.1, size=(N, 1, H))], axis=1)
    got = ms.decide_scen_c(sizes, bitrates, chunk, prev_q, buffer, extra, H, 4.0, 30.0, 1.0, 4.3, ms.MEAN,
                           np.concatenate([w, np.zeros((N, 1))], axis=1))
    _same(got, base, best_j=False)


def test_mean_and_worst_differ_where_the_risk_differs():
    """A fast common future and a rare stall: MEAN takes the high rung the fast future pays for, WORST the low one."""
    bitrates = np.tile([1.0, 2.0, 4.0], (6, 1))
    sizes = bitrates * 4.0
    pred = np.array([[[8.0] * 3, [8.0] * 3, [8.0] * 3, [0.5] * 3]])
    m = ms.decide_scen_c(sizes, bitrates, [0], [2], [4.0], pred, 3, 4.0, 60.0, 1.0, 4.3, ms.MEAN,
                         [[1.0, 1.0, 1.0, 0.05]])
    w = ms.decide_scen_c(sizes, bitrates, [0], [2], [4.0], pred, 3, 4.0, 60.0, 1.0, 4.3, ms.WORST)
    assert m["action"][0] == 2 and w["action"][0] == 0


@pytest.mark.parametrize("bad", [0.0, -1.0, math.nan, math.inf, -math.inf, -0.0])
def test_invalid_scenarios_are_input_errors(bad):
    bitrates = np.tile([1.0, 2.0, 4.0], (6, 1))
    sizes = bitrates * 4.0
    H, K = 4, 3
    pred = np.full((4, K, H), 2.0)
    pred[0, 2, 1] = bad                 # h = 4: read
    pred[1, 1, 3] = bad                 # chunk 4: h = 2, entry 3 is not read
    pred[2, 0, 2] = bad                 # done: nothing is read
    pred[3, 0, 0] = bad                 # chunk 6 = V: h = 0, nothing is read
    for obj in (ms.MEAN, ms.WORST):
        r = ms.decide_scen_c(sizes, bitrates, [0, 4, 1, 6], [1, 1, 1, 1], [5.0] * 4, pred, H, 4.0, 60.0, 1.0, 4.3, obj,
                             done=[0, 0, 1, 0])
        assert r["action"].tolist()[0] == -1 and r["n_errors"] == 1
        assert r["action"][1] >= 0 and r["best_seq"][1].tolist()[2:] == [-1, -1]
        assert r["action"][2] == 0 and r["action"][3] == 0
        assert math.isnan(r["best_J"][0]) and math.isnan(r["best_J"][2]) and math.isnan(r["best_J"][3])
        py = ms.decide_scen(0, 1, 5.0, pred[0], H, bitrates.tolist(), sizes.tolist(), 4.0, 60.0, 1.0, 4.3, obj)
        assert py["action"] == -1 and py["error"]


@pytest.mark.parametrize("w", [[1.0, -1.0], [0.0, 0.0], [math.nan, 1.0], [math.inf, 1.0], [-0.0, -0.0]])
def test_invalid_weights_are_input_errors(w):
    bitrates = np.tile([1.0, 2.0, 4.0], (6, 1))
    sizes = bitrates * 4.0
    pred = np.full((2, 2, 3), 2.0)
    r = ms.decide_scen_c(sizes, bitrates, [0, 0], [1, 1], [5.0, 5.0], pred, 3, 4.0, 60.0, 1.0, 4.3, ms.MEAN,
                         [w, [1.0, 0.0]])
    assert r["action"].tolist()[0] == -1 and r["action"][1] >= 0 and r["n_errors"] == 1


def test_no_finite_aggregate_gives_sequence_zero_and_infinite_j():
    """A subnormal throughput passes the input rule, but sizes / p overflows to inf.  Every Q is then -inf (rw > 0) or
    NaN (rw = 0, or MEAN with weight 0 on that scenario): sequence 0 and best_J = +inf, in both restatements.  A NaN
    Q is never chosen over a finite one."""
    bitrates = np.tile([1.0, 2.0, 4.0], (6, 1))
    sizes = bitrates * 4.0
    pred = np.full((1, 2, 3), 2.0)
    pred[0, 0, 1] = 1e-310
    for rw, obj, w in ((4.3, ms.WORST, None), (0.0, ms.MEAN, None), (4.3, ms.MEAN, [[0.0, 1.0]])):
        c = ms.decide_scen_c(sizes, bitrates, [1], [2], [5.0], pred, 3, 4.0, 60.0, 1.0, rw, obj, w)
        py = ms.decide_scen(1, 2, 5.0, pred[0], 3, bitrates.tolist(), sizes.tolist(), 4.0, 60.0, 1.0, rw, obj,
                            None if w is None else w[0])
        assert c["n_errors"] == 0 and c["best_seq"][0].tolist() == py["best_seq"] == [0, 0, 0]
        assert c["best_J"][0] == py["best_J"] == math.inf
