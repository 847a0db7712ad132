"""CPU-only: MPC over caller-supplied throughput predictions (SPEC §5.6).  The C restatement against the pure-Python
one (both in tests/mpc_pred_oracle.py) on random states, and known answers."""
import itertools
import math

import numpy as np
import pytest

from oracle import mpc_oracle as mo
from helpers import bits_equal
import mpc_pred_oracle as mp


def _world(rng, A, V):
    lad = np.sort(rng.uniform(0.2, 5.0, size=A))
    bitrates = np.tile(lad, (V, 1)) * rng.uniform(0.9, 1.1, size=(V, 1))
    sizes = bitrates * 4.0 * rng.uniform(0.8, 1.2, size=(V, A))
    return bitrates, sizes


def _states(rng, A, H, V, n):
    """n sessions: random chunks, a quarter of them within H of the end of the video (h < H, and h <= 0 past it),
    last_q = -1 for a fifth, per-step predictions spread over a factor of 30."""
    chunk = np.where(rng.random(n) < 0.25, rng.integers(V - H, V + 1, size=n), rng.integers(0, V, size=n))
    prev_q = np.where(rng.random(n) < 0.2, -1, rng.integers(0, A, size=n))
    buffer = np.round(rng.uniform(0, 40, size=n), 9)
    pred = rng.uniform(0.2, 6.0, size=(n, H))
    return chunk.astype(np.int32), prev_q.astype(np.int32), buffer, pred


# (A, H, smooth_penalty, rebuf_penalty)
PENALTIES = [(1.0, 4.3), (0.6, 4.3), (2.5, 1.0), (0.0, 4.3), (1.0, 0.0), (0.0, 0.0)]
SHAPES = [(1, 4), (2, 5), (3, 4), (4, 3), (5, 3), (6, 2), (3, 1)]


@pytest.mark.parametrize("A,H", SHAPES, ids=[f"A{a}H{h}" for a, h in SHAPES])
def test_c_restatement_equals_python_restatement(A, H):
    V, n = 12, 80
    rng = np.random.default_rng(A * 100 + H)
    seen = dict(short=0, past=0, noprev=0, states=0)
    for vw, rw in PENALTIES:
        bitrates, sizes = _world(rng, A, V)
        chunk, prev_q, buffer, pred = _states(rng, A, H, V, n)
        L, B = 4.0, float(rng.choice([20.0, 60.0]))
        c = mp.decide_pred_c(sizes, bitrates, chunk, prev_q, buffer, pred, H, L, B, vw, rw)
        assert c["n_errors"] == 0
        for s in range(n):
            py = mp.decide_pred(int(chunk[s]), int(prev_q[s]), float(buffer[s]), pred[s], H, bitrates.tolist(),
                                sizes.tolist(), L, B, vw, rw)
            h = len(py["best_seq"])
            assert c["action"][s] == py["action"], s
            assert c["best_seq"][s].tolist() == py["best_seq"] + [-1] * (H - h), s
            assert bits_equal(c["best_J"][s], py["best_J"]) == 0, (s, c["best_J"][s], py["best_J"])
            seen["short"] += 0 < V - chunk[s] < H
            seen["past"] += chunk[s] >= V
            seen["noprev"] += prev_q[s] < 0
            seen["states"] += 1
    assert (seen["short"] or H == 1) and seen["past"] and seen["noprev"] and seen["states"] == 480


def test_constant_predictions_reproduce_the_robust_decision():
    """pred[i] = c for every i, c the robust prediction of SPEC §5.2: mpc_oracle.decide_robust's decision."""
    rng = np.random.default_rng(7)
    A, H, V = 4, 4, 10
    bitrates, sizes = _world(rng, A, V)
    U = bitrates.tolist()
    for trial in range(80):
        state = mo.RobustState(K=5)
        state.last_pred = float(rng.uniform(0.5, 4.0)) if trial % 3 else 0.0
        state.errs = list(rng.uniform(0, 0.4, size=int(rng.integers(0, 5))))
        hist = list(rng.uniform(0.3, 5.0, size=int(rng.integers(1, 9))))
        k, q, b = int(rng.integers(0, V)), int(rng.integers(-1, A)), float(rng.uniform(0, 30))
        r = mo.decide_robust(k, q, b, hist, state, H, U, sizes.tolist(), 4.0, 60.0, 1.0, 4.3)
        p = mp.decide_pred(k, q, b, [r["c"]] * H, H, U, sizes.tolist(), 4.0, 60.0, 1.0, 4.3)
        c = mp.decide_pred_c(sizes, bitrates, [k], [q], [b], [r["c"]] * H, H, 4.0, 60.0, 1.0, 4.3)
        assert p["action"] == r["action"] == c["action"][0]
        assert p["best_seq"] == r["best_seq"]
        if r["best_seq"]:
            assert bits_equal(p["best_J"], r["best_J"]) == 0 and bits_equal(c["best_J"][0], r["best_J"]) == 0


def test_huge_predictions_give_the_best_utility_minus_smoothness():
    rng = np.random.default_rng(3)
    A, H, V = 5, 3, 8
    bitrates, sizes = _world(rng, A, V)
    U = bitrates
    for q in (-1, 0, 2, 4):
        k = 2
        best = max(itertools.product(range(A), repeat=H),
                   key=lambda R: sum(U[k + i][R[i]] for i in range(H)) -
                   0.6 * sum(abs(U[k + i][R[i]] - U[k + i][([q] + list(R))[i]]) for i in range(H) if ([q] + list(R))[i] >= 0))
        r = mp.decide_pred_c(sizes, bitrates, [k], [q], [0.0], [1e12] * H, H, 4.0, 60.0, 0.6, 4.3)
        assert tuple(r["best_seq"][0]) == best


def test_tiny_predictions_give_the_lowest_quality():
    rng = np.random.default_rng(4)
    A, H, V = 6, 4, 9
    bitrates, sizes = _world(rng, A, V)
    r = mp.decide_pred_c(sizes, bitrates, [1, 3, 5], [5, -1, 2], [0.0, 10.0, 30.0], np.full((3, H), 1e-6), H, 4.0,
                         60.0, 1.0, 4.3)
    assert r["action"].tolist() == [0, 0, 0]
    assert (r["best_seq"] == 0).all()


def test_a_one_step_dip_reaches_the_search():
    """A dip in the second step's prediction changes the decision where a constant prediction at the mean of the
    steps does not: the search sees every step's own value."""
    bitrates = np.tile([1.0, 2.0, 4.0], (6, 1))
    sizes = bitrates * 4.0
    H, k, q, b = 3, 0, 2, 8.0
    dip = [3.0, 1.0, 3.0]
    flat = [sum(dip) / 3] * 3
    r_dip = mp.decide_pred_c(sizes, bitrates, [k], [q], [b], dip, H, 4.0, 60.0, 1.0, 4.3)
    r_flat = mp.decide_pred_c(sizes, bitrates, [k], [q], [b], flat, H, 4.0, 60.0, 1.0, 4.3)
    assert r_dip["best_seq"][0].tolist() != r_flat["best_seq"][0].tolist()
    assert r_dip["action"][0] != r_flat["action"][0]
    for r, p in ((r_dip, dip), (r_flat, flat)):
        py = mp.decide_pred(k, q, b, p, H, bitrates.tolist(), sizes.tolist(), 4.0, 60.0, 1.0, 4.3)
        assert r["best_seq"][0].tolist() == py["best_seq"]


@pytest.mark.parametrize("bad", [0.0, -1.0, math.nan, math.inf, -math.inf, -0.0])
def test_invalid_predictions_are_input_errors(bad):
    bitrates = np.tile([1.0, 2.0, 4.0], (6, 1))
    sizes = bitrates * 4.0
    H = 4
    pred = np.full((4, H), 2.0)
    pred[0, 1] = bad                 # h = 4: read
    pred[1, 3] = bad                 # chunk 4: h = 2, entry 3 is not read
    pred[2, 2] = bad                 # done: nothing is read
    pred[3, 0] = bad                 # chunk 6 = V: h = 0, nothing is read
    r = mp.decide_pred_c(sizes, bitrates, [0, 4, 1, 6], [1, 1, 1, 1], [5.0] * 4, pred, H, 4.0, 60.0, 1.0, 4.3,
                         done=[0, 0, 1, 0])
    assert r["action"].tolist()[0] == -1 and r["n_errors"] == 1
    assert r["action"][1] >= 0 and r["best_seq"][1].tolist()[2:] == [-1, -1]
    assert r["action"][2] == 0 and r["action"][3] == 0
    assert math.isnan(r["best_J"][0]) and math.isnan(r["best_J"][2]) and math.isnan(r["best_J"][3])
    assert (r["best_seq"][[0, 2, 3]] == -1).all()
    py = mp.decide_pred(0, 1, 5.0, pred[0], H, bitrates.tolist(), sizes.tolist(), 4.0, 60.0, 1.0, 4.3)
    assert py["action"] == -1 and py["error"]


def test_nan_past_the_truncated_horizon_is_ignored():
    bitrates = np.tile([1.0, 2.0, 4.0], (6, 1))
    sizes = bitrates * 4.0
    a = mp.decide_pred_c(sizes, bitrates, [3], [0], [5.0], [2.0, 3.0, 2.5, math.nan, math.nan], 5, 4.0, 60.0, 1.0, 4.3)
    b = mp.decide_pred_c(sizes, bitrates, [3], [0], [5.0], [2.0, 3.0, 2.5, 9.0, 9.0], 5, 4.0, 60.0, 1.0, 4.3)
    assert a["n_errors"] == 0 and a["action"][0] == b["action"][0]
    assert a["best_seq"].tolist() == b["best_seq"].tolist() and bits_equal(a["best_J"], b["best_J"]) == 0


def test_invalid_states_are_input_errors():
    bitrates = np.tile([1.0, 2.0, 4.0], (6, 1))
    sizes = bitrates * 4.0
    r = mp.decide_pred_c(sizes, bitrates, [-1, 2, 2], [0, 3, 2], [5.0] * 3, np.full((3, 2), 2.0), 2, 4.0, 60.0, 1.0,
                         4.3)
    assert r["action"].tolist()[:2] == [-1, -1] and r["action"][2] >= 0 and r["n_errors"] == 2
