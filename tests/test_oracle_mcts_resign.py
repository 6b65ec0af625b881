"""Resignation's host logic without a GPU: the automatic threshold (self_play.resign_threshold_for) on hand-built records and the
calibration draw as tests/mcts_resign_oracle.py restates it (tests/test_gpu_mcts_resign.py compares the kernel's bits with it)."""
import math

import numpy as np
import pytest

from alphaquoridorgnn_b200 import self_play

import mcts_resign_oracle as mr

INF = math.inf


def record(games):
    """games: (flags, plies, resign_min pair, calibration) per game -> a record as play_batch_device returns it (numpy fields)."""
    return {"flags": np.array([g[0] for g in games], np.uint8), "plies": np.array([g[1] for g in games], np.int64),
            "resign_min": np.array([g[2] for g in games], np.float64), "calibration": np.array([g[3] for g in games], bool)}


def test_threshold_reads_the_sides_that_did_not_lose():
    rec = record([
        (1, 10, (-0.9, 0.2), True),    # plies even: the first player (column 0) lost -> the winner's minimum is column 1: 0.2
        (1, 7, (-0.3, -0.95), True),   # plies odd: the second player lost -> column 0: -0.3
        (2, 116, (-0.6, -0.1), True),  # draw: both sides -> -0.6
        (0, 40, (-0.2, -0.7), True),   # unfinished (max_plies): both sides -> -0.7
        (5, 3, (-1.0, -1.0), False),   # not a calibration game: ignored
    ])
    # m = [0.2, -0.3, -0.6, -0.7]; C = 4
    assert self_play.resign_threshold_for(rec, 0.0) == -0.7        # k = 0: the smallest m
    assert self_play.resign_threshold_for(rec, 0.25) == -0.6       # k = 1
    assert self_play.resign_threshold_for(rec, 0.49) == -0.6       # floor(1.96) = 1
    assert self_play.resign_threshold_for(rec, 0.5) == -0.3        # k = 2
    assert self_play.resign_threshold_for(rec, 0.75) == 0.2        # k = 3
    assert self_play.resign_threshold_for(rec, 1.0) == INF         # k = C


@pytest.mark.parametrize("mfp", [0.0, 0.05, 0.1, 0.2, 0.5, 0.99])
def test_threshold_is_the_largest_value_within_the_false_positive_rate(mfp):
    rng = np.random.default_rng(3)
    C = 60
    games = [(int(rng.choice([1, 2, 0])), int(rng.integers(1, 117)), tuple(np.round(rng.uniform(-1, 1, 2), 1)), True) for _ in range(C)]
    rec = record(games)
    v = self_play.resign_threshold_for(rec, mfp)
    m = []
    for f, p, r, _ in games:
        m.append(r[1 - p % 2] if f & 1 else min(r))
    m = np.array(m)
    assert (m < v).sum() / C <= mfp
    bigger = m[m > v]                 # the next larger candidate value already breaks the rate
    if bigger.size:
        assert (m < bigger.min()).sum() / C > mfp
    assert v in m                     # ties: the value is one of the m_c
    assert (m == v).sum() >= 1


def test_ties_count_once_each():
    rec = record([(2, 116, (-0.5, -0.5), True)] * 3 + [(2, 116, (0.1, 0.3), True)])
    assert self_play.resign_threshold_for(rec, 0.5) == -0.5      # k = 2: the third of three equal values
    assert self_play.resign_threshold_for(rec, 0.75) == 0.1


def test_threshold_needs_calibration_games_and_a_rate():
    rec = record([(1, 10, (-0.9, 0.2), False)])
    with pytest.raises(ValueError):
        self_play.resign_threshold_for(rec)
    rec = record([(1, 10, (-0.9, 0.2), True)])
    assert self_play.resign_threshold_for(rec, 0.05) == 0.2
    for bad in (-0.1, 1.5, float("nan")):
        with pytest.raises(ValueError):
            self_play.resign_threshold_for(rec, bad)


@pytest.mark.parametrize("p", [0.1, 0.5])
def test_calibration_fraction_is_within_binomial_bounds(p):
    N = 10 ** 5
    for seed in (7, 12345):
        k = int(mr.is_calibration(seed, np.arange(N), p).sum())
        assert abs(k - N * p) <= 5 * math.sqrt(N * p * (1 - p)), (seed, k)


def test_calibration_depends_on_seed_and_game_id_alone():
    ids = np.arange(20000)
    u = mr.calibration_u(99, ids)
    assert np.array_equal(mr.calibration_u(99, ids[::-1]), u[::-1])               # row order plays no part
    assert np.array_equal(mr.calibration_u(99, ids[5000:7000]), u[5000:7000])     # nor the batch it is drawn in
    assert np.array_equal(mr.is_calibration(99, ids[:300], 0.1), mr.is_calibration(99, ids, 0.1)[:300])
    assert (u >= 0).all() and (u < 1).all()
    a, b = mr.is_calibration(99, ids, 0.5), mr.is_calibration(100, ids, 0.5)      # another seed: an independent draw
    both = int((a & b).sum())
    assert abs(both - 5000) <= 5 * math.sqrt(20000 * 0.25 * 0.75)
    assert not mr.is_calibration(99, ids, 0.0).any() and mr.is_calibration(99, ids, 1.0).all()
