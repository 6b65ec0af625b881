"""The CPU restatement of playout cap randomization (tests/mcts_pcr_oracle.py): the full/fast draw, its rate, its independence of
the other draws, and the self-play game at the edge probabilities."""
import math

import numpy as np
import pytest

import mcts_forced_oracle as mf
import mcts_pcr_oracle as mp
import mcts_resign_oracle as mr
from mcts_noise_oracle import noise_key
from mcts_reuse_oracle import hash_predict

M64 = (1 << 64) - 1


def mix64_int(z):
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def test_draw_restated_in_integers():
    """The numpy draw against the formula in Python integers, for keys that wrap every sum and product."""
    for seed in (0, 1, 12345, M64, 2 ** 63 + 7):
        for g in (0, 1, 77, 2 ** 40 + 3):
            for ply in (0, 1, 5, 199, 2 ** 20):
                key = mix64_int((mix64_int(((seed ^ mp.PCR_DOMAIN) + 0x9E3779B97F4A7C15 * (g + 1)) & M64) + 0xD1B54A32D192ED03 * (ply + 1)) & M64)
                assert mp.full_u(seed, [g], ply)[0] == (key >> 11) * 2.0 ** -53, (seed, g, ply)


def test_domain_is_the_next_digits_of_pi_after_resignation():
    # pi = 3.243F6A88 85A308D3 13198A2E 03707344 A4093822 299F31D0 082EFA98 EC4E6C89 ...
    assert (mr.RESIGN_DOMAIN, mp.PCR_DOMAIN) == (0xA4093822299F31D0, 0x082EFA98EC4E6C89)


@pytest.mark.parametrize("p", [0.1, 0.25, 0.5])
def test_full_fraction_is_within_binomial_bounds(p):
    """100,000 (seed, game, ply) keys: the number of full moves is within 5 standard deviations of n p."""
    g, ply = np.meshgrid(np.arange(500), np.arange(200), indexing="ij")
    hits = sum(int(mp.is_full(seed, g.ravel(), ply.ravel(), p).sum()) for seed in (3, 2 ** 61 + 5))
    n = 2 * g.size
    assert abs(hits - n * p) <= 5 * math.sqrt(n * p * (1 - p)), (hits, n * p)


def test_edge_probabilities_and_independence_of_other_draws():
    g, ply = np.meshgrid(np.arange(300), np.arange(100), indexing="ij")
    g, ply = g.ravel(), ply.ravel()
    u = mp.full_u(9, g, ply)
    assert u.min() >= 0.0 and u.max() < 1.0
    assert not mp.is_full(9, g, ply, 0.0).any() and mp.is_full(9, g, ply, 1.0).all()
    # the full draw is not the noise key's nor the calibration draw's
    assert not np.array_equal(u, (noise_key(9, g, 0) >> np.uint64(11)).astype(np.float64) * 2.0 ** -53)
    full = mp.is_full(9, g, ply, 0.5)
    cal = np.repeat(mr.is_calibration(9, np.arange(300), 0.5), 100)
    assert abs(np.mean(full == cal) - 0.5) < 0.02


def test_partition_is_stable():
    gid = np.arange(1000) * 3 + 11
    out_row, full = mp.partition(4, gid, 6, 0.3)
    f = mp.is_full(4, gid, 6, 0.3)
    assert sorted(out_row.tolist()) == list(range(1000)) and full == int(f.sum())
    assert f[out_row[:full]].all() and not f[out_row[full:]].any()
    assert (np.diff(out_row[:full]) > 0).all() and (np.diff(out_row[full:]) > 0).all()


@pytest.mark.parametrize("kw", [dict(temperature=0, k=2.0), dict(temperature=1.0, alpha=0.3, k=2.0, reuse=True),
                                dict(temperature=1.0, alpha=0.3)])
def test_all_full_is_the_game_without_pcr(kw):
    sims, seed, g = 8, 5, 3
    o = mp.play_game(hash_predict, sims, 2, 1.0, seed, g, **kw)
    ref = mf.play_game(hash_predict, sims, seed, g, kw.get("k") or 0.0, temperature=kw["temperature"], reuse=kw.get("reuse", False),
                       alpha=kw.get("alpha"))
    assert o["states"] == ref["states"] and o["value"] == ref["value"]
    assert all(np.array_equal(a, b) for a, b in zip(o["policy"], ref["policy"])) and len(o["policy"]) == len(ref["policy"])
    assert (o["flags"], o["plies"], o["ply"], o["fast"]) == (ref["flags"], ref["plies"], list(range(ref["plies"])), 0)


def test_no_full_move_records_nothing_and_plays_the_fast_game():
    sims, fast, seed, g = 8, 3, 5, 2
    o = mp.play_game(hash_predict, sims, fast, 0.0, seed, g, temperature=1.0, alpha=0.3, k=2.0)
    ref = mf.play_game(hash_predict, fast, seed, g, 2.0, temperature=1.0)
    assert o["states"] == [] and o["policy"] == [] and o["full"] == 0
    assert (o["flags"], o["plies"], o["fast"]) == (ref["flags"], ref["plies"], ref["plies"])


def test_mixed_game_records_the_full_plies_of_its_draw():
    sims, fast, seed, g, p = 8, 2, 13, 4, 0.4
    o = mp.play_game(hash_predict, sims, fast, p, seed, g, temperature=1.0, alpha=0.3, k=2.0, reuse=True)
    want = [j for j in range(o["plies"]) if mp.is_full(seed, [g], j, p)[0]]
    assert o["ply"] == want and o["full"] == len(want) and o["full"] + o["fast"] == o["plies"]
    assert [s[1] for s in o["states"]] == want   # a position's plies-played is its ply from the start position
