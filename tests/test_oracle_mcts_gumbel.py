"""The CPU restatement of the Gumbel root (tests/mcts_gumbel_oracle.py): mctx's sequential-halving table, the counter-based Gumbel
draw keyed by (seed, game id, ply), and the improved policy of a Gumbel search."""
import numpy as np
import pytest
from scipy import stats

from oracle import mcts_oracle as mo

import mcts_gumbel_oracle as mg
from mcts_reuse_oracle import hash_predict, uniform_predict


def test_considered_visits_table_hand_values():
    assert mg.sequence_of_considered_visits(4, 8) == (0, 0, 0, 0, 1, 1, 2, 2)
    seq = mg.sequence_of_considered_visits(16, 200)
    assert len(seq) == 200
    assert seq[:16] == (0,) * 16 and seq[16] == 1
    assert seq[-6:] == (46, 46, 47, 47, 48, 48)
    for m in (0, 1):
        assert mg.sequence_of_considered_visits(m, 7) == tuple(range(7))


@pytest.mark.parametrize("m", [1, 2, 3, 4, 5, 16, 17, 64, 133, 136])
def test_kernel_formula_is_the_table(m):
    """considered_visit(m, n, k) computes the table without building it; the lengths of the table are n."""
    for n in (0, 1, 2, 3, 7, 15, 16, 31, 49, 63, 199, 200, 511):
        seq = mg.sequence_of_considered_visits(m, n)
        assert len(seq) == n
        assert [mg.considered_visit(m, n, k) for k in range(n)] == list(seq), (m, n)


def test_gumbel_draws_are_standard_gumbel():
    g = mg.gumbel_draw(2024, np.arange(4000), 5, 40).ravel()
    assert np.isfinite(g).all()
    assert stats.kstest(g, stats.gumbel_r.cdf).pvalue > 1e-3
    u = mg.gumbel_uniform(2024, np.arange(4000), 5, 40)
    assert (u > 0).all() and (u < 1).all()
    assert np.array_equal(mg.gumbel_draw(1, [3], 0, 10, 0.0), np.zeros((1, 10)))
    assert np.allclose(mg.gumbel_draw(1, [3], 0, 10, 0.5), 0.5 * mg.gumbel_draw(1, [3], 0, 10), rtol=1e-7)


def test_draw_depends_on_game_ply_and_seed_only():
    base = mg.gumbel_draw(1, [4, 9], 6, 40)
    assert np.array_equal(base[1], mg.gumbel_draw(1, [9], 6, 40)[0])       # not on the other games or the row
    assert np.array_equal(base[1, :20], mg.gumbel_draw(1, [9], 6, 20)[0])  # nor on the number of children
    assert not np.array_equal(base[0], base[1])
    assert not np.array_equal(base[0], mg.gumbel_draw(1, [4], 7, 40)[0])
    assert not np.array_equal(base[0], mg.gumbel_draw(2, [4], 6, 40)[0])
    # its own domain: not the uniforms of the root noise
    import mcts_noise_oracle as mn
    assert not np.array_equal(mg.gumbel_key(1, [4], 6), mn.noise_key(1, [4], 6))


@pytest.mark.parametrize("predict", [hash_predict, uniform_predict])
@pytest.mark.parametrize("considered,sims", [(1, 1), (2, 2), (4, 16), (16, 50), (200, 50)])
def test_gumbel_search_budget_and_improved_policy(mcts_golden, predict, considered, sims):
    states = [mo.COracleState()] + [mo.COracleState(np.array(c["row"], np.uint8), c["plies"]) for c in mcts_golden["roots"]
                                    if c["sims"] == 50 and c["evaluator"] == "hash"][:3]
    for gid, s in enumerate(states):
        o = mg.GumbelSearch(s, considered)
        o.search(predict, sims, seed=11, game_id=gid, ply=3)
        n = o.counts()
        K = len(n)
        assert sum(n) == sims - 1
        m = min(considered, K)
        assert sum(1 for v in n if v) <= m
        pol, choice = o.result()
        assert pol.shape == (K,) and (pol >= 0).all() and abs(pol.sum() - 1.0) < 1e-12
        assert n[choice] == max(n)


def test_scale_zero_is_deterministic_and_seed_independent():
    s = mo.COracleState()
    runs = []
    for seed in (1, 2, 3):
        o = mg.GumbelSearch(s, 4, scale=0.0)
        o.search(hash_predict, 16, seed=seed, game_id=seed, ply=seed)
        runs.append((o.counts(), o.result()[1]))
    assert runs[0] == runs[1] == runs[2]
