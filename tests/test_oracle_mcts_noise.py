"""The CPU restatement of root Dirichlet noise (tests/mcts_noise_oracle.py): the counter-based sampler draws Dirichlet(alpha)
vectors, keyed by (seed, game id, ply), and the noised search is the plain search when the noise has no weight."""
import numpy as np
import pytest
from scipy import stats

from oracle import mcts_oracle as mo

import mcts_noise_oracle as mn
from mcts_reuse_oracle import ReuseSearch, hash_predict

N = 20000


@pytest.mark.parametrize("alpha", [0.03, 0.3, 1.0, 2.5])
@pytest.mark.parametrize("K", [2, 5, 133])
def test_sampler_is_dirichlet(alpha, K):
    eta = mn.dirichlet(12345, np.arange(N), 3, K, alpha)
    assert eta.shape == (N, K)
    assert not np.isnan(eta).any() and (eta >= 0).all()
    assert np.abs(eta.sum(1) - 1.0).max() < 1e-12
    a = float(np.float32(alpha))
    # each coordinate has mean 1/K and variance (1/K)(1 - 1/K)/(K a + 1)
    sd = np.sqrt((1 / K) * (1 - 1 / K) / (K * a + 1)) / np.sqrt(N)
    assert np.abs(eta.mean(0) - 1 / K).max() < 5 * sd
    # one marginal against Beta(a, (K - 1) a), through its CDF.  At small a a sixth of the draws of a coordinate lie within 2^-53
    # of 1, where doubles cannot tell them apart: above 1/2 the CDF is taken as the survival function of the other coordinates'
    # sum, which is Beta((K - 1) a, a) and resolved there.
    for c in (0, K - 1):
        x, rest = eta[:, c], np.delete(eta, c, axis=1).sum(1)
        u = np.where(x <= 0.5, stats.beta(a, (K - 1) * a).cdf(x), stats.beta((K - 1) * a, a).sf(rest))
        p = stats.kstest(u, "uniform").pvalue
        assert p > 1e-3, (alpha, K, c, p)


def test_small_alpha_is_computed_in_logs():
    """At alpha = 0.03 the gamma variates span hundreds of orders of magnitude: for some draws every one of them is below the
    float32 range.  The draw works in logs with the maximum subtracted, so eta is exact there too."""
    key = mn.noise_key(7, np.arange(N), 0)
    lg = mn.log_gamma(key, 2, 0.03)
    tiny = lg.max(1) < np.log(np.finfo(np.float32).tiny)
    assert tiny.sum() > 20
    eta = mn.dirichlet(7, np.arange(N), 0, 2, 0.03)
    assert np.isfinite(eta).all() and np.abs(eta.sum(1) - 1).max() < 1e-12
    assert (eta[tiny].max(1) >= 0.5).all()


def test_draw_depends_on_game_ply_and_seed_only():
    base = mn.dirichlet(1, [4, 9], 6, 40, 0.3)
    assert np.array_equal(base[1], mn.dirichlet(1, [9], 6, 40, 0.3)[0])   # not on the other games or the row
    assert not np.array_equal(base[0], base[1])                             # game id
    assert not np.array_equal(base[0], mn.dirichlet(1, [4], 7, 40, 0.3)[0])  # ply
    assert not np.array_equal(base[0], mn.dirichlet(2, [4], 6, 40, 0.3)[0])  # seed
    assert len({tuple(r) for r in mn.dirichlet(1, np.arange(64), 0, 5, 0.3)}) == 64


def test_warp_order_sum_is_a_sum():
    e = np.random.default_rng(0).random((50, 133))
    assert np.allclose(mn.warp_sum(e), e.sum(1), rtol=1e-14)


def test_zero_fraction_keeps_the_priors_and_the_search(mcts_golden):
    p = np.array([0.1, 0.2, 0.7], np.float32)
    eta = mn.dirichlet(3, [0], 0, 3, 0.3)[0]
    assert np.array_equal(mn.noised_priors(p, eta, 0.0), p)
    assert np.array_equal(mn.noised_priors(p, eta, 1.0), eta.astype(np.float32))
    for c in [r for r in mcts_golden["roots"] if r["sims"] == 50 and r["evaluator"] == "hash"][:3]:
        s = mo.COracleState(np.array(c["row"], np.uint8), c["plies"])
        plain = ReuseSearch(s)
        plain.search(hash_predict, 50)
        zero = mn.NoisedSearch(s, 0.3, 0.0)
        zero.search(hash_predict, 50, seed=5, game_id=1, ply=0)
        noised = mn.NoisedSearch(s, 0.3, 0.25)
        noised.search(hash_predict, 50, seed=5, game_id=1, ply=0)
        assert zero.counts() == plain.counts() == c["visit_counts"]
        assert noised.noised and sum(noised.counts()) == 49


def test_noise_is_applied_once_per_root():
    s = mo.COracleState()
    o = mn.NoisedSearch(s, 0.3)
    o.noise(1, 0, 0)
    assert not o.noised                         # a fresh root has no children to noise before simulation 1
    o.root.evaluate(hash_predict)
    o.noise(1, 0, 0)
    first = [c.p for c in o.root.child_nodes]
    assert all(isinstance(p, np.float32) for p in first)
    o.noise(2, 0, 0)
    assert [c.p for c in o.root.child_nodes] == first
    raw, _ = hash_predict(s)
    eta = mn.dirichlet(1, [0], 0, len(raw), 0.3)[0]
    assert np.array_equal(np.array(first, np.float32), mn.noised_priors(raw, eta, 0.25))
