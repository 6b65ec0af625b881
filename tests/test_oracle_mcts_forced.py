"""The CPU restatement of forced playouts and policy target pruning (tests/mcts_forced_oracle.py): k = 0 is the reference search,
pruning keeps the most visited child and removes only forced visits that PUCT would not have made, and the root rule forces the
first visited child below its n_forced."""
import math

import numpy as np
import pytest

from oracle import mcts_oracle as mo

import mcts_forced_oracle as mf
from mcts_reuse_oracle import hash_predict, uniform_predict

PREDICT = {"hash": hash_predict, "uniform": uniform_predict}


def test_zero_k_is_the_reference_search(mcts_golden):
    """On the roots of mcts_golden.json, whose counts come from the unmodified reference: k = 0 searches the same tree, and pruning
    at k = 0 leaves the counts as they are."""
    for case in mcts_golden["roots"]:
        o = mf.ForcedSearch(mo.COracleState(np.array(case["row"], np.uint8), case["plies"]), 0.0)
        o.search(PREDICT[case["evaluator"]], case["sims"])
        assert o.counts() == case["visit_counts"], case["sims"]
        assert o.pruned() == o.counts()


def random_root(rng, K):
    """Hand-built root children: visits with a few dominant ones, values in [-1, 1] per visit, priors summing to 1 in float32."""
    n = rng.geometric(rng.uniform(0.05, 0.6), K) - 1
    n[rng.integers(K)] += rng.integers(5, 200)
    p = rng.dirichlet(np.full(K, rng.uniform(0.1, 2.0))).astype(np.float32)
    return [mf.node(float(rng.uniform(-1, 1) * v), int(v), p[i]) for i, v in enumerate(n)]


@pytest.mark.parametrize("k", [0.5, 2.0, 8.0])
def test_pruning_properties_on_hand_built_roots(k):
    rng = np.random.default_rng(int(k * 10))
    reduced = zeroed = 0
    for _ in range(400):
        ch = random_root(rng, int(rng.integers(2, 134)))
        before = [c.n for c in ch]
        after = mf.pruned_counts(ch, k)
        t = sum(before)
        b = int(np.argmax(before))
        best = mf.puct(ch[b], t, ch[b].n)
        assert after[b] == before[b] and int(np.argmax(after)) == b        # c* keeps its count, so it stays the first maximum
        for c, n0, n1 in zip(ch, before, after):
            assert 0 <= n1 <= n0                                          # no count rises
            assert n0 - n1 <= math.ceil(mf.n_forced(k, c.p, t))           # none falls by more than ceil(n_forced)
            if 1 < n1 < n0:
                assert mf.puct(c, t, n1) < best                           # a reduced child's PUCT stays below c*'s
            assert n1 != 1 or n0 == 1                                     # a child reduced to one visit goes to 0
            reduced += n1 < n0
            zeroed += n1 == 0 < n0
    assert reduced > 100 and zeroed > 20


def test_pruning_worked_example():
    """t = 100, k = 2, c* = child 0 with PUCT 0.687.  Child 1 (P 0.5, n 12, Q -0.83) has n_forced = 10, but PUCT(1, 3) = 0.729 is
    above c*'s: it keeps 4.  Child 2 (P 0.125, n 6, n_forced 5) may lose 5 and PUCT stays below c*'s down to one visit, so it
    goes to 0.  Child 3 has a Q so high that PUCT wants every visit: it keeps them."""
    ch = [mf.node(-50.0, 80, 0.4), mf.node(10.0, 12, 0.5), mf.node(2.0, 6, 0.125), mf.node(-2.0, 2, 0.08)]
    assert [round(mf.n_forced(2.0, c.p, 100), 3) for c in ch] == [8.944, 10.0, 5.0, 4.0]
    assert mf.pruned_counts(ch, 2.0) == [80, 4, 0, 2]
    assert mf.pruned_counts(ch, 0.0) == [80, 12, 6, 2]


def test_ties_for_the_most_visited_child_resolve_to_the_first():
    ch = [mf.node(0.0, 1, 0.1), mf.node(-9.0, 30, 0.3), mf.node(9.0, 30, 0.3), mf.node(9.0, 30, 0.3)]
    out = mf.pruned_counts(ch, 8.0)
    assert out[1] == 30 and out[2] < 30 and out[3] < 30


def test_the_root_rule_forces_a_visited_child_over_a_larger_puct_score():
    # t = 100: child 0 (P 0.5) needs 10 forced visits at k = 2 and has 3; child 1 has the larger PUCT score
    ch = [mf.node(3.0, 3, 0.5), mf.node(-60.0, 97, 0.5)]   # Q = -1 for child 0, +0.62 for child 1: PUCT prefers child 1 ...
    assert mf.puct(ch[0], 100, 3) < mf.puct(ch[1], 100, 97)
    assert mf.forced_child(ch, 2.0) == 0 and mf.root_child(ch, 2.0) == 0   # ... and the rule still takes child 0
    assert mf.root_child(ch, 0.0) == 1


def test_the_root_rule_takes_the_first_of_several_forced_children():
    ch = [mf.node(0.0, 50, 0.1), mf.node(2.0, 2, 0.3), mf.node(-1.0, 1, 0.3), mf.node(0.0, 47, 0.3)]
    assert mf.forced_child(ch, 2.0) == 1
    ch[1].n = 20
    assert mf.forced_child(ch, 2.0) == 2


def test_an_unvisited_child_is_never_forced():
    ch = [mf.node(0.0, 0, 0.9), mf.node(-50.0, 60, 0.05), mf.node(-30.0, 40, 0.05)]
    assert mf.forced_child(ch, 100.0) is None
    assert mf.root_child(ch, 100.0) == 0   # PUCT takes it, as it would without forcing
    assert mf.pruned_counts(ch, 100.0)[0] == 0


@pytest.mark.parametrize("name", ["hash", "uniform"])
def test_forced_search_spends_the_forced_visits_and_pruning_removes_them(mcts_golden, name):
    """At k = 2 the pruned counts keep the most visited child.  With the hash evaluator the search differs from the plain one and
    the pruning removes visits; with the uniform one (equal priors, all values 0) PUCT already spreads the visits, so it need not."""
    cases = [c for c in mcts_golden["roots"] if c["sims"] == 200 and c["evaluator"] == name]
    removed = changed = 0
    for case in cases:
        s = mo.COracleState(np.array(case["row"], np.uint8), case["plies"])
        o = mf.ForcedSearch(s, 2.0)
        o.search(PREDICT[name], 200)
        counts, pruned = o.counts(), o.pruned()
        assert sum(counts) == 199 and int(np.argmax(pruned)) == int(np.argmax(counts))
        changed += counts != case["visit_counts"]
        removed += sum(counts) - sum(pruned)
    if name == "hash":
        assert removed > 0 and changed > 0
