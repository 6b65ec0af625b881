"""The CPU restatement of tree reuse (tests/mcts_reuse_oracle.py) against the pinned reference search."""
import numpy as np

from oracle import mcts_oracle as mo

from mcts_reuse_oracle import ReuseSearch, hash_predict, node_count, uniform_predict

PREDICT = {"hash": hash_predict, "uniform": uniform_predict}


def _all_nodes(node):
    out, stack = 0, [node]
    while stack:
        nd = stack.pop()
        out += 1
        stack.extend(nd.child_nodes or [])
    return out


def test_search_without_advance_is_the_reference_search(mcts_golden):
    cases = [c for c in mcts_golden["roots"] if c["sims"] == 50]
    assert len(cases) >= 8
    for case in cases:
        st = mo.COracleState(np.array(case["row"], np.uint8), case["plies"])
        rs = ReuseSearch(st)
        rs.search(PREDICT[case["evaluator"]], case["sims"])
        assert rs.counts() == case["visit_counts"]
        assert rs.counts() == mo.pv_mcts_scores(PREDICT[case["evaluator"]], st, case["sims"])
        assert node_count(rs.root) == _all_nodes(rs.root) <= 1 + case["sims"] * 133


def test_advance_keeps_the_visited_child_and_falls_back_to_a_fresh_root():
    rs = ReuseSearch(mo.COracleState())
    rs.search(hash_predict, 50)
    best = rs.actions()[int(np.argmax(rs.counts()))]
    child = rs.root.child_nodes[rs.actions().index(best)]
    n_child, size = child.n, node_count(child)
    assert n_child >= 1 and size > 1
    assert rs.advance([best], capacity=size, reserve=1) == 0          # one node short of room: fresh
    assert rs.root.n == 0 and rs.root.child_nodes is None
    rs = ReuseSearch(mo.COracleState())
    rs.search(hash_predict, 50)
    assert rs.advance([best], capacity=size + 5, reserve=5) == size   # just fits: carried
    assert rs.root.n == n_child and sum(rs.counts()) == n_child - 1
    rs.search(hash_predict, 50)
    assert sum(rs.counts()) == n_child + 50 - 1
    unvisited = [a for a, c in zip(rs.actions(), rs.counts()) if c == 0][0]
    assert rs.advance([unvisited], capacity=10 ** 6, reserve=0) == 0
