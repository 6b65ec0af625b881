"""CPU restatement of tree reuse between moves (AlphaGo Zero), on top of the reference-literal search of oracle/mcts_oracle.py.

The reference builds a fresh root for every move (pv_mcts.py:81).  Reuse is what keeping the child object means in the
reference's own Node class: after the move, the played child becomes the root and keeps its w, n, p and child_nodes.
``ReuseSearch`` states that, plus the arena rule of the GPU (aq_mcts_advance): a subtree is kept only when it was visited and
its node count leaves `reserve` nodes of room in an arena of `capacity` nodes.
"""
import numpy as np

from oracle import mcts_oracle as mo


def hash_predict(state):
    """The hash evaluator of tests/golden/make_golden.py, as tests/test_oracle_golden.py states it for the oracle."""
    r = [int(v) for v in state.row]
    key = (sum(v * (i + 1) * 7919 for i, v in enumerate(r)) + state.plies_played * 104729) % (2 ** 31)
    la = state.legal_actions()
    raw = np.array([(key + a * 40503) % 1009 + 1 for a in la], dtype=np.int64)
    return raw.astype(np.float32) / np.float32(raw.sum()), float(np.float32((key % 2001) - 1000) / np.float32(1000))


def uniform_predict(state):
    la = state.legal_actions()
    return np.full(len(la), 1.0 / len(la), dtype=np.float32), 0.0


def node_count(node):
    """Arena nodes of a subtree: the node itself plus one per child of every expanded node."""
    total, stack = 1, [node]
    while stack:
        nd = stack.pop()
        if nd.child_nodes:
            total += len(nd.child_nodes)
            stack.extend(nd.child_nodes)
    return total


class ReuseSearch:
    def __init__(self, state):
        self.root = mo._Node(state, 0)

    def search(self, predict, sims):
        for _ in range(sims):
            self.root.evaluate(predict)

    def counts(self):
        return [c.n for c in self.root.child_nodes] if self.root.child_nodes else []

    def actions(self):
        return self.root.state.legal_actions() if self.root.child_nodes else []

    def advance(self, path, capacity, reserve):
        """Follow `path` (actions) from the root; keep the node reached when it was visited and its subtree has at most
        capacity - reserve nodes, else start from a fresh root at the same position.  -> nodes carried (0 = fresh)."""
        node, state = self.root, self.root.state
        for a in path:
            state = state.next(a)
            if node is not None:
                la = node.state.legal_actions()
                node = node.child_nodes[la.index(a)] if node.child_nodes and a in la else None
        if node is not None and node.n >= 1 and node_count(node) <= capacity - reserve:
            self.root = node
            return node_count(node)
        self.root = mo._Node(state, 0)
        return 0
