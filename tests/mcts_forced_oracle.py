"""CPU restatement of forced playouts and policy target pruning (KataGo: David J. Wu, "Accelerating Self-Play Learning in Go",
2019), on top of the noised, reusable search of tests/mcts_noise_oracle.py.  The reference has neither.

For a root whose children have priors P_c (np.float32, noised if the root was), visits n_c and value sums w_c, t = sum n_c and
k = float32(forced_k) widened to a Python float:
  n_forced(c) = sqrt(k * P_c * t)                                                  (float64, left to right)
  PUCT(c, m)  = float32(-w_c / n_c) + ((float32(1.25) * P_c) * float32(sqrt(t))) / float32(1 + m)      (float32; Q is 0 when n_c = 0)
  root rule   : the first child with n_c >= 1 and n_c < n_forced(c), else np.argmax of PUCT(c, n_c); PUCT below the root
  pruning     : c* = the first child with the largest n keeps n_c*; any other child with n_c >= 1 starts from m = n_c and, while
                m >= 1, m - 1 >= n_c - n_forced(c) and PUCT(c, m - 1) < PUCT(c*, n_c*), loses one; reduced and m <= 1 -> 0
as aq_mcts_select_forced and aq_mcts_root_counts_pruned (csrc/mcts.cu) compute them.
"""
import math

import numpy as np

from oracle import mcts_oracle as mo

import mcts_resign_oracle as mr
from mcts_noise_oracle import NoisedSearch

C_PUCT = np.float32(mo.C_PUCT)


def n_forced(k, p, t):
    return math.sqrt(float(np.float32(k)) * float(p) * float(t))


def puct(c, t, m):
    """The select score of child c (an oracle node: w, n, p) with the visit count of U replaced by m, in float32."""
    q = np.float32(-c.w / c.n) if c.n else np.float32(0.0)
    return np.float32(q + np.float32(np.float32(C_PUCT * np.float32(c.p)) * np.float32(math.sqrt(t))) / np.float32(1 + m))


def forced_child(children, k):
    """Index of the first visited child below its n_forced, or None."""
    t = sum(c.n for c in children)
    for i, c in enumerate(children):
        if c.n >= 1 and c.n < n_forced(k, c.p, t):
            return i
    return None


def root_child(children, k):
    """The child the forced select takes at the root."""
    f = forced_child(children, k)
    if f is not None:
        return f
    t = sum(c.n for c in children)
    return int(np.argmax([puct(c, t, c.n) for c in children]))


def pruned_counts(children, k):
    """The counts aq_mcts_root_counts_pruned writes for a root with these children."""
    if not children:
        return []
    t = sum(c.n for c in children)
    b = int(np.argmax([c.n for c in children]))
    best = puct(children[b], t, children[b].n)
    out = []
    for i, c in enumerate(children):
        m = c.n
        if i != b and c.n >= 1:
            floor_n = float(c.n) - n_forced(k, c.p, t)
            while m >= 1 and float(m - 1) >= floor_n and puct(c, t, m - 1) < best:
                m -= 1
            if m < c.n and m <= 1:
                m = 0
        out.append(m)
    return out


def node(w, n, p):
    """A hand-built root child."""
    c = mo._Node(None, np.float32(p))
    c.w, c.n = w, n
    return c


class ForcedSearch(NoisedSearch):
    """NoisedSearch (no noise when alpha is None) whose root descents follow the forced-playout rule."""

    def __init__(self, state, k, alpha=None, fraction=0.25):
        super().__init__(state, alpha, fraction)
        self.k = k

    def noise(self, seed, game_id, ply):
        if self.alpha is not None:
            super().noise(seed, game_id, ply)

    def simulate(self, predict):
        root = self.root
        if root.state.is_done() or not root.child_nodes:
            root.evaluate(predict)
            return
        value = -root.child_nodes[root_child(root.child_nodes, self.k)].evaluate(predict)
        root.w += value
        root.n += 1

    def search(self, predict, sims, seed=0, game_id=0, ply=0):
        self.noise(seed, game_id, ply)
        for i in range(sims):
            self.simulate(predict)
            if i == 0:
                self.noise(seed, game_id, ply)

    def pruned(self):
        return pruned_counts(self.root.child_nodes or [], self.k)


def play_game(predict, sims, seed, g, k, temperature=0, reuse=False, alpha=None, v_resign=None, calibration=0.0):
    """One self-play game with forced searches: the move and the recorded policy come from the pruned counts (temperature 0: the
    first most visited child; 1: mcts_resign_oracle.move_draw).  With v_resign, the resignation of mcts_resign_oracle.play_game,
    its statistic read from the unpruned tree.  -> dict(states [(row, plies)], policy [dense 209], value, flags, plies, resign_min)."""
    cal = bool(mr.is_calibration(seed, [g], calibration)[0])
    capacity, reserve = 1 + 2 * sims * mr.MAX_CHILDREN, sims * mr.MAX_CHILDREN
    o = ForcedSearch(mo.COracleState(), k, alpha)
    rmin, seen, pols, ply, flags = [math.inf, math.inf], [], [], 0, None
    while not o.root.state.is_done():
        s = o.root.state
        seen.append((s.row.tolist(), s.plies))
        o.search(predict, sims, seed, g, ply)
        stat = mr.statistic(o.root)
        if not math.isnan(stat):
            rmin[ply & 1] = min(rmin[ply & 1], stat)
        c = np.array(o.pruned(), np.float64)
        dense = np.zeros(209)
        if temperature == 0:
            i = int(np.argmax(c))
            dense[o.actions()[i]] = 1.0
        else:
            dense[o.actions()] = c / c.sum()
            i = mr.move_draw(c, seed, g, ply)
        a = o.actions()[i]
        pols.append(dense)
        if v_resign is not None and not cal and stat < v_resign:
            flags = 1 | 4
            break
        if reuse:
            o.advance([a], capacity, reserve)
        else:
            o = ForcedSearch(s.next(a), k, alpha)
        ply += 1
    if flags is None:
        end = o.root.state
        flags = 1 if end.is_lose() else (2 if end.is_draw() else 0)
    fpv = (-1.0 if ply % 2 == 0 else 1.0) if flags & 1 else 0.0
    return {"states": seen, "policy": pols, "value": [fpv if j % 2 == 0 else -fpv for j in range(len(seen))], "flags": flags,
            "plies": ply, "resign_min": rmin}
