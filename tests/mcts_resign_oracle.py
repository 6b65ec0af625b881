"""CPU restatement of resignation in self-play (AlphaGo Zero), on top of the search oracles of tests/mcts_reuse_oracle.py,
tests/mcts_noise_oracle.py and tests/mcts_gumbel_oracle.py.  The reference has none.

  root_value  = w / n of the root (NaN if n == 0), best child b = the first most visited child, best_q = -(w_b / n_b) (-inf if
                n_b == 0 or there are no children): aq_mcts_root_values, from the oracle tree's own float64 w and n
  s           = max(root_value, best_q), NaN if either is (np.maximum)
  calibration = u < calibration with u = (mix64(mix64((seed ^ RESIGN_DOMAIN) + GOLDEN * (game_id + 1))) >> 11) * 2^-53
  a game resigns at its ply when it is not a calibration game and s < v_resign: its position and policy are recorded, no move is
  played, flags = 1 | 4 and plies = the moves played; resign_min[ply & 1] = min(itself, s) at every ply (NaN s: unchanged).
"""
import math

import numpy as np

from oracle import mcts_oracle as mo

import mcts_gumbel_oracle as mg
from mcts_noise_oracle import GOLDEN, M64, PLY_MUL, NoisedSearch, mix64
from mcts_reuse_oracle import ReuseSearch

RESIGN_DOMAIN = 0xA4093822299F31D0
MAX_CHILDREN = 133


def root_values(root):
    """(root_value, best_q, best child index or -1) of an oracle root (mo._Node)."""
    rv = root.w / root.n if root.n else math.nan
    ch = root.child_nodes or []
    if not ch:
        return rv, -math.inf, -1
    b = int(np.argmax([c.n for c in ch]))
    return rv, (-(ch[b].w / ch[b].n) if ch[b].n else -math.inf), b


def statistic(root):
    rv, bq, _ = root_values(root)
    return float(np.maximum(rv, bq))


def calibration_u(seed, game_id):
    """u in [0, 1) of games game_id (int array): float64 [N]."""
    gid = np.asarray(game_id, dtype=np.int64).astype(np.uint64)
    with np.errstate(over="ignore"):
        z = mix64(mix64(np.uint64((int(seed) ^ RESIGN_DOMAIN) & M64) + np.uint64(GOLDEN) * (gid + np.uint64(1))))
    return (z >> np.uint64(11)).astype(np.float64) * 2.0 ** -53


def is_calibration(seed, game_id, calibration):
    return calibration_u(seed, game_id) < calibration


def move_draw(counts, seed, game_id, ply):
    """The child aq_selfplay_advance draws at temperature 1: the first child with a positive count whose running sum exceeds
    u * total, u = (mix64(mix64(seed + GOLDEN * (game_id + 1)) + PLY_MUL * (ply + 1)) >> 11) * 2^-53 (integer sums are exact)."""
    with np.errstate(over="ignore"):
        z = mix64(mix64(np.uint64(int(seed) & M64) + np.uint64(GOLDEN) * np.uint64(game_id + 1)) + np.uint64(PLY_MUL * (ply + 1) & M64))
    c = np.asarray(counts, np.float64)
    cum = np.cumsum(c)
    target = float(z >> np.uint64(11)) * 2.0 ** -53 * cum[-1]
    over = np.nonzero((c > 0) & (target < cum))[0]
    return int(over[0]) if over.size else int(np.nonzero(c > 0)[0][-1])


def play_game(predict, sims, seed, g, v_resign, calibration, temperature=0, reuse=False, alpha=None, considered=None, max_plies=None):
    """One self-play game with resignation.  The move of a PUCT search is the first most visited child (temperature 0) or, at
    temperature 1, the child move_draw picks (the recorded policy is counts / sum).  A Gumbel search (considered) plays its choice
    and records its improved policy.  -> dict(states [(row, plies)], policy [dense 209], value, flags, plies, resign_min [2],
    calibration)."""
    cal = bool(is_calibration(seed, [g], calibration)[0])
    capacity, reserve = 1 + 2 * sims * MAX_CHILDREN, sims * MAX_CHILDREN

    def fresh(state):
        if considered is not None:
            return mg.GumbelSearch(state, considered)
        return NoisedSearch(state, alpha) if alpha is not None else ReuseSearch(state)

    o = fresh(mo.COracleState())
    rmin, seen, pols, ply, flags = [math.inf, math.inf], [], [], 0, None
    while not o.root.state.is_done() and (max_plies is None or ply < max_plies):
        s = o.root.state
        seen.append((s.row.tolist(), s.plies))
        if considered is not None or alpha is not None:
            o.search(predict, sims, seed, g, ply)
        else:
            o.search(predict, sims)
        stat = statistic(o.root)
        if not math.isnan(stat):
            rmin[ply & 1] = min(rmin[ply & 1], stat)
        dense = np.zeros(209)
        if considered is not None:
            pol, choice = o.result()
            dense[o.actions()] = pol
            a = o.actions()[choice]
        else:
            c = np.array(o.counts(), np.float64)
            if temperature == 0:
                k = int(np.argmax(c))
                dense[o.actions()[k]] = 1.0
                a = o.actions()[k]
            else:
                dense[o.actions()] = c / c.sum()
                a = o.actions()[move_draw(c, seed, g, ply)]
        pols.append(dense)
        if not cal and stat < v_resign:
            flags = 1 | 4
            break
        if reuse:
            o.advance([a], capacity, reserve)
        else:
            o = fresh(s.next(a))
        ply += 1
    if flags is None:
        end = o.root.state
        flags = 1 if end.is_lose() else (2 if end.is_draw() else 0)
    lost = flags & 1
    fpv = (-1.0 if ply % 2 == 0 else 1.0) if lost else 0.0
    return {"states": seen, "policy": pols, "value": [fpv if k % 2 == 0 else -fpv for k in range(len(seen))], "flags": flags,
            "plies": ply, "resign_min": rmin, "calibration": cal}
