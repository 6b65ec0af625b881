"""CPU restatement of playout cap randomization in self-play (KataGo: David J. Wu, "Accelerating Self-Play Learning in Go", 2019,
section 3.1), on top of the forced-playout and resignation oracles of tests/mcts_forced_oracle.py and tests/mcts_resign_oracle.py.
The reference has none.

  full move   : u < p with u = (mix64(mix64((seed ^ PCR_DOMAIN) + GOLDEN * (game_id + 1)) + PLY_MUL * (ply + 1)) >> 11) * 2^-53,
                as aq_selfplay_partition (csrc/mcts.cu) draws it
  full search : `sims` new simulations with the configured root noise (alpha) and forced_k; the position is recorded
  fast search : `fast_sims` new simulations without root noise, the same forced_k; the move is played and nothing is recorded
The move and the recorded policy come from the (pruned) counts as in tests/mcts_forced_oracle.py; k = None is the plain search,
which the forced oracle at k = 0 is.
"""
import math

import numpy as np

from oracle import mcts_oracle as mo

import mcts_forced_oracle as mf
import mcts_resign_oracle as mr
from mcts_noise_oracle import GOLDEN, M64, PLY_MUL, mix64

PCR_DOMAIN = 0x082EFA98EC4E6C89


def full_u(seed, game_id, ply):
    """u in [0, 1) of games game_id (int array) at ply (int or int array of the same shape): float64."""
    gid = np.asarray(game_id, dtype=np.int64).astype(np.uint64)
    pl = np.asarray(ply, dtype=np.int64).astype(np.uint64)
    with np.errstate(over="ignore"):
        a = np.uint64((int(seed) ^ PCR_DOMAIN) & M64) + np.uint64(GOLDEN) * (gid + np.uint64(1))
        z = mix64(mix64(a) + np.uint64(PLY_MUL) * (pl + np.uint64(1)))
    return (z >> np.uint64(11)).astype(np.float64) * 2.0 ** -53


def is_full(seed, game_id, ply, p):
    return full_u(seed, game_id, ply) < p


def partition(seed, game_id, ply, p):
    """What aq_selfplay_partition writes for rows with these game ids: (out_row int64 [n], full_count)."""
    full = is_full(seed, game_id, ply, p)
    rows = np.arange(len(full))
    return np.concatenate([rows[full], rows[~full]]), int(full.sum())


def play_game(predict, sims, fast_sims, p, seed, g, temperature=0, reuse=False, alpha=None, k=None, v_resign=None, calibration=0.0):
    """One self-play game with playout cap randomization.  -> dict(states [(row, plies)], policy [dense 209], ply [int], value,
    flags, plies, resign_min, full, fast): the recorded (full) positions only; full / fast count the searches of each kind."""
    cal = bool(mr.is_calibration(seed, [g], calibration)[0])
    capacity, reserve = 1 + 2 * sims * mr.MAX_CHILDREN, sims * mr.MAX_CHILDREN
    kk = 0.0 if k is None else k
    o = mf.ForcedSearch(mo.COracleState(), kk, alpha)
    rmin, seen, pols, plys, ply, flags, n_full = [math.inf, math.inf], [], [], [], 0, None, 0
    while not o.root.state.is_done():
        s = o.root.state
        full = bool(is_full(seed, [g], ply, p)[0])
        n_full += full
        o.alpha = alpha if full else None   # a fast search is the search without root noise
        o.search(predict, sims if full else fast_sims, seed, g, ply)
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
        if full:
            seen.append((s.row.tolist(), s.plies))
            pols.append(dense)
            plys.append(ply)
        if v_resign is not None and not cal and stat < v_resign:
            flags = 1 | 4
            break
        if reuse:
            o.advance([a], capacity, reserve)
        else:
            o = mf.ForcedSearch(s.next(a), kk, alpha)
        ply += 1
    searches = ply + 1 if flags is not None else ply
    if flags is None:
        end = o.root.state
        flags = 1 if end.is_lose() else (2 if end.is_draw() else 0)
    fpv = (-1.0 if ply % 2 == 0 else 1.0) if flags & 1 else 0.0
    return {"states": seen, "policy": pols, "ply": plys, "value": [fpv if j % 2 == 0 else -fpv for j in plys], "flags": flags,
            "plies": ply, "resign_min": rmin, "full": n_full, "fast": searches - n_full}
