"""Self-play -- drop-in for reference self_play.py, with all games of a run played in lock-step on
the GPU (game-level sharding across ranks needs no communication; SURVEY.md section 8e).

History format is the reference's (self_play.py:51-54,63-66): a list of
``[[player, enemy, walls], policy (209 floats), value]`` pickled to ``./data/<timestamp>.history``."""
import math
import os
import pickle
from datetime import datetime

import numpy as np
import torch

from . import _lib
from . import game_logic as gl
from . import pv_mcts
from .constants import PV_NETWORK_PATH
from .pv_network_gnn import GNNNetwork, POLICY_OUTPUT_SIZE
from .positions import start_states

# Parameters
SP_GAME_COUNT = 50  # Number of games for self-play (self_play.py:19)
SP_TEMPERATURE = 1.0  # Temperature parameter for Boltzmann distribution (self_play.py:20)


def first_player_value(ended_state):
    """1: First player wins, -1: First player loses, 0: Draw (self_play.py:22-27)."""
    if ended_state.is_lose():
        return -1 if ended_state.is_first_player() else 1
    return 0


def write_data(history, directory='./data/'):
    """Save training data to a file (self_play.py:30-37)."""
    now = datetime.now()
    os.makedirs(directory, exist_ok=True)
    path = os.path.join(directory, '{:04}{:02}{:02}{:02}{:02}{:02}.history'.format(
        now.year, now.month, now.day, now.hour, now.minute, now.second))
    with open(path, mode='wb') as f:
        pickle.dump(history, f)
    return path


@torch.no_grad()
def play_batch_device(model, num_games, device=None, sims=None, temperature=SP_TEMPERATURE, seed=None, max_plies=None,
                      policy_dtype=torch.float64, tree_reuse=False, dirichlet_alpha=None, noise_fraction=0.25, gumbel_considered=None,
                      gumbel_scale=1.0, resign_threshold=None, resign_calibration=0.1, forced_k=None, fast_sims=None, full_search_prob=0.25):
    """Execute `num_games` self-play games in lock-step (self_play.py:40-68 per game) and keep the record on the device:
    dict(states uint8[T,32] packed, policy [T,209] search policies over all actions (self_play.py:51-54), value f32[T]
    back-filled game results seen from the player to move (self_play.py:63-66), game int64[T], ply int64[T],
    flags uint8[G] (bit 0 = the player to move at the end has lost, bit 1 = draw), plies int64[G], sims int = new simulations
    run, reused int = searches that continued a carried tree, full_searches / fast_searches int = searches with `sims` / fast_sims
    new simulations).

    Per ply: one search (200 graph-replayed simulation steps in a handful of launches) and ONE library call,
    aq_selfplay_advance -- search policy, its dense 209-wide record, the sampled move, the next states and the compaction of the
    games still running -- then one synchronisation that reads the search's status flags and the number of survivors together.
    A game's moves are drawn from a hash of (seed, game, ply): they do not depend on the other games of the batch.

    tree_reuse=True (AlphaGo Zero; the reference builds a fresh root per move): each search continues the tree of the game's
    previous one below the move played, so its policy counts the carried root visits as well as the `sims` new ones.

    dirichlet_alpha (AlphaZero; the reference has none): every search mixes Dirichlet(dirichlet_alpha) noise into its root priors
    with weight noise_fraction (BatchedMCTS), drawn from (seed, game, ply) like the moves, so a game still does not depend on the
    other games of the batch and a seed reproduces the run.  The record is the same as without noise.

    gumbel_considered (Gumbel AlphaZero; the reference has none): every search uses the Gumbel root of BatchedMCTS, its draw keyed
    by (seed, game, ply), and the ply calls aq_selfplay_advance_chosen: the recorded policy is the search's improved policy
    softmax(logits + sigma(completed Q)) and the move is the search's choice.  `temperature` is not used then.  The record format
    and the value targets are the same.

    resign_threshold (AlphaGo Zero resignation; the reference has none): after each search the ply reads the search's root value
    and its most visited child's value (BatchedMCTS.root_values) and calls aq_selfplay_advance_resign.  With s the larger of the
    two, a game resigns when s < resign_threshold, unless it is one of the calibration games: those, a fraction resign_calibration
    of the games drawn from (seed, game), never resign and measure how often resigning would have been wrong.  A resigned game
    records its last searched position too and ends lost for the player to move (flags bit 0 and bit 2, plies = the moves played;
    the value targets follow as for any loss).  The record gains resign_min f64[num_games, 2], the smallest s each side saw
    (column 0 the first player, +inf where a side never searched), and calibration bool[num_games]; resign_threshold_for picks a
    threshold from them.  None (the default) plays every game to its end, as the reference does.

    forced_k (KataGo's forced playouts and policy target pruning; the reference has none): every search forces visits to its
    visited root children (BatchedMCTS) and returns pruned counts, and the ply records and draws its move from those.  It is meant
    to pair with dirichlet_alpha: the noise still explores, but the visits it forced are taken out of the policy target.  The
    record format, the value targets and resignation are the same (the most visited child is never pruned).

    fast_sims (KataGo's playout cap randomization; the reference has none): each move of each game is full with probability
    full_search_prob, drawn from (seed, game, ply) alone (aq_selfplay_partition), else fast.  A full move searches with `sims` new
    simulations and the configured root noise and forced playouts, and its position is recorded; a fast move searches with
    fast_sims new simulations without root noise (BatchedMCTS.search(fast_sims=...); with forced_k it still forces and prunes, unlike
    KataGo's cheap searches), plays its move as any other and is not recorded: neither a policy nor a value target.  Per ply: the
    partition of the games into full and fast rows (at ply 0 on the start states, which costs one synchronisation before the first
    ply; later at the end of the previous ply), the search, the move, and the one synchronisation, which also reads the number of full
    rows.  The record holds only the full positions, with their real ply; the value targets follow from the game results as ever.
    It combines with tree_reuse, dirichlet_alpha, forced_k and resignation (every game may resign after a full or a fast search),
    not with gumbel_considered.  None (the default) searches every move in full."""
    if policy_dtype not in (torch.float64, torch.float32):
        raise ValueError("policy_dtype must be torch.float64 or torch.float32")
    if resign_threshold is not None:
        if math.isnan(resign_threshold):
            raise ValueError("resign_threshold must be a number (or None), not NaN")
        if not 0.0 <= resign_calibration <= 1.0:
            raise ValueError(f"resign_calibration must be in [0, 1], not {resign_calibration!r}")
    sims = sims or pv_mcts.PV_EVALUATE_COUNT
    pcr = fast_sims is not None
    if pcr:
        if isinstance(fast_sims, bool) or int(fast_sims) != fast_sims or not 1 <= fast_sims <= sims:
            raise ValueError(f"fast_sims must be an integer in [1, sims = {sims}] (or None), not {fast_sims!r}")
        if not 0.0 <= full_search_prob <= 1.0:
            raise ValueError(f"full_search_prob must be in [0, 1], not {full_search_prob!r}")
        if gumbel_considered is not None:
            raise ValueError("fast_sims cannot be combined with gumbel_considered: the Gumbel schedule depends on the budget")
        fast_sims = int(fast_sims)
    dev = gl._dev(device)
    L, P = _lib.load(), _lib.ptr
    seed = (int(seed) if seed is not None else int(torch.seed())) & (2 ** 64 - 1)
    mcts = pv_mcts.searcher_for(model, sims, dev, tree_reuse=tree_reuse, dirichlet_alpha=dirichlet_alpha, noise_fraction=noise_fraction,
                                gumbel_considered=gumbel_considered, gumbel_scale=gumbel_scale, forced_k=forced_k)
    states = start_states(num_games, dev)
    game_id = torch.arange(num_games, device=dev)
    rec_state, rec_policy, rec_game, sizes, searched = [], [], [], [], []
    final_flags = torch.zeros(max(num_games, 1), dtype=torch.uint8, device=dev)
    final_plies = torch.zeros(max(num_games, 1), dtype=torch.int64, device=dev)
    ws = torch.empty((max(1, L.aq_selfplay_ws_bytes(num_games)),), dtype=torch.uint8, device=dev)
    alive = torch.zeros((1,), dtype=torch.int32, device=dev)
    resign = resign_threshold is not None
    if resign:
        resign_min = torch.full((max(num_games, 1), 2), math.inf, dtype=torch.float64, device=dev)
        calibration = torch.zeros(max(num_games, 1), dtype=torch.uint8, device=dev)   # written by the kernel for every game it plays
    ply, sims_run, reused, full_searches = 0, 0, 0, 0
    src_row = path = None
    full = None   # pcr: the number of full rows of the ply, which come first
    if pcr:
        full_count = torch.zeros((1,), dtype=torch.int32, device=dev)
        row_of = torch.empty(max(num_games, 1), dtype=torch.int64, device=dev)   # tree_reuse: a game's row in the last search

        def partition(st, gid, G, count, at_ply):   # -> the rows reordered full first, their input rows; full_count is written
            out, out_id, out_row = torch.empty_like(st), torch.empty_like(gid), torch.empty_like(gid)
            _lib.check(L.aq_selfplay_partition(P(st), P(gid), G, P(count), seed, at_ply, float(full_search_prob), P(out), P(out_id),
                                               P(out_row), P(full_count), _lib.stream_ptr(dev)), "aq_selfplay_partition")
            return out, out_id, out_row
        if num_games:
            with torch.cuda.device(dev):
                states, game_id, _ = partition(states, game_id, num_games, None, 0)
            full = int(full_count.item())
    with torch.cuda.device(dev):
        while states.shape[0] > 0 and (max_plies is None or ply < max_plies):
            G = states.shape[0]
            counts, actions, n, status = mcts.search_async(states, src_row=src_row, path=path, noise_seed=seed, game_id=game_id, ply=ply,
                                                           fast_sims=fast_sims, full_rows=full)
            sims_run += G * sims if full is None else full * sims + (G - full) * fast_sims
            full_searches += G if full is None else full
            dense = torch.empty((G, POLICY_OUTPUT_SIZE), dtype=policy_dtype, device=dev)
            nxt = torch.empty_like(states)
            nxt_id = torch.empty_like(game_id)
            chosen = torch.empty((G,), dtype=torch.int16, device=dev) if tree_reuse else None
            if resign:
                root_value, best_q = mcts.root_values()
                by_counts = gumbel_considered is None
                _lib.check(L.aq_selfplay_advance_resign(P(states), P(counts) if by_counts else None, None if by_counts else P(mcts.last_policy),
                                                        None if by_counts else P(mcts.last_choice), P(actions), P(n), P(game_id), G,
                                                        float(temperature), seed, ply, P(dense), int(policy_dtype == torch.float64), P(chosen),
                                                        P(root_value), P(best_q), float(resign_threshold), float(resign_calibration),
                                                        P(resign_min), P(calibration), P(nxt), P(nxt_id), P(final_flags), P(final_plies), P(alive), P(ws),
                                                        _lib.stream_ptr(dev)), "aq_selfplay_advance_resign")
            elif gumbel_considered is None:
                _lib.check(L.aq_selfplay_advance(P(states), P(counts), P(actions), P(n), P(game_id), G, float(temperature), seed, ply,
                                                 P(dense), int(policy_dtype == torch.float64), P(chosen), P(nxt), P(nxt_id), P(final_flags),
                                                 P(final_plies), P(alive), P(ws), _lib.stream_ptr(dev)), "aq_selfplay_advance")
            else:
                _lib.check(L.aq_selfplay_advance_chosen(P(states), P(mcts.last_policy), P(mcts.last_choice), P(actions), P(n), P(game_id), G,
                                                        ply, P(dense), int(policy_dtype == torch.float64), P(chosen), P(nxt), P(nxt_id),
                                                        P(final_flags), P(final_plies), P(alive), P(ws), _lib.stream_ptr(dev)),
                           "aq_selfplay_advance_chosen")
            parts = [status, alive]
            if mcts.last_kept is not None:
                parts.append((mcts.last_kept > 0).sum(dtype=torch.int32).reshape(1))
            if pcr:   # the next ply's partition, on the survivors
                nxt, nxt_id, _ = partition(nxt, nxt_id, G, alive, ply + 1)
                parts.append(full_count)
            flags = torch.cat(parts).tolist()      # the ply's only synchronisation
            mcts.check_status(flags[:3])
            reused += flags[4] if mcts.last_kept is not None else 0
            keep = G if full is None else full     # pcr: only the full rows are recorded
            rec_state.append(states[:keep])
            rec_policy.append(dense[:keep])
            rec_game.append(game_id[:keep])
            sizes.append(keep)
            searched.append(G)
            ply += 1
            if tree_reuse:
                if pcr:
                    # the partition reorders the games, so a survivor's previous row is looked up by its game id
                    row_of[game_id] = torch.arange(G, device=dev)
                    src_row = row_of[nxt_id[:flags[3]]]
                else:
                    # the compaction keeps game_id ascending, so a survivor's previous row is found by binary search
                    src_row = torch.searchsorted(game_id, nxt_id[:flags[3]])
                path = chosen[src_row].reshape(-1, 1)
            states, game_id = nxt[:flags[3]], nxt_id[:flags[3]]
            if pcr:
                full = flags[-1]
    extra = {}
    if resign:
        extra = {"resign_min": resign_min[:num_games], "calibration": calibration[:num_games] != 0}
    if not sizes:
        z = torch.zeros((0,), dtype=torch.int64, device=dev)
        return {"states": states, "policy": torch.zeros((0, POLICY_OUTPUT_SIZE), dtype=policy_dtype, device=dev),
                "value": torch.zeros((0,), dtype=torch.float32, device=dev), "game": z, "ply": z, "flags": final_flags[:num_games],
                "plies": final_plies[:num_games], "sims": 0, "reused": 0, "full_searches": 0, "fast_searches": 0, **extra}
    sum_searches = sum(searched)
    game = torch.cat(rec_game)
    plyv = torch.repeat_interleave(torch.arange(len(sizes), device=dev), torch.tensor(sizes, device=dev))
    final_flags, final_plies = final_flags[:num_games], final_plies[:num_games]
    # first_player_value of the ended state (self_play.py:22-27): the player to move there has lost; the value target of a
    # position alternates in sign with the ply (self_play.py:63-66); unfinished games (max_plies) count as draws
    lost = (final_flags[game] & 1) != 0
    fpv = torch.where(lost, torch.where(final_plies[game] % 2 == 0, -1.0, 1.0), 0.0)
    value = torch.where(plyv % 2 == 0, fpv, -fpv).to(torch.float32)
    return {"states": torch.cat(rec_state), "policy": torch.cat(rec_policy), "value": value, "game": game, "ply": plyv,
            "flags": final_flags, "plies": final_plies, "sims": sims_run, "reused": reused, "full_searches": full_searches,
            "fast_searches": sum_searches - full_searches, **extra}


def resign_threshold_for(rec, max_false_positive=0.05):
    """AlphaGo Zero's automatic resignation threshold from a self-play record made with resign_threshold set (play_batch_device):
    the largest v with #{c : m_c < v} / C <= max_false_positive, over the C calibration games c, where m_c is the smallest search
    value (resign_min) seen by a side of game c that did not lose it -- both sides of a drawn or unfinished game.  A calibration
    game with m_c < v is one that resigning at v would have lost wrongly.  With k = floor(max_false_positive * C) that is the
    (k+1)-th smallest m_c, or +inf when k >= C.  Raises ValueError when the record has no calibration game."""
    if not 0.0 <= max_false_positive <= 1.0:
        raise ValueError(f"max_false_positive must be in [0, 1], not {max_false_positive!r}")
    asnp = lambda t: t.cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)
    cal = asnp(rec["calibration"]).astype(bool)
    flags, plies, rmin = asnp(rec["flags"])[cal], asnp(rec["plies"])[cal], asnp(rec["resign_min"])[cal]
    C = int(cal.sum())
    if C == 0:
        raise ValueError("the record has no calibration games: play with resign_calibration > 0")
    rows = np.arange(C)
    winner = rmin[rows, 1 - plies % 2]      # the player to move at the end (column plies % 2) is the one who lost
    m = np.where((flags & 1) != 0, winner, rmin.min(axis=1))
    k = math.floor(max_false_positive * C)
    return float(np.sort(m)[k]) if k < C else math.inf


def play_batch(model, num_games, device=None, sims=None, temperature=SP_TEMPERATURE, seed=None, max_plies=None, tree_reuse=False,
               dirichlet_alpha=None, noise_fraction=0.25, gumbel_considered=None, gumbel_scale=1.0, resign_threshold=None,
               resign_calibration=0.1, forced_k=None, fast_sims=None, full_search_prob=0.25):
    """play_batch_device + conversion to the reference's history: a list of [[player, enemy, walls], policy (209 floats), value]
    (self_play.py:51-54, 63-66), games in order, plies in order within a game.  Returns (history, dict with per-game results:
    flags, plies, and with resign_threshold also resign_min and calibration).  With fast_sims the history holds the positions of full
    searches only."""
    rec = play_batch_device(model, num_games, device, sims, temperature, seed, max_plies, tree_reuse=tree_reuse,
                            dirichlet_alpha=dirichlet_alpha, noise_fraction=noise_fraction, gumbel_considered=gumbel_considered,
                            gumbel_scale=gumbel_scale, resign_threshold=resign_threshold, resign_calibration=resign_calibration,
                            forced_k=forced_k, fast_sims=fast_sims, full_search_prob=full_search_prob)
    rows, _ = gl.unpack_rows(rec["states"])
    rows = rows.cpu().numpy()
    pols = rec["policy"].cpu().numpy()
    vals = rec["value"].cpu().numpy()
    gids = rec["game"].cpu().numpy()
    order = np.argsort(gids, kind='stable')                              # plies stay in order within a game
    history = []
    for i in order:
        r = rows[i]
        history.append([[r[0:2].tolist(), r[2:4].tolist(), r[4:].tolist()], pols[i].tolist(), int(vals[i])])
    info = {"flags": rec["flags"].cpu().numpy(), "plies": rec["plies"].cpu().numpy()}
    if resign_threshold is not None:
        info.update(resign_min=rec["resign_min"].cpu().numpy(), calibration=rec["calibration"].cpu().numpy())
    return history, info


def play(model, device=None):
    """Execute one self-play game (self_play.py:40-68)."""
    history, _ = play_batch(model, 1, device)
    return history


def self_play(game_count=None, model_path=None, data_dir='./data/', rank=0, world_size=1, sims=None, seed=None, tree_reuse=False,
              dirichlet_alpha=None, noise_fraction=0.25, gumbel_considered=None, gumbel_scale=1.0, resign_threshold=None,
              resign_calibration=0.1, forced_k=None, fast_sims=None, full_search_prob=0.25):
    """Perform self-play games and save the training data (self_play.py:71-98).  With
    world_size > 1 each rank plays its share of the games on its own GPU and rank 0 writes the file.
    tree_reuse=True keeps each game's search tree between moves; dirichlet_alpha adds AlphaZero root noise to every search;
    gumbel_considered searches with the Gumbel AlphaZero root and records its improved policy; resign_threshold lets games resign,
    resign_calibration of them excepted; forced_k forces root playouts and prunes them from the policy targets; fast_sims gives a
    fraction 1 - full_search_prob of the moves a cheap search and records only the others (see play_batch_device)."""
    game_count = SP_GAME_COUNT if game_count is None else game_count
    model = GNNNetwork()
    model.prep_for_inference(model_path=model_path or (PV_NETWORK_PATH + 'best.pth'))
    mine = game_count // world_size + (1 if rank < game_count % world_size else 0)
    history, _ = play_batch(model, mine, sims=sims, seed=None if seed is None else seed + rank, tree_reuse=tree_reuse,
                            dirichlet_alpha=dirichlet_alpha, noise_fraction=noise_fraction, gumbel_considered=gumbel_considered,
                            gumbel_scale=gumbel_scale, resign_threshold=resign_threshold,
                            resign_calibration=resign_calibration, forced_k=forced_k, fast_sims=fast_sims,
                            full_search_prob=full_search_prob) if mine else ([], None)
    if world_size > 1:
        import torch.distributed as dist
        gathered = [None] * world_size if rank == 0 else None
        dist.gather_object(history, gathered, dst=0)
        if rank == 0:
            history = [h for part in gathered for h in part]
    path = None
    if rank == 0:
        path = write_data(history, data_dir)
        print(f'Self-play: {game_count} games, {len(history)} positions -> {path}')
    del model
    torch.cuda.empty_cache()
    return path


if __name__ == '__main__':
    self_play()
