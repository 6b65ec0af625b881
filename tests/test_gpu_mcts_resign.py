"""Resignation (aq_mcts_root_values, BatchedMCTS.root_values, aq_selfplay_advance_resign, play_batch_device(resign_threshold=...))
against the CPU restatement in tests/mcts_resign_oracle.py.  Priors and values of the hash / uniform evaluators are bit-identical
on both sides and the root values are double quotients of the same sums, so everything but the Gumbel improved policy (an exp per
child, within one float32 ulp as in tests/test_gpu_mcts_gumbel.py) is compared exactly."""
import math

import numpy as np
import pytest
import torch

from alphaquoridorgnn_b200 import _lib, positions, pv_mcts, self_play
from alphaquoridorgnn_b200 import game_logic as gl
from alphaquoridorgnn_b200.pv_network_gnn import GNNNetwork

import mcts_gumbel_oracle as mg
import mcts_resign_oracle as mr
from mcts_noise_oracle import NoisedSearch
from mcts_reuse_oracle import ReuseSearch, hash_predict, uniform_predict
from test_gpu_mcts import EVAL, hash_evaluator
from test_gpu_mcts_gumbel import assert_policy_close
from test_gpu_mcts_noise import fresh_ws
from test_gpu_mcts_reuse import _record_games, capacity, golden_states, pack

pytestmark = pytest.mark.gpu

PREDICT = {"hash": hash_predict, "uniform": uniform_predict}
MC = pv_mcts.MAX_CHILDREN
P = _lib.ptr
SHARED = ("states", "policy", "value", "game", "ply", "flags", "plies")


def abi_root_values(ws, G, max_nodes):
    """(root_value, best_q, best_child) of every row of a workspace, on the host."""
    rv = torch.empty((G,), dtype=torch.float64, device="cuda")
    bq = torch.empty((G,), dtype=torch.float64, device="cuda")
    bc = torch.empty((G,), dtype=torch.int16, device="cuda")
    _lib.check(_lib.load().aq_mcts_root_values(P(ws), G, max_nodes, P(rv), P(bq), P(bc), _lib.stream_ptr()), "aq_mcts_root_values")
    return rv.cpu().numpy(), bq.cpu().numpy(), bc.cpu().numpy()


def same_float(a, b):
    return (a == b) or (math.isnan(a) and math.isnan(b))


def check_root_values(mcts, oracle_roots):
    rv, bq = mcts.root_values()
    ws, G, G_real, max_nodes = mcts._root
    _, _, bc = abi_root_values(ws, G, max_nodes)
    rv, bq = rv.cpu().numpy(), bq.cpu().numpy()
    assert rv.shape == (len(oracle_roots),) and rv.dtype == np.float64
    for r, root in enumerate(oracle_roots):
        want = mr.root_values(root)
        assert same_float(rv[r], want[0]) and same_float(bq[r], want[1]) and int(bc[r]) == want[2], (r, rv[r], bq[r], bc[r], want)


def test_root_values_before_any_search_raise():
    with pytest.raises(ValueError):
        pv_mcts.BatchedMCTS(hash_evaluator, 4).root_values()


def test_unvisited_roots_have_no_values(mcts_golden):
    roots = pack(golden_states(mcts_golden, "hash"))
    G, max_nodes = roots.shape[0], 1 + MC
    rv, bq, bc = abi_root_values(fresh_ws(roots, max_nodes), G, max_nodes)
    assert np.isnan(rv).all() and (bq == -np.inf).all() and (bc == -1).all()


@pytest.mark.parametrize("name", ["hash", "uniform"])
@pytest.mark.parametrize("sims", [1, 2, 16, 50])
def test_root_values_of_fresh_carried_noised_and_gumbel_roots(mcts_golden, name, sims):
    states = golden_states(mcts_golden, name)
    roots = pack(states)
    G = len(states)
    gid = torch.arange(G, device="cuda") + 40
    predict = PREDICT[name]
    # fresh roots
    m = pv_mcts.BatchedMCTS(EVAL[name], sims)
    m.search(roots)
    oracles = [ReuseSearch(s) for s in states]
    for o in oracles:
        o.search(predict, sims)
    check_root_values(m, [o.root for o in oracles])
    # carried roots: the most visited child becomes the next root
    m = pv_mcts.BatchedMCTS(EVAL[name], sims, tree_reuse=True)
    counts, actions, _ = m.search(roots)
    best = torch.gather(actions, 1, torch.argmax(counts, 1, keepdim=True)).squeeze(1)
    nxt, term = gl.next_batch(roots, best)
    alive = torch.nonzero(term == 0).squeeze(1)
    m.search(nxt[alive].contiguous(), src_row=alive, path=best[alive].reshape(-1, 1))
    kept = []
    for r in alive.tolist():
        o = oracles[r]
        o.advance([int(best[r])], capacity(sims), sims * MC)
        o.search(predict, sims)
        kept.append(o.root)
    check_root_values(m, kept)
    # noised roots
    m = pv_mcts.BatchedMCTS(EVAL[name], sims, dirichlet_alpha=0.3)
    m.search(roots, noise_seed=5, game_id=gid, ply=3)
    noised = []
    for r, s in enumerate(states):
        o = NoisedSearch(s, 0.3)
        o.search(predict, sims, 5, 40 + r, 3)
        noised.append(o.root)
    check_root_values(m, noised)
    # Gumbel roots
    m = pv_mcts.BatchedMCTS(EVAL[name], sims, gumbel_considered=4)
    m.search(roots, noise_seed=5, game_id=gid, ply=3)
    gumbel = []
    for r, s in enumerate(states):
        o = mg.GumbelSearch(s, 4)
        o.search(predict, sims, 5, 40 + r, 3)
        gumbel.append(o.root)
    check_root_values(m, gumbel)


def pick_seed(games, calibration):
    """A seed whose calibration games are neither none nor all but two of `games`."""
    for seed in range(1, 1000):
        k = int(mr.is_calibration(seed, np.arange(games), calibration).sum())
        if 1 <= k <= games - 2:
            return seed


def threshold_between(rec, calibration, seed):
    """A threshold that some but not all of the non-calibration games fall below (from a record where nobody resigned): the
    median of their smallest statistics, or just above it when they are all equal."""
    rmin = rec["resign_min"].cpu().numpy().min(axis=1)
    cal = mr.is_calibration(seed, np.arange(rmin.shape[0]), calibration)
    m = np.sort(rmin[~cal])
    if m[0] == m[-1]:
        return float(np.nextafter(m[0], np.inf))
    lo = m[(len(m) - 1) // 2]
    return float((lo + m[m > lo].min()) / 2)


MODES = {"plain-t0": dict(temperature=0), "plain-t1": dict(temperature=1.0), "reuse-t0": dict(temperature=0, tree_reuse=True),
         "reuse-t1": dict(temperature=1.0, tree_reuse=True), "noise-t0": dict(temperature=0, dirichlet_alpha=0.3),
         "gumbel": dict(gumbel_considered=4)}


@pytest.mark.parametrize("mode", list(MODES))
def test_self_play_with_resignation_plays_the_oracle_games(mode):
    games, sims, cal = 8, 12, 0.25
    kw = MODES[mode]
    seed = pick_seed(games, cal)
    full = self_play.play_batch_device(hash_evaluator, games, sims=sims, seed=seed, resign_threshold=-2.0, resign_calibration=1.0, **kw)
    v = threshold_between(full, cal, seed)
    rec = self_play.play_batch_device(hash_evaluator, games, sims=sims, seed=seed, resign_threshold=v, resign_calibration=cal, **kw)
    flags, plies = rec["flags"].cpu().numpy(), rec["plies"].cpu().numpy()
    rmin, calib = rec["resign_min"].cpu().numpy(), rec["calibration"].cpu().numpy()
    game, ply, value = rec["game"].cpu().numpy(), rec["ply"].cpu().numpy(), rec["value"].cpu().numpy()
    for g, (states, pol) in enumerate(_record_games(rec, games)):
        o = mr.play_game(hash_predict, sims, seed, g, v, cal, temperature=kw.get("temperature", 0), reuse=kw.get("tree_reuse", False),
                         alpha=kw.get("dirichlet_alpha"), considered=kw.get("gumbel_considered"))
        assert states == o["states"], (mode, g)
        for k in range(len(states)):
            if "gumbel_considered" in kw:
                assert_policy_close(pol[k].astype(np.float32), o["policy"][k])
            else:
                assert np.array_equal(pol[k], o["policy"][k]), (mode, g, k)
        idx = np.nonzero(game == g)[0]
        assert value[idx[np.argsort(ply[idx])]].tolist() == o["value"], (mode, g)
        assert int(flags[g]) == o["flags"] and int(plies[g]) == o["plies"], (mode, g)
        assert rmin[g].tolist() == o["resign_min"], (mode, g)
        assert bool(calib[g]) == o["calibration"], (mode, g)
    resigned = (flags & 4) != 0
    assert not resigned[calib].any()
    # a game resigns exactly when the smallest statistic of its played-out run falls below the threshold
    assert np.array_equal(resigned, ~calib & (full["resign_min"].cpu().numpy().min(axis=1) < v))
    assert resigned.any()
    if mode not in ("plain-t0", "reuse-t0"):   # greedy games from the start position without noise are all the same game
        assert resigned.sum() < (~calib).sum(), mode


@pytest.mark.parametrize("kw", [dict(), dict(tree_reuse=True), dict(dirichlet_alpha=0.3), dict(gumbel_considered=4)])
def test_thresholds_that_never_resign_give_the_record_without_resignation(kw):
    games, sims, seed = 6, 8, 17
    off = self_play.play_batch_device(hash_evaluator, games, sims=sims, seed=seed, temperature=1.0, **kw)
    assert "resign_min" not in off and "calibration" not in off
    for v, cal in ((-1.5, 0.0), (0.5, 1.0), (2.0, 1.0)):
        on = self_play.play_batch_device(hash_evaluator, games, sims=sims, seed=seed, temperature=1.0, resign_threshold=v,
                                         resign_calibration=cal, **kw)
        for k in SHARED:
            assert torch.equal(on[k], off[k]), (v, cal, k)
        assert on["sims"] == off["sims"] and on["reused"] == off["reused"]
        assert bool(on["calibration"].all()) == (cal == 1.0)
        assert bool(on["calibration"].any()) == (cal != 0.0)
        assert torch.isfinite(on["resign_min"]).all()


def test_a_threshold_above_one_resigns_every_game_at_once():
    games = 5
    rec = self_play.play_batch_device(hash_evaluator, games, sims=8, seed=3, resign_threshold=1.5, resign_calibration=0.0)
    assert rec["states"].shape[0] == games and sorted(rec["game"].tolist()) == list(range(games))
    assert rec["ply"].tolist() == [0] * games and rec["value"].tolist() == [-1.0] * games
    assert rec["plies"].tolist() == [0] * games and rec["flags"].tolist() == [5] * games
    rmin = rec["resign_min"].cpu().numpy()
    assert np.isfinite(rmin[:, 0]).all() and (rmin[:, 1] == np.inf).all()   # the second player never searched
    assert not rec["calibration"].any()


def test_a_game_does_not_depend_on_its_batch():
    """The same games in batches of 1, 37 and 300; the network path pads 300 rows to 512 inside the search."""
    torch.manual_seed(4)
    net = GNNNetwork().cuda().eval()
    net.precision = "fp32"
    kw = dict(sims=4, seed=9, temperature=1.0, max_plies=30, resign_calibration=0.2)
    full = self_play.play_batch_device(net, 300, resign_threshold=-2.0, **dict(kw, resign_calibration=1.0))
    v = threshold_between(full, 0.2, 9)
    recs = {n: self_play.play_batch_device(net, n, resign_threshold=v, **kw) for n in (1, 37, 300)}
    resigned = (recs[300]["flags"] & 4) != 0
    assert resigned.any() and not resigned.all()
    per_game = {n: _record_games(recs[n], n) for n in recs}
    for n in (1, 37):
        for g in range(n):
            assert per_game[n][g][0] == per_game[300][g][0], (n, g)
            assert np.array_equal(per_game[n][g][1], per_game[300][g][1]), (n, g)
        for k in ("flags", "plies", "resign_min", "calibration"):
            assert torch.equal(recs[n][k], recs[300][k][:n]), (n, k)
        for g in range(n):
            a = recs[n]["value"][recs[n]["game"] == g]
            b = recs[300]["value"][recs[300]["game"] == g]
            assert torch.equal(a, b), (n, g)


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_network_graph_replay_equals_eager_loop_with_resignation(prec):
    torch.manual_seed(1)
    net = GNNNetwork().cuda().eval()
    net.precision = prec
    kw = dict(sims=8, seed=11, temperature=1.0, max_plies=40)
    full = self_play.play_batch_device(net, 48, resign_threshold=-2.0, resign_calibration=1.0, **kw)
    v = threshold_between(full, 0.25, 11)
    graph = self_play.play_batch_device(net, 48, resign_threshold=v, resign_calibration=0.25, **kw)
    searcher = pv_mcts.searcher_for(net, 8, gl._dev(None))
    assert searcher.use_graph and searcher._graphs
    searcher.use_graph = False
    eager = self_play.play_batch_device(net, 48, resign_threshold=v, resign_calibration=0.25, **kw)
    for k in SHARED + ("resign_min", "calibration"):
        assert torch.equal(graph[k], eager[k]), (prec, k)
    assert bool(((graph["flags"] & 4) != 0).any())


def resign_call(roots, counts=None, child_policy=None, choice=None, v=0.0, cal=0.5, root_value=True, best_q=True, resign_min=True,
                is_cal=True, G=None, gid=None, seed=0, out=None):
    L = _lib.load()
    G0 = roots.shape[0]
    G = G0 if G is None else G
    actions = torch.zeros((G0, gl.MAX_LEGAL), dtype=torch.int16, device="cuda")
    n = torch.full((G0,), 2, dtype=torch.int16, device="cuda")
    gid = torch.arange(G0, device="cuda") if gid is None else gid
    is_calibration = torch.zeros(int(gid.max()) + 1, dtype=torch.uint8, device="cuda") if out is None else out
    dense = torch.empty((G0, gl.NUM_ACTIONS), dtype=torch.float64, device="cuda")
    rv = torch.zeros(G0, dtype=torch.float64, device="cuda")
    rmin = torch.full((int(gid.max()) + 1, 2), math.inf, dtype=torch.float64, device="cuda")
    nxt, nxt_id = torch.empty_like(roots), torch.empty_like(gid)
    ff, fp = torch.zeros(G0, dtype=torch.uint8, device="cuda"), torch.zeros(G0, dtype=torch.int64, device="cuda")
    alive = torch.zeros(1, dtype=torch.int32, device="cuda")
    ws = torch.empty((L.aq_selfplay_ws_bytes(G0),), dtype=torch.uint8, device="cuda")
    return L.aq_selfplay_advance_resign(P(roots), P(counts), P(child_policy), P(choice), P(actions), P(n), P(gid), G, 1.0, seed, 0, P(dense), 1,
                                        None, P(rv) if root_value else None, P(rv) if best_q else None, v, cal,
                                        P(rmin) if resign_min else None, P(is_calibration) if is_cal else None, P(nxt), P(nxt_id), P(ff),
                                        P(fp), P(alive), P(ws), _lib.stream_ptr())


def test_bad_arguments_are_refused(mcts_golden):
    roots = pack(golden_states(mcts_golden, "hash"))
    G = roots.shape[0]
    counts = torch.ones((G, gl.MAX_LEGAL), dtype=torch.int32, device="cuda")
    pol = torch.full((G, gl.MAX_LEGAL), 0.5, device="cuda")
    ch = torch.zeros((G,), dtype=torch.int16, device="cuda")
    assert resign_call(roots, counts=counts) == 0
    assert resign_call(roots, child_policy=pol, choice=ch) == 0
    bad = [dict(), dict(counts=counts, child_policy=pol, choice=ch), dict(counts=counts, choice=ch), dict(child_policy=pol),
           dict(choice=ch), dict(counts=counts, v=float("nan")), dict(counts=counts, cal=-0.01), dict(counts=counts, cal=1.01),
           dict(counts=counts, cal=float("nan")), dict(counts=counts, root_value=False), dict(counts=counts, best_q=False),
           dict(counts=counts, resign_min=False), dict(counts=counts, is_cal=False), dict(counts=counts, G=0)]
    for kw in bad:
        assert resign_call(roots, **kw) == -1, kw
        with pytest.raises(_lib.AqError):
            _lib.check(resign_call(roots, **kw), "aq_selfplay_advance_resign")
    L = _lib.load()
    max_nodes = 1 + MC
    ws = fresh_ws(roots, max_nodes)
    d = torch.empty(G, dtype=torch.float64, device="cuda")
    b = torch.empty(G, dtype=torch.int16, device="cuda")
    st = _lib.stream_ptr()
    assert L.aq_mcts_root_values(P(ws), G, max_nodes, P(d), P(d), P(b), st) == 0
    for args in ((None, G, max_nodes, P(d), P(d), P(b)), (P(ws), 0, max_nodes, P(d), P(d), P(b)), (P(ws), G, 0, P(d), P(d), P(b)),
                 (P(ws), G, max_nodes, None, P(d), P(b)), (P(ws), G, max_nodes, P(d), None, P(b)), (P(ws), G, max_nodes, P(d), P(d), None)):
        assert L.aq_mcts_root_values(*args, st) == -1
    for kw in (dict(resign_threshold=float("nan")), dict(resign_threshold=0.0, resign_calibration=-0.1),
               dict(resign_threshold=0.0, resign_calibration=1.5), dict(resign_threshold=0.0, resign_calibration=float("nan"))):
        with pytest.raises(ValueError):
            self_play.play_batch_device(hash_evaluator, 2, sims=2, **kw)
    torch.cuda.synchronize()


@pytest.mark.parametrize("cal", [0.1, 0.5])
def test_the_kernel_writes_the_calibration_bit_of_the_oracle(cal):
    """The calibration bit the move kernel used, indexed by game id, for 4,096 rows with scattered ids and three seeds."""
    G = 4096
    roots = positions.random_positions(G, seed=3, games=64)
    counts = torch.ones((G, gl.MAX_LEGAL), dtype=torch.int32, device="cuda")
    gid = torch.randperm(3 * G, generator=torch.Generator().manual_seed(5))[:G].cuda()
    for seed in (0, 99, 2 ** 64 - 1):
        out = torch.full((3 * G,), 7, dtype=torch.uint8, device="cuda")
        _lib.check(resign_call(roots, counts=counts, cal=cal, gid=gid, seed=seed, out=out), "aq_selfplay_advance_resign")
        got = out.cpu().numpy()
        ids = gid.cpu().numpy()
        assert np.array_equal(got[ids], mr.is_calibration(seed, ids, cal).astype(np.uint8)), seed
        untouched = np.ones(3 * G, bool)
        untouched[ids] = False
        assert (got[untouched] == 7).all()


def test_launch_counts(mcts_golden):
    L = _lib.load()
    roots = pack(golden_states(mcts_golden, "hash"))
    G, max_nodes = roots.shape[0], 1 + 4 * MC
    counts = torch.ones((G, gl.MAX_LEGAL), dtype=torch.int32, device="cuda")
    pol = torch.full((G, gl.MAX_LEGAL), 0.5, device="cuda")
    ch = torch.zeros((G,), dtype=torch.int16, device="cuda")
    for kw in (dict(counts=counts), dict(child_policy=pol, choice=ch)):
        c0 = L.aq_launch_count()
        assert resign_call(roots, **kw) == 0
        assert L.aq_launch_count() - c0 == 2
    ws = fresh_ws(roots, max_nodes)
    c0 = L.aq_launch_count()
    abi_root_values(ws, G, max_nodes)
    assert L.aq_launch_count() - c0 == 1
    plies = 6
    for kw in (dict(), dict(tree_reuse=True), dict(gumbel_considered=4)):
        n = []
        for resign in (None, -2.0):
            c0 = L.aq_launch_count()
            self_play.play_batch_device(hash_evaluator, 4, sims=4, seed=3, max_plies=plies, resign_threshold=resign, **kw)
            n.append(L.aq_launch_count() - c0)
        assert n[1] == n[0] + plies, kw   # one aq_mcts_root_values per ply; the advance entry stays two launches
    torch.cuda.synchronize()


def test_play_batch_history_of_resigned_games():
    games, sims, seed = 8, 8, 23
    _, info0 = self_play.play_batch(hash_evaluator, games, sims=sims, seed=seed, resign_threshold=-2.0, resign_calibration=1.0)
    m = info0["resign_min"].min(axis=1)
    v = float(np.median(m))
    history, info = self_play.play_batch(hash_evaluator, games, sims=sims, seed=seed, resign_threshold=v, resign_calibration=0.0)
    assert set(info) == {"flags", "plies", "resign_min", "calibration"} and not info["calibration"].any()
    resigned = (info["flags"] & 4) != 0
    assert resigned.any()
    start = 0
    for g in range(games):
        rows = int(info["plies"][g]) + (1 if resigned[g] else 0)
        vals = [h[2] for h in history[start:start + rows]]
        start += rows
        if resigned[g]:
            assert vals[-1] == -1 and all(a == -b and a in (-1, 1) for a, b in zip(vals[:-1], vals[1:])), (g, vals)
    assert start == len(history)
