"""Forced playouts and policy target pruning (aq_mcts_select_forced, aq_mcts_expand_select_forced, aq_mcts_root_counts_pruned,
BatchedMCTS(forced_k=...), play_batch_device(forced_k=...)) against the CPU restatement in tests/mcts_forced_oracle.py.  Priors and
values of the hash / uniform evaluators are bit-identical on both sides and n_forced and PUCT are computed with the same roundings,
so raw visit counts, pruned counts and self-play records are compared exactly."""
import numpy as np
import pytest
import torch

from alphaquoridorgnn_b200 import _lib, positions, pv_mcts, self_play
from alphaquoridorgnn_b200 import game_logic as gl
from alphaquoridorgnn_b200.pv_network_gnn import GNNNetwork
from oracle import mcts_oracle as mo

import mcts_forced_oracle as mf
from mcts_reuse_oracle import hash_predict, uniform_predict
from test_gpu_mcts import EVAL, hash_evaluator, uniform_evaluator
from test_gpu_mcts_noise import fresh_ws
from test_gpu_mcts_reuse import _record_games, capacity, golden_states, oracle_states, pack

pytestmark = pytest.mark.gpu

PREDICT = {"hash": hash_predict, "uniform": uniform_predict}
MC = pv_mcts.MAX_CHILDREN
P = _lib.ptr
SHARED = ("states", "policy", "value", "game", "ply", "flags", "plies")


@pytest.fixture(scope="module")
def roots():
    """The start position and 24 random positions of mid-game depth."""
    return torch.cat([pack([mo.COracleState()]), positions.random_positions(24, seed=31, games=64)]).contiguous()


def abi_counts(ws, G, max_nodes, forced_k=None):
    """(counts, actions, n_children) of a workspace: aq_mcts_root_counts, or aq_mcts_root_counts_pruned at forced_k."""
    L = _lib.load()
    counts = torch.full((G, gl.MAX_LEGAL), -7, dtype=torch.int32, device="cuda")
    actions = torch.empty((G, gl.MAX_LEGAL), dtype=torch.int16, device="cuda")
    n = torch.empty((G,), dtype=torch.int16, device="cuda")
    if forced_k is None:
        rc = L.aq_mcts_root_counts(P(ws), G, max_nodes, P(counts), P(actions), P(n), None, _lib.stream_ptr())
    else:
        rc = L.aq_mcts_root_counts_pruned(P(ws), G, max_nodes, pv_mcts.C_PUCT, forced_k, P(counts), P(actions), P(n), None,
                                          _lib.stream_ptr())
    _lib.check(rc, "root counts")
    return counts, actions, n


def check(counts, actions, n, r, o, pruned):
    k = int(n[r])
    assert actions[r, :k].tolist() == o.actions(), r
    assert counts[r, :k].tolist() == (o.pruned() if pruned else o.counts()), r
    assert not counts[r, k:].any(), r


@pytest.mark.parametrize("name", ["hash", "uniform"])
@pytest.mark.parametrize("sims", [1, 2, 16, 50])
@pytest.mark.parametrize("k", [0.5, 2.0, 8.0])
def test_raw_and_pruned_counts_match_the_oracle(mcts_golden, roots, name, sims, k):
    states = golden_states(mcts_golden, name) + oracle_states(roots[:8])
    mcts = pv_mcts.BatchedMCTS(EVAL[name], sims, forced_k=k)
    counts, actions, n = mcts.search(pack(states))
    G = len(states)
    raw, raw_a, raw_n = abi_counts(mcts._ws[0], G, 1 + sims * MC)
    again = abi_counts(mcts._ws[0], G, 1 + sims * MC, k)
    assert torch.equal(again[0], counts) and torch.equal(raw_a, actions) and torch.equal(raw_n, n)
    for r, s in enumerate(states):
        o = mf.ForcedSearch(s, k)
        o.search(PREDICT[name], sims)
        check(raw, actions, n, r, o, False)
        check(counts, actions, n, r, o, True)
    assert torch.equal(torch.argmax(counts, 1), torch.argmax(raw, 1))
    if name == "hash" and sims == 50:
        assert not torch.equal(counts, raw)


@pytest.mark.parametrize("name", ["hash", "uniform"])
def test_forced_search_with_noise_matches_the_oracle(mcts_golden, roots, name):
    sims, seed, ply, k = 50, 77, 4, 2.0
    states = golden_states(mcts_golden, name) + oracle_states(roots[:8])
    gids = [3 * r + 1 for r in range(len(states))]
    mcts = pv_mcts.BatchedMCTS(EVAL[name], sims, dirichlet_alpha=0.3, forced_k=k)
    counts, actions, n = mcts.search(pack(states), noise_seed=seed, game_id=torch.tensor(gids), ply=ply)
    raw, _, _ = abi_counts(mcts._ws[0], len(states), 1 + sims * MC)
    for r, s in enumerate(states):
        o = mf.ForcedSearch(s, k, 0.3)
        o.search(PREDICT[name], sims, seed, gids[r], ply)
        check(raw, actions, n, r, o, False)
        check(counts, actions, n, r, o, True)


@pytest.mark.parametrize("alpha", [None, 0.3])
@pytest.mark.parametrize("name", ["hash", "uniform"])
def test_forced_search_with_reuse_matches_the_oracle(mcts_golden, name, alpha):
    """Greedy games with tree reuse: a carried root's visits count in t, and a carried root is noised before its first descent."""
    sims, seed, k = 40, 9, 2.0
    starts = [mo.COracleState()] + golden_states(mcts_golden, name)
    oracles = [mf.ForcedSearch(s, k, alpha) for s in starts]
    mcts = pv_mcts.BatchedMCTS(EVAL[name], sims, tree_reuse=True, dirichlet_alpha=alpha, forced_k=k)
    games, src_row, path, carried = list(range(len(starts))), None, None, 0
    for ply in range(8):
        counts, actions, n = mcts.search(pack([oracles[g].root.state for g in games]), src_row=src_row, path=path, noise_seed=seed,
                                         game_id=torch.tensor(games), ply=ply)
        ws_slot = mcts._last[0]
        raw, _, _ = abi_counts(mcts._ws[ws_slot], len(games), capacity(sims))
        if src_row is not None:
            carried += int((mcts.last_kept > 0).sum())
        nxt, src, pth = [], [], []
        for r, g in enumerate(games):
            o = oracles[g]
            o.search(PREDICT[name], sims, seed, g, ply)
            check(raw, actions, n, r, o, False)
            check(counts, actions, n, r, o, True)
            a = o.actions()[int(np.argmax(o.pruned()))]
            o.advance([a], capacity(sims), sims * MC)
            if not o.root.state.is_done():
                nxt.append(g)
                src.append(r)
                pth.append([a])
        games = nxt
        src_row, path = torch.tensor(src, device="cuda"), torch.tensor(pth, dtype=torch.int16, device="cuda")
    assert carried > len(starts)


MODES = {"t0": dict(temperature=0), "t1": dict(temperature=1.0), "t1-reuse": dict(temperature=1.0, tree_reuse=True),
         "t1-noise": dict(temperature=1.0, dirichlet_alpha=0.3), "t0-noise-reuse": dict(temperature=0, dirichlet_alpha=0.3, tree_reuse=True),
         "t1-noise-resign": dict(temperature=1.0, dirichlet_alpha=0.3, resign_threshold=-2.0, resign_calibration=0.25)}


@pytest.mark.parametrize("mode", list(MODES))
def test_self_play_with_forced_playouts_plays_the_oracle_games(mode):
    """States, policies, values, flags and plies of every game; the resigning run's threshold is below every value, so nothing
    resigns and its record is the one without resignation."""
    games, sims, seed, k = 6, 12, 41, 2.0
    kw = MODES[mode]
    rec = self_play.play_batch_device(hash_evaluator, games, sims=sims, seed=seed, forced_k=k, **kw)
    flags, plies = rec["flags"].cpu().numpy(), rec["plies"].cpu().numpy()
    game, ply, value = rec["game"].cpu().numpy(), rec["ply"].cpu().numpy(), rec["value"].cpu().numpy()
    for g, (states, pol) in enumerate(_record_games(rec, games)):
        o = mf.play_game(hash_predict, sims, seed, g, k, temperature=kw["temperature"], reuse=kw.get("tree_reuse", False),
                         alpha=kw.get("dirichlet_alpha"), v_resign=kw.get("resign_threshold"), calibration=kw.get("resign_calibration", 0.0))
        assert states == o["states"], (mode, g)
        for j in range(len(states)):
            assert np.array_equal(pol[j], o["policy"][j]), (mode, g, j)
        idx = np.nonzero(game == g)[0]
        assert value[idx[np.argsort(ply[idx])]].tolist() == o["value"], (mode, g)
        assert int(flags[g]) == o["flags"] and int(plies[g]) == o["plies"], (mode, g)
        if "resign_threshold" in kw:
            assert rec["resign_min"][g].tolist() == o["resign_min"], (mode, g)
    if "resign_threshold" in kw:
        off = self_play.play_batch_device(hash_evaluator, games, sims=sims, seed=seed, forced_k=k,
                                          **{a: b for a, b in kw.items() if not a.startswith("resign")})
        for key in SHARED:
            assert torch.equal(rec[key], off[key]), key
        assert not ((rec["flags"] & 4) != 0).any()


def test_zero_k_is_the_search_without_forcing(mcts_golden, roots):
    sims = 50
    packed = torch.cat([pack(golden_states(mcts_golden, "hash")), roots]).contiguous()
    plain, a0, n0 = pv_mcts.BatchedMCTS(hash_evaluator, sims).search(packed)
    zero, a1, n1 = pv_mcts.BatchedMCTS(hash_evaluator, sims, forced_k=0.0).search(packed)
    assert torch.equal(plain, zero) and torch.equal(a0, a1) and torch.equal(n0, n1)
    for kw in (dict(temperature=1.0, dirichlet_alpha=0.3, tree_reuse=True), dict(temperature=0)):
        off = self_play.play_batch_device(hash_evaluator, 6, sims=16, seed=8, **kw)
        on = self_play.play_batch_device(hash_evaluator, 6, sims=16, seed=8, forced_k=0.0, **kw)
        for key in SHARED:
            assert torch.equal(on[key], off[key]), (kw, key)
        assert on["sims"] == off["sims"] and on["reused"] == off["reused"]


def test_a_game_does_not_depend_on_its_batch(roots):
    """Same (root, game id, seed, ply) at other rows, in other batches: identical raw and pruned counts."""
    sims, G, k = 20, roots.shape[0], 2.0
    gid = torch.arange(500, 500 + G, device="cuda")
    m1 = pv_mcts.BatchedMCTS(hash_evaluator, sims, dirichlet_alpha=0.3, forced_k=k)
    c1, _, _ = m1.search(roots, noise_seed=3, game_id=gid, ply=6)
    r1, _, _ = abi_counts(m1._ws[0], G, 1 + sims * MC)
    perm = torch.randperm(G, generator=torch.Generator().manual_seed(0)).cuda()
    extra = positions.random_positions(9, seed=5, games=64)
    m2 = pv_mcts.BatchedMCTS(hash_evaluator, sims, dirichlet_alpha=0.3, forced_k=k)
    c2, _, _ = m2.search(torch.cat([extra, roots[perm]]).contiguous(), noise_seed=3,
                         game_id=torch.cat([torch.arange(9, device="cuda"), gid[perm]]), ply=6)
    r2, _, _ = abi_counts(m2._ws[0], G + 9, 1 + sims * MC)
    assert torch.equal(c1[perm], c2[9:]) and torch.equal(r1[perm], r2[9:])
    one = pv_mcts.BatchedMCTS(hash_evaluator, sims, dirichlet_alpha=0.3, forced_k=k)
    c3, _, _ = one.search(roots[7:8], noise_seed=3, game_id=gid[7:8], ply=6)
    assert torch.equal(c3[0], c1[7])


def test_padded_batches_do_not_change_a_game():
    """The network path pads batches above 256 games to a multiple of 256: 300 and 320 real rows both run as 512."""
    torch.manual_seed(2)
    net = GNNNetwork().cuda().eval()
    net.precision = "fp32"
    sims, k = 8, 2.0
    roots = positions.random_positions(300, seed=8, games=64)
    gid = torch.arange(300, device="cuda") * 7
    m1 = pv_mcts.BatchedMCTS(net, sims, dirichlet_alpha=0.3, forced_k=k)
    c1, _, _ = m1.search(roots, noise_seed=12, game_id=gid, ply=1)
    r1, _, _ = abi_counts(m1._ws[0], 512, 1 + sims * MC)
    perm = torch.randperm(300, generator=torch.Generator().manual_seed(1)).cuda()
    roots2 = torch.cat([roots[perm], positions.random_positions(20, seed=9, games=64)]).contiguous()
    gid2 = torch.cat([gid[perm], torch.arange(20, device="cuda") + 5000])
    m2 = pv_mcts.BatchedMCTS(net, sims, dirichlet_alpha=0.3, forced_k=k)
    c2, _, _ = m2.search(roots2, noise_seed=12, game_id=gid2, ply=1)
    r2, _, _ = abi_counts(m2._ws[0], 512, 1 + sims * MC)
    assert torch.equal(c1[perm], c2[:300]) and torch.equal(r1[:300][perm], r2[:300])


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_network_graph_replay_equals_eager_loop_with_forced_playouts(mcts_golden, prec):
    torch.manual_seed(1)
    net = GNNNetwork().cuda().eval()
    net.precision = prec
    roots0 = pack(golden_states(mcts_golden, "hash"))
    gid0 = torch.arange(roots0.shape[0], device="cuda") + 40
    graph = pv_mcts.BatchedMCTS(net, 40, use_graph=True, dirichlet_alpha=0.3, forced_k=2.0)
    eager = pv_mcts.BatchedMCTS(net, 40, use_graph=False, dirichlet_alpha=0.3, forced_k=2.0)
    kw = dict(noise_seed=21, game_id=gid0, ply=2)
    c1, a1, n1 = graph.search(roots0, **kw)
    c2, a2, n2 = eager.search(roots0, **kw)
    c3, _, _ = graph.search(roots0, **kw)
    assert graph.use_graph and graph._graphs and torch.equal(c1, c2) and torch.equal(a1, a2) and torch.equal(n1, n2)
    assert torch.equal(c1, c3)
    assert all(key[-1] == "forced" for key in graph._graphs)
    raw, _, _ = abi_counts(graph._ws[0], roots0.shape[0], 1 + 40 * MC)
    assert int(raw.sum(1).min()) == 39 and bool((c1.sum(1) <= 39).all())
    # tree reuse
    graph = pv_mcts.BatchedMCTS(net, 40, use_graph=True, tree_reuse=True, forced_k=2.0)
    eager = pv_mcts.BatchedMCTS(net, 40, use_graph=False, tree_reuse=True, forced_k=2.0)
    roots, src_row, path, carried = roots0, None, None, 0
    for ply in range(3):
        c1, a1, n1 = graph.search(roots, src_row=src_row, path=path)
        c2, a2, n2 = eager.search(roots, src_row=src_row, path=path)
        assert torch.equal(c1, c2) and torch.equal(a1, a2) and torch.equal(n1, n2), (prec, ply)
        if src_row is not None:
            assert torch.equal(graph.last_kept, eager.last_kept)
            carried += int((graph.last_kept > 0).sum())
        best = torch.gather(a1, 1, torch.argmax(c1, 1, keepdim=True)).squeeze(1)
        nxt, term = gl.next_batch(roots, best)
        alive = torch.nonzero(term == 0).squeeze(1)
        roots, src_row, path = nxt[alive].contiguous(), alive, best[alive].reshape(-1, 1)
    assert graph.use_graph and carried > 0


def test_bad_arguments_are_refused(roots):
    L = _lib.load()
    G, max_nodes = roots.shape[0], 1 + 2 * MC
    ws = fresh_ws(roots, max_nodes)
    st = _lib.stream_ptr()
    leaf = torch.empty((G, gl.STATE_BYTES), dtype=torch.uint8, device="cuda")
    kind = torch.empty((G,), dtype=torch.int32, device="cuda")
    out = uniform_evaluator(roots)
    counts = torch.empty((G, gl.MAX_LEGAL), dtype=torch.int32, device="cuda")
    actions = torch.empty((G, gl.MAX_LEGAL), dtype=torch.int16, device="cuda")
    n = torch.empty((G,), dtype=torch.int16, device="cuda")
    leaves = (P(out["priors"]), P(out["value"]), P(out["mask"]), P(out["pawn"]))

    def calls(k, g=G, w=ws):
        return (L.aq_mcts_select_forced(P(w), g, max_nodes, 1.25, k, P(leaf), P(kind), st),
                L.aq_mcts_expand_select_forced(P(w), g, max_nodes, *leaves, 1.25, k, P(leaf), P(kind), st),
                L.aq_mcts_root_counts_pruned(P(w), g, max_nodes, 1.25, k, P(counts), P(actions), P(n), None, st))

    assert calls(0.0) == (0, 0, 0) and calls(2.0) == (0, 0, 0)
    for k in (-0.5, -1e-30, float("nan"), float("inf"), float("-inf")):
        assert calls(k) == (-1, -1, -1), k
        with pytest.raises(_lib.AqError):
            _lib.check(calls(k)[2], "aq_mcts_root_counts_pruned")
    assert calls(2.0, g=0) == (-1, -1, -1) and calls(2.0, w=None) == (-1, -1, -1)
    assert L.aq_mcts_root_counts_pruned(P(ws), G, max_nodes, 1.25, 2.0, None, P(actions), P(n), None, st) == -1
    for kw in (dict(forced_k=-1.0), dict(forced_k=float("nan")), dict(forced_k=float("inf")), dict(forced_k=True),
               dict(forced_k=2.0, gumbel_considered=4)):
        with pytest.raises(ValueError):
            pv_mcts.BatchedMCTS(hash_evaluator, 8, **kw)
    with pytest.raises(ValueError):
        self_play.play_batch_device(hash_evaluator, 2, sims=2, forced_k=-2.0)
    torch.cuda.synchronize()


def test_a_forced_search_runs_as_many_launches_as_a_plain_one(roots):
    L = _lib.load()
    for kw in (dict(), dict(dirichlet_alpha=0.3), dict(tree_reuse=True)):
        counts = []
        for k in (None, 2.0):
            mcts = pv_mcts.BatchedMCTS(uniform_evaluator, 6, forced_k=k, **kw)
            mcts.search(roots)   # lazy set-up outside the count
            c0 = L.aq_launch_count()
            mcts.search(roots)
            counts.append(L.aq_launch_count() - c0)
        assert counts[0] == counts[1], kw
    torch.cuda.synchronize()
