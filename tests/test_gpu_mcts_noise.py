"""Root Dirichlet noise (aq_mcts_root_noise, BatchedMCTS(dirichlet_alpha=...), play_batch_device(dirichlet_alpha=...)) against the
CPU restatement in tests/mcts_noise_oracle.py.  Priors and values of the hash / uniform evaluators are bit-identical on both sides
and the noised priors are float32 values rounded once from double, so priors and visit counts are compared exactly."""
import numpy as np
import pytest
import torch

from alphaquoridorgnn_b200 import _lib, positions, pv_mcts, self_play
from alphaquoridorgnn_b200 import game_logic as gl
from alphaquoridorgnn_b200.pv_network_gnn import GNNNetwork
from oracle import mcts_oracle as mo

import mcts_noise_oracle as mn
from mcts_reuse_oracle import hash_predict, uniform_predict
from test_gpu_mcts import EVAL, hash_evaluator, uniform_evaluator
from test_gpu_mcts_reuse import _record_games, capacity, check_row, golden_states, oracle_states, pack

pytestmark = pytest.mark.gpu

PREDICT = {"hash": hash_predict, "uniform": uniform_predict}
MC = pv_mcts.MAX_CHILDREN
P = _lib.ptr


@pytest.fixture(scope="module")
def roots():
    """The start position and 40 random positions of mid-game depth."""
    start = pack([mo.COracleState()])
    return torch.cat([start, positions.random_positions(40, seed=21, games=64)]).contiguous()


def noise(ws, G, max_nodes, game_id, seed, ply, alpha, fraction, out=None):
    L = _lib.load()
    return L.aq_mcts_root_noise(P(ws), G, max_nodes, P(game_id), seed, ply, alpha, fraction, P(out), _lib.stream_ptr())


def root_priors(ws, G, max_nodes):
    """The root priors in the workspace (a second noise call is a no-op on a noised root; it only reads them out)."""
    out = torch.full((G, gl.MAX_LEGAL), float("nan"), device="cuda")
    _lib.check(noise(ws, G, max_nodes, None, 0, 0, 1.0, 0.5, out), "aq_mcts_root_noise")
    return out


def simulate(ws, G, max_nodes, evaluator, sims):
    L = _lib.load()
    st = _lib.stream_ptr()
    leaf = torch.empty((G, gl.STATE_BYTES), dtype=torch.uint8, device="cuda")
    kind = torch.empty((G,), dtype=torch.int32, device="cuda")
    for _ in range(sims):
        _lib.check(L.aq_mcts_select(P(ws), G, max_nodes, pv_mcts.C_PUCT, P(leaf), P(kind), st), "select")
        out = evaluator(leaf)
        _lib.check(L.aq_mcts_expand_backup(P(ws), G, max_nodes, P(out["priors"]), P(out["value"]), P(out["mask"]), P(out["pawn"]), st),
                   "expand_backup")


def fresh_ws(packed, max_nodes):
    L = _lib.load()
    G = packed.shape[0]
    ws = torch.empty((L.aq_mcts_ws_bytes(G, max_nodes),), dtype=torch.uint8, device="cuda")
    _lib.check(L.aq_mcts_reset(P(ws), P(packed), G, max_nodes, _lib.stream_ptr()), "aq_mcts_reset")
    return ws


def oracle_noised(state, gid, seed, ply, alpha, fraction):
    raw, _ = hash_predict(state)
    eta = mn.dirichlet(seed, [gid], ply, len(raw), alpha)[0]
    return mn.noised_priors(raw, eta, fraction), eta


@pytest.mark.parametrize("alpha", [0.03, 0.3, 1.0, 2.5])
def test_noised_root_priors_match_the_oracle(roots, alpha):
    """Fresh roots expanded by one simulation through the ABI.  At fraction 1 the kernel's float32 priors are float32(eta): they equal
    the oracle's eta rounded to float32, child by child."""
    G, max_nodes, seed, ply = roots.shape[0], 1 + 4 * MC, 0xC0FFEE, 17
    states = oracle_states(roots)
    gid = torch.arange(1000, 1000 + G, device="cuda")
    for fraction in (0.25, 1.0):
        ws = fresh_ws(roots, max_nodes)
        before = torch.full((G, gl.MAX_LEGAL), float("nan"), device="cuda")
        _lib.check(noise(ws, G, max_nodes, gid, seed, ply, alpha, fraction, before), "aq_mcts_root_noise")
        assert int(torch.count_nonzero(before)) == 0    # not expanded: nothing to noise, nothing noised
        simulate(ws, G, max_nodes, hash_evaluator, 1)
        got = torch.full((G, gl.MAX_LEGAL), float("nan"), device="cuda")
        _lib.check(noise(ws, G, max_nodes, gid, seed, ply, alpha, fraction, got), "aq_mcts_root_noise")
        got = got.cpu().numpy()
        for r, s in enumerate(states):
            want, eta = oracle_noised(s, 1000 + r, seed, ply, alpha, fraction)
            K = len(want)
            assert np.array_equal(got[r, :K], want), (alpha, fraction, r)
            assert not got[r, K:].any()
            if fraction == 1.0:
                assert np.abs(got[r, :K].astype(np.float64) - eta).max() <= 2.0 ** -24 * max(eta.max(), 1e-300)


def test_game_id_null_is_the_row_index(roots):
    G, max_nodes = roots.shape[0], 1 + 4 * MC
    out = []
    for gid in (None, torch.arange(G, device="cuda")):
        ws = fresh_ws(roots, max_nodes)
        simulate(ws, G, max_nodes, hash_evaluator, 1)
        pri = torch.empty((G, gl.MAX_LEGAL), device="cuda")
        _lib.check(noise(ws, G, max_nodes, gid, 5, 2, 0.3, 0.25, pri), "aq_mcts_root_noise")
        out.append(pri)
    assert torch.equal(out[0], out[1])


@pytest.mark.parametrize("name", ["hash", "uniform"])
def test_noised_search_matches_the_oracle(mcts_golden, roots, name):
    sims, seed, ply = 50, 77, 4
    states = golden_states(mcts_golden, name) + oracle_states(roots[:8])
    gids = [3 * r + 1 for r in range(len(states))]
    mcts = pv_mcts.BatchedMCTS(EVAL[name], sims, dirichlet_alpha=0.3)
    counts, actions, n = mcts.search(pack(states), noise_seed=seed, game_id=torch.tensor(gids), ply=ply)
    plain, _, _ = pv_mcts.BatchedMCTS(EVAL[name], sims).search(pack(states))
    for r, s in enumerate(states):
        o = mn.NoisedSearch(s, 0.3)
        o.search(PREDICT[name], sims, seed, gids[r], ply)
        check_row(counts, actions, n, r, o)
    if name == "hash":
        assert not torch.equal(counts, plain)


@pytest.mark.parametrize("name", ["hash", "uniform"])
def test_noised_search_with_reuse_matches_the_oracle(mcts_golden, name):
    """Greedy games with tree reuse: a carried root is noised before its first descent, with the key of the new ply."""
    sims, seed = 40, 9
    starts = [mo.COracleState()] + golden_states(mcts_golden, name)
    oracles = [mn.NoisedSearch(s, 0.3) for s in starts]
    mcts = pv_mcts.BatchedMCTS(EVAL[name], sims, tree_reuse=True, dirichlet_alpha=0.3)
    games, src_row, path, carried = list(range(len(starts))), None, None, 0
    for ply in range(8):
        counts, actions, n = mcts.search(pack([oracles[g].root.state for g in games]), src_row=src_row, path=path, noise_seed=seed,
                                         game_id=torch.tensor(games), ply=ply)
        if src_row is not None:
            carried += int((mcts.last_kept > 0).sum())
        nxt, src, pth = [], [], []
        for r, g in enumerate(games):
            o = oracles[g]
            o.search(PREDICT[name], sims, seed, g, ply)
            check_row(counts, actions, n, r, o)
            a = o.actions()[int(np.argmax(o.counts()))]
            o.advance([a], capacity(sims), sims * MC)
            if not o.root.state.is_done():
                nxt.append(g)
                src.append(r)
                pth.append([a])
        games = nxt
        src_row, path = torch.tensor(src, device="cuda"), torch.tensor(pth, dtype=torch.int16, device="cuda")
    assert carried > len(starts)


def test_zero_fraction_is_the_search_without_noise(mcts_golden, roots):
    sims = 50
    packed = torch.cat([pack(golden_states(mcts_golden, "hash")), roots]).contiguous()
    plain, a0, _ = pv_mcts.BatchedMCTS(hash_evaluator, sims).search(packed)
    zero, a1, _ = pv_mcts.BatchedMCTS(hash_evaluator, sims, dirichlet_alpha=0.03, noise_fraction=0.0).search(packed, noise_seed=1)
    assert torch.equal(plain, zero) and torch.equal(a0, a1)
    # and with reuse over a few plies
    m0 = pv_mcts.BatchedMCTS(hash_evaluator, 20, tree_reuse=True)
    m1 = pv_mcts.BatchedMCTS(hash_evaluator, 20, tree_reuse=True, dirichlet_alpha=0.3, noise_fraction=0.0)
    cur, src_row, path = roots, None, None
    for ply in range(3):
        c0, a0, _ = m0.search(cur, src_row=src_row, path=path)
        c1, _, _ = m1.search(cur, src_row=src_row, path=path, noise_seed=4, ply=ply)
        assert torch.equal(c0, c1), ply
        best = torch.gather(a0, 1, torch.argmax(c0, 1, keepdim=True)).squeeze(1)
        nxt, term = gl.next_batch(cur, best)
        alive = torch.nonzero(term == 0).squeeze(1)
        cur, src_row, path = nxt[alive].contiguous(), alive, best[alive].reshape(-1, 1)


def test_a_game_does_not_depend_on_its_batch(roots):
    """Same (root, game id, seed, ply) at other rows, in other batches: identical root priors and counts."""
    sims, G = 20, roots.shape[0]
    gid = torch.arange(500, 500 + G, device="cuda")
    m1 = pv_mcts.BatchedMCTS(hash_evaluator, sims, dirichlet_alpha=0.3)
    c1, _, _ = m1.search(roots, noise_seed=3, game_id=gid, ply=6)
    p1 = root_priors(m1._ws[0], G, 1 + sims * MC)
    perm = torch.randperm(G, generator=torch.Generator().manual_seed(0)).cuda()
    extra = positions.random_positions(9, seed=5, games=64)
    roots2 = torch.cat([extra, roots[perm]]).contiguous()
    gid2 = torch.cat([torch.arange(9, device="cuda"), gid[perm]])
    m2 = pv_mcts.BatchedMCTS(hash_evaluator, sims, dirichlet_alpha=0.3)
    c2, _, _ = m2.search(roots2, noise_seed=3, game_id=gid2, ply=6)
    p2 = root_priors(m2._ws[0], G + 9, 1 + sims * MC)
    assert torch.equal(c1[perm], c2[9:]) and torch.equal(p1[perm], p2[9:])
    one = pv_mcts.BatchedMCTS(hash_evaluator, sims, dirichlet_alpha=0.3)
    c3, _, _ = one.search(roots[7:8], noise_seed=3, game_id=gid[7:8], ply=6)
    assert torch.equal(c3[0], c1[7])


def test_padded_batches_do_not_change_a_game():
    """The network path pads batches above 256 games to a multiple of 256: 300 and 320 real rows both run as 512."""
    torch.manual_seed(2)
    net = GNNNetwork().cuda().eval()
    net.precision = "fp32"
    sims = 8
    roots = positions.random_positions(300, seed=8, games=64)
    gid = torch.arange(300, device="cuda") * 7
    m1 = pv_mcts.BatchedMCTS(net, sims, dirichlet_alpha=0.3)
    c1, _, _ = m1.search(roots, noise_seed=12, game_id=gid, ply=1)
    p1 = root_priors(m1._ws[0], 512, 1 + sims * MC)[:300]
    perm = torch.randperm(300, generator=torch.Generator().manual_seed(1)).cuda()
    roots2 = torch.cat([roots[perm], positions.random_positions(20, seed=9, games=64)]).contiguous()
    gid2 = torch.cat([gid[perm], torch.arange(20, device="cuda") + 5000])
    m2 = pv_mcts.BatchedMCTS(net, sims, dirichlet_alpha=0.3)
    c2, _, _ = m2.search(roots2, noise_seed=12, game_id=gid2, ply=1)
    p2 = root_priors(m2._ws[0], 512, 1 + sims * MC)[:300]
    assert torch.equal(c1[perm], c2[:300]) and torch.equal(p1[perm], p2)


def test_a_second_noise_call_is_a_no_op(roots):
    G, sims, max_nodes = roots.shape[0], 12, 1 + 12 * MC
    results = []
    for extra in (False, True):
        ws = fresh_ws(roots, max_nodes)
        simulate(ws, G, max_nodes, hash_evaluator, 1)
        first = torch.empty((G, gl.MAX_LEGAL), device="cuda")
        _lib.check(noise(ws, G, max_nodes, None, 1, 0, 0.3, 0.25, first), "aq_mcts_root_noise")
        if extra:   # another key, alpha and fraction: the roots are noised already
            again = torch.empty((G, gl.MAX_LEGAL), device="cuda")
            _lib.check(noise(ws, G, max_nodes, None, 2, 5, 2.5, 1.0, again), "aq_mcts_root_noise")
            assert torch.equal(first, again)
        simulate(ws, G, max_nodes, hash_evaluator, sims - 1)
        results.append(root_priors(ws, G, max_nodes))
        counts = torch.empty((G, gl.MAX_LEGAL), dtype=torch.int32, device="cuda")
        actions = torch.empty((G, gl.MAX_LEGAL), dtype=torch.int16, device="cuda")
        n = torch.empty((G,), dtype=torch.int16, device="cuda")
        _lib.check(_lib.load().aq_mcts_root_counts(P(ws), G, max_nodes, P(counts), P(actions), P(n), None, _lib.stream_ptr()), "counts")
        results.append(counts)
    assert torch.equal(results[0], results[2]) and torch.equal(results[1], results[3])


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_network_graph_replay_equals_eager_loop_with_noise(mcts_golden, prec):
    torch.manual_seed(1)
    net = GNNNetwork().cuda().eval()
    net.precision = prec
    roots0 = pack(golden_states(mcts_golden, "hash"))
    gid0 = torch.arange(roots0.shape[0], device="cuda") + 40
    # fresh roots: the first graph search runs simulation 1 eagerly (warm-up), the second replays the one-step graph for it
    graph = pv_mcts.BatchedMCTS(net, 40, use_graph=True, dirichlet_alpha=0.3)
    eager = pv_mcts.BatchedMCTS(net, 40, use_graph=False, dirichlet_alpha=0.3)
    kw = dict(noise_seed=21, game_id=gid0, ply=2)
    c1, a1, n1 = graph.search(roots0, **kw)
    c2, a2, n2 = eager.search(roots0, **kw)
    c3, _, _ = graph.search(roots0, **kw)
    plain, _, _ = pv_mcts.BatchedMCTS(net, 40, use_graph=True).search(roots0)
    assert graph.use_graph and torch.equal(c1, c2) and torch.equal(a1, a2) and torch.equal(n1, n2) and torch.equal(c1, c3)
    assert int(c1.sum(1).min()) == 39 and not torch.equal(c1, plain)
    # tree reuse
    graph = pv_mcts.BatchedMCTS(net, 40, use_graph=True, tree_reuse=True, dirichlet_alpha=0.3)
    eager = pv_mcts.BatchedMCTS(net, 40, use_graph=False, tree_reuse=True, dirichlet_alpha=0.3)
    roots, gid, src_row, path, carried = roots0, gid0, None, None, 0
    for ply in range(3):
        kw = dict(src_row=src_row, path=path, noise_seed=21, game_id=gid, ply=ply)
        c1, a1, n1 = graph.search(roots, **kw)
        c2, a2, n2 = eager.search(roots, **kw)
        assert torch.equal(c1, c2) and torch.equal(a1, a2) and torch.equal(n1, n2), (prec, ply)
        if src_row is not None:
            assert torch.equal(graph.last_kept, eager.last_kept)
            carried += int((graph.last_kept > 0).sum())
        best = torch.gather(a1, 1, torch.argmax(c1, 1, keepdim=True)).squeeze(1)
        nxt, term = gl.next_batch(roots, best)
        alive = torch.nonzero(term == 0).squeeze(1)
        roots, gid, src_row, path = nxt[alive].contiguous(), gid[alive], alive, best[alive].reshape(-1, 1)
    assert graph.use_graph and carried > 0


def _oracle_noised_game(sims, seed, g, reuse):
    o = mn.NoisedSearch(mo.COracleState(), 0.3)
    seen, ply = [], 0
    while not o.root.state.is_done():
        seen.append((o.root.state.row.tolist(), o.root.state.plies))
        o.search(hash_predict, sims, seed, g, ply)
        a = o.actions()[int(np.argmax(o.counts()))]
        if reuse:
            o.advance([a], capacity(sims), sims * MC)
        else:
            o = mn.NoisedSearch(o.root.state.next(a), 0.3)
        ply += 1
    return seen


@pytest.mark.parametrize("reuse", [False, True])
def test_greedy_self_play_with_noise_plays_the_oracle_games(reuse):
    sims, games, seed = 16, 8, 31
    plain = self_play.play_batch_device(hash_evaluator, games, sims=sims, temperature=0, seed=seed, tree_reuse=reuse)
    first = [s for s, _ in _record_games(plain, games)]
    assert all(s == first[0] for s in first)          # without noise every greedy game from the start position is the same
    rec = self_play.play_batch_device(hash_evaluator, games, sims=sims, temperature=0, dirichlet_alpha=0.3, seed=seed, tree_reuse=reuse)
    again = self_play.play_batch_device(hash_evaluator, games, sims=sims, temperature=0, dirichlet_alpha=0.3, seed=seed, tree_reuse=reuse)
    for k in ("states", "policy", "value", "game", "ply", "flags", "plies"):
        assert torch.equal(rec[k], again[k]), k
    assert rec["sims"] == again["sims"] and rec["reused"] == again["reused"]
    played = [s for s, _ in _record_games(rec, games)]
    assert len({str(s) for s in played}) > 1
    for g, states in enumerate(played):
        assert states == _oracle_noised_game(sims, seed, g, reuse), g


def test_bad_arguments_are_refused(roots):
    G, max_nodes = roots.shape[0], 1 + MC
    ws = fresh_ws(roots, max_nodes)
    for alpha, fraction in ((0.0, 0.25), (-0.3, 0.25), (float("nan"), 0.25), (float("inf"), 0.25), (0.3, -0.01), (0.3, 1.01),
                            (0.3, float("nan"))):
        assert noise(ws, G, max_nodes, None, 0, 0, alpha, fraction) == -1, (alpha, fraction)
        with pytest.raises(_lib.AqError):
            _lib.check(noise(ws, G, max_nodes, None, 0, 0, alpha, fraction), "aq_mcts_root_noise")
    assert noise(ws, 0, max_nodes, None, 0, 0, 0.3, 0.25) == -1
    assert _lib.load().aq_mcts_root_noise(None, G, max_nodes, None, 0, 0, 0.3, 0.25, None, _lib.stream_ptr()) == -1
    assert noise(ws, G, max_nodes, None, 0, 0, 0.3, 0.0) == 0 and noise(ws, G, max_nodes, None, 0, 0, 0.3, 1.0) == 0
    for kw in (dict(dirichlet_alpha=0.0), dict(dirichlet_alpha=float("nan")), dict(dirichlet_alpha=0.3, noise_fraction=1.5)):
        with pytest.raises(ValueError):
            pv_mcts.BatchedMCTS(hash_evaluator, 8, **kw)
    torch.cuda.synchronize()


def test_noise_is_one_launch_and_a_search_gains_two(roots):
    L = _lib.load()
    G, max_nodes = roots.shape[0], 1 + 4 * MC
    ws = fresh_ws(roots, max_nodes)
    for _ in range(2):   # before and after the roots are expanded
        c0 = L.aq_launch_count()
        _lib.check(noise(ws, G, max_nodes, None, 0, 0, 0.3, 0.25), "aq_mcts_root_noise")
        assert L.aq_launch_count() - c0 == 1
        simulate(ws, G, max_nodes, uniform_evaluator, 1)
    counts = []
    for alpha in (None, 0.3):
        mcts = pv_mcts.BatchedMCTS(uniform_evaluator, 4, dirichlet_alpha=alpha)
        mcts.search(roots)   # lazy set-up outside the count
        c0 = L.aq_launch_count()
        mcts.search(roots)
        counts.append(L.aq_launch_count() - c0)
    assert counts[1] == counts[0] + 2
    torch.cuda.synchronize()
