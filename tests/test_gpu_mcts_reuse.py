"""Tree reuse between moves (aq_mcts_advance, BatchedMCTS(tree_reuse=True), play_batch_device(tree_reuse=True)) against the CPU
restatement in tests/mcts_reuse_oracle.py.  Priors and values of the hash / uniform evaluators are bit-identical on both sides,
so every visit count is compared exactly."""
import copy

import numpy as np
import pytest
import torch

from alphaquoridorgnn_b200 import _lib, positions, pv_mcts, self_play
from alphaquoridorgnn_b200 import game_logic as gl
from alphaquoridorgnn_b200.pv_network_gnn import GNNNetwork
from oracle import mcts_oracle as mo

from mcts_reuse_oracle import ReuseSearch, hash_predict, node_count, uniform_predict
from test_gpu_mcts import EVAL, hash_evaluator

pytestmark = pytest.mark.gpu

PREDICT = {"hash": hash_predict, "uniform": uniform_predict}
MC = pv_mcts.MAX_CHILDREN


def capacity(sims):
    return 1 + 2 * sims * MC


def pack(states):
    return gl.pack_rows(np.stack([s.row for s in states]), np.array([s.plies for s in states], np.int16))


def oracle_states(packed):
    rows, plies = gl.unpack_rows(packed)
    return [mo.COracleState(r, int(p)) for r, p in zip(rows.cpu().numpy(), plies.cpu().numpy())]


def golden_states(mcts_golden, name, sims=50):
    return [mo.COracleState(np.array(c["row"], np.uint8), c["plies"]) for c in mcts_golden["roots"]
            if c["sims"] == sims and c["evaluator"] == name]


def check_row(counts, actions, n, r, o):
    k = int(n[r])
    assert actions[r, :k].tolist() == o.actions()
    assert counts[r, :k].tolist() == o.counts()


@pytest.mark.parametrize("name", ["hash", "uniform"])
def test_greedy_game_with_reuse_matches_the_oracle(mcts_golden, name):
    sims = 50
    starts = [mo.COracleState()] + golden_states(mcts_golden, name)
    oracles = [ReuseSearch(s) for s in starts]
    expect_kept = [0] * len(starts)
    mcts = pv_mcts.BatchedMCTS(EVAL[name], sims, tree_reuse=True)
    games, src_row, path, carried = list(range(len(starts))), None, None, 0
    for ply in range(12):
        counts, actions, n = mcts.search(pack([oracles[g].root.state for g in games]), src_row=src_row, path=path)
        kept = mcts.last_kept.tolist() if src_row is not None else [0] * len(games)
        nxt, src, pth = [], [], []
        for r, g in enumerate(games):
            o = oracles[g]
            n_before = o.root.n
            o.search(PREDICT[name], sims)
            check_row(counts, actions, n, r, o)
            assert int(counts[r].sum()) == n_before + sims - 1
            assert kept[r] == expect_kept[g], (ply, g)
            carried += kept[r] > 0
            a = o.actions()[int(np.argmax(o.counts()))]
            expect_kept[g] = o.advance([a], capacity(sims), sims * MC)
            if not o.root.state.is_done():
                nxt.append(g)
                src.append(r)
                pth.append([a])
        games = nxt
        src_row, path = torch.tensor(src, device="cuda"), torch.tensor(pth, dtype=torch.int16, device="cuda")
    assert carried > len(starts)   # the carried branch was exercised, not only fresh roots


def test_two_move_path_carries_a_visited_grandchild_and_refreshes_an_unvisited_one(mcts_golden):
    sims = 50
    starts = golden_states(mcts_golden, "hash")
    mcts = pv_mcts.BatchedMCTS(hash_evaluator, sims, tree_reuse=True)
    mcts.search(pack(starts))
    oracles, dst, src, pth, fresh_rows = [], [], [], [], []
    for r, s in enumerate(starts):
        o = ReuseSearch(s)
        o.search(hash_predict, sims)
        a = o.actions()[int(np.argmax(o.counts()))]
        child = o.root.child_nodes[o.actions().index(a)]
        la = child.state.legal_actions()
        visited = [b for b, c in zip(la, child.child_nodes) if c.n >= 1]
        unvisited = [b for b, c in zip(la, child.child_nodes) if c.n == 0]
        if not (visited and unvisited):   # a reply set the search covered completely, or left unvisited
            continue
        for b in (visited[0], unvisited[0]):
            oc = copy.deepcopy(o)
            kept = oc.advance([a, b], capacity(sims), sims * MC)
            assert (kept > 0) == (b == visited[0])
            if kept == 0:
                fresh_rows.append(len(dst))
            oracles.append((oc, kept))
            dst.append(oc.root.state)
            src.append(r)
            pth.append([a, b])
    assert len(fresh_rows) >= 4 and len(dst) == 2 * len(fresh_rows)
    counts, actions, n = mcts.search(pack(dst), src_row=torch.tensor(src), path=torch.tensor(pth, dtype=torch.int16))
    assert mcts.last_kept.tolist() == [k for _, k in oracles]
    for r, (o, _) in enumerate(oracles):
        o.search(hash_predict, sims)
        check_row(counts, actions, n, r, o)
    plain, _, _ = pv_mcts.BatchedMCTS(hash_evaluator, sims).search(pack([dst[r] for r in fresh_rows]))
    assert torch.equal(counts[fresh_rows], plain)


def test_batch_reshuffle_equals_each_game_searched_alone():
    sims = 30
    roots = positions.random_positions(37, seed=11, games=64)
    extra = positions.random_positions(5, seed=12, games=64)
    mcts = pv_mcts.BatchedMCTS(hash_evaluator, sims, tree_reuse=True)
    counts, actions, _ = mcts.search(roots)
    best = torch.gather(actions, 1, torch.argmax(counts, 1, keepdim=True)).squeeze(1)
    moved, term = gl.next_batch(roots, best)
    keep = [r for r in range(37) if r % 5 != 2 and int(term[r]) == 0]
    order = [keep[i] for i in np.random.default_rng(3).permutation(len(keep))]
    src = order[:10] + [-1] * 5 + order[10:]
    dst = torch.cat([moved[order[:10]], extra, moved[order[10:]]]).contiguous()
    path = torch.stack([best[s] if s >= 0 else best.new_zeros(()) for s in src]).reshape(-1, 1)
    c2, a2, n2 = mcts.search(dst, src_row=torch.tensor(src), path=path)
    kept = mcts.last_kept.tolist()
    assert sum(k > 0 for k in kept) >= 20 and all(kept[10 + i] == 0 for i in range(5))
    for r, s in enumerate(src):
        alone = pv_mcts.BatchedMCTS(hash_evaluator, sims, tree_reuse=True)
        if s >= 0:
            alone.search(roots[s:s + 1])
            c1, a1, n1 = alone.search(dst[r:r + 1], src_row=torch.tensor([0]), path=path[r:r + 1])
            assert alone.last_kept.tolist() == [kept[r]]
        else:
            c1, a1, n1 = alone.search(dst[r:r + 1])
        assert torch.equal(c1[0], c2[r]) and torch.equal(a1[0], a2[r]) and int(n1[0]) == int(n2[r]), r


def _advance(src_ws, G_src, dst_ws, G_dst, max_nodes, roots, src, path, reserve, kept, status):
    L, P = _lib.load(), _lib.ptr
    return L.aq_mcts_advance(P(src_ws), G_src, P(dst_ws), G_dst, max_nodes, P(roots), P(src), P(path),
                             path.shape[1] if path.dim() == 2 else 0, reserve, P(kept), P(status), _lib.stream_ptr())


def _search_abi(ws, G, max_nodes, evaluator, sims):
    L, P = _lib.load(), _lib.ptr
    st = _lib.stream_ptr()
    leaf = torch.empty((G, gl.STATE_BYTES), dtype=torch.uint8, device="cuda")
    kind = torch.empty((G,), dtype=torch.int32, device="cuda")
    for _ in range(sims):
        _lib.check(L.aq_mcts_select(P(ws), G, max_nodes, pv_mcts.C_PUCT, P(leaf), P(kind), st), "select")
        out = evaluator(leaf)
        _lib.check(L.aq_mcts_expand_backup(P(ws), G, max_nodes, P(out["priors"]), P(out["value"]), P(out["mask"]), P(out["pawn"]), st),
                   "expand_backup")
    return _root_counts(ws, G, max_nodes)


def _root_counts(ws, G, max_nodes):
    L, P = _lib.load(), _lib.ptr
    counts = torch.empty((G, gl.MAX_LEGAL), dtype=torch.int32, device="cuda")
    actions = torch.empty((G, gl.MAX_LEGAL), dtype=torch.int16, device="cuda")
    n = torch.empty((G,), dtype=torch.int16, device="cuda")
    _lib.check(L.aq_mcts_root_counts(P(ws), G, max_nodes, P(counts), P(actions), P(n), None, _lib.stream_ptr()), "root_counts")
    return counts, actions, n


def test_capacity_rule_through_the_abi(mcts_golden):
    sims = 20
    starts = golden_states(mcts_golden, "hash")[:3]
    mcts = pv_mcts.BatchedMCTS(hash_evaluator, sims, tree_reuse=True)
    counts, actions, n_src = mcts.search(pack(starts))
    slot, G_src = mcts._last
    src_ws, max_nodes = mcts._ws[slot], capacity(sims)
    L = _lib.load()
    dst_ws = torch.empty((L.aq_mcts_ws_bytes(1, max_nodes),), dtype=torch.uint8, device="cuda")
    kept = torch.empty((1,), dtype=torch.int32, device="cuda")
    status = torch.empty((1,), dtype=torch.int32, device="cuda")
    for r, s in enumerate(starts):
        o = ReuseSearch(s)
        o.search(hash_predict, sims)
        check_row(counts, actions, n_src, r, o)
        a = o.actions()[int(np.argmax(o.counts()))]
        child = o.root.child_nodes[o.actions().index(a)]
        size = node_count(child)   # the oracle's node count = the arena count the GPU reports in `kept`
        root = pack([child.state])
        src = torch.tensor([r], device="cuda")
        path = torch.tensor([[a]], dtype=torch.int16, device="cuda")
        # just fits: carried, with the child's counts as its root counts
        assert _advance(src_ws, G_src, dst_ws, 1, max_nodes, root, src, path, max_nodes - size, kept, status) == 0
        assert kept.tolist() == [size] and status.tolist() == [0]
        c, acts, n = _root_counts(dst_ws, 1, max_nodes)
        k = int(n[0])
        assert acts[0, :k].tolist() == child.state.legal_actions() and c[0, :k].tolist() == [x.n for x in child.child_nodes]
        # one node short: fresh root, and a search from it is a plain search
        assert _advance(src_ws, G_src, dst_ws, 1, max_nodes, root, src, path, max_nodes - size + 1, kept, status) == 0
        assert kept.tolist() == [0] and status.tolist() == [0]
        c, _, _ = _search_abi(dst_ws, 1, max_nodes, hash_evaluator, sims)
        plain, _, _ = pv_mcts.BatchedMCTS(hash_evaluator, sims).search(root)
        assert torch.equal(c, plain)


def test_bad_input_is_refused(mcts_golden):
    sims = 10
    starts = golden_states(mcts_golden, "hash")[:2]
    mcts = pv_mcts.BatchedMCTS(hash_evaluator, sims, tree_reuse=True)
    counts, actions, _ = mcts.search(pack(starts))
    a = int(actions[0, int(torch.argmax(counts[0]))])
    good = pack([starts[0].next(a)])
    path = torch.tensor([[a]], dtype=torch.int16)
    with pytest.raises(_lib.AqError):            # a root that is not where the path leads
        mcts.search(pack([starts[1]]), src_row=torch.tensor([0]), path=path)
    mcts.search(pack(starts))
    with pytest.raises(_lib.AqError):            # source game out of range
        mcts.search(good, src_row=torch.tensor([7]), path=path)
    mcts.search(pack(starts))
    with pytest.raises(_lib.AqError):
        mcts.search(good, src_row=torch.tensor([-2]), path=path)
    mcts.search(pack(starts))
    with pytest.raises(ValueError):              # more simulations than the arena was sized for
        mcts.search(good, sims=sims + 1, src_row=torch.tensor([0]), path=path)
    with pytest.raises(ValueError):
        pv_mcts.BatchedMCTS(hash_evaluator, None, tree_reuse=True)
    with pytest.raises(ValueError):
        pv_mcts.BatchedMCTS(hash_evaluator, sims).search(good, src_row=torch.tensor([0]), path=path)
    slot, G_src = mcts._last
    src_ws, max_nodes = mcts._ws[slot], capacity(sims)
    L = _lib.load()
    dst_ws = torch.empty((L.aq_mcts_ws_bytes(1, max_nodes),), dtype=torch.uint8, device="cuda")
    kept = torch.empty((1,), dtype=torch.int32, device="cuda")
    status = torch.zeros((1,), dtype=torch.int32, device="cuda")
    src, dpath = torch.tensor([0], device="cuda"), path.cuda()
    assert _advance(src_ws, G_src, dst_ws, 1, max_nodes, good, src, dpath, 0, kept, status) == 0
    assert status.tolist() == [0] and kept.tolist()[0] > 0
    assert _advance(src_ws, G_src, dst_ws, 1, max_nodes, good, src, dpath[:, :0], 0, kept, status) == -1         # path_len 0 (AQ_ERR_ARG)
    assert _advance(src_ws, G_src, src_ws, 1, max_nodes, good, src, dpath, 0, kept, status) == -1                  # same workspace
    assert _advance(src_ws, G_src, src_ws[64:], 1, max_nodes, good, src, dpath, 0, kept, status) == -1             # overlapping
    assert _advance(src_ws, G_src, dst_ws, 1, max_nodes, good, src, dpath, max_nodes, kept, status) == -1          # no room at all
    torch.cuda.synchronize()


def test_network_graph_replay_equals_eager_loop_with_reuse(mcts_golden):
    torch.manual_seed(1)
    net = GNNNetwork().cuda().eval()
    roots0 = pack(golden_states(mcts_golden, "hash"))
    for prec in ("fp32", "bf16"):
        net.precision = prec
        graph = pv_mcts.BatchedMCTS(net, 40, use_graph=True, tree_reuse=True)
        eager = pv_mcts.BatchedMCTS(net, 40, use_graph=False, tree_reuse=True)
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
        assert len(graph._graphs) >= 2   # one graph set per workspace: the key holds the workspace pointer


def _oracle_reuse_game(sims, follow=None):
    """Greedy (follow=None) or recorded (follow = list of actions) self-play of one game with reuse on the oracle.
    -> (positions searched, search counts per ply, searches that continued a carried tree)."""
    o = ReuseSearch(mo.COracleState())
    seen, counts, reused, kept, ply = [], [], 0, 0, 0
    while not o.root.state.is_done():
        seen.append((o.root.state.row.tolist(), o.root.state.plies))
        reused += kept > 0
        o.search(hash_predict, sims)
        counts.append(o.counts())
        if follow is None:
            a = o.actions()[int(np.argmax(o.counts()))]
        elif ply < len(follow):
            a = follow[ply]
        else:
            break
        kept = o.advance([a], capacity(sims), sims * MC)
        ply += 1
    return seen, counts, reused


def _record_games(rec, num_games):
    rows, plies = gl.unpack_rows(rec["states"])
    rows, plies = rows.cpu().numpy(), plies.cpu().numpy()
    game, ply = rec["game"].cpu().numpy(), rec["ply"].cpu().numpy()
    pol = rec["policy"].cpu().numpy()
    out = []
    for g in range(num_games):
        idx = np.nonzero(game == g)[0]
        idx = idx[np.argsort(ply[idx])]
        out.append(([(rows[i].tolist(), int(plies[i])) for i in idx], pol[idx]))
    return out


def test_self_play_with_reuse_plays_the_oracle_game():
    sims = 24
    rec = self_play.play_batch_device(hash_evaluator, 6, sims=sims, temperature=0, seed=0, tree_reuse=True)
    seen, _, reused = _oracle_reuse_game(sims)
    for g, (states, _) in enumerate(_record_games(rec, 6)):
        assert states == seen, g
        assert int(rec["plies"][g]) == len(seen)
    assert rec["reused"] == 6 * reused and reused > 0
    assert rec["sims"] == 6 * len(seen) * sims


def test_self_play_with_reuse_at_temperature_one_follows_the_oracle():
    """Sampled games of different lengths: survivors are mapped to their previous rows as games end."""
    sims = 12
    rec = self_play.play_batch_device(hash_evaluator, 6, sims=sims, temperature=1.0, seed=5, tree_reuse=True)
    lengths = set()
    for g, (states, pol) in enumerate(_record_games(rec, 6)):
        follow = []
        for (r0, p0), (r1, p1) in zip(states[:-1], states[1:]):
            s = mo.COracleState(np.array(r0, np.uint8), p0)
            follow += [a for a in s.legal_actions() if s.next(a).row.tolist() == r1]
        seen, counts, _ = _oracle_reuse_game(sims, follow)
        assert seen == states, g
        for k, c in enumerate(counts):
            la = mo.COracleState(np.array(states[k][0], np.uint8), states[k][1]).legal_actions()
            want = np.zeros(gl.NUM_ACTIONS)
            want[la] = np.array(c, np.float64) / float(sum(c))
            assert np.array_equal(pol[k], want), (g, k)
        lengths.add(len(states))
    assert len(lengths) > 1


def test_host_sampled_moves_at_temperature_one_match_the_oracle(mcts_golden):
    sims = 24
    starts = golden_states(mcts_golden, "hash")
    oracles = [ReuseSearch(s) for s in starts]
    rng = np.random.default_rng(7)
    mcts = pv_mcts.BatchedMCTS(hash_evaluator, sims, tree_reuse=True)
    games, src_row, path = list(range(len(starts))), None, None
    for ply in range(4):
        counts, actions, n = mcts.search(pack([oracles[g].root.state for g in games]), src_row=src_row, path=path)
        nxt, src, pth = [], [], []
        for r, g in enumerate(games):
            o = oracles[g]
            o.search(hash_predict, sims)
            check_row(counts, actions, n, r, o)
            c = np.array(o.counts(), np.float64)
            a = int(rng.choice(o.actions(), p=c / c.sum()))
            o.advance([a], capacity(sims), sims * MC)
            if not o.root.state.is_done():
                nxt.append(g)
                src.append(r)
                pth.append([a])
        games = nxt
        src_row, path = torch.tensor(src), torch.tensor(pth, dtype=torch.int16)
