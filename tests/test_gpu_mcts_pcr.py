"""Playout cap randomization (the prefix entry points aq_mcts_*_rows, aq_selfplay_partition, BatchedMCTS.search(fast_sims=...,
full_rows=...), play_batch_device(fast_sims=..., full_search_prob=...)).  A full row must be exactly the plain search of its root, a
fast row exactly the plain fast_sims search without noise, and self-play games exactly those of tests/mcts_pcr_oracle.py."""
import warnings

import numpy as np
import pytest
import torch

from alphaquoridorgnn_b200 import _lib, positions, pv_mcts, self_play
from alphaquoridorgnn_b200 import game_logic as gl
from alphaquoridorgnn_b200.pv_network_gnn import GNNNetwork
from oracle import mcts_oracle as mo

import mcts_forced_oracle as mf
import mcts_pcr_oracle as mp
from mcts_reuse_oracle import hash_predict, uniform_predict
from test_gpu_mcts import EVAL, hash_evaluator, uniform_evaluator
from test_gpu_mcts_forced import abi_counts, check
from test_gpu_mcts_reuse import _record_games, capacity, golden_states, pack

pytestmark = pytest.mark.gpu

PREDICT = {"hash": hash_predict, "uniform": uniform_predict}
MC = pv_mcts.MAX_CHILDREN
P = _lib.ptr
SHARED = ("states", "policy", "value", "game", "ply", "flags", "plies")


@pytest.fixture(scope="module")
def roots():
    """The start position and 23 random positions of mid-game depth."""
    return torch.cat([pack([mo.COracleState()]), positions.random_positions(23, seed=31, games=64)]).contiguous()


# ----------------------------------------------------------------------------------------------------------------------------------
# prefix entry points

def zero_ws(packed, max_nodes):
    """A workspace reset for these roots whose unused bytes are 0, so that two workspaces can be compared byte for byte."""
    L = _lib.load()
    G = packed.shape[0]
    ws = torch.zeros((L.aq_mcts_ws_bytes(G, max_nodes),), dtype=torch.uint8, device="cuda")
    _lib.check(L.aq_mcts_reset(P(ws), P(packed), G, max_nodes, _lib.stream_ptr()), "aq_mcts_reset")
    return ws


def ws_parts(ws, G, max_nodes):
    """(games [G,64], hot [G, max_nodes * 16], cold [G, max_nodes * 16]) byte views of a workspace laid out for G games."""
    off, half = (G * 64 + 255) // 256 * 256, G * max_nodes * 16
    return ws[:G * 64].view(G, 64), ws[off:off + half].view(G, -1), ws[off + half:off + 2 * half].view(G, -1)


def run_sims(ws, G, rows, max_nodes, evaluator, sims, k=None, noise=True):
    """sims simulations of games [0, rows) through the prefix entry points (rows None: the plain entry points on all G), with root
    noise before and after simulation 1, as a search runs them; -> (leaf states, leaf kinds)."""
    L, st = _lib.load(), _lib.stream_ptr()
    sfx, dims, n = ("", (G,), G) if rows is None else ("_rows", (G, rows), rows)
    mode = "" if k is None else "_forced"
    fk = () if k is None else (k,)
    sel, exs = getattr(L, "aq_mcts_select" + mode + sfx), getattr(L, "aq_mcts_expand_select" + mode + sfx)
    exb, nz = getattr(L, "aq_mcts_expand_backup" + sfx), getattr(L, "aq_mcts_root_noise" + sfx)
    leaf = torch.zeros((G, gl.STATE_BYTES), dtype=torch.uint8, device="cuda")
    kind = torch.zeros((G,), dtype=torch.int32, device="cuda")
    gid = torch.arange(G, device="cuda") * 5 + 1

    def block(steps):
        _lib.check(sel(P(ws), *dims, max_nodes, pv_mcts.C_PUCT, *fk, P(leaf), P(kind), st), "select")
        for i in range(steps):
            out = evaluator(leaf[:n])
            leaves = (P(ws), *dims, max_nodes, P(out["priors"]), P(out["value"]), P(out["mask"]), P(out["pawn"]))
            if i + 1 < steps:
                _lib.check(exs(*leaves, pv_mcts.C_PUCT, *fk, P(leaf), P(kind), st), "expand_select")
            else:
                _lib.check(exb(*leaves, st), "expand_backup")

    for steps in (1, sims - 1):
        if noise:
            _lib.check(nz(P(ws), *dims, max_nodes, P(gid), 7, 3, 0.3, 0.25, None, st), "root_noise")
        block(steps)
    return leaf, kind


@pytest.mark.parametrize("k", [None, 2.0])
def test_prefix_entry_points_over_all_rows_equal_the_plain_ones(roots, k):
    sims = 12
    G, max_nodes = roots.shape[0], 1 + sims * MC
    ws1, ws2 = zero_ws(roots, max_nodes), zero_ws(roots, max_nodes)
    l1, k1 = run_sims(ws1, G, None, max_nodes, hash_evaluator, sims, k)
    l2, k2 = run_sims(ws2, G, G, max_nodes, hash_evaluator, sims, k)
    assert torch.equal(ws1, ws2) and torch.equal(l1, l2) and torch.equal(k1, k2)


@pytest.mark.parametrize("k", [None, 2.0])
@pytest.mark.parametrize("rows", [1, 9, 23])
def test_prefix_entry_points_leave_the_other_rows_and_search_the_prefix(roots, k, rows):
    sims = 12
    G, max_nodes = roots.shape[0], 1 + sims * MC
    ws = zero_ws(roots, max_nodes)
    before = [t.clone() for t in ws_parts(ws, G, max_nodes)]
    leaf, kind = run_sims(ws, G, rows, max_nodes, hash_evaluator, sims, k)
    after = ws_parts(ws, G, max_nodes)
    for b, a in zip(before, after):
        assert torch.equal(a[rows:], b[rows:])
    alone = zero_ws(roots[:rows].contiguous(), max_nodes)
    leaf1, kind1 = run_sims(alone, rows, None, max_nodes, hash_evaluator, sims, k)
    for a, b in zip(ws_parts(ws, G, max_nodes), ws_parts(alone, rows, max_nodes)):
        assert torch.equal(a[:rows], b)
    assert torch.equal(leaf[:rows], leaf1) and torch.equal(kind[:rows], kind1)
    assert not leaf[rows:].any() and not kind[rows:].any()


def test_prefix_entry_points_refuse_rows_out_of_range(roots):
    L, st = _lib.load(), _lib.stream_ptr()
    G, max_nodes = roots.shape[0], 1 + 2 * MC
    ws = zero_ws(roots, max_nodes)
    leaf = torch.empty((G, gl.STATE_BYTES), dtype=torch.uint8, device="cuda")
    kind = torch.empty((G,), dtype=torch.int32, device="cuda")
    out = uniform_evaluator(roots)
    leaves = (P(out["priors"]), P(out["value"]), P(out["mask"]), P(out["pawn"]))

    def calls(rows):
        return (L.aq_mcts_select_rows(P(ws), G, rows, max_nodes, 1.25, P(leaf), P(kind), st),
                L.aq_mcts_select_forced_rows(P(ws), G, rows, max_nodes, 1.25, 2.0, P(leaf), P(kind), st),
                L.aq_mcts_expand_backup_rows(P(ws), G, rows, max_nodes, *leaves, st),
                L.aq_mcts_expand_select_rows(P(ws), G, rows, max_nodes, *leaves, 1.25, P(leaf), P(kind), st),
                L.aq_mcts_expand_select_forced_rows(P(ws), G, rows, max_nodes, *leaves, 1.25, 2.0, P(leaf), P(kind), st),
                L.aq_mcts_root_noise_rows(P(ws), G, rows, max_nodes, None, 1, 0, 0.3, 0.25, None, st))

    assert calls(G) == (0,) * 6 and calls(1) == (0,) * 6
    for rows in (0, -1, G + 1, 2 ** 40):
        assert calls(rows) == (-1,) * 6, rows
    torch.cuda.synchronize()


# ----------------------------------------------------------------------------------------------------------------------------------
# partition

def partition(states, gid, count, seed, ply, p):
    L = _lib.load()
    G = states.shape[0]
    out = torch.full_like(states, 0xEE)
    out_id = torch.full((G,), -5, dtype=torch.int64, device="cuda")
    out_row = torch.full((G,), -5, dtype=torch.int64, device="cuda")
    full = torch.full((1,), -9, dtype=torch.int32, device="cuda")
    rc = L.aq_selfplay_partition(P(states), P(gid), G, P(count), seed, ply, p, P(out), P(out_id), P(out_row), P(full), _lib.stream_ptr())
    return rc, out, out_id, out_row, full


def test_partition_matches_the_oracle_draw():
    G = 4000
    states = positions.random_positions(G, seed=3, games=64)
    gid = torch.arange(G, device="cuda") * 3 + 17
    for seed in (0, 12345, 2 ** 64 - 3):
        for ply in (0, 1, 7, 150):
            for p in (0.0, 0.1, 0.25, 0.6, 1.0):
                rc, out, out_id, out_row, full = partition(states, gid, None, seed, ply, p)
                assert rc == 0
                want, want_full = mp.partition(seed, gid.cpu().numpy(), ply, p)
                assert int(full) == want_full and out_row.cpu().numpy().tolist() == want.tolist(), (seed, ply, p)
                assert torch.equal(out_id, gid[out_row]) and torch.equal(out, states[out_row])


def test_partition_honours_the_device_count():
    L = _lib.load()
    G = 3000
    states = positions.random_positions(G, seed=4, games=64)
    gid = torch.arange(G, device="cuda") + 1000
    for n in (0, 1, 1023, 1024, 1025, 2500, G, G + 50):
        count = torch.tensor([n], dtype=torch.int32, device="cuda")
        c0 = L.aq_launch_count()
        rc, out, out_id, out_row, full = partition(states, gid, count, 99, 5, 0.3)
        assert rc == 0 and L.aq_launch_count() - c0 == 1
        m = min(n, G)
        want, want_full = mp.partition(99, gid[:m].cpu().numpy(), 5, 0.3)
        assert int(full) == want_full and out_row[:m].cpu().numpy().tolist() == want.tolist(), n
        assert torch.equal(out[:m], states[out_row[:m]]) and torch.equal(out_id[:m], gid[out_row[:m]])
        assert bool((out_row[m:] == -5).all()) and bool((out_id[m:] == -5).all()) and bool((out[m:] == 0xEE).all())


# ----------------------------------------------------------------------------------------------------------------------------------
# the search

def plain(evaluator, packed, sims, k, alpha=None, **kw):
    """(counts, actions, n, raw counts, root values) of a plain search of these roots."""
    m = pv_mcts.BatchedMCTS(evaluator, sims, dirichlet_alpha=alpha, forced_k=k)
    c, a, n = m.search(packed, **kw)
    raw = abi_counts(m._ws[0], packed.shape[0], 1 + sims * MC)[0]
    return c, a, n, raw, m.root_values()


def check_split(got, packed, evaluator, sims, fast, full, k, alpha, gid, seed, ply):
    c, a, n, raw, rv = got
    G = packed.shape[0]
    if full:
        want = plain(evaluator, packed[:full].contiguous(), sims, k, alpha, noise_seed=seed, game_id=gid[:full], ply=ply)
        for x, y in zip((c, a, n, raw, rv[0], rv[1]), want[:4] + want[4]):
            assert torch.equal(x[:full], y)
    if full < G:
        want = plain(evaluator, packed[full:].contiguous(), fast, k)
        for x, y in zip((c, a, n, raw, rv[0], rv[1]), want[:4] + want[4]):
            assert torch.equal(x[full:], y)


@pytest.mark.parametrize("name", ["hash", "uniform"])
@pytest.mark.parametrize("fast", [1, 4, 16])
@pytest.mark.parametrize("share", ["none", "one", "half", "all"])
def test_full_rows_are_plain_searches_and_fast_rows_plain_fast_searches(mcts_golden, roots, name, fast, share):
    sims, seed, ply, k, alpha = 16, 77, 4, 2.0, 0.3
    packed = torch.cat([pack(golden_states(mcts_golden, name)), roots]).contiguous()
    G = packed.shape[0]
    full = {"none": 0, "one": 1, "half": G // 2, "all": G}[share]
    gid = torch.arange(G, device="cuda") * 3 + 1
    m = pv_mcts.BatchedMCTS(EVAL[name], sims, dirichlet_alpha=alpha, forced_k=k)
    c, a, n = m.search(packed, noise_seed=seed, game_id=gid, ply=ply, fast_sims=fast, full_rows=full)
    raw = abi_counts(m._ws[0], G, 1 + sims * MC)[0]
    check_split((c, a, n, raw, m.root_values()), packed, EVAL[name], sims, fast, full, k, alpha, gid, seed, ply)


@pytest.mark.parametrize("name", ["hash", "uniform"])
def test_pcr_without_noise_or_forcing(mcts_golden, roots, name):
    sims, fast = 16, 4
    packed = torch.cat([pack(golden_states(mcts_golden, name)), roots]).contiguous()
    G = packed.shape[0]
    m = pv_mcts.BatchedMCTS(EVAL[name], sims)
    c, a, n = m.search(packed, fast_sims=fast, full_rows=G // 3)
    raw = abi_counts(m._ws[0], G, 1 + sims * MC)[0]
    assert torch.equal(raw, c)
    check_split((c, a, n, raw, m.root_values()), packed, EVAL[name], sims, fast, G // 3, None, None, torch.arange(G, device="cuda"), 0, 0)
    c2, a2, n2 = pv_mcts.BatchedMCTS(EVAL[name], sims).search(packed, fast_sims=sims, full_rows=G // 3)
    c3, a3, n3 = pv_mcts.BatchedMCTS(EVAL[name], sims).search(packed)
    assert torch.equal(c2, c3) and torch.equal(a2, a3) and torch.equal(n2, n3)


@pytest.mark.parametrize("name", ["hash", "uniform"])
def test_pcr_search_with_reuse_matches_the_oracle(mcts_golden, name):
    """Six plies of greedy games with tree reuse, noise and forced playouts; each ply the games are ordered full first by the draw."""
    sims, fast, seed, k, alpha, p = 20, 5, 9, 2.0, 0.3, 0.5
    starts = [mo.COracleState()] + golden_states(mcts_golden, name)
    oracles = [mf.ForcedSearch(s, k, alpha) for s in starts]
    mcts = pv_mcts.BatchedMCTS(EVAL[name], sims, tree_reuse=True, dirichlet_alpha=alpha, forced_k=k)
    games, prev, carried = list(range(len(starts))), None, 0
    for ply in range(6):
        order = [g for g in games if mp.is_full(seed, [g], ply, p)[0]]
        full = len(order)
        order += [g for g in games if not mp.is_full(seed, [g], ply, p)[0]]
        src_row = path = None
        if prev is not None:
            src_row = torch.tensor([prev[g][0] for g in order], device="cuda")
            path = torch.tensor([[prev[g][1]] for g in order], dtype=torch.int16, device="cuda")
        counts, actions, n = mcts.search(pack([oracles[g].root.state for g in order]), src_row=src_row, path=path, noise_seed=seed,
                                         game_id=torch.tensor(order, device="cuda"), ply=ply, fast_sims=fast, full_rows=full)
        raw, _, _ = abi_counts(mcts._ws[mcts._last[0]], len(order), capacity(sims))
        if src_row is not None:
            carried += int((mcts.last_kept > 0).sum())
        prev, games = {}, []
        for r, g in enumerate(order):
            o = oracles[g]
            o.alpha = alpha if r < full else None
            o.search(PREDICT[name], sims if r < full else fast, seed, g, ply)
            check(raw, actions, n, r, o, False)
            check(counts, actions, n, r, o, True)
            a = o.actions()[int(np.argmax(o.pruned()))]
            o.advance([a], capacity(sims), sims * MC)
            if not o.root.state.is_done():
                games.append(g)
                prev[g] = (r, a)
    assert carried > len(starts)


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_network_graph_replay_equals_eager_loop_with_pcr(prec):
    """700 rows, 300 full: the graph path lays them out as [300 full | 212 copies | 400 fast | 112 copies] = 1,024 rows and runs
    phase B over 512; the eager loop does not pad.  Then a second ply continues the trees."""
    torch.manual_seed(1)
    net = GNNNetwork().cuda().eval()
    net.precision = prec
    sims, fast, k, alpha, full = 8, 2, 2.0, 0.3, 300
    roots = positions.random_positions(700, seed=8, games=64)
    gid = torch.arange(700, device="cuda") * 7
    kw = dict(noise_seed=21, game_id=gid, ply=2, fast_sims=fast, full_rows=full)
    graph = pv_mcts.BatchedMCTS(net, sims, use_graph=True, tree_reuse=True, dirichlet_alpha=alpha, forced_k=k)
    eager = pv_mcts.BatchedMCTS(net, sims, use_graph=False, tree_reuse=True, dirichlet_alpha=alpha, forced_k=k)
    c1, a1, n1 = graph.search(roots, **kw)
    c2, a2, n2 = eager.search(roots, **kw)
    assert graph.use_graph and graph._root[1] == 1024 and eager._root[1] == 700
    assert any(key[0] == 1024 and key[-2:] == (512, "forced-rows") for key in graph._graphs)
    assert torch.equal(c1, c2) and torch.equal(a1, a2) and torch.equal(n1, n2)
    for x, y in zip(graph.root_values(), eager.root_values()):
        assert torch.equal(x, y)
    if prec == "fp32":   # a full row is the plain search of its root, a fast row the plain fast search without noise
        p = plain(net, roots[:full].contiguous(), sims, k, alpha, noise_seed=21, game_id=gid[:full], ply=2)
        assert torch.equal(c1[:full], p[0]) and torch.equal(a1[:full], p[1])
        p = plain(net, roots[full:].contiguous(), fast, k)
        assert torch.equal(c1[full:], p[0]) and torch.equal(a1[full:], p[1])
    # ply 3: the survivors, reordered so that other games are full; src_row names rows of the previous search in the caller's order
    best = torch.gather(a1, 1, torch.argmax(c1, 1, keepdim=True)).squeeze(1)
    nxt, term = gl.next_batch(roots, best)
    alive = torch.nonzero(term == 0).squeeze(1)
    alive = torch.cat([alive[alive >= 350], alive[alive < 350]])
    kw = dict(src_row=alive, path=best[alive].reshape(-1, 1), noise_seed=21, game_id=gid[alive], ply=3, fast_sims=fast, full_rows=320)
    c1, a1, n1 = graph.search(nxt[alive].contiguous(), **kw)
    c2, a2, n2 = eager.search(nxt[alive].contiguous(), **kw)
    assert torch.equal(c1, c2) and torch.equal(a1, a2) and torch.equal(n1, n2)
    assert torch.equal(graph.last_kept, eager.last_kept) and int((graph.last_kept > 0).sum()) > 300
    assert graph.use_graph


# ----------------------------------------------------------------------------------------------------------------------------------
# self-play

MODES = {"t0-forced": dict(temperature=0, forced_k=2.0),
         "t1-noise": dict(temperature=1.0, dirichlet_alpha=0.3),
         "t0-reuse": dict(temperature=0, tree_reuse=True),
         "t1-noise-forced-reuse": dict(temperature=1.0, dirichlet_alpha=0.3, forced_k=2.0, tree_reuse=True),
         "t1-noise-forced-resign": dict(temperature=1.0, dirichlet_alpha=0.3, forced_k=2.0, resign_threshold=-0.3, resign_calibration=0.25)}


@pytest.mark.parametrize("mode", list(MODES))
def test_self_play_with_pcr_plays_the_oracle_games(mode):
    games, sims, fast, p, seed = 6, 12, 3, 0.5, 41
    kw = MODES[mode]
    rec = self_play.play_batch_device(hash_evaluator, games, sims=sims, seed=seed, fast_sims=fast, full_search_prob=p, **kw)
    flags, plies = rec["flags"].cpu().numpy(), rec["plies"].cpu().numpy()
    game, ply, value = rec["game"].cpu().numpy(), rec["ply"].cpu().numpy(), rec["value"].cpu().numpy()
    n_full = n_fast = 0
    for g, (states, pol) in enumerate(_record_games(rec, games)):
        o = mp.play_game(hash_predict, sims, fast, p, seed, g, temperature=kw["temperature"], reuse=kw.get("tree_reuse", False),
                         alpha=kw.get("dirichlet_alpha"), k=kw.get("forced_k"), v_resign=kw.get("resign_threshold"),
                         calibration=kw.get("resign_calibration", 0.0))
        assert states == o["states"], (mode, g)
        assert len(pol) == len(o["policy"]) and all(np.array_equal(a, b) for a, b in zip(pol, o["policy"])), (mode, g)
        idx = np.nonzero(game == g)[0]
        idx = idx[np.argsort(ply[idx])]
        assert ply[idx].tolist() == o["ply"] and value[idx].tolist() == o["value"], (mode, g)
        assert int(flags[g]) == o["flags"] and int(plies[g]) == o["plies"], (mode, g)
        if "resign_threshold" in kw:
            assert rec["resign_min"][g].tolist() == o["resign_min"], (mode, g)
        n_full, n_fast = n_full + o["full"], n_fast + o["fast"]
    assert (rec["full_searches"], rec["fast_searches"]) == (n_full, n_fast) and n_full and n_fast
    assert rec["sims"] == n_full * sims + n_fast * fast
    if "resign_threshold" in kw:
        assert ((rec["flags"] & 4) != 0).any()


def test_all_full_is_the_record_without_pcr():
    for kw in (dict(temperature=1.0, dirichlet_alpha=0.3, forced_k=2.0, tree_reuse=True), dict(temperature=0)):
        off = self_play.play_batch_device(hash_evaluator, 6, sims=12, seed=8, **kw)
        on = self_play.play_batch_device(hash_evaluator, 6, sims=12, seed=8, fast_sims=3, full_search_prob=1.0, **kw)
        for key in SHARED:
            assert torch.equal(on[key], off[key]), (kw, key)
        assert (on["sims"], on["reused"], on["full_searches"], on["fast_searches"]) == (off["sims"], off["reused"], off["full_searches"], 0)


def test_no_full_move_records_nothing_and_plays_the_fast_games():
    on = self_play.play_batch_device(hash_evaluator, 6, sims=12, seed=8, temperature=1.0, dirichlet_alpha=0.3, forced_k=2.0,
                                     fast_sims=3, full_search_prob=0.0)
    off = self_play.play_batch_device(hash_evaluator, 6, sims=3, seed=8, temperature=1.0, forced_k=2.0)
    assert on["states"].shape[0] == 0 and on["policy"].shape[0] == 0 and on["value"].shape[0] == 0
    assert torch.equal(on["flags"], off["flags"]) and torch.equal(on["plies"], off["plies"])
    assert (on["full_searches"], on["fast_searches"], on["sims"]) == (0, off["full_searches"], off["sims"])


def test_a_game_does_not_depend_on_its_batch():
    kw = dict(sims=10, seed=17, temperature=1.0, dirichlet_alpha=0.3, forced_k=2.0, tree_reuse=True, fast_sims=2, full_search_prob=0.4)
    small = self_play.play_batch_device(hash_evaluator, 4, **kw)
    big = self_play.play_batch_device(hash_evaluator, 9, **kw)
    for (s1, p1), (s2, p2) in zip(_record_games(small, 4), _record_games(big, 4)):
        assert s1 == s2 and np.array_equal(p1, p2)
    assert torch.equal(small["flags"], big["flags"][:4]) and torch.equal(small["plies"], big["plies"][:4])


def test_play_batch_history_holds_only_full_positions():
    games, seed, p = 6, 5, 0.3
    history, info = self_play.play_batch(hash_evaluator, games, sims=8, seed=seed, fast_sims=2, full_search_prob=p)
    want = sum(int(mp.is_full(seed, [g], np.arange(info["plies"][g]), p).sum()) for g in range(games))
    assert len(history) == want and 0 < want < int(info["plies"].sum())
    rec = self_play.play_batch_device(hash_evaluator, games, sims=8, seed=seed, fast_sims=2, full_search_prob=p)
    rows = [r for states, _ in _record_games(rec, games) for r, _ in states]
    assert [h[0] for h in history] == [[r[0:2], r[2:4], r[4:]] for r in rows]
    assert all(abs(sum(h[1]) - 1.0) < 1e-9 for h in history)


# ----------------------------------------------------------------------------------------------------------------------------------
# arguments, launches, synchronisations

def test_bad_arguments_are_refused(roots):
    L = _lib.load()
    G = roots.shape[0]
    m = pv_mcts.BatchedMCTS(hash_evaluator, 8)
    for kw in (dict(fast_sims=0), dict(fast_sims=9), dict(fast_sims=2.5), dict(fast_sims=True), dict(fast_sims=2, full_rows=-1),
               dict(fast_sims=2, full_rows=G + 1), dict(fast_sims=2, full_rows=1.5), dict(full_rows=3)):
        with pytest.raises(ValueError):
            m.search(roots, **kw)
    with pytest.raises(ValueError):
        pv_mcts.BatchedMCTS(hash_evaluator, 8, gumbel_considered=4).search(roots, fast_sims=2, full_rows=1)
    for kw in (dict(fast_sims=0), dict(fast_sims=3), dict(fast_sims=1, full_search_prob=float("nan")),
               dict(fast_sims=1, full_search_prob=-0.1), dict(fast_sims=1, full_search_prob=1.5), dict(fast_sims=1, gumbel_considered=4)):
        with pytest.raises(ValueError):
            self_play.play_batch_device(hash_evaluator, 2, sims=2, **kw)
    gid = torch.arange(G, device="cuda")
    for p in (float("nan"), -0.1, 1.5, float("inf")):
        assert partition(roots, gid, None, 1, 0, p)[0] == -1, p
    out = torch.empty_like(roots)
    ids = torch.empty_like(gid)
    full = torch.empty((1,), dtype=torch.int32, device="cuda")
    st = _lib.stream_ptr()
    assert L.aq_selfplay_partition(P(roots), P(gid), 0, None, 1, 0, 0.5, P(out), P(ids), P(ids), P(full), st) == -1
    assert L.aq_selfplay_partition(P(roots), P(gid), G, None, 1, 0, 0.5, P(out), P(ids), P(ids), None, st) == -1
    assert L.aq_selfplay_partition(None, P(gid), G, None, 1, 0, 0.5, P(out), P(ids), P(ids), P(full), st) == -1
    torch.cuda.synchronize()


def test_launches_and_synchronisations(roots):
    """A PCR search launches what an n-step search over all rows and an (N - n)-step search over the full rows launch together,
    less the second search's reset and counts read (one launch each); a PCR self-play ply still synchronises once."""
    L = _lib.load()
    G, sims, fast, full = roots.shape[0], 12, 4, 9

    def launches(f):
        f()   # lazy set-up outside the count
        c0 = L.aq_launch_count()
        f()
        return L.aq_launch_count() - c0

    for kw in (dict(), dict(forced_k=2.0), dict(tree_reuse=True)):
        m = pv_mcts.BatchedMCTS(uniform_evaluator, sims, **kw)
        a = launches(lambda: pv_mcts.BatchedMCTS(uniform_evaluator, fast, **kw).search(roots))
        b = launches(lambda: pv_mcts.BatchedMCTS(uniform_evaluator, sims - fast, **kw).search(roots[:full].contiguous()))
        assert launches(lambda: m.search(roots, fast_sims=fast, full_rows=full)) == a + b - 2, kw

    def syncs(**kw):
        with warnings.catch_warnings(record=True) as w:
            warnings.simplefilter("always")
            torch.cuda.set_sync_debug_mode("warn")
            try:
                self_play.play_batch_device(uniform_evaluator, 5, sims=6, seed=2, **kw)
            finally:
                torch.cuda.set_sync_debug_mode("default")
        return sum(str(x.message).startswith("called a synchronizing") for x in w)

    syncs(max_plies=1)   # the debug mode warns once about itself on first use
    for kw in (dict(), dict(tree_reuse=True, dirichlet_alpha=0.3)):
        plain_n = [syncs(max_plies=m, **kw) for m in (2, 3)]
        pcr_n = [syncs(max_plies=m, fast_sims=2, full_search_prob=0.5, **kw) for m in (2, 3)]
        assert pcr_n[1] - pcr_n[0] == plain_n[1] - plain_n[0], kw     # the same synchronisations per ply
        assert pcr_n[1] == plain_n[1] + 1, kw                          # and one more for the partition of the start states
    torch.cuda.synchronize()
