"""The Gumbel root (aq_mcts_gumbel_root, the _gumbel select kernels, aq_mcts_gumbel_result, BatchedMCTS(gumbel_considered=...),
play_batch_device(gumbel_considered=...)) against the CPU restatement in tests/mcts_gumbel_oracle.py.  Priors and values of the
hash / uniform evaluators are bit-identical on both sides and the root scores are float32 values rounded once from double, so root
scores, visit counts and choices are compared exactly; improved policies (an exp per child) within one float32 ulp."""
import numpy as np
import pytest
import torch

from alphaquoridorgnn_b200 import _lib, positions, pv_mcts, self_play
from alphaquoridorgnn_b200 import game_logic as gl
from alphaquoridorgnn_b200.pv_network_gnn import GNNNetwork
from oracle import mcts_oracle as mo

import mcts_gumbel_oracle as mg
from mcts_reuse_oracle import hash_predict, uniform_predict
from test_gpu_mcts import EVAL, hash_evaluator, uniform_evaluator
from test_gpu_mcts_noise import fresh_ws, simulate
from test_gpu_mcts_reuse import _record_games, golden_states, oracle_states, pack

pytestmark = pytest.mark.gpu

PREDICT = {"hash": hash_predict, "uniform": uniform_predict}
MC = pv_mcts.MAX_CHILDREN
P = _lib.ptr
ULPS = []   # measured improved-policy differences, in float32 ulps


@pytest.fixture(scope="module")
def roots():
    """The start position and 24 random positions of mid-game depth."""
    start = pack([mo.COracleState()])
    return torch.cat([start, positions.random_positions(24, seed=31, games=64)]).contiguous()


def gumbel_root(ws, G, max_nodes, game_id, seed, ply, considered, scale, sims, out=None):
    return _lib.load().aq_mcts_gumbel_root(P(ws), G, max_nodes, P(game_id), seed, ply, considered, scale, sims, P(out), _lib.stream_ptr())


def root_scores(ws, G, max_nodes):
    """The stored base scores (a second call is a no-op on a root with Gumbel state; it only reads them out)."""
    out = torch.full((G, gl.MAX_LEGAL), float("nan"), device="cuda")
    _lib.check(gumbel_root(ws, G, max_nodes, None, 0, 0, 1, 1.0, 1, out), "aq_mcts_gumbel_root")
    return out


def assert_policy_close(got, want):
    """got float32, want float64: within one float32 ulp of want, entry by entry."""
    got = np.asarray(got, np.float32)
    w32 = np.asarray(want).astype(np.float32)
    ulp = np.spacing(np.maximum(np.abs(w32), np.float32(np.finfo(np.float32).tiny)))
    d = np.abs(got.astype(np.float64) - np.asarray(want)) / ulp
    ULPS.append(float(d.max()) if d.size else 0.0)
    assert (np.abs(got - w32) <= ulp).all(), d.max()


@pytest.mark.parametrize("scale", [1.0, 0.0, 2.5])
def test_root_scores_match_the_oracle(roots, scale):
    G, max_nodes, seed, ply = roots.shape[0], 1 + 4 * MC, 0xBEEF, 9
    states = oracle_states(roots)
    gid = torch.arange(700, 700 + G, device="cuda")
    ws = fresh_ws(roots, max_nodes)
    before = torch.full((G, gl.MAX_LEGAL), float("nan"), device="cuda")
    _lib.check(gumbel_root(ws, G, max_nodes, gid, seed, ply, 4, scale, 8, before), "aq_mcts_gumbel_root")
    assert int(torch.count_nonzero(before)) == 0    # not expanded: no Gumbel state
    simulate(ws, G, max_nodes, hash_evaluator, 1)
    got = torch.full((G, gl.MAX_LEGAL), float("nan"), device="cuda")
    _lib.check(gumbel_root(ws, G, max_nodes, gid, seed, ply, 4, scale, 8, got), "aq_mcts_gumbel_root")
    got = got.cpu().numpy()
    for r, s in enumerate(states):
        raw, _ = hash_predict(s)
        want = mg.base_scores(raw, mg.gumbel_draw(seed, [700 + r], ply, len(raw), scale)[0])
        assert np.array_equal(got[r, :len(raw)], want), (scale, r)
        assert not got[r, len(raw):].any()


def _oracle_search(state, predict, considered, sims, seed, gid, ply, scale=1.0):
    o = mg.GumbelSearch(state, considered, scale)
    o.search(predict, sims, seed, gid, ply)
    return o


def check_gumbel_row(mcts, counts, actions, n, r, o):
    k = int(n[r])
    assert actions[r, :k].tolist() == o.actions()
    assert counts[r, :k].tolist() == o.counts()
    pol, choice = o.result()
    assert int(mcts.last_choice[r]) == choice
    got = mcts.last_policy[r].cpu().numpy()
    assert_policy_close(got[:k], pol)
    assert not got[k:].any()


@pytest.mark.parametrize("name", ["hash", "uniform"])
@pytest.mark.parametrize("sims", [1, 2, 16, 50])
@pytest.mark.parametrize("considered", [1, 2, 4, 16, 200])
def test_gumbel_search_matches_the_oracle(mcts_golden, roots, name, considered, sims):
    seed, ply = 77, 4
    states = golden_states(mcts_golden, name) + oracle_states(roots[:6])
    gids = [5 * r + 2 for r in range(len(states))]
    mcts = pv_mcts.BatchedMCTS(EVAL[name], sims, gumbel_considered=considered)
    counts, actions, n = mcts.search(pack(states), noise_seed=seed, game_id=torch.tensor(gids), ply=ply)
    assert mcts.last_policy.shape == (len(states), gl.MAX_LEGAL) and mcts.last_choice.dtype == torch.int16
    for r, s in enumerate(states):
        check_gumbel_row(mcts, counts, actions, n, r, _oracle_search(s, PREDICT[name], considered, sims, seed, gids[r], ply))
        assert int(counts[r].sum()) == sims - 1
        visited = int((counts[r] > 0).sum())
        assert visited <= min(considered, int(n[r]))


def test_zero_scale_is_deterministic_and_seed_independent(mcts_golden, roots):
    sims = 16
    states = golden_states(mcts_golden, "hash") + oracle_states(roots[:6])
    out = []
    for seed in (1, 2):
        mcts = pv_mcts.BatchedMCTS(hash_evaluator, sims, gumbel_considered=4, gumbel_scale=0.0)
        c, a, n = mcts.search(pack(states), noise_seed=seed, ply=seed)
        out.append((c, mcts.last_policy, mcts.last_choice))
        for r, s in enumerate(states):
            check_gumbel_row(mcts, c, a, n, r, _oracle_search(s, hash_predict, 4, sims, seed, r, seed, 0.0))
    assert all(torch.equal(x, y) for x, y in zip(*out))


def test_game_id_null_is_the_row_index(roots):
    out = []
    for gid in (None, torch.arange(roots.shape[0])):
        mcts = pv_mcts.BatchedMCTS(hash_evaluator, 12, gumbel_considered=4)
        out.append(mcts.search(roots, noise_seed=3, game_id=gid, ply=1)[0])
    assert torch.equal(out[0], out[1])


def test_a_game_does_not_depend_on_its_batch(roots):
    """Same (root, game id, seed, ply) at other rows, in other batches: identical root scores, counts, policies and choices."""
    sims, G = 20, roots.shape[0]
    gid = torch.arange(500, 500 + G, device="cuda")
    m1 = pv_mcts.BatchedMCTS(hash_evaluator, sims, gumbel_considered=8)
    c1, _, _ = m1.search(roots, noise_seed=3, game_id=gid, ply=6)
    s1 = root_scores(m1._ws[0], G, 1 + sims * MC)
    perm = torch.randperm(G, generator=torch.Generator().manual_seed(0)).cuda()
    extra = positions.random_positions(9, seed=5, games=64)
    roots2 = torch.cat([extra, roots[perm]]).contiguous()
    gid2 = torch.cat([torch.arange(9, device="cuda"), gid[perm]])
    m2 = pv_mcts.BatchedMCTS(hash_evaluator, sims, gumbel_considered=8)
    c2, _, _ = m2.search(roots2, noise_seed=3, game_id=gid2, ply=6)
    s2 = root_scores(m2._ws[0], G + 9, 1 + sims * MC)
    assert torch.equal(c1[perm], c2[9:]) and torch.equal(s1[perm], s2[9:])
    assert torch.equal(m1.last_policy[perm], m2.last_policy[9:]) and torch.equal(m1.last_choice[perm], m2.last_choice[9:])
    one = pv_mcts.BatchedMCTS(hash_evaluator, sims, gumbel_considered=8)
    c3, _, _ = one.search(roots[7:8], noise_seed=3, game_id=gid[7:8], ply=6)
    assert torch.equal(c3[0], c1[7]) and torch.equal(one.last_policy[0], m1.last_policy[7])


def test_padded_batches_do_not_change_a_game():
    """The network path pads batches above 256 games to a multiple of 256: 300 and 320 real rows both run as 512."""
    torch.manual_seed(2)
    net = GNNNetwork().cuda().eval()
    net.precision = "fp32"
    sims = 8
    roots = positions.random_positions(300, seed=8, games=64)
    gid = torch.arange(300, device="cuda") * 7
    m1 = pv_mcts.BatchedMCTS(net, sims, gumbel_considered=4)
    c1, _, _ = m1.search(roots, noise_seed=12, game_id=gid, ply=1)
    assert m1.last_policy.shape[0] == 300
    perm = torch.randperm(300, generator=torch.Generator().manual_seed(1)).cuda()
    roots2 = torch.cat([roots[perm], positions.random_positions(20, seed=9, games=64)]).contiguous()
    gid2 = torch.cat([gid[perm], torch.arange(20, device="cuda") + 5000])
    m2 = pv_mcts.BatchedMCTS(net, sims, gumbel_considered=4)
    c2, _, _ = m2.search(roots2, noise_seed=12, game_id=gid2, ply=1)
    assert torch.equal(c1[perm], c2[:300])
    assert torch.equal(m1.last_policy[perm], m2.last_policy[:300]) and torch.equal(m1.last_choice[perm], m2.last_choice[:300])


def test_a_second_init_call_is_a_no_op(roots):
    L = _lib.load()
    G, sims, max_nodes = roots.shape[0], 12, 1 + 12 * MC
    results = []
    for extra in (False, True):
        ws = fresh_ws(roots, max_nodes)
        simulate(ws, G, max_nodes, hash_evaluator, 1)
        first = torch.empty((G, gl.MAX_LEGAL), device="cuda")
        _lib.check(gumbel_root(ws, G, max_nodes, None, 1, 0, 4, 1.0, sims, first), "aq_mcts_gumbel_root")
        if extra:   # another key, considered, scale and budget: the roots have their Gumbel state already
            again = torch.empty((G, gl.MAX_LEGAL), device="cuda")
            _lib.check(gumbel_root(ws, G, max_nodes, None, 2, 5, 16, 3.0, 40, again), "aq_mcts_gumbel_root")
            assert torch.equal(first, again)
        mcts = pv_mcts.BatchedMCTS(hash_evaluator, sims)
        buf = {"leaf": torch.empty((G, gl.STATE_BYTES), dtype=torch.uint8, device="cuda"),
               "kind": torch.empty((G,), dtype=torch.int32, device="cuda")}
        for _ in range(sims - 1):
            mcts._step(ws, G, max_nodes, buf, lambda s: hash_evaluator(buf["leaf"]), _lib.stream_ptr(), 1, gumbel=True)
        counts = torch.empty((G, gl.MAX_LEGAL), dtype=torch.int32, device="cuda")
        actions = torch.empty((G, gl.MAX_LEGAL), dtype=torch.int16, device="cuda")
        n = torch.empty((G,), dtype=torch.int16, device="cuda")
        _lib.check(L.aq_mcts_root_counts(P(ws), G, max_nodes, P(counts), P(actions), P(n), None, _lib.stream_ptr()), "counts")
        policy = torch.empty((G, gl.MAX_LEGAL), device="cuda")
        choice = torch.empty((G,), dtype=torch.int16, device="cuda")
        _lib.check(L.aq_mcts_gumbel_result(P(ws), G, max_nodes, P(policy), P(choice), _lib.stream_ptr()), "result")
        results.append((counts, policy, choice))
    assert all(torch.equal(x, y) for x, y in zip(*results))


def test_roots_without_gumbel_state_search_with_puct(roots):
    """The _gumbel kernels on roots that never got Gumbel state run PUCT; the result reports policy 0 and choice -1."""
    L = _lib.load()
    G, sims = roots.shape[0], 10
    plain, _, _ = pv_mcts.BatchedMCTS(hash_evaluator, sims).search(roots)
    mcts = pv_mcts.BatchedMCTS(hash_evaluator, sims)
    max_nodes = 1 + sims * MC
    ws = fresh_ws(roots, max_nodes)
    buf = {"leaf": torch.empty((G, gl.STATE_BYTES), dtype=torch.uint8, device="cuda"),
           "kind": torch.empty((G,), dtype=torch.int32, device="cuda")}
    mcts._step(ws, G, max_nodes, buf, lambda s: hash_evaluator(buf["leaf"]), _lib.stream_ptr(), sims, gumbel=True)
    counts = torch.empty((G, gl.MAX_LEGAL), dtype=torch.int32, device="cuda")
    actions = torch.empty((G, gl.MAX_LEGAL), dtype=torch.int16, device="cuda")
    n = torch.empty((G,), dtype=torch.int16, device="cuda")
    _lib.check(L.aq_mcts_root_counts(P(ws), G, max_nodes, P(counts), P(actions), P(n), None, _lib.stream_ptr()), "counts")
    policy = torch.full((G, gl.MAX_LEGAL), 1.0, device="cuda")
    choice = torch.zeros((G,), dtype=torch.int16, device="cuda")
    _lib.check(L.aq_mcts_gumbel_result(P(ws), G, max_nodes, P(policy), P(choice), _lib.stream_ptr()), "result")
    assert torch.equal(counts, plain) and not policy.any() and bool((choice == -1).all())


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_network_graph_replay_equals_eager_loop_with_gumbel(mcts_golden, prec):
    torch.manual_seed(1)
    net = GNNNetwork().cuda().eval()
    net.precision = prec
    roots = pack(golden_states(mcts_golden, "hash"))
    gid = torch.arange(roots.shape[0], device="cuda") + 40
    # the first graph search runs each step mode's first simulation eagerly (warm-up), the second replays graphs only
    graph = pv_mcts.BatchedMCTS(net, 40, use_graph=True, gumbel_considered=8)
    eager = pv_mcts.BatchedMCTS(net, 40, use_graph=False, gumbel_considered=8)
    kw = dict(noise_seed=21, game_id=gid, ply=2)
    c1, a1, n1 = graph.search(roots, **kw)
    p1, ch1 = graph.last_policy, graph.last_choice
    c2, a2, n2 = eager.search(roots, **kw)
    c3, _, _ = graph.search(roots, **kw)
    plain, _, _ = pv_mcts.BatchedMCTS(net, 40, use_graph=True).search(roots)
    assert graph.use_graph and torch.equal(c1, c2) and torch.equal(a1, a2) and torch.equal(n1, n2) and torch.equal(c1, c3)
    assert torch.equal(p1, eager.last_policy) and torch.equal(ch1, eager.last_choice)
    assert torch.equal(p1, graph.last_policy) and torch.equal(ch1, graph.last_choice)
    assert int(c1.sum(1).min()) == 39 and not torch.equal(c1, plain)
    assert torch.allclose(p1.sum(1).double(), torch.ones(p1.shape[0], dtype=torch.float64, device="cuda"), atol=1e-5)


def _oracle_gumbel_game(sims, considered, seed, g, max_plies):
    s, seen, pols, ply = mo.COracleState(), [], [], 0
    while not s.is_done() and ply < max_plies:
        seen.append((s.row.tolist(), s.plies))
        o = _oracle_search(s, hash_predict, considered, sims, seed, g, ply)
        pol, choice = o.result()
        dense = np.zeros(gl.NUM_ACTIONS)
        dense[o.actions()] = pol
        pols.append(dense)
        s = s.next(o.actions()[choice])
        ply += 1
    L = len(seen)
    fpv = (-1.0 if L % 2 == 0 else 1.0) if s.is_lose() else 0.0
    return seen, pols, [fpv if k % 2 == 0 else -fpv for k in range(L)]


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_gumbel_self_play_plays_the_oracle_games(dtype):
    sims, games, seed, considered, max_plies = 16, 6, 31, 4, 8
    rec = self_play.play_batch_device(hash_evaluator, games, sims=sims, seed=seed, max_plies=max_plies, policy_dtype=dtype,
                                      gumbel_considered=considered)
    again = self_play.play_batch_device(hash_evaluator, games, sims=sims, seed=seed, max_plies=max_plies, policy_dtype=dtype,
                                        gumbel_considered=considered, temperature=0)
    for k in ("states", "policy", "value", "game", "ply", "flags", "plies"):
        assert torch.equal(rec[k], again[k]), k   # temperature plays no part
    assert rec["policy"].dtype == dtype
    played = _record_games(rec, games)
    assert len({str(s) for s, _ in played}) > 1
    game, value = rec["game"].cpu().numpy(), rec["value"].cpu().numpy()
    ply = rec["ply"].cpu().numpy()
    for g, (states, pol) in enumerate(played):
        seen, want_pol, want_val = _oracle_gumbel_game(sims, considered, seed, g, max_plies)
        assert states == seen, g
        for k in range(len(seen)):
            assert_policy_close(pol[k].astype(np.float32), want_pol[k])
        idx = np.nonzero(game == g)[0]
        assert value[idx[np.argsort(ply[idx])]].tolist() == want_val, g


def test_gumbel_self_play_to_the_end():
    """Whole games: every game ends, values are +-1 or 0, and every recorded policy is a distribution."""
    rec = self_play.play_batch_device(hash_evaluator, 4, sims=8, seed=3, gumbel_considered=4)
    assert bool((rec["flags"] != 0).all())
    assert torch.allclose(rec["policy"].sum(1), torch.ones(rec["policy"].shape[0], dtype=torch.float64, device="cuda"), atol=1e-6)
    assert set(rec["value"].tolist()) <= {-1.0, 0.0, 1.0}


def test_bad_arguments_are_refused(roots):
    L = _lib.load()
    G, max_nodes = roots.shape[0], 1 + MC
    ws = fresh_ws(roots, max_nodes)
    for considered, scale, sims in ((0, 1.0, 8), (-1, 1.0, 8), (4, -0.5, 8), (4, float("nan"), 8), (4, float("inf"), 8), (4, 1.0, 0),
                                    (4, 1.0, -3)):
        assert gumbel_root(ws, G, max_nodes, None, 0, 0, considered, scale, sims) == -1, (considered, scale, sims)
        with pytest.raises(_lib.AqError):
            _lib.check(gumbel_root(ws, G, max_nodes, None, 0, 0, considered, scale, sims), "aq_mcts_gumbel_root")
    assert gumbel_root(ws, 0, max_nodes, None, 0, 0, 4, 1.0, 8) == -1
    assert L.aq_mcts_gumbel_root(None, G, max_nodes, None, 0, 0, 4, 1.0, 8, None, _lib.stream_ptr()) == -1
    assert gumbel_root(ws, G, max_nodes, None, 0, 0, 1, 0.0, 1) == 0
    pol = torch.empty((G, gl.MAX_LEGAL), device="cuda")
    ch = torch.empty((G,), dtype=torch.int16, device="cuda")
    assert L.aq_mcts_gumbel_result(P(ws), G, max_nodes, None, P(ch), _lib.stream_ptr()) == -1
    assert L.aq_mcts_gumbel_result(P(ws), G, max_nodes, P(pol), None, _lib.stream_ptr()) == -1
    assert L.aq_mcts_gumbel_result(P(ws), 0, max_nodes, P(pol), P(ch), _lib.stream_ptr()) == -1
    leaf = torch.empty((G, gl.STATE_BYTES), dtype=torch.uint8, device="cuda")
    assert L.aq_mcts_select_gumbel(P(ws), G, max_nodes, 1.25, P(leaf), None, _lib.stream_ptr()) == -1
    assert L.aq_selfplay_advance_chosen(None, P(pol), P(ch), None, None, None, G, 0, None, 0, None, None, None, None, None, None, None,
                                        _lib.stream_ptr()) == -1
    for kw in (dict(gumbel_considered=0), dict(gumbel_considered=2.5), dict(gumbel_considered=True),
               dict(gumbel_considered=4, gumbel_scale=-1.0), dict(gumbel_considered=4, gumbel_scale=float("nan")),
               dict(gumbel_considered=4, gumbel_scale=float("inf")), dict(gumbel_considered=4, tree_reuse=True),
               dict(gumbel_considered=4, dirichlet_alpha=0.3)):
        with pytest.raises(ValueError):
            pv_mcts.BatchedMCTS(hash_evaluator, 8, **kw)
    torch.cuda.synchronize()


def test_launch_counts(roots):
    L = _lib.load()
    G, sims, max_nodes = roots.shape[0], 4, 1 + 4 * MC
    ws = fresh_ws(roots, max_nodes)
    simulate(ws, G, max_nodes, uniform_evaluator, 1)
    leaf = torch.empty((G, gl.STATE_BYTES), dtype=torch.uint8, device="cuda")
    kind = torch.empty((G,), dtype=torch.int32, device="cuda")
    pol = torch.empty((G, gl.MAX_LEGAL), device="cuda")
    ch = torch.empty((G,), dtype=torch.int16, device="cuda")
    calls = [lambda: gumbel_root(ws, G, max_nodes, None, 0, 0, 4, 1.0, sims),
             lambda: L.aq_mcts_select_gumbel(P(ws), G, max_nodes, 1.25, P(leaf), P(kind), _lib.stream_ptr()),
             lambda: L.aq_mcts_gumbel_result(P(ws), G, max_nodes, P(pol), P(ch), _lib.stream_ptr())]
    for call in calls:
        c0 = L.aq_launch_count()
        _lib.check(call(), "gumbel entry point")
        assert L.aq_launch_count() - c0 == 1
    out = uniform_evaluator(leaf)
    c0 = L.aq_launch_count()
    _lib.check(L.aq_mcts_expand_select_gumbel(P(ws), G, max_nodes, P(out["priors"]), P(out["value"]), P(out["mask"]), P(out["pawn"]),
                                              1.25, P(leaf), P(kind), _lib.stream_ptr()), "aq_mcts_expand_select_gumbel")
    assert L.aq_launch_count() - c0 == 1
    counts = []
    for considered in (None, 4):
        mcts = pv_mcts.BatchedMCTS(uniform_evaluator, sims, gumbel_considered=considered)
        mcts.search(roots)   # lazy set-up outside the count
        c0 = L.aq_launch_count()
        mcts.search(roots)
        counts.append(L.aq_launch_count() - c0)
    assert counts[1] == counts[0] + 2
    # aq_selfplay_advance_chosen: two launches, as aq_selfplay_advance
    n = torch.full((G,), 2, dtype=torch.int16, device="cuda")
    actions = torch.zeros((G, gl.MAX_LEGAL), dtype=torch.int16, device="cuda")
    gid = torch.arange(G, device="cuda")
    dense = torch.empty((G, gl.NUM_ACTIONS), dtype=torch.float64, device="cuda")
    nxt, nxt_id = torch.empty_like(roots), torch.empty_like(gid)
    ff, fp = torch.zeros(G, dtype=torch.uint8, device="cuda"), torch.zeros(G, dtype=torch.int64, device="cuda")
    alive = torch.zeros(1, dtype=torch.int32, device="cuda")
    sp_ws = torch.empty((L.aq_selfplay_ws_bytes(G),), dtype=torch.uint8, device="cuda")
    c0 = L.aq_launch_count()
    _lib.check(L.aq_selfplay_advance_chosen(P(roots), P(pol), P(ch.zero_()), P(actions), P(n), P(gid), G, 0, P(dense), 1, None, P(nxt),
                                            P(nxt_id), P(ff), P(fp), P(alive), P(sp_ws), _lib.stream_ptr()), "aq_selfplay_advance_chosen")
    assert L.aq_launch_count() - c0 == 2
    torch.cuda.synchronize()


def test_report_policy_ulps():
    """Runs last in the module: the largest improved-policy difference measured above, in float32 ulps."""
    if ULPS:
        print(f"\ngumbel improved policy: max difference {max(ULPS):.3f} float32 ulp over {len(ULPS)} rows")
