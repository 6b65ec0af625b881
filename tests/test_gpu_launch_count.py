"""How many kernels each entry point launches: the aq_launch_count() delta of one eager call.  bench.py reports gpu_launches from
the same counter, so these numbers pin both which kernels an entry point runs for its arguments and that every launch is counted."""
import pytest
import torch

from alphaquoridorgnn_b200 import _lib, positions, train_network
from alphaquoridorgnn_b200 import game_logic as gl
from alphaquoridorgnn_b200.pv_network_gnn import GNNNetwork

pytestmark = pytest.mark.gpu

P = _lib.ptr
SIMS = 4
MAX_NODES = 1 + 2 * SIMS * 133   # room for a carried subtree (pv_mcts.BatchedMCTS with tree_reuse)


def launches(call, what):
    """Kernels the library launched during call(), which returns the entry point's status."""
    L = _lib.load()
    c0 = L.aq_launch_count()
    _lib.check(call(), what)
    n = L.aq_launch_count() - c0
    torch.cuda.synchronize()
    return n


@pytest.fixture(scope="module")
def net():
    torch.manual_seed(0)
    return GNNNetwork().cuda().eval()


@pytest.fixture(scope="module")
def boards():
    return positions.random_positions(16384, seed=7)


def leaf_outputs(B):
    L = _lib.load()
    return dict(priors=torch.empty((B, 209), device="cuda"), value=torch.empty((B,), device="cuda"),
                mask=torch.empty((B, 8), dtype=torch.int32, device="cuda"), pawn=torch.empty((B, 8), dtype=torch.uint8, device="cuda"),
                ws=torch.empty((L.aq_leaf_eval_ws_floats(B),), device="cuda"))


def leaf_eval(net, packed, prec, out):
    """-> the call of aq_leaf_eval (the weights, and at precision 1 their prepared tiles, are made ready before it)."""
    L = _lib.load()
    flat, prep = P(net.flat_parameters()), P(net.prepared_weights()) if prec == 1 else None
    return lambda: L.aq_leaf_eval(flat, prep, P(packed), packed.shape[0], P(out["priors"]), P(out["value"]), P(out["mask"]), P(out["pawn"]),
                                  P(out["ws"]), prec, _lib.stream_ptr())


@pytest.mark.parametrize("prec,B,want", [(1, 256, 3), (1, 16384, 2), (0, 16384, 4)])
def test_leaf_eval(net, boards, prec, B, want):
    assert launches(leaf_eval(net, boards[:B], prec, leaf_outputs(B)), "aq_leaf_eval") == want


@pytest.mark.parametrize("B,with_ws,want", [(16384, True, 2), (256, False, 1)])
def test_legal_mask(boards, B, with_ws, want):
    L = _lib.load()
    packed = boards[:B]
    mask = torch.empty((B, 8), dtype=torch.int32, device="cuda")
    pawn = torch.empty((B, 8), dtype=torch.uint8, device="cuda")
    ws = torch.empty((L.aq_legal_mask_ws_bytes(B),), dtype=torch.uint8, device="cuda") if with_ws else None
    call = lambda: L.aq_legal_mask_ws(P(packed), B, P(mask), P(pawn), P(ws), ws.numel() if with_ws else 0, _lib.stream_ptr())
    assert launches(call, "aq_legal_mask_ws") == want


@pytest.mark.parametrize("B,want", [(0, 1), (300, 2)])
def test_compact_priors(net, boards, B, want):
    L = _lib.load()
    out = leaf_outputs(max(B, 1))
    if B:
        _lib.check(leaf_eval(net, boards[:B], 0, out)(), "aq_leaf_eval")
    offsets = torch.empty((B + 1,), dtype=torch.int32, device="cuda")
    compact = torch.empty((max(B, 1) * gl.MAX_LEGAL,), device="cuda")
    call = lambda: L.aq_compact_priors(P(out["priors"]), P(out["mask"]), P(out["pawn"]), B, P(offsets), P(compact), _lib.stream_ptr())
    assert launches(call, "aq_compact_priors") == want


def training_forward(net, packed, prec):
    L = _lib.load()
    B = packed.shape[0]
    policy, value = torch.empty((B, 209), device="cuda"), torch.empty((B,), device="cuda")
    saved = torch.empty((L.aq_gnn_saved_floats(B),), device="cuda")
    _lib.check(L.aq_gnn_forward(P(net.flat_parameters()), P(packed), None, None, B, P(policy), P(value), P(saved), prec, _lib.stream_ptr()),
               "aq_gnn_forward")
    return saved


def test_gnn_forward(net, boards):
    L = _lib.load()
    B = 256
    policy, value = torch.empty((B, 209), device="cuda"), torch.empty((B,), device="cuda")
    call = lambda: L.aq_gnn_forward(P(net.flat_parameters()), P(boards[:B]), None, None, B, P(policy), P(value), None, 0, _lib.stream_ptr())
    assert launches(call, "aq_gnn_forward") == 2


@pytest.mark.parametrize("prec", [0, 1])
def test_gnn_backward(net, boards, prec):
    L = _lib.load()
    B = 256
    saved = training_forward(net, boards[:B], prec)
    dp, dv = torch.randn((B, 209), device="cuda") * 1e-3, torch.randn((B,), device="cuda") * 1e-3
    grads = torch.empty_like(net.flat_parameters())
    ws = torch.empty((L.aq_gnn_backward_ws_floats(B),), device="cuda")
    call = lambda: L.aq_gnn_backward(P(net.flat_parameters()), P(saved), P(dp), P(dv), B, P(grads), P(ws), prec, _lib.stream_ptr())
    assert launches(call, "aq_gnn_backward") == 4


@pytest.mark.parametrize("prec", [0, 1])
def test_train_backward_step(boards, prec):
    L = _lib.load()
    torch.manual_seed(1)
    model = GNNNetwork().cuda().train()
    B = 256
    saved = training_forward(model, boards[:B], prec)
    flat = model.flat_parameters()
    pt = torch.softmax(torch.randn((B, 209), device="cuda"), 1)
    vt = torch.randint(-1, 2, (B,), device="cuda").float()
    loss, grads = torch.empty((2,), device="cuda"), torch.empty_like(flat)
    m, v = torch.zeros_like(flat), torch.zeros_like(flat)
    ws = torch.empty((L.aq_gnn_backward_ws_floats(B),), device="cuda")
    comm = train_network.PeerCommunicator(0, 1, flat.device)
    try:
        call = lambda: L.aq_train_backward_step(comm.handle, P(flat), P(saved), P(pt), P(vt), B, B, P(loss), P(grads), P(m), P(v), P(ws),
                                                prec, 1e-3, 0.9, 0.999, 1e-8, _lib.stream_ptr())
        assert launches(call, "aq_train_backward_step") == 4
    finally:
        comm.close()


def test_mcts_and_selfplay(net, boards):
    """One search of SIMS simulations through the ABI, counting select and the fused expand + select; then the subtree of each root's
    most visited child is carried into a second workspace (aq_mcts_advance), and one self-play ply is taken from the counts."""
    L = _lib.load()
    st = _lib.stream_ptr()
    G = 64
    roots = boards[:G]
    ws = [torch.empty((L.aq_mcts_ws_bytes(G, MAX_NODES),), dtype=torch.uint8, device="cuda") for _ in range(2)]
    leaf = torch.empty((G, gl.STATE_BYTES), dtype=torch.uint8, device="cuda")
    kind = torch.empty((G,), dtype=torch.int32, device="cuda")
    out = leaf_outputs(G)
    _lib.check(L.aq_mcts_reset(P(ws[0]), P(roots), G, MAX_NODES, st), "aq_mcts_reset")
    assert launches(lambda: L.aq_mcts_select(P(ws[0]), G, MAX_NODES, 1.25, P(leaf), P(kind), st), "aq_mcts_select") == 1
    for i in range(SIMS):
        _lib.check(leaf_eval(net, leaf, 0, out)(), "aq_leaf_eval")
        args = (P(ws[0]), G, MAX_NODES, P(out["priors"]), P(out["value"]), P(out["mask"]), P(out["pawn"]))
        if i + 1 < SIMS:
            assert launches(lambda: L.aq_mcts_expand_select(*args, 1.25, P(leaf), P(kind), st), "aq_mcts_expand_select") == 1
        else:
            _lib.check(L.aq_mcts_expand_backup(*args, st), "aq_mcts_expand_backup")
    counts = torch.empty((G, gl.MAX_LEGAL), dtype=torch.int32, device="cuda")
    actions = torch.empty((G, gl.MAX_LEGAL), dtype=torch.int16, device="cuda")
    n = torch.empty((G,), dtype=torch.int16, device="cuda")
    _lib.check(L.aq_mcts_root_counts(P(ws[0]), G, MAX_NODES, P(counts), P(actions), P(n), None, st), "aq_mcts_root_counts")

    best = torch.gather(actions, 1, torch.argmax(counts, 1, keepdim=True)).contiguous()
    moved, _ = gl.next_batch(roots, best.squeeze(1))
    src = torch.arange(G, device="cuda")
    kept, status = torch.empty((G,), dtype=torch.int32, device="cuda"), torch.empty((1,), dtype=torch.int32, device="cuda")
    call = lambda: L.aq_mcts_advance(P(ws[0]), G, P(ws[1]), G, MAX_NODES, P(moved), P(src), P(best), 1, SIMS * 133, P(kept), P(status), st)
    assert launches(call, "aq_mcts_advance") == 1
    assert status.item() == 0 and (kept > 0).any()

    policy = torch.empty((G, 209), device="cuda")
    chosen = torch.empty((G,), dtype=torch.int16, device="cuda")
    nxt, nxt_id = torch.empty_like(roots), torch.empty((G,), dtype=torch.int64, device="cuda")
    flags, plies = torch.empty((G,), dtype=torch.uint8, device="cuda"), torch.empty((G,), dtype=torch.int64, device="cuda")
    alive = torch.empty((1,), dtype=torch.int32, device="cuda")
    sp_ws = torch.empty((L.aq_selfplay_ws_bytes(G),), dtype=torch.uint8, device="cuda")
    call = lambda: L.aq_selfplay_advance(P(roots), P(counts), P(actions), P(n), P(src), G, 1.0, 3, 0, P(policy), 0, P(chosen), P(nxt),
                                         P(nxt_id), P(flags), P(plies), P(alive), P(sp_ws), st)
    assert launches(call, "aq_selfplay_advance") == 2


@pytest.mark.parametrize("with_edges,want", [(False, 0), (True, 2)])
def test_edges_to_open_mask(boards, with_edges, want):
    L = _lib.load()
    B = 64
    ei = gl.build_graph_batch(boards[:B], with_edge_index=True)["edge_index"]
    E = ei.shape[1] if with_edges else 0
    open_mask = torch.empty(((B * 81 + 3) // 4 * 4,), dtype=torch.uint8, device="cuda")
    bad = torch.empty((1,), dtype=torch.int32, device="cuda")
    call = lambda: L.aq_edges_to_open_mask(P(ei[0]), P(ei[1]), E, B, P(open_mask), P(bad), _lib.stream_ptr())
    assert launches(call, "aq_edges_to_open_mask") == want
    assert bad.item() == 0
