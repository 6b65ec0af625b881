"""The leaf evaluation (aq_leaf_eval: legal mask, GCN trunk, policy / value heads) at every batch-size branch of its kernels, board by
board.

The launch shapes (trunk grid and passes, heads tiles, fp32 heads grid cap, legal-mask lanes, fused legal warpgroup rounds, the ragged
prior scan's pieces) are chosen from the batch size; tests/leaf_probes.py lists the boundaries.  A board's arithmetic does not depend
on where it sits in the batch, so at every size:
  placement   the batch in order, rotated by one and reversed gives bit-identical priors, value, mask and pawn for every board once the
              order is undone, and the probe boards (leaf_probes.probe_positions) are bit-identical to the same board evaluated alone;
              mask and pawn equal the golden data; every output word is written (outputs start as NaN / -1 / 0xAB);
  content     every board against the oracle in the content metric of leaf_probes (legal log-probabilities and value):
                fp32 (precision 0)  vs the exact fp64 oracle,            bar 1e-5 (NVIDIA B200 at 1,000 W: worst 3.3e-7 log-prob,
                                    1.3e-7 value);
                bf16 (precision 1)  vs the fp64 rounding-point oracle,   bar 5e-3 (gnn_oracle.forward_tc_emulation; B200: worst 1.7e-3
                                    log-prob, 6.1e-4 value over the 20,000 boards -- an fp32 accumulator that rounds to the other
                                    bf16 / fp16 neighbour than the fp64 one moves a board by this much; the same emulation run in
                                    fp32 on the CPU is 6e-4 from the fp64 one on 3,000 of these boards);
              priors of illegal actions are exactly 0.  The measured worst board of each size is printed;
  callers     predict_batch, HostLeafEvaluator (f32 wire: the exact gather of the dense priors, f16: the same values rounded to half;
              offsets the running popcount of the mask) and, around the two-chunk threshold, aq_leaf_eval_host with a context are
              bit-identical to aq_leaf_eval.
The ragged-prior scan (legal_count_scan_kernel, pieces of 16,384 boards with a running carry) is checked at up to 50,001 boards
through aq_compact_priors and the host compact path.  The network is leaf_probes.leaf_model(); the fp32 bar is >= 100x below the
distance to the reference of any board a placement mistake would use (tests/test_oracle_leaf_probes.py).  The bf16 bar is not: there
placement rests on the bit-identity checks alone."""
import ctypes
import time

import numpy as np
import pytest
import torch

from alphaquoridorgnn_b200 import _lib
from alphaquoridorgnn_b200 import game_logic as gl
from alphaquoridorgnn_b200.pv_network_gnn import GNNNetwork, HostLeafEvaluator
from oracle import quoridor_oracle as qo

import leaf_probes as lp
import train_probes as tp

pytestmark = pytest.mark.gpu
PREC = {"fp32": 0, "bf16": 1, "bf16-raw": 1}   # bf16-raw: precision 1 without the prepared weight tiles (each CTA builds its own)
RAW_SIZES = (5, 593, 4097, 9473)
CASES = [(B, m) for B in lp.LEAF_BATCH_SIZES for m in ("fp32", "bf16")] + [(B, "bf16-raw") for B in RAW_SIZES]


@pytest.fixture(scope="module")
def leaf(traj):
    t0 = time.perf_counter()
    ref = lp.leaf_model()
    net = GNNNetwork()
    net.load_state_dict(ref.state_dict())
    net = net.cuda().eval()

    class Ctx:
        pass
    c = Ctx()
    c.net, c.flat = net, net.flat_parameters()
    c.rows, c.plies, c.mask, c.pawn = traj["rows"], traj["plies"], traj["mask"], traj["pawn"]
    c.perm = tp.permutation(traj["rows"])
    n = max(lp.LEAF_BATCH_SIZES)
    c.ids = c.perm[:n]
    c.legal = lp.dense_legal(traj["mask"][c.ids])
    exact, v_exact = lp.oracle_outputs(ref, traj["rows"][c.ids])
    emul, v_emul = lp.oracle_outputs(ref, traj["rows"][c.ids], emulate_tc=True)
    c.want = {0: (lp.restrict(exact, c.legal), v_exact), 1: (lp.restrict(emul, c.legal), v_emul)}
    la = qo.legal_actions_batch(traj["rows"][c.ids], traj["plies"][c.ids])
    c.actions, c.nact = la["actions"], la["n"].astype(np.int64)
    c.packed = gl.pack_rows(traj["rows"][c.ids], traj["plies"][c.ids], "cuda")
    c.alone = {}   # (row id, mode) -> outputs of a one-board evaluation
    print(f"\nleaf-eval oracle for {n} boards: {time.perf_counter() - t0:.1f} s")
    yield c
    print(f"\ntests/test_gpu_leaf_eval_batch_regimes.py: wall time {time.perf_counter() - t0:.1f} s")


def _leaf(net, packed, mode):
    """aq_leaf_eval; outputs start as garbage so that every word must be written."""
    L, P = _lib.load(), _lib.ptr
    B = packed.shape[0]
    pri = torch.full((B, 209), float("nan"), device="cuda")
    val = torch.full((B,), float("nan"), device="cuda")
    msk = torch.full((B, 8), -1, dtype=torch.int32, device="cuda")
    pwn = torch.full((B, 8), 0xAB, dtype=torch.uint8, device="cuda")
    ws = torch.empty((L.aq_leaf_eval_ws_floats(B),), device="cuda")
    prep = net.prepared_weights() if mode == "bf16" else None
    _lib.check(L.aq_leaf_eval(P(net.flat_parameters()), P(prep), P(packed), B, P(pri), P(val), P(msk), P(pwn), P(ws), PREC[mode],
                              _lib.stream_ptr()), "aq_leaf_eval")
    return pri, val, msk, pwn


def _bits(out):
    pri, val, msk, pwn = out
    return pri.view(torch.int32), val.view(torch.int32), msk, pwn


def _same(a, b):
    return all(torch.equal(x, y) for x, y in zip(_bits(a), _bits(b)))


def _ragged(dense, actions, nact):
    """Dense priors [B,209] gathered in legal_actions() order."""
    B = len(nact)
    take = np.arange(actions.shape[1])[None, :] < nact[:, None]
    return dense[np.repeat(np.arange(B), nact), actions[take].astype(np.int64)]


@pytest.mark.parametrize("B,mode", CASES, ids=[f"{B}-{m}" for B, m in CASES])
def test_leaf_eval_at_every_batch_regime(leaf, B, mode):
    net, prec = leaf.net, PREC[mode]
    net.precision = "fp32" if prec == 0 else "bf16"
    ids = leaf.ids[:B]
    packed = leaf.packed[:B]
    out = _leaf(net, packed, mode)
    pri, val, msk, pwn = out
    assert torch.isfinite(pri).all() and torch.isfinite(val).all()
    assert np.array_equal(msk.cpu().numpy().view(np.uint32), leaf.mask[ids]) and np.array_equal(pwn.cpu().numpy(), leaf.pawn[ids])
    # ---- placement: other orders, and probe boards alone ---------------------------------------------------------------------------
    for name, order in (("rotated", (torch.arange(B, device="cuda") + 1) % B), ("reversed", torch.arange(B - 1, -1, -1, device="cuda"))):
        moved = _leaf(net, packed[order].contiguous(), mode)
        undo = torch.empty_like(order)
        undo[order] = torch.arange(B, device="cuda")
        for what, g, w in zip(("priors", "value", "mask", "pawn"), _bits(tuple(t[undo] for t in moved)), _bits(out)):
            if not torch.equal(g, w):
                bad = (g != w).reshape(B, -1).any(1).nonzero()[:8, 0].tolist()
                pytest.fail(f"B={B} {mode} {name}: {what} of boards {bad} depend on where they sit in the batch")
    for i in lp.probe_positions(B):
        key = (int(ids[i]), mode)
        if key not in leaf.alone:
            leaf.alone[key] = _leaf(net, packed[i:i + 1].clone(), mode)
        assert _same(tuple(t[i:i + 1] for t in out), leaf.alone[key]), f"B={B} {mode}: board {i} differs from its one-board evaluation"
    # ---- content against the oracle --------------------------------------------------------------------------------------------------
    dense = pri.cpu().numpy()
    legal = leaf.legal[:B]
    assert not dense[~legal].any(), "an illegal action has a non-zero prior"
    want_logp, want_v = leaf.want[prec]
    pe, ve = lp.errors(lp.kernel_logp(dense, legal), val.cpu().numpy(), want_logp[:B], want_v[:B], legal)
    bar = lp.FP32_BAR if prec == 0 else lp.BF16_BAR
    worst = int(np.argmax(np.maximum(pe, ve)))
    print(f"B={B} {mode}: worst vs {'exact' if prec == 0 else 'rounding-point'} oracle: log-prob {pe.max():.2e}, value {ve.max():.2e} "
          f"(board {worst}; bar {bar:.0e})")
    assert pe.max() <= bar and ve.max() <= bar, (B, mode, worst, pe.max(), ve.max())
    if mode == "bf16-raw":
        return
    # ---- the other callers of the same kernels --------------------------------------------------------------------------------------
    got = net.predict_batch(packed)
    assert _same((got["priors"], got["value"], got["mask"], got["pawn"]), out)
    nact = leaf.nact[:B]
    want_off = np.concatenate([[0], np.cumsum(nact)]).astype(np.int32)
    gathered = _ragged(dense, leaf.actions[:B], nact)
    host = torch.from_numpy(gl.pack_rows_host(leaf.rows[ids], leaf.plies[ids])).pin_memory()
    for wire in ("f32", "f16"):
        ev = HostLeafEvaluator(net, B, wire=wire)
        res = ev.evaluate(B, states=host)
        assert np.array_equal(res["offsets"], want_off), wire
        assert np.array_equal(res["priors"].view(np.uint16 if wire == "f16" else np.uint32),
                              (gathered.astype(np.float16) if wire == "f16" else gathered).view(np.uint16 if wire == "f16" else np.uint32)), wire
        assert np.array_equal(res["value"].view(np.uint32), val.cpu().numpy().view(np.uint32)), wire
        assert np.array_equal(res["mask"], msk.cpu().numpy()) and np.array_equal(res["pawn"], pwn.cpu().numpy()), wire
        ev.close()
    if lp.HOST_CHUNK_MIN - 1 <= B <= lp.HOST_CHUNK_MIN + 1:   # one chunk / two chunks of a multiple of 128 boards
        L, P = _lib.load(), _lib.ptr
        hp = torch.full((B, 209), float("nan")).pin_memory()
        hv = torch.full((B,), float("nan")).pin_memory()
        hm = torch.full((B, 8), -1, dtype=torch.int32).pin_memory()
        hw = torch.full((B, 8), 0xAB, dtype=torch.uint8).pin_memory()
        ws = torch.empty((L.aq_leaf_eval_host_ws_bytes(B),), dtype=torch.uint8, device="cuda")
        ctx = ctypes.c_void_p()
        _lib.check(L.aq_host_ctx_create(ctypes.byref(ctx)), "aq_host_ctx_create")
        try:
            prep = net.prepared_weights() if prec == 1 else None
            _lib.check(L.aq_leaf_eval_host(P(leaf.flat), P(prep), P(host), B, P(hp), P(hv), P(hm), P(hw), P(ws), prec, ctx,
                                           _lib.stream_ptr()), "aq_leaf_eval_host")
        finally:
            L.aq_host_ctx_destroy(ctx)
        assert _same((hp, hv, hm, hw), tuple(t.cpu() for t in out)), f"aq_leaf_eval_host at B={B} {mode}"
    del out, got
    torch.cuda.empty_cache()


@pytest.mark.parametrize("B", lp.SCAN_BATCH_SIZES)
def test_ragged_priors_across_scan_pieces(leaf, B):
    """aq_compact_priors and the host compact path (HostLeafEvaluator, f32 wire) past one, two and three pieces of the ragged-prior
    scan: offsets equal the running popcount of the legal masks, the ragged priors equal the gather of the dense priors in
    legal_actions() order.  Rows repeat from 46,032 boards on (the distinct trajectory positions)."""
    net = leaf.net
    net.precision = "bf16"
    ids = np.resize(leaf.perm, B)
    rows, plies = leaf.rows[ids], leaf.plies[ids]
    out = net.predict_batch(gl.pack_rows(rows, plies, "cuda"))
    assert np.array_equal(out["mask"].cpu().numpy().view(np.uint32), leaf.mask[ids])
    count = np.unpackbits(leaf.mask[ids].view(np.uint8), axis=1).sum(1).astype(np.int64)
    want_off = np.concatenate([[0], np.cumsum(count)]).astype(np.int32)
    la = qo.legal_actions_batch(rows, plies)
    assert np.array_equal(la["n"].astype(np.int64), count)
    gathered = _ragged(out["priors"].cpu().numpy(), la["actions"], count)
    L, P = _lib.load(), _lib.ptr
    offsets = torch.full((B + 1,), -1, dtype=torch.int32, device="cuda")
    compact = torch.full((B * 136,), float("nan"), device="cuda")
    _lib.check(L.aq_compact_priors(P(out["priors"]), P(out["mask"]), P(out["pawn"]), B, P(offsets), P(compact), _lib.stream_ptr()),
               "aq_compact_priors")
    got_off = offsets.cpu().numpy()
    if not np.array_equal(got_off, want_off):
        first = int(np.argmax(got_off != want_off))
        pytest.fail(f"B={B}: offsets differ from board {first} on (scan piece {first // lp.SCAN_PIECE})")
    assert np.array_equal(compact[:len(gathered)].cpu().numpy().view(np.uint32), gathered.view(np.uint32))
    ev = HostLeafEvaluator(net, B, with_mask=False)
    res = ev.evaluate(B, states=torch.from_numpy(gl.pack_rows_host(rows, plies)).pin_memory())
    assert np.array_equal(res["offsets"], want_off)
    assert np.array_equal(res["priors"].view(np.uint32), gathered.view(np.uint32))
    assert np.array_equal(res["value"].view(np.uint32), out["value"].cpu().numpy().view(np.uint32))
    ev.close()
    print(f"B={B}: {lp.scan_pieces(B)} scan pieces, {int(want_off[-1])} ragged priors exact")
    del out, compact
    torch.cuda.empty_cache()
