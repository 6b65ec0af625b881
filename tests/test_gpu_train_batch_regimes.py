"""The training backward at every batch-size branch of its kernels, one probe board at a time.

heads_backward_kernel, heads_wgrad_tc_kernel, gcn_backward_tc2_kernel, atb_jobs_kernel and loss_grad_kernel choose their launch shape
from the batch size (tests/train_probes.py lists the boundaries).  A gradient summed over a large batch cannot show a board dropped,
counted twice or paired with its neighbour's activations (it moves by ~1/B), so these tests drive the C ABI with an upstream gradient
that is zero except on probe boards and compare with the gradient of the probe boards alone:
  fp32 (precision 0)  vs the fp64 oracle of the probes (gnn_oracle.probe_grads_fp64): rel-L2 <= 1e-5 per tensor (norm floor 1e-3 of the
                      largest) and flat;
  bf16 (precision 1)  vs the same kernels on a compact batch of only the probe boards with the same upstream rows: bit-identical for a
                      single probe (the other boards add exact zeros to every accumulator, and a board's own arithmetic does not depend
                      on where it sits), flat and per-tensor rel-L2 <= 1e-5 for the 8-board joint set (its boards are summed in another
                      order); the compact batches are anchored by a 40-board set against the exact fp64 oracle.
Every tolerance-based comparison also checks that the wrong references a kernel mistake would produce are >= 100 bars away.
The fused loss path (loss inside heads_backward_kernel<true, kNB>, aq_train_backward_step) is compared with the unfused entry points at
the same sizes, and once end to end at B = 13,001 with the real loss against the fp64 oracle."""
import time

import numpy as np
import pytest
import torch

from alphaquoridorgnn_b200 import _lib
from alphaquoridorgnn_b200 import game_logic as gl
from alphaquoridorgnn_b200.pv_network_gnn import FLAT_PARAM_ORDER, GNNNetwork, POLICY_OUTPUT_SIZE
from alphaquoridorgnn_b200.train_network import FlatTrainer
from oracle import gnn_oracle

import train_probes as tp

pytestmark = pytest.mark.gpu
BAR = 1e-5   # fp32 probes vs the fp64 oracle; bf16 joint sets vs their compact batch
PRECS = {0: "fp32", 1: "bf16"}


class _Batch:
    """One aq_gnn_forward with saved activations, then aq_gnn_backward as often as needed with a chosen upstream gradient."""

    def __init__(self, flat, rows, plies, prec):
        L, P = _lib.load(), _lib.ptr
        self.L, self.flat, self.prec = L, flat, prec
        self.B = B = len(rows)
        self.packed = gl.pack_rows(rows, plies, "cuda")
        self.policy = torch.empty((B, POLICY_OUTPUT_SIZE), device="cuda")
        self.value = torch.empty((B,), device="cuda")
        self.saved = torch.zeros((L.aq_gnn_saved_floats(B),), device="cuda")
        _lib.check(L.aq_gnn_forward(P(flat), P(self.packed), None, None, B, P(self.policy), P(self.value), P(self.saved), prec,
                                    _lib.stream_ptr()), "aq_gnn_forward")
        self.ws = torch.empty((L.aq_gnn_backward_ws_floats(B),), device="cuda")
        self.grads = torch.empty_like(flat)
        self.dp = torch.zeros((B, POLICY_OUTPUT_SIZE), device="cuda")
        self.dv = torch.zeros((B,), device="cuda")

    def backward(self):
        P = _lib.ptr
        self.grads.fill_(float("nan"))   # every element must be written
        _lib.check(self.L.aq_gnn_backward(P(self.flat), P(self.saved), P(self.dp), P(self.dv), self.B, P(self.grads), P(self.ws), self.prec,
                                          _lib.stream_ptr()), "aq_gnn_backward")
        return self.grads.clone()

    def probe(self, positions, row_ids):
        """Gradient with the upstream rows of `row_ids` (gnn_oracle.probe_upstream) at `positions`, zero elsewhere."""
        dp, dv = gnn_oracle.probe_upstream(row_ids)
        idx = torch.as_tensor(np.asarray(positions, np.int64), device="cuda")
        self.dp[idx] = torch.from_numpy(dp).cuda()
        self.dv[idx] = torch.from_numpy(dv).cuda()
        g = self.backward()
        self.dp[idx] = 0.0
        self.dv[idx] = 0.0
        return g


@pytest.fixture(scope="module")
def probe(traj):
    t0 = time.perf_counter()
    ref = tp.probe_model()
    net = GNNNetwork()
    net.load_state_dict(ref.state_dict())
    net = net.cuda().train()

    class Ctx:
        pass
    c = Ctx()
    c.ref, c.net, c.flat = ref, net, net.flat_parameters()
    c.rows, c.plies = traj["rows"], traj["plies"]
    c.perm = tp.permutation(traj["rows"])
    c.oracle = tp.ProbeOracle(ref, traj["rows"])
    c.compact = {}   # (row ids, precision) -> flat gradient of the compact batch of those boards

    def compact(ids, prec):
        key = (tuple(int(r) for r in ids), prec)
        if key not in c.compact:
            b = _Batch(c.flat, c.rows[list(key[0])], c.plies[list(key[0])], prec)
            c.compact[key] = b.probe(np.arange(len(ids)), key[0])
        return c.compact[key]
    c.compact_grads = compact
    yield c
    print(f"\ntests/test_gpu_train_batch_regimes.py: wall time {time.perf_counter() - t0:.1f} s")


def _check_fp32(probe, got, ids, what):
    """-> (error, what, tensor) of an fp32 gradient against the fp64 oracle of the probe boards `ids`."""
    per, flat, name = probe.oracle.errors(got.cpu().numpy(), probe.oracle.grads(ids))
    assert per <= BAR and flat <= BAR, (what, name, per, flat)
    return max(per, flat), what, name


@pytest.mark.parametrize("prec", [0, 1], ids=["fp32", "bf16"])
@pytest.mark.parametrize("B", tp.BATCH_SIZES)
def test_probe_board_gradients_at_every_batch_regime(probe, B, prec):
    """aq_gnn_backward at batch B with the upstream gradient on single probe boards (tile / slot / grid-pass edges, batch tail) and on
    one joint set of 8 random boards: see the module docstring for the references and bars."""
    ids = probe.perm[:B]
    batch = _Batch(probe.flat, probe.rows[ids], probe.plies[ids], prec)
    saved_bits = batch.saved.view(torch.int32).clone()
    assert torch.isfinite(batch.policy).all() and torch.isfinite(batch.value).all()
    # the zero-upstream path of every kernel really produces exact zeros (no 0 * inf, no stale slot)
    zero = batch.backward()
    assert int(torch.count_nonzero(zero)) == 0, int(torch.count_nonzero(zero))
    worst = (0.0, None, None)
    for i in tp.probe_positions(B):
        got = batch.probe([i], [ids[i]])
        assert torch.isfinite(got).all(), (B, i)
        if prec == 0:
            drop, swap = tp.single_probe_margins(probe.oracle, probe.perm, B, i)
            assert min(drop, swap) >= tp.MARGIN * BAR, (B, i, drop, swap)
            worst = max(worst, _check_fp32(probe, got, [ids[i]], f"position {i}"), key=lambda t: t[0])
        else:
            want = probe.compact_grads([ids[i]], 1)
            if not torch.equal(got, want):
                rel = ((got - want).double().norm() / want.double().norm()).item()
                pytest.fail(f"bf16 probe at position {i} of B={B} differs from the single-board batch: rel-L2 {rel:.2e}")
    pos = tp.joint_positions(B)
    joint_ids = ids[pos]
    got = batch.probe(pos, joint_ids)
    drop = tp.joint_drop_margin(probe.oracle, probe.perm[:B], pos)
    assert drop >= tp.MARGIN * BAR, (B, drop)
    if prec == 0:
        worst = max(worst, _check_fp32(probe, got, joint_ids, "joint set"), key=lambda t: t[0])
        print(f"B={B} fp32: worst rel-L2 vs the fp64 oracle over {len(tp.probe_positions(B))} single probes + joint set {worst[0]:.2e} "
              f"({worst[1]}, {worst[2]})")
    else:
        want = probe.compact_grads(joint_ids, 1)
        per, flat, _ = probe.oracle.errors(got.cpu().numpy(), want.cpu().numpy())
        assert per <= BAR and flat <= BAR, (B, per, flat)
        print(f"B={B} bf16: single probes bit-identical to their one-board batch; joint set vs its {len(pos)}-board batch "
              f"per-tensor {per:.2e}, flat {flat:.2e}")
    # aq_gnn_backward takes `saved` as const: nothing of the forward's record changed under all these backward passes
    assert torch.equal(batch.saved.view(torch.int32), saved_bits)


def test_bf16_compact_probe_batch_against_the_exact_oracle(probe):
    """Anchor of the compact bf16 batches: 40 probe boards at B = 40 (below kSlots, idle trunk-backward CTAs) against the exact fp64
    oracle, with the rule of the benchmarked batches: flat rel-L2 <= 2 x (rounding-point oracle vs exact) + 2e-2.  Its bar is what bf16
    operands do to a gradient; where a board sits in a batch is checked by the bit-identity of the single probes."""
    ids = probe.perm[:40]
    got = probe.compact_grads(ids, 1).cpu().numpy()
    exact = probe.oracle.grads(ids)
    implied = tp.rel_l2(probe.oracle.grads(ids, emulate_tc=True), exact)
    err = tp.rel_l2(got, exact)
    drop = tp.joint_drop_margin(probe.oracle, probe.perm, np.arange(40))
    print(f"bf16 40-board probe batch: flat rel-L2 vs exact fp64 oracle {err:.2e} (rounding-point oracle vs exact {implied:.2e}, "
          f"bar {2 * implied + 2e-2:.2e}); one board dropped moves the reference by >= {drop:.2e}")
    assert err <= 2 * implied + 2e-2, (err, implied)
    # the same 40 boards at fp32 are within the fp32 bar: the compact batch itself is no special case
    assert drop >= tp.MARGIN * BAR, drop
    _check_fp32(probe, probe.compact_grads(ids, 0), ids, "40-board batch")


def _targets(B, seed):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    pt = torch.softmax(2 * torch.randn((B, POLICY_OUTPUT_SIZE), device="cuda", generator=g), dim=1)
    vt = torch.randint(-1, 2, (B,), device="cuda", generator=g).float()
    return pt, vt


@pytest.mark.parametrize("prec", [0, 1], ids=["fp32", "bf16"])
@pytest.mark.parametrize("B", tp.BATCH_SIZES)
def test_fused_loss_path_at_every_batch_regime(probe, B, prec):
    """FlatTrainer's default step (loss gradient inside heads_backward_kernel<true, kNB>, aq_train_backward_step) against the unfused
    entry points (collective "nccl", world 1: aq_loss_grad + aq_gnn_backward, which the probe test covers) with lr = 0, and the same
    batch as a part of a larger global batch B_total (the 'mean' losses divide by B_total):
      fused vs unfused      gradients <= 1e-6 max|g|; loss <= 2e-5 relative;
      B_total = 4B          gradients x 4 bit-identical (a power-of-two scale is exact in every operand, bf16 tiles included); loss x 4
                            within 2e-5 relative;
      B_total = 3B (fp32)   gradients x 3 within 1e-6 max|g|.  Not at bf16: the trunk and head weight-gradient MMAs take the upstream
                            gradients as bf16 operands, and bf16(x / 3) x 3 differs from bf16(x) by up to 2^-9 relative (measured
                            0.8 .. 6.7e-3 max|g| on a B200), so a 1/3 scale is only as exact as bf16.
    The loss scalars are sums of float atomics, one per CTA (up to 1,184 of them in loss_grad_kernel), in launch order: their last
    bits differ from call to call and grow with the number of partial sums (measured up to 5.3e-6 relative at B = 9,537)."""
    ids = probe.perm[:B]
    packed = gl.pack_rows(probe.rows[ids], probe.plies[ids], "cuda")
    pt, vt = _targets(B, B)
    flat0 = probe.flat.clone()
    runs = (("fused", {}, B), ("plain", {"collective": "nccl"}, B), ("quarter", {}, 4 * B)) + ((("third", {}, 3 * B),) if prec == 0 else ())
    out = {}
    for name, kw, total in runs:
        tr = FlatTrainer(probe.net, lr=0.0, precision=PRECS[prec], **kw)   # a fresh trainer per size: buffers of B = 20,000 are ~5 GB
        assert tr.collective == ("nccl" if kw else "p2p")
        loss = tr.step(packed, pt, vt, total).clone()
        out[name] = (loss, tr.grads.clone())
        del tr
    torch.cuda.empty_cache()
    assert torch.equal(probe.flat, flat0)   # lr 0 leaves the weights alone
    (lf, gf), (lp, gp), (l4, g4) = out["fused"], out["plain"], out["quarter"]
    assert torch.isfinite(gf).all() and torch.isfinite(lf).all()
    gmax = gp.abs().max().item()
    d_plain = (gf - gp).abs().max().item()
    loss_tol = 2e-5 * lf.abs().max().item()
    dl_plain, dl_quarter = (lf - lp).abs().max().item(), (4 * l4 - lf).abs().max().item()
    msg = (f"B={B} {PRECS[prec]}: fused vs unfused max|dg| {d_plain / gmax:.1e} max|g|, loss {dl_plain:.1e}; B_total = 4B: "
           f"{'bit-identical' if torch.equal(4 * g4, gf) else 'DIFFERENT'} gradients, loss {dl_quarter:.1e}")
    if prec == 0:
        l3, g3 = out["third"]
        d_third = (3 * g3 - gf).abs().max().item()
        msg += f"; B_total = 3B: max|3 g' - g| {d_third / gmax:.1e} max|g|, loss {(3 * l3 - lf).abs().max().item():.1e}"
    print(msg)
    assert d_plain <= 1e-6 * gmax, (d_plain, gmax)
    assert dl_plain <= loss_tol, (dl_plain, loss_tol)
    assert torch.equal(4 * g4, gf)
    assert dl_quarter <= loss_tol, (dl_quarter, loss_tol)
    if prec == 0:
        assert d_third <= 1e-6 * gmax, (d_third, gmax)
        assert (3 * l3 - lf).abs().max().item() <= loss_tol


def test_fused_training_step_end_to_end_at_13001_against_the_fp64_oracle(probe):
    """The whole fp32 training step at B = 13,001 (every backward kernel strides) on diverse positions with the real loss, against the
    chunked fp64 oracle: flat gradient rel-L2 <= 1e-4, loss <= 1e-5."""
    B = 13001
    ids = probe.perm[:B]
    torch.manual_seed(13)
    pt = torch.softmax(2 * torch.randn(B, POLICY_OUTPUT_SIZE), dim=1)
    vt = torch.randint(-1, 2, (B,)).float()
    t0 = time.perf_counter()
    loss64, g_ref = gnn_oracle.oracle_grads_fp64(probe.ref, probe.rows[ids], pt, vt)
    t_oracle = time.perf_counter() - t0
    flat_ref = torch.cat([g_ref[n].reshape(-1) for n in FLAT_PARAM_ORDER])
    tr = FlatTrainer(probe.net, lr=0.0, precision="fp32")
    loss = tr.step(gl.pack_rows(probe.rows[ids], probe.plies[ids], "cuda"), pt.cuda(), vt.cuda(), B).sum().item()
    err = tp.rel_l2(tr.grads.cpu().double().numpy(), flat_ref.numpy())
    print(f"fp32 training step at B={B}: flat rel-L2 vs fp64 oracle {err:.2e}, loss {loss:.7f} vs {loss64:.7f} "
          f"(oracle {t_oracle:.1f} s on the CPU)")
    assert err <= 1e-4, err
    assert abs(loss - loss64) <= 1e-5
