"""CPU checks of the probe-board reference of the training-backward tests (tests/train_probes.py, gnn_oracle.probe_grads_fp64):
the probe-only reference equals the full-batch fp64 gradient with zero upstream rows, and the wrong references a kernel mistake
would produce stay far outside the bars of tests/test_gpu_train_batch_regimes.py."""
import numpy as np
from oracle import gnn_oracle

import train_probes as tp

BAR = 1e-5   # the tolerance-based bars of the GPU test (fp32 probes vs the oracle, bf16 joint sets vs their compact batch)


def test_probe_reference_equals_the_full_batch_gradient_with_zero_upstream_rows(traj):
    """A 200-board batch whose upstream gradient is zero except on 24 probe boards has the gradient of those 24 boards alone."""
    ref = tp.probe_model()
    perm = tp.permutation(traj["rows"])
    B = 200
    ids = perm[:B]
    probes = np.sort(np.random.default_rng(5).choice(B, 24, replace=False))
    dp = np.zeros((B, gnn_oracle.POLICY_OUTPUT_SIZE), np.float32)
    dv = np.zeros((B,), np.float32)
    dp[probes], dv[probes] = gnn_oracle.probe_upstream(ids[probes])
    full = gnn_oracle.probe_grads_fp64(ref, traj["rows"][ids], dp, dv)
    oracle = tp.ProbeOracle(ref, traj["rows"])
    want = np.concatenate([full[n].numpy().reshape(-1) for n in oracle.slices])
    got = oracle.grads(ids[probes])
    per, flat, _ = oracle.errors(got, want)
    assert per <= 1e-12 and flat <= 1e-12, (per, flat)
    # the upstream gradient of a board depends on its row id only
    a, b = gnn_oracle.probe_upstream([ids[7], ids[3]]), gnn_oracle.probe_upstream([ids[3]])
    assert np.array_equal(a[0][1], b[0][0]) and a[1][1] == b[1][0]
    # and the zero rows really contribute nothing: the same batch with every upstream row zero has a zero gradient
    zero = gnn_oracle.probe_grads_fp64(ref, traj["rows"][ids[:16]], np.zeros((16, 209), np.float32), np.zeros(16, np.float32))
    assert all(float(g.abs().max()) == 0.0 for g in zero.values())


def test_wrong_probe_references_are_far_outside_the_bars(traj):
    """For every batch size of the GPU test: a single probe's reference computed for its swap partner's row, and a joint set's
    reference with one board left out, are each at least 100 bars away from the true reference (flat rel-L2)."""
    ref = tp.probe_model()
    perm = tp.permutation(traj["rows"])
    oracle = tp.ProbeOracle(ref, traj["rows"])
    worst_swap, worst_drop = np.inf, np.inf
    for B in tp.BATCH_SIZES:
        for i in tp.probe_positions(B):
            drop, swap = tp.single_probe_margins(oracle, perm, B, i)
            assert drop >= tp.MARGIN * BAR and swap >= tp.MARGIN * BAR, (B, i, drop, swap)
            worst_swap = min(worst_swap, swap)
        d = tp.joint_drop_margin(oracle, perm, tp.joint_positions(B))
        assert d >= tp.MARGIN * BAR, (B, d)
        worst_drop = min(worst_drop, d)
    print(f"smallest swap distance {worst_swap:.2e}, smallest joint-set drop distance {worst_drop:.2e} (bar {BAR:.0e})")


def test_probe_plan_covers_every_branch():
    """Every batch size is in range of the trajectories and every probe list is within its batch; the heads-backward pass boundaries
    of the plan are the ones of backward_to_partials."""
    assert [tp.heads_backward_pass(B) for B in (1, 1184, 1185, 2367, 2368, 8191, 8192)] == [1184, 1184, 2368, 2368, 4736, 4736, 9472]
    assert len(set(tp.BATCH_SIZES)) == len(tp.BATCH_SIZES) == 21
    for B in tp.BATCH_SIZES:
        pos = tp.probe_positions(B)
        assert pos and pos[0] == 0 and pos[-1] == B - 1 and len(set(pos)) == len(pos)
        j = tp.joint_positions(B)
        assert len(j) == min(tp.N_JOINT, B) and len(set(j.tolist())) == len(j) and j.max() < B
    rows = np.random.default_rng(0).integers(0, 3, (50, 4)).astype(np.uint8)
    perm = tp.permutation(rows)
    assert np.array_equal(perm, tp.permutation(rows)) and len(np.unique(rows[perm], axis=0)) == len(perm)
