"""CPU checks of the leaf-evaluation batch plan (tests/leaf_probes.py): a board's oracle reference does not depend on the chunk it was
computed in, the wrong boards a placement mistake would use stay far outside the fp32 bar of tests/test_gpu_leaf_eval_batch_regimes.py,
and the launch-shape restatements reach the branches the plan names."""
import numpy as np

import leaf_probes as lp
import train_probes as tp


def test_cached_oracle_equals_a_direct_call_on_any_slice(traj):
    """The chunked references of perm[:N] equal a direct oracle call on sub-slices that start inside a chunk and cross chunk
    boundaries."""
    ref = lp.leaf_model()
    perm = tp.permutation(traj["rows"])
    rows = traj["rows"][perm[:2100]]
    for emulate in (False, True):
        logp, value = lp.oracle_outputs(ref, rows, emulate_tc=emulate)
        for lo, hi in ((0, 1), (5, 17), (1000, 1100), (2047, 2049), (2099, 2100)):
            lg, vg = lp.oracle_outputs(ref, rows[lo:hi], emulate_tc=emulate)
            assert np.abs(lg - logp[lo:hi]).max() <= 1e-12 and np.abs(vg - value[lo:hi]).max() <= 1e-12, (emulate, lo, hi)


def test_wrong_boards_are_far_outside_the_fp32_bar(traj):
    """For every batch size and probe position: the references of the neighbour, of the same tile row one heads tile away and of the same
    trunk group one pass away are each >= 100 fp32 bars from the true reference in the content metric.  The bf16 bar is not held to
    this: the rounding-point oracle and the kernels round at the same points, but an fp32 accumulator that lands on the other side of a
    bf16 rounding boundary than the fp64 one moves a board by about as much as the closest distinct boards differ.  Placement at bf16
    rests on the bit-identity checks instead (a board in any order and alone), which need no margin."""
    ref = lp.leaf_model()
    perm = tp.permutation(traj["rows"])
    need = sorted({k for B in lp.LEAF_BATCH_SIZES for i in lp.probe_positions(B) for k in [i] + lp.wrong_positions(B, i)})
    at = {k: n for n, k in enumerate(need)}
    ids = perm[need]
    logp, value = lp.oracle_outputs(ref, traj["rows"][ids])
    legal = lp.dense_legal(traj["mask"][ids])
    worst = (np.inf, None)
    for B in lp.LEAF_BATCH_SIZES:
        for i in lp.probe_positions(B):
            for j in lp.wrong_positions(B, i):
                d = lp.wrong_board_distance(logp, value, legal, at[i], at[j])
                assert d >= lp.MARGIN * lp.FP32_BAR, (B, i, j, d)
                worst = min(worst, (d, (B, i, j)), key=lambda t: t[0])
    # what the existing absolute bars (bf16 priors 2e-3, values 5e-3 against the exact oracle) have to cover: the rounding-point
    # oracle against the exact one, on the same boards
    le, ve = lp.oracle_outputs(ref, traj["rows"][ids], emulate_tc=True)
    pe, vd = lp.errors(lp.restrict(le, legal), ve, lp.restrict(logp, legal), value, legal)
    pa = np.abs(np.exp(lp.restrict(le, legal)) - np.exp(lp.restrict(logp, legal))).max()
    print(f"closest wrong board {worst[0]:.2e} at (B, i, j) = {worst[1]} = {worst[0] / lp.FP32_BAR:.0f} fp32 bars, "
          f"{worst[0] / lp.BF16_BAR:.1f} bf16 bars; rounding-point vs exact oracle over {len(ids)} boards: log-prob {pe.max():.2e}, "
          f"prior {pa:.2e}, value {vd.max():.2e}")


def test_leaf_plan_reaches_every_branch():
    """The restated launch shapes put the plan's batch sizes where their comments say, and every probe list lies in its batch."""
    sizes = lp.LEAF_BATCH_SIZES
    assert len(set(sizes)) == len(sizes) and list(sizes) == sorted(sizes) and max(sizes) <= 46032
    assert [lp.trunk_grid(B, 1) for B in (1, 4, 5, 591, 592, 593)] == [1, 1, 2, 148, 148, 148]
    assert [lp.trunk_grid(B, 0) for B in (1, 148, 149)] == [1, 148, 148]
    assert max(lp.trunk_pass(B, 1, B - 1) for B in (591, 592)) == 0 and lp.trunk_pass(593, 1, 592) == 1
    assert lp.trunk_pass(1184, 1, 1183) == 1 and lp.trunk_pass(1185, 1, 1184) == 2
    assert lp.trunk_pass(149, 0, 148) == 1 and lp.trunk_pass(148, 0, 147) == 0
    assert [lp.heads_tiles(B) for B in (1, 127, 128, 129)] == [1, 1, 1, 2]
    assert [lp.heads_fp32_grid(B) for B in (4, 5, 1184, 1185)] == [1, 1, 148, 148]
    assert (1184 - 1) // (lp.SMS * lp.HEADS_FP32_WARPS) == 0 and 1184 // (lp.SMS * lp.HEADS_FP32_WARPS) == 1
    assert [lp.legal_round(B, B - 1) for B in (4096, 9471, 9472, 9473, 18944, 18945)] == [0, 0, 0, 1, 1, 2]
    assert [lp.scan_pieces(B) for B in lp.SCAN_BATCH_SIZES] == [1, 1, 2, 2, 3, 4]
    assert lp.scan_pieces(16384) == 1 and lp.scan_pieces(20000) == 2
    assert max(B for B in sizes if B < lp.FUSED_MIN) == lp.FUSED_MIN - 1 and lp.FUSED_MIN in sizes
    for B in sizes:
        pos = lp.probe_positions(B)
        assert pos and pos[0] == 0 and pos[-1] == B - 1 and len(set(pos)) == len(pos)
        for i in pos:
            assert all(0 <= j < B and j != i for j in lp.wrong_positions(B, i))
    assert lp.wrong_positions(593, 592) == [0, 464, 591] and lp.wrong_positions(1, 0) == []
