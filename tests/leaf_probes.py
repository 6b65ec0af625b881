"""Batch plan of the leaf-evaluation tests at every batch-size branch of its kernels (tests/test_gpu_leaf_eval_batch_regimes.py) and of
their CPU check (tests/test_oracle_leaf_probes.py) -- test infrastructure.

aq_leaf_eval (legal mask, GCN trunk, policy / value heads) picks its launch shapes from the batch size.  A board's arithmetic does not
depend on where it sits in the batch, so where a board's outputs land is checked without a tolerance (the same boards in another
order, a board alone); the oracle only has to pin down what is computed.  The batch at size B holds the trajectory rows perm[:B]
(train_probes.permutation: distinct positions in a fixed random order), so a board has the same row id at every size and its
references are computed once.

The content metric of a board is max(max over its legal actions |log p - log p_ref|, |v - v_ref|): log-probabilities, because with
the random-init test network every prior lies within a factor ~2 of 1/|legal| and an absolute bar on the priors cannot tell one
board from another."""
import numpy as np
import torch

from oracle import gnn_oracle

import train_probes as tp

SMS = 148             # SMs of a B200 (aq_num_sms): grid cap of the trunk and of the fp32 heads
KG = 4                # kG (gnn_tc2.cu): boards in flight per trunk CTA, one per group
HEADS_TILE = 128      # kTile (heads_tc.cu): boards per heads_forward_tc_kernel CTA
HEADS_FP32_WARPS = 8  # kHeadThreads / 32 (gnn_forward.cu): boards per heads_forward_kernel CTA, one per warp
LEGAL_ROUND = 64      # kLegalStates (gnn_tc2.cu): states per round of the fused legal warpgroup
FUSED_MIN = 4096      # kLeafFusedMin (gnn_forward.cu): from here precision 1 computes the legal mask inside the trunk launch
SCAN_PIECE = 16 * 1024  # kScanRun x 1024 (gnn_forward.cu): boards per piece of legal_count_scan_kernel
HOST_CHUNK_MIN = 4096   # aq_leaf_eval_host with a context: two chunks of a multiple of 128 boards from here
MARGIN = 100.0        # a wrong board's reference must be this many bars from the true one
PLANE_SCALE = 30.0    # leaf_model: layer-1 weight columns of the pawn and wall planes (features 0, 2, 4, 5) x this
FP32_BAR = 1e-5       # content bar of the fp32 path against the exact fp64 oracle (B200: worst 3.3e-7)
BF16_BAR = 5e-3       # content bar of the bf16 path against the rounding-point oracle (B200: worst 1.7e-3 over 20,000 boards)
ORACLE_CHUNK = 1024   # boards per oracle call (the edge-list formulation in float64 is ~80 MB per 1,024 boards)

# One batch just below and one just above every boundary of the inference launch shapes (csrc/), with the branch each reaches.
LEAF_BATCH_SIZES = (
    1,       # trunk CTA 0 with three idle groups; one heads tile of 128 rows with one board; legal_mask_kernel<32>
    2,       # two groups of trunk CTA 0 busy
    4,       # trunk CTA 0 full (kG = 4), one board per group
    5,       # second trunk CTA (grid ceil(B / kG)) with one board; fp32 heads: 5 of the 8 warps of one CTA
    127,     # last heads tile one row short of kTile = 128 (heads_tc.cu)
    128,     # exactly one full heads tile
    129,     # second heads tile with one row
    148,     # fp32 trunk: one board per CTA of grid min(B, SMs) (gcn_forward_fp32_kernel)
    149,     # fp32 trunk: CTA 0 takes a second board (grid stride SMs)
    591,     # bf16 trunk: 148 CTAs, the last group idle
    592,     # 148 CTAs x kG = 4 groups: every group one board, one pass
    593,     # second trunk pass: group 0 of CTA 0 takes board 592 -- the software-pipelined next-board node_phase and its adjacency
             # buffer parity run
    1024,    # last batch of legal_mask_kernel<32> (unfused path, aq_legal_mask_ws)
    1025,    # legal_mask_kernel<8>
    1184,    # fp32 heads: 148 CTAs x 8 warps fill one pass; bf16 trunk: two full passes
    1185,    # fp32 heads: grid cap, warp 0 of CTA 0 takes board 1,184; bf16 trunk: third pass
    4095,    # last unfused batch: legal-mask kernels, then trunk, then heads (kLeafFusedMin = 4,096)
    4096,    # fused: the trunk launch's fifth warpgroup computes the legal mask (one 64-state round per CTA)
    4097,    # fused, one board past a multiple of 592 in the last round
    9471,    # last batch inside the first 64-state round of the legal warpgroup (148 x 4 x 16 = 9,472 boards per round)
    9472,    # exactly one full round
    9473,    # second round: its counters at parity 1, board 9,472 the round's only state
    16384,   # the benchmarked batch (bench.py --batch 16384): one full scan piece of legal_count_scan_kernel
    18944,   # exactly two full legal rounds
    18945,   # third round: the parity-0 counters reused ("last used two rounds ago", legal_warpgroup)
    20000,   # 34 trunk passes (last partial), three legal rounds, two scan pieces
)

# batch sizes of the ragged-prior scan: one piece, one board past it, two pieces, one past two, and a ragged fourth piece
SCAN_BATCH_SIZES = (16383, 16384, 16385, 32768, 32769, 50001)


def leaf_model():
    """train_probes.probe_model() with the layer-1 weights of the pawn and wall planes scaled by PLANE_SCALE.  The two wall-count
    planes are the same at all 81 nodes and dominate the mean-pooled vector of the plain random-init network, so boards with the same
    walls in hand come out nearly alike: the closest wrong board of a probe position is 5.6e-5 from the true one in the content metric.
    The scale makes a board's outputs depend on where its pawns and walls are (closest wrong board 4.6e-3; |Z| <= 18 stays far from
    the fp16 limit of the trunk's aggregation operand)."""
    ref = tp.probe_model()
    with torch.no_grad():
        w = ref.gcn_layers[0].lin.weight
        w[:, [0, 2, 4, 5]] *= PLANE_SCALE
    return ref


def trunk_grid(B, precision):
    """CTAs of the trunk launch: gcn_forward_fp32_kernel min(B, SMs) (one board per CTA), gcn_forward_tc2_kernel
    min(ceil(B / kG), SMs) (kG boards per CTA)."""
    return min(B, SMS) if precision == 0 else min((B + KG - 1) // KG, SMS)


def trunk_stride(B, precision):
    """Boards between two passes of one trunk group (grid stride)."""
    return trunk_grid(B, precision) * (1 if precision == 0 else KG)


def trunk_pass(B, precision, i):
    return i // trunk_stride(B, precision)


def heads_tiles(B):
    """CTAs of heads_forward_tc_kernel: ceil(B / kTile)."""
    return (B + HEADS_TILE - 1) // HEADS_TILE


def heads_fp32_grid(B):
    """CTAs of heads_forward_kernel: min(ceil(B / 8), SMs)."""
    return min((B + HEADS_FP32_WARPS - 1) // HEADS_FP32_WARPS, SMS)


def legal_round(B, i):
    """Round of the fused legal warpgroup that computes board i's mask: state k of a CTA is board first + (k & 3) + (k >> 2) x stride,
    so board i is state 4 x (pass of i) + group, and a round holds 64 states."""
    return (KG * trunk_pass(B, 1, i) + i % KG) // LEGAL_ROUND


def scan_pieces(B):
    """Pieces of legal_count_scan_kernel (a running carry passes between them)."""
    return (B + SCAN_PIECE - 1) // SCAN_PIECE


def probe_positions(B):
    """Boards of a batch compared one by one with their one-board evaluation: group, tile, pass and round edges, and the tail."""
    cand = (0, 1, 3, 4, 127, 128, 591, 592, 9471, 9472, B - 2, B - 1)
    return sorted({c for c in cand if 0 <= c < B})


def wrong_positions(B, i):
    """Boards whose outputs a placement mistake would hand board i: the neighbour, the same tile row in the next / previous heads tile
    and, from one full trunk pass on, the same group one pass away."""
    cand = [i + 1 if i + 1 < B else i - 1, i + HEADS_TILE, i - HEADS_TILE]
    if B >= SMS * KG:
        cand += [i + SMS * KG, i - SMS * KG]
    return sorted({j for j in cand if 0 <= j < B and j != i})


def dense_legal(mask):
    """uint32 [N,8] legal masks -> bool [N,209]."""
    return np.unpackbits(np.ascontiguousarray(mask).view(np.uint8), axis=1, bitorder="little")[:, :gnn_oracle.POLICY_OUTPUT_SIZE].astype(bool)


def oracle_outputs(ref, rows, emulate_tc=False, chunk=ORACLE_CHUNK):
    """fp64 forward of the boards `rows`: (log-softmax over all 209 actions [N,209], value [N]).  emulate_tc: with the rounding points
    of the bf16 tensor-core path (gnn_oracle.forward_tc_emulation).  Computed in chunks; a board's reference does not depend on its
    chunk."""
    import copy
    ref64 = copy.deepcopy(ref).double()
    n = len(rows)
    logp = np.empty((n, gnn_oracle.POLICY_OUTPUT_SIZE), np.float64)
    value = np.empty((n,), np.float64)
    with torch.no_grad():
        for lo in range(0, n, chunk):
            hi = min(n, lo + chunk)
            x, ei, batch = gnn_oracle.graph_inputs_from_rows(rows[lo:hi], dtype=torch.float64)
            p, v = gnn_oracle.forward_tc_emulation(ref64, x, ei, batch) if emulate_tc else ref64(x, ei, batch)
            logp[lo:hi] = torch.log(p).numpy()
            value[lo:hi] = v[:, 0].numpy()
    return logp, value


def restrict(logp, legal):
    """Log-probabilities of predict(): the distribution restricted to the legal actions and renormalised (`_oracle_predict`).  Entries
    of illegal actions are -inf."""
    m = np.where(legal, logp, -np.inf)
    top = m.max(axis=1, keepdims=True)
    return m - (top + np.log(np.exp(m - top).sum(axis=1, keepdims=True)))


def errors(logp_legal, value, want_logp_legal, want_value, legal):
    """Per-board content error (module docstring): -> (policy error [N], value error [N])."""
    d = np.abs(np.where(legal, logp_legal, 0.0) - np.where(legal, want_logp_legal, 0.0))
    return d.max(axis=1), np.abs(np.asarray(value, np.float64) - want_value)


def kernel_logp(priors, legal):
    """log of the kernel's (legal-masked, renormalised) priors, -inf off the legal actions."""
    p = np.asarray(priors, np.float64)
    with np.errstate(divide="ignore"):
        return np.where(legal, np.log(p), -np.inf)


def wrong_board_distance(logp, value, legal, i, j):
    """Distance, in the content metric, between board i's reference and what board i would get if a kernel used board j's trunk or
    head output with board i's legal mask."""
    want = restrict(logp[i:i + 1], legal[i:i + 1])
    got = restrict(logp[j:j + 1], legal[i:i + 1])
    pe, ve = errors(got, value[j:j + 1], want, value[i:i + 1], legal[i:i + 1])
    return max(float(pe[0]), float(ve[0]))
