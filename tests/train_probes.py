"""Probe-board plan of the training-backward tests at every batch-size branch (tests/test_gpu_train_batch_regimes.py) and of their CPU
check (tests/test_oracle_train_probes.py) -- test infrastructure.

A batch of B boards gets an upstream gradient (dpolicy, dvalue) that is zero on every board except a few probe boards.  Everything from
the heads back to the weights is linear in the upstream gradient, so the parameter gradient of the whole batch is the gradient of the
probe boards alone (gnn_oracle.probe_grads_fp64): a reference that costs milliseconds at any B.  A gradient summed over all B boards
would move by only ~1/B if a kernel dropped a board, counted it twice or paired one board's upstream gradient with its neighbour's
activations; for a single probe board the same mistakes move it by O(1).

Positions are the distinct rows of tests/golden/trajectories.npz (46,032 of its 54,459 rows; games repeat their opening positions) under
a fixed permutation, so adjacent boards of a batch are unrelated positions and a board paired with the wrong neighbour gives a
different gradient."""
import numpy as np

from alphaquoridorgnn_b200.pv_network_gnn import FLAT_PARAM_ORDER
from oracle import gnn_oracle

PERM_SEED = 20261
MODEL_SEED = 0
N_JOINT = 8          # boards of the joint probe set of a batch
SLOTS = 148          # kSlots (gnn_backward.cu): partial-gradient slots, heads-backward grid cap; also the trunk-backward grid (gnn_tc2_bwd.cu)
MARGIN = 100.0       # a probe reference with one board dropped or swapped must be this many bars away from the true one

# One batch just below and one just above every boundary of the training backward's launch shapes (csrc/), with the branch each reaches.
BATCH_SIZES = (
    1,       # one board: 147 of the kSlots = 148 trunk-backward CTAs idle (gnn_tc2_bwd.cu), one kWgTile tile, one AQ_HEAD_CHUNK_ROWS chunk
    2,       # two boards in one heads-backward CTA (256 threads, kNB = 1) and one 64-board tile
    63,      # last board before the second kWgTile = 64 tile (heads_wgrad_tc.cu) / AQ_HEAD_CHUNK_ROWS = 64 row chunk (gnn_backward.cu)
    64,      # exactly one full tile / row chunk
    65,      # second tile / head row chunk with one board
    147,     # one idle gcn_backward_tc2_kernel CTA left (grid kSlots = 148); 147 trunk-backward partial slots with a board
    148,     # every trunk-backward CTA has exactly one board
    149,     # CTA 0 of the trunk backward takes a second board (grid stride of kSlots)
    1184,    # heads backward at 256 threads: 148 CTAs x 8 warps x kNB = 1 boards in one pass (B <= 1184 branch, gnn_backward.cu)
    1185,    # heads backward at kHbThreads = 512 threads with kNB = 1 (never compared before)
    2367,    # last batch with kNB = 1 (kNB = 2 from kSlots x kHbThreads / 32 = 2,368)
    2368,    # kNB = 2, one pass
    4736,    # kNB = 2: 148 x 16 x 2 = 4,736 boards fill exactly one grid pass of the heads backward
    4737,    # kNB = 2 with a grid stride: CTA 0's first warp takes board 4,736 on its second pass
    8191,    # last batch with kNB = 2 (strided)
    8192,    # kNB = 4 (B >= 8192), one pass
    9472,    # 148 x 64: heads_wgrad_tc_kernel one tile per CTA; kNB = 4 one pass (148 x 16 x 4); loss_grad_kernel 1,184 CTAs x 8 boards
    9473,    # 149 tiles: CTA 0 of heads_wgrad_tc_kernel takes a second tile (tensor-memory accumulation, mbarrier parity flip) with one board;
             # the heads backward and loss_grad_kernel stride
    9537,    # 9,472 + 65: CTA 0 takes a full second tile, CTA 1 a second tile with one board
    13001,   # 204 tiles: 56 CTAs take two tiles; every kernel strides
    20000,   # 313 tiles: 17 CTAs take three tiles (two parity flips); heads backward and loss_grad_kernel take three passes
)


def permutation(rows):
    """Row ids of the distinct positions of `rows` (first occurrence of each) in a fixed random order."""
    _, first = np.unique(rows, axis=0, return_index=True)
    return np.random.default_rng(PERM_SEED).permutation(np.sort(first))


def probe_model():
    """The random-init network of the tests (GCN biases non-zero so that their path is exercised), as the fp32 CPU oracle model."""
    import torch
    torch.manual_seed(MODEL_SEED)
    ref = gnn_oracle.GraphPolicyValueNetworkOracle()
    with torch.no_grad():
        for layer in ref.gcn_layers:
            layer.bias.uniform_(-0.1, 0.1)
    return ref


def heads_backward_shape(B):
    """(threads, kNB) of heads_backward_kernel at batch B, restated from backward_to_partials (gnn_backward.cu)."""
    threads = 256 if B <= 1184 else 512
    nb = 4 if B >= 8192 else 2 if B >= SLOTS * (512 // 32) else 1
    return threads, nb


def heads_backward_pass(B):
    """Boards the heads backward covers in one grid pass; board number `pass` is the first one a warp takes on its second pass."""
    threads, nb = heads_backward_shape(B)
    return SLOTS * (threads // 32) * nb


def probe_positions(B):
    """Single-board probe positions of a batch: tile, slot and grid-pass edges, and the tail of the batch."""
    p = heads_backward_pass(B)
    cand = (0, 1, 63, 64, 147, 148, p - 1, p, 9471, 9472, B - 65, B - 64, B - 2, B - 1)
    return sorted({c for c in cand if 0 <= c < B})


def joint_positions(B):
    """N_JOINT distinct positions drawn at random (seeded by B), sorted; every board when B < N_JOINT."""
    return np.sort(np.random.default_rng(B).choice(B, min(N_JOINT, B), replace=False))


def swap_partner(B, i):
    """Position whose row a kernel would use if it paired board i's upstream gradient with its neighbour's activations."""
    return i + 1 if i + 1 < B else i - 1 if i > 0 else 1


class ProbeOracle:
    """Cached flat fp64 reference gradients of probe sets (FLAT_PARAM_ORDER, the order of the kernels' flat gradient buffer)."""

    def __init__(self, ref, rows):
        self.ref, self.rows = ref, rows
        self._cache = {}
        self.slices, off = {}, 0
        named = dict(ref.named_parameters())
        for n in FLAT_PARAM_ORDER:
            k = named[n].numel()
            self.slices[n] = slice(off, off + k)
            off += k

    def grads(self, row_ids, upstream_ids=None, emulate_tc=False):
        """Gradient of the boards `row_ids` (trajectory rows), board k receiving the upstream gradient of row upstream_ids[k]
        (default: its own, gnn_oracle.probe_upstream)."""
        row_ids = tuple(int(r) for r in row_ids)
        upstream_ids = row_ids if upstream_ids is None else tuple(int(r) for r in upstream_ids)
        key = (row_ids, upstream_ids, emulate_tc)
        g = self._cache.get(key)
        if g is None:
            dp, dv = gnn_oracle.probe_upstream(upstream_ids)
            gd = gnn_oracle.probe_grads_fp64(self.ref, self.rows[list(row_ids)], dp, dv, emulate_tc=emulate_tc)
            g = self._cache[key] = np.concatenate([gd[n].numpy().reshape(-1) for n in FLAT_PARAM_ORDER])
        return g

    def errors(self, got, want):
        """-> (worst per-tensor rel-L2, flat rel-L2, name of the worst tensor).  Per tensor the error is divided by max(|want_tensor|, 1e-3 max_t |want_t|): a
        tensor whose gradient is three orders below the largest one is held to the same absolute error as one at that floor."""
        got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
        norms = {n: np.linalg.norm(want[s]) for n, s in self.slices.items()}
        floor = 1e-3 * max(norms.values())
        per = {n: np.linalg.norm(got[s] - want[s]) / max(norms[n], floor) for n, s in self.slices.items()}
        flat = np.linalg.norm(got - want) / np.linalg.norm(want)
        worst = max(per, key=per.get)
        return per[worst], flat, worst


def rel_l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


def single_probe_margins(oracle, perm, B, i):
    """Flat rel-L2 of two wrong references from the true one of the single probe at position i: the probe dropped (zero gradient,
    distance 1) and its upstream gradient paired with the swap partner's row."""
    want = oracle.grads([perm[i]])
    swapped = oracle.grads([perm[swap_partner(B, i)]], upstream_ids=[perm[i]])
    return 1.0, rel_l2(swapped, want)


def joint_drop_margin(oracle, perm, positions):
    """Smallest flat rel-L2 between the joint set's reference and the reference with one of its boards left out."""
    ids = [perm[i] for i in positions]
    want = oracle.grads(ids)
    if len(ids) == 1:
        return 1.0
    return min(rel_l2(oracle.grads(ids[:k] + ids[k + 1:]), want) for k in range(len(ids)))
