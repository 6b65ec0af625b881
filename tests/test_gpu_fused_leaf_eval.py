"""Leaf evaluation at precision 1 computes the legal mask inside the trunk launch from 4,096 boards on (a fifth warpgroup of every
trunk CTA, with a task list in shared memory; smaller batches run the legal-mask kernels first).  Checked bit for bit: mask and pawn
moves against the golden data, priors and value against the separate entry points (legal mask + trunk + heads), a batch whose
searches overflow every CTA's task list, and back-to-back calls."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

from alphaquoridorgnn_b200 import _lib, positions
from alphaquoridorgnn_b200 import game_logic as gl
from alphaquoridorgnn_b200.pv_network_gnn import GNNNetwork

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "..", "alphaquoridorgnn_b200", "csrc")

# Number of path searches the prepare step leaves for a state (LegalPrep::offs[4] in legal_steps.cuh), from the host build of the
# same headers: the popcount of the task sets.
_COUNT_SRC = r'''
#include "legal_steps.cuh"
using namespace aq;
extern "C" void count_searches(const AqState *states, long long B, int *out) {
    for (long long b = 0; b < B; ++b) {
        const AqState s = states[b];
        const Open base = open_from_walls(s.hwalls, s.vwalls);
        const int me = s.ppos, en = 80 - (int)s.epos;
        WallSets ws{};
        if (s.pwalls > 0) ws = wall_sets(s.hwalls, s.vwalls);
        const PathCuts pc[2] = {find_path_cuts(base, me, en, goal_row0()), find_path_cuts(base, en, me, goal_row8())};
        u64 set[4];
        legal_task_sets(ws, pc, set);
        out[b] = __builtin_popcountll(set[0]) + __builtin_popcountll(set[1]) + __builtin_popcountll(set[2]) + __builtin_popcountll(set[3]);
    }
}
'''


@pytest.fixture(scope="module")
def net():
    torch.manual_seed(0)
    n = GNNNetwork().cuda().eval()
    n.precision = "bf16"
    return n


def _np(t):
    return t.cpu().numpy()


def _leaf(net, packed):
    """aq_leaf_eval at precision 1; outputs start as garbage so that every word must be written."""
    L, P = _lib.load(), _lib.ptr
    B = packed.shape[0]
    pri = torch.full((B, 209), float("nan"), device="cuda")
    val = torch.full((B,), float("nan"), device="cuda")
    msk = torch.full((B, 8), -1, dtype=torch.int32, device="cuda")
    pwn = torch.full((B, 8), 0xAB, dtype=torch.uint8, device="cuda")
    ws = torch.empty((L.aq_leaf_eval_ws_floats(B),), device="cuda")
    _lib.check(L.aq_leaf_eval(P(net.flat_parameters()), P(net.prepared_weights()), P(packed), B, P(pri), P(val), P(msk), P(pwn), P(ws), 1,
                              _lib.stream_ptr()), "aq_leaf_eval")
    return pri, val, msk, pwn


def _unfused(net, packed):
    """The same evaluation through the separate entry points: legal mask (two-phase form above 4,096 states), trunk, heads."""
    L, P = _lib.load(), _lib.ptr
    B = packed.shape[0]
    flat, prep = net.flat_parameters(), net.prepared_weights()
    msk = torch.zeros((B, 8), dtype=torch.int32, device="cuda")
    pwn = torch.zeros((B, 8), dtype=torch.uint8, device="cuda")
    ws = torch.empty((L.aq_legal_mask_ws_bytes(B),), dtype=torch.uint8, device="cuda")
    _lib.check(L.aq_legal_mask_ws(P(packed), B, P(msk), P(pwn), P(ws), ws.numel(), _lib.stream_ptr()), "aq_legal_mask_ws")
    pooled = torch.empty((B, 128), device="cuda")
    _lib.check(L.aq_gcn_trunk_forward(P(flat), P(prep), P(packed), B, P(pooled), 1, _lib.stream_ptr()), "aq_gcn_trunk_forward")
    pri = torch.empty((B, 209), device="cuda")
    val = torch.empty((B,), device="cuda")
    _lib.check(L.aq_heads_forward(P(flat), P(prep), P(pooled), B, P(pri), P(val), P(msk), 1, _lib.stream_ptr()), "aq_heads_forward")
    return pri, val, msk, pwn


def test_fused_mask_and_pawn_match_golden(net, traj):
    packed = gl.pack_rows(traj["rows"], traj["plies"])
    B = packed.shape[0]
    _, _, msk, pwn = _leaf(net, packed)
    assert np.array_equal(_np(msk).view(np.uint32), traj["mask"]) and np.array_equal(_np(pwn), traj["pawn"])
    lo = 0
    for n in (1, 3, 5, 31, 592, 777, 4095, 4097, 16383, 20000):   # uneven slices: partial rounds and CTAs with unequal board counts
        hi = min(B, lo + n)
        _, _, msk, pwn = _leaf(net, packed[lo:hi])
        assert np.array_equal(_np(msk).view(np.uint32), traj["mask"][lo:hi]), (lo, hi)
        assert np.array_equal(_np(pwn), traj["pawn"][lo:hi]), (lo, hi)
        lo = hi


@pytest.mark.parametrize("B", [1, 5, 777, 4096, 16384])
def test_fused_leaf_eval_is_bit_identical_to_separate_entry_points(net, B):
    _, (packed,) = positions.mixed_batches(1, B, seed=3)
    got, want = _leaf(net, packed), _unfused(net, packed)
    for name, g, w in zip(("priors", "value", "mask", "pawn"), got, want):
        assert torch.equal(g, w), name


def test_fused_task_list_overflow_is_exact(net, traj, tmp_path_factory):
    """Only the positions with the most searches (>= 39 each), tiled so that every round of 64 states of every CTA needs more
    entries than the shared-memory task list has (2,048): the states that do not fit run their searches in place."""
    d = tmp_path_factory.mktemp("count")
    src, lib = d / "count.cu", d / "libcount.so"
    src.write_text(_COUNT_SRC)
    subprocess.check_call(["nvcc", "-O2", "-std=c++17", "--expt-relaxed-constexpr", "-Wno-deprecated-gpu-targets", "-I", CSRC,
                           "-Xcompiler", "-fPIC", "-shared", "-o", str(lib), str(src)], env=dict(os.environ, CC="/usr/bin/gcc"))
    host = gl.pack_rows_host(traj["rows"], traj["plies"])
    counts = np.zeros(len(host), np.int32)
    ctypes.CDLL(str(lib)).count_searches(ctypes.c_void_p(host.ctypes.data), ctypes.c_longlong(len(host)), ctypes.c_void_p(counts.ctypes.data))
    hard = np.argsort(-counts, kind="stable")[:16]
    assert counts[hard].min() * 64 > 2048, counts[hard]
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    idx = np.resize(hard, sms * 4 * 64 * 2)      # every CTA: 512 states, 8 full rounds
    packed = gl.pack_rows(traj["rows"][idx], traj["plies"][idx])
    got, want = _leaf(net, packed), _unfused(net, packed)
    assert np.array_equal(_np(got[2]).view(np.uint32), traj["mask"][idx]) and np.array_equal(_np(got[3]), traj["pawn"][idx])
    for name, g, w in zip(("priors", "value"), got[:2], want[:2]):
        assert torch.equal(g, w), name


def test_fused_back_to_back_calls_with_different_task_counts(net, traj):
    """Batches with many / no / few path searches, of different sizes, one after another on one stream without synchronisation."""
    rows, plies = traj["rows"], traj["plies"]
    nwalls = (rows[:, 4:] != 0).sum(1)
    sets = {"hard": np.argsort(-nwalls)[:6000], "easy": np.argsort(nwalls, kind="stable")[:5000], "mid": np.arange(5000, 12001)}
    packed = {k: gl.pack_rows(rows[i], plies[i]) for k, i in sets.items()}
    outs = [(k, _leaf(net, packed[k])) for k in ("hard", "easy", "hard", "mid", "easy", "mid", "hard")]
    torch.cuda.synchronize()
    ref = {k: _unfused(net, packed[k]) for k in sets}
    for k, (pri, val, msk, pwn) in outs:
        assert np.array_equal(_np(msk).view(np.uint32), traj["mask"][sets[k]]), k
        assert np.array_equal(_np(pwn), traj["pawn"][sets[k]]), k
        assert torch.equal(pri, ref[k][0]) and torch.equal(val, ref[k][1]), k
