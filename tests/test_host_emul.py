"""CPU check of the bitboard algorithm used by the CUDA legal-mask kernels: the same device headers
(csrc/aq_common.cuh and the per-state steps of csrc/legal_steps.cuh, __host__ __device__) are compiled
for the host and run on every golden position.  No GPU needed; the GPU tests then cover the warp-level
plumbing."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "host_emul", "emul.cu")
LIB = os.path.join(HERE, "host_emul", "libemul.so")


@pytest.fixture(scope="module")
def emul():
    hdrs = [os.path.join(HERE, "..", "alphaquoridorgnn_b200", "csrc", h) for h in ("aq_common.cuh", "legal_steps.cuh")]
    if not os.path.exists(LIB) or os.path.getmtime(LIB) < max(os.path.getmtime(f) for f in [SRC] + hdrs):
        subprocess.check_call(["nvcc", "-O2", "-std=c++17", "--expt-relaxed-constexpr", "-Wno-deprecated-gpu-targets",
                               "-Xcompiler", "-fPIC", "-shared", "-o", LIB, SRC],
                              env=dict(os.environ, CC="/usr/bin/gcc"))
    return ctypes.CDLL(LIB)


def _p(a):
    return ctypes.c_void_p(a.ctypes.data)


def test_bitboard_algorithm_matches_reference_goldens(emul, traj, graph_golden):
    rows, plies = np.ascontiguousarray(traj["rows"]), np.ascontiguousarray(traj["plies"])
    B = len(rows)
    st = np.zeros((B, 32), np.uint8)
    emul.emul_pack(_p(rows), _p(plies), ctypes.c_longlong(B), _p(st))
    mask = np.zeros((B, 8), np.uint32)
    pawn = np.zeros((B, 8), np.uint8)
    emul.emul_legal_mask(_p(st), ctypes.c_longlong(B), _p(mask), _p(pawn))
    assert np.array_equal(mask, traj["mask"])
    assert np.array_equal(pawn, traj["pawn"])
    idx = graph_golden["index"]
    sub = np.ascontiguousarray(st[idx])
    om = np.zeros((len(idx), 81), np.uint8)
    emul.emul_open_mask(_p(sub), ctypes.c_longlong(len(idx)), _p(om))
    assert np.array_equal(om, graph_golden["open"])


def test_path_length_matches_reference_heuristic(emul, traj, agents_golden):
    """agents.heuristic_eval of the unmodified reference = (dist_enemy - dist_mover) / 48 for the bitboard flood fill."""
    idx = np.array(agents_golden["heuristic"]["index"])
    rows, plies = np.ascontiguousarray(traj["rows"][idx]), np.ascontiguousarray(traj["plies"][idx])
    st = np.zeros((len(idx), 32), np.uint8)
    emul.emul_pack(_p(rows), _p(plies), ctypes.c_longlong(len(idx)), _p(st))
    dist = np.zeros((len(idx), 2), np.int16)
    emul.emul_shortest_paths(_p(st), ctypes.c_longlong(len(idx)), _p(dist))
    assert (dist >= -1).all() and (dist == -1).sum() >= 1  # -1: the other pawn seals the only corridor (agents.py:41)
    got = (dist[:, 1].astype(np.int64) - dist[:, 0]) / 48
    assert np.array_equal(got, np.array(agents_golden["heuristic"]["value"]))
