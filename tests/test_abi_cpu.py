"""CPU-side checks of the boundary: the shared library loads, exports every symbol include/aqgnn.h
declares, host-side packing matches the device layout, and the product fails loudly without CUDA."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from alphaquoridorgnn_b200 import _lib, build
from alphaquoridorgnn_b200 import game_logic as gl

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_builds_and_exports_every_header_symbol():
    path = build.build()
    lib = ctypes.CDLL(path)
    header = open(os.path.join(ROOT, "include", "aqgnn.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(aq_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in aqgnn.h but not exported"
    assert declared == set(_lib.SYMBOLS), (declared ^ set(_lib.SYMBOLS))
    L = _lib.load()
    assert L.aq_version() >= 100
    assert L.aq_param_count() == 64082  # BASELINE.md: 64,082 fp32 parameters


def test_sass_is_sm100a():
    import subprocess
    out = subprocess.run(["cuobjdump", "-lelf", build.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out


def test_every_kernel_launch_goes_through_aq_launch():
    """aq_launch (csrc/aq_common.cuh) sets the shared-memory limit, chooses a programmatic launch and counts the launch
    (aq_launch_count, bench.py's gpu_launches); a launch written any other way would go uncounted."""
    csrc = os.path.join(ROOT, "alphaquoridorgnn_b200", "csrc")
    for name in sorted(os.listdir(csrc)):
        with open(os.path.join(csrc, name)) as f:
            text = f.read()
        assert "<<<" not in text, name
        if name != "aq_common.cuh":
            assert "cudaLaunchKernelEx" not in text and "cudaFuncSetAttribute" not in text, name


def test_host_packing_matches_struct_layout(traj):
    rows, plies = traj["rows"][:5000], traj["plies"][:5000]
    packed = gl.pack_rows_host(rows, plies)
    assert packed.shape == (5000, 32) and packed.dtype == np.uint8
    h = packed[:, 0:8].copy().view(np.uint64)[:, 0]
    v = packed[:, 8:16].copy().view(np.uint64)[:, 0]
    for s in (0, 7, 31, 32, 63):
        assert np.array_equal((h >> np.uint64(s)) & np.uint64(1), (rows[:, 4 + s] == 1).astype(np.uint64))
        assert np.array_equal((v >> np.uint64(s)) & np.uint64(1), (rows[:, 4 + s] == 2).astype(np.uint64))
    assert np.array_equal(packed[:, 16:20], rows[:, 0:4])
    assert np.array_equal(packed[:, 20:22].copy().view(np.uint16)[:, 0], plies.astype(np.uint16))
    assert not packed[:, 22:].any()


def test_rows_from_arrays_and_state_record_keeping():
    s = gl.State()
    assert s.player == [76, 10] and s.enemy == [76, 10] and len(s.walls) == 64
    t = s.next(67)
    assert t.player == [76, 10] and t.enemy == [67, 10] and t.plies_played == 1          # KA7
    t = s.next(81)
    assert t.enemy == [76, 9] and t.walls[63] == 1                                           # KA8
    t = s.next(81 + 64 + 9)
    assert t.walls[54] == 2                                                                  # KA9
    assert gl.State(player=[40, 5], enemy=[5, 5]).is_lose()
    assert gl.State(plies_played=116).is_draw() and not gl.State(plies_played=115).is_draw()  # KA12
    rows = gl.rows_from_arrays([s.to_array(), t.to_array()])
    assert rows.shape == (2, 68) and rows[0, 0] == 76 and rows[1, 4 + 54] == 2
    with pytest.raises(ValueError):
        gl.State(board_size=5)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_fails_loudly_without_cuda():
    with pytest.raises(_lib.AqError):
        gl.State().legal_actions()
    from alphaquoridorgnn_b200.pv_network_gnn import GNNNetwork
    net = GNNNetwork()
    with pytest.raises(_lib.AqError):
        net(torch.zeros((1, 68), dtype=torch.uint8))
    with pytest.raises(_lib.AqError):
        net.predict(gl.State())
