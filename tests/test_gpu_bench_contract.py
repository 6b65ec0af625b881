"""bench.py prints ONE JSON line with every key its readers rely on (a short run at a small batch), and --dump-outputs writes what its
last timed step computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
B, STEPS = 2048, 3


@pytest.fixture(scope="module")
def bench_run(tmp_path_factory):
    dump = str(tmp_path_factory.mktemp("bench_outputs"))
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(STEPS), "--warmup", "3", "--batch", str(B),
                          "--skip-extra", "--skip-cpu", "--dump-outputs", dump], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0]), dump


def test_bench_line_has_every_contract_key(bench_run):
    d, _ = bench_run
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
              "data", "config", "roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks", "kernels", "extra"):
        assert k in d, k
    assert d["steps"] == 3 and d["n_gpus"] == 1 and d["value"] > 0 and d["gpu_launches"] > 0
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert k in d["roofline"], k
    for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"):
        assert k in d["e2e"], k
    assert d["e2e"]["value"] > 0 and d["e2e"]["value"] != d["value"]
    assert "workload" in d["config"] and "sm_mhz" in d["clocks"]


def test_dumped_outputs_are_the_last_timed_step(bench_run):
    """The dump equals GNNNetwork.predict_batch on the batch of the last timed step, rebuilt from bench.py's seeds (weights from seed 0,
    positions.mixed_batches(4, B, seed=1); timed step i evaluates batch i % 4)."""
    import torch
    from alphaquoridorgnn_b200 import positions
    from alphaquoridorgnn_b200.pv_network_gnn import GNNNetwork
    d, dump = bench_run
    names = ("board_index", "priors", "value", "mask", "pawn")
    assert sorted(os.listdir(dump)) == sorted(n + ".npy" for n in names)
    assert sum(os.path.getsize(os.path.join(dump, f)) for f in os.listdir(dump)) <= 64 << 20
    got = {n: np.load(os.path.join(dump, n + ".npy")) for n in names}
    assert all(v.dtype in (np.float32, np.float64) for v in got.values())
    assert np.array_equal(got["board_index"], np.arange(B))
    torch.manual_seed(0)
    net = GNNNetwork().cuda().eval()
    net.precision = d["config"]["precision"]
    _, batches = positions.mixed_batches(4, B, seed=1, device="cuda:0")
    want = net.predict_batch(batches[(STEPS - 1) % 4])
    assert np.array_equal(got["mask"], want["mask"].cpu().numpy().view(np.uint32).astype(np.float64))
    assert np.array_equal(got["pawn"], want["pawn"].cpu().numpy().astype(np.float32))
    assert np.abs(got["priors"] - want["priors"].cpu().numpy()).max() <= 1e-6
    assert np.abs(got["value"] - want["value"].cpu().numpy()).max() <= 1e-6
