"""Where CUDA-graph capture is not supported, the tree search and the training step warn once, run eagerly from then on and compute
what their use_graph=False twins compute.  Capture is refused in torch.cuda.CUDAGraph.capture_begin, before any stream capture
begins."""
import numpy as np
import pytest
import torch

from alphaquoridorgnn_b200 import game_logic as gl
from alphaquoridorgnn_b200 import positions, pv_mcts, train_network
from alphaquoridorgnn_b200.pv_network_gnn import GNNNetwork

pytestmark = pytest.mark.gpu


@pytest.fixture
def no_capture(monkeypatch):
    def refuse(self, *args, **kwargs):
        raise RuntimeError("stream capture is not supported here")
    monkeypatch.setattr(torch.cuda.CUDAGraph, "capture_begin", refuse)


def _net(seed):
    torch.manual_seed(seed)
    return GNNNetwork().cuda().eval()


def test_search_without_capture_is_the_eager_search(no_capture):
    net = _net(1)
    roots = positions.random_positions(64, seed=4, games=64)
    graph = pv_mcts.BatchedMCTS(net, 40)
    eager = pv_mcts.BatchedMCTS(net, 40, use_graph=False)
    with pytest.warns(UserWarning, match="CUDA-graph capture of the MCTS simulation step failed"):
        c1, a1, n1 = graph.search(roots)
    assert not graph.use_graph and not graph._graphs
    c2, a2, n2 = eager.search(roots)
    assert torch.equal(c1, c2) and torch.equal(a1, a2) and torch.equal(n1, n2)
    assert int(c1.sum(1).min()) == 39


def test_training_step_without_capture_is_the_eager_step(no_capture, traj):
    rng = np.random.default_rng(2)
    packed = gl.pack_rows(traj["rows"][rng.choice(len(traj["rows"]), 200, replace=False)])
    torch.manual_seed(4)
    pt = torch.softmax(2 * torch.randn(200, 209), 1).cuda()
    vt = torch.randint(-1, 2, (200,)).float().cuda()
    graph = train_network.FlatTrainer(_net(7).train(), lr=1e-3)
    eager = train_network.FlatTrainer(_net(7).train(), lr=1e-3, use_graph=False)
    with pytest.warns(UserWarning, match="CUDA-graph capture of the training step failed"):
        for step in range(3):   # the second step with the same inputs is the one that captures
            lg = graph.step(packed, pt, vt, 200).clone()
            le = eager.step(packed, pt, vt, 200).clone()
            assert graph.use_graph == (step == 0)
            # the loss scalars are summed with float atomics, in an order that differs from launch to launch
            assert (lg - le).abs().max().item() <= 1e-5
            assert torch.equal(graph.grads, eager.grads) and torch.equal(graph.flat, eager.flat)
    assert graph.kernels_per_step == eager.kernels_per_step
    graph.check()
