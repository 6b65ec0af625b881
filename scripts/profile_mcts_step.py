"""Three simulation steps of the lock-step MCTS at G = 4,096 (after 60 steps of warm-up, so that the trees have depth) bracketed by
cudaProfilerStart/Stop:  ncu --profile-from-start off --metrics gpu__time_duration.sum ... python scripts/profile_mcts_step.py"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from alphaquoridorgnn_b200 import _lib, positions, pv_mcts
from alphaquoridorgnn_b200.pv_network_gnn import GNNNetwork, PRECISIONS

G, sims = 4096, 200
torch.manual_seed(0)
net = GNNNetwork().cuda().eval()
net.precision = "bf16"
roots = positions.random_positions(G, seed=5, games=G)
m = pv_mcts.BatchedMCTS(net, sims, use_graph=False)
L, P = _lib.load(), _lib.ptr
max_nodes = 1 + sims * pv_mcts.MAX_CHILDREN
ws, buf = m._workspace(G, max_nodes), m._buffers(G)
st = _lib.stream_ptr()
L.aq_mcts_reset(P(ws), P(roots), G, max_nodes, st)
flat, prep = net.flat_parameters(), net.prepared_weights()


def evaluate(s):
    _lib.check(L.aq_leaf_eval(P(flat), P(prep), P(buf["leaf"]), G, P(buf["priors"]), P(buf["value"]), P(buf["mask"]), P(buf["pawn"]),
                              P(buf["pooled"]), PRECISIONS["bf16"], s), "aq_leaf_eval")
    return buf


for _ in range(60):
    m._step(ws, G, max_nodes, buf, evaluate, st)
torch.cuda.synchronize()
torch.cuda.profiler.start()
for _ in range(3):
    m._step(ws, G, max_nodes, buf, evaluate, st)
torch.cuda.synchronize()
torch.cuda.profiler.stop()
print("done")
