"""CPU oracle for the floating-point half of the hot path -- TEST INFRASTRUCTURE, NOT PRODUCT.

Restates ``GraphPolicyValueNetwork`` (/root/reference/pv_network_gnn.py:23-64) in plain
PyTorch.  The reference builds its layers from ``torch_geometric.nn.GCNConv`` and
``global_mean_pool`` (pv_network_gnn.py:13,33,35,56,59).  torch_geometric is NOT vendored in
/root/reference, NOT pinned by its requirements.txt, and NOT installed in this image, so the
arithmetic below restates the published PyG 2.x algorithm with GCNConv's default arguments
(improved=False, cached=False, add_self_loops=True, normalize=True, bias=True, aggr='add',
flow='source_to_target'; SURVEY.md section 3.4).

PARITY UNPINNED: the reference ships no test, golden vector or checkpoint for the GNN, and the
third-party layer cannot be imported here.  What pins this file instead is
``dense_forward_fp64`` -- an independent dense-matrix restatement (A_hat = D^-1/2 (A+I) D^-1/2
built from the reference's own is_wall_blocking via the golden open-direction masks) that
tests/test_oracle_gnn.py compares with the edge-list formulation.

state_dict keys equal the reference's (gcn_layers.{i}.lin.weight, gcn_layers.{i}.bias,
policy_head.{0,2}.{weight,bias}, value_head.{0,2}.{weight,bias}).
"""
import copy
import math

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

NUM_FEATURES = 6          # pv_network_gnn.py:17
HIDDEN_DIM = 128          # pv_network_gnn.py:18
NUM_GCN_LAYERS = 3        # pv_network_gnn.py:19
BOARD_SIZE = 9
POLICY_OUTPUT_SIZE = BOARD_SIZE ** 2 + 2 * (BOARD_SIZE - 1) ** 2  # pv_network_gnn.py:20


def gcn_norm(edge_index, num_nodes, dtype):
    """PyG gcn_norm with add_self_loops=True, improved=False, flow='source_to_target':
    drop existing self loops, append (i,i) for every node with weight 1, degree over the
    TARGET index, w_e = deg^-1/2[src] * deg^-1/2[dst], inf -> 0."""
    src, dst = edge_index[0], edge_index[1]
    keep = src != dst
    loops = torch.arange(num_nodes, dtype=edge_index.dtype, device=edge_index.device)
    src = torch.cat([src[keep], loops])
    dst = torch.cat([dst[keep], loops])
    ones = torch.ones(src.numel(), dtype=dtype, device=edge_index.device)
    deg = torch.zeros(num_nodes, dtype=dtype, device=edge_index.device).index_add_(0, dst, ones)
    dis = deg.pow(-0.5)
    dis = dis.masked_fill(torch.isinf(dis), 0.0)
    return src, dst, dis[src] * ones * dis[dst]


class _Lin(nn.Module):
    """PyG ``Linear(in, out, bias=False, weight_initializer='glorot')``."""

    def __init__(self, n_in, n_out):
        super().__init__()
        self.weight = nn.Parameter(torch.empty(n_out, n_in))
        a = math.sqrt(6.0 / (n_in + n_out))
        nn.init.uniform_(self.weight, -a, a)

    def forward(self, x):
        return x @ self.weight.t()


class GCNConvOracle(nn.Module):
    """GCNConv(in, out) with default kwargs: out = scatter_add(w_e * (x W^T)[src] -> dst) + bias."""

    def __init__(self, n_in, n_out):
        super().__init__()
        self.lin = _Lin(n_in, n_out)
        self.bias = nn.Parameter(torch.zeros(n_out))

    def forward(self, x, edge_index):
        src, dst, w = gcn_norm(edge_index, x.shape[0], x.dtype)  # cached=False: every call
        z = self.lin(x)
        out = torch.zeros_like(z).index_add_(0, dst, w.unsqueeze(1) * z[src])
        return out + self.bias


def global_mean_pool(x, batch, num_graphs=None):
    if num_graphs is None:
        num_graphs = int(batch.max().item()) + 1
    s = torch.zeros(num_graphs, x.shape[1], dtype=x.dtype, device=x.device).index_add_(0, batch, x)
    c = torch.zeros(num_graphs, dtype=x.dtype, device=x.device).index_add_(0, batch, torch.ones_like(batch, dtype=x.dtype))
    return s / c.clamp(min=1).unsqueeze(1)


class GraphPolicyValueNetworkOracle(nn.Module):
    """pv_network_gnn.py:23-64."""

    def __init__(self, num_features=NUM_FEATURES, hidden_dim=HIDDEN_DIM, num_gcn_layers=NUM_GCN_LAYERS,
                 policy_output_size=POLICY_OUTPUT_SIZE):
        super().__init__()
        self.gcn_layers = nn.ModuleList([GCNConvOracle(num_features, hidden_dim)])
        for _ in range(num_gcn_layers - 1):
            self.gcn_layers.append(GCNConvOracle(hidden_dim, hidden_dim))
        self.policy_head = nn.Sequential(nn.Linear(hidden_dim, hidden_dim // 2), nn.ReLU(),
                                         nn.Linear(hidden_dim // 2, policy_output_size), nn.Softmax(dim=1))
        self.value_head = nn.Sequential(nn.Linear(hidden_dim, hidden_dim // 2), nn.ReLU(),
                                        nn.Linear(hidden_dim // 2, 1), nn.Tanh())

    def forward(self, x, edge_index, batch):
        for layer in self.gcn_layers:
            x = F.relu(layer(x, edge_index))
        x = global_mean_pool(x, batch)
        return self.policy_head(x), self.value_head(x)


def training_loss(policy_pred, value_pred, policy_target, value_target):
    """train_network.py:54-55,85-89: CrossEntropyLoss applied to the network's SOFTMAX
    OUTPUT (so log_softmax runs on probabilities -- kept literally) + MSELoss, both 'mean'."""
    policy_loss = nn.CrossEntropyLoss()(policy_pred, policy_target)
    value_loss = nn.MSELoss()(value_pred.squeeze(), value_target)
    return policy_loss + value_loss, policy_loss, value_loss


# ---- graph inputs from row68 states (uses the integer oracle) ------------------------------
def graph_inputs_from_rows(rows, dtype=torch.float32):
    """rows uint8[B,68] -> (x [B*81,6], edge_index int64[2,E], batch int64[B*81]) in the
    canonical layout of SURVEY.md section 8a A6 (nodes row-major, per node U,D,L,R)."""
    from oracle import quoridor_oracle as qo

    rows = np.ascontiguousarray(rows, dtype=np.uint8)
    B = rows.shape[0]
    planes = qo.planes_batch(rows)                      # [B,6,9,9]
    x = torch.from_numpy(planes.reshape(B, 6, 81).transpose(0, 2, 1).reshape(B * 81, 6).copy()).to(dtype)
    opn = qo.open_mask_batch(rows)                      # [B,81]
    off = np.array([-9, 9, -1, 1])
    srcs, dsts = [], []
    node = np.arange(81)
    for d in range(4):
        has = ((opn >> d) & 1).astype(bool)             # [B,81]
        b, v = np.nonzero(has)
        srcs.append(b * 81 + v)
        dsts.append(b * 81 + v + off[d])
    src = np.concatenate(srcs)
    dst = np.concatenate(dsts)
    order = np.lexsort((dst, src))  # deterministic; summation order is not part of the contract
    edge_index = torch.from_numpy(np.stack([src[order], dst[order]]).astype(np.int64))
    batch = torch.from_numpy(np.repeat(np.arange(B), 81).astype(np.int64))
    del node
    return x, edge_index, batch


def dense_forward_fp64(state_dict, rows):
    """Independent dense restatement in numpy float64: X_{l+1} = relu(A_hat (X_l W^T) + b)."""
    from oracle import quoridor_oracle as qo

    rows = np.ascontiguousarray(rows, dtype=np.uint8)
    B = rows.shape[0]
    sd = {k: v.detach().double().cpu().numpy() for k, v in state_dict.items()}
    planes = qo.planes_batch(rows).astype(np.float64)
    opn = qo.open_mask_batch(rows)
    off = (-9, 9, -1, 1)
    pol = np.zeros((B, sd["policy_head.2.weight"].shape[0]))
    val = np.zeros((B, 1))
    n_layers = len([k for k in sd if k.endswith("lin.weight")])
    for b in range(B):
        A = np.eye(81)
        for v in range(81):
            for d in range(4):
                if (opn[b, v] >> d) & 1:
                    A[v + off[d], v] = 1.0  # message from source v into target v+off
        deg = A.sum(axis=1)                 # in-degree incl. self loop
        dis = deg ** -0.5
        Ahat = dis[:, None] * A * dis[None, :]
        X = planes[b].reshape(6, 81).T
        for l in range(n_layers):
            X = np.maximum(Ahat @ (X @ sd[f"gcn_layers.{l}.lin.weight"].T) + sd[f"gcn_layers.{l}.bias"], 0.0)
        g = X.mean(axis=0)
        h = np.maximum(sd["policy_head.0.weight"] @ g + sd["policy_head.0.bias"], 0.0)
        z = sd["policy_head.2.weight"] @ h + sd["policy_head.2.bias"]
        z = np.exp(z - z.max())
        pol[b] = z / z.sum()
        h = np.maximum(sd["value_head.0.weight"] @ g + sd["value_head.0.bias"], 0.0)
        val[b] = np.tanh(sd["value_head.2.weight"] @ h + sd["value_head.2.bias"])
    return pol, val


# ---- the tensor-core path's rounding points, emulated (test infrastructure) -----------------------------------------------
class _Round(torch.autograd.Function):
    """x -> x rounded to bfloat16 / float16 and back, gradient passed straight through: what storing an operand in a 16-bit tile
    does to the forward pass, with the backward pass seeing the rounded operand (as the kernels' saved tiles do)."""

    @staticmethod
    def forward(ctx, t, dtype):
        return t.to(torch.float32).to(dtype).to(t.dtype)

    @staticmethod
    def backward(ctx, g):
        return g, None


def forward_tc_emulation(model, x, edge_index, batch):
    """GraphPolicyValueNetworkOracle.forward with the rounding points of the bf16 tensor-core path (DESIGN.md section 5) and exact
    (caller's dtype, normally float64) accumulation everywhere else:
      trunk  W1, W2, W3 -> bf16; X1, X2 -> bf16 (the feature-major tiles); Z2, Z3 -> fp16 and the A_hat coefficients -> fp16 (the
             aggregation MMA's operands); layer 1's 6-wide input is carried as a bf16 hi/lo pair (~16 mantissa bits: left exact here);
             the last layer feeds the mean pool from the fp32 accumulator (no rounding);
      heads  pooled -> bf16, Wp0, Wv0, Wp2 -> bf16, policy hidden -> bf16; the value head's second layer, biases, softmax and tanh in
             full precision.
    Comparing the CUDA path with THIS isolates kernel errors from the error bf16 operands imply (the difference between this and the
    exact forward is what the stated bf16 tolerances cover)."""
    bf, hf = torch.bfloat16, torch.float16
    src, dst, w = gcn_norm(edge_index, x.shape[0], x.dtype)
    h = x
    n_layers = len(model.gcn_layers)
    for i, layer in enumerate(model.gcn_layers):
        z = h @ _Round.apply(layer.lin.weight, bf).t()
        we = w
        if i > 0:
            z, we = _Round.apply(z, hf), _Round.apply(w, hf)
        out = torch.zeros_like(z).index_add_(0, dst, we.unsqueeze(1) * z[src]) + layer.bias
        h = F.relu(out)
        if i + 1 < n_layers:
            h = _Round.apply(h, bf)
    g = _Round.apply(global_mean_pool(h, batch), bf)
    ph, vh = model.policy_head, model.value_head
    hp = _Round.apply(F.relu(g @ _Round.apply(ph[0].weight, bf).t() + ph[0].bias), bf)
    policy = torch.softmax(hp @ _Round.apply(ph[2].weight, bf).t() + ph[2].bias, dim=1)
    hv = F.relu(g @ _Round.apply(vh[0].weight, bf).t() + vh[0].bias)
    value = torch.tanh(hv @ vh[2].weight.t() + vh[2].bias)
    return policy, value


# ---- training-gradient references (test infrastructure) ------------------------------------------------------------------------
def oracle_grads_fp64(ref, rows, pt, vt, chunk=512, emulate_tc=False):
    """fp64 oracle autograd of the reference loss (train_network.py:54-55,85-89: both 'mean' over the batch), accumulated over chunks
    of boards so that the edge-list formulation fits in memory: mean over B = sum over chunks of (chunk mean x n_chunk / B).
    emulate_tc: the forward pass carries the tensor-core path's rounding points (forward_tc_emulation).
    Returns (loss, {parameter name: gradient})."""
    ref64 = copy.deepcopy(ref).double()
    B = len(rows)
    total = 0.0
    for lo in range(0, B, chunk):
        hi = min(B, lo + chunk)
        x, ei, batch = graph_inputs_from_rows(rows[lo:hi], dtype=torch.float64)
        p64, v64 = forward_tc_emulation(ref64, x, ei, batch) if emulate_tc else ref64(x, ei, batch)
        loss, _, _ = training_loss(p64, v64, pt[lo:hi].double(), vt[lo:hi].double())
        (loss * ((hi - lo) / B)).backward()
        total += loss.item() * (hi - lo) / B
    return total, {n: p.grad for n, p in ref64.named_parameters()}


def probe_upstream(row_ids):
    """Upstream gradient of probe boards: dpolicy ~ N(0,1)[209] and dvalue ~ N(0,1) in float32, drawn from a generator seeded by each
    board's row id -- the same board gets the same upstream gradient in every batch it is placed in.  -> (dpolicy [n,209], dvalue [n])."""
    dp = np.empty((len(row_ids), POLICY_OUTPUT_SIZE), np.float32)
    dv = np.empty((len(row_ids),), np.float32)
    for i, r in enumerate(row_ids):
        g = np.random.default_rng(int(r))
        dp[i] = g.standard_normal(POLICY_OUTPUT_SIZE, dtype=np.float32)
        dv[i] = g.standard_normal(dtype=np.float32)
    return dp, dv


def probe_grads_fp64(ref, rows, dpolicy, dvalue, emulate_tc=False):
    """fp64 gradient with respect to the parameters of sum_b (policy_b . dpolicy_b + value_b * dvalue_b) over the given boards.
    Every operation from the outputs back to the weights is linear in the upstream gradient, so this is also the gradient of any
    larger batch that holds these boards and has zero upstream rows everywhere else (as long as its activations are finite): a
    reference for a few probe boards of a batch of any size.  emulate_tc as in oracle_grads_fp64.  -> {parameter name: gradient}."""
    ref64 = copy.deepcopy(ref).double()
    x, ei, batch = graph_inputs_from_rows(rows, dtype=torch.float64)
    p64, v64 = forward_tc_emulation(ref64, x, ei, batch) if emulate_tc else ref64(x, ei, batch)
    dp = torch.as_tensor(np.asarray(dpolicy), dtype=torch.float64).reshape(p64.shape)
    dv = torch.as_tensor(np.asarray(dvalue), dtype=torch.float64).reshape(v64.shape)
    ((p64 * dp).sum() + (v64 * dv).sum()).backward()
    return {n: p.grad for n, p in ref64.named_parameters()}
