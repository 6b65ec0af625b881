"""Network training -- drop-in for reference train_network.py (train_network.py:14-107): newest
./data/*.history, batch 128 shuffled, loss = CrossEntropyLoss(softmax output, target) + MSELoss,
Adam(lr=1e-3) with the 1.0 / 0.5 / 0.25 LambdaLR schedule, 100 epochs, weights saved to latest.pth.

The step runs entirely in libaqgnn.so on flat buffers (forward with saved activations, fused loss
gradient, atomic-free backward, Adam).  Data parallel: every rank computes its slice of each global
batch, gradients are summed with ONE all-reduce of the flat 64,082-float buffer (NCCL over NVLink on
GPUs), and every rank applies the identical Adam update."""
import os
import pickle
from pathlib import Path

import numpy as np
import torch

from . import _lib
from . import game_logic as gl
from .constants import PV_NETWORK_PATH
from .pv_network_gnn import GNNNetwork, POLICY_OUTPUT_SIZE

NUM_EPOCH = 100   # train_network.py:14
BATCH_SIZE = 128  # train_network.py:15


def load_data(directory='./data'):
    # Load the latest training data (train_network.py:18-23)
    history_path = sorted(Path(directory).glob('*.history'))[-1]
    with history_path.open(mode='rb') as f:
        return pickle.load(f)


def lr_lambda(epoch):
    """train_network.py:59-65"""
    if epoch >= 80:
        return 0.25
    elif epoch >= 50:
        return 0.5
    return 1.0


def shard_bounds(n, rank, world_size):
    """Contiguous split of a batch of n samples over the ranks (sizes differ by at most one)."""
    base, rem = divmod(n, world_size)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


class PeerAccessUnavailable(_lib.AqError):
    """The ranks cannot map each other's memory (no CUDA IPC / no peer access between the GPUs)."""


class PeerCommunicator:
    """The ranks of one box mapped into each other's address space (CUDA IPC over NVLink; csrc/dp_comm.cu), for the fused
    all-reduce + Adam kernel.  Handles are exchanged through torch.distributed (any backend)."""

    def __init__(self, rank, world_size, device):
        import ctypes
        self.L = _lib.load()
        self.rank, self.world, self.device = rank, world_size, device
        self._h = ctypes.c_void_p()
        handle = (ctypes.c_ubyte * 64)()
        with torch.cuda.device(device):
            rc = self.L.aq_comm_create(rank, world_size, ctypes.byref(self._h), handle)
            err = self.L.aq_last_error_string().decode() if rc else ""
            if world_size == 1:
                _lib.check(rc, "aq_comm_create")
                return
            # every rank must take the same decision: exchange (ok, handle), map the peers, exchange ok again
            import torch.distributed as dist
            gathered = [None] * world_size
            dist.all_gather_object(gathered, (rc == 0, bytes(handle), err))
            if all(g[0] for g in gathered):
                blob = (ctypes.c_ubyte * (64 * world_size)).from_buffer_copy(b"".join(g[1] for g in gathered))
                rc = self.L.aq_comm_open(self._h, blob)
                err = self.L.aq_last_error_string().decode() if rc else ""
                opened = [None] * world_size
                dist.all_gather_object(opened, (rc == 0, err))
                bad = [f"rank {r}: {e}" for r, (ok, e) in enumerate(opened) if not ok]
            else:
                bad = [f"rank {r}: {g[2]}" for r, g in enumerate(gathered) if not g[0]]
            if bad:
                self.close()
                raise PeerAccessUnavailable("; ".join(bad))

    @property
    def handle(self):
        return self._h

    def status(self):
        """-> (optimiser steps completed on the device, status: 0 ok, 1 = a peer did not arrive in time).  Synchronises."""
        import ctypes
        out = (ctypes.c_int64 * 2)()
        with torch.cuda.device(self.device):
            _lib.check(self.L.aq_comm_status(self._h, out, _lib.stream_ptr(self.device)), "aq_comm_status")
        return int(out[0]), int(out[1])

    def set_step(self, step, betas=(0.9, 0.999)):
        with torch.cuda.device(self.device):
            _lib.check(self.L.aq_comm_set_step(self._h, int(step), betas[0], betas[1], _lib.stream_ptr(self.device)), "aq_comm_set_step")

    def close(self):
        if self._h:
            with torch.cuda.device(self.device):
                self.L.aq_comm_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class FlatTrainer:
    """One model replica + Adam state on flat buffers; step() = forward / loss / backward / gradient all-reduce / Adam.

    collective: "p2p"  -- the default: the optimiser step is ONE kernel that reduces the partial gradients, all-reduces them over
                          NVLink peer memory and applies Adam (aq_train_backward_step; csrc/dp_comm.cu); the whole step is 6 kernels
                          and is replayed as a CUDA graph per batch shape (use_graph);
                "nccl" -- the checked alternative: the same backward kernels, torch.distributed.all_reduce of the flat gradient,
                          aq_adam_step.  Also what a world spanning several boxes needs."""

    def __init__(self, model, lr=0.001, betas=(0.9, 0.999), eps=1e-8, rank=0, world_size=1, precision=None, collective="p2p",
                 use_graph=True):
        from .pv_network_gnn import PRECISIONS
        if collective not in ("p2p", "nccl"):
            raise ValueError("collective must be 'p2p' or 'nccl'")
        self.model, self.lr, self.betas, self.eps = model, lr, betas, eps
        self.prec = PRECISIONS[precision if precision is not None else model.train_precision]
        self.rank, self.world = rank, world_size
        self.flat = model.flat_parameters()
        _lib.require_cuda(self.flat, "model parameters")
        self.exp_avg = torch.zeros_like(self.flat)
        self.exp_avg_sq = torch.zeros_like(self.flat)
        self.grads = torch.zeros_like(self.flat)
        self.step_count = 0
        self.loss = torch.zeros(2, device=self.flat.device)
        self.collective, self.use_graph = collective, use_graph
        self.comm = None
        if collective == "p2p":
            try:
                self.comm = PeerCommunicator(rank, world_size, self.flat.device)
            except PeerAccessUnavailable as e:  # raised on every rank alike (the ranks exchange their outcome)
                import warnings
                warnings.warn(f"peer memory is not available ({e}); the gradient all-reduce falls back to torch.distributed")
                self.collective = "nccl"
        self._bufs, self._graphs = {}, {}
        self.kernels_per_step = None   # this library's kernel launches in one step, counted on the last eagerly run step

    def _buffers(self, b):
        buf = self._bufs.get(b)
        if buf is None:
            L, dev = _lib.load(), self.flat.device
            if len(self._bufs) >= 8:  # a training loop has one full batch size and one tail (each with workspace + inputs)
                self._bufs.clear()
                self._graphs.clear()
            buf = self._bufs[b] = {
                "policy": torch.empty((b, POLICY_OUTPUT_SIZE), dtype=torch.float32, device=dev),
                "value": torch.empty((b,), dtype=torch.float32, device=dev),
                "saved": torch.empty((L.aq_gnn_saved_floats(b),), dtype=torch.float32, device=dev),
                "ws": torch.empty((L.aq_gnn_backward_ws_floats(b),), dtype=torch.float32, device=dev),
                "dp": torch.empty((b, POLICY_OUTPUT_SIZE), dtype=torch.float32, device=dev) if self.collective == "nccl" else None,
                "dv": torch.empty((b,), dtype=torch.float32, device=dev) if self.collective == "nccl" else None,
            }
        return buf

    def inputs(self, b):
        """Persistent input tensors (packed uint8[b,32], policy_target f32[b,209], value_target f32[b]) a data loader can fill in
        place (e.g. torch.index_select(..., out=...)): a step on tensors whose addresses repeat is replayed as one CUDA graph."""
        key = ("in", b)
        buf = self._bufs.get(key)
        if buf is None:
            dev = self.flat.device
            buf = self._bufs[key] = (torch.empty((b, gl.STATE_BYTES), dtype=torch.uint8, device=dev),
                                     torch.empty((b, POLICY_OUTPUT_SIZE), dtype=torch.float32, device=dev),
                                     torch.empty((b,), dtype=torch.float32, device=dev))
        return buf

    def _enqueue(self, buf, packed, policy_target, value_target, b, global_batch, lr, st):
        """The library calls of one step on stream `st` (eagerly, or under CUDA-graph capture)."""
        L, P = _lib.load(), _lib.ptr
        c0 = L.aq_launch_count()
        _lib.check(L.aq_gnn_forward(P(self.flat), P(packed), None, None, b, P(buf["policy"]), P(buf["value"]), P(buf["saved"]), self.prec, st),
                   "aq_gnn_forward")
        _lib.check(L.aq_train_backward_step(self.comm.handle, P(self.flat), P(buf["saved"]), P(policy_target), P(value_target), b, global_batch,
                                            P(self.loss), P(self.grads), P(self.exp_avg), P(self.exp_avg_sq), P(buf["ws"]), self.prec, lr,
                                            self.betas[0], self.betas[1], self.eps, st), "aq_train_backward_step")
        self.kernels_per_step = L.aq_launch_count() - c0

    def step(self, packed, policy_target, value_target, global_batch, lr_scale=1.0):
        """packed uint8[b,32], policy_target f32[b,209], value_target f32[b]: this rank's slice of a
        global batch of `global_batch` samples (b may be 0).  Returns the loss tensor [policy, value]
        contribution of this rank (already divided by the global batch size)."""
        L, P = _lib.load(), _lib.ptr
        flat = self.model.flat_parameters()
        if flat.data_ptr() != self.flat.data_ptr() or flat.device != self.flat.device:
            # the module was moved (.to) or its storage replaced (load_state_dict(assign=True)) since the last step: follow it, keep
            # the Adam moments (on the new device), so that the update does not go into an orphaned buffer
            if self.comm is not None and flat.device != self.flat.device:
                raise _lib.AqError("the model moved to another device: create a new FlatTrainer (its peer communicator is bound to the old one)")
            self.flat = flat
            self.exp_avg, self.exp_avg_sq = self.exp_avg.to(flat.device), self.exp_avg_sq.to(flat.device)
            self.grads, self.loss = torch.zeros_like(flat), torch.zeros(2, device=flat.device)
            self._bufs.clear()
            self._graphs.clear()
        dev = self.flat.device
        b = packed.shape[0]
        lr = float(self.lr * lr_scale)
        with torch.cuda.device(dev):
            st = _lib.stream_ptr(dev)
            if self.collective == "p2p":
                if b == 0:  # an empty shard still takes part in the exchange: zero gradient through the plain entry point
                    self.grads.zero_()
                    self.loss.zero_()
                    _lib.check(L.aq_dp_adam_step(self.comm.handle, P(self.flat), P(self.grads), P(self.exp_avg), P(self.exp_avg_sq), lr,
                                                 self.betas[0], self.betas[1], self.eps, st), "aq_dp_adam_step")
                else:
                    for t, name in ((packed, "packed"), (policy_target, "policy_target"), (value_target, "value_target")):
                        if not (t.is_cuda and t.is_contiguous()):
                            raise ValueError(f"{name} must be a contiguous CUDA tensor")
                    buf = self._buffers(b)
                    args = (buf, packed, policy_target, value_target, b, int(global_batch), lr)
                    # a step whose input addresses repeat (FlatTrainer.inputs(), or a loader that reuses its batch tensors) is
                    # replayed as one CUDA graph; the first step with a key runs eagerly, the second is captured
                    key = (b, int(global_batch), lr, packed.data_ptr(), policy_target.data_ptr(), value_target.data_ptr())
                    graph = self._graphs.get(key) if self.use_graph else None
                    if self.use_graph and graph is None and key in self._graphs:
                        graph = self._graphs[key] = _lib.capture_graph(dev, lambda cst: self._enqueue(*args, cst), "the training step")
                        self.use_graph = graph is not None
                    if graph is not None:
                        graph.replay()   # also right after the capture: capture records, it does not execute
                    else:
                        if self.use_graph:
                            if len(self._graphs) >= 16:
                                self._graphs.clear()
                            self._graphs[key] = None
                        self._enqueue(*args, st)
                self.step_count += 1
            else:
                if b > 0:
                    buf = self._buffers(b)
                    _lib.check(L.aq_gnn_forward(P(self.flat), P(packed), None, None, b, P(buf["policy"]), P(buf["value"]), P(buf["saved"]), self.prec, st),
                               "aq_gnn_forward")
                    _lib.check(L.aq_loss_grad(P(buf["policy"]), P(buf["value"]), P(policy_target), P(value_target), b, global_batch, P(self.loss),
                                              P(buf["dp"]), P(buf["dv"]), st), "aq_loss_grad")
                    _lib.check(L.aq_gnn_backward(P(self.flat), P(buf["saved"]), P(buf["dp"]), P(buf["dv"]), b, P(self.grads), P(buf["ws"]), self.prec, st),
                               "aq_gnn_backward")
                else:
                    self.grads.zero_()
                    self.loss.zero_()
                if self.world > 1:
                    import torch.distributed as dist
                    dist.all_reduce(self.grads)  # one 256 KB all-reduce per step; losses divide by the global batch already
                self.step_count += 1
                _lib.check(L.aq_adam_step(P(self.flat), P(self.grads), P(self.exp_avg), P(self.exp_avg_sq), self.flat.numel(),
                                          self.step_count, lr, self.betas[0], self.betas[1], self.eps, 1.0, st),
                           "aq_adam_step")
        if hasattr(self.model, "mark_weights_changed"):
            self.model.mark_weights_changed()  # the flat buffer was written through a raw pointer
        return self.loss

    def check(self):
        """Synchronises and raises if the peer exchange timed out or the device step counter disagrees with the host's."""
        if self.comm is not None:
            steps, status = self.comm.status()
            if status:
                raise _lib.AqError("data-parallel step: a peer rank did not arrive within the kernel's time-out")
            if steps != self.step_count:
                raise _lib.AqError(f"device step counter {steps} != host step count {self.step_count}")


def train_on_history(model, history, num_epochs=NUM_EPOCH, batch_size=BATCH_SIZE, rank=0, world_size=1, seed=0,
                     verbose=True):
    """The training loop of train_network.py:69-104 on an in-memory history."""
    dev = model.flat_parameters().device
    s, p, v = zip(*history)
    rows = model.preprocess_input(s)                                   # train_network.py:37
    packed = gl.pack_rows(rows, None, dev)
    p = torch.tensor(np.array(p), dtype=torch.float32, device=dev)     # policy targets
    v = torch.tensor(np.array(v), dtype=torch.float32, device=dev)     # value targets
    return train_on_buffer(model, packed, p, v, num_epochs, batch_size, rank, world_size, seed, verbose)


def train_on_buffer(model, packed, p, v, num_epochs=NUM_EPOCH, batch_size=BATCH_SIZE, rank=0, world_size=1, seed=0, verbose=True):
    """The same loop on a self-play record that is already on the device (self_play.play_batch_device): packed states
    uint8[M,32], policy targets f32[M,209], value targets f32[M]."""
    dev = model.flat_parameters().device
    packed, p, v = packed.to(dev), p.to(device=dev, dtype=torch.float32), v.to(device=dev, dtype=torch.float32)
    M = packed.shape[0]
    trainer = FlatTrainer(model, lr=0.001, rank=rank, world_size=world_size)
    gen = torch.Generator(device='cpu')
    gen.manual_seed(seed)                                              # same shuffle on every rank
    losses = []
    model.train()
    for epoch in range(num_epochs):
        perm = torch.randperm(M, generator=gen).to(dev)                # DataLoader(shuffle=True)
        ep = torch.zeros(2, device=dev)
        for start in range(0, M, batch_size):
            idx = perm[start:start + batch_size]
            lo, hi = shard_bounds(idx.numel(), rank, world_size)
            mine = idx[lo:hi]
            bp, bt, bv = trainer.inputs(mine.numel())   # gathered in place: the step's addresses repeat, so it replays as a CUDA graph
            if mine.numel():
                torch.index_select(packed, 0, mine, out=bp)
                torch.index_select(p, 0, mine, out=bt)
                torch.index_select(v, 0, mine, out=bv)
            ep += trainer.step(bp, bt, bv, idx.numel(), lr_lambda(epoch))
        if world_size > 1:
            import torch.distributed as dist
            dist.all_reduce(ep)
        losses.append(ep.tolist())
        if verbose and rank == 0:
            print(f"\rEpoch {epoch + 1}/{num_epochs} | Policy Loss: {losses[-1][0]:.4f} | Value Loss: {losses[-1][1]:.4f}", end='')
    if verbose and rank == 0:
        print('')
    trainer.check()
    return losses


def train_network(data_dir='./data', model_dir=None, num_epochs=NUM_EPOCH, rank=0, world_size=1):
    model_dir = PV_NETWORK_PATH if model_dir is None else model_dir
    # Load the model (train_network.py:28-30)
    model = GNNNetwork()
    model.load_state_dict(torch.load(os.path.join(model_dir, 'best.pth'), map_location='cuda'))
    model = model.to('cuda')
    history = load_data(data_dir)
    losses = train_on_history(model, history, num_epochs, BATCH_SIZE, rank, world_size)
    if rank == 0:
        torch.save(model.state_dict(), os.path.join(model_dir, 'latest.pth'))  # train_network.py:107
    return losses


if __name__ == '__main__':
    train_network()
