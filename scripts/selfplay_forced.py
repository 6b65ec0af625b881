"""Whole-game lock-step self-play at temperature 1 with root Dirichlet noise only, noise plus forced playouts and policy target pruning,
and forced playouts alone (play_batch_device(dirichlet_alpha=..., forced_k=...)).  One untimed run of each configuration (module
loads, arenas, graph captures), then three timed runs of each, alternating.  Per run: wall time, new simulations/s, the time per call
of the counts read after each search (CUDA events around each aq_mcts_root_counts / aq_mcts_root_counts_pruned on the search stream),
the share of root-child visits the pruning removed, the mean entropy of the recorded policy rows and the mean number of children
with a non-zero target.  To count the removed visits, every search of every configuration also reads its raw counts
(aq_mcts_root_counts, one launch per ply, outside the per-call timing).  Last, the select step alone: aq_mcts_select and
aq_mcts_select_forced alternating on the trees of a finished 200-simulation search, CUDA events around each call.  The card's name,
power limit and max SM clock are read in the same process.

    python scripts/selfplay_forced.py [games] [sims] [--k K] [--alpha A] [--fraction F] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from alphaquoridorgnn_b200 import _lib, pv_mcts, self_play
from alphaquoridorgnn_b200 import game_logic as gl
from alphaquoridorgnn_b200.positions import random_positions
from alphaquoridorgnn_b200.pv_network_gnn import GNNNetwork

ap = argparse.ArgumentParser()
ap.add_argument("games", type=int, nargs="?", default=4096)
ap.add_argument("sims", type=int, nargs="?", default=200)
ap.add_argument("--k", type=float, default=2.0)
ap.add_argument("--alpha", type=float, default=0.3)
ap.add_argument("--fraction", type=float, default=0.25)
ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
cli = ap.parse_args()
games, sims, out_path = cli.games, cli.sims, cli.out

if not torch.cuda.is_available():
    sys.exit("selfplay_forced.py measures on the GPU and needs one")
torch.manual_seed(0)
net = GNNNetwork().cuda().eval()
net.precision = "bf16"
L = _lib.load()
P = _lib.ptr

# instrumentation: CUDA events around every counts read (one per search)
events = {"aq_mcts_root_counts": [], "aq_mcts_root_counts_pruned": []}
_orig = {name: getattr(L, name) for name in events}


def timed(name):
    def call(*a):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rc = _orig[name](*a)
        e1.record()
        events[name].append((e0, e1))
        return rc
    return call


for name in events:
    setattr(L, name, timed(name))

# the raw counts of every search, summed on the device next to the counts the search returned
visits = torch.zeros(2, dtype=torch.int64, device="cuda")   # [raw, returned]
_search_async = pv_mcts.BatchedMCTS.search_async


def search_async(self, *a, **kw):
    out = _search_async(self, *a, **kw)
    ws, G, G_real, max_nodes = self._root
    if G_real:
        raw = torch.empty((G, gl.MAX_LEGAL), dtype=torch.int32, device="cuda")
        act = torch.empty((G, gl.MAX_LEGAL), dtype=torch.int16, device="cuda")
        n = torch.empty((G,), dtype=torch.int16, device="cuda")
        _lib.check(_orig["aq_mcts_root_counts"](P(ws), G, max_nodes, P(raw), P(act), P(n), None, _lib.stream_ptr()), "raw counts")
        visits[0] += raw[:G_real].sum()
        visits[1] += out[0].sum()
    return out


pv_mcts.BatchedMCTS.search_async = search_async


def per_call_us(name):
    ms = [e0.elapsed_time(e1) for e0, e1 in events[name]]
    return (len(ms), round(1e3 * sum(ms) / len(ms), 2) if ms else None, round(1e3 * max(ms), 2) if ms else None)


def run(alpha, k, seed):
    for v in events.values():
        v.clear()
    visits.zero_()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    rec = self_play.play_batch_device(net, games, "cuda", sims=sims, temperature=1.0, seed=seed, policy_dtype=torch.float32,
                                      dirichlet_alpha=alpha, noise_fraction=cli.fraction, forced_k=k)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    pol = rec["policy"].double()
    entropy = -(torch.where(pol > 0, pol * torch.log(torch.where(pol > 0, pol, 1.0)), 0.0)).sum(1)
    raw, kept = visits.tolist()
    plain, pruned = per_call_us("aq_mcts_root_counts"), per_call_us("aq_mcts_root_counts_pruned")
    return {"dirichlet_alpha": alpha, "forced_k": k, "temperature": 1.0, "seconds": round(dt, 4),
            "new_sims_per_s_M": round(rec["sims"] / dt / 1e6, 2), "plies": int(rec["ply"].max()) + 1, "searches": int(rec["game"].shape[0]),
            "root_counts_calls": plain[0], "root_counts_us_per_call_mean": plain[1], "root_counts_us_per_call_max": plain[2],
            "root_counts_pruned_calls": pruned[0], "root_counts_pruned_us_per_call_mean": pruned[1],
            "root_counts_pruned_us_per_call_max": pruned[2], "root_visits": raw, "root_visits_pruned_share": round(1 - kept / raw, 5),
            "policy_entropy_mean": round(float(entropy.mean()), 4), "nonzero_targets_mean": round(float((pol > 0).sum(1).double().mean()), 3)}


def select_step():
    """aq_mcts_select vs aq_mcts_select_forced on the same trees (a finished forced search of `sims` simulations from mid-game roots):
    the select writes only the leaf it chose, so both can run over and over on one tree."""
    roots = random_positions(games, seed=5, games=64)
    mcts = pv_mcts.BatchedMCTS(net, sims, forced_k=cli.k)
    mcts.search(roots)
    ws, G, _, max_nodes = mcts._root
    leaf = torch.empty((G, gl.STATE_BYTES), dtype=torch.uint8, device="cuda")
    kind = torch.empty((G,), dtype=torch.int32, device="cuda")
    st = _lib.stream_ptr()
    calls = {"aq_mcts_select": lambda: L.aq_mcts_select(P(ws), G, max_nodes, pv_mcts.C_PUCT, P(leaf), P(kind), st),
             "aq_mcts_select_forced": lambda: L.aq_mcts_select_forced(P(ws), G, max_nodes, pv_mcts.C_PUCT, cli.k, P(leaf), P(kind), st)}
    for f in calls.values():
        for _ in range(20):
            _lib.check(f(), "select")
    ev = {name: [] for name in calls}
    for _ in range(200):
        for name, f in calls.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _lib.check(f(), name)
            e1.record()
            ev[name].append((e0, e1))
    torch.cuda.synchronize()
    out = {"select_step": True, "games": G, "root_visits": sims, "forced_k": cli.k}
    for name, es in ev.items():
        ms = sorted(e0.elapsed_time(e1) for e0, e1 in es)
        out[name + "_us_median"] = round(1e3 * ms[len(ms) // 2], 2)
        out[name + "_us_mean"] = round(1e3 * sum(ms) / len(ms), 2)
    return out


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()
header = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None, "games": games, "sims": sims,
          "precision": "bf16", "temperature": 1.0, "dirichlet_alpha": cli.alpha, "noise_fraction": cli.fraction, "forced_k": cli.k}
print(json.dumps(header), flush=True)
configs = [(cli.alpha, None), (cli.alpha, cli.k), (None, cli.k)]
for c in configs:
    run(*c, 1)
results = []
for rep in range(3):
    for c in configs:
        r = run(*c, 7 + rep)
        r["rep"] = rep
        results.append(r)
        print(json.dumps(r), flush=True)
results.append(select_step())
print(json.dumps(results[-1]), flush=True)
if out_path:
    with open(out_path, "w") as f:
        f.write(json.dumps(header) + "\n" + "".join(json.dumps(r) + "\n" for r in results))
