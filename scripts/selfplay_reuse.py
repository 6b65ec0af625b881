"""Whole-game lock-step self-play with tree reuse off and on (play_batch_device(tree_reuse=...)), alternating, three timed runs
each after one untimed run of each (module loads, arenas, graph captures).  Per run: wall time, new simulations/s, mean root
visits per decision, share of searches that continued a carried tree, aq_mcts_advance time per ply (CUDA events around each
call on the search stream) and the bytes of the node arenas.  The card's name and power limit are read in the same process.

    python scripts/selfplay_reuse.py [games] [sims] [--out FILE]
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
from alphaquoridorgnn_b200.pv_network_gnn import GNNNetwork

ap = argparse.ArgumentParser()
ap.add_argument("games", type=int, nargs="?", default=4096)
ap.add_argument("sims", type=int, nargs="?", default=200)
ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
cli = ap.parse_args()
games, sims, out_path = cli.games, cli.sims, cli.out

if not torch.cuda.is_available():
    sys.exit("selfplay_reuse.py measures on the GPU and needs one")
torch.manual_seed(0)
net = GNNNetwork().cuda().eval()
net.precision = "bf16"
L = _lib.load()

# instrumentation: root visits of every search, and CUDA events around every aq_mcts_advance
visits, advance_events = [], []
_orig_search = pv_mcts.BatchedMCTS.search_async
_orig_advance = L.aq_mcts_advance


def search_async(self, roots, *a, **k):
    counts, actions, n, status = _orig_search(self, roots, *a, **k)
    visits.append(counts.sum(1, dtype=torch.int64) + 1)   # root n = 1 + sum of its children's visits
    return counts, actions, n, status


def advance(*a):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    rc = _orig_advance(*a)
    e1.record()
    advance_events.append((e0, e1))
    return rc


pv_mcts.BatchedMCTS.search_async = search_async
L.aq_mcts_advance = advance


def run(reuse, seed):
    visits.clear()
    advance_events.clear()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    rec = self_play.play_batch_device(net, games, "cuda", sims=sims, seed=seed, policy_dtype=torch.float32, tree_reuse=reuse)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    v = torch.cat(visits)
    searches = int(rec["game"].shape[0])
    adv_ms = [e0.elapsed_time(e1) for e0, e1 in advance_events]
    mcts = pv_mcts.searcher_for(net, sims, "cuda", tree_reuse=reuse)
    ws_bytes = sum(int(w.numel()) for w in mcts._ws if w is not None)
    return {"tree_reuse": reuse, "seconds": round(dt, 4), "new_sims_per_s_M": round(rec["sims"] / dt / 1e6, 2),
            "plies": len(visits), "searches": searches, "mean_root_visits": round(float(v.double().mean()), 2),
            "carried_share": round(rec["reused"] / searches, 4),
            "advance_us_per_ply_mean": round(1e3 * sum(adv_ms) / len(adv_ms), 1) if adv_ms else None,
            "advance_us_per_ply_max": round(1e3 * max(adv_ms), 1) if adv_ms else None,
            "workspace_bytes": ws_bytes}


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()
header = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None, "games": games, "sims": sims,
          "precision": "bf16"}
print(json.dumps(header), flush=True)
run(False, 1)
run(True, 1)
results = []
for rep in range(3):
    for reuse in (False, True):
        r = run(reuse, 7 + rep)
        r["rep"] = rep
        results.append(r)
        print(json.dumps(r), flush=True)
if out_path:
    with open(out_path, "w") as f:
        f.write(json.dumps(header) + "\n" + "".join(json.dumps(r) + "\n" for r in results))
