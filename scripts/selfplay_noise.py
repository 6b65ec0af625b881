"""Whole-game lock-step self-play with root Dirichlet noise off and on (play_batch_device(dirichlet_alpha=...)), each with tree reuse
off and on, at temperature 1 and 0.  One untimed run of each configuration (module loads, arenas, graph captures), then three timed
runs of each, alternating.  Per run: wall time, new simulations/s, aq_mcts_root_noise time per call (CUDA events around each call on
the search stream) and, for diversity, the number of distinct games (move sequences so far) and distinct positions among the games
still running at plies 10, 20 and 40.  The card's name and power limit are read in the same process.

    python scripts/selfplay_noise.py [games] [sims] [--alpha A] [--fraction F] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from alphaquoridorgnn_b200 import _lib, self_play
from alphaquoridorgnn_b200.pv_network_gnn import GNNNetwork

ap = argparse.ArgumentParser()
ap.add_argument("games", type=int, nargs="?", default=4096)
ap.add_argument("sims", type=int, nargs="?", default=200)
ap.add_argument("--alpha", type=float, default=0.3)
ap.add_argument("--fraction", type=float, default=0.25)
ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
cli = ap.parse_args()
games, sims, out_path = cli.games, cli.sims, cli.out
PLIES = (10, 20, 40)

if not torch.cuda.is_available():
    sys.exit("selfplay_noise.py measures on the GPU and needs one")
torch.manual_seed(0)
net = GNNNetwork().cuda().eval()
net.precision = "bf16"
L = _lib.load()

# instrumentation: CUDA events around every aq_mcts_root_noise (two per search)
noise_events = []
_orig_noise = L.aq_mcts_root_noise


def root_noise(*a):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    rc = _orig_noise(*a)
    e1.record()
    noise_events.append((e0, e1))
    return rc


L.aq_mcts_root_noise = root_noise


def diversity(rec):
    """{ply: [distinct games, distinct positions, games running]} over the games that reached the ply."""
    states = rec["states"].cpu().numpy()
    game, ply = rec["game"].cpu().numpy(), rec["ply"].cpu().numpy()
    order = np.lexsort((ply, game))
    states, game, ply = states[order], game[order], ply[order]
    out = {}
    for p in PLIES:
        at = np.nonzero(ply == p)[0]
        if not len(at):
            out[p] = [0, 0, 0]
            continue
        # a game's records are contiguous and in ply order: the ones up to ply p are rows at - p .. at
        seqs = {states[i - p:i + 1].tobytes() for i in at}
        out[p] = [len(seqs), len({states[i].tobytes() for i in at}), int(len(at))]
    return out


def run(alpha, reuse, temperature, seed):
    noise_events.clear()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    rec = self_play.play_batch_device(net, games, "cuda", sims=sims, temperature=temperature, seed=seed, policy_dtype=torch.float32,
                                      tree_reuse=reuse, dirichlet_alpha=alpha, noise_fraction=cli.fraction)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    noise_ms = [e0.elapsed_time(e1) for e0, e1 in noise_events]
    return {"dirichlet_alpha": alpha, "tree_reuse": reuse, "temperature": temperature, "seconds": round(dt, 4),
            "new_sims_per_s_M": round(rec["sims"] / dt / 1e6, 2), "plies": int(rec["ply"].max()) + 1, "searches": int(rec["game"].shape[0]),
            "noise_calls": len(noise_ms),
            "noise_us_per_call_mean": round(1e3 * sum(noise_ms) / len(noise_ms), 1) if noise_ms else None,
            "noise_us_per_call_max": round(1e3 * max(noise_ms), 1) if noise_ms else None,
            "noise_share_of_wall": round(sum(noise_ms) / 1e3 / dt, 5) if noise_ms else None,
            "distinct_games_positions_running": {str(p): v for p, v in diversity(rec).items()}}


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()
header = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None, "games": games, "sims": sims,
          "precision": "bf16", "dirichlet_alpha": cli.alpha, "noise_fraction": cli.fraction}
print(json.dumps(header), flush=True)
configs = [(alpha, reuse, temp) for temp in (1.0, 0.0) for reuse in (False, True) for alpha in (None, cli.alpha)]
for c in configs:
    run(*c, 1)
results = []
for rep in range(3):
    for c in configs:
        r = run(*c, 7 + rep)
        r["rep"] = rep
        results.append(r)
        print(json.dumps(r), flush=True)
if out_path:
    with open(out_path, "w") as f:
        f.write(json.dumps(header) + "\n" + "".join(json.dumps(r) + "\n" for r in results))
