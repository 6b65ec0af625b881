"""Whole-game lock-step self-play with the PUCT root at 200 simulations against the Gumbel root (play_batch_device(
gumbel_considered=...)) at 16, 32, 64 and 200 simulations, bf16.  One untimed run of each configuration (module loads, arenas,
graph captures), then three timed runs of each, alternating.  Per run: wall time, positions (searches) per second, new simulations
per second, and the time per call of aq_mcts_gumbel_root / aq_mcts_gumbel_result (CUDA events around each call on the search
stream).  The card's name and power limit are read in the same process.

    python scripts/selfplay_gumbel.py [games] [--considered M] [--scale S] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from alphaquoridorgnn_b200 import _lib, self_play
from alphaquoridorgnn_b200.pv_network_gnn import GNNNetwork

ap = argparse.ArgumentParser()
ap.add_argument("games", type=int, nargs="?", default=4096)
ap.add_argument("--considered", type=int, default=16)
ap.add_argument("--scale", type=float, default=1.0)
ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
cli = ap.parse_args()
games, out_path = cli.games, cli.out

if not torch.cuda.is_available():
    sys.exit("selfplay_gumbel.py measures on the GPU and needs one")
torch.manual_seed(0)
net = GNNNetwork().cuda().eval()
net.precision = "bf16"
L = _lib.load()

# instrumentation: CUDA events around every aq_mcts_gumbel_root and aq_mcts_gumbel_result (one of each per search)
events = {"aq_mcts_gumbel_root": [], "aq_mcts_gumbel_result": []}


def timed(name):
    orig = getattr(L, name)

    def call(*a):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rc = orig(*a)
        e1.record()
        events[name].append((e0, e1))
        return rc
    setattr(L, name, call)


for name in events:
    timed(name)


def run(considered, sims, seed):
    for v in events.values():
        v.clear()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    rec = self_play.play_batch_device(net, games, "cuda", sims=sims, seed=seed, policy_dtype=torch.float32, gumbel_considered=considered,
                                      gumbel_scale=cli.scale)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    r = {"root": "puct" if considered is None else "gumbel", "considered": considered, "sims": sims, "seconds": round(dt, 4),
         "positions": int(rec["game"].shape[0]), "positions_per_s": round(rec["game"].shape[0] / dt, 1),
         "new_sims_per_s_M": round(rec["sims"] / dt / 1e6, 2), "plies": int(rec["ply"].max()) + 1,
         "mean_game_plies": round(float(rec["plies"].double().mean()), 2),
         "draws": int(((rec["flags"] & 2) != 0).sum())}
    for name, ev in events.items():
        ms = [e0.elapsed_time(e1) for e0, e1 in ev]
        r[name] = {"calls": len(ms), "us_per_call_mean": round(1e3 * sum(ms) / len(ms), 1), "us_per_call_max": round(1e3 * max(ms), 1),
                   "share_of_wall": round(sum(ms) / 1e3 / dt, 5)} if ms else None
    return r


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()
header = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None, "games": games, "precision": "bf16",
          "gumbel_considered": cli.considered, "gumbel_scale": cli.scale, "temperature_puct": self_play.SP_TEMPERATURE}
print(json.dumps(header), flush=True)
configs = [(None, 200)] + [(cli.considered, s) for s in (16, 32, 64, 200)]
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
