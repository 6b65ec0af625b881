"""Whole-game lock-step self-play at temperature 1 with root noise and forced playouts, without and with playout cap randomization
(play_batch_device(fast_sims=..., full_search_prob=...)).  One untimed run of each arm (module loads, arenas, graph captures), then
three timed runs of each, alternating.  Per run: wall time, games/s, full and fast searches, recorded positions, new simulations/s,
and the number and host time of the CUDA-graph captures the run made.  The simulation phases are timed with CUDA events around each
BatchedMCTS._simulate call that captured nothing: phase A (every row, the searcher's step mode) and phase B (the full-row prefix,
"-rows" mode), per simulation step, by batch size; the first ply's searches run at the full 4,096 rows.  The card's name and power
limit are read in the same process.

    python scripts/selfplay_pcr.py [games] [sims] [--fast F] [--p P] [--k K] [--alpha A] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time
from collections import defaultdict

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from alphaquoridorgnn_b200 import _lib, pv_mcts, self_play
from alphaquoridorgnn_b200.pv_network_gnn import GNNNetwork

ap = argparse.ArgumentParser()
ap.add_argument("games", type=int, nargs="?", default=4096)
ap.add_argument("sims", type=int, nargs="?", default=200)
ap.add_argument("--fast", type=int, default=50)
ap.add_argument("--p", type=float, default=0.25)
ap.add_argument("--k", type=float, default=2.0)
ap.add_argument("--alpha", type=float, default=0.3)
ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
cli = ap.parse_args()
games, sims = cli.games, cli.sims

if not torch.cuda.is_available():
    sys.exit("selfplay_pcr.py measures on the GPU and needs one")
torch.manual_seed(0)
net = GNNNetwork().cuda().eval()
net.precision = "bf16"

# instrumentation: graph captures (count, host time) and CUDA events around every simulation phase that captured nothing
captures = []
_capture = _lib.capture_graph


def capture_graph(*a, **kw):
    t0 = time.perf_counter()
    g = _capture(*a, **kw)
    captures.append(time.perf_counter() - t0)
    return g


_lib.capture_graph = capture_graph
phases = []   # (phase, batch rows, phase rows, simulations, start event, end event)
_simulate = pv_mcts.BatchedMCTS._simulate


def simulate(self, n, step, key, st):
    if key is None or n == 0:
        return _simulate(self, n, step, key, st)
    c0, warm = len(captures), key[-1] in self._warm
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = _simulate(self, n, step, key, st)
    e1.record()
    if len(captures) == c0 and warm:
        b = key[-1].endswith("-rows")
        phases.append(("B" if b else "A", key[0], key[-2] if b else key[0], n, e0, e1))
    return out


pv_mcts.BatchedMCTS._simulate = simulate


def run(fast, seed):
    captures.clear()
    phases.clear()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    rec = self_play.play_batch_device(net, games, "cuda", sims=sims, temperature=1.0, seed=seed, policy_dtype=torch.float32,
                                      dirichlet_alpha=cli.alpha, forced_k=cli.k, fast_sims=fast, full_search_prob=cli.p)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    steps = defaultdict(lambda: [0, 0.0])
    for ph, G, rows, n, e0, e1 in phases:
        s = steps[(ph, G, rows)]
        s[0] += n
        s[1] += e0.elapsed_time(e1)
    at_full = {f"{ph}_{rows}_rows": round(1e3 * ms / n, 2) for (ph, G, rows), (n, ms) in sorted(steps.items()) if G == games}
    return {"fast_sims": fast, "full_search_prob": cli.p if fast else None, "seconds": round(dt, 4), "games_per_s": round(games / dt, 1),
            "full_searches": rec["full_searches"], "fast_searches": rec["fast_searches"], "recorded_positions": int(rec["states"].shape[0]),
            "new_sims": rec["sims"], "new_sims_per_s_M": round(rec["sims"] / dt / 1e6, 2), "plies": int(rec["plies"].max()),
            "graph_captures": len(captures), "graph_capture_s": round(sum(captures), 3),
            "step_us_at_first_batch": at_full}


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()
header = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None, "games": games, "sims": sims,
          "precision": "bf16", "temperature": 1.0, "dirichlet_alpha": cli.alpha, "forced_k": cli.k, "fast_sims": cli.fast,
          "full_search_prob": cli.p}
print(json.dumps(header), flush=True)
arms = [None, cli.fast]
for fast in arms:
    r = run(fast, 1)
    r["warmup"] = True
    print(json.dumps(r), flush=True)
results = []
for rep in range(3):
    for fast in arms:
        r = run(fast, 7 + rep)
        r["rep"] = rep
        results.append(r)
        print(json.dumps(r), flush=True)
if cli.out:
    with open(cli.out, "w") as f:
        f.write(json.dumps(header) + "\n" + "".join(json.dumps(r) + "\n" for r in results))
