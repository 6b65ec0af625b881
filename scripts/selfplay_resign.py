"""What resignation costs and saves in whole-game lock-step self-play (play_batch_device(resign_threshold=...)), 4,096 games x 200
simulations, bf16.

An untrained network's values say nothing, so the script first trains one from a fixed seed with the repository's own loop:
`--cycles` cycles of 4,096-game self-play at `--train-sims` simulations (PUCT, temperature 1: with an untrained network these games
end decided often enough to give the value head a signal, where Gumbel games of such a network are nearly all draws), each
followed by `--epochs` epochs of train_on_buffer on its record.  It reports the value spread the
network reaches on the positions of a self-play record.  Then, one untimed run of each configuration first:
  1. cost when nothing resigns: resign_threshold=-2 against resignation off, alternating, three runs each: wall time and the time
     per call of aq_mcts_root_values (CUDA events around each call on the search stream);
  2. calibration: one run with resign_calibration=1.0, then v* = resign_threshold_for(rec, 0.05);
  3. resignation at v* with resign_calibration=0.1 against off, alternating, three runs each: wall time, searches run, positions
     recorded, games resigned and the false-positive rate seen among the calibration games (those whose non-losing sides' smallest
     statistic fell below v*).
The card's name and power limit are read in the same process.  The numbers hold for this network only.

    python scripts/selfplay_resign.py [games] [--cycles N] [--epochs E] [--train-sims S] [--out FILE]
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

from alphaquoridorgnn_b200 import _lib, self_play, train_network
from alphaquoridorgnn_b200.pv_network_gnn import GNNNetwork

ap = argparse.ArgumentParser()
ap.add_argument("games", type=int, nargs="?", default=4096)
ap.add_argument("--sims", type=int, default=200)
ap.add_argument("--cycles", type=int, default=4)
ap.add_argument("--epochs", type=int, default=1)
ap.add_argument("--train-sims", type=int, default=32)
ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
cli = ap.parse_args()
games, sims = cli.games, cli.sims

if not torch.cuda.is_available():
    sys.exit("selfplay_resign.py measures on the GPU and needs one")
L = _lib.load()
lines = []


def emit(d):
    lines.append(d)
    print(json.dumps(d), flush=True)


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()
emit({"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None, "games": games, "sims": sims, "precision": "bf16",
      "temperature": self_play.SP_TEMPERATURE, "train_cycles": cli.cycles, "train_epochs": cli.epochs, "train_sims": cli.train_sims})

# ---- a network with informative values: self-play + train_on_buffer, from a fixed seed
torch.manual_seed(0)
net = GNNNetwork().cuda().eval()
net.precision = "bf16"
t0 = time.perf_counter()
for cycle in range(cli.cycles):
    rec = self_play.play_batch_device(net, games, "cuda", sims=cli.train_sims, seed=100 + cycle, policy_dtype=torch.float32)
    losses = train_network.train_on_buffer(net, rec["states"], rec["policy"], rec["value"], num_epochs=cli.epochs, batch_size=256,
                                           seed=cycle, verbose=False)
    net.eval()
    emit({"train_cycle": cycle, "positions": int(rec["game"].shape[0]), "draws": int(((rec["flags"] & 2) != 0).sum()),
          "mean_game_plies": round(float(rec["plies"].double().mean()), 2), "last_loss": losses[-1] if losses else None})
train_s = time.perf_counter() - t0
with torch.no_grad():
    sample = rec["states"][torch.randperm(rec["states"].shape[0], generator=torch.Generator().manual_seed(0))[:8192].cuda()]
    v = net.predict_batch(sample)["value"].double().cpu().numpy()
q = np.quantile(v, [0.05, 0.25, 0.5, 0.75, 0.95])
emit({"value_spread": {"positions": int(v.size), "mean": round(float(v.mean()), 4), "std": round(float(v.std()), 4),
                       "mean_abs": round(float(np.abs(v).mean()), 4), "q05_25_50_75_95": [round(float(x), 4) for x in q],
                       "share_abs_above_0.5": round(float((np.abs(v) > 0.5).mean()), 4)}, "train_seconds": round(train_s, 1)})

# ---- instrumentation: CUDA events around every aq_mcts_root_values
events = []
orig = L.aq_mcts_root_values


def timed_root_values(*a):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    rc = orig(*a)
    e1.record()
    events.append((e0, e1))
    return rc


L.aq_mcts_root_values = timed_root_values


def run(threshold, calibration, seed):
    events.clear()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    rec = self_play.play_batch_device(net, games, "cuda", sims=sims, seed=seed, policy_dtype=torch.float32, resign_threshold=threshold,
                                      resign_calibration=calibration)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    flags = rec["flags"]
    r = {"threshold": threshold, "calibration": calibration if threshold is not None else None, "seed": seed, "seconds": round(dt, 4),
         "searches": int(rec["game"].shape[0]), "positions_recorded": int(rec["game"].shape[0]), "sims_run": rec["sims"],
         "plies": int(rec["ply"].max()) + 1, "mean_game_plies": round(float(rec["plies"].double().mean()), 2),
         "resigned": int(((flags & 4) != 0).sum()), "draws": int(((flags & 2) != 0).sum())}
    if events:
        ms = [e0.elapsed_time(e1) for e0, e1 in events]
        r["aq_mcts_root_values"] = {"calls": len(ms), "us_per_call_mean": round(1e3 * sum(ms) / len(ms), 1),
                                    "us_per_call_max": round(1e3 * max(ms), 1), "share_of_wall": round(sum(ms) / 1e3 / dt, 5)}
    return r, rec


def false_positives(rec, v):
    """Calibration games whose non-losing sides' smallest statistic fell below v (resigning at v would have lost them wrongly)."""
    cal = rec["calibration"].cpu().numpy()
    flags, plies, rmin = rec["flags"].cpu().numpy()[cal], rec["plies"].cpu().numpy()[cal], rec["resign_min"].cpu().numpy()[cal]
    m = np.where((flags & 1) != 0, rmin[np.arange(cal.sum()), 1 - plies % 2], rmin.min(axis=1))
    return int(cal.sum()), int((m < v).sum())


# 1. cost when nothing resigns
for c in ((None, 0.1), (-2.0, 0.0)):
    run(*c, 1)
for rep in range(3):
    for c in ((None, 0.1), (-2.0, 0.0)):
        r, _ = run(*c, 7 + rep)
        r.update(measurement="no_resign_cost", rep=rep)
        emit(r)

# 2. calibration: every game plays out
r, rec = run(-2.0, 1.0, 50)
v_star = self_play.resign_threshold_for(rec, 0.05)
C, fp = false_positives(rec, v_star)
r.update(measurement="calibration", v_star=v_star, calibration_games=C, would_be_false_positives=fp)
emit(r)

# 3. resignation at v*
run(v_star, 0.1, 2)
for rep in range(3):
    for c in ((None, 0.1), (v_star, 0.1)):
        r, rec = run(*c, 60 + rep)
        r.update(measurement="resign_at_v_star", rep=rep)
        if c[0] is not None:
            C, fp = false_positives(rec, v_star)
            r.update(calibration_games=C, false_positives=fp, false_positive_rate=round(fp / C, 4) if C else None)
        emit(r)
if cli.out:
    with open(cli.out, "w") as f:
        f.write("".join(json.dumps(d) + "\n" for d in lines))
