"""Resignation in self-play: game length, throughput and calibration at several resign thresholds, with the shipped checkpoints.

Workloads (one JSON line per workload and threshold):
  c4     Connect Four, 16,384 trees, 800 simulations per move, tree reuse, auto-restart: a window of --rounds graphed evaluator
         round trips after --settle untimed ones (games of every length are in flight, as in a throughput run); plies per
         game are those of the games that finished in the window
  bt6    Breakthrough 6x6, one generation of 1,024 games (one game per tree), 200 simulations per move
  train  the Trainer-default generation: 500 Connect Four games in a pool of 500 trees, 100 simulations per move
Fields:
  plies_per_game       moves played per finished game (a resigned game counts the moves before its resignation)
  resign_threshold_suggested  resign_threshold_for(records, 0.05, threshold) over the finished games
  games_per_s, sims_per_s
  resign_share         resigned games / finished games
  false_positive_rate  calibration games: players who did not lose but whose minimum r was below the threshold, per
                       calibration game (resign_false / resign_samples)
  generation_s         bt6 / train: wall time of ExampleGenerator.generate_examples; c4: the timed window
Thresholds: off (resign_threshold=None) and the values of --thresholds; calibration share --disabled (default 0.1).

usage: python scripts/resign_selfplay.py [--workloads c4 bt6 train] [--thresholds -0.9 -0.8 -0.7]
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from alphazero_openspiel_b200.engine import game_shape  # noqa: E402
from alphazero_openspiel_b200.examplegenerator import ExampleGenerator, SelfPlayRunner, resign_threshold_for  # noqa: E402
from alphazero_openspiel_b200.network import Net  # noqa: E402

C4 = "connect_four"
BT6 = "breakthrough(rows=6,columns=6)"
CKPT = {C4: "tests/golden/example_model_connect_four.pth", BT6: "tests/golden/example_model_breakthrough_6x6.pth"}


def load_net(game):
    shape, n_actions = game_shape(game)
    net = Net(shape, n_actions)
    net.load_state_dict(torch.load(os.path.join(ROOT, CKPT[game]), map_location="cpu", weights_only=True))
    return net.eval()


def summary(d, seconds):
    games = max(1, d["games"])
    return {"games": d["games"], "plies_per_game": d["moves"] / games, "games_per_s": d["games"] / seconds,
            "sims_per_s": d["sims"] / seconds, "resign_share": d["resigns"] / games,
            "false_positive_rate": (d["resign_false"] / d["resign_samples"]) if d["resign_samples"] else None,
            "resigns": d["resigns"], "resign_samples": d["resign_samples"], "resign_false": d["resign_false"],
            "generation_s": seconds, "overflow": d["overflow"]}


def window(game, trees, playouts, thr, disabled, settle, rounds):
    r = SelfPlayRunner(load_net(game), game, "cuda:0", trees, n_playouts=playouts, seed=0xC4, resign_threshold=thr,
                       resign_disabled_fraction=disabled)
    r.round(settle)
    r.drain()
    torch.cuda.synchronize()
    c0 = r.counters()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    done, closes = 0, []
    while done < rounds:
        n = min(500, rounds - done)
        r.round(n)
        done += n
        if done < rounds:
            recs = r.drain()     # keeps the record buffer from filling (synchronises the stream)
            closes.append(recs[recs["kind"] == 1])
    e1.record()
    torch.cuda.synchronize()
    recs = r.drain()
    closes = np.concatenate(closes + [recs[recs["kind"] == 1]])
    c1 = r.counters()
    r.close()
    out = summary({k: c1[k] - c0[k] for k in c1}, e0.elapsed_time(e1) / 1e3)
    # games from the initial position: the closing record's ply is the number of moves played (resigned: before resigning)
    out["plies_per_game"] = float(closes["ply"].mean()) if len(closes) else None
    out["resign_threshold_suggested"] = None if thr is None else resign_threshold_for(closes, 0.05, thr)
    return out


def generation(game, n_games, playouts, thr, disabled):
    gen = ExampleGenerator(load_net(game), game, torch.device("cuda:0"), n_playouts=playouts, seed=7, resign_threshold=thr,
                           resign_disabled_fraction=disabled)
    torch.cuda.synchronize()
    t0 = time.time()
    gen.generate_examples(n_games)
    torch.cuda.synchronize()
    out = summary(gen.last_stats, time.time() - t0)
    out["resign_threshold_suggested"] = gen.last_stats.get("resign_threshold_suggested")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", nargs="+", default=["c4", "bt6", "train"], choices=["c4", "bt6", "train"])
    ap.add_argument("--thresholds", type=float, nargs="+", default=[-0.9, -0.8, -0.7])
    ap.add_argument("--disabled", type=float, default=0.1)
    ap.add_argument("--settle", type=int, default=40000, help="c4: untimed round trips first (longer than one game)")
    ap.add_argument("--rounds", type=int, default=20000, help="c4: timed round trips")
    ap.add_argument("--warm", action="store_true", help="one untimed generation of each generation workload first")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("resign_selfplay.py needs a CUDA device")
    print(json.dumps({"device": torch.cuda.get_device_name(0)}), flush=True)
    for w in args.workloads:
        if args.warm and w != "c4":
            generation(C4 if w == "train" else BT6, 64, 20, None, args.disabled)
        for thr in [None] + args.thresholds:
            if w == "c4":
                out = window(C4, 16384, 800, thr, args.disabled, args.settle, args.rounds)
            elif w == "bt6":
                out = generation(BT6, 1024, 200, thr, args.disabled)
            else:
                out = generation(C4, 500, 100, thr, args.disabled)
            print(json.dumps(dict(workload=w, threshold=thr, **out)), flush=True)


if __name__ == "__main__":
    main()
