"""Playout cap randomization in self-play: games, training examples and simulations per second, with the shipped checkpoints.

Workloads (one JSON line per workload and setting):
  c4     Connect Four, 16,384 trees, 800 simulations per full search, tree reuse, auto-restart: a window of --rounds graphed
         evaluator round trips after --settle untimed ones (games of every length are in flight, as in a throughput run)
  bt6    Breakthrough 6x6, one generation of 1,024 games (one game per tree), 200 simulations per full search
  train  the Trainer-default generation: 500 Connect Four games in a pool of 500 trees, 100 simulations per full search
Settings: off (fast_playouts=None), then full_search_fraction --fraction (default 0.25) with fast_playouts = N/8 and N/4.
Fields:
  games_per_s          finished games per second
  examples_per_s       full-search ply records (the training examples) per second
  sims_per_s
  plies_per_game       moves played per finished game
  fast_share           fast searches / searched positions
  seconds              c4: the timed window; bt6 / train: wall time of ExampleGenerator.generate_examples
  device, power_limit_w  the GPU and its power limit, read in the same run

usage: python scripts/playout_cap_selfplay.py [--workloads c4 bt6 train] [--fraction 0.25]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from alphazero_openspiel_b200.engine import game_shape  # noqa: E402
from alphazero_openspiel_b200.examplegenerator import ExampleGenerator, SelfPlayRunner  # noqa: E402
from alphazero_openspiel_b200.network import Net  # noqa: E402

C4 = "connect_four"
BT6 = "breakthrough(rows=6,columns=6)"
CKPT = {C4: "tests/golden/example_model_connect_four.pth", BT6: "tests/golden/example_model_breakthrough_6x6.pth"}


def load_net(game):
    shape, n_actions = game_shape(game)
    net = Net(shape, n_actions)
    net.load_state_dict(torch.load(os.path.join(ROOT, CKPT[game]), map_location="cpu", weights_only=True))
    return net.eval()


def power_limit_w():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
        return float(out.splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        return None


def summary(d, n_searched, n_fast, seconds):
    games = max(1, d["games"])
    return {"games": d["games"], "games_per_s": d["games"] / seconds, "examples_per_s": (n_searched - n_fast) / seconds,
            "sims_per_s": d["sims"] / seconds, "plies_per_game": d["moves"] / games,
            "fast_share": n_fast / max(1, n_searched), "seconds": seconds, "overflow": d["overflow"]}


def window(game, trees, playouts, fast, fraction, settle, rounds):
    r = SelfPlayRunner(load_net(game), game, "cuda:0", trees, n_playouts=playouts, seed=0xC4, fast_playouts=fast,
                       full_search_fraction=fraction)
    r.round(settle)
    r.drain()
    torch.cuda.synchronize()
    c0 = r.counters()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    done, searched, n_fast = 0, 0, 0
    while done < rounds:
        n = min(500, rounds - done)
        r.round(n)
        done += n
        if done < rounds:
            recs = r.drain()     # keeps the record buffer from filling (synchronises the stream)
            searched += int((recs["kind"] == 0).sum())
            n_fast += int(((recs["kind"] == 0) & (recs["end"] == 3)).sum())
    e1.record()
    torch.cuda.synchronize()
    recs = r.drain()
    searched += int((recs["kind"] == 0).sum())
    n_fast += int(((recs["kind"] == 0) & (recs["end"] == 3)).sum())
    c1 = r.counters()
    r.close()
    return summary({k: c1[k] - c0[k] for k in c1}, searched, n_fast, e0.elapsed_time(e1) / 1e3)


def generation(game, n_games, playouts, fast, fraction):
    gen = ExampleGenerator(load_net(game), game, torch.device("cuda:0"), n_playouts=playouts, seed=7, fast_playouts=fast,
                           full_search_fraction=fraction)
    torch.cuda.synchronize()
    t0 = time.time()
    gen.generate_examples(n_games)
    torch.cuda.synchronize()
    s = gen.last_stats
    return summary(s, s["moves"] + s["resigns"], s["fast_searches"], time.time() - t0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", nargs="+", default=["c4", "bt6", "train"], choices=["c4", "bt6", "train"])
    ap.add_argument("--fraction", type=float, default=0.25, help="full_search_fraction of the playout-cap settings")
    ap.add_argument("--settle", type=int, default=40000, help="c4: untimed round trips first (longer than one game)")
    ap.add_argument("--rounds", type=int, default=20000, help="c4: timed round trips")
    ap.add_argument("--warm", action="store_true", help="one untimed generation of each generation workload first")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("playout_cap_selfplay.py needs a CUDA device")
    print(json.dumps({"device": torch.cuda.get_device_name(0), "power_limit_w": power_limit_w()}), flush=True)
    for w in args.workloads:
        game, playouts = {"c4": (C4, 800), "bt6": (BT6, 200), "train": (C4, 100)}[w]
        if args.warm and w != "c4":
            generation(game, 64, 20, None, args.fraction)
        for fast in (None, playouts // 8, playouts // 4):
            if w == "c4":
                out = window(game, 16384, playouts, fast, args.fraction, args.settle, args.rounds)
            else:
                out = generation(game, 1024 if w == "bt6" else 500, playouts, fast, args.fraction)
            print(json.dumps(dict(workload=w, fast_playouts=fast, full_search_fraction=None if fast is None else args.fraction,
                                  device=torch.cuda.get_device_name(0), power_limit_w=power_limit_w(), **out)), flush=True)


if __name__ == "__main__":
    main()
