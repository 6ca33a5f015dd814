"""Forced playouts and policy target pruning in self-play: throughput and policy-target statistics, with the shipped
checkpoints.

Workloads (one JSON line per workload and setting):
  c4     Connect Four, 16,384 trees, 800 simulations per full search, tree reuse, auto-restart: a window of --rounds graphed
         evaluator round trips after --settle untimed ones (games of every length are in flight, as in a throughput run)
  bt6    Breakthrough 6x6, one generation of 1,024 games (one game per tree), 200 simulations per full search
Settings: off (forced_playouts=None); k = 2; k = 2 with playout cap randomization (fast_playouts = N/8, 25 % full searches).
Fields:
  sims_per_s, games_per_s
  examples_per_s       full-search ply records (the training examples) per second
  target_nonzero       mean number of non-zero policy-target entries per example
  target_entropy       mean entropy (nats) of the policy targets counts / sum(counts)
  pruned_visits        mean root_n - sum(counts) per example: the visits pruned from the target (within one of the true
                       figure, because a reused root carries one visit of its own)
  seconds              c4: the timed window; bt6: wall time of ExampleGenerator.generate_examples
  device, power_limit_w  the GPU and its power limit, read in the same run

usage: python scripts/forced_playouts_selfplay.py [--workloads c4 bt6] [--settle N] [--rounds N]
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


class TargetStats:
    """Policy-target statistics of the full-search ply records (the training examples)."""

    def __init__(self):
        self.n = 0
        self.nonzero = 0
        self.entropy = 0.0
        self.pruned = 0

    def add(self, recs):
        ex = recs[(recs["kind"] == 0) & (recs["end"] != 3)]
        if len(ex) == 0:
            return
        counts = ex["counts"].astype(np.float64)
        total = counts.sum(axis=1)
        ok = total > 0
        p = counts[ok] / total[ok][:, None]
        with np.errstate(divide="ignore", invalid="ignore"):
            h = -np.where(p > 0, p * np.log(p), 0.0).sum(axis=1)
        self.n += int(ok.sum())
        self.nonzero += int((counts[ok] > 0).sum())
        self.entropy += float(h.sum())
        self.pruned += int((ex["root_n"][ok].astype(np.int64) - total[ok].astype(np.int64)).sum())

    def fields(self, seconds):
        n = max(1, self.n)
        return {"examples_per_s": self.n / seconds, "target_nonzero": self.nonzero / n, "target_entropy": self.entropy / n,
                "pruned_visits": self.pruned / n}


def summary(d, stats, seconds):
    return dict({"games": d["games"], "games_per_s": d["games"] / seconds, "sims_per_s": d["sims"] / seconds,
                 "seconds": seconds, "overflow": d["overflow"]}, **stats.fields(seconds))


def window(game, trees, playouts, k, fast, settle, rounds):
    r = SelfPlayRunner(load_net(game), game, "cuda:0", trees, n_playouts=playouts, seed=0xC4, forced_playouts=k,
                       fast_playouts=fast, full_search_fraction=0.25)
    r.round(settle)
    r.drain()
    torch.cuda.synchronize()
    c0 = r.counters()
    stats = TargetStats()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    done, chunks = 0, []
    while done < rounds:
        n = min(500, rounds - done)
        r.round(n)
        done += n
        if done < rounds:
            chunks.append(r.drain())     # keeps the record buffer from filling (synchronises the stream)
    e1.record()
    torch.cuda.synchronize()
    chunks.append(r.drain())
    c1 = r.counters()
    r.close()
    for c in chunks:
        stats.add(c)
    return summary({k: c1[k] - c0[k] for k in c1}, stats, e0.elapsed_time(e1) / 1e3)


def generation(game, n_games, playouts, k, fast):
    gen = ExampleGenerator(load_net(game), game, torch.device("cuda:0"), n_trees=n_games, n_playouts=playouts, seed=7,
                           forced_playouts=k, fast_playouts=fast, full_search_fraction=0.25)
    torch.cuda.synchronize()
    t0 = time.time()
    recs, s = gen._play(n_games)
    torch.cuda.synchronize()
    seconds = time.time() - t0
    stats = TargetStats()
    stats.add(recs)
    return summary(s, stats, seconds)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", nargs="+", default=["c4", "bt6"], choices=["c4", "bt6"])
    ap.add_argument("--settle", type=int, default=40000, help="c4: untimed round trips first (longer than one game)")
    ap.add_argument("--rounds", type=int, default=20000, help="c4: timed round trips")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("forced_playouts_selfplay.py needs a CUDA device")
    print(json.dumps({"device": torch.cuda.get_device_name(0), "power_limit_w": power_limit_w()}), flush=True)
    for w in args.workloads:
        game, playouts = {"c4": (C4, 800), "bt6": (BT6, 200)}[w]
        for k, fast in ((None, None), (2.0, None), (2.0, playouts // 8)):
            if w == "c4":
                out = window(game, 16384, playouts, k, fast, args.settle, args.rounds)
            else:
                out = generation(game, 1024, playouts, k, fast)
            print(json.dumps(dict(workload=w, forced_playouts=k, fast_playouts=fast,
                                  full_search_fraction=None if fast is None else 0.25, settle=args.settle if w == "c4" else None,
                                  rounds=args.rounds if w == "c4" else None, device=torch.cuda.get_device_name(0),
                                  power_limit_w=power_limit_w(), **out)), flush=True)


if __name__ == "__main__":
    main()
