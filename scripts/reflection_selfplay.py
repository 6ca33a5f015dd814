"""Left-right reflection: self-play throughput with reflected evaluations (SelfPlayRunner(reflect_evaluations=True),
AZ_F_REFLECT) and the graphed training step with reflected minibatches (Trainer(reflect_minibatches=True)), each off / on,
alternated in one run.

Workloads (one JSON line per workload, setting and repetition):
  c4     Connect Four, 16,384 trees, 800 simulations per search, tree reuse, auto-restart, the shipped checkpoint: a window
         of --rounds graphed evaluator round trips after --settle untimed ones
  bt8    Breakthrough 8x8, 4,096 trees, 200 simulations per search, the same window; there is no shipped 8x8 checkpoint, so
         the network has seeded random weights (the evaluator's cost does not depend on them)
  train  Trainer(device_training=True, graph_step=True), Connect Four, batch 256: --steps graphed optimisation steps over a
         device replay buffer of 65,536 random-playout positions, after 20 untimed ones
Fields: sims_per_s (self-play), ms_per_step (train), seconds of the timed window (CUDA events / a host clock around work
that ends in a device synchronise), device and power_limit_w read in the same run.

usage: python scripts/reflection_selfplay.py [--workloads c4 bt8 train] [--settle N] [--rounds N] [--steps N] [--reps N]
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
from alphazero_openspiel_b200 import engine as E  # noqa: E402
from alphazero_openspiel_b200.examplegenerator import SelfPlayRunner  # noqa: E402
from alphazero_openspiel_b200.network import Net  # noqa: E402

C4 = "connect_four"
BT8 = "breakthrough"


def load_net(game):
    shape, n_actions = E.game_shape(game)
    torch.manual_seed(0)
    net = Net(shape, n_actions)
    if game == C4:
        ck = os.path.join(ROOT, "tests/golden/example_model_connect_four.pth")
        net.load_state_dict(torch.load(ck, map_location="cpu", weights_only=True))
    return net.eval()


def power_limit_w():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
        return float(out.splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        return None


def selfplay_window(game, trees, playouts, reflect, settle, rounds):
    r = SelfPlayRunner(load_net(game), game, "cuda:0", trees, n_playouts=playouts, seed=0xC4,
                       reflect_evaluations=reflect)
    r.round(settle)
    r.drain()
    torch.cuda.synchronize()
    c0 = r.counters()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    done = 0
    while done < rounds:
        n = min(500, rounds - done)
        r.round(n)
        done += n
        if done < rounds:
            r.drain()                    # keeps the record buffer from filling (synchronises the stream)
    e1.record()
    torch.cuda.synchronize()
    c1 = r.counters()
    r.close()
    seconds = e0.elapsed_time(e1) / 1e3
    return {"sims_per_s": (c1["sims"] - c0["sims"]) / seconds, "seconds": seconds, "overflow": c1["overflow"]}


def replay_buffer(n, seed=5):
    """A device replay buffer of n random-playout Connect Four positions (one per game, random lengths)."""
    from alphazero_openspiel_b200.device_replay import DeviceReplay
    from alphazero_openspiel_b200.replay import ExampleBatch
    hist, lens = E.game_random_playouts(C4, n, seed, 42)
    rng = np.random.RandomState(seed)
    lens = torch.from_numpy((rng.rand(n) * (lens.cpu().numpy() + 1)).astype(np.int32)).to(hist.device)
    bb = E.game_replay_dev(C4, hist, lens)["bb"].cpu().numpy().view(np.uint64)
    ln = lens.cpu().numpy()
    h = hist.cpu().numpy().astype(np.int16)
    h[np.arange(42)[None, :] >= ln[:, None]] = -1
    batch = ExampleBatch(C4, np.arange(n + 1), bb, ln, h, ln, rng.dirichlet(np.ones(7), n), rng.uniform(-1, 1, n))
    rb = DeviceReplay(C4, "cuda:0")
    rb.append(batch)
    return rb


def train_window(rb, reflect, steps):
    from alphazero_openspiel_b200.train import Trainer
    torch.manual_seed(0)
    np.random.seed(0)
    tr = Trainer(device="cuda:0", batch_size=256, device_training=True, graph_step=True, reflect_minibatches=reflect,
                 save=False)
    tr.current_net.train()
    first, pol, val = rb.remove_duplicates()
    for _ in range(20):
        tr.net_step_device(rb, first, pol, val)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        lp, _ = tr.net_step_device(rb, first, pol, val)
    torch.cuda.synchronize()
    seconds = time.perf_counter() - t0
    return {"ms_per_step": seconds / steps * 1e3, "seconds": seconds, "loss_p": float(lp)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", nargs="+", default=["c4", "bt8", "train"], choices=["c4", "bt8", "train"])
    ap.add_argument("--settle", type=int, default=2000, help="self-play: untimed round trips first")
    ap.add_argument("--rounds", type=int, default=3000, help="self-play: timed round trips")
    ap.add_argument("--steps", type=int, default=2000, help="train: timed optimisation steps")
    ap.add_argument("--reps", type=int, default=2, help="off / on pairs per workload")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("reflection_selfplay.py needs a CUDA device")
    dev = torch.cuda.get_device_name(0)
    print(json.dumps({"device": dev, "power_limit_w": power_limit_w()}), flush=True)
    rb = replay_buffer(65536) if "train" in args.workloads else None
    for w in args.workloads:
        for rep in range(args.reps):
            for reflect in (False, True):
                if w == "train":
                    out = train_window(rb, reflect, args.steps)
                    extra = {"steps": args.steps, "batch_size": 256}
                else:
                    game, trees, playouts = {"c4": (C4, 16384, 800), "bt8": (BT8, 4096, 200)}[w]
                    out = selfplay_window(game, trees, playouts, reflect, args.settle, args.rounds)
                    extra = {"trees": trees, "playouts": playouts, "settle": args.settle, "rounds": args.rounds}
                print(json.dumps(dict(workload=w, reflect=reflect, rep=rep, device=dev, power_limit_w=power_limit_w(),
                                      **extra, **out)), flush=True)


if __name__ == "__main__":
    main()
