"""Evaluator-cache hit rate and the step kernel's time on the bench.py self-play workload.

Runs bench.py's self-play setup (seeded random-init net, or the shipped checkpoint for bt6, device Dirichlet noise, random
starts, sim cap 16) with the evaluator cache on or off and prints one JSON line per run:
  hit_rate      cache_hits / expansions: the share of leaf expansions served from the cache (no evaluator row)
  k_step_ms     az_step (cache insert + k_step) per round trip, CUDA events around each launch of an un-graphed pass
  nn_ms         the ResNet forward per round trip, measured the same way
  sims_per_s    simulations per second over graphed round trips (CUDA events)

usage: python scripts/eval_cache_stats.py [--config c4|bt6|bt8] [--log2 N ...] [--cycle-budget N ...] [--no-cache]
Every combination of --log2 and --cycle-budget is one run (0 = the default).
"""
import argparse
import itertools
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from alphazero_openspiel_b200 import _lib as L  # noqa: E402
from alphazero_openspiel_b200.engine import game_shape  # noqa: E402
from alphazero_openspiel_b200.examplegenerator import SelfPlayRunner  # noqa: E402
from alphazero_openspiel_b200.network import Net  # noqa: E402

CONFIGS = {
    "c4": ("connect_four", 800, 16384, None),
    "bt6": ("breakthrough(rows=6,columns=6)", 200, 1024, "tests/golden/example_model_breakthrough_6x6.pth"),
    "bt8": ("breakthrough", 800, 8192, None),
}


def run(game, playouts, trees, ckpt, cache, log2, budget, settle, timed, probe):
    shape, n_actions = game_shape(game)
    torch.manual_seed(0)
    net = Net(shape, n_actions)
    if ckpt:
        net.load_state_dict(torch.load(os.path.join(ROOT, ckpt), map_location="cpu", weights_only=True))
    net.eval()
    r = SelfPlayRunner(net, game, "cuda:0", trees, n_playouts=playouts, c_puct=2.5, use_dirichlet=True, seed=0xC4,
                       random_start_mod=21, max_sims_per_step=16, eval_cache=cache, eval_cache_log2=log2,
                       step_cycle_budget=budget or None)
    r.round(settle)
    torch.cuda.synchronize()
    c0 = r.counters()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    r.round(timed)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    c1 = r.counters()
    ev = r.evaluator
    steps = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(probe)]
    nns = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(probe)]
    with torch.no_grad():
        for a, b in zip(steps, nns):
            a[0].record()
            r.engine.step(ev.priors, ev.values, None, ev.obs, L.OBS_BF16_NHWC)
            a[1].record()
            r.engine.compact()
            b[0].record()
            ev()
            b[1].record()
    torch.cuda.synchronize()
    d = {k: c1[k] - c0[k] for k in c1}
    out = {"game": game, "trees": trees, "playouts": playouts, "eval_cache": bool(r.engine.flags & L.F_EVAL_CACHE),
           "eval_cache_log2": int(r.engine.eval_cache_log2), "step_cycle_budget": int(r.engine.cfg.step_cycle_budget),
           "hit_rate": d["cache_hits"] / max(1, d["expansions"]), "cache_hits": d["cache_hits"],
           "expansions": d["expansions"], "terminal": d["terminal"], "root_evals": d["root_evals"],
           "sims_per_eval_slot": d["sims"] / (trees * timed), "ms_per_round_trip": ms / timed,
           "sims_per_s": d["sims"] / (ms / 1e3), "overflow": d["overflow"],
           "k_step_ms": sum(a.elapsed_time(b) for a, b in steps) / probe,
           "nn_ms": sum(a.elapsed_time(b) for a, b in nns) / probe,
           "device_gb": r.engine.device_bytes / 1e9}
    r.close()
    del r, ev
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="c4", choices=sorted(CONFIGS))
    ap.add_argument("--log2", type=int, nargs="+", default=[0])
    ap.add_argument("--cycle-budget", type=int, nargs="+", default=[0])
    ap.add_argument("--no-cache", action="store_true")
    ap.add_argument("--settle", type=int, default=3000, help="untimed round trips first (fills the cache)")
    ap.add_argument("--rounds", type=int, default=1000, help="timed round trips")
    ap.add_argument("--probe", type=int, default=100, help="un-graphed round trips timed launch by launch")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("eval_cache_stats.py needs a CUDA device")
    game, playouts, trees, ckpt = CONFIGS[args.config]
    print(json.dumps({"device": torch.cuda.get_device_name(0)}), flush=True)
    for log2, budget in itertools.product(args.log2, args.cycle_budget):
        print(json.dumps(run(game, playouts, trees, ckpt, not args.no_cache, log2, budget, args.settle, args.rounds,
                             args.probe)), flush=True)


if __name__ == "__main__":
    main()
