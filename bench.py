#!/usr/bin/env python
"""bench.py -- self-play MCTS throughput of the B200 engine (BASELINE.json metric: MCTS simulations/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # our arm
    python bench.py ... --dump-outputs DIR                         # + training records of a tree sample as DIR/*.npy
    python bench.py --impl reference [--steps K] [--warmup W]      # CPU arm: the oracle port of the reference
    torchrun ... bench.py --gpus N ...                             # one rank per GPU, NCCL

Default workload (BASELINE.json configs[2], `--config c4`): Connect Four, 800 sims/move, 16,384 concurrent trees per GPU,
Dirichlet root noise, tree reuse, synthetic start positions (k = counter % 21 random plies), random-init ResNet of the
reference architecture in bf16.  `--config bt6 | bt8 | train` select BASELINE configs [1], [3], [4].

One evaluator ROUND TRIP for every tree = az_step (consume + PUCT simulations + move bookkeeping + observation encode)
followed by the batched ResNet forward, one CUDA-graph replay.  One bench "step" = ROUNDS_PER_STEP (50) round trips, so
that the driver's `--steps 20` times 1,000 round trips (~0.7 s), not 14 ms.  Before the warm-up an untimed SETTLE phase
runs the pool into steady state whatever --warmup says (at least 1,500 round trips and until every tree has moved twice
on average and games are finishing): the first searches of a fresh pool run in lock step and are ~40 % faster than the
steady state (VERDICT r01).  Weak scaling: every GPU runs its own independent pool; there is no data-path collective.

One JSON line on stdout (rank 0).  `value` = simulations completed in the timed region (device counters,
summed over ranks) / max-over-ranks CUDA-event time.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ROUNDS_PER_STEP = 50
SETTLE_MIN_ROUNDS, SETTLE_MAX_ROUNDS = 1500, 12000
DUMP_TREES = 4096
# BASELINE.json configs by index; trees = concurrent games per GPU
CONFIGS = {
    "c4": {"index": 2, "game": "connect_four", "playouts": 800, "trees": 16384},
    "bt6": {"index": 1, "game": "breakthrough(rows=6,columns=6)", "playouts": 200, "trees": 1024,
            "checkpoint": os.path.join("tests", "golden", "example_model_breakthrough_6x6.pth")},
    "bt8": {"index": 3, "game": "breakthrough", "playouts": 800, "trees": 8192},
    "train": {"index": 4, "game": "connect_four", "playouts": 100, "trees": 0},
}


_REAL_STDOUT = None


def emit(line):
    """The one JSON line of this run, on the process's original stdout."""
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def conv_dram_traffic(game, trees):
    """dram__bytes_read.sum + dram__bytes_write.sum per conv launch (averaged over the conv launches of one evaluation)
    from the committed `ncu --set full` capture of this shape: profiles/conv_traffic.json is written by
    scripts/summarize_ncu_traffic.py from the raw csv.  None when no capture of this (game, trees) exists."""
    path = os.path.join(ROOT, "profiles", "conv_traffic.json")
    try:
        with open(path) as f:
            return json.load(f).get("%s/%d" % (game, trees), {}).get("bytes_per_launch")
    except Exception:
        return None

FLOPS_PER_EVAL = {"connect_four": 17211600, "breakthrough(rows=6,columns=6)": 16282800, "breakthrough": 31097600}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.rows = []
        self.proc = None
        self.n0 = 0

    def mark(self):
        self.n0 = len(self.rows)

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows, where = self.rows[self.n0:], "timed region"
        if not rows:
            rows, where = self.rows[-5:], "end of warm-up (timed region shorter than the sampling latency)"
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, val in zip(names, f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "sampled_during": where}


def algorithmic_bytes(d, game_cells, num_actions):
    """SURVEY 8(d) bytes/simulation summed over the region, from the engine's counters (delta dict)."""
    state_bytes = 16
    return (8 * d["depth"] + 20 * d["children"]                       # select: per level 8 B node + 20 B per child
            + 24 * (d["depth"] + d["sims"])                           # backup: N,Q read+write along the path
            + d["expansions"] * (8 + 4 * (num_actions + 1) + 2 * 4 * game_cells)  # link + fp32 NN out + bf16 NN in
            + 20 * d["legal"]                                         # child records written at expansion
            + state_bytes * d["sims"])                                # root position read


def cpu_baseline(game, n_playouts, seconds_budget=20.0, max_plies=None):
    """The oracle's Python port of the reference's multi-process self-play (examplegenerator.py) on host cores."""
    import torch
    from oracle import ref_port, ref_net, pyspiel_shim
    torch.manual_seed(0)
    g = pyspiel_shim.load_game(game)
    net = ref_net.RefNet(g.information_state_normalized_vector_shape(), g.num_distinct_actions())
    net.eval()
    cores = os.cpu_count() or 2
    workers = max(1, min(cores - 1, 32))
    # bounded sample: every worker plays the first `max_plies` plies of one game
    if max_plies is None:
        per_ply = n_playouts / 450.0  # ~450 sims/s/process for the Python path (BASELINE.md section 3)
        max_plies = max(1, int(seconds_budget / max(per_ply, 1e-3)))
        max_plies = min(max_plies, 12)
    res = ref_port.time_selfplay(net, game, workers, workers, n_playouts=n_playouts, c_puct=2.5,
                                 dirichlet_ratio=0.25, temperature=1.0, backup="on-policy", max_plies=max_plies)
    sample = ("%d games x first %d plies, %d sims/move, %d worker processes + 1 evaluator process (fp32 CPU ResNet), "
              "%d sims in %.1f s" % (res["n_games"], max_plies, n_playouts, workers, res["sims"], res["seconds"]))
    # BASELINE config 1 shape: one process, in-process Net.predict, 100 sims/move (first 8 plies, bounded)
    torch.set_num_threads(1)
    np_state = None
    try:
        import numpy as np
        np_state = np.random.get_state()
        np.random.seed(0)
        t0 = time.time()
        st = {}
        ref_port.selfplay_game(net.predict, game, pyspiel_shim.load_game, stats=st, n_playouts=100, c_puct=2.5,
                               dirichlet_ratio=0.25, temperature=1.0, backup="on-policy", max_plies=8)
        single = st.get("sims", 0) / max(time.time() - t0, 1e-9)
    finally:
        if np_state is not None:
            np.random.set_state(np_state)
    return {"value": res["sims_per_s"], "unit": "sims/s", "cores": workers + 1, "kind": "port", "sample": sample,
            "host_cpus": cores, "games_per_s_equiv": res["sims_per_s"] / (n_playouts * 25.0),
            "single_process_100sims_sims_per_s": single}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    game = args.game
    vals = []
    base = None
    for _ in range(max(1, min(args.steps, 3)) if args.ref_repeat else 1):
        base = cpu_baseline(game, args.playouts, seconds_budget=args.cpu_seconds)
        vals.append(base["value"])
    v = sum(vals) / len(vals)
    base["value"] = v
    line = {"metric": "mcts_simulations_per_sec", "value": v, "unit": "sims/s", "impl": "reference",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * float(base["sample"].split(" sims in ")[1].split(" s")[0]) / max(args.steps, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": {"workload": workload_name(args), "trees_per_gpu": args.trees,
                                            "n_playouts": args.playouts, "game": game},
            "cpu_baseline": base,
            "e2e": {"value": v, "unit": "sims/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def workload_name(args):
    return "BASELINE configs[%d]: %s batched self-play, %d sims/move, %d concurrent trees per GPU" % (
        CONFIGS[args.config]["index"], args.game, args.playouts, args.trees)


def build_net(args, shape, n_actions):
    """Random-init weights of the reference architecture (no checkpoints off-box), except where BASELINE names a shipped
    model that travels as a test fixture (config [1]: tests/golden/example_model_breakthrough_6x6.pth)."""
    import torch
    from alphazero_openspiel_b200.network import Net
    torch.manual_seed(0)
    net = Net(shape, n_actions)
    weights = "random-init weights"
    ck = CONFIGS[args.config].get("checkpoint")
    if ck and args.game == CONFIGS[args.config]["game"] and os.path.exists(os.path.join(ROOT, ck)):
        net.load_state_dict(torch.load(os.path.join(ROOT, ck), map_location="cpu", weights_only=True))
        weights = "shipped checkpoint " + os.path.basename(ck)
    net.eval()
    return net, weights


def settle(runner, n_trees, dev, drain):
    """Untimed: run the pool into steady state (see the module docstring).  Returns the round trips spent."""
    import torch
    rounds = 0
    while True:
        runner.round(250)
        rounds += 250
        if rounds % 1000 == 0:
            drain()
        c = runner.counters()
        torch.cuda.synchronize(dev)
        if rounds >= SETTLE_MIN_ROUNDS and c["moves"] >= 2 * n_trees and c["games"] > 0:
            break
        if rounds >= SETTLE_MAX_ROUNDS:
            break
    drain()
    return rounds


def dump_move(args):
    """--dump-outputs writes each sample tree's search number dump_move(args) (1-based): a lower bound on the searches every
    tree has finished when the last timed step ends.  A search of n playouts takes at most n + 3 round trips (one evaluation
    per playout, the root evaluation, the move and the re-rooting), and by then the run has made at least the settle
    minimum plus the warm-up and timed steps' round trips."""
    rounds = (0 if args.no_settle else SETTLE_MIN_ROUNDS) + (args.warmup + args.steps) * ROUNDS_PER_STEP
    return rounds // (args.playouts + 3)


def dump_trees(n_trees):
    """The fixed, seeded sample of trees whose searches --dump-outputs writes (at most DUMP_TREES of them)."""
    import numpy as np
    return np.sort(np.random.RandomState(0).choice(n_trees, min(n_trees, DUMP_TREES), replace=False))


def dump_outputs(path, records, trees, move, game):
    """What the self-play path hands its caller, the training record of a search (policy target, root value, the position
    searched and the move played), for search number `move` of every tree in `trees`, as float arrays path/<name>.npy.
    Which move a tree is on when the last timed step ends depends on timing (the step kernel's cycle budget is a clock
    bound); what each search computes does not, so this selection is the same from run to run for the same arguments.
    A tree that has not finished that search (an arena overflow stops a tree) gives a row of NaN."""
    import numpy as np
    from alphazero_openspiel_b200.engine import game_shape, parse_game_name
    from alphazero_openspiel_b200.examplegenerator import boards_from_bitboards, policy_targets_batch
    gid, rows, cols = parse_game_name(game)
    n_actions = game_shape(game)[1]
    recs = np.concatenate(records)
    recs = recs[np.lexsort((recs["ply"], recs["game_seq"], recs["tree"]))]
    first = np.searchsorted(recs["tree"], recs["tree"])          # index of each tree's first search
    recs = recs[np.arange(len(recs)) - first == move - 1]
    slot = np.searchsorted(trees, recs["tree"])
    n = len(trees)
    out = {"tree": trees.astype(np.float64)}
    for name in ("game_seq", "ply", "action", "root_q"):
        out[name] = np.full((n,), np.nan)
        out[name][slot] = recs[name]
    out["policy"] = np.full((n, n_actions), np.nan)
    out["policy"][slot] = policy_targets_batch(recs["counts"], recs["actions"], recs["n_legal"], n_actions)
    out["board"] = np.full((n, 4, rows, cols), np.nan, dtype=np.float32)
    out["board"][slot] = boards_from_bitboards(gid, rows, cols, recs["bb"], recs["ply"])
    os.makedirs(path, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), a)
    if len(recs) < n:
        sys.stderr.write("WARNING: --dump-outputs: %d of %d sample trees had not finished search %d (rows of NaN)\n"
                         % (n - len(recs), n, move))


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from alphazero_openspiel_b200 import _lib as L
    from alphazero_openspiel_b200.engine import game_shape, parse_game_name
    from alphazero_openspiel_b200.examplegenerator import SelfPlayRunner
    from alphazero_openspiel_b200.network import Net

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    L.load()  # fail loudly if the CUDA extension is missing

    game = args.game
    shape, n_actions = game_shape(game)
    _, rows, cols = parse_game_name(game)
    net, weights = build_net(args, shape, n_actions)
    if world > 1:
        from alphazero_openspiel_b200 import parallel
        parallel.broadcast_weights(net, src=0, device=dev)  # NCCL: the per-generation weight broadcast

    runner = SelfPlayRunner(net, game, dev, args.trees, n_playouts=args.playouts, c_puct=2.5, use_dirichlet=True,
                            dirichlet_ratio=0.25, temperature=1.0, backup="on-policy", seed=0xC4 + rank,
                            auto_restart=True, random_start_mod=21, max_sims_per_step=args.sim_cap, records=True,
                            use_graph=not args.no_graph, evaluator=args.evaluator,
                            keep_search_tree=not args.no_keep_tree, node_capacity=args.node_capacity,
                            virtual_loss=args.virtual_loss, step_cycle_budget=args.cycle_budget)
    rps = ROUNDS_PER_STEP
    n_rounds = args.steps * rps
    # --dump-outputs keeps the sample trees' training records from every drain up to the end of the timed steps
    dump = args.dump_outputs and rank == 0
    kept, sample = [], dump_trees(args.trees) if dump else None

    def drain():
        recs = runner.drain()
        if dump:
            kept.append(recs[(recs["kind"] == 0) & np.isin(recs["tree"], sample)])

    # ---- settle (untimed, steady state) + warm-up (untimed, W steps).  nvidia-smi needs up to a second to deliver its
    # first sample, so the clock sampler is started before the warm-up; only samples taken after mark() are reported.
    settle_rounds = 0 if args.no_settle else settle(runner, args.trees, dev, drain)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    runner.round(args.warmup * rps)
    drain()
    torch.cuda.synchronize(dev)
    if rank == 0:
        t_wait = time.time()
        while not sampler.rows and time.time() - t_wait < 3.0:
            runner.round(rps)
            torch.cuda.synchronize(dev)
        drain()
        torch.cuda.synchronize(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- timed region: K steps = K * 50 round trips, CUDA events on the launching stream
    c0 = runner.counters()
    barrier()
    sampler.mark()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    runner.round(n_rounds)
    ev1.record()
    torch.cuda.synchronize(dev)
    barrier()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if rank == 0 else None
    c1 = runner.counters()
    d = {k: c1[k] - c0[k] for k in c1}

    # ---- e2e: same metric through the public API with HOST buffers: host weights -> device (H2D), K steps,
    # training records + counters back to host memory (D2H), wall clock around all of it
    host_net = Net(shape, n_actions)
    host_net.load_state_dict(net.state_dict())
    for t in list(host_net.parameters()) + list(host_net.buffers()):
        t.data = t.data.pin_memory()
    h2d = sum(t.numel() * t.element_size() for t in list(host_net.parameters()) + list(host_net.buffers()))
    drain()
    if dump:
        dump_outputs(args.dump_outputs, kept, sample, dump_move(args), game)
    barrier()
    e0 = runner.counters()
    t0 = time.perf_counter()
    runner.load_weights(host_net)
    runner.round(n_rounds)
    recs = runner.drain()
    e1 = runner.counters()
    torch.cuda.synchronize(dev)
    t_e2e = time.perf_counter() - t0
    d2h = recs.nbytes + 8 * len(L.CTR_NAMES)
    e2e_sims = e1["sims"] - e0["sims"]

    # ---- per-launch durations of the hand-written kernels, live, CUDA events around each launch (un-graphed pass)
    n_probe = min(n_rounds, 200)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_probe)]
    nn_evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_probe)]
    p0 = runner.counters()
    ev = runner.evaluator
    fused = hasattr(ev, "timing")
    if fused:
        ev.timing = []
    for a, b in zip(evs, nn_evs):
        a[0].record()
        runner.engine.step(ev.priors, ev.values, None, ev.obs, L.OBS_BF16_NHWC)
        a[1].record()
        if runner._async_compact:
            runner.engine.compact()
        b[0].record()
        ev()
        b[1].record()
    torch.cuda.synchronize(dev)
    p1 = runner.counters()
    pd = {k: p1[k] - p0[k] for k in p1}
    step_ms = sum(a.elapsed_time(b) for a, b in evs) / n_probe
    nn_ms = sum(a.elapsed_time(b) for a, b in nn_evs) / n_probe
    alg_bytes_per_launch = algorithmic_bytes(pd, rows * cols, n_actions) / n_probe
    conv_ms, conv_n, stem_ms = 0.0, 0, 0.0
    by_name = {}
    if fused:
        for name, e0_, e1_ in ev.timing:
            acc = by_name.setdefault(name, [0.0, 0])
            acc[0] += e0_.elapsed_time(e1_)
            acc[1] += 1
            if name == "stem":
                stem_ms += e0_.elapsed_time(e1_)
            elif name.startswith("conv"):
                conv_ms += e0_.elapsed_time(e1_)
                conv_n += 1
        ev.timing = None

    # ---- reduce over ranks
    stats = torch.tensor([ms, float(d["sims"]), float(d["moves"]), float(d["games"]), float(d["overflow"]),
                          t_e2e, float(e2e_sims)], dtype=torch.float64, device=dev)
    if world > 1:
        mx = stats.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(stats, op=dist.ReduceOp.SUM)
        ms, t_e2e = float(mx[0]), float(mx[5])
    else:
        ms, t_e2e = float(stats[0]), float(stats[5])
    sims, moves, games, overflow, e2e_sims = float(stats[1]), float(stats[2]), float(stats[3]), float(stats[4]), \
        float(stats[6])
    node_bytes, node_cap = runner.engine.device_bytes, int(runner.engine.cfg.node_capacity)
    rows_per_round = runner.evaluator.batch if hasattr(runner.evaluator, "batch") else args.trees
    runner.close()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = load_peaks()
    value = sims / (ms / 1e3)
    evals_per_s = rows_per_round * world * n_rounds / (ms / 1e3)
    flops = FLOPS_PER_EVAL.get(game, 0)
    hbm_ach = alg_bytes_per_launch / (step_ms / 1e3) / 1e9
    nn_tflops = rows_per_round * flops / (nn_ms / 1e3) / 1e12
    tree_roofline = {"kernel": "k_step (select/expand/backup/advance/encode)", "bound": "hbm",
                     "achieved": hbm_ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": hbm_ach / peaks["hbm_gbs"],
                     "traffic": None, "peak_source": peaks["source"], "avg_launch_ms": step_ms,
                     "algorithmic_bytes_per_launch": alg_bytes_per_launch,
                     "share_of_step": step_ms / (step_ms + nn_ms)}
    conv_roofline = None
    if fused and conv_n:
        # dominant kernel: k_conv8 (3x3 conv, 50->50 filters, nine launches per evaluation).  Per launch the algorithm
        # needs boards x 2*HW*50*50*9 FLOPs and reads / writes every [B][H][W][64] bf16 tensor it touches once:
        # in + out (+ residual) (+ second output) = 2-4 tensors -> HBM is the binding roofline of the launch.
        conv_flops = rows_per_round * 2.0 * rows * cols * 50 * 50 * 9
        tensor_bytes = rows_per_round * rows * cols * 64 * 2.0
        n_tensors = {"conv": 2, "conv+res": 3, "conv+out2": 3, "conv+res+out2": 4}
        conv_bytes = sum(n_tensors.get(k, 2) * tensor_bytes * v[1] for k, v in by_name.items() if k.startswith("conv")) / conv_n
        avg_conv_ms = conv_ms / conv_n
        ach = conv_bytes / (avg_conv_ms / 1e3) / 1e9
        conv_roofline = {"kernel": "k_conv8 (tcgen05 implicit-GEMM 3x3 conv, TMA in/out, fused BN/LeakyReLU/residual epilogue)",
                         "bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": ach / peaks["hbm_gbs"], "traffic": conv_dram_traffic(game, rows_per_round),
                         "peak_source": peaks["source"],
                         "avg_launch_ms": avg_conv_ms, "launches_per_step": rps * conv_n / n_probe,
                         "algorithmic_bytes_per_launch": conv_bytes, "algorithmic_flops_per_launch": conv_flops,
                         "tensor_tflops": conv_flops / (avg_conv_ms / 1e3) / 1e12,
                         "tensor_frac_of_burst_peak": conv_flops / (avg_conv_ms / 1e3) / 1e12 / peaks["bf16_tflops"],
                         "stem_avg_launch_ms": stem_ms / n_probe,
                         "share_of_step": conv_ms / n_probe / (step_ms + nn_ms),
                         "launch_ms_by_kind": {k: v[0] / v[1] for k, v in sorted(by_name.items())},
                         "note": "averaged over the conv launches of one evaluation; traffic = dram read+write per "
                                 "launch averaged the same way from the committed ncu --set full capture "
                                 "(profiles/conv_traffic.json), null when this shape was not captured"}
    launches_per_round = (2 if not args.no_keep_tree else 1) + (len(by_name) and sum(v[1] for v in by_name.values()) // n_probe)
    line = {
        "metric": "mcts_simulations_per_sec", "value": value, "unit": "sims/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args), "game": game, "n_playouts": args.playouts,
                   "trees_per_gpu": args.trees, "parallelism": "independent game pool per GPU (x%d)" % world,
                   "rounds_per_step": rps, "settle_rounds": settle_rounds,
                   "step": "%d evaluator round trips (az_step + ResNet forward, one CUDA graph replay each)" % rps,
                   "evaluator": ("ResNet 5x50 bf16, hand-written tcgen05 implicit-GEMM convs + FC head kernels (az_resnet.cu)"
                                 if args.evaluator == "fused" else "ResNet 5x50 bf16 channels-last via PyTorch")
                   + ", " + weights,
                   "noise": "device Dirichlet(0.3), ratio 0.25", "start": "counter % 21 random plies",
                   "sim_cap_per_step": args.sim_cap, "step_cycle_budget": int(runner.engine.cfg.step_cycle_budget),
                   "cuda_graph": not args.no_graph,
                   "virtual_loss_leaves": args.virtual_loss,
                   "l2_policy": "working set (%.1f GB node arenas + %.0f MB activations per round trip) exceeds the 126 MB L2"
                                % (node_bytes / 1e9, rows_per_round * rows * cols * 64 * 2 * 3 / 1e6)},
        "ms_per_round_trip": ms / n_rounds,
        "games_per_sec": games / (ms / 1e3), "moves_per_sec": moves / (ms / 1e3), "evals_per_sec": evals_per_s,
        "sims_per_eval_slot": sims / (rows_per_round * world * n_rounds), "overflow": overflow,
        "peak_nodes_per_tree": c1.get("peak_nodes"), "node_capacity": node_cap,
        "e2e": {"value": e2e_sims / t_e2e, "unit": "sims/s", "h2d_bytes_per_step": h2d / args.steps,
                "d2h_bytes_per_step": d2h / args.steps,
                "what": "SelfPlayRunner.load_weights(host net) + round(K*50) + drain()/counters() to host, wall clock"},
        # our kernels per round trip: k_step, k_compact, stem + 9 convs + FC head
        "gpu_launches": n_rounds * world * launches_per_round,
        "roofline": conv_roofline if fused else tree_roofline,
        "tree_roofline": tree_roofline,
        "nn_roofline": {"kernel": "ResNet forward (%s): stem + 9 convs + FC head" % args.evaluator, "bound": "tensor",
                        "achieved": nn_tflops, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                        "frac": nn_tflops / peaks["bf16_tflops_sustained"], "avg_forward_ms": nn_ms,
                        "flops_per_eval": flops, "peak_source": peaks["source"]},
        "clocks": clocks,
    }
    if world == 1 and not args.no_cpu_baseline:
        try:
            line["cpu_baseline"] = cpu_baseline(game, args.playouts, seconds_budget=args.cpu_seconds)
        except Exception as e:  # the baseline must never hide the GPU number
            line["cpu_baseline"] = {"value": None, "unit": "sims/s", "cores": 0, "kind": "port",
                                    "sample": "failed: %r" % (e,)}
    if overflow:
        sys.stderr.write("WARNING: %d arena/record overflows in the timed region -- raise --node-capacity\n" % overflow)
    emit(line)
    if world > 1:
        dist.destroy_process_group()


def run_train(args):
    """BASELINE configs[4]: the reference's full train.py loop (train.py:272-293) with the Trainer defaults of
    train.py:24-49 -- 500 games / generation at 100 sims/move, 500 optimisation steps of batch 256 (Adam 1e-3, wd 1e-4) --
    self-play generation sharded over the GPUs (one process per GPU), records all-gathered, rank 0 trains, NCCL weight
    broadcast.  One bench "step" = one generation (generate -> train -> broadcast); wall clock with device synchronisation
    on both sides (the loop is host-driven by nature), max over ranks."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from alphazero_openspiel_b200 import _lib as L, parallel
    from alphazero_openspiel_b200.train import Trainer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    L.load()
    torch.manual_seed(0)
    np.random.seed(rank)
    tr = Trainer(name="bench", name_game=args.game, device=dev, save=False, n_playouts_train=args.playouts,
                 array_buffer=not args.list_buffer, device_training=not args.list_buffer,
                 graph_step=not (args.list_buffer or args.eager_train or args.ddp), ddp=args.ddp)
    gens = args.steps if args.generations is None else max(1, args.generations)

    def sync():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()

    def one_generation():
        sync()
        t0 = time.perf_counter()
        tr.generation += 1
        tr.generate_examples(tr.n_games_per_generation)
        sync()
        t1 = time.perf_counter()
        tr.train_network()
        sync()
        t2 = time.perf_counter()
        return t1 - t0, t2 - t1, dict(tr.last_generation_stats)

    one_generation()  # warm-up generation (CUDA graph capture, cuDNN autotune, allocator)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        sampler.mark()
    gen_s, train_s, sims, games = [], [], 0, 0
    for _ in range(gens):
        g, t, st = one_generation()
        gen_s.append(g)
        train_s.append(t)
        sims += st.get("sims", 0)
        games += st.get("games", 0)
    # the weight broadcast alone (it is the tail of train_network): NCCL broadcast of one flat fp32 bucket
    sync()
    t0 = time.perf_counter()
    for _ in range(10):
        parallel.broadcast_weights(tr.current_net, src=0, device=dev)
    sync()
    bcast_ms = (time.perf_counter() - t0) / 10 * 1e3
    tot = torch.tensor([sum(gen_s), sum(train_s), float(sims)], dtype=torch.float64, device=dev)
    if world > 1:
        mx = tot.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = tot.clone()
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        tot = torch.stack([mx[0], mx[1], sm[2]])
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        gen_t, train_t, all_sims = float(tot[0]), float(tot[1]), float(tot[2])
        wall = gen_t + train_t
        line = {"metric": "selfplay_games_per_sec_full_train_loop", "value": games / wall, "unit": "games/s",
                "n_gpus": world, "steps": gens, "warmup": 1, "ms_per_step": 1e3 * wall / gens, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f64 search / bf16 evaluator / fp32 training",
                "data": "synthetic",
                "config": {"workload": "BASELINE configs[4]: full train.py loop, %s, Trainer defaults (%d games/generation, "
                                       "%d sims/move, %d x batch %d Adam steps), generation on %d GPU(s) + NCCL weight broadcast"
                                       % (args.game, tr.n_games_per_generation, args.playouts, tr.n_batches_per_generation,
                                          tr.batch_size, world),
                           "step": "one generation: generate_examples -> train_network -> broadcast"},
                "generation_s": gen_t / gens, "train_s": train_t / gens, "broadcast_ms": bcast_ms,
                "sims_per_sec_in_generation": all_sims / gen_t if gen_t > 0 else None,
                "games_per_generation": games / gens, "buffer": "arrays on device" if not args.list_buffer else "python lists",
                "train_step": ("one CUDA graph per optimisation step" if tr.graph_step else "eager PyTorch") +
                              (", data-parallel over %d ranks (gradient all-reduce)" % world if tr.ddp and world > 1
                               else (", rank 0 trains + NCCL weight broadcast" if world > 1 else "")),
                "clocks": clocks}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps; one step = %d evaluator round trips" % ROUNDS_PER_STEP)
    ap.add_argument("--warmup", type=int, default=5, help="untimed warm-up steps after the settle phase")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c4", choices=sorted(CONFIGS), help="BASELINE.json config (default: configs[2])")
    ap.add_argument("--game", default=None)
    ap.add_argument("--trees", type=int, default=None)
    ap.add_argument("--playouts", type=int, default=None)
    ap.add_argument("--sim-cap", type=int, default=16)
    ap.add_argument("--cycle-budget", type=int, default=None,
                    help="az_config.step_cycle_budget: SM cycles after which a tree starts no further in-kernel simulation "
                         "(default: SelfPlayRunner's choice by pool size)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-settle", action="store_true", help="profiling runs: skip the steady-state settle phase")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=20.0)
    ap.add_argument("--ref-repeat", action="store_true")
    ap.add_argument("--evaluator", default="fused", choices=["fused", "torch"])
    ap.add_argument("--node-capacity", type=int, default=0)
    ap.add_argument("--virtual-loss", type=int, default=0, help="K leaves in flight per tree (non-bit-exact mode); 0 = off")
    ap.add_argument("--generations", type=int, default=None, help="--config train: generations timed (default: --steps)")
    ap.add_argument("--ddp", action="store_true", help="--config train: data-parallel optimisation steps (NCCL gradient all-reduce)")
    ap.add_argument("--eager-train", action="store_true", help="--config train: eager optimisation steps (no CUDA graph)")
    ap.add_argument("--list-buffer", action="store_true", help="--config train: the reference's Python-list replay buffer")
    ap.add_argument("--no-keep-tree", action="store_true", help="experiment: fresh tree every move (no re-root compaction)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="self-play configs: after the timed steps write the training records of a fixed sample of trees as "
                         "DIR/<name>.npy (see dump_outputs), for comparing the outputs of two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    # stdout carries ONE JSON line and nothing else: whatever libraries write to file descriptor 1 (NCCL prints its version
    # banner there when NCCL_DEBUG is VERSION or higher, as on some boxes) is sent to stderr; emit() writes to the real stdout
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    cfg = CONFIGS[args.config]
    args.game = args.game or cfg["game"]
    args.trees = args.trees or cfg["trees"]
    args.playouts = args.playouts or cfg["playouts"]
    if args.warmup < 3:
        args.warmup = 3
    if args.dump_outputs and (args.impl == "reference" or args.config == "train"):
        ap.error("--dump-outputs is for the self-play configs (c4, bt6, bt8) of --impl ours")
    if args.dump_outputs and dump_move(args) < 1:
        ap.error("--dump-outputs: too few round trips for every tree to finish a search; raise --steps or --warmup")
    if args.impl == "reference":
        run_reference(args)
    elif args.config == "train":
        run_train(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
