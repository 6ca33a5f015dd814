"""Drop-in for the reference's examplegenerator.py self-play generator, batched on the GPU.

  ExampleGenerator(net, game_name, device, n_pools=1, n_processes=1, **kwargs)   examplegenerator.py:80-104
      .generate_examples(n_games) -> list[game] of list[[info_state_str, board (C+1,H,W) float64,
                                                          policy list[A], value]]  examplegenerator.py:164-175

The reference runs one OS process per game plus a `handle_gpu` process that batches whichever boards happen
to be ready (examplegenerator.py:57-77,106-138).  Here every game is a search tree in HBM; one az_step() +
one batched bf16 ResNet forward advances ALL games by one evaluator round trip, with both captured in a single
CUDA graph.  `n_pools` / `n_processes` are accepted for signature parity and ignored: parallelism is the
number of concurrent trees (`n_trees`, default min(n_games, 16384)).  With torch.distributed initialised
(one process per GPU) each rank plays its share of the games and the training records are all-gathered over
NCCL (parallel.gather_records); weights are broadcast with parallel.broadcast_weights.

Host-side conversion of device records to the reference's example format uses the reference's own numpy
expressions (visit counts -> normalised -> remove_illegal_actions), so policy targets are bit-identical
(SURVEY A.9).
"""
import copy
import logging
import time

import numpy as np
import torch

from . import _lib as L
from .engine import Engine, parse_game_name, record_dtype
from .network import BatchedEvaluator

logger = logging.getLogger("alphazero")

DEFAULT_MAX_TREES = 16384


def boards_from_bitboards(game_id, rows, cols, bb, ply):
    """Vectorised state_to_board (network.py:9-18) from canonical bitboards: -> float64 [n, 4, rows, cols]."""
    n = bb.shape[0]
    cells = rows * cols
    shifts = np.arange(cells, dtype=np.uint64)
    p0 = ((bb[:, 0:1] >> shifts) & np.uint64(1)).astype(np.float64)
    p1 = ((bb[:, 1:2] >> shifts) & np.uint64(1)).astype(np.float64)
    empty = 1.0 - p0 - p1
    cur = np.broadcast_to((ply.astype(np.int64) & 1).astype(np.float64)[:, None], (n, cells))
    if game_id == L.GAME_CONNECT_FOUR:
        planes = [empty, p1, p0, cur]       # empty, 'o' (player 1), 'x' (player 0)  -- SURVEY B.2
    else:
        planes = [p0, p1, empty, cur]       # black, white, empty                   -- SURVEY B.3
    return np.stack(planes, axis=1).reshape(n, 4, rows, cols)


def policy_target(counts, actions, n_legal, num_actions):
    """Visit counts -> the reference's policy target list (mcts.py:161-162 + alphazerobot.py:7-18,89-93)."""
    visits = [0] * num_actions
    legal = []
    for k in range(n_legal):
        visits[int(actions[k])] = int(counts[k])
        legal.append(int(actions[k]))
    total = sum(visits)
    probs = np.array([float(v) / total for v in visits])
    mask = np.zeros(probs.shape, dtype=bool)
    mask[legal] = True
    probs[~mask] = 0.0
    if np.sum(probs) > 1e-6:
        probs = probs / np.sum(probs)
    else:
        probs = np.zeros(len(probs))
        probs[legal] = 1. / len(legal)
    out = [0.0] * num_actions
    for a in legal:
        out[a] = probs[a]
    return out


def policy_targets_batch(counts, actions, n_legal, num_actions):
    """Vectorised policy_target for many records: float64 [n, num_actions], bit-identical to the per-record expressions
    (IEEE division is elementwise; the row sums run over the same contiguous vectors as np.sum on one record)."""
    n = counts.shape[0]
    maxc = counts.shape[1]
    valid = np.arange(maxc)[None, :] < n_legal[:, None]
    rows = np.repeat(np.arange(n), maxc).reshape(n, maxc)[valid]
    cols = actions.astype(np.int64)[valid]
    visits = np.zeros((n, num_actions), dtype=np.float64)
    visits[rows, cols] = counts[valid]
    total = counts.astype(np.int64).sum(axis=1).astype(np.float64) * valid.any(axis=1)
    probs = visits / total[:, None]                      # float(v) / sum(visits)               mcts.py:161-162
    s = np.array([np.sum(probs[i]) for i in range(n)]) if num_actions >= 8 else probs.sum(axis=1)
    ok = s > 1e-6                                        # remove_illegal_actions               alphazerobot.py:12-17
    out = np.zeros_like(probs)
    out[ok] = probs[ok] / s[ok][:, None]
    if not ok.all():
        legal_mask = np.zeros((n, num_actions), dtype=bool)
        legal_mask[rows, cols] = True
        uni = legal_mask / np.maximum(n_legal, 1)[:, None].astype(np.float64)
        out[~ok] = uni[~ok]
    return out


def records_to_games(records, game_name, backup="on-policy"):
    """Device training records -> list of games in the reference's example format (game_utils.py:168-204).
    Only games that have their closing (kind 1) record are returned.  A fast search's ply record (F_PLAYOUT_CAP, end 3) is
    no example, but its action stays in the history (the key) of the examples after it."""
    gid, rows, cols = parse_game_name(game_name)
    num_actions = 7 if gid == L.GAME_CONNECT_FOUR else rows * cols * 12
    if len(records) == 0:
        return []
    order = np.lexsort((records["kind"], records["ply"], records["game_seq"], records["tree"]))
    recs = records[order]
    boards = boards_from_bitboards(gid, rows, cols, recs["bb"], recs["ply"])
    ply_mask = recs["kind"] == 0
    pol_rows = np.full((len(recs),), -1, dtype=np.int64)
    pol_rows[ply_mask] = np.arange(int(ply_mask.sum()))
    pols = policy_targets_batch(recs["counts"][ply_mask], recs["actions"][ply_mask], recs["n_legal"][ply_mask], num_actions)
    key = recs["tree"].astype(np.int64) * (1 << 32) + recs["game_seq"].astype(np.int64)
    starts = np.flatnonzero(np.r_[True, key[1:] != key[:-1]])
    ends = np.r_[starts[1:], len(recs)]
    games = []
    for s, e in zip(starts, ends):
        if recs["kind"][e - 1] != 1:
            continue  # unfinished game
        history = []
        game = []
        # A game that did not start at the initial position (random_start_mod > 0: k random plies first) has no action
        # history for its first k plies: its start position goes into the key instead, so that remove_duplicates
        # (train.py:176-198 keys on example[0]) never merges different positions.  The reference always starts at ply 0
        # (game_utils.py:150-154), where the key is exactly its information_state string.
        prefix = start_key_prefix(recs["bb"][s], recs["ply"][s])
        reward = float(recs["root_q"][e - 1])  # kind-1 record carries returns()[0]
        for i in range(s, e - 1):
            r = recs[i]
            if r["end"] == 3:
                history.append(int(r["action"]))
                continue
            pol = pols[pol_rows[i]].tolist()
            if backup == "soft-Z":
                value = -float(r["root_q"])
            elif backup == "A0C":
                value = float(r["v_a0c"])
            elif backup == "off-policy":
                value = float(r["v_offpolicy"])
            else:
                # on-policy (game_utils.py:168-169,200-204): returns()[0] for player 0 to move, negated for player 1.  The
                # sign comes from the position's real ply, not from the index of the example inside the game.
                value = reward if (int(r["ply"]) & 1) == 0 else -reward
            game.append([prefix + ", ".join(str(a) for a in history), boards[i], pol, value])
            history.append(int(r["action"]))
        games.append(game)
    return games


def resign_threshold_for(records, target_fp, current):
    """Resign threshold calibrated on the no-resign games (F_RESIGN records of kind 1 with end == 2): the minimum r of every
    player of such a game who did not lose, sorted v_1 <= ... <= v_n, gives v_(k+1) with k = floor(target_fp * n), capped at
    1.0 -- so at most a target_fp share of those players would have resigned below it.  `current` when there is no value
    (n == 0) or k >= n.  A player who never moved (minimum 2.0) has no value."""
    ends = records[(records["kind"] == 1) & (records["end"] == 2)]
    ret0 = ends["root_q"]
    v = np.concatenate([ends["v_a0c"][ret0 >= 0], ends["v_offpolicy"][ret0 <= 0]]).astype(np.float64)
    v = np.sort(v[v <= 1.0])
    k = int(np.floor(target_fp * len(v)))
    if k >= len(v):
        return current
    return min(float(v[k]), 1.0)


def start_key_prefix(bb, ply):
    """'' for a game from the initial position, else a tag of the position the game started from."""
    if int(ply) == 0:
        return ""
    return "start=%x/%x/%d; " % (int(bb[0]), int(bb[1]), int(ply))


class SelfPlayRunner:
    """Engine + batched evaluator wired together; one `round()` = az_step + ResNet forward in one CUDA graph."""

    def __init__(self, net, game_name, device, n_trees, n_playouts=100, c_puct=2.5, use_dirichlet=True,
                 dirichlet_ratio=0.25, temperature=1.0, num_probabilistic_actions=1000, keep_search_tree=True,
                 backup="on-policy", seed=0, max_games=0, auto_restart=True, random_start_mod=0,
                 max_sims_per_step=16, records=True, use_graph=True, noise_mode=None, node_capacity=0,
                 record_capacity=0, evaluator="fused", virtual_loss=0, step_cycle_budget=None, eval_cache=None,
                 eval_cache_log2=0, resign_threshold=None, resign_disabled_fraction=0.1, fast_playouts=None,
                 full_search_fraction=0.25, forced_playouts=None, **_ignored):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise L.EngineUnavailable("SelfPlayRunner needs a CUDA device; there is no CPU fallback")
        dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.device = torch.device("cuda", dev_index)
        flags = L.F_SAMPLE_MOVES
        if keep_search_tree:
            flags |= L.F_KEEP_TREE | L.F_ASYNC_COMPACT   # re-root compaction on a side stream, next to the evaluator
        if auto_restart:
            flags |= L.F_AUTO_RESTART
        if records:
            flags |= L.F_RECORDS
            if backup == "off-policy":
                flags |= L.F_OFFPOLICY
        if random_start_mod > 0:
            flags |= L.F_RANDOM_START
        if resign_threshold is not None:
            flags |= L.F_RESIGN     # resignation (an extension: the reference plays every game to its end)
        if fast_playouts is not None:
            # playout cap randomization (an extension: the reference runs every search with n_playouts): a
            # full_search_fraction share of the searches is full, the others run fast_playouts simulations without root
            # noise, and their positions are no training examples
            flags |= L.F_PLAYOUT_CAP
        if forced_playouts is not None:
            # forced playouts and policy target pruning (an extension the reference does not have): every visited root
            # child of a search with root noise gets at least sqrt(k * P * N) visits, and the visits it got only from that
            # floor are taken out of the policy target and the move choice
            flags |= L.F_FORCED_PLAYOUTS
        if noise_mode is None:
            noise_mode = L.NOISE_DIRICHLET if use_dirichlet else L.NOISE_NONE
        # virtual_loss = K > 0: K leaves in flight per tree (AZ_F_VIRTUAL_LOSS, NOT bit-exact with the reference), for pools
        # too small to fill the evaluator with one row per tree; the evaluator batch becomes n_trees * K rows
        leaves = int(virtual_loss) if virtual_loss and int(virtual_loss) > 0 else 1
        if virtual_loss and int(virtual_loss) > 0:
            flags |= L.F_VIRTUAL_LOSS
        if step_cycle_budget is None:
            # time bound on a tree's in-kernel (terminal-leaf) simulations per launch, in SM cycles: the longer the evaluator
            # of a round trip runs, the more k_step time an extra simulation per row is worth (measured, profiles/
            # r02_summary.md: 16,384 Connect Four trees best at 60-80 k, 1,024 Breakthrough 6x6 trees at 30 k)
            step_cycle_budget = 64000 if n_trees * leaves >= 4096 else 30000
        self.backup = backup
        self.game_name = game_name
        with torch.cuda.device(self.device):
            n_rows = n_trees * leaves
            if evaluator == "fused":      # hand-written tcgen05 convs (csrc/az_resnet.cu)
                from .nn_fused import FusedEvaluator
                self.evaluator = FusedEvaluator(net, n_rows, self.device)
            elif evaluator == "torch":    # cuDNN/cuBLAS through PyTorch (numerics reference for the fused path)
                self.evaluator = BatchedEvaluator(net, n_rows, self.device, use_graph=False)
            else:
                raise ValueError("evaluator must be 'fused' or 'torch'")
            # eval_cache (None = on where it is exact): expand leaves whose position was already evaluated from a device
            # table of the evaluator's outputs (F_EVAL_CACHE) instead of sending them to the evaluator again.  Results are
            # unchanged only if an output row depends on that row's board alone: true of the fused evaluator, not promised
            # by cuDNN / cuBLAS (torch evaluator).  Virtual-loss mode has no cache.
            cache_ok = getattr(self.evaluator, "row_independent", False) and not (flags & L.F_VIRTUAL_LOSS)
            if eval_cache is None:
                eval_cache = cache_ok
            elif eval_cache and not cache_ok:
                raise ValueError("eval_cache needs the fused evaluator (with its own FC head) and virtual_loss=0")
            if eval_cache:
                flags |= L.F_EVAL_CACHE
            self.engine = Engine(game_name, n_trees, n_playouts=n_playouts, c_puct=c_puct,
                                 dirichlet_ratio=dirichlet_ratio, temperature=temperature,
                                 num_probabilistic_actions=num_probabilistic_actions, noise_mode=noise_mode,
                                 eval_mode=L.EVAL_EXTERNAL, flags=flags, seed=seed, device=dev_index,
                                 max_sims_per_step=max_sims_per_step, start_plies_mod=random_start_mod,
                                 max_games=max_games, node_capacity=node_capacity,
                                 record_capacity=record_capacity, leaves_per_tree=leaves,
                                 step_cycle_budget=step_cycle_budget, eval_cache_log2=eval_cache_log2)
        if resign_threshold is not None:
            self.set_resign(resign_threshold, resign_disabled_fraction)
        if fast_playouts is not None:
            self.set_playout_cap(fast_playouts, full_search_fraction)
        if forced_playouts is not None:
            self.set_forced_playouts(forced_playouts)
        self.use_graph = use_graph
        self._graph = None
        self._first = True
        self.rounds = 0
        self._async_compact = bool(keep_search_tree)
        self._side = torch.cuda.Stream(self.device) if self._async_compact else None
        self._ev_fork = torch.cuda.Event()
        self._ev_join = torch.cuda.Event()

    def load_weights(self, net):
        """New generation's weights (host or device Net) into the captured evaluator, in place."""
        with torch.cuda.device(self.device):
            self.evaluator.load(net)
            if self.engine.flags & L.F_EVAL_CACHE:
                self.engine.invalidate_eval_cache()

    def set_resign(self, threshold, disabled_fraction=0.1):
        """Resign threshold and share of no-resign calibration games (needs resign_threshold at construction).  Takes effect
        on the next round, also in an already captured graph."""
        with torch.cuda.device(self.device):
            self.engine.set_resign(threshold, int(round(float(disabled_fraction) * 1000)))

    def set_playout_cap(self, fast_playouts, full_search_fraction=0.25):
        """Simulations of a fast search and share of full searches (needs fast_playouts at construction).  Takes effect for
        the searches that begin from the next round on, also in an already captured graph."""
        with torch.cuda.device(self.device):
            self.engine.set_playout_cap(fast_playouts, int(round(float(full_search_fraction) * 1000)))

    def set_forced_playouts(self, k):
        """k of the forced playouts (needs forced_playouts at construction; 0 forces nothing, 2.0 is KataGo's value).  Takes
        effect for the searches that begin from the next round on, also in an already captured graph."""
        with torch.cuda.device(self.device):
            self.engine.set_forced_playouts(k)

    @torch.no_grad()
    def _round_eager(self):
        ev = self.evaluator
        self.engine.step(ev.priors, ev.values, None, ev.obs, L.OBS_BF16_NHWC)
        if self._async_compact:
            # fork: k_compact (re-rooting of the trees that just moved) runs next to the evaluator, join before next step
            main = torch.cuda.current_stream(self.device)
            self._ev_fork.record(main)
            self._side.wait_event(self._ev_fork)
            self.engine.compact(self._side)
            self._ev_join.record(self._side)
            ev()
            main.wait_event(self._ev_join)
        else:
            ev()

    @torch.no_grad()
    def round(self, n=1):
        """n evaluator round trips for every tree."""
        with torch.cuda.device(self.device):
            if self._first:
                # first call: no evaluator outputs yet -- produce the initial requests, then evaluate them
                self.engine.step(None, None, None, self.evaluator.obs, L.OBS_BF16_NHWC)
                if self._async_compact:
                    self.engine.compact()
                self.evaluator()
                self._first = False
            if self.use_graph and self._graph is None:
                s = torch.cuda.Stream(self.device)
                s.wait_stream(torch.cuda.current_stream(self.device))
                with torch.cuda.stream(s):
                    for _ in range(3):
                        self._round_eager()
                torch.cuda.current_stream(self.device).wait_stream(s)
                self.rounds += 3
                self._graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self._graph):
                    self._round_eager()
                self.rounds += 1  # capture does not execute, but keep the count conservative
            for _ in range(n):
                if self.use_graph:
                    self._graph.replay()
                else:
                    self._round_eager()
            self.rounds += n

    def counters(self):
        return self.engine.counters()

    def drain(self):
        return self.engine.drain_records()

    def all_idle(self):
        """Every tree finished (or is stuck in AZ_PH_ERROR after an arena / depth overflow, which never leaves that phase:
        counters()['overflow'] tells the two apart)."""
        ph = self.engine.phases()
        return int(((ph != L.PH_IDLE) & (ph != L.PH_ERROR)).sum().item()) == 0

    def close(self):
        self.engine.close()


class ExampleGenerator:
    def __init__(self, net, game_name, device, n_pools=1, n_processes=1, **kwargs):
        self.is_test = bool(kwargs.pop("is_test", False))          # examplegenerator.py:93: a generator for generate_tests
        self.generate_statistics = bool(kwargs.pop("generate_statistics", False))
        self.net2 = None                                            # second network of zero-vs-zero (tournament.py:44-48)
        self.n_pools = n_pools            # accepted for signature parity; the GPU batch replaces pools/processes
        self.n_processes = n_processes
        self.net = copy.deepcopy(net)     # weights are frozen for the whole call (examplegenerator.py:86-87)
        self.net.to("cpu")
        self.net.eval()
        self.device = torch.device(device) if not isinstance(device, torch.device) else device
        self.game_name = game_name
        self.kwargs = kwargs
        self.rank0_only = bool(self.kwargs.pop("rank0_only", False))
        # resignation: with resign_threshold set, last_stats["resign_threshold_suggested"] is the threshold at which a
        # resign_false_positive share of the calibration games' non-losing players would have resigned
        self.resign_false_positive = float(self.kwargs.pop("resign_false_positive", 0.05))
        self.last_stats = {}

    def _resign_suggestion(self, records, stats):
        current = self.kwargs.get("resign_threshold")
        stats["resign_threshold_suggested"] = None if current is None else \
            resign_threshold_for(records, self.resign_false_positive, current)

    def generate_examples(self, n_games):
        """Play n_games self-play games (split over ranks when torch.distributed is initialised)."""
        from . import parallel
        rank, world = parallel.rank_world()
        share = n_games // world + (1 if rank < n_games % world else 0)
        t0 = time.time()
        records, stats = self._play(share, seed_offset=rank)
        if world > 1:
            records = parallel.gather_records(records, self.device)
        self._resign_suggestion(records, stats)     # on the gathered records: every rank derives the same value
        backup = str(self.kwargs.get("backup", "on-policy"))
        # rank0_only (Trainer: only rank 0 trains): the other ranks skip the host-side conversion and return no games
        games = [] if (self.rank0_only and rank != 0) else records_to_games(records, self.game_name, backup)
        stats["seconds"] = time.time() - t0
        self.last_stats = stats
        logger.info("Generated " + str(len(games)) + " games")
        return games

    def generate_batch(self, n_games):
        """Same games as generate_examples, as a replay.ExampleBatch (arrays) instead of Python lists: the conversion of
        16,384 games to the reference's list format costs seconds of host time, the arrays are built in milliseconds
        (SURVEY 8(f) rank 3).  `ExampleBatch.to_games()` gives the reference format on demand."""
        from . import parallel
        from .replay import ExampleBatch
        rank, world = parallel.rank_world()
        share = n_games // world + (1 if rank < n_games % world else 0)
        t0 = time.time()
        records, stats = self._play(share, seed_offset=rank)
        if world > 1:
            records = parallel.gather_records(records, self.device)
        self._resign_suggestion(records, stats)
        if self.rank0_only and rank != 0:
            records = records[:0]
        batch = ExampleBatch.from_records(records, self.game_name, str(self.kwargs.get("backup", "on-policy")))
        stats["seconds"] = time.time() - t0
        self.last_stats = stats
        logger.info("Generated " + str(batch.n_games) + " games")
        return batch

    def generate_tests(self, n_games, game_fn, n_playouts_mcts):
        """examplegenerator.py:177-195: n_games PAIRS of evaluation games (each `game_fn` call of the reference plays one game
        with either side moving first) -> average reward in [-1, 1], (avg, statistics) with generate_statistics.  `game_fn`
        is one of the reference's match-up functions (game_utils.py:51-145) or its name; all pairs run at once on the GPU
        (evaluate.py).  kwargs follow the reference: c_puct / n_playouts / temperature for the AlphaZero side of
        test_zero_vs_mcts (tournament.py:24 puts n_playouts into kwargs["settings1"]), settings1 / settings2 for
        test_zero_vs_zero, `net2` attribute for a second network.  Per-move tree statistics are not collected: the
        statistics list is empty."""
        from . import evaluate
        name = game_fn if isinstance(game_fn, str) else getattr(game_fn, "__name__", str(game_fn))
        kw = dict(self.kwargs)
        s1 = dict(kw.get("settings1") or {})
        s2 = dict(kw.get("settings2") or {})
        zero = {k: kw[k] for k in ("c_puct", "n_playouts", "temperature", "keep_search_tree", "use_probabilistic_actions")
                if k in kw}
        seed = int(kw.get("seed", np.random.randint(0, 2 ** 31 - 1)))
        dev = self.device
        if name == "test_zero_vs_mcts":
            zero.update(s1)
            a, b = evaluate.zero_vs_mcts(self.net, self.game_name, n_games, n_playouts_mcts, device=dev, seed=seed, **zero)
        elif name == "test_net_vs_mcts":
            a, b = evaluate.net_vs_mcts(self.net, self.game_name, n_games, n_playouts_mcts, device=dev, seed=seed)
        elif name == "test_zero_vs_zero":
            a, b = evaluate.zero_vs_zero(self.net, self.game_name, n_games, net2=self.net2, settings1=s1, settings2=s2,
                                         device=dev, seed=seed)
        elif name == "test_zero_vs_random":
            a, b = evaluate.zero_vs_random(self.net, self.game_name, n_games, device=dev, seed=seed,
                                           **{k: v for k, v in zero.items() if k in ("c_puct", "n_playouts", "keep_search_tree")})
        elif name == "test_net_vs_random":
            a, b = evaluate.net_vs_random(self.net, self.game_name, n_games, device=dev, seed=seed)
        else:
            raise ValueError("unknown evaluation game function %r" % (name,))
        avg_reward = (a + b) / 2.0            # sum(score1 + score2) / (2 * n_games)
        return (avg_reward, []) if self.generate_statistics else avg_reward

    def _play(self, n_games, seed_offset=0):
        kw = dict(self.kwargs)
        n_trees = int(kw.pop("n_trees", min(max(n_games, 1), DEFAULT_MAX_TREES)))
        n_trees = max(1, min(n_trees, max(n_games, 1)))
        seed = int(kw.pop("seed", np.random.randint(0, 2 ** 31 - 1))) + seed_offset
        if self.device.type != "cuda":
            raise L.EngineUnavailable("ExampleGenerator needs a CUDA device; there is no CPU fallback")
        if n_games == 0:
            gid, _, _ = parse_game_name(self.game_name)
            maxc = 7 if gid == L.GAME_CONNECT_FOUR else 48
            return np.empty((0,), dtype=record_dtype(maxc, (72 + 6 * maxc + 7) // 8 * 8)), {}
        runner = SelfPlayRunner(self.net, self.game_name, self.device, n_trees, seed=seed, max_games=n_games,
                                auto_restart=True, records=True, **kw)
        chunks = []
        # Drain the device record buffer before it can fill.  A tree emits one record per move (two when the game ends) and
        # runs at most max(1, max_sims_per_step) simulations per round, so at most 2 * n_trees * sims_per_round / n_playouts
        # records arrive per round; drain when half the capacity could be used.  With fast searches (fast_playouts) moves come
        # up to n_playouts / fast_playouts times faster: the bound takes the smallest playout count.
        n_playouts = max(1, int(kw.get("n_playouts", 100)))
        min_playouts = n_playouts if kw.get("fast_playouts") is None else max(1, min(n_playouts, int(kw["fast_playouts"])))
        cap = int(kw.get("max_sims_per_step", 16))
        sims_per_round = cap if cap > 0 else 64    # no count cap: the cycle budget / tree depth bound it far below this
        capacity = int(runner.engine.cfg.record_capacity)
        drain_every = max(64, int(capacity * min_playouts / (4.0 * sims_per_round * n_trees)) // 64 * 64)
        # upper bound on the round trips a generation can need: every game <= max plies, every ply <= n_playouts + 2 rounds
        max_plies = 42 if runner.engine.game_id == L.GAME_CONNECT_FOUR else 8 * runner.engine.rows * runner.engine.cols
        max_rounds = (n_games // n_trees + 2) * max_plies * (n_playouts + 3) + 1024
        since_drain = 0
        try:
            while True:
                runner.round(64)
                since_drain += 64
                if runner.all_idle():
                    break
                if since_drain >= drain_every:
                    chunks.append(runner.drain())
                    since_drain = 0
                    if runner.counters()["overflow"]:
                        break                # raised below: a tree in AZ_PH_ERROR never finishes
                if runner.rounds > max_rounds:
                    raise RuntimeError("self-play did not finish within %d round trips" % max_rounds)
            chunks.append(runner.drain())
            stats = runner.counters()
            stats["rounds"] = runner.rounds
            stats["fast_searches"] = int(sum(((c["kind"] == 0) & (c["end"] == 3)).sum() for c in chunks))
            if stats["overflow"]:
                raise RuntimeError("search arena / record buffer overflow (%d); raise node_capacity" %
                                   stats["overflow"])
        finally:
            runner.close()
        return np.concatenate(chunks), stats
