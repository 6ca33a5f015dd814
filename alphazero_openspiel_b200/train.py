"""Drop-in for the caller of the self-play path: the reference's Trainer (train.py:21-298) -- SURVEY 8(f) rank 1.

Same hyper-parameter attributes and method names (generate_examples / train_network / net_step / remove_duplicates /
update_buffer_size / run).  Self-play generation goes through the GPU ExampleGenerator; the optimisation step is plain
PyTorch (MSE value loss + cross-entropy against the visit-count targets, Adam lr 1e-3, weight decay 1e-4, train.py:85-128).
With torch.distributed initialised (one process per GPU): every rank plays its share of the games, the records are
all-gathered, rank 0 trains and the new weights are broadcast over NCCL (parallel.broadcast_weights) -- the reference
"broadcasts" by pickling a deepcopy of the net into every handler process (examplegenerator.py:121).
Strength evaluation (test_agent, train.py:238-270): all four match-ups run batched on the GPU (evaluate.py); the MCTS
opponent is the reference's own search in UCT mode with its random-rollout evaluator, on the device.
"""
import logging
import time
from datetime import datetime

import numpy as np
import torch
import torch.nn as nn

from . import parallel
from .engine import game_shape, reflect_actions
from .examplegenerator import ExampleGenerator
from .network import Net
from .replay import reflect_bits

logger = logging.getLogger("alphazero")


class Trainer:
    def __init__(self, name="openspieltest", backup="on-policy", name_game="connect_four", device=None, **overrides):
        # Experiment parameters (train.py:24-33)
        self.name_game = name_game
        self.name_run = name
        self.model_path = "models/"
        self.save = True
        self.save_n_gens = 10
        self.test_n_gens = 10
        self.n_tests = 200
        self.use_gpu = True
        self.n_pools = 1
        self.n_processes = 1
        # Algorithm parameters (train.py:35-49)
        self.n_games_per_generation = 500
        self.n_batches_per_generation = 500
        self.n_games_buffer_max = 20000
        self.batch_size = 256
        self.lr = 0.001
        self.n_games_buffer = 4 * self.n_games_per_generation
        self.temperature = 1.0
        self.dirichlet_ratio = 0.25
        self.uct_train = 2.5
        self.uct_test = 2.5
        self.n_playouts_train = 100
        self.backup = backup
        self.tree_strap = False
        self.it = 0
        self.n_generations = 201
        # Extension (SURVEY 8(f) rank 3): keep the replay buffer as arrays (replay.ExampleBatch) instead of Python lists.
        # Same sampling calls, duplicate merging and losses; `self.buffer` stays empty in this mode.
        self.array_buffer = False
        # Extension (SURVEY 8(f) rank 1): keep the replay buffer ON THE DEVICE (device_replay.DeviceReplay): duplicates are
        # merged by a device sort + segment mean and every minibatch is gathered / encoded by the az_observations kernel, so an
        # optimisation step moves only its 256 sample indices over PCIe.  Implies the array form of the examples.
        self.device_training = False
        # Extension: with torch.distributed, `ddp=True` trains data-parallel -- every rank takes batch_size / world of each
        # minibatch and the gradients are averaged with one NCCL all-reduce per step -- instead of rank 0 training alone.
        self.ddp = False
        # Extension: capture the whole device optimisation step (forward, losses, backward, Adam) in ONE CUDA graph with
        # static minibatch buffers -- the 5x50 network at batch 256 is launch-bound in eager mode (~60 kernels of a few
        # microseconds per step).  Same arithmetic, same sampling calls.  Needs device_training; not combined with ddp.
        self.graph_step = False
        # Extension: resignation in self-play (AlphaGo Zero; the reference plays every game to its end).  A game resigns once
        # its mover's root value and best child value are both below resign_threshold (-1: never, until the first
        # calibration); a resign_disabled_fraction share of the games never resigns, and after every generation the
        # threshold becomes the one at which a resign_false_positive share of those games' non-losing players would have
        # resigned.
        self.resign = False
        self.resign_false_positive = 0.05
        self.resign_disabled_fraction = 0.1
        self.resign_threshold = -1.0
        # Extension: playout cap randomization in self-play (KataGo; the reference runs every search with n_playouts_train).
        # With fast_playouts set, a full_search_fraction share of the searches is full; the others run fast_playouts
        # simulations without root noise, still choose the move, and their positions are no training examples.
        self.fast_playouts = None
        self.full_search_fraction = 0.25
        # Extension: forced playouts and policy target pruning in self-play (KataGo; the reference has neither).  With
        # forced_playouts = k (2.0 in the paper), every visited root child of a search with root noise gets at least
        # sqrt(k * P * N) visits, and the visits it got only from that floor are pruned from its policy target.
        self.forced_playouts = None
        # Extension: left-right reflection, the one symmetry of both games (AlphaGo Zero; the reference uses every position
        # as it is).  With reflect_evaluations, self-play evaluates a position mirrored (column c <-> cols-1-c) when a hash of
        # the engine seed and the position says so, and maps the policy back.  With reflect_minibatches, every sampled
        # training example is mirrored, board planes and policy target, when a hash of (optimisation step, row) says so.
        self.reflect_evaluations = False
        self.reflect_minibatches = False
        for k, v in overrides.items():
            if not hasattr(self, k):
                raise TypeError("unknown Trainer setting %r" % k)
            setattr(self, k, v)
        if "n_games_buffer" not in overrides:
            self.n_games_buffer = 4 * self.n_games_per_generation

        self.generation = 0
        self.buffer = []
        self.abuffer = None
        self.dbuffer = None
        self.state_shape, self.num_distinct_actions = game_shape(self.name_game)
        self.games_played = 0
        self.start_time = datetime.now().strftime("%Y-%m-%d-%H-%M-%S")
        if device is None:
            device = torch.device("cuda", torch.cuda.current_device()) if (self.use_gpu and torch.cuda.is_available()) \
                else torch.device("cpu")
        self.device = torch.device(device)
        self.current_net = Net(self.state_shape, self.num_distinct_actions, device=self.device)
        self.current_net.to(self.device)
        parallel.broadcast_weights(self.current_net, src=0, device=self.device)  # identical initial weights on every rank
        self.optimizer = torch.optim.Adam(self.current_net.parameters(), lr=self.lr, weight_decay=0.0001,
                                          capturable=bool(self.graph_step and self.device.type == "cuda"))
        self._step_graph = None
        self._gids = None
        self._perm = None
        self.criterion_value = nn.MSELoss()
        self.current_net.eval()
        self.last_generation_stats = {}

    # ------------------------------------------------------------------ optimisation (train.py:95-154)
    def _reflect_rows(self):
        """reflect_minibatches: the minibatch rows of this optimisation step (self.it) to mirror, bool [batch_size] (for
        the whole minibatch: ddp slices it like the sample ids); None when off."""
        return reflect_bits(self.it, self.batch_size) if self.reflect_minibatches else None

    def _host_perm(self):
        if self._perm is None:
            self._perm = reflect_actions(self.name_game)
        return self._perm

    def net_step_arrays(self, batch, first, pol, val):
        """net_step on the array form of the buffer (replay.ExampleBatch after remove_duplicates): same sampling call,
        same losses; the board planes are rebuilt for the sampled minibatch only."""
        self.current_net.zero_grad()
        sample_ids = np.random.randint(len(first), size=self.batch_size)
        boards, p = batch.boards(first[sample_ids]), pol[sample_ids]
        refl = self._reflect_rows()
        if refl is not None:
            boards[refl] = boards[refl][..., ::-1]
            p[refl] = p[refl][:, self._host_perm()]
        x = torch.from_numpy(boards).float().to(self.device)
        p_t, v_t = self.current_net(x)
        p_r = torch.tensor(p).float().to(self.device)
        v_r = torch.tensor(val[sample_ids]).float().to(self.device)
        loss_v = self.criterion_value(v_t, v_r.unsqueeze(1))
        loss_p = -torch.sum(p_r * torch.log(p_t)) / p_r.size()[0]
        (loss_v + loss_p).backward()
        self.optimizer.step()
        self.it += 1
        return loss_p, loss_v

    def net_step_device(self, replay, first, pol, val):
        """net_step (train.py:95-130) on the device replay buffer: the same `np.random.randint` sampling call, the board planes
        of the sampled examples come from the az_observations gather kernel, targets are gathered on the device; with
        `ddp` every rank trains on its slice of the minibatch and the gradients are averaged over NCCL."""
        sample_ids = np.random.randint(int(first.numel()), size=self.batch_size)
        refl = self._reflect_rows()
        rank, world = parallel.rank_world()
        if self.graph_step and not (self.ddp and world > 1):
            return self._net_step_graphed(replay, first, pol, val, sample_ids, refl)
        self.current_net.zero_grad()
        if self.ddp and world > 1:
            sample_ids = sample_ids[rank::world]
            refl = None if refl is None else refl[rank::world]
        ids = torch.from_numpy(sample_ids).to(self.device)
        refl = None if refl is None else torch.from_numpy(refl).to(self.device)
        x = replay.boards(first[ids], refl)
        p_t, v_t = self.current_net(x)
        p_r = pol[ids].float()
        if refl is not None:
            p_r = torch.where(refl[:, None], p_r[:, replay.reflect_perm], p_r)
        v_r = val[ids].float()
        loss_v = self.criterion_value(v_t, v_r.unsqueeze(1))
        loss_p = -torch.sum(p_r * torch.log(p_t)) / p_r.size()[0]
        (loss_v + loss_p).backward()
        if self.ddp and world > 1:
            parallel.allreduce_gradients(self.current_net, self.device)
        self.optimizer.step()
        self.it += 1
        return loss_p, loss_v

    def _net_step_graphed(self, replay, first, pol, val, sample_ids, refl=None):
        """The device step as ONE CUDA-graph replay: minibatch gather (az_observations kernel + two index_selects from the
        de-duplicated targets), forward, MSE + cross-entropy, backward, Adam.  Per step the host only draws the sample ids
        (the reference's np.random.randint call) and copies 2 KB of indices to the device; the graph is re-captured
        when a new generation brings new target tensors.  refl (reflect_minibatches): the rows to mirror travel as bit 32
        of the same indices (the ids are below 2^31)."""
        dev = self.device
        if getattr(self, "_gids", None) is None:
            self._gids = torch.zeros(self.batch_size, dtype=torch.int64, device=dev)
            self._graph_key = None
            self._graph_warm = False
        gids = np.ascontiguousarray(sample_ids, dtype=np.int64)
        perm = None
        if refl is not None:
            gids = gids | (refl.astype(np.int64) << 32)
            perm = replay.reflect_perm         # (built here: no host-to-device copy inside the capture)
        # (pageable source: the driver stages the 2 KB before returning, so the next step may overwrite sample_ids)
        self._gids.copy_(torch.from_numpy(gids))

        def step():
            ids = self._gids
            rows = None
            if perm is not None:
                rows = (ids >> 32).to(torch.uint8)
                ids = ids & 0xFFFFFFFF
            x = replay.boards(first[ids], rows)
            p_r = pol[ids].float()
            if perm is not None:
                p_r = torch.where(rows[:, None].bool(), p_r[:, perm], p_r)
            v_r = val[ids].float().unsqueeze(1)
            self.optimizer.zero_grad(set_to_none=False)
            p_t, v_t = self.current_net(x)
            loss_v = self.criterion_value(v_t, v_r)
            loss_p = -torch.sum(p_r * torch.log(p_t)) / p_r.size()[0]
            (loss_v + loss_p).backward()
            self.optimizer.step()
            return loss_p.detach(), loss_v.detach()

        if not self._graph_warm:
            # the very first step runs eagerly on a side stream (cuDNN / allocator warm-up, gradient and Adam state
            # allocation); it is a real optimisation step
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                self.optimizer.zero_grad(set_to_none=False)
                out = step()
            torch.cuda.current_stream(dev).wait_stream(side)
            self._graph_warm = True
            self.it += 1
            return out[0].clone(), out[1].clone()
        key = (first.data_ptr(), pol.data_ptr(), val.data_ptr(), int(first.numel()), replay.bb.data_ptr(),
               perm is not None)
        if key != self._graph_key:
            torch.cuda.current_stream(dev).synchronize()
            self._step_graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self._step_graph):
                self._glp, self._glv = step()
            self._graph_key = key          # (capture does not execute: the replay below performs this step)
        self._step_graph.replay()
        self.it += 1
        return self._glp.clone(), self._glv.clone()

    def net_step(self, flattened_buffer):
        self.current_net.zero_grad()
        sample_ids = np.random.randint(len(flattened_buffer), size=self.batch_size)
        boards = [flattened_buffer[i][1] for i in sample_ids]
        pol = [flattened_buffer[i][2] for i in sample_ids]
        val = [flattened_buffer[i][3] for i in sample_ids]
        refl = self._reflect_rows()
        if refl is not None:
            # an empty policy is replaced below by the network's output, which already refers to the mirrored input
            perm = self._host_perm()
            boards = [b[..., ::-1] if r else b for b, r in zip(boards, refl)]
            pol = [np.asarray(item)[perm].tolist() if (r and item) else item for item, r in zip(pol, refl)]
        x = torch.from_numpy(np.array(boards)).float().to(self.device)
        p_t, v_t = self.current_net(x)
        pol = [item if item else p_t[i, :].to("cpu").tolist() for i, item in enumerate(pol)]
        p_r = torch.tensor(np.array(pol)).float().to(self.device)
        v_r = torch.tensor(np.array(val)).float().to(self.device)
        loss_v = self.criterion_value(v_t, v_r.unsqueeze(1))
        loss_p = -torch.sum(p_r * torch.log(p_t)) / p_r.size()[0]
        (loss_v + loss_p).backward()
        self.optimizer.step()
        self.it += 1
        return loss_p, loss_v

    def train_network(self):
        rank, world = parallel.rank_world()
        losses = []
        if rank == 0 or (self.ddp and self.device_training):
            self.current_net.train()
            if self.device_training:
                first, pol, val = self.dbuffer.remove_duplicates()
            elif self.array_buffer:
                first, pol, val = self.abuffer.remove_duplicates()
            else:
                flat = self.remove_duplicates([sample for game in self.buffer for sample in game])
            run_p = run_v = 0
            for i in range(self.n_batches_per_generation):
                if self.device_training:
                    loss_p, loss_v = self.net_step_device(self.dbuffer, first, pol, val)
                elif self.array_buffer:
                    loss_p, loss_v = self.net_step_arrays(self.abuffer, first, pol, val)
                else:
                    loss_p, loss_v = self.net_step(flat)
                run_p += loss_p
                run_v += loss_v
                if i % 100 == 99:
                    logger.info("Batch: " + str(i) + "Loss policy: " + str(run_p / 100.) + "Loss value: " + str(run_v / 100.))
                    losses.append((float(run_p) / 100., float(run_v) / 100.))
                    run_p = run_v = 0
            self.current_net.eval()
        if world > 1:
            # rank 0's weights to everyone; under ddp the parameters are already equal and this only re-synchronises the
            # BatchNorm running statistics, which every rank accumulated from its own slice of the minibatches
            parallel.broadcast_weights(self.current_net, src=0, device=self.device)
        return losses

    @staticmethod
    def remove_duplicates(flattened_buffer):
        """Merge examples with the same information-state key: policies and values are averaged (train.py:156-201).
        Like the reference, the FIRST example of a key is the accumulator object and is mutated in place."""
        start = time.time()
        merged, n_val, n_pol = {}, {}, {}
        for item in flattened_buffer:
            key = item[0]
            acc = merged.get(key)
            if acc is None:
                merged[key], n_val[key], n_pol[key] = item, 1, 1
                continue
            if item[2] and acc[2]:
                acc[2] = [sum(pair) for pair in zip(acc[2], item[2])]
                n_pol[key] += 1
            elif item[2]:
                acc[2] = item[2]
            acc[3] += item[3]
            n_val[key] += 1
        for key, acc in merged.items():
            if acc[2]:
                acc[2] = [x / n_pol[key] for x in acc[2]]
            acc[3] = acc[3] / n_val[key]
        out = list(merged.values())
        logger.info("Removing duplicates: %d -> %d samples in %.2f s" % (len(flattened_buffer), len(out), time.time() - start))
        return out

    # ------------------------------------------------------------------ generation (train.py:203-236)
    def generate_examples(self, n_games, **engine_kwargs):
        start = time.time()
        if self.resign:
            engine_kwargs = dict(engine_kwargs, resign_threshold=self.resign_threshold,
                                 resign_disabled_fraction=self.resign_disabled_fraction,
                                 resign_false_positive=self.resign_false_positive)
        if self.fast_playouts is not None:
            engine_kwargs = dict(engine_kwargs, fast_playouts=self.fast_playouts,
                                 full_search_fraction=self.full_search_fraction)
        if self.forced_playouts is not None:
            engine_kwargs = dict(engine_kwargs, forced_playouts=self.forced_playouts)
        if self.reflect_evaluations:
            engine_kwargs = dict(engine_kwargs, reflect_evaluations=True)
        generator = ExampleGenerator(self.current_net, self.name_game, self.device,
                                     n_playouts=self.n_playouts_train, temperature=self.temperature,
                                     dirichlet_ratio=self.dirichlet_ratio, c_puct=self.uct_train, backup=self.backup,
                                     tree_strap=self.tree_strap, n_pools=self.n_pools, n_processes=self.n_processes,
                                     rank0_only=not (self.ddp and self.device_training), **engine_kwargs)
        if self.device_training:
            from .device_replay import DeviceReplay
            new = generator.generate_batch(n_games)
            n_new = new.n_games
            if self.dbuffer is None:
                self.dbuffer = DeviceReplay(self.name_game, self.device)
            self.dbuffer.append(new)
        elif self.array_buffer:
            from .replay import ExampleBatch
            new = generator.generate_batch(n_games)
            n_new = new.n_games
            self.abuffer = new if self.abuffer is None else ExampleBatch.concat([self.abuffer, new])
        else:
            games = generator.generate_examples(n_games)
            n_new = len(games)
            for examples in games:
                self.buffer.append(examples)
        self.games_played += self.n_games_per_generation
        self.last_generation_stats = dict(generator.last_stats, seconds=time.time() - start, games=n_new)
        if self.resign:
            self.last_generation_stats["resign_threshold"] = self.resign_threshold
            self.resign_threshold = generator.last_stats["resign_threshold_suggested"]
            logger.info("Resignation: %d resigned, %d calibration games, %d false positives; threshold %.4f -> %.4f" % (
                generator.last_stats.get("resigns", 0), generator.last_stats.get("resign_samples", 0),
                generator.last_stats.get("resign_false", 0), self.last_generation_stats["resign_threshold"],
                self.resign_threshold))
        logger.info("Finished Generating Data. Took: " + str(time.time() - start) + " seconds")
        self.update_buffer_size()
        if self.device_training:
            self.dbuffer.keep_last_games(self.n_games_buffer)
        elif self.array_buffer:
            self.abuffer = self.abuffer.last_games(self.n_games_buffer)
        elif len(self.buffer) > self.n_games_buffer:
            del self.buffer[:len(self.buffer) - self.n_games_buffer]

    def update_buffer_size(self):
        if self.generation % 2 == 0 and self.n_games_buffer < self.n_games_buffer_max:
            self.n_games_buffer += self.n_games_per_generation

    def test_agent(self):
        """train.py:238-270: the network alone against a uniform-random player, then -- through
        ExampleGenerator.generate_tests -- the network alone against the 100- and 200-simulation MCTS bot and the full
        AlphaZero bot against the 200-simulation MCTS bot, n_tests game pairs each, all batched on the GPU (evaluate.py;
        the MCTS bot is the device UCT + random-rollout bot described there)."""
        from . import evaluate
        if parallel.rank_world()[0] != 0:
            return None
        if self.device.type != "cuda":
            logger.info("test_agent needs the GPU engine; skipped on %s" % self.device)
            return None
        start = time.time()
        logger.info("Testing...")
        generator = ExampleGenerator(self.current_net, self.name_game, self.device, is_test=True,
                                     temperature=self.temperature, dirichlet_ratio=self.dirichlet_ratio,
                                     c_puct=self.uct_test, n_pools=self.n_pools, n_processes=self.n_processes)
        out = {}
        s1, s2 = evaluate.net_vs_random(self.current_net, self.name_game, self.n_tests, device=self.device)
        out["net_vs_random"] = (s1 + s2) / 2
        logger.info("Average score vs random (net only):" + str(out["net_vs_random"]))
        out["net_vs_mcts100"] = generator.generate_tests(self.n_tests, "test_net_vs_mcts", 100)
        logger.info("Average score vs mcts100 (net only):" + str(out["net_vs_mcts100"]))
        out["zero_vs_mcts200"] = generator.generate_tests(self.n_tests, "test_zero_vs_mcts", 200)
        logger.info("Average score vs mcts200:" + str(out["zero_vs_mcts200"]))
        out["net_vs_mcts200"] = generator.generate_tests(self.n_tests, "test_net_vs_mcts", 200)
        logger.info("Average score vs mcts200 (net only):" + str(out["net_vs_mcts200"]))
        logger.info("Testing took: " + str(time.time() - start) + "seconds")
        return out

    def run(self, **engine_kwargs):
        """Main loop (train.py:272-293): generate -> train -> (save)."""
        import os
        rank, _ = parallel.rank_world()
        self.test_agent()                                       # train.py:275 (before the loop)
        while self.generation < self.n_generations:
            self.generation += 1
            self.generate_examples(self.n_games_per_generation, **engine_kwargs)
            self.train_network()
            if self.save and rank == 0 and self.generation % self.save_n_gens == 0:     # train.py:285-288
                os.makedirs(self.model_path, exist_ok=True)
                torch.save(self.current_net.state_dict(), self.model_path + self.name_run + str(self.generation) + ".pth")
            if self.generation % self.test_n_gens == 0:         # train.py:290-291
                self.test_agent()
