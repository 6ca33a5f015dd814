"""Pure-Python restatement of the reference's self-play path (CPU ORACLE -- test infrastructure only).

This is the CPU baseline bench.py times (the reference itself is not part of this repository).  It restates, with flat parallel lists instead of linked Node objects:

    PortMCTS          <- mcts.py:92-203   (search / playout / expand_root_dirichlet / update_root)
      ._pick          <- mcts.py:38-52,68-80  Node.select + get_value (PUCT and use_puct=False branches)
      ._grow          <- mcts.py:54-66    Node.expand
      ._credit        <- mcts.py:82-89    Node.update_recursive
    rollout_policy    <- mcts.py:205-223  MCTS.random_rollout
    strip_illegal     <- alphazerobot.py:7-18   remove_illegal_actions
    PortBot.step      <- alphazerobot.py:42-93
    selfplay_game     <- game_utils.py:148-206  play_game_self (all four `backup` targets)
    board_planes      <- network.py:9-18  state_to_board
    PortGenerator     <- examplegenerator.py:17-22,39-175  worker pool + batching evaluator process

The arithmetic (operation order, Python-float fp64, first-max tie-breaking, global numpy RNG call
order) is kept identical so results are bit-equal to the reference; tests/test_oracle_golden.py pins that against
the reference's recorded outputs (tests/golden/).
"""
import math
import os
import time

import numpy as np


class PortMCTS:
    def __init__(self, policy_fn, num_distinct_actions, c_puct=2.5, n_playouts=100, use_dirichlet=True,
                 dirichlet_ratio=0.25, use_puct=True, **_ignored):
        self.use_puct = use_puct
        self.policy_fn = policy_fn
        self.num_distinct_actions = num_distinct_actions
        self.c_puct = c_puct
        self.n_playouts = n_playouts
        self.use_dirichlet = use_dirichlet
        self.dirichlet_ratio = dirichlet_ratio
        self.stats = {"sims": 0, "depth": 0, "children": 0, "expand": 0, "legal": 0, "terminal": 0, "root_evals": 0}
        # The reference stores use_puct per Node, children inherit it from their parent (mcts.py:64) and the first root is
        # built WITHOUT the flag (mcts.py:122): a tree scores with the UCT formula only if its root was created by
        # update_root on a leaf root (mcts.py:199-200).  One flag per tree reproduces that.
        self.fresh(uct=False)

    # flat storage: index 0.. ; kids[i] is None (leaf) or (actions, ids) in insertion (= legal) order
    def fresh(self, uct):
        self.tree_uct = uct
        self.visits = [0]
        self.mean = [0]
        self.prior = [0.0]
        self.up = [-1]
        self.kids = [None]
        self.root = 0

    def _grow(self, node, prior_ps, legal_actions):
        if self.kids[node] is None:
            acts, ids = [], []
            self.kids[node] = (acts, ids)
        else:
            acts, ids = self.kids[node]
        for a in legal_actions:
            if a in acts:
                self.prior[ids[acts.index(a)]] = prior_ps[a]
            else:
                self.visits.append(0)
                self.mean.append(0)
                self.prior.append(prior_ps[a])
                self.up.append(node)
                self.kids.append(None)
                acts.append(a)
                ids.append(len(self.visits) - 1)
        if not acts:
            self.kids[node] = None

    def _pick(self, node):
        acts, ids = self.kids[node]
        root_term = math.sqrt(self.visits[node])
        best_k, best_v = 0, None
        for k, j in enumerate(ids):
            if not self.tree_uct:
                v = self.mean[j] + self.c_puct * self.prior[j] * root_term / (self.visits[j] + 1)
            elif self.visits[j] == 0:      # mcts.py:80: unvisited children first, in insertion order
                v = float("inf")
            else:
                v = self.mean[j] + self.c_puct * self.prior[j] * math.sqrt(math.log(self.visits[node]) / self.visits[j])
            if best_v is None or v > best_v:
                best_k, best_v = k, v
        return ids[best_k], acts[best_k]

    def _credit(self, node, value):
        while node >= 0:
            n = self.visits[node]
            self.mean[node] = (n * self.mean[node] + value) / (n + 1)
            self.visits[node] = n + 1
            value = -value
            node = self.up[node]

    def playout(self, state):
        node = self.root
        mover = state.current_player()
        depth = 0
        while self.kids[node] is not None and not state.is_terminal():
            mover = state.current_player()
            self.stats["children"] += len(self.kids[node][1])
            node, action = self._pick(node)
            state.apply_action(action)
            depth += 1
        if not state.is_terminal():
            prior_ps, leaf_value = self.policy_fn(state)
            legal = state.legal_actions(state.current_player())
            self._grow(node, prior_ps, legal)
            self.stats["expand"] += 1
            self.stats["legal"] += len(legal)
        else:
            leaf_value = -state.player_return(mover)
            self.stats["terminal"] += 1
        self.stats["sims"] += 1
        self.stats["depth"] += depth
        self._credit(node, -leaf_value)

    def root_child_visits(self):
        out = [0] * self.num_distinct_actions
        if self.kids[self.root] is not None:
            for a, j in zip(*self.kids[self.root]):
                out[a] = self.visits[j]
        return out

    def get_normalized_visit_counts(self):
        visits = self.root_child_visits()
        total = sum(visits)
        return [float(v) / total for v in visits]

    def expand_root_dirichlet(self, state):
        prior_ps, _ = self.policy_fn(state)
        legal = state.legal_actions(state.current_player())
        prior_ps = (1.0 - self.dirichlet_ratio) * np.array(prior_ps)
        eta = list(np.random.dirichlet(0.3 * np.ones(len(legal))))
        for i, a in enumerate(legal):
            prior_ps[a] = prior_ps[a] + 0.25 * eta[i]
        self._grow(self.root, prior_ps, legal)
        self.stats["root_evals"] += 1

    def search(self, state):
        if self.use_dirichlet:
            self.expand_root_dirichlet(state)
        for _ in range(self.n_playouts):
            self.playout(state.clone())
        return self.get_normalized_visit_counts()

    def update_root(self, action):
        if self.kids[self.root] is None:
            self.fresh(uct=not self.use_puct)
            return
        acts, ids = self.kids[self.root]
        self.root = ids[acts.index(action)]  # ValueError here == the reference's KeyError
        self.up[self.root] = -1

    # --- value targets, game_utils.py:172-194 ---
    def target_soft_z(self):
        return -self.mean[self.root]

    def target_a0c(self):
        _, ids = self.kids[self.root]
        return max([self.mean[j] if self.visits[j] > 0 else -99.0 for j in ids])

    def target_off_policy(self):
        node, sign, value = self.root, 1.0, None
        while self.kids[node] is not None:
            value = self.mean[node]
            _, ids = self.kids[node]
            best, best_v = ids[0], None
            for j in ids:
                v = self.visits[j] + self.prior[j] if self.visits[j] > 0 else -99.0
                if best_v is None or v > best_v:
                    best, best_v = j, v
            node = best
            sign *= -1.0
        if self.visits[node] > 0:
            value = self.mean[node]
            sign *= -1.0
        return value * sign


def rollout_policy(num_distinct_actions):
    """mcts.py:205-223 (MCTS.random_rollout) as a policy_fn: uniform priors, value = return of one random playout for the
    player to move; one np.random.choice per ply on the global numpy RNG."""
    def fn(state):
        work = state.clone()
        starter = work.current_player()
        while not work.is_terminal():
            work.apply_action(np.random.choice(work.legal_actions()))
        return np.ones(num_distinct_actions), work.player_return(starter)
    return fn


def strip_illegal(probs, legal_actions):
    keep = np.zeros(probs.shape, dtype=bool)
    keep[legal_actions] = True
    probs[~keep] = 0.0
    if np.sum(probs) > 1e-6:
        return probs / np.sum(probs)
    out = np.zeros(len(probs))
    out[legal_actions] = 1. / len(legal_actions)
    return out


class PortBot:
    def __init__(self, game, player, policy_fn, self_play=False, keep_search_tree=True, **kwargs):
        self.num_distinct_actions = game.num_distinct_actions()
        self.policy_fn = policy_fn
        self.kwargs = kwargs
        self.sample = self_play or bool(kwargs.get("use_probabilistic_actions"))
        self.uniform_random = bool(kwargs.get("use_random_actions", False))
        self.sample_plies = int(kwargs.get("num_probabilistic_actions", 1000))
        self.temperature = float(kwargs.get("temperature", 1.0))
        self.self_play = self_play
        self.keep_search_tree = keep_search_tree
        self.mcts = PortMCTS(policy_fn, self.num_distinct_actions, **kwargs)

    def step(self, state):
        if self.keep_search_tree:
            hist = state.history()
            if self.self_play:
                if hist:
                    self.mcts.update_root(hist[-1])
            elif len(hist) >= 2:
                self.mcts.update_root(hist[-2])
                self.mcts.update_root(hist[-1])
        else:
            self.mcts = PortMCTS(self.policy_fn, self.num_distinct_actions, **self.kwargs)
        nvc = np.array(self.mcts.search(state))
        legal = state.legal_actions(state.current_player())
        nvc_legal = strip_illegal(nvc, legal)
        heated = nvc_legal ** (1. / self.temperature)
        probs = heated / sum(heated)
        n_moves = len(state.history())
        if self.uniform_random and n_moves < self.sample_plies:
            action = np.random.choice(legal)
        elif self.sample and n_moves < self.sample_plies:
            action = np.random.choice(len(probs), p=probs)
        else:
            action = np.argmax(probs)
        return [(a, nvc_legal[a]) for a in legal], action


def board_planes(state, state_shape):
    c, h, w = state_shape
    out = np.zeros((c + 1, h, w)) + state.current_player()
    out[:-1] = np.asarray(state.information_state_as_normalized_vector()).reshape(state_shape)
    out[-1] = np.zeros((1, h, w)) + state.current_player()
    return out


def selfplay_game(policy_fn, game_name, load_game, stats=None, **kwargs):
    """game_utils.py:148-206.  `load_game` is the pyspiel-shaped loader (oracle.pyspiel_shim.load_game)."""
    game = load_game(game_name)
    state = game.new_initial_state()
    shape = game.information_state_normalized_vector_shape()
    n_actions = game.num_distinct_actions()
    bot = PortBot(game, 0, policy_fn, self_play=True, **kwargs)
    backup = str(kwargs.get("backup", "on-policy"))
    max_plies = int(kwargs.get("max_plies", 0))  # port-only knob: bounded sample for the CPU baseline timing
    examples = []
    while not state.is_terminal():
        if max_plies and len(examples) >= max_plies:
            break
        policy, action = bot.step(state)
        sparse = dict(policy)
        dense = [sparse.get(i, 0.0) for i in range(n_actions)]
        if backup == "on-policy":
            examples.append([state.information_state(), board_planes(state, shape), dense, None])
        if backup == "soft-Z":
            examples.append([state.information_state(), board_planes(state, shape), dense, bot.mcts.target_soft_z()])
        if backup == "A0C":
            examples.append([state.information_state(), board_planes(state, shape), dense, bot.mcts.target_a0c()])
        if backup == "off-policy":
            examples.append([state.information_state(), board_planes(state, shape), dense,
                             bot.mcts.target_off_policy()])
        state.apply_action(action)
    if backup == "on-policy":
        reward = state.returns()[0]
        for ex in examples:
            ex[3] = reward
            reward *= -1
    if stats is not None:
        for k, v in bot.mcts.stats.items():
            stats[k] = stats.get(k, 0) + v
        stats["plies"] = stats.get("plies", 0) + len(examples)
    return examples


# ---------------------------------------------------------------------------------------------
# Multi-process generator (examplegenerator.py): one OS process per game worker, one evaluator
# process that batches whatever boards are ready into a single forward.
# ---------------------------------------------------------------------------------------------

class PipeEvaluator:  # examplegenerator.py:39-54
    def __init__(self, conn, shape):
        self.conn = conn
        self.shape = shape

    def __call__(self, state):
        self.conn.send(board_planes(state, self.shape))
        pi, vi = self.conn.recv()
        return pi, float(vi[0])


def _worker(job):  # examplegenerator.py:17-22
    conn, game_name, kwargs = job
    from . import pyspiel_shim
    game = pyspiel_shim.load_game(game_name)
    stats = {}
    t0 = time.time()
    ex = selfplay_game(PipeEvaluator(conn, game.information_state_normalized_vector_shape()), game_name,
                       pyspiel_shim.load_game, stats=stats, **kwargs)
    stats["t_start"], stats["t_end"] = t0, time.time()
    return ex, stats


def _serve(net, conns, device):  # examplegenerator.py:57-77 (forward with autograd enabled, as shipped)
    import torch
    torch.set_num_threads(1)
    net.to(device)
    while True:
        ready, batch = [], []
        for c in conns:
            if c.poll():
                ready.append(c)
                batch.append(c.recv())
        if batch:
            x = torch.from_numpy(np.array(batch)).float().to(device)
            p, v = net.forward(x)
            p, v = p.tolist(), v.tolist()
            for i, c in enumerate(ready):
                c.send((p[i], v[i]))


def _seed_worker():
    np.random.seed()
    try:
        import torch
        torch.set_num_threads(1)
    except Exception:
        pass


class PortGenerator:
    """examplegenerator.py:80-175 on the CPU (device argument kept for signature parity)."""

    def __init__(self, net, game_name, device="cpu", n_pools=1, n_processes=1, **kwargs):
        import copy
        self.net = copy.deepcopy(net).to("cpu")
        self.game_name = game_name
        self.device = device
        self.n_pools = n_pools
        self.n_processes = n_processes
        self.kwargs = kwargs
        self.last_stats = {}

    def generate_examples(self, n_games):
        import copy
        from torch import multiprocessing as mp
        ctx = mp.get_context("spawn")
        pools = []
        per_pool = int(n_games / self.n_pools)
        for _ in range(self.n_pools):
            pairs = [ctx.Pipe() for _ in range(per_pool)]
            pool = ctx.Pool(processes=self.n_processes, initializer=_seed_worker)
            server = ctx.Process(target=_serve, args=(copy.deepcopy(self.net), [p for p, _ in pairs], "cpu"))
            server.start()
            res = pool.map_async(_worker, [(c, self.game_name, self.kwargs) for _, c in pairs])
            pools.append((pool, server, res))
        games, stats = [], {}
        for pool, server, res in pools:
            for ex, st in res.get():
                games.append(ex)
                for k, v in st.items():
                    if k == "t_start":
                        stats[k] = min(stats.get(k, v), v)
                    elif k == "t_end":
                        stats[k] = max(stats.get(k, v), v)
                    else:
                        stats[k] = stats.get(k, 0) + v
            pool.close()
            pool.join()
            server.terminate()
            server.join()
        self.last_stats = stats
        return games


def dedupe_examples(flat):
    """train.py:156-201 remove_duplicates, restated: per key, element-wise policy sum / count and value sum / count;
    the first example of each key is the accumulator and is mutated in place (as in the reference)."""
    first, vcount, pcount = {}, {}, {}
    for ex in flat:
        k = ex[0]
        if k not in first:
            first[k] = ex
            vcount[k] = 1
            pcount[k] = 1
        else:
            tgt = first[k]
            if ex[2] and tgt[2]:
                tgt[2] = [sum(x) for x in zip(tgt[2], ex[2])]
                pcount[k] += 1
            elif ex[2]:
                tgt[2] = ex[2]
            tgt[3] += ex[3]
            vcount[k] += 1
    for k in first:
        if first[k][2]:
            first[k][2] = [x / pcount[k] for x in first[k][2]]
        first[k][3] = first[k][3] / vcount[k]
    return list(first.values())


def train_step(net, optimizer, flat, batch_size, device="cpu"):
    """train.py:95-130 net_step restated for the fp32 reference net: returns (loss_policy, loss_value)."""
    import torch
    net.zero_grad()
    ids = np.random.randint(len(flat), size=batch_size)
    x = torch.from_numpy(np.array([flat[i][1] for i in ids])).float().to(device)
    p_t, v_t = net(x)
    p_r = [flat[i][2] if flat[i][2] else p_t[j, :].to("cpu").tolist() for j, i in enumerate(ids)]
    p_r = torch.tensor(np.array(p_r)).float().to(device)
    v_r = torch.tensor(np.array([flat[i][3] for i in ids])).float().to(device)
    loss_v = torch.nn.MSELoss()(v_t, v_r.unsqueeze(1))
    loss_p = -torch.sum(p_r * torch.log(p_t)) / p_r.size()[0]
    (loss_v + loss_p).backward()
    optimizer.step()
    return loss_p, loss_v


def time_selfplay(net, game_name, n_games, n_processes, **kwargs):
    """Wall-clock the multi-process generator; returns dict(sims_per_s, games_per_s, plies, cores, seconds)."""
    gen = PortGenerator(net, game_name, "cpu", n_pools=1, n_processes=n_processes, **kwargs)
    games = gen.generate_examples(n_games)
    st = gen.last_stats
    dt = st["t_end"] - st["t_start"]  # first worker start .. last worker end (process spawn / imports excluded)
    plies = sum(len(g) for g in games)
    sims = st.get("sims", plies * int(kwargs.get("n_playouts", 100)))
    return {"sims_per_s": sims / dt, "games_per_s": len(games) / dt, "plies": plies, "seconds": dt, "sims": sims,
            "cores": n_processes + 1, "host_cpus": os.cpu_count(), "n_games": len(games)}
