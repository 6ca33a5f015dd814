"""Records tests/golden/reference_crosscheck.json: what the reference's own Python (mcts.py, alphazerobot.py,
game_utils.py, train.py) returns in the cases of the reference cross-checks in tests/test_oracle_golden.py and
tests/test_trainer.py (self-play games, a 300-playout search, the random-rollout evaluator, use_puct=False trees,
NeuralNetBot / play_game and Trainer.remove_duplicates).

The reference is not part of this repository.  The vectors are recorded from the oracle's restatement of it
(oracle/ref_port.py) and, for NeuralNetBot / play_game, which the port does not restate, from this package's host code:
in exactly these cases both returned what the unmodified reference returned, bit for bit.  Given a checkout of the
reference, the script checks that again before it writes anything:

    python tests/golden/make_golden_crosscheck.py [REFERENCE_CHECKOUT]
"""
import copy
import ctypes as C
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import cbind, pyspiel_shim, ref_port  # noqa: E402

L = cbind.lib()
GAMES = ["connect_four", "breakthrough(rows=6,columns=6)"]


def hash_policy(seed):
    def fn(st):
        A = st.get_game().num_distinct_actions()
        pri = (C.c_double * A)()
        v = C.c_double()
        L.oz_synth_eval(C.byref(st.raw()), 1, seed, 2 if A == 7 else 4, pri, C.byref(v))
        return list(pri), v.value
    return fn


def fake_buffer(rng, n=300, n_keys=60, A=7):
    """The example buffer of tests/test_trainer.py (same RNG calls)."""
    flat = []
    for _ in range(n):
        k = int(rng.randint(n_keys))
        pol = rng.dirichlet(np.ones(A)).tolist() if rng.rand() > 0.1 else []
        flat.append([str(k), rng.rand(4, 6, 7), pol, float(rng.choice([-1.0, 0.0, 1.0]))])
    return flat


def selfplay(play_game_self):
    """play_game_self(hash policy 123, 25 playouts) under np.random.seed(11), both games, on- and off-policy targets."""
    out = []
    for game in GAMES:
        for backup in ["on-policy", "off-policy"]:
            np.random.seed(11)
            ex = play_game_self(hash_policy(123), game, backup)
            boards = [np.asarray(e[1]) for e in ex]
            assert all(np.array_equal(b, b.astype(np.int64)) for b in boards)  # 0/1 planes: stored as integers
            out.append({"game": game, "backup": backup, "keys": [e[0] for e in ex],
                        "boards": [b.astype(np.int64).ravel().tolist() for b in boards],
                        "policies": [[[i, float(p)] for i, p in enumerate(e[2]) if p != 0.0] for e in ex],
                        "values": [float(e[3]) for e in ex]})
    return out


def search300(new_mcts):
    """One 300-playout search of the Connect Four start position, hash policy 123, no root noise."""
    s = pyspiel_shim.load_game("connect_four").new_initial_state()
    counts, root_q = new_mcts(hash_policy(123), s)
    return {"counts": [int(c) for c in counts], "root_q": float(root_q)}


def rollouts(random_rollout, rollout_search):
    """The random-rollout evaluator on six positions per game (priors, value, next draw of the numpy RNG), then a
    40-playout search driven by it under np.random.seed(5)."""
    out = []
    for game in GAMES:
        g = pyspiel_shim.load_game(game)
        A = g.num_distinct_actions()
        s = g.new_initial_state()
        evals = []
        for ply in range(6):
            np.random.seed(100 + ply)
            pri, v = random_rollout(A)(s)
            evals.append({"priors": [float(p) for p in pri], "value": float(v), "next_draw": np.random.random_sample()})
            s.apply_action(s.legal_actions()[ply % len(s.legal_actions())])
        np.random.seed(5)
        visits = rollout_search(A, g.new_initial_state())
        out.append({"game": game, "evals": evals, "search": [float(x) for x in visits]})
    return out


def uct_trees(new_uct_mcts):
    """use_puct=False, 80 playouts, hash policy 31: three moves per tree, with and without root noise, from a fresh tree and
    from one whose root came from update_root on a leaf root."""
    out = []
    for game in GAMES:
        g = pyspiel_shim.load_game(game)
        A = g.num_distinct_actions()
        for dirichlet in (False, True):
            for leaf_update_first in (False, True):
                m = new_uct_mcts(hash_policy(31), A, dirichlet)
                s = g.new_initial_state()
                if leaf_update_first:
                    first = s.legal_actions()[1]
                    s.apply_action(first)
                    m.update_root(first)
                moves = []
                for move in range(3):
                    np.random.seed(70 + move)
                    counts, root_q = m.search_root(s)
                    moves.append({"counts": [float(c) for c in counts], "root_q": float(root_q)})
                    act = int(np.argmax(counts))
                    m.update_root(act)
                    s.apply_action(act)
                out.append({"game": game, "dirichlet": dirichlet, "leaf_update_first": leaf_update_first, "moves": moves})
    return out


def netbot_games(bot_module, game_utils_module):
    """NeuralNetBot (hash policies 3 and 4): five steps from the start, then one play_game."""
    out = []
    for game in GAMES:
        g = pyspiel_shim.load_game(game)
        fa, fb = hash_policy(3), hash_policy(4)
        s = g.new_initial_state()
        steps = []
        for _ in range(5):
            pol, act = bot_module.NeuralNetBot(g, 0, fa).step(s)
            steps.append({"policy": [[int(a), float(p)] for a, p in pol], "action": int(act)})
            s.apply_action(int(act))
        result = game_utils_module.play_game(g, bot_module.NeuralNetBot(g, 0, fa), bot_module.NeuralNetBot(g, 1, fb))
        out.append({"game": game, "steps": steps, "play_game": float(result)})
    return out


def remove_duplicates(fn):
    """remove_duplicates on the buffer of tests/test_trainer.py (RandomState(0))."""
    merged = fn(copy.deepcopy(fake_buffer(np.random.RandomState(0))))
    return {"keys": [e[0] for e in merged], "policies": [[float(p) for p in e[2]] for e in merged],
            "values": [float(e[3]) for e in merged]}


class PortUCT:
    def __init__(self, fn, A, dirichlet):
        self.m = ref_port.PortMCTS(fn, A, n_playouts=80, use_dirichlet=dirichlet, use_puct=False)

    def update_root(self, a):
        self.m.update_root(a)

    def search_root(self, s):
        counts = self.m.search(s)
        return counts, self.m.mean[self.m.root]


def port_search300(fn, s):
    m = ref_port.PortMCTS(fn, 7, use_dirichlet=False, n_playouts=300)
    m.search(s)
    return m.root_child_visits(), m.mean[m.root]


def port_rollout_search(A, s):
    return ref_port.PortMCTS(ref_port.rollout_policy(A), A, n_playouts=40, use_dirichlet=False).search(s)


def record():
    from alphazero_openspiel_b200 import alphazerobot, game_utils
    return {
        "selfplay": selfplay(lambda fn, game, backup: ref_port.selfplay_game(fn, game, pyspiel_shim.load_game,
                                                                             n_playouts=25, backup=backup)),
        "search300": search300(port_search300),
        "rollouts": rollouts(ref_port.rollout_policy, port_rollout_search),
        "uct": uct_trees(PortUCT),
        "netbot": netbot_games(alphazerobot, game_utils),
        "remove_duplicates": remove_duplicates(ref_port.dedupe_examples),
    }


def from_reference(path):
    """The same cases, run by the reference itself."""
    pyspiel_shim.install()
    sys.path.insert(0, path)
    import alphazerobot as ref_bot
    import game_utils as ref_gu
    import mcts as ref_mcts
    import train as ref_train

    def search300_ref(fn, s):
        m = ref_mcts.MCTS(fn, 7, use_dirichlet=False, n_playouts=300)
        m.search(s)
        return [m.root.children[a].N for a in range(7)], m.root.Q

    def rollout_search_ref(A, s):
        m = ref_mcts.MCTS(None, A, n_playouts=40, use_dirichlet=False)
        m.policy_fn = m.random_rollout
        return m.search(s)

    class RefUCT:
        def __init__(self, fn, A, dirichlet):
            self.m = ref_mcts.MCTS(fn, A, n_playouts=80, use_dirichlet=dirichlet, use_puct=False)

        def update_root(self, a):
            self.m.update_root(a)

        def search_root(self, s):
            counts = self.m.search(s)
            return counts, self.m.root.Q

    return {
        "selfplay": selfplay(lambda fn, game, backup: ref_gu.play_game_self(fn, game, n_playouts=25, backup=backup)),
        "search300": search300(search300_ref),
        "rollouts": rollouts(lambda A: ref_mcts.MCTS(None, A, n_playouts=40, use_dirichlet=False).random_rollout,
                             rollout_search_ref),
        "uct": uct_trees(RefUCT),
        "netbot": netbot_games(ref_bot, ref_gu),
        "remove_duplicates": remove_duplicates(ref_train.Trainer.remove_duplicates),
    }


if __name__ == "__main__":
    gold = record()
    if len(sys.argv) > 1:
        ref = from_reference(os.path.abspath(sys.argv[1]))
        for k in gold:
            assert ref[k] == gold[k], "the reference differs from the recorded vectors in %r" % k
        print("the reference returns the recorded vectors")
    path = os.path.join(HERE, "reference_crosscheck.json")
    with open(path, "w") as f:
        json.dump(gold, f)
    print("wrote", path, os.path.getsize(path))
