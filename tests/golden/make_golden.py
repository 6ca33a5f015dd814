"""Generates tests/golden/reference_golden.json by running the UNMODIFIED reference (mcts.py, alphazerobot.py,
game_utils.py, network.py of a checkout of danielwillemsen/alphazero-openspiel) over oracle.pyspiel_shim.  The reference
is not part of this repository, so the vectors are committed; re-run this script to regenerate them:

    python tests/golden/make_golden.py REFERENCE_CHECKOUT
"""
import ctypes as C
import json
import os
import shutil
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import pyspiel_shim, cbind  # noqa: E402

pyspiel = pyspiel_shim.install()
REF = os.path.abspath(sys.argv[1])
sys.path.insert(0, REF)
import torch  # noqa: E402
import mcts as ref_mcts  # noqa: E402
import game_utils as ref_game_utils  # noqa: E402
import network as ref_network  # noqa: E402

L = cbind.lib()
FIXTURE_16 = [1, 2, 1, 2, 3, 4, 5, 6, 3, 4, 5, 3, 3, 1, 5, 2]  # test_mcts.py:12-27


def hash_eval(seed):
    def fn(st):
        A = st.get_game().num_distinct_actions()
        pri = (C.c_double * A)()
        v = C.c_double()
        L.oz_synth_eval(C.byref(st.raw()), 1, seed, 2 if A == 7 else 4, pri, C.byref(v))
        return list(pri), v.value
    return fn


def root_dump(m, A):
    kids = m.root.children
    return {"root_n": m.root.N, "root_q": float(m.root.Q),
            "n": [kids[a].N if a in kids else -1 for a in range(A)],
            "q": [float(kids[a].Q) if a in kids else 0.0 for a in range(A)],
            "p": [float(kids[a].P) if a in kids else 0.0 for a in range(A)]}


def known_answers():
    out = []
    g = pyspiel.load_game("connect_four")
    uni7 = lambda st: ([1 / 7] * 7, 0.0)  # noqa: E731
    for hist, n in [([], 100), ([], 800), (FIXTURE_16, 100), (FIXTURE_16, 800)]:
        s = g.new_initial_state()
        for a in hist:
            s.apply_action(a)
        m = ref_mcts.MCTS(uni7, 7, use_dirichlet=False, n_playouts=n)
        m.search(s)
        out.append({"game": "connect_four", "history": hist, "n_playouts": n, "evaluator": "uniform",
                    "use_dirichlet": False, **root_dump(m, 7)})
    # tree reuse: search, update_root(3), search (SURVEY C.3)
    s = g.new_initial_state()
    m = ref_mcts.MCTS(uni7, 7, use_dirichlet=False, n_playouts=100)
    m.search(s)
    m.update_root(3)
    s.apply_action(3)
    m.search(s)
    out.append({"game": "connect_four", "history": [3], "n_playouts": 100, "evaluator": "uniform",
                "use_dirichlet": False, "reuse_after": [[], 3], **root_dump(m, 7)})
    g6 = pyspiel.load_game("breakthrough(rows=6,columns=6)")
    m = ref_mcts.MCTS(lambda st: ([1 / 432] * 432, 0.0), 432, use_dirichlet=False, n_playouts=200)
    m.search(g6.new_initial_state())
    d = root_dump(m, 432)
    out.append({"game": "breakthrough(rows=6,columns=6)", "history": [], "n_playouts": 200, "evaluator": "uniform",
                "use_dirichlet": False, "root_n": d["root_n"], "root_q": d["root_q"],
                "legal": g6.new_initial_state().legal_actions(),
                "n_legal_order": [d["n"][a] for a in g6.new_initial_state().legal_actions()]})
    return out


def hash_searches():
    """Reference MCTS with the hash evaluator and injected (recorded) Dirichlet noise, incl. re-rooted second searches."""
    out = []
    for game, A in [("connect_four", 7), ("breakthrough(rows=6,columns=6)", 432), ("breakthrough", 768)]:
        g = pyspiel.load_game(game)
        rng = np.random.RandomState(7)
        for trial in range(6):
            s = g.new_initial_state()
            for _ in range(rng.randint(0, 14)):
                if s.is_terminal():
                    break
                s.apply_action(int(rng.choice(s.legal_actions())))
            if s.is_terminal():
                continue
            n_playouts = [50, 200, 800][trial % 3]
            np.random.seed(1000 + trial)
            m = ref_mcts.MCTS(hash_eval(77), A, n_playouts=n_playouts)
            case = {"game": game, "history": s.history(), "n_playouts": n_playouts, "evaluator": "hash77",
                    "searches": []}
            for rep in range(2):
                st = np.random.get_state()
                noise = np.random.dirichlet(0.3 * np.ones(len(s.legal_actions())))
                np.random.set_state(st)
                m.search(s)
                kids = m.root.children
                legal = s.legal_actions()
                case["searches"].append({"noise": [float(x) for x in noise], "legal": legal, "root_n": m.root.N,
                                         "root_q": float(m.root.Q), "n": [kids[a].N for a in legal],
                                         "q": [float(kids[a].Q) for a in legal],
                                         "p": [float(kids[a].P) for a in legal]})
                best = legal[int(np.argmax([kids[a].N for a in legal]))]
                case["searches"][-1]["then_action"] = best
                m.update_root(best)
                s.apply_action(best)
                if s.is_terminal():
                    break
            out.append(case)
    return out


def selfplay_examples():
    out = []
    for game in ["connect_four", "breakthrough(rows=6,columns=6)"]:
        for backup in ["on-policy", "soft-Z", "A0C", "off-policy"]:
            np.random.seed(5)
            ex = ref_game_utils.play_game_self(hash_eval(77), game, n_playouts=30, backup=backup, c_puct=2.5)
            out.append({"game": game, "backup": backup, "np_seed": 5, "n_playouts": 30,
                        "keys": [e[0] for e in ex], "values": [float(e[3]) for e in ex],
                        "policies": [[[i, float(p)] for i, p in enumerate(e[2]) if p != 0.0] for e in ex],
                        "board_sums": [float(np.sum(e[1] * np.arange(e[1].size).reshape(e[1].shape))) for e in ex]})
    return out


def encoding_pins():
    """SURVEY B.4: the shipped checkpoints pin the observation / action encodings of the game restatement."""
    res = {}
    ck = os.path.join(REF, "models", "example_model_connect_four.pth")
    shutil.copyfile(ck, os.path.join(HERE, "example_model_connect_four.pth"))  # weights are data, kept as a fixture
    g = pyspiel.load_game("connect_four")
    net = ref_network.Net([3, 6, 7], 7)
    net.load_state_dict(torch.load(ck, map_location="cpu", weights_only=True))
    net.eval()
    rng = np.random.RandomState(0)
    hists, boards = [], []
    while len(hists) < 64:
        s = g.new_initial_state()
        for _ in range(rng.randint(0, 30)):
            if s.is_terminal():
                break
            s.apply_action(int(rng.choice(s.legal_actions())))
        if s.is_terminal():
            continue
        hists.append(s.history())
        boards.append(ref_network.state_to_board(s, [3, 6, 7]))
    with torch.no_grad():
        p, v = net(torch.from_numpy(np.array(boards)).float())
    res["c4"] = {"histories": hists, "p": p.numpy().astype(np.float64).tolist(),
                 "v": v.numpy()[:, 0].astype(np.float64).tolist()}
    # 16-ply fixture: column 5 wins for x; the trained net must see it
    s = g.new_initial_state()
    for a in FIXTURE_16:
        s.apply_action(a)
    pp, vv = net.predict(s)
    res["c4_fixture16"] = {"p": pp, "v": vv}
    # breakthrough 6x6: policy mass on legal moves under the B.3 encoding
    ck6 = os.path.join(REF, "models", "example_model_breakthrough(6x6).pth")
    g6 = pyspiel.load_game("breakthrough(rows=6,columns=6)")
    net6 = ref_network.Net([3, 6, 6], 432)
    net6.load_state_dict(torch.load(ck6, map_location="cpu", weights_only=True))
    net6.eval()
    masses = []
    for _ in range(200):
        s = g6.new_initial_state()
        for _ in range(rng.randint(0, 40)):
            if s.is_terminal():
                break
            s.apply_action(int(rng.choice(s.legal_actions())))
        if s.is_terminal():
            continue
        pp, _ = net6.predict(s)
        masses.append(sum(pp[a] for a in s.legal_actions()))
    res["bt6_legal_mass_mean"] = float(np.mean(masses))
    return res


if __name__ == "__main__":
    golden = {"known_answers": known_answers(), "hash_searches": hash_searches(), "selfplay": selfplay_examples(),
              "encoding_pins": encoding_pins()}
    with open(os.path.join(HERE, "reference_golden.json"), "w") as f:
        json.dump(golden, f)
    print("wrote", os.path.join(HERE, "reference_golden.json"), os.path.getsize(os.path.join(HERE, "reference_golden.json")))
    print("bt6 legal mass", golden["encoding_pins"]["bt6_legal_mass_mean"], "c4 fixture16", golden["encoding_pins"]["c4_fixture16"])
