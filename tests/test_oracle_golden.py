"""CPU: the oracle (C restatement + Python port + RefNet) and the drop-in's host code against the golden vectors of the
UNMODIFIED reference: tests/golden/reference_golden.json (tests/golden/make_golden.py) and
tests/golden/reference_crosscheck.json (tests/golden/make_golden_crosscheck.py)."""
import ctypes as C
import json
import os

import numpy as np
import pytest

from oracle import cbind, pyspiel_shim, ref_port

HERE = os.path.dirname(os.path.abspath(__file__))
with open(os.path.join(HERE, "golden", "reference_golden.json")) as f:
    GOLD = json.load(f)
with open(os.path.join(HERE, "golden", "reference_crosscheck.json")) as f:
    CROSS = json.load(f)
L = cbind.lib()


def _state(game, hist):
    s = pyspiel_shim.load_game(game).new_initial_state()
    for a in hist:
        s.apply_action(a)
    return s


def _eval_cb(kind, seed):
    def cb(sp, pp, vp, _u):
        A = L.oz_num_actions(sp)
        L.oz_synth_eval(sp, kind, seed, 2 if A == 7 else 4, pp, vp)
    return cbind.EVAL_FN(cb)


def _hash_policy(seed):
    def fn(st):
        A = st.get_game().num_distinct_actions()
        pri = (C.c_double * A)()
        v = C.c_double()
        L.oz_synth_eval(C.byref(st.raw()), 1, seed, 2 if A == 7 else 4, pri, C.byref(v))
        return list(pri), v.value
    return fn


def test_known_answer_vectors_c_oracle():
    """SURVEY C.3 vectors (uniform evaluator) reproduced by the C oracle."""
    for case in GOLD["known_answers"]:
        game = case["game"]
        A = pyspiel_shim.load_game(game).num_distinct_actions()
        t = L.oz_tree_new(A, 2.5, case["n_playouts"], 0, 0.25)
        cb = _eval_cb(0, 0)
        counts = (C.c_int64 * A)()
        if "reuse_after" in case:
            s0 = _state(game, case["reuse_after"][0])
            L.oz_tree_search(t, C.byref(s0.raw()), cb, None, None, counts)
            L.oz_tree_update_root(t, case["reuse_after"][1])
        s = _state(game, case["history"])
        L.oz_tree_search(t, C.byref(s.raw()), cb, None, None, counts)
        assert L.oz_tree_root_n(t) == case["root_n"]
        assert L.oz_tree_root_q(t) == case["root_q"]
        if "n" in case:
            n = (C.c_int64 * A)()
            q = (C.c_double * A)()
            p = (C.c_double * A)()
            L.oz_tree_root_children(t, n, q, p)
            assert list(n) == case["n"] and list(q) == case["q"]
        else:
            assert [counts[a] for a in case["legal"]] == case["n_legal_order"]
        L.oz_tree_free(t)


def test_known_answers_are_the_survey_vectors():
    ka = GOLD["known_answers"]
    assert ka[0]["n"] == [15, 14, 14, 14, 14, 14, 14] and ka[0]["root_n"] == 100
    assert ka[1]["n"] == [115, 114, 114, 114, 114, 114, 114]
    assert ka[2]["n"] == [3, 3, 3, 3, 3, 81, 3] and ka[2]["root_q"] == -0.81
    assert ka[3]["n"] == [6, 6, 7, 6, 6, 762, 6]
    assert ka[4]["root_n"] == 114 and ka[4]["n"] == [17, 16, 16, 16, 16, 16, 16]
    assert ka[5]["n_legal_order"] == [13] * 7 + [12] * 9


@pytest.mark.parametrize("impl", ["c", "port"])
def test_hash_evaluator_searches_with_injected_noise(impl):
    """Reference visit counts / Q / P (incl. Dirichlet-mixed priors and re-rooted second searches), bit-exact."""
    for case in GOLD["hash_searches"]:
        game = case["game"]
        g = pyspiel_shim.load_game(game)
        A = g.num_distinct_actions()
        s = _state(game, case["history"])
        if impl == "c":
            t = L.oz_tree_new(A, 2.5, case["n_playouts"], 1, 0.25)
            cb = _eval_cb(1, 77)
        else:
            m = ref_port.PortMCTS(_hash_policy(77), A, n_playouts=case["n_playouts"])
        for srch in case["searches"]:
            legal = s.legal_actions()
            assert legal == srch["legal"]
            if impl == "c":
                counts = (C.c_int64 * A)()
                nz = (C.c_double * len(legal))(*srch["noise"])
                L.oz_tree_search(t, C.byref(s.raw()), cb, None, nz, counts)
                n = (C.c_int64 * A)()
                q = (C.c_double * A)()
                p = (C.c_double * A)()
                L.oz_tree_root_children(t, n, q, p)
                got = ([n[a] for a in legal], [q[a] for a in legal], [p[a] for a in legal],
                       L.oz_tree_root_n(t), L.oz_tree_root_q(t))
            else:
                import numpy.random as npr
                orig = npr.dirichlet
                npr.dirichlet = lambda alpha, _n=srch["noise"]: np.array(_n)  # inject the recorded draw
                try:
                    m.search(s)
                finally:
                    npr.dirichlet = orig
                acts, ids = m.kids[m.root]
                assert acts == legal
                got = ([m.visits[j] for j in ids], [m.mean[j] for j in ids], [m.prior[j] for j in ids],
                       m.visits[m.root], m.mean[m.root])
            assert got[0] == srch["n"], (game, case["history"])
            assert got[1] == srch["q"] and got[2] == srch["p"]
            assert got[3] == srch["root_n"] and got[4] == srch["root_q"]
            a = srch["then_action"]
            if impl == "c":
                L.oz_tree_update_root(t, a)
            else:
                m.update_root(a)
            s.apply_action(a)
        if impl == "c":
            L.oz_tree_free(t)


def test_selfplay_examples_port_vs_golden():
    """play_game_self examples for all four backup targets under np.random.seed(5), from the reference."""
    for case in GOLD["selfplay"]:
        np.random.seed(case["np_seed"])
        ex = ref_port.selfplay_game(_hash_policy(77), case["game"], pyspiel_shim.load_game,
                                    n_playouts=case["n_playouts"], backup=case["backup"], c_puct=2.5)
        assert [e[0] for e in ex] == case["keys"]
        assert [float(e[3]) for e in ex] == case["values"]
        pol = [[[i, float(p)] for i, p in enumerate(e[2]) if p != 0.0] for e in ex]
        assert pol == case["policies"]
        sums = [float(np.sum(e[1] * np.arange(e[1].size).reshape(e[1].shape))) for e in ex]
        assert sums == case["board_sums"]


def test_encoding_pins_with_shipped_checkpoint():
    """SURVEY B.4: reference Net outputs on 64 Connect Four positions (shipped checkpoint) reproduced by the
    oracle's RefNet over the oracle's observation planes -> pins plane order, row orientation and action ids."""
    import torch
    from oracle import ref_net
    pins = GOLD["encoding_pins"]
    sd = torch.load(os.path.join(HERE, "golden", "example_model_connect_four.pth"), map_location="cpu",
                    weights_only=True)
    net = ref_net.RefNet([3, 6, 7], 7).eval()
    net.load_state_dict(sd)  # same key names as the reference checkpoints (SURVEY C.1)
    boards = []
    for h in pins["c4"]["histories"]:
        boards.append(ref_port.board_planes(_state("connect_four", h), [3, 6, 7]))
    with torch.no_grad():
        p, v = net(torch.from_numpy(np.array(boards)).float())
    assert np.abs(p.numpy() - np.array(pins["c4"]["p"])).max() < 1e-5
    assert np.abs(v.numpy()[:, 0] - np.array(pins["c4"]["v"])).max() < 1e-5
    assert int(np.argmax(pins["c4_fixture16"]["p"])) == 5 and pins["c4_fixture16"]["v"] > 0.5
    assert pins["bt6_legal_mass_mean"] > 0.98


def test_breakthrough_encoding_pins_with_shipped_checkpoint():
    """Same pin for Breakthrough 6x6 (tests/golden/make_golden_bt6.py): the reference Net with its shipped 6x6 checkpoint on
    64 positions -> priors [432] / value reproduced by the oracle's RefNet over the oracle's planes (plane order black /
    white / empty, row 0 = black's home row, action id = ((r*C + c)*6 + dir)*2 + capture, SURVEY B.3); the legal-move lists
    of the game restatement carry 0.98 of the trained policy mass, which no other numbering does (SURVEY B.4)."""
    import torch
    from oracle import ref_net
    pins = np.load(os.path.join(HERE, "golden", "bt6_pins.npz"))
    sd = torch.load(os.path.join(HERE, "golden", "example_model_breakthrough_6x6.pth"), map_location="cpu",
                    weights_only=True)
    net = ref_net.RefNet([3, 6, 6], 432).eval()
    net.load_state_dict(sd)
    game = "breakthrough(rows=6,columns=6)"
    boards, mass = [], []
    for i, h in enumerate(pins["histories"]):
        st = _state(game, [int(a) for a in h if a >= 0])
        boards.append(ref_port.board_planes(st, [3, 6, 6]))
        legal = st.legal_actions()
        assert legal == [int(a) for a in pins["legal"][i] if a >= 0]
        mass.append(float(pins["p"][i, legal].sum()))
    with torch.no_grad():
        p, v = net(torch.from_numpy(np.array(boards)).float())
    assert np.abs(p.numpy() - pins["p"]).max() < 1e-5
    assert np.abs(v.numpy()[:, 0] - pins["v"]).max() < 1e-5
    assert np.mean(mass) > 0.97


def test_game_rules_properties():
    """Random playouts: legal lists ascending, terminal <=> no legal moves, returns zero-sum, C4 draw only at 42."""
    rng = np.random.RandomState(1)
    for game in ["connect_four", "breakthrough(rows=6,columns=6)", "breakthrough", "breakthrough(rows=8,columns=5)"]:
        g = pyspiel_shim.load_game(game)
        for _ in range(60):
            s = g.new_initial_state()
            while not s.is_terminal():
                legal = s.legal_actions()
                assert legal == sorted(set(legal)) and len(legal) > 0
                assert s.current_player() == len(s.history()) % 2
                assert all(0 <= a < g.num_distinct_actions() for a in legal)
                illegal = [a for a in range(min(g.num_distinct_actions(), 40)) if a not in legal]
                if illegal:
                    c = s.clone()
                    with pytest.raises(RuntimeError):
                        c.apply_action(illegal[0])
                s.apply_action(int(rng.choice(legal)))
            r = s.returns()
            assert r[0] == -r[1] and s.legal_actions() == [] and s.current_player() == -4
            if game == "connect_four":
                assert (r[0] != 0) or len(s.history()) == 42
            else:
                assert r[0] != 0
                assert r[(len(s.history()) - 1) % 2] == 1.0  # the mover wins in breakthrough
    s = pyspiel_shim.load_game("breakthrough(rows=6,columns=6)").new_initial_state()
    assert s.legal_actions() == [74, 76, 84, 86, 88, 96, 98, 100, 108, 110, 112, 120, 122, 124, 132, 134]


def test_port_and_c_oracle_vs_live_reference():
    """play_game_self and a 300-playout search as the unmodified reference returns them (mcts.py / game_utils.py run over
    the shim; recorded in reference_crosscheck.json): the port's self-play and the C oracle's search reproduce them."""
    fn = _hash_policy(123)
    for case in CROSS["selfplay"]:
        np.random.seed(11)
        b = ref_port.selfplay_game(fn, case["game"], pyspiel_shim.load_game, n_playouts=25, backup=case["backup"])
        A = pyspiel_shim.load_game(case["game"]).num_distinct_actions()
        assert len(b) == len(case["keys"])
        for i, y in enumerate(b):
            dense = [0.0] * A
            for a, p in case["policies"][i]:
                dense[a] = p
            assert y[0] == case["keys"][i] and y[2] == dense and y[3] == case["values"][i]
            assert np.array_equal(y[1].ravel(), np.array(case["boards"][i]))
    s = pyspiel_shim.load_game("connect_four").new_initial_state()
    t = L.oz_tree_new(7, 2.5, 300, 0, 0.25)
    counts = (C.c_int64 * 7)()
    L.oz_tree_search(t, C.byref(s.raw()), _eval_cb(1, 123), None, None, counts)
    assert list(counts) == CROSS["search300"]["counts"]
    assert L.oz_tree_root_q(t) == CROSS["search300"]["root_q"]
    L.oz_tree_free(t)


def test_random_rollout_evaluator_matches_live_reference():
    """MCTS.random_rollout (mcts.py:205-223, SURVEY 8(f).4): the oracle port and the drop-in's host implementation draw the
    reference's playouts from the same numpy seed (same priors, value and RNG position afterwards); a whole search driven
    by it gives the reference's visit distribution."""
    from alphazero_openspiel_b200.mcts import MCTS as OurMCTS
    for case in CROSS["rollouts"]:
        g = pyspiel_shim.load_game(case["game"])
        A = g.num_distinct_actions()
        ours = OurMCTS(None, A)                      # no engine is created before a search
        port_fn = ref_port.rollout_policy(A)
        s = g.new_initial_state()
        for ply, want in enumerate(case["evals"]):
            for fn in (ours.random_rollout, port_fn):
                np.random.seed(100 + ply)
                pri, v = fn(s)
                assert (list(pri), v, np.random.random_sample()) == (want["priors"], want["value"], want["next_draw"])
            s.apply_action(s.legal_actions()[ply % len(s.legal_actions())])
        port = ref_port.PortMCTS(port_fn, A, n_playouts=40, use_dirichlet=False)
        np.random.seed(5)
        assert list(port.search(g.new_initial_state())) == case["search"]


def test_uct_mode_port_vs_live_reference():
    """use_puct=False (mcts.py:80, SURVEY 8(f).4) exactly as the reference behaves: the flag lives on the nodes, the first
    root is built without it (mcts.py:122), so only a tree whose root came from update_root on a leaf root (mcts.py:199-200)
    scores with the UCT formula.  The port gives the reference's visit distributions and root Q through both kinds of
    tree."""
    fn = _hash_policy(31)
    for case in CROSS["uct"]:
        g = pyspiel_shim.load_game(case["game"])
        A = g.num_distinct_actions()
        port = ref_port.PortMCTS(fn, A, n_playouts=80, use_dirichlet=case["dirichlet"], use_puct=False)
        s = g.new_initial_state()
        if case["leaf_update_first"]:     # what a second player's bot does before its first search: the UCT tree
            first = s.legal_actions()[1]
            s.apply_action(first)
            port.update_root(first)
            assert port.tree_uct
        for move, want in enumerate(case["moves"]):
            np.random.seed(70 + move)
            b = port.search(s)
            assert list(b) == want["counts"] and port.mean[port.root] == want["root_q"]
            act = int(np.argmax(b))
            port.update_root(act)
            s.apply_action(act)


def test_neuralnetbot_and_play_game_match_live_reference():
    """The host-only pieces of the match-up harness (alphazerobot.py:96-118, game_utils.py:16-35): the reference's
    policies, actions and game results for the same policy functions."""
    from alphazero_openspiel_b200 import alphazerobot as our_bot, game_utils as our_gu
    for case in CROSS["netbot"]:
        g = pyspiel_shim.load_game(case["game"])
        fa, fb = _hash_policy(3), _hash_policy(4)
        s = g.new_initial_state()
        for want in case["steps"]:
            po, ao = our_bot.NeuralNetBot(g, 0, fa).step(s)
            assert ao == want["action"] and [[int(a), float(p)] for a, p in po] == want["policy"]
            s.apply_action(int(ao))
        got = our_gu.play_game(g, our_bot.NeuralNetBot(g, 0, fa), our_bot.NeuralNetBot(g, 1, fb))
        assert got == case["play_game"]
