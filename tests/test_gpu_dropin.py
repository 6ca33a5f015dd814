"""GPU parity of the drop-in Python API (MCTS / AlphaZeroBot / play_game_self / Net / ExampleGenerator)
against the oracle's port of the reference (oracle.ref_port, pinned to the reference's recorded outputs in test_oracle_golden)."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def shim():
    from oracle import pyspiel_shim
    return pyspiel_shim.install()  # stands in for the caller's OpenSpiel


def _hash_policy(seed=77):
    from oracle import cbind
    lib = cbind.lib()

    def fn(state):
        A = state.get_game().num_distinct_actions()
        pri = (C.c_double * A)()
        v = C.c_double()
        lib.oz_synth_eval(C.byref(state.raw()), 1, seed, 2 if A == 7 else 4, pri, C.byref(v))
        return list(pri), v.value
    return fn


@pytest.mark.parametrize("game", ["connect_four", "breakthrough(rows=6,columns=6)"])
def test_mcts_search_update_root_matches_reference_port(shim, game):
    from oracle import ref_port
    from alphazero_openspiel_b200.mcts import MCTS
    g = shim.load_game(game)
    A = g.num_distinct_actions()
    fn = _hash_policy()
    for dirichlet in (True, False):
        ours = MCTS(fn, A, n_playouts=120, use_dirichlet=dirichlet, game_name=game)
        ref = ref_port.PortMCTS(fn, A, n_playouts=120, use_dirichlet=dirichlet)
        s = g.new_initial_state()
        for move in range(4):
            np.random.seed(10 + move)
            a = ours.search(s)
            np.random.seed(10 + move)
            b = ref.search(s)
            assert a == b
            assert ours.root.N == ref.visits[ref.root] and ours.root.Q == ref.mean[ref.root]
            kids = ours.root.children
            acts, ids = ref.kids[ref.root]
            assert list(kids.keys()) == acts
            for act, j in zip(acts, ids):
                assert kids[act].N == ref.visits[j] and kids[act].Q == ref.mean[j] and kids[act].P == ref.prior[j]
            sz, a0c, off = ours.value_targets()
            assert sz == ref.target_soft_z() and a0c == ref.target_a0c() and off == ref.target_off_policy()
            act = int(np.argmax(a))
            ours.update_root(act)
            ref.update_root(act)
            s.apply_action(act)
        with pytest.raises(KeyError):
            ours.update_root(A + 5 if game == "connect_four" else 0)


@pytest.mark.parametrize("game", ["connect_four", "breakthrough(rows=6,columns=6)"])
def test_mcts_playout_matches_reference_port(shim, game):
    """MCTS.playout(state) (mcts.py:126-153): one simulation per call, the caller's state is walked to the leaf in place,
    no root Dirichlet expansion.  After every playout the root statistics and the leaf reached equal the port's; a search()
    afterwards continues from the same tree.  A position two plies from the end exercises the terminal-leaf branch."""
    from oracle import ref_port
    from alphazero_openspiel_b200.mcts import MCTS
    g = shim.load_game(game)
    A = g.num_distinct_actions()
    fn = _hash_policy()
    s = g.new_initial_state()
    if game == "connect_four":
        for a in [3, 3, 4, 4, 5, 0]:      # x threatens 2-3-4-5-6: terminal leaves appear within a few playouts
            s.apply_action(a)
    ours = MCTS(fn, A, n_playouts=50, use_dirichlet=True, game_name=game)
    ref = ref_port.PortMCTS(fn, A, n_playouts=50, use_dirichlet=True)
    terminal_leaves = 0
    for i in range(70):
        a, b = s.clone(), s.clone()
        ours.playout(a)
        ref.playout(b)
        assert a.history() == b.history(), i
        terminal_leaves += a.is_terminal()
        assert ours.root.N == ref.visits[ref.root] and ours.root.Q == ref.mean[ref.root]
        kids = ours.root.children
        acts, ids = ref.kids[ref.root]
        assert list(kids.keys()) == acts
        for act, j in zip(acts, ids):
            assert kids[act].N == ref.visits[j] and kids[act].Q == ref.mean[j] and kids[act].P == ref.prior[j]
    if game == "connect_four":
        assert terminal_leaves > 0
    np.random.seed(3)
    x = ours.search(s)
    np.random.seed(3)
    y = ref.search(s)
    assert x == y


@pytest.mark.parametrize("game", ["connect_four", "breakthrough(rows=6,columns=6)"])
def test_mcts_use_puct_false_matches_reference_port(shim, game):
    """use_puct=False (mcts.py:80; SURVEY 8(f).4) with the reference's actual semantics (the port is pinned to the live
    reference in test_oracle_golden): a freshly constructed MCTS still searches with PUCT, a tree whose root was created by
    update_root on a leaf root searches with the UCT formula -- visit counts, Q and tree reuse equal the port's."""
    from oracle import ref_port
    from alphazero_openspiel_b200.mcts import MCTS
    g = shim.load_game(game)
    A = g.num_distinct_actions()
    fn = _hash_policy(5)
    seen = []
    for leaf_update_first in (False, True):
        ours = MCTS(fn, A, n_playouts=90, use_dirichlet=True, use_puct=False, game_name=game)
        ref = ref_port.PortMCTS(fn, A, n_playouts=90, use_dirichlet=True, use_puct=False)
        s = g.new_initial_state()
        if leaf_update_first:
            first = s.legal_actions()[1]       # what a second player's bot does before its first search
            s.apply_action(first)
            ours.update_root(first)
            ref.update_root(first)
        for move in range(3):
            np.random.seed(60 + move)
            a = ours.search(s)
            np.random.seed(60 + move)
            b = ref.search(s)
            assert list(a) == list(b)
            assert ours.root.N == ref.visits[ref.root] and ours.root.Q == ref.mean[ref.root]
            if move == 0:
                seen.append(list(a))
            act = int(np.argmax(a))
            ours.update_root(act)
            ref.update_root(act)
            s.apply_action(act)
        assert ref.tree_uct == leaf_update_first


def test_mcts_with_random_rollout_evaluator_matches_port(shim):
    """MCTS.random_rollout as policy_fn (mcts.py:205-223; SURVEY 8(f).4): the device search consumes the host rollouts in
    the reference's order, so visit counts equal the port's from the same numpy seed."""
    from oracle import ref_port
    from alphazero_openspiel_b200.mcts import MCTS
    game = "connect_four"
    g = shim.load_game(game)
    A = g.num_distinct_actions()
    ours = MCTS(None, A, n_playouts=60, use_dirichlet=False, game_name=game)
    ours.policy_fn = ours.random_rollout
    ref = ref_port.PortMCTS(ref_port.rollout_policy(A), A, n_playouts=60, use_dirichlet=False)
    s = g.new_initial_state()
    for move in range(3):
        np.random.seed(40 + move)
        a = ours.search(s)
        np.random.seed(40 + move)
        b = ref.search(s)
        assert list(a) == list(b) and ours.root.N == ref.visits[ref.root] and ours.root.Q == ref.mean[ref.root]
        act = int(np.argmax(a))
        ours.update_root(act)
        ref.update_root(act)
        s.apply_action(act)


@pytest.mark.parametrize("game,backup", [("connect_four", "on-policy"), ("connect_four", "soft-Z"),
                                         ("connect_four", "A0C"), ("connect_four", "off-policy"),
                                         ("breakthrough(rows=6,columns=6)", "off-policy")])
def test_play_game_self_matches_reference_port(shim, game, backup):
    """Whole games through AlphaZeroBot.step with the global numpy RNG: examples must be identical."""
    from oracle import ref_port
    from alphazero_openspiel_b200.game_utils import play_game_self
    fn = _hash_policy(5)
    np.random.seed(42)
    ours = play_game_self(fn, game, n_playouts=40, backup=backup, c_puct=2.5)
    np.random.seed(42)
    ref = ref_port.selfplay_game(fn, game, shim.load_game, n_playouts=40, backup=backup, c_puct=2.5)
    assert len(ours) == len(ref) > 4
    for a, b in zip(ours, ref):
        assert a[0] == b[0]
        assert np.array_equal(a[1], b[1])
        assert list(a[2]) == list(b[2])
        assert a[3] == b[3]


def test_bot_two_player_mode_and_restart(shim):
    """keep_search_tree with two update_root calls per step (alphazerobot.py:60-64) and argmax moves."""
    from oracle import ref_port
    from alphazero_openspiel_b200.alphazerobot import AlphaZeroBot
    g = shim.load_game("connect_four")
    fn = _hash_policy(9)
    ours = AlphaZeroBot(g, 0, fn, n_playouts=50, use_dirichlet=False)
    ref = ref_port.PortBot(g, 0, fn, n_playouts=50, use_dirichlet=False)
    s = g.new_initial_state()
    rng = np.random.RandomState(0)
    while not s.is_terminal() and len(s.history()) < 14:
        pa, aa = ours.step(s)
        pb, ab = ref.step(s)
        assert aa == ab and [(x, float(y)) for x, y in pa] == [(x, float(y)) for x, y in pb]
        s.apply_action(int(aa))
        if not s.is_terminal():
            s.apply_action(int(rng.choice(s.legal_actions())))
    ours.restart()
    assert ours.mcts.root.N == 0 and ours.mcts.root.is_leaf()


def test_net_matches_fp32_reference_and_bf16_evaluator(shim):
    """Net == oracle RefNet in fp32 (same state_dict); BatchedEvaluator (bf16, folded BN) within bf16 tolerance."""
    import torch
    from oracle import ref_net
    from alphazero_openspiel_b200.network import Net, BatchedEvaluator
    from alphazero_openspiel_b200 import engine as E, _lib as L
    for game in ("connect_four", "breakthrough(rows=6,columns=6)"):
        shape, A = E.game_shape(game)
        torch.manual_seed(3)
        ref = ref_net.RefNet(shape, A).eval()
        with torch.no_grad():  # non-trivial BatchNorm statistics
            for m in ref.modules():
                if isinstance(m, torch.nn.BatchNorm2d):
                    m.running_mean.uniform_(-0.3, 0.3)
                    m.running_var.uniform_(0.5, 1.5)
                    m.weight.uniform_(0.5, 1.5)
                    m.bias.uniform_(-0.2, 0.2)
        net = Net(shape, A).eval()
        net.load_state_dict(ref.state_dict())
        B = 256
        hist, lens = E.game_random_playouts(game, B, seed=5, max_plies=20)
        out = E.game_replay_dev(game, hist, lens, L.OBS_F32_NCHW)
        out_bf = E.game_replay_dev(game, hist, lens, L.OBS_BF16_NHWC)
        x = out["obs"].cpu()
        with torch.no_grad():
            p_ref, v_ref = ref(x)
            p_net, v_net = net(x)
        assert torch.equal(p_ref, p_net) and torch.equal(v_ref, v_net)
        ev = BatchedEvaluator(net, B, "cuda:0")
        p, v = ev.eval_batch(out_bf["obs"])
        # bf16 tolerance: 8-bit mantissa through 11 layers
        assert (p.cpu() - p_ref).abs().max().item() < 3e-2
        assert (v.cpu() - v_ref[:, 0]).abs().max().item() < 6e-2
        assert (p.cpu().argmax(1) == p_ref.argmax(1)).float().mean().item() > 0.9


def test_example_generator_contract(shim):
    """ExampleGenerator.generate_examples: n_games finished games in the reference's example format, consistent
    with the game rules (boards replay from the info-state string, targets are distributions over legal moves)."""
    import torch
    from alphazero_openspiel_b200.examplegenerator import ExampleGenerator
    from alphazero_openspiel_b200.network import Net
    from tests import oracle_util as ou
    torch.manual_seed(0)
    net = Net([3, 6, 7], 7).eval()
    gen = ExampleGenerator(net, "connect_four", torch.device("cuda:0"), n_playouts=30, c_puct=2.5,
                           dirichlet_ratio=0.25, temperature=1.0, backup="on-policy", n_trees=16, seed=3)
    games = gen.generate_examples(40)
    assert len(games) == 40
    assert gen.last_stats["overflow"] == 0 and gen.last_stats["games"] == 40
    for game in games:
        assert 7 <= len(game) <= 42
        for i, (key, board, pol, value) in enumerate(game):
            hist = [int(t) for t in key.split(", ")] if key else []
            assert len(hist) == i
            ref = ou.replay("connect_four", hist)
            assert board.dtype == np.float64 and np.array_equal(board, ref["board"])
            assert len(pol) == 7 and abs(sum(pol) - 1.0) < 1e-12
            assert all((p == 0.0) for a, p in enumerate(pol) if a not in ref["legal"])
            assert value in (-1.0, 0.0, 1.0)
        vals = [ex[3] for ex in game]
        assert all(vals[i] == -vals[i + 1] for i in range(len(vals) - 1))
    # soft-Z / A0C / off-policy targets are finite numbers in [-1, 1]
    gen2 = ExampleGenerator(net, "connect_four", torch.device("cuda:0"), n_playouts=30, backup="off-policy",
                            n_trees=8, seed=4)
    for game in gen2.generate_examples(8):
        assert all(-1.0 <= ex[3] <= 1.0 for ex in game)


def test_baseline_config1_shipped_checkpoint_game(shim):
    """BASELINE.json configs[0]: one Connect Four self-play game, 100 sims/move, the shipped example checkpoint, the
    evaluator Net.predict on the CPU in fp32 -- through the drop-in (search on the GPU) and through the oracle's port of
    the reference: identical examples for the same numpy seed."""
    import os
    import torch
    from oracle import ref_port
    from alphazero_openspiel_b200.game_utils import play_game_self
    from alphazero_openspiel_b200.network import Net
    ck = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "example_model_connect_four.pth")
    net = Net([3, 6, 7], 7)
    net.load_state_dict(torch.load(ck, map_location="cpu", weights_only=True))  # reference key names load unchanged
    net.eval()
    kwargs = dict(n_playouts=100, c_puct=2.5, dirichlet_ratio=0.25, temperature=1.0, backup="on-policy")
    np.random.seed(2024)
    ours = play_game_self(net.predict, "connect_four", **kwargs)
    np.random.seed(2024)
    ref = ref_port.selfplay_game(net.predict, "connect_four", shim.load_game, **kwargs)
    assert len(ours) == len(ref) >= 7
    for a, b in zip(ours, ref):
        assert a[0] == b[0] and np.array_equal(a[1], b[1]) and list(a[2]) == list(b[2]) and a[3] == b[3]


def test_example_generator_many_short_searches_never_overflows_records(shim):
    """More training records than the device buffer holds (1 M): the generator must drain in time, not overflow."""
    import torch
    from alphazero_openspiel_b200.examplegenerator import ExampleGenerator
    from alphazero_openspiel_b200.network import Net
    torch.manual_seed(0)
    net = Net([3, 6, 7], 7).eval()
    gen = ExampleGenerator(net, "connect_four", torch.device("cuda:0"), n_playouts=3, n_trees=4096, seed=9)
    games = gen.generate_examples(70000)
    assert len(games) == 70000 and gen.last_stats["overflow"] == 0
    assert sum(len(g) for g in games) == gen.last_stats["moves"] > (1 << 20)


def test_shipped_checkpoint_beats_random_through_the_whole_stack(shim):
    """End-to-end behavioural pin of the UNPINNED game restatement (SURVEY B.4 / tournament.py:19-27 in spirit): the
    reference's trained Connect Four checkpoint + 100-playout search on the device kernels + the tcgen05 evaluator must
    crush a uniform-random opponent from both sides.  A wrong plane order, row orientation, action id or value sign
    anywhere between az_step's observation encode and the policy/value head would turn this into coin flips."""
    import os
    import torch
    from alphazero_openspiel_b200.evaluate import zero_vs_random
    from alphazero_openspiel_b200.network import Net
    ck = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "example_model_connect_four.pth")
    net = Net([3, 6, 7], 7)
    net.load_state_dict(torch.load(ck, map_location="cpu", weights_only=True))
    net.eval()
    # 8 playouts: the result is decided by the network's policy / value, not by brute-force search
    # (measured, 256 pairs: shipped checkpoint (1.0, 1.0); untrained network (0.48, 0.60); at 100 playouts even the
    #  untrained network scores 0.97 against random, so that setting would not discriminate)
    s_first, s_second = zero_vs_random(net, "connect_four", n_pairs=64, n_playouts=8, seed=3)
    assert s_first >= 0.95 and s_second >= 0.95, (s_first, s_second)
    torch.manual_seed(0)
    blank = Net([3, 6, 7], 7).eval()
    b_first, b_second = zero_vs_random(blank, "connect_four", n_pairs=64, n_playouts=8, seed=3)
    assert b_first <= 0.85 and b_second <= 0.85, (b_first, b_second)


def test_net_only_match_up_and_trainer_test_agent(shim):
    """evaluate.net_vs_random (`test_net_vs_random`, game_utils.py:100-112: NeuralNetBot = argmax of the policy over the legal
    moves, no search): the reference's trained checkpoint beats a random player clearly and beats what an untrained network
    scores; Trainer.test_agent runs both batched match-ups."""
    import os
    import torch
    from alphazero_openspiel_b200.evaluate import net_vs_random
    from alphazero_openspiel_b200.network import Net
    from alphazero_openspiel_b200.train import Trainer
    ck = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "example_model_connect_four.pth")
    net = Net([3, 6, 7], 7)
    net.load_state_dict(torch.load(ck, map_location="cpu", weights_only=True))
    net.eval()
    t1, t2 = net_vs_random(net, "connect_four", n_pairs=128, seed=1)
    torch.manual_seed(0)
    b1, b2 = net_vs_random(Net([3, 6, 7], 7).eval(), "connect_four", n_pairs=128, seed=1)
    assert t1 + t2 > 1.2 and t1 + t2 > b1 + b2 + 0.4, (t1, t2, b1, b2)
    tr = Trainer(n_tests=8, n_playouts_train=8)
    tr.current_net.load_state_dict(net.state_dict())
    out = tr.test_agent()      # train.py:238-270: net vs random, net vs mcts100, zero vs mcts200, net vs mcts200
    assert set(out) == {"net_vs_random", "net_vs_mcts100", "zero_vs_mcts200", "net_vs_mcts200"}
    assert all(-1.0 <= v <= 1.0 for v in out.values())
    assert out["net_vs_random"] > 0.5


def test_tournament_alphazero_vs_mcts_with_the_shipped_breakthrough_checkpoint(shim):
    """tournament.py:19-27, the reference's only published number: with models/example_model_breakthrough(6x6).pth an
    AlphaZero bot with 100 playouts "should win over 99% of games" against the MCTS bot with 200 playouts.  Here both bots
    run batched on the device (evaluate.zero_vs_mcts through ExampleGenerator.generate_tests; the MCTS bot is the UCT +
    random-rollout bot of evaluate.py) -- an end-to-end pin of the Breakthrough game kernels, the observation encoding and
    the large-action-space evaluator head.  The untrained network does not get there."""
    import os
    import torch
    from alphazero_openspiel_b200.examplegenerator import ExampleGenerator
    from alphazero_openspiel_b200.game_utils import test_zero_vs_mcts, test_zero_vs_zero
    from alphazero_openspiel_b200.network import Net
    game = "breakthrough(rows=6,columns=6)"
    ck = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "example_model_breakthrough_6x6.pth")
    net = Net([3, 6, 6], 432)
    net.load_state_dict(torch.load(ck, map_location="cpu", weights_only=True))
    net.eval()
    gen = ExampleGenerator(net, game, torch.device("cuda:0"), is_test=True, generate_statistics=False, seed=11)
    gen.kwargs["settings1"] = {"n_playouts": 100}
    avg = gen.generate_tests(48, test_zero_vs_mcts, 200)          # 96 games
    win_rate = avg * 0.5 + 0.5
    assert win_rate >= 0.95, win_rate
    torch.manual_seed(0)
    blank = ExampleGenerator(Net([3, 6, 6], 432).eval(), game, torch.device("cuda:0"), is_test=True, seed=11)
    blank.kwargs["settings1"] = {"n_playouts": 100}
    assert blank.generate_tests(48, test_zero_vs_mcts, 200) * 0.5 + 0.5 < win_rate - 0.1
    # zero vs zero (tournament.py:30-53): more playouts must not lose to fewer with the same network
    gen2 = ExampleGenerator(net, game, torch.device("cuda:0"), is_test=True, generate_statistics=True, seed=5)
    gen2.kwargs["settings1"] = {"n_playouts": 200, "use_probabilistic_actions": True}
    gen2.kwargs["settings2"] = {"n_playouts": 20, "use_probabilistic_actions": True}
    avg2, stats = gen2.generate_tests(32, test_zero_vs_zero, None)
    assert -1.0 <= avg2 <= 1.0 and stats == []
    assert avg2 > 0.0, avg2
