"""Left-right reflection (AZ_F_REFLECT in self-play, Trainer(reflect_minibatches=True) in training): the game symmetry on the
oracle's games, the training minibatch rule on the host, and on the GPU the engine against the restatement of
tests/selfplay_rule.py, the evaluator rows, the eval cache, the gather kernel and the Trainer paths."""
import ctypes as C

import numpy as np
import pytest

from tests import oracle_util as ou
from tests import selfplay_rule as sr
from tests.selfplay_rule import BT6, BT8, C4

GAMES = [C4, BT6, BT8]


def _random_histories(game, n, seed):
    from oracle import pyspiel_shim
    rng = np.random.RandomState(seed)
    g = pyspiel_shim.load_game(game)
    out = []
    for _ in range(n):
        s, hist = g.new_initial_state(), []
        stop = rng.randint(0, 80)
        while not s.is_terminal() and len(hist) < stop:
            a = int(rng.choice(s.legal_actions()))
            s.apply_action(a)
            hist.append(a)
        out.append(hist)
    return out


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("game", GAMES)
def test_reflect_actions_is_the_involution_of_the_rule(game):
    from alphazero_openspiel_b200 import _lib as L
    from alphazero_openspiel_b200.engine import game_shape, parse_game_name, reflect_actions
    gid, rows, cols = parse_game_name(game)
    perm = reflect_actions(game)
    assert len(perm) == game_shape(game)[1]
    assert np.array_equal(perm[perm], np.arange(len(perm)))
    assert list(perm) == [sr.reflect_action(a, gid, cols) for a in range(len(perm))]
    assert (perm != np.arange(len(perm))).sum() > len(perm) // 2
    lib = L.load()
    out = np.zeros(len(perm), np.int32)
    assert lib.az_reflect_actions(7, 6, 6, out.ctypes.data) != 0 and b"unknown game_id" in lib.az_last_error()
    assert lib.az_reflect_actions(L.GAME_BREAKTHROUGH, 9, 9, out.ctypes.data) != 0
    assert lib.az_reflect_actions(L.GAME_CONNECT_FOUR, 6, 7, None) != 0


@pytest.mark.parametrize("game", GAMES)
def test_reflection_is_a_symmetry_of_the_game(game):
    """On random positions s, R(s) built by replaying the reflected history: legal(R(s)) = R(legal(s)),
    apply(R(s), R(a)) = R(apply(s, a)), the same outcome, and state_to_board(R(s)) = state_to_board(s) with the columns
    flipped -- also for boards_from_bitboards, the numpy planes of the training path."""
    from oracle import pyspiel_shim
    from alphazero_openspiel_b200.engine import parse_game_name, reflect_actions
    from alphazero_openspiel_b200.examplegenerator import boards_from_bitboards
    gid, rows, cols = parse_game_name(game)
    perm = reflect_actions(game)
    g = pyspiel_shim.load_game(game)
    n_terminal = 0
    for hist in _random_histories(game, 150, 3):
        s, rs = g.new_initial_state(), g.new_initial_state()
        for a in hist:
            s.apply_action(a)
            rs.apply_action(int(perm[a]))
            b0, b1 = s.bitboards()
            assert rs.bitboards() == (sr.mirror(b0, rows, cols), sr.mirror(b1, rows, cols))
        assert sorted(rs.legal_actions()) == sorted(int(perm[a]) for a in s.legal_actions())
        assert rs.is_terminal() == s.is_terminal() and rs.returns() == s.returns()
        n_terminal += s.is_terminal()
        for a in s.legal_actions():
            t, rt = s.clone(), rs.clone()
            t.apply_action(a)
            rt.apply_action(int(perm[a]))
            assert rt.bitboards() == tuple(sr.mirror(x, rows, cols) for x in t.bitboards())
        board, rboard = ou.replay(game, hist)["board"], ou.replay(game, [int(perm[a]) for a in hist])["board"]
        assert np.array_equal(rboard, board[..., ::-1])
        bb = np.array([s.bitboards(), rs.bitboards()], dtype=np.uint64)
        planes = boards_from_bitboards(gid, rows, cols, bb, np.array([len(hist)] * 2))
        assert np.array_equal(planes[1], planes[0][..., ::-1])
        if not s.is_terminal():     # (the oracle's board marks a terminal position's player plane differently)
            assert np.array_equal(planes[0], board)
    assert n_terminal > 0


def test_cabi_reflect_flag_and_entry_points():
    from alphazero_openspiel_b200 import _lib as L
    lib = L.load()
    assert L.F_REFLECT == 1 << 16 and hasattr(lib, "az_observations_reflected") and hasattr(lib, "az_reflect_actions")
    for other, ev, name in ((L.F_MANUAL, L.EVAL_HASH, b"AZ_F_MANUAL"), (L.F_UCT, L.EVAL_HASH, b"AZ_F_UCT"),
                            (0, L.EVAL_ROLLOUT, b"AZ_EVAL_ROLLOUT")):
        cfg = L.AzConfig()
        cfg.game_id, cfg.n_trees, cfg.n_playouts, cfg.c_puct = 0, 4, 10, 2.5
        cfg.eval_mode = ev
        cfg.flags = L.F_REFLECT | other
        h = C.c_void_p()
        assert lib.az_create(C.byref(cfg), C.byref(h)) != 0
        assert b"AZ_F_REFLECT" in lib.az_last_error() and name in lib.az_last_error()


def test_restatement_reflects_evaluations():
    """The restatement's evaluator answers for R(s) on about half of the positions, and the restated games differ from the
    plain ones."""
    from oracle import pyspiel_shim
    g = pyspiel_shim.load_game(BT6)
    on, off = sr.Rule(BT6, 1, reflect=True, seed=5), sr.Rule(BT6, 1, seed=5)
    hits = total = 0
    for hist in _random_histories(BT6, 60, 4):
        s = g.new_initial_state()
        for a in hist:
            s.apply_action(a)
        if s.is_terminal():
            continue
        hits += sr.evaluate(on, s)[0] != sr.evaluate(off, s)[0]
        total += 1
    assert 0.3 * total < hits < 0.7 * total
    reflected = [sr.selfplay_game(sr.Rule(C4, 60, reflect=True, seed=5), t)[0] for t in range(4)]
    assert reflected != [sr.selfplay_game(sr.Rule(C4, 60, seed=5), t)[0] for t in range(4)]


def _trainer_pair(recs, **kw):
    import torch
    from alphazero_openspiel_b200.replay import ExampleBatch
    from alphazero_openspiel_b200.train import Trainer
    batch = ExampleBatch.from_records(recs, C4)
    merged = Trainer.remove_duplicates([ex for g in batch.to_games() for ex in g])
    first, pol, val = batch.remove_duplicates()
    torch.manual_seed(3)
    a = Trainer(device="cpu", batch_size=32, use_gpu=False, **kw)
    b = Trainer(device="cpu", batch_size=32, use_gpu=False, array_buffer=True, **kw)
    b.current_net.load_state_dict(a.current_net.state_dict())
    a.current_net.train()
    b.current_net.train()
    return a, b, merged, batch, first, pol, val


def _inputs(net):
    seen = []
    net.register_forward_pre_hook(lambda mod, args: seen.append(args[0].detach().clone()))
    return seen


def test_training_bits_leave_the_global_rng_alone():
    """The sample ids of net_step / net_step_arrays, and the RNG state after the step, are the same with the option on and
    off; the minibatch rows are mirrored exactly where replay.reflect_bits says so."""
    from alphazero_openspiel_b200.replay import reflect_bits
    recs = sr.oracle_records(n_games=9)
    boards = {}
    for on in (False, True):
        a, b, merged, batch, first, pol, val = _trainer_pair(recs, reflect_minibatches=on)
        seen_a, seen_b = _inputs(a.current_net), _inputs(b.current_net)
        states = []
        for step in range(3):
            np.random.seed(40 + step)
            a.net_step(merged)
            states.append(np.random.get_state()[1].copy())
            np.random.seed(40 + step)
            b.net_step_arrays(batch, first, pol, val)
            assert np.array_equal(np.random.get_state()[1], states[-1])
        boards[on] = (states, [x.numpy() for x in seen_a], [x.numpy() for x in seen_b])
    for k in range(3):
        assert np.array_equal(boards[False][0][k], boards[True][0][k])
        bits = reflect_bits(k, 32)
        assert 0 < bits.sum() < 32
        off, on = boards[False][2][k], boards[True][2][k]
        assert np.array_equal(on[bits], off[bits][..., ::-1]) and np.array_equal(on[~bits], off[~bits])


def test_list_and_array_paths_build_the_same_reflected_minibatch():
    """Same seeds, same buffer: the list buffer (net_step) and the array buffer (net_step_arrays) see the same mirrored
    boards, take the same losses and end with the same weights; the reflection changes the losses."""
    import torch
    recs = sr.oracle_records(n_games=9)
    losses = {}
    for on in (True, False):
        a, b, merged, batch, first, pol, val = _trainer_pair(recs, reflect_minibatches=on)
        seen_a, seen_b = _inputs(a.current_net), _inputs(b.current_net)
        out = []
        for step in range(3):
            np.random.seed(20 + step)
            la = a.net_step(merged)
            np.random.seed(20 + step)
            lb = b.net_step_arrays(batch, first, pol, val)
            assert float(la[0]) == float(lb[0]) and float(la[1]) == float(lb[1])
            assert torch.equal(seen_a[-1], seen_b[-1])
            out.append(float(la[0]))
        for x, y in zip(a.current_net.parameters(), b.current_net.parameters()):
            assert torch.equal(x, y)
        losses[on] = out
    assert losses[True] != losses[False]


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("game,n_trees,n_playouts", [(C4, 64, 100), (BT6, 16, 200), (BT8, 8, 120)])
@pytest.mark.parametrize("keep", [1, 0])
def test_selfplay_with_reflection_bit_exact(game, n_trees, n_playouts, keep):
    """Whole games with the hash evaluator: every ply record and every counter equal the restatement's, whose evaluator
    answers for R(s) whenever m(s)."""
    rule = sr.Rule(game, n_playouts, reflect=True, keep_tree=keep, seed=1234)
    recs, ctr = sr.engine_selfplay(rule, n_trees)
    sr.check_against_rule(recs, ctr, rule, n_trees)
    if game == C4 and keep:
        plain, _ = sr.engine_selfplay(sr.Rule(game, n_playouts, keep_tree=keep, seed=1234), n_trees)
        assert not (np.array_equal(plain["counts"], recs["counts"]) and np.array_equal(plain["action"], recs["action"]))


@pytest.mark.gpu
@pytest.mark.parametrize("game,n_trees,n_playouts", [(C4, 64, 100), (BT6, 16, 200)])
def test_reflection_with_playout_cap_forced_playouts_and_resignation(game, n_trees, n_playouts):
    rule = sr.Rule(game, n_playouts, resign=(0.0, 300), playout_cap=(n_playouts // 4, 250), forced=2.0, reflect=True,
                   keep_tree=1, seed=4321)
    recs, ctr = sr.engine_selfplay(rule, n_trees)
    ends, stats = sr.check_against_rule(recs, ctr, rule, n_trees)
    assert ends[1] > 0 and stats["forced"] > 0 and stats["pruned"] > 0
    plies = recs[recs["kind"] == 0]
    assert (plies["end"] == 3).any() and (plies["end"] == 0).any()


def _planes(game, bb, ply, obs_format, device):
    """az_observations of positions (bb uint64 [n, 2], ply [n]) in obs_format, as a device tensor."""
    import torch
    from alphazero_openspiel_b200 import _lib as L
    from alphazero_openspiel_b200.engine import parse_game_name
    gid, rows, cols = parse_game_name(game)
    n = len(ply)
    bb_d = torch.from_numpy(np.ascontiguousarray(bb, dtype=np.uint64).view(np.int64)).to(device)
    ply_d = torch.from_numpy(np.asarray(ply, dtype=np.int32)).to(device)
    shape = (n, rows, cols, 4) if obs_format == L.OBS_BF16_NHWC else (n, 4, rows, cols)
    out = torch.zeros(shape, dtype=torch.bfloat16 if obs_format == L.OBS_BF16_NHWC else torch.float32, device=device)
    st = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
    L.check(L.load().az_observations(gid, rows, cols, n, C.c_void_p(bb_d.data_ptr()), C.c_void_p(ply_d.data_ptr()), None,
                                     C.c_void_p(out.data_ptr()), obs_format, st))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("game", [C4, BT6])
@pytest.mark.parametrize("obs_format", [1, 2])
@pytest.mark.parametrize("vl", [0, 4])
def test_external_evaluator_rows_are_reflected(game, obs_format, vl):
    """AZ_EVAL_EXTERNAL with a deterministic, non-symmetric row function of the observation rows.  A requesting tree's row
    holds the planes of its position, columns flipped iff m(s); after the next step a freshly expanded root's priors are
    row[R(a)].  Exact kernel: every request, positions from az_request_info.  Virtual-loss kernel (4 leaves in flight):
    the root requests (a childless root is the first leaf of its search), positions from az_positions."""
    import torch
    from alphazero_openspiel_b200 import engine as E, _lib as L
    seed, n_trees = 21, 64
    # no tree reuse: every search expands a fresh root; sampled moves: the trees play different games
    flags = L.F_REFLECT | L.F_SAMPLE_MOVES | (L.F_VIRTUAL_LOSS if vl else 0)
    eng = E.Engine(game, n_trees, n_playouts=24, noise_mode=L.NOISE_NONE, eval_mode=L.EVAL_EXTERNAL, flags=flags, seed=seed,
                   leaves_per_tree=max(vl, 1))
    dev, K, A = eng.device, eng.rows_per_tree, eng.num_actions
    perm = E.reflect_actions(game)
    flip_dim = 2 if obs_format == L.OBS_BF16_NHWC else 3
    obs = eng.new_obs(obs_format)
    gen = torch.Generator().manual_seed(5)
    W = torch.rand((obs[0].numel(), A), generator=gen).to(dev)
    wv = (torch.rand(obs[0].numel(), generator=gen) - 0.5).to(dev)
    eng.step(None, None, None, obs, obs_format)
    n_rows = n_roots = n_flipped = 0
    for _ in range(40):
        ph = eng.status()["phase"]
        before = eng.root_stats(offpolicy=False)
        pos = eng.positions()
        if vl:
            req = [t for t in range(n_trees) if ph[t] == L.PH_LEAF_EVAL and before["n_children"][t] == 0]
            bb, ply = pos["bb"][req], pos["ply"][req]
        else:
            info = eng.request_info()
            req = [t for t in range(n_trees) if ph[t] in (L.PH_ROOT_EVAL, L.PH_LEAF_EVAL)]
            bb, ply = info["bb"][req], info["ply"][req]
        if req:
            want = _planes(game, bb, ply, obs_format, dev)
            flips = torch.tensor([sr.m(seed, int(b[0]), int(b[1]), int(p)) for b, p in zip(bb, ply)], device=dev)
            want = torch.where(flips.view(-1, 1, 1, 1), want.flip(flip_dim), want)
            assert torch.equal(obs[torch.tensor(req, device=dev) * K], want)
            n_rows += len(req)
            n_flipped += int(flips.sum())
        x = obs.reshape(obs.shape[0], -1).float()
        priors, values = (0.01 + x @ W).contiguous(), torch.tanh(x @ wv).contiguous()
        roots = [t for t in range(n_trees) if ph[t] == L.PH_LEAF_EVAL and before["n_children"][t] == 0]
        rows = priors.double().cpu().numpy()
        eng.step(priors, values, None, obs, obs_format)
        after, pos2 = eng.root_stats(offpolicy=False), eng.positions()
        for t in roots:
            if pos2["ply"][t] != pos["ply"][t] or not np.array_equal(pos2["bb"][t], pos["bb"][t]):
                continue                                             # the search ended in this step
            m = sr.m(seed, int(pos["bb"][t][0]), int(pos["bb"][t][1]), int(pos["ply"][t]))
            acts = after["child_action"][t, :after["n_children"][t]]
            cols_ = perm[acts] if m else acts
            assert np.array_equal(after["child_p"][t, :len(acts)], rows[t * K, cols_])
            n_roots += 1
    eng.close()
    assert n_rows > 100 and n_roots > 50 and 0 < n_flipped < n_rows


@pytest.mark.gpu
def test_eval_cache_with_reflection_gives_the_same_games():
    """Fused evaluator and the shipped Connect Four checkpoint: the same records with the evaluator cache on and off."""
    on, c_on = sr.runner_games(C4, 512, True, reflect_evaluations=True)
    off, c_off = sr.runner_games(C4, 512, False, reflect_evaluations=True)
    assert c_on["overflow"] == 0 and c_off["overflow"] == 0
    assert c_on["cache_hits"] > 0 and c_off["cache_hits"] == 0
    sr.same_records(on, off)


@pytest.mark.gpu
@pytest.mark.parametrize("game", [C4, BT6])
def test_reflected_gather_kernel(game):
    """az_observations_reflected: a null flag array gives az_observations bit for bit (both formats), flagged rows hold the
    planes with flipped columns; DeviceReplay.boards(ids, reflect) equals the numpy planes flipped on the same rows."""
    import torch
    from alphazero_openspiel_b200 import _lib as L
    from alphazero_openspiel_b200.device_replay import DeviceReplay
    from alphazero_openspiel_b200.engine import parse_game_name
    from alphazero_openspiel_b200.replay import ExampleBatch
    gid, rows, cols = parse_game_name(game)
    dev = torch.device("cuda:0")
    hist = _random_histories(game, 200, 9)
    bb = np.array([ou.replay(game, h)["bb"] for h in hist], dtype=np.uint64)
    ply = np.array([len(h) for h in hist], dtype=np.int32)
    flags = np.random.RandomState(1).rand(len(ply)) < 0.5
    bb_d = torch.from_numpy(bb.view(np.int64)).to(dev)
    ply_d = torch.from_numpy(ply).to(dev)
    flags_d = torch.from_numpy(flags.astype(np.uint8)).to(dev)
    for fmt in (L.OBS_F32_NCHW, L.OBS_BF16_NHWC):
        want = _planes(game, bb, ply, fmt, dev)
        for refl in (None, flags_d):
            got = torch.zeros_like(want)
            L.check(L.load().az_observations_reflected(gid, rows, cols, len(ply), C.c_void_p(bb_d.data_ptr()),
                                                       C.c_void_p(ply_d.data_ptr()), None,
                                                       None if refl is None else C.c_void_p(refl.data_ptr()),
                                                       C.c_void_p(got.data_ptr()), fmt, None))
            torch.cuda.synchronize()
            if refl is None:
                assert torch.equal(got, want)
            else:
                flip = torch.from_numpy(flags).to(dev).view(-1, 1, 1, 1)
                assert torch.equal(got, torch.where(flip, want.flip(2 if fmt == L.OBS_BF16_NHWC else 3), want))
    if game == C4:
        batch = ExampleBatch.from_records(sr.oracle_records(n_games=6, playouts=15, seed=4), C4)
        rb = DeviceReplay(C4, "cuda:0")
        rb.append(batch)
        rng = np.random.RandomState(2)
        ids = rng.randint(len(rb), size=300)
        fl = rng.rand(300) < 0.5
        got = rb.boards(torch.from_numpy(ids).to(dev), torch.from_numpy(fl).to(dev)).cpu().numpy()
        host = batch.boards(ids)
        host[fl] = host[fl][..., ::-1]
        assert np.array_equal(got.astype(np.float64), host)


@pytest.mark.gpu
def test_reflected_minibatches_take_the_same_steps_on_every_path():
    """Trainer(reflect_minibatches=True): the array, eager device and graphed device paths take the same optimisation steps
    (tolerances of tests/test_trainer.py::test_device_replay_matches_the_array_buffer)."""
    import torch
    from alphazero_openspiel_b200.device_replay import DeviceReplay
    from alphazero_openspiel_b200.replay import ExampleBatch
    from alphazero_openspiel_b200.train import Trainer
    recs = sr.oracle_records(n_games=12, playouts=15, seed=4)
    losses = {}
    for mode in ("array", "device", "graph", "array_plain"):
        torch.manual_seed(3)
        tr = Trainer(device="cuda:0", batch_size=64, array_buffer=True, device_training=mode in ("device", "graph"),
                     graph_step=mode == "graph", reflect_minibatches=mode != "array_plain")
        np.random.seed(8)
        if mode in ("device", "graph"):
            tr.dbuffer = DeviceReplay(C4, "cuda:0")
            tr.dbuffer.append(ExampleBatch.from_records(recs, C4))
            first, pol, val = tr.dbuffer.remove_duplicates()
            tr.current_net.train()
            out = [tr.net_step_device(tr.dbuffer, first, pol, val) for _ in range(4)]
        else:
            tr.abuffer = ExampleBatch.from_records(recs, C4)
            first, pol, val = tr.abuffer.remove_duplicates()
            tr.current_net.train()
            out = [tr.net_step_arrays(tr.abuffer, first, pol, val) for _ in range(4)]
        losses[mode] = [(float(a), float(b)) for a, b in out]
    for other in ("device", "graph"):
        for k, ((pa, va), (pd, vd)) in enumerate(zip(losses["array"], losses[other])):
            tol = 1e-4 if k < 2 else 2e-3
            assert abs(pa - pd) < tol * max(1.0, abs(pa)) and abs(va - vd) < tol * max(1.0, abs(va)), (other, k, losses)
    assert losses["array"][0][0] != losses["array_plain"][0][0]


@pytest.mark.gpu
def test_trainer_with_both_reflections_end_to_end():
    from alphazero_openspiel_b200.train import Trainer
    tr = Trainer(device="cuda:0", n_games_per_generation=32, n_batches_per_generation=10, batch_size=64, n_playouts_train=10,
                 device_training=True, graph_step=True, reflect_minibatches=True, reflect_evaluations=True, save=False)
    for gen in range(2):
        tr.generation += 1
        tr.generate_examples(tr.n_games_per_generation, seed=gen + 1)
        assert tr.last_generation_stats["overflow"] == 0 and tr.last_generation_stats["games"] == 32
        tr.train_network()
    assert tr.it == 20 and tr.dbuffer.n_games == 64
