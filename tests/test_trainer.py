"""Trainer drop-in (SURVEY 8(f) rank 1): CPU parity of remove_duplicates / net_step with the oracle's restatement of
train.py (and with what the reference's own remove_duplicates returns, tests/golden/reference_crosscheck.json); GPU
end-to-end generations."""
import copy
import json
import os

import numpy as np
import pytest
import torch

from tests import selfplay_rule as sr


def _fake_buffer(rng, n=300, n_keys=60, A=7):
    flat = []
    for _ in range(n):
        k = int(rng.randint(n_keys))
        pol = rng.dirichlet(np.ones(A)).tolist() if rng.rand() > 0.1 else []
        flat.append([str(k), rng.rand(4, 6, 7), pol, float(rng.choice([-1.0, 0.0, 1.0]))])
    return flat


def test_remove_duplicates_matches_oracle_and_reference():
    from alphazero_openspiel_b200.train import Trainer
    from oracle import ref_port
    rng = np.random.RandomState(0)
    buf = _fake_buffer(rng)
    a = Trainer.remove_duplicates(copy.deepcopy(buf))
    b = ref_port.dedupe_examples(copy.deepcopy(buf))
    assert len(a) == len(b) <= 60
    for x, y in zip(a, b):
        assert x[0] == y[0] and x[2] == y[2] and x[3] == y[3] and np.array_equal(x[1], y[1])
    # in-place accumulation quirk: the first example of every key is the returned (mutated) object
    mine = copy.deepcopy(buf)
    out = Trainer.remove_duplicates(mine)
    firsts = {}
    for ex in mine:
        firsts.setdefault(ex[0], ex)
    assert all(o is firsts[o[0]] for o in out)
    # what the reference's own Trainer.remove_duplicates returns for this buffer (tests/golden/make_golden_crosscheck.py)
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_crosscheck.json")) as f:
        c = json.load(f)["remove_duplicates"]
    assert [x[0] for x in a] == c["keys"]
    assert [x[2] for x in a] == c["policies"] and [x[3] for x in a] == c["values"]


def test_net_step_matches_oracle_restatement_on_cpu():
    """Same seed, same buffer, same initial weights: losses and updated weights are identical (fp32, CPU)."""
    from alphazero_openspiel_b200.train import Trainer
    from oracle import ref_port, ref_net
    rng = np.random.RandomState(1)
    buf = _fake_buffer(rng, n=400, n_keys=400)
    torch.manual_seed(5)
    tr = Trainer(device="cpu", batch_size=32, use_gpu=False)
    ref = ref_net.RefNet([3, 6, 7], 7)
    ref.load_state_dict(tr.current_net.state_dict())
    opt = torch.optim.Adam(ref.parameters(), lr=0.001, weight_decay=0.0001)
    tr.current_net.train()
    ref.train()
    for step in range(3):
        np.random.seed(100 + step)
        lp, lv = tr.net_step(buf)
        np.random.seed(100 + step)
        rp, rv = ref_port.train_step(ref, opt, buf, 32)
        assert float(lp) == float(rp) and float(lv) == float(rv)
    for (ka, va), (kb, vb) in zip(tr.current_net.state_dict().items(), ref.state_dict().items()):
        assert ka == kb and torch.equal(va, vb)
    assert tr.it == 3


def test_update_buffer_size_schedule():
    from alphazero_openspiel_b200.train import Trainer
    tr = Trainer(device="cpu", use_gpu=False, n_games_per_generation=10, n_games_buffer_max=60)
    assert tr.n_games_buffer == 40
    sizes = []
    for g in range(1, 8):
        tr.generation = g
        tr.update_buffer_size()
        sizes.append(tr.n_games_buffer)
    assert sizes == [40, 50, 50, 60, 60, 60, 60]  # grows every second generation up to the cap (train.py:295-298)


@pytest.mark.gpu
def test_trainer_generations_end_to_end():
    """Two tiny generations on the GPU: games enter the FIFO buffer, the network trains, weights change."""
    from alphazero_openspiel_b200.train import Trainer
    torch.manual_seed(0)
    np.random.seed(0)
    tr = Trainer(n_games_per_generation=24, n_batches_per_generation=6, batch_size=32, n_playouts_train=20,
                 n_generations=2, backup="soft-Z")
    before = copy.deepcopy(tr.current_net.state_dict())
    tr.run(n_trees=24, seed=11)
    assert tr.generation == 2 and len(tr.buffer) == 48 and tr.it == 12
    assert all(len(g) >= 7 for g in tr.buffer)
    after = tr.current_net.state_dict()
    assert any(not torch.equal(before[k].cpu(), after[k].cpu()) for k in before if "weight" in k)
    assert all(torch.isfinite(v).all() for v in after.values())
    assert tr.last_generation_stats["overflow"] == 0 and not tr.current_net.training


@pytest.mark.gpu
def test_array_buffer_generations_match_the_list_buffer():
    """Trainer(array_buffer=True): the same two generations as the list-buffer Trainer from the same seeds -- same games in
    the buffer (device self-play is deterministic for a seed), same number of optimisation steps."""
    from alphazero_openspiel_b200.train import Trainer
    nets = []
    for array_buffer in (False, True):
        torch.manual_seed(0)
        np.random.seed(0)
        tr = Trainer(n_games_per_generation=24, n_batches_per_generation=6, batch_size=32, n_playouts_train=20,
                     n_generations=2, backup="on-policy", array_buffer=array_buffer)
        tr.run(n_trees=24, seed=11)
        assert tr.generation == 2 and tr.it == 12
        if array_buffer:
            assert tr.abuffer.n_games == 48 and tr.buffer == []
            games = tr.abuffer.to_games()
        else:
            games = tr.buffer
        # generation 1's games are identical (same initial weights, same seed); their targets are not compared because
        # remove_duplicates has merged them in place with generation 2's, which depends on the (noisy) GPU training
        nets.append((copy.deepcopy(tr.current_net.state_dict()), [[ex[0] for ex in g] for g in games[:24]]))
    assert nets[0][1] == nets[1][1]
    # (cuDNN's backward kernels are not bit-reproducible from run to run on the GPU, and Adam amplifies the last-bit
    # differences: the CPU test below pins the array path bit for bit; here both trainings must simply have happened)
    for sd, _ in nets:
        assert all(torch.isfinite(v.float()).all() for v in sd.values())


def test_example_batch_is_a_lossless_form_of_the_reference_examples():
    """replay.ExampleBatch (SURVEY 8(f) rank 3): from_records + to_games == records_to_games for every value target;
    concat / last_games follow the buffer list semantics."""
    from alphazero_openspiel_b200.examplegenerator import records_to_games
    from alphazero_openspiel_b200.replay import ExampleBatch
    recs = sr.oracle_records()
    for backup in ["on-policy", "soft-Z", "A0C", "off-policy"]:
        want = records_to_games(recs, "connect_four", backup)
        b = ExampleBatch.from_records(recs, "connect_four", backup)
        got = b.to_games()
        assert b.n_games == len(want) == 6 and len(b) == sum(len(g) for g in want)
        for gw, gg in zip(want, got):
            assert len(gw) == len(gg)
            for x, y in zip(gw, gg):
                assert x[0] == y[0] and np.array_equal(x[1], y[1]) and x[2] == y[2] and x[3] == y[3]
    b = ExampleBatch.from_records(recs, "connect_four")
    two = ExampleBatch.concat([b, b])
    assert two.n_games == 12 and len(two) == 2 * len(b)
    tail = two.last_games(5)
    assert tail.n_games == 5
    for gx, gy in zip(tail.to_games(), two.to_games()[-5:]):
        assert len(gx) == len(gy)
        assert all(x[0] == y[0] and np.array_equal(x[1], y[1]) and x[2] == y[2] and x[3] == y[3] for x, y in zip(gx, gy))
    assert ExampleBatch.from_records(recs[recs["kind"] == 0], "connect_four").n_games == 0   # unfinished games dropped


def test_array_remove_duplicates_and_net_step_match_the_list_path():
    """Same merged examples (order, averaged targets bit-equal, first example of a key updated in place) and, from the same
    seeds and initial weights, the same losses and weights after a few optimisation steps."""
    from alphazero_openspiel_b200.replay import ExampleBatch
    from alphazero_openspiel_b200.train import Trainer
    recs = sr.oracle_records(n_games=9)
    batch = ExampleBatch.from_records(recs, "connect_four")
    games = batch.to_games()
    flat = [ex for g in games for ex in g]
    merged = Trainer.remove_duplicates(flat)
    first, pol, val = batch.remove_duplicates()
    assert len(merged) == len(first) < len(flat)                    # the oracle games share their opening positions
    for m, i, p, v in zip(merged, first, pol, val):
        assert m[0] == batch.key(i) and m[2] == p.tolist() and m[3] == v
        assert m is flat[i]                                          # reference: the first example IS the accumulator
        assert batch.policy[i].tolist() == m[2] and batch.value[i] == m[3]
    torch.manual_seed(3)
    a = Trainer(device="cpu", batch_size=16, use_gpu=False)
    b = Trainer(device="cpu", batch_size=16, use_gpu=False, array_buffer=True)
    b.current_net.load_state_dict(a.current_net.state_dict())
    a.current_net.train()
    b.current_net.train()
    for step in range(3):
        np.random.seed(20 + step)
        la = a.net_step(merged)
        np.random.seed(20 + step)
        lb = b.net_step_arrays(batch, first, pol, val)
        assert float(la[0]) == float(lb[0]) and float(la[1]) == float(lb[1])
    for x, y in zip(a.current_net.parameters(), b.current_net.parameters()):
        assert torch.equal(x, y)


def test_random_start_games_get_signs_from_the_ply_and_keys_from_the_start_position():
    """ADVICE r01 (medium): with random_start_mod > 0 a game may begin with player 1 to move and has no action history for
    its first plies.  The on-policy value is returns()[0] for player 0 to move and its negation for player 1
    (game_utils.py:168-169,200-204) -- from the position's real ply -- and the de-duplication key carries the start
    position so that different positions never share a key.  Both example forms agree."""
    from alphazero_openspiel_b200.examplegenerator import records_to_games
    from alphazero_openspiel_b200.replay import ExampleBatch
    recs = sr.oracle_records(n_games=12, start_mod=9, seed=3)
    games = records_to_games(recs, "connect_four", "on-policy")
    batch = ExampleBatch.from_records(recs, "connect_four", "on-policy")
    assert len(games) == 12 and batch.n_games == 12
    odd_starts = 0
    keys = set()
    for g, gb in zip(games, batch.to_games()):
        ret0 = None
        for ex, exb in zip(g, gb):
            board = ex[1]
            player = int(board[3, 0, 0])                     # current-player plane (network.py:16-17)
            n_pieces = int(board[1].sum() + board[2].sum())
            assert player == n_pieces % 2
            if ret0 is None:
                ret0 = ex[3] if player == 0 else -ex[3]
                odd_starts += player
                assert (n_pieces == 0) == (not ex[0].startswith("start="))
            assert ex[3] == (ret0 if player == 0 else -ret0)
            assert ex[0] == exb[0] and ex[3] == exb[3] and np.array_equal(ex[1], exb[1])
            keys.add((ex[0], board.tobytes()))
    assert odd_starts > 0                                    # the case the old index-based sign got wrong
    # one key never names two different positions
    assert len({k for k, _ in keys}) == len(keys)
    first, _, _ = batch.remove_duplicates()
    assert len(first) == len({k for k, _ in keys})


@pytest.mark.gpu
def test_device_replay_matches_the_array_buffer():
    """device_replay.DeviceReplay (SURVEY 8(f) ranks 1 + 3): duplicates merged on the device equal ExampleBatch.remove_duplicates
    (same first-occurrence order, averaged targets within 1e-12), the az_observations gather kernel reproduces
    state_to_board (network.py:9-18) bit for bit, and Trainer(device_training=True) takes the same optimisation steps as
    the host array path from the same seeds (same sample ids -> same minibatches; fp32 losses agree to 1e-5)."""
    from alphazero_openspiel_b200.device_replay import DeviceReplay
    from alphazero_openspiel_b200.replay import ExampleBatch
    from alphazero_openspiel_b200.train import Trainer
    recs = sr.oracle_records(n_games=12, playouts=15, seed=4)
    host = ExampleBatch.concat([ExampleBatch.from_records(recs, "connect_four"), ExampleBatch.from_records(recs, "connect_four")])
    dev = DeviceReplay("connect_four", "cuda:0")
    dev.append(ExampleBatch.from_records(recs, "connect_four"))
    dev.append(ExampleBatch.from_records(recs, "connect_four"))
    assert len(dev) == len(host) and dev.n_games == host.n_games == 24
    import copy as _copy
    f_h, p_h, v_h = _copy.deepcopy(host).remove_duplicates()
    f_d, p_d, v_d = dev.remove_duplicates()
    assert np.array_equal(f_d.cpu().numpy(), f_h)
    assert np.abs(p_d.cpu().numpy() - p_h).max() < 1e-12 and np.abs(v_d.cpu().numpy() - v_h).max() < 1e-12
    ids = torch.arange(len(dev), device="cuda:0")
    assert np.array_equal(dev.boards(ids).cpu().numpy().astype(np.float64), host.boards())
    dev.keep_last_games(5)
    assert dev.n_games == 5 and len(dev) == len(host.last_games(5))
    # same optimisation steps from the same seeds
    losses = {}
    for mode in ("array", "device"):
        torch.manual_seed(3)
        tr = Trainer(device="cuda:0", batch_size=64, array_buffer=True, device_training=(mode == "device"))
        np.random.seed(8)
        if mode == "device":
            tr.dbuffer = DeviceReplay("connect_four", "cuda:0")
            tr.dbuffer.append(ExampleBatch.from_records(recs, "connect_four"))
            first, pol, val = tr.dbuffer.remove_duplicates()
            tr.current_net.train()
            out = [tr.net_step_device(tr.dbuffer, first, pol, val) for _ in range(4)]
        else:
            tr.abuffer = ExampleBatch.from_records(recs, "connect_four")
            first, pol, val = tr.abuffer.remove_duplicates()
            tr.current_net.train()
            out = [tr.net_step_arrays(tr.abuffer, first, pol, val) for _ in range(4)]
        losses[mode] = [(float(a), float(b)) for a, b in out]
    # fp32 training on the GPU: the first steps agree to 1e-4, later ones drift apart slowly (non-deterministic cuDNN
    # reductions, last-bit differences of the device-summed targets) -- bounded at 2e-3 over four steps
    for k, ((pa, va), (pd, vd)) in enumerate(zip(losses["array"], losses["device"])):
        tol = 1e-4 if k < 2 else 2e-3
        assert abs(pa - pd) < tol * max(1.0, abs(pa)) and abs(va - vd) < tol * max(1.0, abs(va)), (k, losses)
    # the whole optimisation step as one CUDA graph (Trainer(graph_step=True)): same losses as the eager device steps
    torch.manual_seed(3)
    tg = Trainer(device="cuda:0", batch_size=64, device_training=True, graph_step=True)
    np.random.seed(8)
    tg.dbuffer = DeviceReplay("connect_four", "cuda:0")
    tg.dbuffer.append(ExampleBatch.from_records(recs, "connect_four"))
    first, pol, val = tg.dbuffer.remove_duplicates()
    tg.current_net.train()
    got = [tuple(float(t) for t in tg.net_step_device(tg.dbuffer, first, pol, val)) for _ in range(4)]
    assert tg.it == 4
    for k, ((pd, vd), (pg, vg)) in enumerate(zip(losses["device"], got)):
        tol = 1e-4 if k < 2 else 2e-3
        assert abs(pg - pd) < tol * max(1.0, abs(pd)) and abs(vg - vd) < tol * max(1.0, abs(vd)), (k, losses["device"], got)
    # whole generations through Trainer.run's pieces
    tr = Trainer(device="cuda:0", n_games_per_generation=32, n_batches_per_generation=10, batch_size=64, n_playouts_train=10,
                 device_training=True, save=False)
    tr.generation += 1
    tr.generate_examples(tr.n_games_per_generation)
    tr.train_network()
    assert tr.dbuffer.n_games == 32 and tr.it == 10


def test_device_replay_key_hash_groups_like_the_reference_keys():
    """device_replay.key_hash (host part of the device buffer): two examples get the same 64-bit hash exactly when the
    reference's info-state keys (action history; plus the start position of random-start games) are equal."""
    from alphazero_openspiel_b200.device_replay import key_hash
    from alphazero_openspiel_b200.replay import ExampleBatch
    for start_mod in (0, 9):
        recs = sr.oracle_records(n_games=12, start_mod=start_mod, seed=3)
        b = ExampleBatch.concat([ExampleBatch.from_records(recs, "connect_four")] * 2)
        h = key_hash(b)
        keys = [b.key(i) for i in range(len(b))]
        by_key, by_hash = {}, {}
        for i, (k, x) in enumerate(zip(keys, h.tolist())):
            by_key.setdefault(k, []).append(i)
            by_hash.setdefault(x, []).append(i)
        assert sorted(by_key.values()) == sorted(by_hash.values())
        assert len(by_key) < len(b)          # duplicates exist (every game appears twice)
