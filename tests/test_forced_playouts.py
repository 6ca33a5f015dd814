"""Forced playouts and policy target pruning in batched self-play (AZ_F_FORCED_PLAYOUTS): the rule as tests/selfplay_rule.py
restates it on top of the reference port's search, the conversion of pruned records into training examples, and on the GPU
the engine against the restatement and through the Python layers."""
import ctypes as C
import math

import numpy as np
import pytest

from tests import oracle_util as ou
from tests import selfplay_rule as sr
from tests.selfplay_rule import BT6, BT8, C4


def _non_best_ones(counts):
    """Entries other than the first maximum that equal 1."""
    star = int(np.argmax(counts))
    return sum(1 for i, c in enumerate(counts) if i != star and c == 1)


# ---------------------------------------------------------------------------------------------------------------- CPU
def _roots():
    """Hand-built roots (counts, q, prior, N_root) that reach every branch of the pruning rule."""
    rng = np.random.RandomState(7)
    roots = [
        # a child with many forced visits and a low Q; a 1-visit child; an unvisited child
        ([60, 12, 1, 0, 27], [0.1, -0.6, -0.9, 0.0, 0.05], [0.3, 0.25, 0.05, 0.1, 0.3], 101),
        # a child with a high Q: its PUCT at N - 1 is above c*'s, so it keeps its count
        ([40, 30, 10], [0.0, 0.9, -0.2], [0.2, 0.2, 0.6], 81),
        # equal counts: the first is c*
        ([20, 20, 5], [0.0, -0.1, -0.5], [0.4, 0.4, 0.2], 46),
    ]
    for _ in range(300):
        n = rng.randint(2, 12)
        prior = rng.dirichlet(np.ones(n) * 0.5).tolist()
        counts = rng.multinomial(rng.randint(1, 800), rng.dirichlet(np.ones(n))).tolist()
        q = rng.uniform(-1, 1, n).tolist()
        roots.append((counts, q, prior, sum(counts) + rng.randint(0, 2)))
    return roots


def test_prune_on_hand_built_roots():
    rule = sr.Rule(C4, 100, forced=2.0)
    c_puct = rule.cfg.c_puct
    reduced = high_q_kept = ones_dropped = 0
    for counts, q, prior, n_root in _roots():
        out = rule.prune(counts, q, prior, n_root)
        star = int(np.argmax(counts))
        sq = math.sqrt(n_root)
        s_star = q[star] + c_puct * prior[star] * sq / (counts[star] + 1)
        assert out[star] == counts[star]
        assert int(np.argmax(out)) == star
        for i, (n_c, n) in enumerate(zip(counts, out)):
            assert 0 <= n <= n_c
            if i == star:
                continue
            if n == 0 and n_c > 0 and (n_c == 1 or n_c - rule.floor(prior[i], n_root) <= 1):
                ones_dropped += n_c == 1 or n != n_c
                continue  # a remainder of 1 went to 0
            assert n >= n_c - rule.floor(prior[i], n_root)
            assert n != 1
            if n < n_c:
                reduced += 1
                # the child's PUCT at its pruned count stays below c*'s
                assert q[i] + c_puct * prior[i] * sq / (n + 1) < s_star
            elif n_c > 1 and q[i] + c_puct * prior[i] * sq / n_c >= s_star:
                high_q_kept += 1
    first = rule.prune(*_roots()[0])
    assert first[0] == 60 and first[1] < 12 and first[2] == 0 and first[3] == 0
    assert rule.prune(*_roots()[1])[1] == 30
    assert reduced > 50 and high_q_kept > 10 and ones_dropped > 10


@pytest.mark.parametrize("game,n_games,n_playouts", [(C4, 16, 100), (BT6, 4, 200)])
def test_restated_games_force_and_prune(game, n_games, n_playouts):
    """With k = 2 the restated games do force selections and prune counts, and no non-best count is 1."""
    rule = sr.Rule(game, n_playouts, forced=2.0, seed=5)
    stats = {}
    for t in range(n_games):
        plies, _, _ = sr.selfplay_game(rule, t, stats=stats)
        for p in plies:
            assert _non_best_ones(p["counts"]) == 0
            assert sum(p["counts"]) <= p["root_n"]
    assert stats["forced"] > 0 and stats["pruned"] > 0


def test_pruned_targets_become_the_examples():
    """records_to_games: the policy targets of the examples are the pruned counts normalised; no non-best entry is 1/sum."""
    from alphazero_openspiel_b200.examplegenerator import records_to_games
    rule = sr.Rule(C4, 60, forced=2.0, seed=3)
    games = [(t, *sr.selfplay_game(rule, t)[:2], 0) for t in range(8)]
    lists = records_to_games(sr.records(C4, games), C4)
    assert len(lists) == len(games)
    n_pruned_rows = 0
    for ex_list, (_, plies, _, _) in zip(lists, games):
        assert len(ex_list) == len(plies)
        hist = []
        for ex, p in zip(ex_list, plies):
            legal = ou.replay(C4, hist)["legal"]
            pol = np.asarray(ex[2], dtype=np.float64)
            total = sum(p["counts"])
            want = np.array(p["counts"], dtype=np.float64) / total
            assert np.allclose(pol[legal], want / want.sum(), rtol=0, atol=1e-15)
            star = int(np.argmax(p["counts"]))
            for i, a in enumerate(legal):
                if i != star:
                    assert pol[a] != 1.0 / total
            n_pruned_rows += total < p["root_n"] - 1
            hist.append(p["action"])
    assert n_pruned_rows > 0


def test_cabi_forced_playouts_flag_and_entry_point():
    from alphazero_openspiel_b200 import _lib as L
    lib = L.load()
    assert hasattr(lib, "az_set_forced_playouts") and L.F_FORCED_PLAYOUTS == 1 << 15
    for other, noise, name in ((L.F_MANUAL, L.NOISE_COUNTER, b"AZ_F_MANUAL"), (L.F_UCT, L.NOISE_COUNTER, b"AZ_F_UCT"),
                               (0, L.NOISE_NONE, b"AZ_NOISE_NONE")):
        cfg = L.AzConfig()
        cfg.game_id, cfg.n_trees, cfg.n_playouts, cfg.c_puct = 0, 4, 10, 2.5
        cfg.noise_mode = noise
        cfg.flags = L.F_FORCED_PLAYOUTS | other
        h = C.c_void_p()
        assert lib.az_create(C.byref(cfg), C.byref(h)) != 0
        assert b"AZ_F_FORCED_PLAYOUTS" in lib.az_last_error() and name in lib.az_last_error()
    assert lib.az_set_forced_playouts(None, 2.0, None) != 0 and b"null engine" in lib.az_last_error()


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("game,n_trees,n_playouts", [(C4, 64, 100), (BT6, 16, 200), (BT8, 8, 120)])
@pytest.mark.parametrize("keep", [1, 0])
def test_selfplay_with_forced_playouts_bit_exact(game, n_trees, n_playouts, keep):
    """Whole games with k = 2: every ply record and every counter equal the restatement's, which forces and prunes."""
    rule = sr.Rule(game, n_playouts, forced=2.0, keep_tree=keep, seed=1234)
    recs, ctr = sr.engine_selfplay(rule, n_trees)
    _, stats = sr.check_against_rule(recs, ctr, rule, n_trees)
    assert stats["forced"] > 0 and stats["pruned"] > 0
    if game == C4 and keep:
        # a per-step simulation cap, by count or by SM cycles, changes no record
        for cap, budget in ((1, 0), (0, 20000)):
            r2, c2 = sr.engine_selfplay(rule, n_trees, max_sims_per_step=cap, step_cycle_budget=budget)
            sr.same_records(r2, recs)
            assert all(c2[k] == ctr[k] for k in ("sims", "moves", "games", "root_evals"))


@pytest.mark.gpu
@pytest.mark.parametrize("game,n_trees,n_playouts", [(C4, 64, 100), (BT6, 16, 200)])
def test_forced_playouts_with_playout_cap(game, n_trees, n_playouts):
    """25 % full searches, fast = N/4: only the full searches are forced and pruned."""
    rule = sr.Rule(game, n_playouts, playout_cap=(n_playouts // 4, 250), forced=2.0, seed=4242)
    recs, ctr = sr.engine_selfplay(rule, n_trees)
    _, stats = sr.check_against_rule(recs, ctr, rule, n_trees)
    assert stats["forced"] > 0 and stats["pruned"] > 0
    plies = recs[recs["kind"] == 0]
    assert (plies["end"] == 3).any() and (plies["end"] == 0).any()


@pytest.mark.gpu
@pytest.mark.parametrize("game,n_trees,n_playouts", [(C4, 64, 100), (BT6, 16, 200)])
def test_forced_playouts_with_resignation(game, n_trees, n_playouts):
    rule = sr.Rule(game, n_playouts, resign=(0.0, 300), forced=2.0, keep_tree=1, seed=4321)
    recs, ctr = sr.engine_selfplay(rule, n_trees)
    ends, _ = sr.check_against_rule(recs, ctr, rule, n_trees)
    assert ends[1] * 5 >= n_trees


@pytest.mark.gpu
def test_flag_alone_changes_nothing():
    """AZ_F_FORCED_PLAYOUTS without an az_set_forced_playouts call (k = 0): the records and counters are the plain engine's."""
    from alphazero_openspiel_b200 import _lib as L
    plain = sr.Rule(C4, 100, seed=77)
    on, c_on = sr.engine_selfplay(plain, 64, L.F_FORCED_PLAYOUTS)
    off, c_off = sr.engine_selfplay(plain, 64)
    sr.same_records(on, off)
    assert c_on == c_off


@pytest.mark.gpu
def test_set_forced_playouts_rejects_bad_arguments():
    from alphazero_openspiel_b200 import engine as E, _lib as L
    plain = E.Engine(C4, 4, n_playouts=40, flags=L.F_RECORDS, noise_mode=L.NOISE_COUNTER)
    with pytest.raises(RuntimeError, match="without AZ_F_FORCED_PLAYOUTS"):
        plain.set_forced_playouts(2.0)
    plain.close()
    eng = E.Engine(C4, 4, n_playouts=40, flags=L.F_RECORDS | L.F_FORCED_PLAYOUTS, noise_mode=L.NOISE_COUNTER)
    for k in (-1.0, float("nan"), float("inf")):
        with pytest.raises(RuntimeError, match="finite and >= 0"):
            eng.set_forced_playouts(k)
    eng.set_forced_playouts(0.0)
    eng.set_forced_playouts(2.0)
    eng.close()


@pytest.mark.gpu
def test_new_k_reaches_a_captured_graph():
    """az_set_forced_playouts on a runner whose round trip is already captured: after a drain-and-discard window longer
    than one search, every record is pruned (no non-best count of 1)."""
    from alphazero_openspiel_b200.examplegenerator import SelfPlayRunner
    n_playouts = 40
    r = SelfPlayRunner(sr.net(C4), C4, "cuda:0", 256, n_playouts=n_playouts, seed=3, forced_playouts=0.0)
    r.round(100)
    assert r._graph is not None
    before = r.drain()
    plies = before[before["kind"] == 0]
    assert len(plies) > 0
    assert sum(_non_best_ones(list(p["counts"][:p["n_legal"]])) for p in plies) > 0
    r.set_forced_playouts(2.0)
    r.round(3 * n_playouts)  # every search that began before the call has finished
    r.drain()
    r.round(200)
    after = r.drain()
    ctr = r.counters()
    r.close()
    plies = after[after["kind"] == 0]
    assert len(plies) > 0 and ctr["overflow"] == 0
    assert sum(_non_best_ones(list(p["counts"][:p["n_legal"]])) for p in plies) == 0


@pytest.mark.gpu
def test_eval_cache_with_forced_playouts_gives_the_same_games():
    """Fused evaluator and the shipped Connect Four checkpoint: the same records with the evaluator cache on and off."""
    on, c_on = sr.runner_games(C4, 512, True, forced_playouts=2.0)
    off, c_off = sr.runner_games(C4, 512, False, forced_playouts=2.0)
    assert c_on["overflow"] == 0 and c_off["overflow"] == 0
    assert c_on["cache_hits"] > 0 and c_off["cache_hits"] == 0
    sr.same_records(on, off)


@pytest.mark.gpu
def test_virtual_loss_mode_with_forced_playouts():
    """K = 4 leaves in flight: games finish, every record's counts sum to at most root_n and no non-best count is 1."""
    from alphazero_openspiel_b200 import _lib as L
    n_trees = 32
    recs, ctr = sr.engine_selfplay(sr.Rule(C4, 40, forced=2.0, seed=5), n_trees, L.F_VIRTUAL_LOSS, leaves_per_tree=4)
    assert int((recs["kind"] == 1).sum()) == n_trees and ctr["overflow"] == 0
    plies = recs[recs["kind"] == 0]
    pruned = 0
    for p in plies:
        counts = list(p["counts"][:p["n_legal"]])
        assert sum(counts) <= p["root_n"] and _non_best_ones(counts) == 0
        pruned += sum(counts) < p["root_n"] - 1
    assert pruned > 0


def _assert_pruned_examples(recs):
    plies = recs[recs["kind"] == 0]
    assert len(plies) > 0
    assert sum(_non_best_ones(list(p["counts"][:p["n_legal"]])) for p in plies) == 0
    assert int((plies["counts"].sum(axis=1) < plies["root_n"] - 1).sum()) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("game", [C4, BT6])
def test_example_generator_with_forced_playouts(game):
    from alphazero_openspiel_b200.examplegenerator import ExampleGenerator, records_to_games
    n_trees, n_games = 128, 256
    gen = ExampleGenerator(sr.net(game), game, "cuda:0", n_trees=n_trees, n_playouts=40, seed=11, forced_playouts=2.0)
    recs, stats = gen._play(n_games)
    assert stats["overflow"] == 0 and stats["games"] == n_games
    _assert_pruned_examples(recs)
    games = records_to_games(recs, game)
    assert len(games) == n_games and sum(len(g) for g in games) == stats["moves"]


@pytest.mark.gpu
def test_trainer_with_forced_playouts():
    from alphazero_openspiel_b200.train import Trainer
    tr = Trainer(name_game=C4, forced_playouts=2.0, n_games_per_generation=64, n_playouts_train=20, save=False)
    for seed in (1, 2):
        n_before = sum(len(g) for g in tr.buffer)
        tr.generate_examples(64, seed=seed)
        s = tr.last_generation_stats
        assert s["games"] == 64 and s["overflow"] == 0
        assert sum(len(g) for g in tr.buffer) - n_before == s["moves"]
