"""Playout cap randomization in batched self-play (AZ_F_PLAYOUT_CAP): the self-play restatement of tests/selfplay_rule.py
against the C oracle's game, the per-search decision in it, the conversion of records with fast searches into training
examples, and on the GPU the engine against the restatement and through the Python layers."""
import ctypes as C

import numpy as np
import pytest

from tests import oracle_util as ou
from tests import selfplay_rule as sr
from tests.selfplay_rule import BT6, BT8, C4


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("keep", [1, 0])
@pytest.mark.parametrize("game,n_games,n_playouts,noise,k", [
    pytest.param(C4, 32, 100, 2, None, id="connect_four-32-100-2"),
    pytest.param(C4, 8, 60, 0, None, id="connect_four-8-60-0"),
    pytest.param(BT6, 8, 200, 2, None, id="breakthrough(rows=6,columns=6)-8-200-2"),
    pytest.param(C4, 16, 100, 2, 0.0, id="connect_four-16-100-2-k0"),
    pytest.param(BT6, 4, 200, 2, 0.0, id="breakthrough(rows=6,columns=6)-4-200-2-k0")])
def test_restatement_is_the_c_oracle_game(game, n_games, n_playouts, noise, k, keep):
    """Without playout cap randomization, and without forced playouts or with k = 0, the restated game is the C oracle's:
    records, returns and counters."""
    rule = sr.Rule(game, n_playouts, forced=k, use_dirichlet=noise, keep_tree=keep, seed=5)
    for t in range(n_games):
        plies, ret, ctr = sr.selfplay_game(rule, t)
        want, want_ret, want_ctr = ou.selfplay_game(rule.cfg, t)
        assert plies == want and ret == want_ret and ctr[:7] == want_ctr[:7]
        if not keep:
            assert ctr[7] == want_ctr[7]
        cut = sr.selfplay_game(rule, t, max_plies=5)
        cfg = type(rule.cfg).from_buffer_copy(rule.cfg)
        cfg.max_plies = 5
        assert cut[0] == ou.selfplay_game(cfg, t)[0] and cut[2][:7] == ou.selfplay_game(cfg, t)[2][:7]


@pytest.mark.parametrize("game,n_games,n_playouts", [(C4, 64, 100), (BT6, 16, 200)])
def test_all_full_searches_is_the_plain_game(game, n_games, n_playouts):
    plain = sr.Rule(game, n_playouts, seed=5)
    pcr = sr.Rule(game, n_playouts, playout_cap=(n_playouts // 4, 1000), seed=5)
    for t in range(n_games):
        plies, ret, ctr = sr.selfplay_game(pcr, t)
        want, want_ret, want_ctr = ou.selfplay_game(plain.cfg, t)
        assert plies == want and ret == want_ret and ctr[:7] == want_ctr[:7]


@pytest.mark.parametrize("game,n_games,n_playouts", [(C4, 64, 100), (BT6, 16, 200)])
def test_all_fast_searches_at_n_is_the_game_without_noise(game, n_games, n_playouts):
    """permille 0 and fast = n_playouts: every search is fast, which differs from a full one only by its missing root noise."""
    plain = sr.Rule(game, n_playouts, use_dirichlet=0, seed=5)
    pcr = sr.Rule(game, n_playouts, playout_cap=(n_playouts, 0), seed=5)
    for t in range(n_games):
        plies, ret, ctr = sr.selfplay_game(pcr, t)
        want, want_ret, want_ctr = ou.selfplay_game(plain.cfg, t)
        assert all(p["end"] == 3 for p in plies)
        assert [dict(p, end=0) for p in plies] == want and ret == want_ret and ctr[:7] == want_ctr[:7]


@pytest.mark.parametrize("keep", [1, 0])
@pytest.mark.parametrize("game,n_games,n_playouts", [(C4, 32, 100), (BT6, 8, 200)])
def test_fast_searches_follow_stream_7(game, n_games, n_playouts, keep):
    """Every search runs its own target: after the search the root has the visits its kept subtree already had plus the
    target, which is fast_playouts exactly at the stream-7 plies.  The sims counter is the sum of the targets, and the full
    searches (no fast one) expand the root with noise."""
    rule = sr.Rule(game, n_playouts, playout_cap=(n_playouts // 4, 250), keep_tree=keep, seed=9)
    n_fast = n_full = 0
    for t in range(n_games):
        plies, _, ctr = sr.selfplay_game(rule, t)
        kept, hist = 0, []
        for p in plies:
            assert p["root_n"] == kept + rule.target(t, p["ply"]), (t, p["ply"])
            fast = rule.is_fast(t, p["ply"])
            n_fast, n_full = n_fast + fast, n_full + (not fast)
            if keep:
                kept = p["counts"][ou.replay(game, hist)["legal"].index(p["action"])]
            hist.append(p["action"])
        assert ctr[0] == sum(rule.target(t, p["ply"]) for p in plies)
        assert ctr[6] == sum(not rule.is_fast(t, p["ply"]) for p in plies)
    assert n_fast > 2 * n_full > 0


def test_fast_searches_are_no_examples():
    """records_to_games and ExampleBatch.from_records: one example per full search and none per fast one; the key of an
    example is the whole action history before it, fast plies included; values for every backup; to_games() agrees."""
    from alphazero_openspiel_b200.examplegenerator import records_to_games
    from alphazero_openspiel_b200.replay import ExampleBatch
    rule = sr.Rule(C4, 40, playout_cap=(10, 250), seed=3)
    games = [(t, *sr.selfplay_game(rule, t)[:2], 0) for t in range(12)]
    recs = sr.records(C4, games, shuffle_seed=1)
    assert int((recs["end"] == 3).sum()) > 2 * int(((recs["kind"] == 0) & (recs["end"] == 0)).sum())
    for backup in ["on-policy", "soft-Z", "A0C", "off-policy"]:
        lists = records_to_games(recs, C4, backup)
        batch = ExampleBatch.from_records(recs, C4, backup)
        conv = batch.to_games()
        assert len(lists) == len(games) == batch.n_games == len(conv)
        for g, (ex_list, (_, plies, ret, _)) in enumerate(zip(lists, games)):
            full = [(k, p) for k, p in enumerate(plies) if not rule.is_fast(g, p["ply"])]
            assert len(ex_list) == len(full) == batch.game_ptr[g + 1] - batch.game_ptr[g] == len(conv[g])
            lo = batch.game_ptr[g]
            for i, (ex, (k, p)) in enumerate(zip(ex_list, full)):
                want = {"on-policy": ret[0] if (p["ply"] & 1) == 0 else -ret[0], "soft-Z": -p["root_q"],
                        "A0C": p["v_a0c"], "off-policy": p["v_offpolicy"]}[backup]
                key = ", ".join(str(q["action"]) for q in plies[:k])
                assert ex[0] == key == batch.key(lo + i) == conv[g][i][0]
                assert ex[3] == want == batch.value[lo + i] == conv[g][i][3]
                assert batch.ply[lo + i] == p["ply"]
                assert np.array_equal(ex[1], conv[g][i][1]) and ex[2] == conv[g][i][2]


def test_cabi_playout_cap_flag_and_entry_point():
    from alphazero_openspiel_b200 import _lib as L
    lib = L.load()
    assert hasattr(lib, "az_set_playout_cap") and L.F_PLAYOUT_CAP == 1 << 14
    cfg = L.AzConfig()
    cfg.game_id, cfg.n_trees, cfg.n_playouts, cfg.c_puct = 0, 4, 10, 2.5
    cfg.flags = L.F_PLAYOUT_CAP | L.F_MANUAL
    h = C.c_void_p()
    assert lib.az_create(C.byref(cfg), C.byref(h)) != 0
    assert b"AZ_F_PLAYOUT_CAP" in lib.az_last_error() and b"AZ_F_MANUAL" in lib.az_last_error()
    assert lib.az_set_playout_cap(None, 5, 250, None) != 0 and b"null engine" in lib.az_last_error()


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("game,n_trees,n_playouts", [(C4, 64, 100), (BT6, 16, 200), (BT8, 8, 120)])
@pytest.mark.parametrize("keep", [1, 0])
def test_selfplay_with_playout_cap_bit_exact(game, n_trees, n_playouts, keep):
    """Whole games with 25 % full searches and fast = N/4: every ply record (with its end flag) and every counter equal the
    restatement's."""
    rule = sr.Rule(game, n_playouts, playout_cap=(n_playouts // 4, 250), keep_tree=keep, seed=1234)
    recs, ctr = sr.engine_selfplay(rule, n_trees)
    ends, _ = sr.check_against_rule(recs, ctr, rule, n_trees)
    assert ends[3] > 0
    if game == C4 and keep:
        # a per-step simulation cap, by count or by SM cycles, changes no record
        for cap, budget in ((1, 0), (0, 20000)):
            r2, c2 = sr.engine_selfplay(rule, n_trees, max_sims_per_step=cap, step_cycle_budget=budget)
            sr.same_records(r2, recs)
            assert all(c2[k] == ctr[k] for k in ("sims", "moves", "games", "root_evals"))


@pytest.mark.gpu
def test_flag_alone_changes_nothing():
    """AZ_F_PLAYOUT_CAP without an az_set_playout_cap call: every search is full, the records are the plain engine's."""
    from alphazero_openspiel_b200 import _lib as L
    plain = sr.Rule(C4, 100, seed=77)
    on, c_on = sr.engine_selfplay(plain, 64, L.F_PLAYOUT_CAP)
    off, c_off = sr.engine_selfplay(plain, 64)
    sr.same_records(on, off)
    assert c_on == c_off


@pytest.mark.gpu
def test_set_playout_cap_rejects_bad_arguments():
    from alphazero_openspiel_b200 import engine as E, _lib as L
    plain = E.Engine(C4, 4, n_playouts=40, flags=L.F_RECORDS)
    with pytest.raises(RuntimeError, match="without AZ_F_PLAYOUT_CAP"):
        plain.set_playout_cap(10, 250)
    plain.close()
    eng = E.Engine(C4, 4, n_playouts=40, flags=L.F_RECORDS | L.F_PLAYOUT_CAP)
    for fast, permille in ((0, 250), (41, 250), (10, -1), (10, 1001)):
        with pytest.raises(RuntimeError, match="outside"):
            eng.set_playout_cap(fast, permille)
    eng.set_playout_cap(1, 0)
    eng.set_playout_cap(40, 1000)
    eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("game,n_trees,n_playouts", [(C4, 64, 100), (BT6, 16, 200)])
def test_playout_cap_with_resignation(game, n_trees, n_playouts):
    """Resignation is checked at every searched root, fast or full: the records are the resignation rule restated over the
    game with playout cap randomization."""
    rule = sr.Rule(game, n_playouts, resign=(0.0, 300), playout_cap=(n_playouts // 4, 250), keep_tree=1, seed=4321)
    recs, ctr = sr.engine_selfplay(rule, n_trees)
    ends, _ = sr.check_against_rule(recs, ctr, rule, n_trees)
    assert ends[3] > 0 and ends[1] * 5 >= n_trees


@pytest.mark.gpu
def test_eval_cache_with_playout_cap_gives_the_same_games():
    """Fused evaluator and the shipped Connect Four checkpoint: the same records with the evaluator cache on and off."""
    on, c_on = sr.runner_games(C4, 512, True, fast_playouts=10, full_search_fraction=0.25)
    off, c_off = sr.runner_games(C4, 512, False, fast_playouts=10, full_search_fraction=0.25)
    assert c_on["overflow"] == 0 and c_off["overflow"] == 0
    assert c_on["cache_hits"] > 0 and c_off["cache_hits"] == 0
    assert int((on["end"][on["kind"] == 0] == 3).sum()) > 0
    sr.same_records(on, off)


@pytest.mark.gpu
def test_new_playout_cap_reaches_a_captured_graph():
    """az_set_playout_cap on a runner whose round trip is already captured takes effect on the next replay."""
    from alphazero_openspiel_b200.examplegenerator import SelfPlayRunner
    r = SelfPlayRunner(sr.net(C4), C4, "cuda:0", 256, n_playouts=20, seed=3, fast_playouts=5, full_search_fraction=1.0)
    r.round(200)
    assert r._graph is not None
    before = r.drain()
    assert int((before["kind"] == 0).sum()) > 0 and int((before["end"][before["kind"] == 0] == 3).sum()) == 0
    r.set_playout_cap(5, 0.25)
    r.round(200)
    after = r.drain()
    ctr = r.counters()
    r.close()
    assert int((after["end"][after["kind"] == 0] == 3).sum()) > 0 and ctr["overflow"] == 0


@pytest.mark.gpu
def test_virtual_loss_mode_with_playout_cap():
    """K = 4 leaves in flight: the fast plies are the stream-7 ones and every search runs exactly its target."""
    from alphazero_openspiel_b200 import _lib as L
    n_trees, n_playouts, fast = 32, 40, 10
    rule = sr.Rule(C4, n_playouts, playout_cap=(fast, 250), seed=5)
    recs, ctr = sr.engine_selfplay(rule, n_trees, L.F_VIRTUAL_LOSS, leaves_per_tree=4)
    plies = recs[recs["kind"] == 0]
    assert int((recs["kind"] == 1).sum()) == n_trees and ctr["overflow"] == 0
    want = np.array([3 if rule.is_fast(int(t), int(p)) else 0 for t, p in zip(plies["tree"], plies["ply"])])
    assert np.array_equal(plies["end"], want) and (want == 3).any() and (want == 0).any()
    assert ctr["sims"] == sum(fast if e == 3 else n_playouts for e in plies["end"])


@pytest.mark.gpu
@pytest.mark.parametrize("game", [C4, BT6])
def test_example_generator_with_playout_cap(game):
    """Mostly fast searches and a record buffer that the n_playouts-based drain interval would let overflow: the generation
    finishes, every full-search ply record is an example and last_stats counts the fast ones."""
    from alphazero_openspiel_b200.examplegenerator import ExampleGenerator, records_to_games
    n_trees, n_games, n_playouts, fast, capacity = 128, 512, 40, 4, 8192
    gen = ExampleGenerator(sr.net(game), game, "cuda:0", n_trees=n_trees, n_playouts=n_playouts, seed=11, fast_playouts=fast,
                           full_search_fraction=0.1, max_sims_per_step=1, record_capacity=capacity)
    recs, stats = gen._play(n_games)
    assert stats["overflow"] == 0 and stats["games"] == n_games
    # the drain interval sized with n_playouts alone, at the records per round trip this generation produced
    old_interval = max(64, int(capacity * n_playouts / (4.0 * 1 * n_trees)) // 64 * 64)
    assert len(recs) / stats["rounds"] * old_interval > capacity
    kind0 = recs["kind"] == 0
    n_fast = int((kind0 & (recs["end"] == 3)).sum())
    assert stats["fast_searches"] == n_fast > 0
    games = records_to_games(recs, game)
    assert len(games) == n_games
    assert sum(len(g) for g in games) == int((kind0 & (recs["end"] != 3)).sum()) == stats["moves"] - n_fast


@pytest.mark.gpu
def test_trainer_with_playout_cap():
    from alphazero_openspiel_b200.train import Trainer
    tr = Trainer(name_game=C4, fast_playouts=5, n_games_per_generation=64, n_playouts_train=20, save=False)
    for seed in (1, 2):
        n_before = sum(len(g) for g in tr.buffer)
        tr.generate_examples(64, seed=seed)
        s = tr.last_generation_stats
        assert s["games"] == 64 and s["fast_searches"] > 0 and s["overflow"] == 0
        assert sum(len(g) for g in tr.buffer) - n_before == s["moves"] - s["fast_searches"]
