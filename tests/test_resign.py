"""Resignation in batched self-play (AZ_F_RESIGN): the rule restated on top of the self-play game of
tests/selfplay_rule.py, the threshold calibration, the conversion of resigned games into training examples, and on the GPU
the engine against the restated rule and through the Python layers."""
import ctypes as C

import numpy as np
import pytest

from tests import oracle_util as ou
from tests import selfplay_rule as sr
from tests.selfplay_rule import BT6, BT8, C4


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("game,n_games,n_playouts", [(C4, 64, 100), (BT6, 16, 200)])
def test_oracle_never_firing_threshold_changes_nothing(game, n_games, n_playouts):
    """The restated rule with resignation on, threshold -1 and no calibration games: the game played with it off."""
    off = sr.Rule(game, n_playouts, seed=5)
    on = sr.Rule(game, n_playouts, resign=(-1.0, 0), seed=5)
    for t in range(n_games):
        a, ra, ca = sr.selfplay_game(off, t)
        b, rb, cb, end, rmin = sr.oracle_game(on, t)
        assert a == b and ra == rb and ca == cb
        assert end == 0 and rmin == [2.0, 2.0]


@pytest.mark.parametrize("game,n_games,n_playouts", [(C4, 32, 100), (BT6, 8, 200)])
def test_oracle_resigning_threshold_ends_games_early(game, n_games, n_playouts):
    """A threshold that fires: the game stops at the first position with r < threshold, its last ply record has action -1,
    the resigner gets -1; every earlier position had r >= threshold; the plies before are those of the C oracle's
    unresigned game."""
    thr = 0.0
    off = sr.Rule(game, n_playouts, seed=5)
    on = sr.Rule(game, n_playouts, resign=(thr, 0), seed=5)
    resigned = 0
    for t in range(n_games):
        full, ret_full, _ = ou.selfplay_game(off.cfg, t)
        plies, ret, _, end, _ = sr.oracle_game(on, t)
        assert all(sr.resign_r(p) >= thr for p in plies[:-1])
        if end == 1:
            resigned += 1
            last = plies[-1]
            assert last["action"] == -1 and sr.resign_r(last) < thr
            m = last["ply"] & 1
            assert ret[m] == -1.0 and ret[1 - m] == 1.0
            assert len(plies) <= len(full)
            assert [dict(p, action=None) for p in plies] == [dict(p, action=None) for p in full[:len(plies)]]
            assert [p["action"] for p in plies[:-1]] == [p["action"] for p in full[:len(plies) - 1]]
        else:
            assert end == 0 and plies == full and ret == ret_full
    assert resigned * 5 >= n_games


def test_oracle_calibration_games_keep_the_minimum_r():
    """permille 1000: no game resigns; each player's minimum r over its own searched positions is reported."""
    rule = sr.Rule(C4, 60, resign=(0.9, 1000), seed=8)
    for t in range(16):
        plies, _, _, end, rmin = sr.oracle_game(rule, t)
        assert end == 2
        for m in (0, 1):
            mine = [sr.resign_r(p) for p in plies if (p["ply"] & 1) == m]
            assert rmin[m] == (min(mine) if mine else 2.0)


def test_resign_threshold_for():
    from alphazero_openspiel_b200.engine import record_dtype
    from alphazero_openspiel_b200.examplegenerator import resign_threshold_for
    dt = record_dtype(7, 120)

    def recs(rows):   # rows of (end, returns()[0], min r of player 0, min r of player 1)
        out = np.zeros(len(rows), dtype=dt)
        out["kind"] = 1
        for i, (end, ret0, a, b) in enumerate(rows):
            out[i]["end"], out[i]["root_q"], out[i]["v_a0c"], out[i]["v_offpolicy"] = end, ret0, a, b
        return out

    # non-losing players only: the winner of a decided game, both players of a draw; never-moved (2.0) and end != 2 ignored
    r = recs([(2, 1.0, -0.5, -0.9), (2, -1.0, -0.95, -0.3), (2, 0.0, -0.7, -0.2), (2, 1.0, 2.0, -0.1), (1, -1.0, 0.0, 0.0),
              (0, 1.0, -0.99, -0.99)])
    # values: -0.5 (g0 p0), -0.3 (g1 p1), -0.7, -0.2 (g2 both) -> sorted [-0.7, -0.5, -0.3, -0.2]
    assert resign_threshold_for(r, 0.0, -1.0) == -0.7
    assert resign_threshold_for(r, 0.25, -1.0) == -0.5
    assert resign_threshold_for(r, 0.5, -1.0) == -0.3
    assert resign_threshold_for(r, 0.8, -1.0) == -0.2       # k = 3: the last value
    assert resign_threshold_for(r, 1.0, -0.42) == -0.42     # k = n: keep the current threshold
    assert resign_threshold_for(r[:0], 0.05, -0.42) == -0.42
    assert resign_threshold_for(recs([(1, -1.0, 0.0, 0.0)]), 0.05, -0.6) == -0.6
    # ties: at most a target_fp share of the values lies strictly below the threshold
    t = recs([(2, 1.0, -0.4, 0.0)] * 3 + [(2, 1.0, -0.8, 0.0)])
    assert resign_threshold_for(t, 0.25, -1.0) == -0.4 and resign_threshold_for(t, 0.5, -1.0) == -0.4
    assert resign_threshold_for(t, 0.0, -1.0) == -0.8
    rng = np.random.RandomState(0)
    big = recs([(2, 1.0, float(v), 0.0) for v in np.round(rng.uniform(-1, 1, 200), 2)])
    for fp in (0.0, 0.01, 0.05, 0.1, 0.5):
        thr = resign_threshold_for(big, fp, -1.0)
        assert np.mean(big["v_a0c"] < thr) <= fp


def test_resigned_games_convert_to_examples():
    """records_to_games and ExampleBatch.from_records need no change for resigned games: every searched position, the resign
    position included, is an example; the on-policy value is +-1 with the sign of the player to move there."""
    from alphazero_openspiel_b200.examplegenerator import records_to_games
    from alphazero_openspiel_b200.replay import ExampleBatch
    game = C4
    rule = sr.Rule(game, 40, resign=(0.0, 0), seed=3)
    games = []
    for t in range(12):
        plies, ret, _, end, _ = sr.oracle_game(rule, t)
        games.append((t, plies, ret, end))
    recs = sr.records(game, games, shuffle_seed=1)
    assert sum(e == 1 for _, _, _, e in games) >= 3 and sum(e == 0 for _, _, _, e in games) >= 1
    for backup in ["on-policy", "soft-Z", "A0C", "off-policy"]:
        lists = records_to_games(recs, game, backup)
        batch = ExampleBatch.from_records(recs, game, backup)
        assert len(lists) == len(games) == batch.n_games
        for g, (ex_list, (_, plies, ret, end)) in enumerate(zip(lists, games)):
            assert len(ex_list) == len(plies) == batch.game_ptr[g + 1] - batch.game_ptr[g]
            vals = batch.value[batch.game_ptr[g]:batch.game_ptr[g + 1]]
            for i, (ex, p) in enumerate(zip(ex_list, plies)):
                want = {"on-policy": ret[0] if (p["ply"] & 1) == 0 else -ret[0], "soft-Z": -p["root_q"],
                        "A0C": p["v_a0c"], "off-policy": p["v_offpolicy"]}[backup]
                assert ex[3] == want and vals[i] == want
                if backup == "on-policy" and end == 1:
                    assert abs(want) == 1.0
                    if i == len(plies) - 1:
                        assert want == -1.0       # the resigner's own example
            assert batch.to_games()[g][-1][0] == ex_list[-1][0]


def test_cabi_resign_flag_and_entry_point():
    from alphazero_openspiel_b200 import _lib as L
    lib = L.load()
    assert hasattr(lib, "az_set_resign") and L.F_RESIGN == 1 << 13
    assert L.CTR_NAMES[-3:] == ["resigns", "resign_samples", "resign_false"]
    assert L.AzRecord.end.offset == 28 and C.sizeof(L.AzRecord) == 72
    cfg = L.AzConfig()
    cfg.game_id, cfg.n_trees, cfg.n_playouts, cfg.c_puct = 0, 4, 10, 2.5
    cfg.flags = L.F_RESIGN | L.F_MANUAL
    h = C.c_void_p()
    assert lib.az_create(C.byref(cfg), C.byref(h)) != 0
    assert b"AZ_F_RESIGN" in lib.az_last_error() and b"AZ_F_MANUAL" in lib.az_last_error()
    assert lib.az_set_resign(None, -0.5, 100, None) != 0


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("game,n_trees,n_playouts", [(C4, 64, 100), (BT6, 16, 200), (BT8, 8, 120)])
@pytest.mark.parametrize("keep", [1, 0])
def test_selfplay_with_resignation_bit_exact(game, n_trees, n_playouts, keep):
    """Whole games with resignation on (hash evaluator, counter noise + sampling, 30 % calibration games): every ply record,
    the closing record (end kind, returns, minimum r) and every counter equal the restated rule's."""
    rule = sr.Rule(game, n_playouts, resign=(0.0, 300), keep_tree=keep, seed=1234)
    recs, ctr = sr.engine_selfplay(rule, n_trees)
    ends, _ = sr.check_against_rule(recs, ctr, rule, n_trees)
    assert ends[1] * 5 >= n_trees and ends[2] > 0
    if game == C4 and keep:
        # a per-step simulation cap, by count or by SM cycles, changes no record
        for cap, budget in ((1, 0), (0, 20000)):
            r2, c2 = sr.engine_selfplay(rule, n_trees, max_sims_per_step=cap, step_cycle_budget=budget)
            sr.same_records(r2, recs)
            assert all(c2[k] == ctr[k] for k in ("sims", "moves", "games", "resigns", "resign_samples", "resign_false"))


@pytest.mark.gpu
def test_eval_cache_with_resignation_gives_the_same_games():
    """Fused evaluator and the shipped Connect Four checkpoint: the same records with the evaluator cache on and off."""
    on, c_on = sr.runner_games(C4, 512, True, resign_threshold=-0.2, resign_disabled_fraction=0.3)
    off, c_off = sr.runner_games(C4, 512, False, resign_threshold=-0.2, resign_disabled_fraction=0.3)
    assert c_on["overflow"] == 0 and c_off["overflow"] == 0
    assert c_on["cache_hits"] > 0 and c_off["cache_hits"] == 0
    assert c_on["resigns"] > 0 and c_on["resigns"] == c_off["resigns"]
    sr.same_records(on, off)


@pytest.mark.gpu
def test_new_threshold_reaches_a_captured_graph():
    """az_set_resign on a runner whose round trip is already captured takes effect on the next replay."""
    from alphazero_openspiel_b200.examplegenerator import SelfPlayRunner
    r = SelfPlayRunner(sr.net(C4), C4, "cuda:0", 256, n_playouts=20, seed=3, resign_threshold=-1.0,
                       resign_disabled_fraction=0.0)
    r.round(200)
    assert r._graph is not None
    before = r.counters()
    assert before["resigns"] == 0 and before["sims"] > 0
    r.set_resign(0.5, 0.0)
    r.round(200)
    after = r.counters()
    r.close()
    assert after["resigns"] > 0 and after["overflow"] == 0


@pytest.mark.gpu
def test_virtual_loss_mode_with_resignation():
    from alphazero_openspiel_b200.examplegenerator import ExampleGenerator
    gen = ExampleGenerator(sr.net(C4), C4, "cuda:0", n_trees=32, virtual_loss=4, n_playouts=40, seed=5,
                           resign_threshold=-0.2, resign_disabled_fraction=0.2)
    games = gen.generate_examples(128)
    s = gen.last_stats
    assert len(games) == 128 and s["games"] == 128 and s["overflow"] == 0
    assert s["resigns"] > 0 and s["resign_samples"] > 0
    assert s["resign_threshold_suggested"] is not None


@pytest.mark.gpu
@pytest.mark.parametrize("game", [C4, BT6])
def test_example_generator_resigns_with_the_shipped_checkpoint(game):
    """Same seed with and without a resign threshold: one game per tree, so a resigned game is a prefix of the same tree's
    full game; plies per game drop, and the examples of a resigned game carry the resigner's loss."""
    from alphazero_openspiel_b200.examplegenerator import ExampleGenerator, records_to_games
    n = 128
    out = {}
    for thr in (None, -0.2):
        gen = ExampleGenerator(sr.net(game), game, "cuda:0", n_trees=n, n_playouts=40, seed=21, resign_threshold=thr,
                               resign_disabled_fraction=0.2)
        recs, stats = gen._play(n)
        assert stats["overflow"] == 0 and stats["games"] == n
        out[thr] = (recs[np.lexsort((recs["kind"], recs["ply"], recs["tree"]))], stats)
    full, s_full = out[None]
    res, s_res = out[-0.2]
    assert s_full["resigns"] == 0 and s_res["resigns"] > 0
    assert s_res["moves"] / n < s_full["moves"] / n
    closes = res[res["kind"] == 1]
    assert int((closes["end"] == 1).sum()) == s_res["resigns"]
    games = records_to_games(res, game)
    for t, ex in zip(closes["tree"], games):
        mine = res[(res["tree"] == t) & (res["kind"] == 0)]
        ref = full[(full["tree"] == t) & (full["kind"] == 0)]
        assert len(mine) <= len(ref)
        assert np.array_equal(mine["counts"], ref["counts"][:len(mine)])
        close = closes[closes["tree"] == t][0]
        if close["end"] == 1:
            loser = int(mine["ply"][-1]) & 1
            assert close["root_q"] == (-1.0 if loser == 0 else 1.0) and mine["action"][-1] == -1
            assert [e[3] for e in ex] == [(-1.0 if (int(p) & 1) == loser else 1.0) for p in mine["ply"]]


@pytest.mark.gpu
def test_trainer_adopts_the_suggested_threshold():
    from alphazero_openspiel_b200.train import Trainer
    tr = Trainer(name_game=C4, resign=True, resign_disabled_fraction=0.5, n_games_per_generation=96, n_playouts_train=20,
                 save=False)
    assert tr.resign_threshold == -1.0
    tr.generate_examples(96, seed=1)
    s1 = tr.last_generation_stats
    assert s1["resign_threshold"] == -1.0 and s1["resigns"] == 0 and s1["resign_samples"] > 0
    suggested = s1["resign_threshold_suggested"]
    assert suggested != -1.0 and tr.resign_threshold == suggested
    tr.generate_examples(96, seed=2)
    s2 = tr.last_generation_stats
    assert s2["resign_threshold"] == suggested and tr.resign_threshold == s2["resign_threshold_suggested"]
