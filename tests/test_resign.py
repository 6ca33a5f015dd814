"""Resignation in batched self-play (AZ_F_RESIGN): the rule restated on top of the C oracle's self-play, the threshold
calibration, the conversion of resigned games into training examples, and on the GPU the engine against the restated rule and
through the Python layers."""
import ctypes as C

import numpy as np
import pytest

from tests import oracle_util as ou

C4 = "connect_four"
BT6 = "breakthrough(rows=6,columns=6)"
BT8 = "breakthrough"


class _Rule:
    """An oracle self-play configuration (tests/oracle_util.selfplay_cfg) plus the engine's AZ_F_RESIGN parameters."""

    def __init__(self, cfg, resign, threshold, permille):
        self.cfg, self.resign, self.threshold, self.permille = cfg, resign, threshold, permille


def _cfg(game, n_playouts, resign=0, threshold=0.0, permille=0, **kw):
    return _Rule(ou.selfplay_cfg(game, n_playouts, **kw), resign, threshold, permille)


def _oracle_game(rule, tree, game_seq=0):
    """The resignation rule of AZ_F_RESIGN (include/az_b200.h), restated on top of the CPU oracle's whole-game self-play.

    Resignation changes nothing before the position where it happens: noise, move sampling and the evaluator are counter
    hashes of the position and the tree's searches do not depend on later moves.  So the oracle's full game, played to its
    end, holds every search a resigning game runs, and:
      - a calibration game (counter stream 6 % 1000 < permille) is the full game; it keeps each player's minimum r;
      - any other game stops at its first searched position with r = max(-root_q, v_a0c) < threshold: that position's
        record with action -1, the resigner gets -1, and the search counters are those of the oracle's game cut after that
        search (max_plies);
      - a game in which r never falls below the threshold is the full game.
    -> (ply dicts, returns[2], counters[8], end kind as az_record.end, minimum r [2] (2.0: not a calibration game / never
    moved))"""
    from oracle import cbind
    cfg = rule.cfg
    plies, ret, ctr = ou.selfplay_game(cfg, tree, game_seq)
    rmin = [2.0, 2.0]
    if not rule.resign:
        return plies, ret, ctr, 0, rmin
    if cbind.lib().oz_counter(cfg.seed, tree, game_seq, 0, 0, 6) % 1000 < rule.permille:
        for p in plies:
            m = p["ply"] & 1
            if _r(p) < rmin[m]:
                rmin[m] = _r(p)
        return plies, ret, ctr, 2, rmin
    for k, p in enumerate(plies):
        if _r(p) < rule.threshold:
            cut = type(cfg).from_buffer_copy(cfg)
            cut.max_plies = k + 1
            _, _, ctr = ou.selfplay_game(cut, tree, game_seq)
            m = p["ply"] & 1
            return plies[:k] + [dict(p, action=-1)], [-1.0, 1.0] if m == 0 else [1.0, -1.0], ctr, 1, rmin
    return plies, ret, ctr, 0, rmin


def _r(p):
    return max(-p["root_q"], p["v_a0c"])


def _same_records(a, b):
    assert len(a) == len(b)
    for f in a.dtype.names:
        assert np.array_equal(a[f], b[f]), f


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("game,n_games,n_playouts", [(C4, 64, 100), (BT6, 16, 200)])
def test_oracle_never_firing_threshold_changes_nothing(game, n_games, n_playouts):
    """The restated rule with resignation on, threshold -1 and no calibration games: the game played with it off."""
    off = _cfg(game, n_playouts, seed=5)
    on = _cfg(game, n_playouts, resign=1, threshold=-1.0, permille=0, seed=5)
    for t in range(n_games):
        a, ra, ca = ou.selfplay_game(off.cfg, t)
        b, rb, cb, end, rmin = _oracle_game(on, t)
        assert a == b and ra == rb and ca == cb
        assert end == 0 and rmin == [2.0, 2.0]


@pytest.mark.parametrize("game,n_games,n_playouts", [(C4, 32, 100), (BT6, 8, 200)])
def test_oracle_resigning_threshold_ends_games_early(game, n_games, n_playouts):
    """A threshold that fires: the game stops at the first position with r < threshold, its last ply record has action -1,
    the resigner gets -1; every earlier position had r >= threshold; the plies before are those of the unresigned game."""
    thr = 0.0
    off = _cfg(game, n_playouts, seed=5)
    on = _cfg(game, n_playouts, resign=1, threshold=thr, permille=0, seed=5)
    resigned = 0
    for t in range(n_games):
        full, ret_full, _ = ou.selfplay_game(off.cfg, t)
        plies, ret, _, end, _ = _oracle_game(on, t)
        assert all(_r(p) >= thr for p in plies[:-1])
        if end == 1:
            resigned += 1
            last = plies[-1]
            assert last["action"] == -1 and _r(last) < thr
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
    cfg = _cfg(C4, 60, resign=1, threshold=0.9, permille=1000, seed=8)
    for t in range(16):
        plies, _, _, end, rmin = _oracle_game(cfg, t)
        assert end == 2
        for m in (0, 1):
            mine = [_r(p) for p in plies if (p["ply"] & 1) == m]
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


def _records_from_oracle(game, cfg, trees):
    """Engine-format records (kind 0 per searched position, closing kind-1 record) of oracle games."""
    from alphazero_openspiel_b200.engine import record_dtype
    dt = record_dtype(7, (72 + 6 * 7 + 7) // 8 * 8)
    rows, games = [], []
    for t in trees:
        plies, ret, _, end, _ = _oracle_game(cfg, t)
        hist = []
        for r in plies:
            rec = np.zeros((), dtype=dt)
            rec["tree"], rec["ply"], rec["action"] = t, r["ply"], r["action"]
            rec["n_legal"], rec["root_n"], rec["bb"] = r["n_legal"], r["root_n"], r["bb"]
            rec["root_q"], rec["v_a0c"], rec["v_offpolicy"] = r["root_q"], r["v_a0c"], r["v_offpolicy"]
            rec["counts"][:r["n_legal"]] = r["counts"]
            rec["actions"][:] = -1
            rec["actions"][:r["n_legal"]] = ou.replay(game, hist)["legal"]
            rows.append(rec)
            hist.append(r["action"])
        close = np.zeros((), dtype=dt)
        close["tree"], close["kind"], close["end"], close["root_q"] = t, 1, end, ret[0]
        close["ply"] = plies[-1]["ply"] if end == 1 else plies[-1]["ply"] + 1   # the engine's kind-1 ply
        rows.append(close)
        games.append((plies, ret, end))
    recs = np.array(rows, dtype=dt)
    return recs[np.random.RandomState(1).permutation(len(recs))], games


def test_resigned_games_convert_to_examples():
    """records_to_games and ExampleBatch.from_records need no change for resigned games: every searched position, the resign
    position included, is an example; the on-policy value is +-1 with the sign of the player to move there."""
    from alphazero_openspiel_b200.examplegenerator import records_to_games
    from alphazero_openspiel_b200.replay import ExampleBatch
    game = C4
    cfg = _cfg(game, 40, resign=1, threshold=0.0, permille=0, seed=3)
    recs, games = _records_from_oracle(game, cfg, range(12))
    assert sum(e == 1 for _, _, e in games) >= 3 and sum(e == 0 for _, _, e in games) >= 1
    for backup in ["on-policy", "soft-Z", "A0C", "off-policy"]:
        lists = records_to_games(recs, game, backup)
        batch = ExampleBatch.from_records(recs, game, backup)
        assert len(lists) == len(games) == batch.n_games
        for g, (ex_list, (plies, ret, end)) in enumerate(zip(lists, games)):
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
def _engine_selfplay(game, n_trees, n_playouts, seed, keep, threshold, permille, max_sims_per_step=0, step_cycle_budget=0):
    from alphazero_openspiel_b200 import engine as E, _lib as L
    flags = L.F_RECORDS | L.F_OFFPOLICY | L.F_SAMPLE_MOVES | L.F_RESIGN | (L.F_KEEP_TREE if keep else 0)
    eng = E.Engine(game, n_trees, n_playouts=n_playouts, noise_mode=L.NOISE_COUNTER, flags=flags, eval_mode=L.EVAL_HASH,
                   seed=seed, max_sims_per_step=max_sims_per_step, step_cycle_budget=step_cycle_budget)
    eng.set_resign(threshold, permille)
    for _ in range(4000):
        for _ in range(64):
            eng.step()
        if int((eng.phases() != L.PH_IDLE).sum()) == 0:
            break
    assert int((eng.phases() != L.PH_IDLE).sum()) == 0
    recs = eng.drain_records()
    ctr = eng.counters()
    eng.close()
    return recs[np.lexsort((recs["kind"], recs["ply"], recs["tree"]))], ctr


@pytest.mark.gpu
@pytest.mark.parametrize("game,n_trees,n_playouts", [(C4, 64, 100), (BT6, 16, 200), (BT8, 8, 120)])
@pytest.mark.parametrize("keep", [1, 0])
def test_selfplay_with_resignation_bit_exact(game, n_trees, n_playouts, keep):
    """Whole games with resignation on (hash evaluator, counter noise + sampling, 30 % calibration games): every ply record,
    the closing record (end kind, returns, minimum r) and every counter equal the oracle."""
    seed, thr, permille = 1234, 0.0, 300
    recs, ctr = _engine_selfplay(game, n_trees, n_playouts, seed, keep, thr, permille)
    assert ctr["overflow"] == 0
    cfg = _cfg(game, n_playouts, resign=1, threshold=thr, permille=permille, keep_tree=keep, seed=seed)
    tot = np.zeros(8, dtype=np.int64)
    n_end = {0: 0, 1: 0, 2: 0}
    false_pos = moves = 0
    for t in range(n_trees):
        ref, ret, c, end, rmin = _oracle_game(cfg, t)
        tot += np.array(c, dtype=np.int64)
        mine = recs[recs["tree"] == t]
        plies, close = mine[mine["kind"] == 0], mine[mine["kind"] == 1]
        assert len(plies) == len(ref) and len(close) == 1
        for r, g in zip(ref, plies):
            assert g["ply"] == r["ply"] and g["n_legal"] == r["n_legal"] and g["end"] == 0
            assert list(g["counts"][:r["n_legal"]]) == r["counts"], (t, r["ply"])
            assert g["action"] == r["action"]
            assert (int(g["bb"][0]), int(g["bb"][1])) == r["bb"] and g["root_n"] == r["root_n"]
            assert g["root_q"] == r["root_q"] and g["v_a0c"] == r["v_a0c"] and g["v_offpolicy"] == r["v_offpolicy"]
        e = close[0]
        assert e["end"] == end and e["root_q"] == ret[0]
        if end == 1:
            assert e["ply"] == ref[-1]["ply"] and (int(e["bb"][0]), int(e["bb"][1])) == ref[-1]["bb"]
        if end == 2:
            assert e["v_a0c"] == rmin[0] and e["v_offpolicy"] == rmin[1]
            false_pos += int(rmin[0] < thr and ret[0] >= 0) + int(rmin[1] < thr and ret[1] >= 0)
        n_end[end] += 1
        moves += sum(r["action"] >= 0 for r in ref)
    assert n_end[1] * 5 >= n_trees and n_end[2] > 0
    assert ctr["resigns"] == n_end[1] and ctr["resign_samples"] == n_end[2] and ctr["resign_false"] == false_pos
    assert ctr["games"] == n_trees and ctr["moves"] == moves
    assert ctr["sims"] == tot[0] and ctr["depth"] == tot[1] and ctr["children"] == tot[2]
    assert ctr["expansions"] == tot[3] and ctr["legal"] == tot[4] and ctr["terminal"] == tot[5]
    assert ctr["root_evals"] == tot[6]
    if game == C4 and keep:
        # a per-step simulation cap, by count or by SM cycles, changes no record
        for cap, budget in ((1, 0), (0, 20000)):
            r2, c2 = _engine_selfplay(game, n_trees, n_playouts, seed, keep, thr, permille, cap, budget)
            _same_records(r2, recs)
            assert all(c2[k] == ctr[k] for k in ("sims", "moves", "games", "resigns", "resign_samples", "resign_false"))


def _net(game):
    import os
    import torch
    from alphazero_openspiel_b200.engine import game_shape
    from alphazero_openspiel_b200.network import Net
    shape, n_actions = game_shape(game)
    name = "example_model_connect_four.pth" if game == C4 else "example_model_breakthrough_6x6.pth"
    net = Net(shape, n_actions)
    ck = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name)
    net.load_state_dict(torch.load(ck, map_location="cpu", weights_only=True))
    return net.eval()


def _runner_games(game, n_trees, cache, threshold, n_playouts=40, **kw):
    """One game per tree (max_games = n_trees) of a seeded SelfPlayRunner -> (records sorted, counters)."""
    from alphazero_openspiel_b200.examplegenerator import SelfPlayRunner
    r = SelfPlayRunner(_net(game), game, "cuda:0", n_trees, n_playouts=n_playouts, seed=31, max_games=n_trees,
                       eval_cache=cache, resign_threshold=threshold, resign_disabled_fraction=0.3, **kw)
    recs = []
    for _ in range(400):
        r.round(100)
        recs.append(r.drain())
        if r.all_idle():
            break
    assert r.all_idle()
    ctr = r.counters()
    r.close()
    recs = np.concatenate(recs)
    return recs[np.lexsort((recs["kind"], recs["ply"], recs["tree"]))], ctr


@pytest.mark.gpu
def test_eval_cache_with_resignation_gives_the_same_games():
    """Fused evaluator and the shipped Connect Four checkpoint: the same records with the evaluator cache on and off."""
    on, c_on = _runner_games(C4, 512, True, -0.2)
    off, c_off = _runner_games(C4, 512, False, -0.2)
    assert c_on["overflow"] == 0 and c_off["overflow"] == 0
    assert c_on["cache_hits"] > 0 and c_off["cache_hits"] == 0
    assert c_on["resigns"] > 0 and c_on["resigns"] == c_off["resigns"]
    _same_records(on, off)


@pytest.mark.gpu
def test_new_threshold_reaches_a_captured_graph():
    """az_set_resign on a runner whose round trip is already captured takes effect on the next replay."""
    from alphazero_openspiel_b200.examplegenerator import SelfPlayRunner
    r = SelfPlayRunner(_net(C4), C4, "cuda:0", 256, n_playouts=20, seed=3, resign_threshold=-1.0,
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
    gen = ExampleGenerator(_net(C4), C4, "cuda:0", n_trees=32, virtual_loss=4, n_playouts=40, seed=5,
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
        gen = ExampleGenerator(_net(game), game, "cuda:0", n_trees=n, n_playouts=40, seed=21, resign_threshold=thr,
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
