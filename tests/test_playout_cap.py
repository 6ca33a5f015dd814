"""Playout cap randomization in batched self-play (AZ_F_PLAYOUT_CAP): the per-search decision restated in the C oracle's
self-play, the conversion of records with fast searches into training examples, and on the GPU the engine against the oracle
and through the Python layers."""
import ctypes as C

import numpy as np
import pytest

from tests import oracle_util as ou

C4 = "connect_four"
BT6 = "breakthrough(rows=6,columns=6)"
BT8 = "breakthrough"


class _Rule:
    """An oracle self-play configuration (tests/oracle_util.selfplay_cfg) plus the engine's AZ_F_PLAYOUT_CAP parameters
    (fast = 0: off)."""

    def __init__(self, cfg, fast, permille):
        self.cfg, self.fast, self.permille = cfg, fast, permille


def _cfg(game, n_playouts, fast=0, permille=1000, **kw):
    return _Rule(ou.selfplay_cfg(game, n_playouts, **kw), fast, permille)


def _is_fast(rule, tree, ply, game_seq=0):
    """The decision of AZ_F_PLAYOUT_CAP (include/az_b200.h, counter stream 7) for the search at root ply `ply`."""
    from oracle import cbind
    return bool(rule.fast) and cbind.lib().oz_counter(rule.cfg.seed, tree, game_seq, ply, 0, 7) % 1000 >= rule.permille


def _target(rule, tree, ply):
    return rule.fast if _is_fast(rule, tree, ply) else rule.cfg.n_playouts


def _selfplay_game(rule, tree, max_plies=0):
    """oracle/az_oracle.c:oz_selfplay_game (counter noise and sampling, hash evaluator) restated with the reference port's
    search (oracle/ref_port.PortMCTS), so that every search can run its own playout count and noise: a fast search runs
    rule.fast simulations without the root noise expansion.  With rule.fast = 0 it is the C oracle's game, record for record
    (test_restatement_is_the_c_oracle_game).  -> (ply dicts as tests/oracle_util.selfplay_game, returns[2], counters[8])"""
    from oracle import cbind, pyspiel_shim, ref_port
    lib, cfg = cbind.lib(), rule.cfg
    game = pyspiel_shim.load_game(("connect_four" if cfg.game == 0 else
                                   "breakthrough(rows=%d,columns=%d)" % (cfg.rows, cfg.cols)))
    A = game.num_distinct_actions()

    def policy(state):
        pri, v = (C.c_double * A)(), C.c_double()
        lib.oz_synth_eval(C.byref(state.raw()), cfg.eval_kind, cfg.seed, cfg.eval_shift, pri, C.byref(v))
        return list(pri), v.value

    mcts = ref_port.PortMCTS(policy, A, c_puct=cfg.c_puct, dirichlet_ratio=cfg.dirichlet_ratio)
    st = game.new_initial_state()
    plies, first, last = [], True, -1
    while not st.is_terminal():
        if max_plies and len(plies) >= max_plies:
            break
        if cfg.keep_tree:
            if not first:
                mcts.update_root(last)
        else:
            mcts.fresh(uct=False)
        first = False
        ply = st.raw().ply
        legal = st.legal_actions()
        if cfg.use_dirichlet and not _is_fast(rule, tree, ply):
            # expand_root_dirichlet with the counter-uniform noise eta_i = u_i / sum(u) of the oracle and the engine
            u = [float((lib.oz_counter(cfg.seed, tree, 0, ply, i, 1) >> 11) + 1) * (1.0 / 9007199254740992.0)
                 for i in range(len(legal))]
            total = 0.0
            for x in u:
                total += x
            prior, _ = policy(st)
            prior = (1.0 - cfg.dirichlet_ratio) * np.array(prior)
            for i, a in enumerate(legal):
                prior[a] = prior[a] + 0.25 * (u[i] / total)
            mcts._grow(mcts.root, prior, legal)
            mcts.stats["root_evals"] += 1
        for _ in range(_target(rule, tree, ply)):
            mcts.playout(st.clone())
        visits = mcts.root_child_visits()
        counts = [visits[a] for a in legal]
        if cfg.sample_moves and ply < cfg.num_probabilistic_actions:
            r = ((lib.oz_counter(cfg.seed, tree, 0, ply, 0, 2) >> 32) * sum(counts)) >> 32
            cum = 0
            for a, c in zip(legal, counts):
                cum += c
                if cum > r:
                    action = a
                    break
        else:
            action = legal[int(np.argmax(counts))]
        plies.append({"ply": ply, "action": action, "n_legal": len(legal), "bb": st.bitboards(),
                      "root_q": mcts.mean[mcts.root], "root_n": mcts.visits[mcts.root], "v_a0c": mcts.target_a0c(),
                      "v_offpolicy": mcts.target_off_policy(), "counts": counts})
        st.apply_action(action)
        last = action
    k = mcts.stats
    ctr = [k["sims"], k["depth"], k["children"], k["expand"], k["legal"], k["terminal"], k["root_evals"], len(mcts.visits)]
    return plies, list(st.returns()), ctr


def _r(p):
    return max(-p["root_q"], p["v_a0c"])


def _oracle_game(rule, tree, threshold=None, permille=0):
    """The game with playout cap randomization; with a resign threshold, AZ_F_RESIGN restated on top of it as in
    tests/test_resign.py: resignation changes no search before it, so a resigning game is the full game cut at its first
    searched position (fast or full) with r < threshold, and a calibration game (counter stream 6) is the full game.
    -> (ply dicts, returns[2], counters[8], end kind of the closing record)"""
    from oracle import cbind
    plies, ret, ctr = _selfplay_game(rule, tree)
    if threshold is None:
        return plies, ret, ctr, 0
    if cbind.lib().oz_counter(rule.cfg.seed, tree, 0, 0, 0, 6) % 1000 < permille:
        return plies, ret, ctr, 2
    for k, p in enumerate(plies):
        if _r(p) < threshold:
            _, _, ctr = _selfplay_game(rule, tree, max_plies=k + 1)
            m = p["ply"] & 1
            return plies[:k] + [dict(p, action=-1)], [-1.0, 1.0] if m == 0 else [1.0, -1.0], ctr, 1
    return plies, ret, ctr, 0


def _same_records(a, b):
    assert len(a) == len(b)
    for f in a.dtype.names:
        assert np.array_equal(a[f], b[f]), f


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("keep", [1, 0])
@pytest.mark.parametrize("game,n_games,n_playouts,noise", [(C4, 32, 100, 2), (C4, 8, 60, 0), (BT6, 8, 200, 2)])
def test_restatement_is_the_c_oracle_game(game, n_games, n_playouts, noise, keep):
    """Without playout cap randomization the restated game is the C oracle's: records, returns and counters."""
    rule = _cfg(game, n_playouts, use_dirichlet=noise, keep_tree=keep, seed=5)
    for t in range(n_games):
        plies, ret, ctr = _selfplay_game(rule, t)
        want, want_ret, want_ctr = ou.selfplay_game(rule.cfg, t)
        assert plies == want and ret == want_ret and ctr[:7] == want_ctr[:7]
        if not keep:
            assert ctr[7] == want_ctr[7]
        cut = _selfplay_game(rule, t, max_plies=5)
        cfg = type(rule.cfg).from_buffer_copy(rule.cfg)
        cfg.max_plies = 5
        assert cut[0] == ou.selfplay_game(cfg, t)[0] and cut[2][:7] == ou.selfplay_game(cfg, t)[2][:7]


@pytest.mark.parametrize("game,n_games,n_playouts", [(C4, 64, 100), (BT6, 16, 200)])
def test_all_full_searches_is_the_plain_game(game, n_games, n_playouts):
    plain = _cfg(game, n_playouts, seed=5)
    pcr = _cfg(game, n_playouts, fast=n_playouts // 4, permille=1000, seed=5)
    for t in range(n_games):
        plies, ret, ctr = _selfplay_game(pcr, t)
        want, want_ret, want_ctr = ou.selfplay_game(plain.cfg, t)
        assert plies == want and ret == want_ret and ctr[:7] == want_ctr[:7]


@pytest.mark.parametrize("game,n_games,n_playouts", [(C4, 64, 100), (BT6, 16, 200)])
def test_all_fast_searches_at_n_is_the_game_without_noise(game, n_games, n_playouts):
    """permille 0 and fast = n_playouts: every search is fast, which differs from a full one only by its missing root noise."""
    plain = _cfg(game, n_playouts, use_dirichlet=0, seed=5)
    pcr = _cfg(game, n_playouts, fast=n_playouts, permille=0, seed=5)
    for t in range(n_games):
        plies, ret, ctr = _selfplay_game(pcr, t)
        want, want_ret, want_ctr = ou.selfplay_game(plain.cfg, t)
        assert plies == want and ret == want_ret and ctr[:7] == want_ctr[:7]


@pytest.mark.parametrize("keep", [1, 0])
@pytest.mark.parametrize("game,n_games,n_playouts", [(C4, 32, 100), (BT6, 8, 200)])
def test_fast_searches_follow_stream_7(game, n_games, n_playouts, keep):
    """Every search runs its own target: after the search the root has the visits its kept subtree already had plus the
    target, which is fast_playouts exactly at the stream-7 plies.  The sims counter is the sum of the targets, and the full
    searches (no fast one) expand the root with noise."""
    rule = _cfg(game, n_playouts, fast=n_playouts // 4, permille=250, keep_tree=keep, seed=9)
    n_fast = n_full = 0
    for t in range(n_games):
        plies, _, ctr = _selfplay_game(rule, t)
        kept, hist = 0, []
        for p in plies:
            assert p["root_n"] == kept + _target(rule, t, p["ply"]), (t, p["ply"])
            fast = _is_fast(rule, t, p["ply"])
            n_fast, n_full = n_fast + fast, n_full + (not fast)
            if keep:
                kept = p["counts"][ou.replay(game, hist)["legal"].index(p["action"])]
            hist.append(p["action"])
        assert ctr[0] == sum(_target(rule, t, p["ply"]) for p in plies)
        assert ctr[6] == sum(not _is_fast(rule, t, p["ply"]) for p in plies)
    assert n_fast > 2 * n_full > 0


def _records_from_oracle(game, cfg, trees):
    """Engine-format records of oracle games with playout cap randomization: kind 0 per searched position (end 3 for a fast
    search), then the closing kind-1 record; shuffled."""
    from alphazero_openspiel_b200.engine import record_dtype
    dt = record_dtype(7, (72 + 6 * 7 + 7) // 8 * 8)
    rows, games = [], []
    for t in trees:
        plies, ret, _ = _selfplay_game(cfg, t)
        hist = []
        for r in plies:
            rec = np.zeros((), dtype=dt)
            rec["tree"], rec["ply"], rec["action"] = t, r["ply"], r["action"]
            rec["end"] = 3 if _is_fast(cfg, t, r["ply"]) else 0
            rec["n_legal"], rec["root_n"], rec["bb"] = r["n_legal"], r["root_n"], r["bb"]
            rec["root_q"], rec["v_a0c"], rec["v_offpolicy"] = r["root_q"], r["v_a0c"], r["v_offpolicy"]
            rec["counts"][:r["n_legal"]] = r["counts"]
            rec["actions"][:] = -1
            rec["actions"][:r["n_legal"]] = ou.replay(game, hist)["legal"]
            rows.append(rec)
            hist.append(r["action"])
        close = np.zeros((), dtype=dt)
        close["tree"], close["kind"], close["root_q"], close["ply"] = t, 1, ret[0], plies[-1]["ply"] + 1
        rows.append(close)
        games.append((plies, ret))
    recs = np.array(rows, dtype=dt)
    return recs[np.random.RandomState(1).permutation(len(recs))], games


def test_fast_searches_are_no_examples():
    """records_to_games and ExampleBatch.from_records: one example per full search and none per fast one; the key of an
    example is the whole action history before it, fast plies included; values for every backup; to_games() agrees."""
    from alphazero_openspiel_b200.examplegenerator import records_to_games
    from alphazero_openspiel_b200.replay import ExampleBatch
    cfg = _cfg(C4, 40, fast=10, permille=250, seed=3)
    recs, games = _records_from_oracle(C4, cfg, range(12))
    assert int((recs["end"] == 3).sum()) > 2 * int(((recs["kind"] == 0) & (recs["end"] == 0)).sum())
    for backup in ["on-policy", "soft-Z", "A0C", "off-policy"]:
        lists = records_to_games(recs, C4, backup)
        batch = ExampleBatch.from_records(recs, C4, backup)
        conv = batch.to_games()
        assert len(lists) == len(games) == batch.n_games == len(conv)
        for g, (ex_list, (plies, ret)) in enumerate(zip(lists, games)):
            full = [(k, p) for k, p in enumerate(plies) if not _is_fast(cfg, g, p["ply"])]
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
def _engine_selfplay(game, n_trees, n_playouts, seed, keep, fast, permille, flags=0, max_sims_per_step=0,
                     step_cycle_budget=0, resign=None, **kw):
    """One game per tree with the hash evaluator, counter noise and sampling; fast = None: no az_set_playout_cap call."""
    from alphazero_openspiel_b200 import engine as E, _lib as L
    flags |= L.F_RECORDS | L.F_OFFPOLICY | L.F_SAMPLE_MOVES | (L.F_KEEP_TREE if keep else 0)
    if resign is not None:
        flags |= L.F_RESIGN
    eng = E.Engine(game, n_trees, n_playouts=n_playouts, noise_mode=L.NOISE_COUNTER, flags=flags, eval_mode=L.EVAL_HASH,
                   seed=seed, max_sims_per_step=max_sims_per_step, step_cycle_budget=step_cycle_budget, **kw)
    if fast is not None:
        eng.set_playout_cap(fast, permille)
    if resign is not None:
        eng.set_resign(*resign)
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


def _check_against_oracle(recs, ctr, cfg, n_trees, threshold=None, permille=0):
    tot = np.zeros(8, dtype=np.int64)
    n_fast = moves = resigned = 0
    for t in range(n_trees):
        ref, ret, c, end = _oracle_game(cfg, t, threshold, permille)
        tot += np.array(c, dtype=np.int64)
        mine = recs[recs["tree"] == t]
        plies, close = mine[mine["kind"] == 0], mine[mine["kind"] == 1]
        assert len(plies) == len(ref) and len(close) == 1
        for r, g in zip(ref, plies):
            fast = _is_fast(cfg, t, r["ply"])
            assert g["ply"] == r["ply"] and g["n_legal"] == r["n_legal"] and g["end"] == (3 if fast else 0)
            assert list(g["counts"][:r["n_legal"]]) == r["counts"], (t, r["ply"])
            assert g["action"] == r["action"]
            assert (int(g["bb"][0]), int(g["bb"][1])) == r["bb"] and g["root_n"] == r["root_n"]
            assert g["root_q"] == r["root_q"] and g["v_a0c"] == r["v_a0c"] and g["v_offpolicy"] == r["v_offpolicy"]
            n_fast += fast
        assert close[0]["end"] == end and close[0]["root_q"] == ret[0]
        moves += sum(r["action"] >= 0 for r in ref)
        resigned += end == 1
    assert n_fast > 0
    assert ctr["overflow"] == 0 and ctr["games"] == n_trees and ctr["moves"] == moves and ctr["resigns"] == resigned
    assert ctr["sims"] == tot[0] and ctr["depth"] == tot[1] and ctr["children"] == tot[2]
    assert ctr["expansions"] == tot[3] and ctr["legal"] == tot[4] and ctr["terminal"] == tot[5]
    assert ctr["root_evals"] == tot[6]
    return resigned


@pytest.mark.gpu
@pytest.mark.parametrize("game,n_trees,n_playouts", [(C4, 64, 100), (BT6, 16, 200), (BT8, 8, 120)])
@pytest.mark.parametrize("keep", [1, 0])
def test_selfplay_with_playout_cap_bit_exact(game, n_trees, n_playouts, keep):
    """Whole games with 25 % full searches and fast = N/4: every ply record (with its end flag) and every counter equal the
    oracle's."""
    from alphazero_openspiel_b200 import _lib as L
    seed, fast, permille = 1234, n_playouts // 4, 250
    recs, ctr = _engine_selfplay(game, n_trees, n_playouts, seed, keep, fast, permille, L.F_PLAYOUT_CAP)
    cfg = _cfg(game, n_playouts, fast=fast, permille=permille, keep_tree=keep, seed=seed)
    _check_against_oracle(recs, ctr, cfg, n_trees)
    if game == C4 and keep:
        # a per-step simulation cap, by count or by SM cycles, changes no record
        for cap, budget in ((1, 0), (0, 20000)):
            r2, c2 = _engine_selfplay(game, n_trees, n_playouts, seed, keep, fast, permille, L.F_PLAYOUT_CAP, cap, budget)
            _same_records(r2, recs)
            assert all(c2[k] == ctr[k] for k in ("sims", "moves", "games", "root_evals"))


@pytest.mark.gpu
def test_flag_alone_changes_nothing():
    """AZ_F_PLAYOUT_CAP without an az_set_playout_cap call: every search is full, the records are the plain engine's."""
    from alphazero_openspiel_b200 import _lib as L
    on, c_on = _engine_selfplay(C4, 64, 100, 77, 1, None, 0, L.F_PLAYOUT_CAP)
    off, c_off = _engine_selfplay(C4, 64, 100, 77, 1, None, 0)
    _same_records(on, off)
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
    oracle's game with playout cap randomization."""
    from alphazero_openspiel_b200 import _lib as L
    seed, fast, permille, thr, calib = 4321, n_playouts // 4, 250, 0.0, 300
    recs, ctr = _engine_selfplay(game, n_trees, n_playouts, seed, 1, fast, permille, L.F_PLAYOUT_CAP, resign=(thr, calib))
    cfg = _cfg(game, n_playouts, fast=fast, permille=permille, keep_tree=1, seed=seed)
    resigned = _check_against_oracle(recs, ctr, cfg, n_trees, thr, calib)
    assert resigned * 5 >= n_trees


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


def _runner_games(game, n_trees, cache, n_playouts=40, **kw):
    """One game per tree (max_games = n_trees) of a seeded SelfPlayRunner -> (records sorted, counters)."""
    from alphazero_openspiel_b200.examplegenerator import SelfPlayRunner
    r = SelfPlayRunner(_net(game), game, "cuda:0", n_trees, n_playouts=n_playouts, seed=31, max_games=n_trees,
                       eval_cache=cache, **kw)
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
def test_eval_cache_with_playout_cap_gives_the_same_games():
    """Fused evaluator and the shipped Connect Four checkpoint: the same records with the evaluator cache on and off."""
    on, c_on = _runner_games(C4, 512, True, fast_playouts=10, full_search_fraction=0.25)
    off, c_off = _runner_games(C4, 512, False, fast_playouts=10, full_search_fraction=0.25)
    assert c_on["overflow"] == 0 and c_off["overflow"] == 0
    assert c_on["cache_hits"] > 0 and c_off["cache_hits"] == 0
    assert int((on["end"][on["kind"] == 0] == 3).sum()) > 0
    _same_records(on, off)


@pytest.mark.gpu
def test_new_playout_cap_reaches_a_captured_graph():
    """az_set_playout_cap on a runner whose round trip is already captured takes effect on the next replay."""
    from alphazero_openspiel_b200.examplegenerator import SelfPlayRunner
    r = SelfPlayRunner(_net(C4), C4, "cuda:0", 256, n_playouts=20, seed=3, fast_playouts=5, full_search_fraction=1.0)
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
    n_trees, n_playouts, fast, seed = 32, 40, 10, 5
    recs, ctr = _engine_selfplay(C4, n_trees, n_playouts, seed, 1, fast, 250, L.F_PLAYOUT_CAP | L.F_VIRTUAL_LOSS,
                                 leaves_per_tree=4)
    cfg = _cfg(C4, n_playouts, fast=fast, permille=250, seed=seed)
    plies = recs[recs["kind"] == 0]
    assert int((recs["kind"] == 1).sum()) == n_trees and ctr["overflow"] == 0
    want = np.array([3 if _is_fast(cfg, int(t), int(p)) else 0 for t, p in zip(plies["tree"], plies["ply"])])
    assert np.array_equal(plies["end"], want) and (want == 3).any() and (want == 0).any()
    assert ctr["sims"] == sum(fast if e == 3 else n_playouts for e in plies["end"])


@pytest.mark.gpu
@pytest.mark.parametrize("game", [C4, BT6])
def test_example_generator_with_playout_cap(game):
    """Mostly fast searches and a record buffer that the n_playouts-based drain interval would let overflow: the generation
    finishes, every full-search ply record is an example and last_stats counts the fast ones."""
    from alphazero_openspiel_b200.examplegenerator import ExampleGenerator, records_to_games
    n_trees, n_games, n_playouts, fast, capacity = 128, 512, 40, 4, 8192
    gen = ExampleGenerator(_net(game), game, "cuda:0", n_trees=n_trees, n_playouts=n_playouts, seed=11, fast_playouts=fast,
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
