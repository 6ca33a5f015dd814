"""Forced playouts and policy target pruning in batched self-play (AZ_F_FORCED_PLAYOUTS): the rule restated on top of the
reference port's search, the conversion of pruned records into training examples, and on the GPU the engine against the
restatement and through the Python layers."""
import ctypes as C
import math

import numpy as np
import pytest

from tests import oracle_util as ou
from tests import test_playout_cap as pc

C4 = "connect_four"
BT6 = "breakthrough(rows=6,columns=6)"
BT8 = "breakthrough"


def _cfg(game, n_playouts, k=0.0, fast=0, permille=1000, **kw):
    """tests/test_playout_cap._cfg plus the engine's AZ_F_FORCED_PLAYOUTS k (0: no search is forced)."""
    rule = pc._cfg(game, n_playouts, fast=fast, permille=permille, **kw)
    rule.k = k
    return rule


def _floor(k, prior, n_root):
    """nf(c) = sqrt((k * P(c)) * N_root) (include/az_b200.h, AZ_F_FORCED_PLAYOUTS)."""
    return math.sqrt(k * prior * n_root)


def _prune(counts, q, prior, n_root, k, c_puct):
    """Policy target pruning of the root child counts (legal order) of a forced search; q / prior of the same children."""
    star = int(np.argmax(counts))  # the first maximal count
    sq = math.sqrt(n_root)
    s_star = q[star] + c_puct * prior[star] * sq / (counts[star] + 1)
    out = list(counts)
    for i, n_c in enumerate(counts):
        if i == star or n_c == 0:
            continue
        lo = n_c - _floor(k, prior[i], n_root)
        n = n_c
        # the PUCT score at n - 1 visits is q + c_puct * P * sqrt(N_root) / n
        while n > 0 and n - 1 >= lo and q[i] + c_puct * prior[i] * sq / n < s_star:
            n -= 1
        out[i] = 0 if n == 1 else n
    return out


def _port_class():
    from oracle import ref_port

    class ForcedPort(ref_port.PortMCTS):
        """The reference port's search with the forced-playout root selection while forced_k > 0: the first visited root
        child below its floor is taken (its score is +inf, and the first maximum wins)."""
        forced_k = 0.0
        n_forced = 0

        def _pick(self, node):
            if node == self.root and self.forced_k > 0:
                acts, ids = self.kids[node]
                n_root = self.visits[node]
                for a, j in zip(acts, ids):
                    if 1 <= self.visits[j] < _floor(self.forced_k, self.prior[j], n_root):
                        self.n_forced += 1
                        return j, a
            return super()._pick(node)
    return ForcedPort


def _is_forced(rule, tree, ply):
    return rule.k > 0 and bool(rule.cfg.use_dirichlet) and not pc._is_fast(rule, tree, ply)


def _selfplay_game(rule, tree, max_plies=0, stats=None):
    """tests/test_playout_cap._selfplay_game (the C oracle's counter-mode self-play game on the reference port's search)
    with forced playouts at the root of every forced search and its pruned counts in the move choice and the record.
    stats (a dict) accumulates "forced" selections and "pruned" visits.  -> (ply dicts, returns[2], counters[8])"""
    from oracle import cbind, pyspiel_shim
    lib, cfg = cbind.lib(), rule.cfg
    game = pyspiel_shim.load_game(("connect_four" if cfg.game == 0 else
                                   "breakthrough(rows=%d,columns=%d)" % (cfg.rows, cfg.cols)))
    A = game.num_distinct_actions()

    def policy(state):
        pri, v = (C.c_double * A)(), C.c_double()
        lib.oz_synth_eval(C.byref(state.raw()), cfg.eval_kind, cfg.seed, cfg.eval_shift, pri, C.byref(v))
        return list(pri), v.value

    mcts = _port_class()(policy, A, c_puct=cfg.c_puct, dirichlet_ratio=cfg.dirichlet_ratio)
    st = game.new_initial_state()
    plies, first, last, pruned = [], True, -1, 0
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
        if cfg.use_dirichlet and not pc._is_fast(rule, tree, ply):
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
        forced = _is_forced(rule, tree, ply)
        mcts.forced_k = rule.k if forced else 0.0
        for _ in range(pc._target(rule, tree, ply)):
            mcts.playout(st.clone())
        visits = mcts.root_child_visits()
        counts = [visits[a] for a in legal]
        if forced:
            ids = dict(zip(*mcts.kids[mcts.root]))
            counts = _prune(counts, [mcts.mean[ids[a]] for a in legal], [mcts.prior[ids[a]] for a in legal],
                            mcts.visits[mcts.root], rule.k, cfg.c_puct)
            pruned += sum(visits[a] for a in legal) - sum(counts)
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
    if stats is not None:
        stats["forced"] = stats.get("forced", 0) + mcts.n_forced
        stats["pruned"] = stats.get("pruned", 0) + pruned
    k = mcts.stats
    ctr = [k["sims"], k["depth"], k["children"], k["expand"], k["legal"], k["terminal"], k["root_evals"], len(mcts.visits)]
    return plies, list(st.returns()), ctr


def _oracle_game(rule, tree, threshold=None, permille=0, stats=None):
    """The game with forced playouts; with a resign threshold, AZ_F_RESIGN restated on top of it as in
    tests/test_playout_cap._oracle_game (the resignation ply record carries the pruned counts too).
    -> (ply dicts, returns[2], counters[8], end kind of the closing record)"""
    from oracle import cbind
    plies, ret, ctr = _selfplay_game(rule, tree, stats=stats)
    if threshold is None:
        return plies, ret, ctr, 0
    if cbind.lib().oz_counter(rule.cfg.seed, tree, 0, 0, 0, 6) % 1000 < permille:
        return plies, ret, ctr, 2
    for k, p in enumerate(plies):
        if pc._r(p) < threshold:
            _, _, ctr = _selfplay_game(rule, tree, max_plies=k + 1)
            m = p["ply"] & 1
            return plies[:k] + [dict(p, action=-1)], [-1.0, 1.0] if m == 0 else [1.0, -1.0], ctr, 1
    return plies, ret, ctr, 0


def _non_best_ones(counts):
    """Entries other than the first maximum that equal 1."""
    star = int(np.argmax(counts))
    return sum(1 for i, c in enumerate(counts) if i != star and c == 1)


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("keep", [1, 0])
@pytest.mark.parametrize("game,n_games,n_playouts", [(C4, 16, 100), (BT6, 4, 200)])
def test_restatement_at_k0_is_the_c_oracle_game(game, n_games, n_playouts, keep):
    rule = _cfg(game, n_playouts, k=0.0, keep_tree=keep, seed=5)
    for t in range(n_games):
        plies, ret, ctr = _selfplay_game(rule, t)
        want, want_ret, want_ctr = ou.selfplay_game(rule.cfg, t)
        assert plies == want and ret == want_ret and ctr[:7] == want_ctr[:7]


@pytest.mark.parametrize("game,n_games,n_playouts", [(C4, 16, 100), (BT6, 4, 200)])
def test_restatement_at_k0_with_playout_cap_is_its_game(game, n_games, n_playouts):
    rule = _cfg(game, n_playouts, k=0.0, fast=n_playouts // 4, permille=250, seed=9)
    for t in range(n_games):
        assert _selfplay_game(rule, t) == pc._selfplay_game(rule, t)


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
    k, c_puct = 2.0, 2.5
    reduced = high_q_kept = ones_dropped = 0
    for counts, q, prior, n_root in _roots():
        out = _prune(counts, q, prior, n_root, k, c_puct)
        star = int(np.argmax(counts))
        sq = math.sqrt(n_root)
        s_star = q[star] + c_puct * prior[star] * sq / (counts[star] + 1)
        assert out[star] == counts[star]
        assert int(np.argmax(out)) == star
        for i, (n_c, n) in enumerate(zip(counts, out)):
            assert 0 <= n <= n_c
            if i == star:
                continue
            if n == 0 and n_c > 0 and (n_c == 1 or n_c - _floor(k, prior[i], n_root) <= 1):
                ones_dropped += n_c == 1 or n != n_c
                continue  # a remainder of 1 went to 0
            assert n >= n_c - _floor(k, prior[i], n_root)
            assert n != 1
            if n < n_c:
                reduced += 1
                # the child's PUCT at its pruned count stays below c*'s
                assert q[i] + c_puct * prior[i] * sq / (n + 1) < s_star
            elif n_c > 1 and q[i] + c_puct * prior[i] * sq / n_c >= s_star:
                high_q_kept += 1
    first = _prune(*_roots()[0], k, c_puct)
    assert first[0] == 60 and first[1] < 12 and first[2] == 0 and first[3] == 0
    assert _prune(*_roots()[1], k, c_puct)[1] == 30
    assert reduced > 50 and high_q_kept > 10 and ones_dropped > 10


@pytest.mark.parametrize("game,n_games,n_playouts", [(C4, 16, 100), (BT6, 4, 200)])
def test_restated_games_force_and_prune(game, n_games, n_playouts):
    """With k = 2 the restated games do force selections and prune counts, and no non-best count is 1."""
    rule = _cfg(game, n_playouts, k=2.0, seed=5)
    stats = {}
    for t in range(n_games):
        plies, _, _ = _selfplay_game(rule, t, stats=stats)
        for p in plies:
            assert _non_best_ones(p["counts"]) == 0
            assert sum(p["counts"]) <= p["root_n"]
    assert stats["forced"] > 0 and stats["pruned"] > 0


def test_pruned_targets_become_the_examples():
    """records_to_games: the policy targets of the examples are the pruned counts normalised; no non-best entry is 1/sum."""
    from alphazero_openspiel_b200.examplegenerator import records_to_games
    from alphazero_openspiel_b200.engine import record_dtype
    rule = _cfg(C4, 60, k=2.0, seed=3)
    dt = record_dtype(7, (72 + 6 * 7 + 7) // 8 * 8)
    rows, games = [], []
    for t in range(8):
        plies, ret, _ = _selfplay_game(rule, t)
        hist = []
        for r in plies:
            rec = np.zeros((), dtype=dt)
            rec["tree"], rec["ply"], rec["action"] = t, r["ply"], r["action"]
            rec["n_legal"], rec["root_n"], rec["bb"] = r["n_legal"], r["root_n"], r["bb"]
            rec["root_q"], rec["v_a0c"], rec["v_offpolicy"] = r["root_q"], r["v_a0c"], r["v_offpolicy"]
            rec["counts"][:r["n_legal"]] = r["counts"]
            rec["actions"][:] = -1
            rec["actions"][:r["n_legal"]] = ou.replay(C4, hist)["legal"]
            rows.append(rec)
            hist.append(r["action"])
        close = np.zeros((), dtype=dt)
        close["tree"], close["kind"], close["root_q"], close["ply"] = t, 1, ret[0], plies[-1]["ply"] + 1
        rows.append(close)
        games.append(plies)
    lists = records_to_games(np.array(rows, dtype=dt), C4)
    assert len(lists) == len(games)
    n_pruned_rows = 0
    for ex_list, plies in zip(lists, games):
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
def _engine_selfplay(game, n_trees, n_playouts, seed, keep, k, flags=0, max_sims_per_step=0, step_cycle_budget=0,
                     resign=None, fast=None, permille=0, **kw):
    """One game per tree with the hash evaluator, counter noise and sampling; k = None: no az_set_forced_playouts call."""
    from alphazero_openspiel_b200 import engine as E, _lib as L
    flags |= L.F_RECORDS | L.F_OFFPOLICY | L.F_SAMPLE_MOVES | (L.F_KEEP_TREE if keep else 0)
    if resign is not None:
        flags |= L.F_RESIGN
    if fast is not None:
        flags |= L.F_PLAYOUT_CAP
    eng = E.Engine(game, n_trees, n_playouts=n_playouts, noise_mode=L.NOISE_COUNTER, flags=flags, eval_mode=L.EVAL_HASH,
                   seed=seed, max_sims_per_step=max_sims_per_step, step_cycle_budget=step_cycle_budget, **kw)
    if k is not None:
        eng.set_forced_playouts(k)
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


def _check_against_oracle(recs, ctr, rule, n_trees, threshold=None, permille=0):
    """Every ply record (counts, action, root_n, root_q, v_a0c, v_offpolicy, end) and every counter equal the restatement's.
    -> (games that resigned, restatement stats)"""
    tot = np.zeros(8, dtype=np.int64)
    stats = {}
    moves = resigned = 0
    for t in range(n_trees):
        ref, ret, c, end = _oracle_game(rule, t, threshold, permille, stats)
        tot += np.array(c, dtype=np.int64)
        mine = recs[recs["tree"] == t]
        plies, close = mine[mine["kind"] == 0], mine[mine["kind"] == 1]
        assert len(plies) == len(ref) and len(close) == 1
        for r, g in zip(ref, plies):
            fast = pc._is_fast(rule, t, r["ply"])
            assert g["ply"] == r["ply"] and g["n_legal"] == r["n_legal"] and g["end"] == (3 if fast else 0)
            assert list(g["counts"][:r["n_legal"]]) == r["counts"], (t, r["ply"])
            assert g["action"] == r["action"]
            assert (int(g["bb"][0]), int(g["bb"][1])) == r["bb"] and g["root_n"] == r["root_n"]
            assert g["root_q"] == r["root_q"] and g["v_a0c"] == r["v_a0c"] and g["v_offpolicy"] == r["v_offpolicy"]
        assert close[0]["end"] == end and close[0]["root_q"] == ret[0]
        moves += sum(r["action"] >= 0 for r in ref)
        resigned += end == 1
    assert ctr["overflow"] == 0 and ctr["games"] == n_trees and ctr["moves"] == moves and ctr["resigns"] == resigned
    assert ctr["sims"] == tot[0] and ctr["depth"] == tot[1] and ctr["children"] == tot[2]
    assert ctr["expansions"] == tot[3] and ctr["legal"] == tot[4] and ctr["terminal"] == tot[5]
    assert ctr["root_evals"] == tot[6]
    return resigned, stats


@pytest.mark.gpu
@pytest.mark.parametrize("game,n_trees,n_playouts", [(C4, 64, 100), (BT6, 16, 200), (BT8, 8, 120)])
@pytest.mark.parametrize("keep", [1, 0])
def test_selfplay_with_forced_playouts_bit_exact(game, n_trees, n_playouts, keep):
    """Whole games with k = 2: every ply record and every counter equal the restatement's, which forces and prunes."""
    from alphazero_openspiel_b200 import _lib as L
    seed = 1234
    recs, ctr = _engine_selfplay(game, n_trees, n_playouts, seed, keep, 2.0, L.F_FORCED_PLAYOUTS)
    rule = _cfg(game, n_playouts, k=2.0, keep_tree=keep, seed=seed)
    _, stats = _check_against_oracle(recs, ctr, rule, n_trees)
    assert stats["forced"] > 0 and stats["pruned"] > 0
    if game == C4 and keep:
        # a per-step simulation cap, by count or by SM cycles, changes no record
        for cap, budget in ((1, 0), (0, 20000)):
            r2, c2 = _engine_selfplay(game, n_trees, n_playouts, seed, keep, 2.0, L.F_FORCED_PLAYOUTS, cap, budget)
            pc._same_records(r2, recs)
            assert all(c2[k] == ctr[k] for k in ("sims", "moves", "games", "root_evals"))


@pytest.mark.gpu
@pytest.mark.parametrize("game,n_trees,n_playouts", [(C4, 64, 100), (BT6, 16, 200)])
def test_forced_playouts_with_playout_cap(game, n_trees, n_playouts):
    """25 % full searches, fast = N/4: only the full searches are forced and pruned."""
    from alphazero_openspiel_b200 import _lib as L
    seed, fast, permille = 4242, n_playouts // 4, 250
    recs, ctr = _engine_selfplay(game, n_trees, n_playouts, seed, 1, 2.0, L.F_FORCED_PLAYOUTS, fast=fast,
                                 permille=permille)
    rule = _cfg(game, n_playouts, k=2.0, fast=fast, permille=permille, seed=seed)
    _, stats = _check_against_oracle(recs, ctr, rule, n_trees)
    assert stats["forced"] > 0 and stats["pruned"] > 0
    plies = recs[recs["kind"] == 0]
    assert (plies["end"] == 3).any() and (plies["end"] == 0).any()


@pytest.mark.gpu
@pytest.mark.parametrize("game,n_trees,n_playouts", [(C4, 64, 100), (BT6, 16, 200)])
def test_forced_playouts_with_resignation(game, n_trees, n_playouts):
    from alphazero_openspiel_b200 import _lib as L
    seed, thr, calib = 4321, 0.0, 300
    recs, ctr = _engine_selfplay(game, n_trees, n_playouts, seed, 1, 2.0, L.F_FORCED_PLAYOUTS, resign=(thr, calib))
    rule = _cfg(game, n_playouts, k=2.0, keep_tree=1, seed=seed)
    resigned, _ = _check_against_oracle(recs, ctr, rule, n_trees, thr, calib)
    assert resigned * 5 >= n_trees


@pytest.mark.gpu
def test_flag_alone_changes_nothing():
    """AZ_F_FORCED_PLAYOUTS without an az_set_forced_playouts call (k = 0): the records and counters are the plain engine's."""
    from alphazero_openspiel_b200 import _lib as L
    on, c_on = _engine_selfplay(C4, 64, 100, 77, 1, None, L.F_FORCED_PLAYOUTS)
    off, c_off = _engine_selfplay(C4, 64, 100, 77, 1, None)
    pc._same_records(on, off)
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
    r = SelfPlayRunner(pc._net(C4), C4, "cuda:0", 256, n_playouts=n_playouts, seed=3, forced_playouts=0.0)
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
    on, c_on = pc._runner_games(C4, 512, True, forced_playouts=2.0)
    off, c_off = pc._runner_games(C4, 512, False, forced_playouts=2.0)
    assert c_on["overflow"] == 0 and c_off["overflow"] == 0
    assert c_on["cache_hits"] > 0 and c_off["cache_hits"] == 0
    pc._same_records(on, off)


@pytest.mark.gpu
def test_virtual_loss_mode_with_forced_playouts():
    """K = 4 leaves in flight: games finish, every record's counts sum to at most root_n and no non-best count is 1."""
    from alphazero_openspiel_b200 import _lib as L
    n_trees = 32
    recs, ctr = _engine_selfplay(C4, n_trees, 40, 5, 1, 2.0, L.F_FORCED_PLAYOUTS | L.F_VIRTUAL_LOSS, leaves_per_tree=4)
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
    gen = ExampleGenerator(pc._net(game), game, "cuda:0", n_trees=n_trees, n_playouts=40, seed=11, forced_playouts=2.0)
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
