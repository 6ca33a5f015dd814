"""The self-play rule of the step kernels with their extensions (include/az_b200.h: AZ_F_RESIGN, AZ_F_PLAYOUT_CAP,
AZ_F_FORCED_PLAYOUTS, AZ_F_REFLECT), restated once for the tests on top of the C oracle's counter-mode self-play game and
the reference port's search; the engine-format records of restated games; and the GPU harness that runs the engine with
the settings of the same Rule and checks it against the restatement record for record (tests only)."""
import ctypes as C
import math
import os

import numpy as np

from oracle import cbind, pyspiel_shim, ref_port
from tests import oracle_util as ou

C4 = "connect_four"
BT6 = "breakthrough(rows=6,columns=6)"
BT8 = "breakthrough"


class Rule:
    """An oracle self-play configuration (oracle_util.selfplay_cfg) plus the engine's extensions, each off when None:
    resign = (threshold, calibration permille), playout_cap = (fast_playouts, full permille), forced = k, and reflect."""

    def __init__(self, game, n_playouts, resign=None, playout_cap=None, forced=None, reflect=False, **cfg_kw):
        self.game, self.cfg = game, ou.selfplay_cfg(game, n_playouts, **cfg_kw)
        self.resign, self.playout_cap, self.forced, self.reflect = resign, playout_cap, forced, reflect

    def is_fast(self, tree, ply):
        """AZ_F_PLAYOUT_CAP: the search at root ply `ply` is fast iff counter stream 7 % 1000 >= the full permille."""
        return (self.playout_cap is not None
                and cbind.lib().oz_counter(self.cfg.seed, tree, 0, ply, 0, 7) % 1000 >= self.playout_cap[1])

    def target(self, tree, ply):
        """The simulations the search at root ply `ply` runs."""
        return self.playout_cap[0] if self.is_fast(tree, ply) else self.cfg.n_playouts

    def is_forced(self, tree, ply):
        """AZ_F_FORCED_PLAYOUTS: a search with root noise (so not a fast one) is forced iff k > 0."""
        return bool(self.forced) and bool(self.cfg.use_dirichlet) and not self.is_fast(tree, ply)

    def is_calibration(self, tree):
        """AZ_F_RESIGN: the game never resigns iff counter stream 6 % 1000 < the calibration permille."""
        return cbind.lib().oz_counter(self.cfg.seed, tree, 0, 0, 0, 6) % 1000 < self.resign[1]

    def floor(self, prior, n_root):
        """nf(c) = sqrt((k * P(c)) * N_root)."""
        return math.sqrt(self.forced * prior * n_root)

    def prune(self, counts, q, prior, n_root):
        """Policy target pruning of the root child counts (legal order) of a forced search; q / prior of the same children."""
        c_puct = self.cfg.c_puct
        star = int(np.argmax(counts))  # the first maximal count
        sq = math.sqrt(n_root)
        s_star = q[star] + c_puct * prior[star] * sq / (counts[star] + 1)
        out = list(counts)
        for i, n_c in enumerate(counts):
            if i == star or n_c == 0:
                continue
            lo = n_c - self.floor(prior[i], n_root)
            n = n_c
            # the PUCT score at n - 1 visits is q + c_puct * P * sqrt(N_root) / n
            while n > 0 and n - 1 >= lo and q[i] + c_puct * prior[i] * sq / n < s_star:
                n -= 1
            out[i] = 0 if n == 1 else n
        return out


def resign_r(p):
    """r = max(-root_q, v_a0c) of a ply dict: the mover's value that AZ_F_RESIGN compares with the threshold."""
    return max(-p["root_q"], p["v_a0c"])


# ---------------------------------------------------------------------------------------------------------- reflection
def mirror(x, rows, cols):
    """R on a cell mask: column c <-> cols-1-c."""
    y = 0
    for r in range(rows):
        for c in range(cols):
            if (x >> (r * cols + c)) & 1:
                y |= 1 << (r * cols + cols - 1 - c)
    return y


def reflect_action(a, game_id, cols):
    """R on actions, written out from the games' encodings (include/az_b200.h, AZ_F_REFLECT)."""
    if game_id == 0:
        return 6 - a
    cap, d, cell = a & 1, (a >> 1) % 6, (a >> 1) // 6
    r, c = divmod(cell, cols)
    return ((r * cols + cols - 1 - c) * 6 + (2 - d % 3) + 3 * (d // 3)) * 2 + cap


def m(seed, b0, b1, ply):
    """m(s): position (b0, b1, ply) is evaluated reflected (counter stream 8)."""
    return bool(cbind.lib().oz_counter(seed, b0, b1, ply & 1, 0, 8) & 1)


def evaluate(rule, state):
    """The hash evaluator (oz_synth_eval) at `state`; with rule.reflect it answers for R(s) whenever m(s): the prior of a
    is the output of oz_synth_eval_bb on the mirrored bitboards at R(a), the value is as it is.  -> (priors, value)"""
    lib, cfg = cbind.lib(), rule.cfg
    n_actions = state.get_game().num_distinct_actions()
    ply = state.raw().ply
    if rule.reflect:
        b0, b1 = state.bitboards()
        if m(cfg.seed, b0, b1, ply):
            rbb = np.array([mirror(b0, cfg.rows, cfg.cols), mirror(b1, cfg.rows, cfg.cols)], dtype=np.uint64)
            plies = np.array([ply], dtype=np.int32)
            pri, val = np.zeros(n_actions, np.float32), np.zeros(1, np.float32)
            lib.oz_synth_eval_bb(n_actions, 1, rbb.ctypes.data, plies.ctypes.data, cfg.eval_kind, cfg.seed,
                                 cfg.eval_shift, pri.ctypes.data, val.ctypes.data)
            return [float(pri[reflect_action(a, cfg.game, cfg.cols)]) for a in range(n_actions)], float(val[0])
    pri, v = (C.c_double * n_actions)(), C.c_double()
    lib.oz_synth_eval(C.byref(state.raw()), cfg.eval_kind, cfg.seed, cfg.eval_shift, pri, C.byref(v))
    return list(pri), v.value


# ------------------------------------------------------------------------------------------------------- restatement
class _ForcedPort(ref_port.PortMCTS):
    """The reference port's search with the forced-playout root selection while `forcing` (the Rule of a forced search) is
    set: the first visited root child below its floor is taken (its score is +inf, and the first maximum wins)."""
    forcing = None
    n_forced = 0

    def _pick(self, node):
        if node == self.root and self.forcing is not None:
            acts, ids = self.kids[node]
            n_root = self.visits[node]
            for a, j in zip(acts, ids):
                if 1 <= self.visits[j] < self.forcing.floor(self.prior[j], n_root):
                    self.n_forced += 1
                    return j, a
        return super()._pick(node)


def selfplay_game(rule, tree, max_plies=0, stats=None):
    """oracle/az_oracle.c:oz_selfplay_game (counter noise and sampling, hash evaluator) restated with the reference port's
    search (oracle/ref_port.PortMCTS), so that every search can run its own playout count, noise and root selection: a
    fast search runs rule.target simulations without the root noise expansion, a forced search forces root playouts and
    its pruned counts are the record's and the ones the move is sampled from, and rule.reflect reflects the evaluations.
    With every extension off it is the C oracle's game, record for record (tests/test_playout_cap.py).  stats (a dict)
    accumulates "forced" selections and "pruned" visits.
    -> (ply dicts as tests/oracle_util.selfplay_game, whose end is 3 for a fast search, returns[2], counters[8])"""
    lib, cfg = cbind.lib(), rule.cfg
    game = pyspiel_shim.load_game(rule.game)
    mcts = _ForcedPort(lambda state: evaluate(rule, state), game.num_distinct_actions(), c_puct=cfg.c_puct,
                       dirichlet_ratio=cfg.dirichlet_ratio)
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
        fast = rule.is_fast(tree, ply)
        if cfg.use_dirichlet and not fast:
            # expand_root_dirichlet with the counter-uniform noise eta_i = u_i / sum(u) of the oracle and the engine
            u = [float((lib.oz_counter(cfg.seed, tree, 0, ply, i, 1) >> 11) + 1) * (1.0 / 9007199254740992.0)
                 for i in range(len(legal))]
            total = 0.0
            for x in u:
                total += x
            prior, _ = evaluate(rule, st)
            prior = (1.0 - cfg.dirichlet_ratio) * np.array(prior)
            for i, a in enumerate(legal):
                prior[a] = prior[a] + 0.25 * (u[i] / total)
            mcts._grow(mcts.root, prior, legal)
            mcts.stats["root_evals"] += 1
        forced = rule.is_forced(tree, ply)
        mcts.forcing = rule if forced else None
        for _ in range(rule.target(tree, ply)):
            mcts.playout(st.clone())
        visits = mcts.root_child_visits()
        counts = [visits[a] for a in legal]
        if forced:
            ids = dict(zip(*mcts.kids[mcts.root]))
            counts = rule.prune(counts, [mcts.mean[ids[a]] for a in legal], [mcts.prior[ids[a]] for a in legal],
                                mcts.visits[mcts.root])
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
                      "v_offpolicy": mcts.target_off_policy(), "counts": counts, "end": 3 if fast else 0})
        st.apply_action(action)
        last = action
    if stats is not None:
        stats["forced"] = stats.get("forced", 0) + mcts.n_forced
        stats["pruned"] = stats.get("pruned", 0) + pruned
    k = mcts.stats
    ctr = [k["sims"], k["depth"], k["children"], k["expand"], k["legal"], k["terminal"], k["root_evals"], len(mcts.visits)]
    return plies, list(st.returns()), ctr


def oracle_game(rule, tree, stats=None):
    """selfplay_game with the resignation rule of AZ_F_RESIGN on top.  Resignation changes nothing before the position where
    it happens: noise, move sampling and the evaluator are counter hashes of the position and the tree's searches do not
    depend on later moves.  So the full game, played to its end, holds every search a resigning game runs, and:
      - a calibration game (Rule.is_calibration) is the full game; it keeps each player's minimum r;
      - any other game stops at its first searched position, fast or full, with r < threshold: that position's record
        with action -1, the resigner gets -1, and the search counters are those of the game cut after that search;
      - a game in which r never falls below the threshold is the full game.
    stats go to selfplay_game of the full game.
    -> (ply dicts, returns[2], counters[8], end kind as az_record.end, minimum r [2] (2.0: not a calibration game / never
    moved))"""
    plies, ret, ctr = selfplay_game(rule, tree, stats=stats)
    rmin = [2.0, 2.0]
    if rule.resign is None:
        return plies, ret, ctr, 0, rmin
    if rule.is_calibration(tree):
        for p in plies:
            mover = p["ply"] & 1
            if resign_r(p) < rmin[mover]:
                rmin[mover] = resign_r(p)
        return plies, ret, ctr, 2, rmin
    for k, p in enumerate(plies):
        if resign_r(p) < rule.resign[0]:
            _, _, ctr = selfplay_game(rule, tree, max_plies=k + 1)
            mover = p["ply"] & 1
            return plies[:k] + [dict(p, action=-1)], [-1.0, 1.0] if mover == 0 else [1.0, -1.0], ctr, 1, rmin
    return plies, ret, ctr, 0, rmin


def records(game_name, games, shuffle_seed=None):
    """Engine-format records of finished games, each (tree, ply dicts, returns[2], end kind): a kind-0 record per searched
    position, with the ply dict's end (3: a fast search) and its legal actions replayed from the initial position (left
    -1 for a game that starts elsewhere, a random-start game), then the closing kind-1 record with the end kind,
    returns()[0] and the engine's kind-1 ply (the resign position's for end = 1, else the last ply + 1).  The arrival
    order of the engine's records is arbitrary: with a shuffle_seed they are permuted."""
    from alphazero_openspiel_b200.engine import parse_game_name, record_dtype
    maxc = 7 if parse_game_name(game_name)[0] == 0 else 48
    dt = record_dtype(maxc, (72 + 6 * maxc + 7) // 8 * 8)
    rows = []
    for tree, plies, ret, end in games:
        st = pyspiel_shim.load_game(game_name).new_initial_state() if plies[0]["ply"] == 0 else None
        for p in plies:
            rec = np.zeros((), dtype=dt)
            rec["tree"], rec["ply"], rec["action"], rec["end"] = tree, p["ply"], p["action"], p["end"]
            rec["n_legal"], rec["root_n"], rec["bb"] = p["n_legal"], p["root_n"], p["bb"]
            rec["root_q"], rec["v_a0c"], rec["v_offpolicy"] = p["root_q"], p["v_a0c"], p["v_offpolicy"]
            rec["counts"][:p["n_legal"]] = p["counts"]
            rec["actions"][:] = -1
            if st is not None:
                rec["actions"][:p["n_legal"]] = st.legal_actions()
                if p["action"] >= 0:
                    st.apply_action(p["action"])
            rows.append(rec)
        close = np.zeros((), dtype=dt)
        close["tree"], close["kind"], close["end"], close["root_q"] = tree, 1, end, ret[0]
        close["ply"] = plies[-1]["ply"] if end == 1 else plies[-1]["ply"] + 1
        rows.append(close)
    recs = np.array(rows, dtype=dt)
    return recs if shuffle_seed is None else recs[np.random.RandomState(shuffle_seed).permutation(len(recs))]


def oracle_records(n_games=6, game=C4, playouts=20, seed=9, start_mod=0):
    """Training records of the C oracle's self-play games of trees 0..2, each played twice, so that histories repeat
    across games; shuffled."""
    cfg = ou.selfplay_cfg(game, playouts, use_dirichlet=2, sample_moves=1, seed=seed, start_mod=start_mod)
    recs = records(game, [(t, *ou.selfplay_game(cfg, t % 3)[:2], 0) for t in range(n_games)], shuffle_seed=1)
    if start_mod:   # random-start games have no history from the initial position: Connect Four legal = non-full columns
        for i in np.flatnonzero(recs["kind"] == 0):
            occ = int(recs["bb"][i, 0]) | int(recs["bb"][i, 1])
            recs["actions"][i, :recs["n_legal"][i]] = [c for c in range(7) if not (occ >> (35 + c)) & 1]
    return recs


# ---------------------------------------------------------------------------------------------------------------- GPU
def engine_selfplay(rule, n_trees, flags=0, **engine_kw):
    """One game per tree of the engine with the hash evaluator, counter noise and sampling, and the extensions of `rule`:
    their flags and their az_set_* calls.  flags: further engine flags (for a flag alone, no setter is called).
    -> (records sorted by tree, ply and kind; counters)"""
    from alphazero_openspiel_b200 import engine as E, _lib as L
    cfg = rule.cfg
    flags |= L.F_RECORDS | L.F_OFFPOLICY | L.F_SAMPLE_MOVES | (L.F_KEEP_TREE if cfg.keep_tree else 0)
    flags |= L.F_RESIGN if rule.resign is not None else 0
    flags |= L.F_PLAYOUT_CAP if rule.playout_cap is not None else 0
    flags |= L.F_FORCED_PLAYOUTS if rule.forced is not None else 0
    flags |= L.F_REFLECT if rule.reflect else 0
    eng = E.Engine(rule.game, n_trees, n_playouts=cfg.n_playouts, noise_mode=L.NOISE_COUNTER, flags=flags,
                   eval_mode=L.EVAL_HASH, seed=cfg.seed, **engine_kw)
    if rule.resign is not None:
        eng.set_resign(*rule.resign)
    if rule.playout_cap is not None:
        eng.set_playout_cap(*rule.playout_cap)
    if rule.forced is not None:
        eng.set_forced_playouts(rule.forced)
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


def check_against_rule(recs, ctr, rule, n_trees):
    """The records and counters of engine_selfplay(rule, n_trees) equal oracle_game's: every field of every ply record
    (end 3 exactly on the fast searches), the closing record (end kind, returns()[0]; for end = 1 the resign position, for
    end = 2 both players' minimum r) and every counter, the resignation ones included.
    -> (games per closing end kind 0..2 and fast-search ply records as 3, the restatement's "forced" / "pruned" stats)"""
    tot = np.zeros(8, dtype=np.int64)
    ends = {0: 0, 1: 0, 2: 0, 3: 0}
    stats = {"forced": 0, "pruned": 0}
    moves = false_pos = 0
    for t in range(n_trees):
        ref, ret, c, end, rmin = oracle_game(rule, t, stats)
        tot += np.array(c, dtype=np.int64)
        mine = recs[recs["tree"] == t]
        plies, close = mine[mine["kind"] == 0], mine[mine["kind"] == 1]
        assert len(plies) == len(ref) and len(close) == 1
        for r, g in zip(ref, plies):
            assert g["ply"] == r["ply"] and g["n_legal"] == r["n_legal"] and g["end"] == r["end"]
            assert list(g["counts"][:r["n_legal"]]) == r["counts"], (t, r["ply"])
            assert g["action"] == r["action"]
            assert (int(g["bb"][0]), int(g["bb"][1])) == r["bb"] and g["root_n"] == r["root_n"]
            assert g["root_q"] == r["root_q"] and g["v_a0c"] == r["v_a0c"] and g["v_offpolicy"] == r["v_offpolicy"]
            ends[3] += r["end"] == 3
        e = close[0]
        assert e["end"] == end and e["root_q"] == ret[0]
        if end == 1:
            assert e["ply"] == ref[-1]["ply"] and (int(e["bb"][0]), int(e["bb"][1])) == ref[-1]["bb"]
        if end == 2:
            assert e["v_a0c"] == rmin[0] and e["v_offpolicy"] == rmin[1]
            thr = rule.resign[0]
            false_pos += int(rmin[0] < thr and ret[0] >= 0) + int(rmin[1] < thr and ret[1] >= 0)
        ends[end] += 1
        moves += sum(r["action"] >= 0 for r in ref)
    assert ctr["overflow"] == 0 and ctr["games"] == n_trees and ctr["moves"] == moves
    assert ctr["resigns"] == ends[1] and ctr["resign_samples"] == ends[2] and ctr["resign_false"] == false_pos
    assert ctr["sims"] == tot[0] and ctr["depth"] == tot[1] and ctr["children"] == tot[2]
    assert ctr["expansions"] == tot[3] and ctr["legal"] == tot[4] and ctr["terminal"] == tot[5]
    assert ctr["root_evals"] == tot[6]
    return ends, stats


def same_records(a, b):
    assert len(a) == len(b)
    for f in a.dtype.names:
        assert np.array_equal(a[f], b[f]), f


def net(game):
    """The shipped checkpoint of the game (Connect Four, else 6x6 Breakthrough), in eval mode on the CPU."""
    import torch
    from alphazero_openspiel_b200.engine import game_shape
    from alphazero_openspiel_b200.network import Net
    shape, n_actions = game_shape(game)
    name = "example_model_connect_four.pth" if game == C4 else "example_model_breakthrough_6x6.pth"
    out = Net(shape, n_actions)
    ck = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name)
    out.load_state_dict(torch.load(ck, map_location="cpu", weights_only=True))
    return out.eval()


def runner_games(game, n_trees, cache, n_playouts=40, **kw):
    """One game per tree (max_games = n_trees) of a seeded SelfPlayRunner with the shipped checkpoint -> (records sorted,
    counters)."""
    from alphazero_openspiel_b200.examplegenerator import SelfPlayRunner
    r = SelfPlayRunner(net(game), game, "cuda:0", n_trees, n_playouts=n_playouts, seed=31, max_games=n_trees,
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
