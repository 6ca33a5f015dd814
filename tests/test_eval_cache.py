"""The evaluator cache (AZ_F_EVAL_CACHE): leaves whose position was already evaluated are expanded from stored evaluator
outputs.  The search results must be exactly those of the run without the cache."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

C4 = "connect_four"
BT6 = "breakthrough(rows=6,columns=6)"


def _net(game, seed=0):
    import os
    import torch
    from alphazero_openspiel_b200.engine import game_shape
    from alphazero_openspiel_b200.network import Net
    shape, n_actions = game_shape(game)
    torch.manual_seed(seed)
    net = Net(shape, n_actions)
    if game == BT6 and seed == 0:
        ck = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "example_model_breakthrough_6x6.pth")
        net.load_state_dict(torch.load(ck, map_location="cpu", weights_only=True))
    return net.eval()


@pytest.mark.parametrize("game,n", [(C4, 16384), (BT6, 1024)])
def test_fused_evaluator_output_does_not_depend_on_the_row(game, n):
    """The precondition of the cache's exactness: the same boards in a random order give exactly the permuted outputs."""
    import torch
    from alphazero_openspiel_b200 import _lib as L
    from alphazero_openspiel_b200.engine import game_random_playouts, game_replay_dev
    from alphazero_openspiel_b200.nn_fused import FusedEvaluator
    hist, lens = game_random_playouts(game, n, seed=11, max_plies=40)
    lens = torch.remainder(torch.arange(n, device=lens.device, dtype=torch.int32), lens + 1)  # every depth of the game
    obs = game_replay_dev(game, hist, lens, L.OBS_BF16_NHWC)["obs"]
    ev = FusedEvaluator(_net(game), n, "cuda:0")
    assert ev.row_independent
    p, v = ev.eval_batch(obs)
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(5)).to(obs.device)
    pp, vp = ev.eval_batch(obs[perm])
    assert torch.equal(pp, p[perm]) and torch.equal(vp, v[perm])


def _selfplay(game, n_trees, cache, rounds, log2=0):
    """rounds evaluator round trips of a seeded SelfPlayRunner -> (ply records, counters)."""
    from alphazero_openspiel_b200.examplegenerator import SelfPlayRunner
    r = SelfPlayRunner(_net(game), game, "cuda:0", n_trees, n_playouts=50, seed=77, random_start_mod=9, eval_cache=cache,
                       eval_cache_log2=log2)
    recs = []
    for _ in range(0, rounds, 100):
        r.round(100)
        recs.append(r.drain())
    ctr = r.counters()
    r.close()
    recs = np.concatenate(recs)
    return recs[recs["kind"] == 0], ctr


def _two_generations(game, n_trees, cache, net2):
    """Every tree plays one game, then load_weights(net2) and every tree plays the same game again from its start position:
    -> (ply records of game 1, ply records of game 2, counters after game 1, counters after game 2)."""
    from alphazero_openspiel_b200.examplegenerator import SelfPlayRunner
    r = SelfPlayRunner(_net(game), game, "cuda:0", n_trees, n_playouts=30, seed=77, random_start_mod=9, eval_cache=cache,
                       max_games=n_trees)
    out = []
    for gen in range(2):
        if gen == 1:
            r.load_weights(net2)
            r.engine.reset()          # the same start positions (game_seq 0) as the first generation
        for _ in range(200):
            r.round(100)
            if r.all_idle():
                break
        assert r.all_idle()
        recs = r.drain()
        out.append(recs[recs["kind"] == 0])
        out.append(r.counters())
    r.close()
    return out[0], out[2], out[1], out[3]


def _assert_same_searches(a, b, n_trees, min_searches):
    def keyed(r):
        return {(int(t), int(g), int(p)): i for i, (t, g, p) in enumerate(zip(r["tree"], r["game_seq"], r["ply"]))}
    ka, kb = keyed(a), keyed(b)
    both = sorted(set(ka) & set(kb))
    assert len(both) >= min_searches * n_trees
    ia = np.array([ka[k] for k in both])
    ib = np.array([kb[k] for k in both])
    for f in ["counts", "actions", "action", "root_q", "bb", "root_n", "n_legal"]:
        assert np.array_equal(a[f][ia], b[f][ib]), f


@pytest.mark.parametrize("game,n_trees,log2", [(C4, 4096, 0), (BT6, 1024, 0), (C4, 4096, 4), (BT6, 1024, 4)])
def test_cache_on_gives_the_searches_of_cache_off(game, n_trees, log2):
    """Same seed with and without the cache: every search both runs finished has the same visit counts, move, root value and
    position.  log2 = 4 (16 slots) makes nearly every insert collide with another position."""
    on, c_on = _selfplay(game, n_trees, True, 500, log2)
    off, c_off = _selfplay(game, n_trees, False, 500)
    assert c_on["overflow"] == 0 and c_off["overflow"] == 0 and c_off["cache_hits"] == 0
    assert c_on["cache_hits"] > 0
    _assert_same_searches(on, off, n_trees, 3)


def test_cache_serves_no_entry_of_replaced_weights():
    """load_weights, then the same games again: the table still holds the first weights' outputs for exactly these positions,
    and none of them may be served.  Both runs switch weights with every tree idle, so the switch falls at the same point
    of every search (mid-game, how far a tree has got at a given round depends on the cache and on timing)."""
    game, n_trees = C4, 1024
    net2 = _net(game, seed=9)
    on1, on2, c_on1, c_on2 = _two_generations(game, n_trees, True, net2)
    off1, off2, _, c_off2 = _two_generations(game, n_trees, False, net2)
    assert c_on2["overflow"] == 0 and c_off2["overflow"] == 0
    assert c_on1["cache_hits"] > 0 and c_on2["cache_hits"] > c_on1["cache_hits"]
    _assert_same_searches(on1, off1, n_trees, 3)
    _assert_same_searches(on2, off2, n_trees, 3)
    g1, g2 = on1[np.lexsort((on1["ply"], on1["tree"]))], on2[np.lexsort((on2["ply"], on2["tree"]))]
    assert not np.array_equal(g1["counts"], g2["counts"])    # the new weights change the searches


@pytest.mark.parametrize("game,n_trees,n_playouts", [(C4, 256, 60), (BT6, 256, 24)])
def test_cached_external_evaluator_path_matches_the_oracle(game, n_trees, n_playouts):
    """The external-evaluator path with the cache, answered by a host evaluator that is a pure function of the position:
    the records equal the C oracle's ply by ply, with fewer evaluator rows than expansions."""
    import torch
    from oracle import cbind
    from tests import oracle_util as ou
    from alphazero_openspiel_b200 import engine as E, _lib as L
    seed = 2024
    flags = L.F_RECORDS | L.F_OFFPOLICY | L.F_KEEP_TREE | L.F_SAMPLE_MOVES | L.F_EVAL_CACHE
    eng = E.Engine(game, n_trees, n_playouts=n_playouts, noise_mode=L.NOISE_COUNTER, eval_mode=L.EVAL_EXTERNAL, flags=flags,
                   seed=seed)
    A = eng.num_actions
    shift = 2 if game == C4 else 4
    olib = cbind.lib()
    pri_h = torch.zeros((n_trees, A), dtype=torch.float32).pin_memory()
    val_h = torch.zeros((n_trees,), dtype=torch.float32).pin_memory()
    pri_d = torch.zeros((n_trees, A), dtype=torch.float32, device=eng.device)
    val_d = torch.zeros((n_trees,), dtype=torch.float32, device=eng.device)
    eng.step()
    answered = 0
    for _ in range(200000):
        info = eng.request_info(max_depth=1)
        bb = np.ascontiguousarray(info["bb"])
        ply = np.ascontiguousarray(info["ply"])
        if int((ply >= 0).sum()) == 0 and int((eng.phases() != L.PH_IDLE).sum()) == 0:
            break
        answered += int((ply >= 0).sum())
        olib.oz_synth_eval_bb(A, n_trees, bb.ctypes.data, ply.ctypes.data, 1, seed, shift, pri_h.data_ptr(), val_h.data_ptr())
        pri_d.copy_(pri_h, non_blocking=True)
        val_d.copy_(val_h, non_blocking=True)
        eng.step(pri_d, val_d)
        torch.cuda.synchronize()
    recs = eng.drain_records()
    ctr = eng.counters()
    eng.close()
    assert ctr["overflow"] == 0 and int((recs["kind"] == 1).sum()) == n_trees
    assert ctr["cache_hits"] > 0 and answered + ctr["cache_hits"] <= ctr["expansions"] + ctr["root_evals"]
    cfg = ou.selfplay_cfg(game, n_playouts, use_dirichlet=2, sample_moves=1, keep_tree=1, seed=seed)
    for t in range(n_trees):
        plies = recs[(recs["tree"] == t) & (recs["kind"] == 0)]
        plies = plies[np.argsort(plies["ply"])]
        ref, _, _ = ou.selfplay_game(cfg, t)
        assert len(plies) == len(ref)
        for r, g in zip(ref, plies):
            assert list(g["counts"][:r["n_legal"]]) == r["counts"] and g["action"] == r["action"], (t, r["ply"])
            assert g["root_q"] == r["root_q"] and g["root_n"] == r["root_n"]
            assert g["v_a0c"] == r["v_a0c"] and g["v_offpolicy"] == r["v_offpolicy"]
            assert (int(g["bb"][0]), int(g["bb"][1])) == r["bb"]
