"""Helpers that drive the CPU oracle (tests only)."""
import ctypes as C

import numpy as np

from oracle import cbind


def selfplay_cfg(game_name, n_playouts, c_puct=2.5, dirichlet_ratio=0.25, use_dirichlet=2, sample_moves=1,
                 num_prob=1000, keep_tree=1, eval_kind=1, eval_shift=None, seed=0, start_mod=0, max_plies=0):
    from oracle.pyspiel_shim import parse_game_name
    gid, rows, cols = parse_game_name(game_name)
    cfg = cbind.OzSelfplayCfg()
    cfg.game, cfg.rows, cfg.cols = gid, rows, cols
    cfg.n_playouts, cfg.c_puct, cfg.dirichlet_ratio = n_playouts, c_puct, dirichlet_ratio
    cfg.use_dirichlet, cfg.sample_moves, cfg.num_probabilistic_actions = use_dirichlet, sample_moves, num_prob
    cfg.keep_tree, cfg.eval_kind = keep_tree, eval_kind
    cfg.eval_shift = (2 if gid == 0 else 4) if eval_shift is None else eval_shift
    cfg.seed, cfg.start_random_plies_mod, cfg.max_plies = seed, start_mod, max_plies
    return cfg


def selfplay_game(cfg, tree, game_seq=0, max_out=512):
    """-> (list of ply dicts, returns[2], counters[8]); a ply dict's end is the engine ply record's, 0: the C oracle runs
    no fast searches"""
    lib = cbind.lib()
    recs = (cbind.OzPlyRecord * max_out)()
    ret = (C.c_double * 2)()
    ctr = (C.c_uint64 * 8)()
    n = lib.oz_selfplay_game(C.byref(cfg), tree, game_seq, recs, max_out, ret, ctr)
    assert n <= max_out
    out = []
    for i in range(n):
        r = recs[i]
        out.append({"ply": r.ply, "action": r.action, "n_legal": r.n_legal, "bb": (int(r.bb[0]), int(r.bb[1])),
                    "root_q": r.root_q, "root_n": int(r.root_n), "v_a0c": r.v_a0c, "v_offpolicy": r.v_offpolicy,
                    "counts": list(r.counts[:r.n_legal]), "end": 0})
    return out, [ret[0], ret[1]], list(ctr)


def replay(game_name, history):
    """-> dict(bb, terminal, returns0, legal, board(4,H,W) float64) via the oracle games."""
    from oracle import pyspiel_shim
    g = pyspiel_shim.load_game(game_name)
    s = g.new_initial_state()
    for a in history:
        s.apply_action(int(a))
    lib = cbind.lib()
    board = (C.c_double * (4 * g.rows * g.cols))()
    lib.oz_board(C.byref(s.raw()), board)
    b = np.array(board).reshape(4, g.rows, g.cols)
    return {"bb": s.bitboards(), "terminal": s.is_terminal(), "returns0": s.returns()[0],
            "legal": s.legal_actions(), "board": b, "player": s.raw().player}
