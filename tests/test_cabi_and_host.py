"""CPU: the C-ABI library loads and exports every symbol include/az_b200.h declares; host-side logic."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    text = open(os.path.join(ROOT, "include", "az_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(az_[a-z_0-9]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from alphazero_openspiel_b200 import _lib as L, build
    build.build()
    lib = C.CDLL(L.LIB_PATH)
    syms = _header_symbols()
    assert len(syms) >= 20
    for name in syms:
        assert hasattr(lib, name), "libaz_b200.so does not export %s" % name
        assert name in L.SIGNATURES, "ctypes binding misses %s" % name
    assert set(L.SIGNATURES) == set(syms)
    assert L.load().az_version() == 1


def test_config_struct_layout_matches_header():
    from alphazero_openspiel_b200 import _lib as L
    # field order/size as declared in the header: 6 int32, 5 double, 10 int32/uint32, 1 uint64, 2 int32 (appended in r02)
    assert C.sizeof(L.AzConfig) == 6 * 4 + 5 * 8 + 10 * 4 + 8 + 2 * 4
    assert L.AzConfig.seed.offset == 104 and L.AzConfig.c_puct.offset == 24 and L.AzConfig.leaves_per_tree.offset == 112
    assert C.sizeof(L.AzRecord) == 72


def test_no_cpu_fallback_fails_loudly():
    """Without a GPU the product must raise, never compute on the CPU."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from alphazero_openspiel_b200 import _lib as L
    from alphazero_openspiel_b200.engine import Engine
    from alphazero_openspiel_b200.examplegenerator import ExampleGenerator, SelfPlayRunner
    from alphazero_openspiel_b200.network import Net
    with pytest.raises(L.EngineUnavailable):
        Engine("connect_four", 4)
    net = Net([3, 6, 7], 7)
    with pytest.raises(L.EngineUnavailable):
        SelfPlayRunner(net, "connect_four", "cpu", 4)
    with pytest.raises(L.EngineUnavailable):
        ExampleGenerator(net, "connect_four", torch.device("cpu")).generate_examples(2)
    # the raw C-ABI reports an error code + message instead of crashing
    lib = L.load()
    cfg = L.AzConfig()
    cfg.game_id, cfg.n_trees, cfg.n_playouts, cfg.c_puct = 0, 4, 10, 2.5
    h = C.c_void_p()
    rc = lib.az_create(C.byref(cfg), C.byref(h))
    assert rc != 0 and len(lib.az_last_error()) > 0


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "alphazero_openspiel_b200")
    for dirpath, _, files in os.walk(pkg):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, fn)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), fn
                assert "az_oracle" not in text, fn


def test_parse_game_name():
    from alphazero_openspiel_b200.engine import parse_game_name, game_shape
    assert parse_game_name("connect_four") == (0, 6, 7)
    assert parse_game_name("connect_four()") == (0, 6, 7)
    assert parse_game_name("breakthrough") == (1, 8, 8)
    assert parse_game_name("breakthrough()") == (1, 8, 8)
    assert parse_game_name("breakthrough(rows=6,columns=6)") == (1, 6, 6)
    assert parse_game_name("breakthrough(columns=5,rows=7)") == (1, 7, 5)
    assert game_shape("breakthrough(rows=6,columns=6)") == ([3, 6, 6], 432)
    with pytest.raises(ValueError):
        parse_game_name("tic_tac_toe")


def test_remove_illegal_actions_and_policy_target_follow_the_reference_expressions():
    from alphazero_openspiel_b200.alphazerobot import remove_illegal_actions
    from alphazero_openspiel_b200.examplegenerator import policy_target
    from oracle.ref_port import strip_illegal
    rng = np.random.RandomState(0)
    for A, L_ in [(7, 5), (432, 17), (768, 30)]:
        for _ in range(20):
            legal = sorted(rng.choice(A, size=L_, replace=False).tolist())
            counts = rng.randint(0, 300, size=L_)
            counts[rng.randint(L_)] += 1
            visits = [0] * A
            for a, c in zip(legal, counts):
                visits[a] = int(c)
            nvc = np.array([float(v) / sum(visits) for v in visits])  # mcts.py:161-162
            want = strip_illegal(nvc.copy(), legal)
            got = remove_illegal_actions(nvc.copy(), legal)
            assert np.array_equal(want, got)
            pol = policy_target(counts, np.array(legal), L_, A)
            assert pol == [want[a] if a in legal else 0.0 for a in range(A)]
    # the vectorised batch version used by records_to_games is bit-identical to the per-record expressions
    from alphazero_openspiel_b200.examplegenerator import policy_targets_batch
    for A, maxc in [(7, 7), (432, 48), (768, 48)]:
        n = 64
        n_legal = rng.randint(1, min(maxc, A) + 1, size=n)
        counts = np.zeros((n, maxc), dtype=np.int32)
        actions = np.full((n, maxc), -1, dtype=np.int16)
        for i in range(n):
            actions[i, :n_legal[i]] = sorted(rng.choice(A, size=n_legal[i], replace=False).tolist())
            counts[i, :n_legal[i]] = rng.randint(0, 900, size=n_legal[i])
            counts[i, rng.randint(n_legal[i])] += 1
        batch = policy_targets_batch(counts, actions, n_legal, A)
        for i in range(n):
            assert batch[i].tolist() == policy_target(counts[i], actions[i], int(n_legal[i]), A)
    # all-zero mass -> uniform over legal (alphazerobot.py:15-17)
    z = remove_illegal_actions(np.zeros(7), [1, 3])
    assert z.tolist() == [0, 0.5, 0, 0.5, 0, 0, 0]


def test_records_to_games_from_oracle_records():
    """Device record format -> reference example format, checked with records synthesised from the oracle."""
    from alphazero_openspiel_b200.examplegenerator import records_to_games
    from tests import oracle_util as ou, selfplay_rule as sr
    game = "connect_four"
    cfg = ou.selfplay_cfg(game, 25, use_dirichlet=2, sample_moves=1, seed=3)
    expect = [ou.selfplay_game(cfg, t)[:2] for t in range(3)]
    recs = sr.records(game, [(t, plies, ret, 0) for t, (plies, ret) in enumerate(expect)], shuffle_seed=0)
    for backup in ["on-policy", "soft-Z", "A0C", "off-policy"]:
        games = records_to_games(recs, game, backup)
        assert len(games) == 3
        for gme, (plies, ret) in zip(games, expect):
            assert len(gme) == len(plies)
            hist = []
            for i, (ex, r) in enumerate(zip(gme, plies)):
                assert ex[0] == ", ".join(str(a) for a in hist)
                assert np.array_equal(ex[1], ou.replay(game, hist)["board"])
                assert abs(sum(ex[2]) - 1.0) < 1e-12
                want = {"on-policy": ret[0] * (-1) ** i, "soft-Z": -r["root_q"], "A0C": r["v_a0c"],
                        "off-policy": r["v_offpolicy"]}[backup]
                assert ex[3] == want
                hist.append(r["action"])
    assert records_to_games(recs[recs["kind"] == 0], game) == []  # unfinished games are not returned


def test_boards_from_bitboards_breakthrough():
    from alphazero_openspiel_b200.examplegenerator import boards_from_bitboards
    from tests import oracle_util as ou
    rng = np.random.RandomState(2)
    from oracle import pyspiel_shim
    for game, gid, rows, cols in [("breakthrough(rows=6,columns=6)", 1, 6, 6), ("breakthrough", 1, 8, 8),
                                  ("connect_four", 0, 6, 7)]:
        g = pyspiel_shim.load_game(game)
        bbs, plies, boards = [], [], []
        for _ in range(20):
            s = g.new_initial_state()
            for _ in range(rng.randint(0, 25)):
                if s.is_terminal():
                    break
                s.apply_action(int(rng.choice(s.legal_actions())))
            if s.is_terminal():
                continue
            bbs.append(s.bitboards())
            plies.append(len(s.history()))
            boards.append(ou.replay(game, s.history())["board"])
        got = boards_from_bitboards(gid, rows, cols, np.array(bbs, dtype=np.uint64), np.array(plies, dtype=np.int32))
        assert np.array_equal(got, np.array(boards))


def test_conv_weight_image_layout():
    """pack_conv3x3: [ky][kx*50 + co][chunk position][8] (160 rows, 150 used) with chunk c of row r stored at position
    c ^ (r & 7) (the SWIZZLE_128B K-major image the conv kernel bulk-copies into shared memory); pure host code."""
    import torch
    from alphazero_openspiel_b200.nn_fused import pack_conv3x3
    w = torch.arange(64 * 64 * 9, dtype=torch.float32).reshape(64, 64, 3, 3) % 251   # bf16-exact small integers
    img = pack_conv3x3(w).float()
    assert tuple(img.shape) == (3, 160, 8, 8)
    for ky, kx, co, c in [(0, 0, 0, 0), (1, 2, 5, 3), (2, 1, 49, 7), (0, 2, 17, 6), (2, 2, 49, 0)]:
        r = kx * 50 + co
        got = img[ky, r, c ^ (r & 7)]
        assert torch.equal(got, w[co, c * 8:c * 8 + 8, ky, kx])
    assert float(img[:, 150:].abs().max()) == 0.0      # padding rows of the N dimension
