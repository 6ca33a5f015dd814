"""`pyspiel`-shaped shim over the C oracle games (CPU ORACLE -- test infrastructure only).

Exposes exactly the API subset the reference calls (SURVEY Appendix B.1), with the pre-Feb-2020
OpenSpiel method names (`information_state_normalized_vector_shape`, ...), so that the reference's
own mcts.py / alphazerobot.py / game_utils.py run unmodified over it:

    from oracle import pyspiel_shim; pyspiel_shim.install()   # registers sys.modules['pyspiel']
    sys.path.insert(0, REFERENCE_CHECKOUT); import game_utils

Real pyspiel is absent (no network); game semantics follow SURVEY Appendix B.2/B.3.
"""
import ctypes as C
import re
import sys
import types

from . import cbind


def parse_game_name(name):
    """'connect_four' | 'breakthrough' | 'breakthrough(rows=6,columns=6)' -> (game_id, rows, cols)."""
    name = name.strip()
    if name == "connect_four":
        return cbind.GAME_CONNECT_FOUR, 6, 7
    m = re.fullmatch(r"breakthrough(?:\((.*)\))?", name)
    if not m:
        raise ValueError("unknown game: " + name)
    rows = cols = 8
    if m.group(1):
        for kv in m.group(1).split(","):
            k, v = kv.split("=")
            if k.strip() == "rows":
                rows = int(v)
            elif k.strip() == "columns":
                cols = int(v)
            else:
                raise ValueError("unknown breakthrough parameter " + k)
    return cbind.GAME_BREAKTHROUGH, rows, cols


class State:
    __slots__ = ("_s", "_hist", "_game")

    def __init__(self, game, _raw=None, _hist=None):
        self._game = game
        self._s = cbind.OzState()
        if _raw is None:
            cbind.lib().oz_init(C.byref(self._s), game.game_id, game.rows, game.cols)
            self._hist = []
        else:
            C.memmove(C.byref(self._s), C.byref(_raw), C.sizeof(cbind.OzState))
            self._hist = list(_hist)

    def clone(self):
        return State(self._game, self._s, self._hist)

    def current_player(self):
        return cbind.lib().oz_current_player(C.byref(self._s))

    def is_terminal(self):
        return bool(cbind.lib().oz_terminal(C.byref(self._s)))

    def legal_actions(self, player=None):
        buf = (C.c_int32 * cbind.OZ_MAX_LEGAL)()
        n = cbind.lib().oz_legal(C.byref(self._s), buf)
        if player is not None and n and player != self._s.player:
            return []
        return list(buf[:n])

    def apply_action(self, action):
        if cbind.lib().oz_apply(C.byref(self._s), int(action)) != 0:
            raise RuntimeError("illegal action %r" % (action,))
        self._hist.append(int(action))

    def returns(self):
        out = (C.c_double * 2)()
        cbind.lib().oz_returns(C.byref(self._s), out)
        return [out[0], out[1]]

    def player_return(self, player):
        return self.returns()[player]

    def history(self):
        return list(self._hist)

    def information_state(self, player=None):
        return ", ".join(str(a) for a in self._hist)

    def information_state_as_normalized_vector(self, player=None):
        n = 3 * self._game.rows * self._game.cols
        out = (C.c_float * n)()
        cbind.lib().oz_normalized_vector(C.byref(self._s), out)
        return list(out)

    def bitboards(self):
        out = (C.c_uint64 * 2)()
        cbind.lib().oz_bitboards(C.byref(self._s), out)
        return int(out[0]), int(out[1])

    def raw(self):
        return self._s

    def get_game(self):
        return self._game

    def __str__(self):
        g = self._game
        sym = ".xo" if g.game_id == cbind.GAME_CONNECT_FOUR else ".bw"
        rows = []
        for r in range(g.rows - 1, -1, -1):
            rows.append("".join(sym[self._s.cell[r * g.cols + c]] for c in range(g.cols)))
        return "\n".join(rows) + "\n"


class Game:
    def __init__(self, name):
        self.name = name
        self.game_id, self.rows, self.cols = parse_game_name(name)

    def num_distinct_actions(self):
        return 7 if self.game_id == cbind.GAME_CONNECT_FOUR else self.rows * self.cols * 12

    def new_initial_state(self):
        return State(self)

    def information_state_normalized_vector_shape(self):
        return [3, self.rows, self.cols]

    def num_players(self):
        return 2

    def __str__(self):
        return self.name


class Bot:
    def __init__(self, game=None, player=None):
        self._game = game
        self._player = player


def load_game(name):
    return Game(name)


def install():
    """Register this shim as `pyspiel` and a stub `open_spiel.python.algorithms.mcts` (eval harness only)."""
    mod = types.ModuleType("pyspiel")
    mod.Game = Game
    mod.State = State
    mod.Bot = Bot
    mod.load_game = load_game
    sys.modules["pyspiel"] = mod
    for name in ("open_spiel", "open_spiel.python", "open_spiel.python.algorithms",
                 "open_spiel.python.algorithms.mcts"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["open_spiel"].python = sys.modules["open_spiel.python"]
    sys.modules["open_spiel.python"].algorithms = sys.modules["open_spiel.python.algorithms"]
    sys.modules["open_spiel.python.algorithms"].mcts = sys.modules["open_spiel.python.algorithms.mcts"]
    return mod
