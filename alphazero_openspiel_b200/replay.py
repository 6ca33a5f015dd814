"""Array form of the training examples (SURVEY 8(f) rank 3): the replay buffer as a few numpy arrays instead of Python lists.

The reference moves examples around as `[info_state_str, board ndarray, policy list, value]` lists (game_utils.py:168-194,
train.py:108-120): converting 16,384 device-generated games into that format costs more host time than playing them.
`ExampleBatch` keeps the same information as arrays -- bitboards + ply (the board planes are rebuilt only for the sampled
minibatch), the action history (which IS the reference's info-state key), policy and value targets -- converts loss-lessly
to the reference format (`to_games`, equal to `examplegenerator.records_to_games`), and implements `Trainer.remove_duplicates`
(train.py:156-201) as a grouped sum with the reference's semantics: groups in first-occurrence order, sums in buffer order
(so the float64 results are bit-identical), and the first example of every key updated in place like the reference's
accumulator object.
"""
import numpy as np

from . import _lib as L
from .engine import parse_game_name
from .examplegenerator import boards_from_bitboards, policy_targets_batch


def _mix64(x):
    """splitmix64 finaliser (csrc/az_games.cuh mix64) on uint64 arrays."""
    x = x + np.uint64(0x9E3779B97F4A7C15)
    x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return x ^ (x >> np.uint64(31))


def reflect_bits(step, n):
    """Trainer(reflect_minibatches=True): example j of optimisation step `step` is reflected iff the top bit of
    mix64(mix64(step) + j) is set -> bool [n].  Stateless, so it draws nothing from numpy's global RNG and the sample ids
    stay those of the reference."""
    with np.errstate(over="ignore"):
        h = _mix64(_mix64(np.full(1, step, dtype=np.uint64)) + np.arange(n, dtype=np.uint64))
    return (h >> np.uint64(63)).astype(bool)


class ExampleBatch:
    """Examples of whole games, game after game, ply after ply.

    game_ptr [G+1]  examples of game g are rows game_ptr[g] : game_ptr[g+1]
    bb [N,2] uint64, ply [N] int32            position (canonical bitboards), enough to rebuild the board planes
    hist [N,Lmax] int16 (-1 padded), hist_len [N]   actions played before the position == the info-state key
    policy [N,A] float64, value [N] float64   targets (policy rows sum to 1)
    start [N,3] uint64                        (bb0, bb1, ply) of the position the example's game started from when that
                                              was not the initial position (random_start_mod > 0), else zeros: part of
                                              the key, because such a game has no action history for its first plies
    """

    def __init__(self, game_name, game_ptr, bb, ply, hist, hist_len, policy, value, start=None):
        self.game_name = game_name
        self.game_id, self.rows, self.cols = parse_game_name(game_name)
        self.game_ptr = np.asarray(game_ptr, dtype=np.int64)
        self.bb, self.ply, self.hist, self.hist_len = bb, ply, hist, hist_len
        self.policy, self.value = policy, value
        self.start = np.zeros((len(ply), 3), np.uint64) if start is None else start

    def __len__(self):
        return int(self.bb.shape[0])

    @property
    def n_games(self):
        return len(self.game_ptr) - 1

    # ------------------------------------------------------------------ construction
    @staticmethod
    def empty(game_name, num_actions):
        return ExampleBatch(game_name, np.zeros(1, np.int64), np.zeros((0, 2), np.uint64), np.zeros(0, np.int32),
                            np.full((0, 1), -1, np.int16), np.zeros(0, np.int32), np.zeros((0, num_actions)), np.zeros(0),
                            np.zeros((0, 3), np.uint64))

    @staticmethod
    def from_records(records, game_name, backup="on-policy"):
        """Device training records (engine.record_dtype) -> examples of the finished games, in (tree, game_seq) order.
        Same selection, ordering and value targets as examplegenerator.records_to_games (game_utils.py:168-204): a fast
        search's ply record (F_PLAYOUT_CAP, end 3) is no example, but its action is in the history of the examples after it."""
        gid, rows, cols = parse_game_name(game_name)
        num_actions = 7 if gid == L.GAME_CONNECT_FOUR else rows * cols * 12
        if len(records) == 0:
            return ExampleBatch.empty(game_name, num_actions)
        order = np.lexsort((records["kind"], records["ply"], records["game_seq"], records["tree"]))
        recs = records[order]
        key = recs["tree"].astype(np.int64) * (1 << 32) + recs["game_seq"].astype(np.int64)
        starts = np.flatnonzero(np.r_[True, key[1:] != key[:-1]])
        ends = np.r_[starts[1:], len(recs)]
        finished = recs["kind"][ends - 1] == 1                       # the closing record carries returns()[0]
        starts, ends = starts[finished], ends[finished]
        if len(starts) == 0:
            return ExampleBatch.empty(game_name, num_actions)
        n_ply = ends - 1 - starts                                    # ply records per game
        g_rec = np.repeat(np.arange(len(starts)), n_ply)             # game of every ply record
        k_rec = np.arange(int(n_ply.sum())) - np.r_[0, np.cumsum(n_ply)][g_rec]   # its index inside its game
        full = recs["end"][starts[g_rec] + k_rec] != 3               # the examples: ply records of full searches
        g_of, k_of = g_rec[full], k_rec[full]                        # game of every example, its ply index in the game
        game_ptr = np.r_[0, np.cumsum(np.bincount(g_of, minlength=len(starts)))]
        n = int(game_ptr[-1])
        src = starts[g_of] + k_of                                    # row in recs
        ex = recs[src]
        policy = policy_targets_batch(ex["counts"], ex["actions"], ex["n_legal"], num_actions)
        if backup == "soft-Z":
            value = -ex["root_q"].astype(np.float64)
        elif backup == "A0C":
            value = ex["v_a0c"].astype(np.float64)
        elif backup == "off-policy":
            value = ex["v_offpolicy"].astype(np.float64)
        else:  # on-policy: returns()[0] for player 0 to move, negated for player 1 (game_utils.py:168-169,198-203); the sign
            # comes from the position's real ply (a random-start game may begin with player 1 to move)
            reward = recs["root_q"][ends - 1].astype(np.float64)[g_of]
            value = np.where((ex["ply"] & 1) == 0, reward, -reward)
        # action history before every position: row i holds the first k_of[i] actions of its game
        lmax = max(int(n_ply.max()) - 1, 1)
        cols_ = np.arange(lmax)[None, :]
        take = np.minimum(starts[g_of][:, None] + cols_, len(recs) - 1)
        hist = np.where(cols_ < k_of[:, None], recs["action"][take].astype(np.int16), np.int16(-1))
        first = recs[starts[g_of]]                                   # first record of every example's game
        late = first["ply"] > 0
        start = np.zeros((n, 3), np.uint64)
        start[late, 0:2] = first["bb"][late]
        start[late, 2] = first["ply"][late].astype(np.uint64)
        return ExampleBatch(game_name, game_ptr, ex["bb"].copy(), ex["ply"].astype(np.int32), hist,
                            k_of.astype(np.int32), policy, value, start)

    @staticmethod
    def concat(batches):
        batches = [b for b in batches if b is not None]
        assert batches, "nothing to concatenate"
        lmax = max(b.hist.shape[1] for b in batches)
        hists = [np.pad(b.hist, ((0, 0), (0, lmax - b.hist.shape[1])), constant_values=-1) for b in batches]
        ptr = [np.zeros(1, np.int64)]
        off = 0
        for b in batches:
            ptr.append(b.game_ptr[1:] + off)
            off += len(b)
        f = batches[0]
        return ExampleBatch(f.game_name, np.concatenate(ptr), np.concatenate([b.bb for b in batches]),
                            np.concatenate([b.ply for b in batches]), np.concatenate(hists),
                            np.concatenate([b.hist_len for b in batches]), np.concatenate([b.policy for b in batches]),
                            np.concatenate([b.value for b in batches]), np.concatenate([b.start for b in batches]))

    def last_games(self, n_games):
        """The most recent n_games games (the reference trims its buffer list from the front, train.py:232-234)."""
        if n_games >= self.n_games:
            return self
        g0 = self.n_games - n_games
        lo = int(self.game_ptr[g0])
        return ExampleBatch(self.game_name, self.game_ptr[g0:] - lo, self.bb[lo:], self.ply[lo:], self.hist[lo:],
                            self.hist_len[lo:], self.policy[lo:], self.value[lo:], self.start[lo:])

    # ------------------------------------------------------------------ views
    def boards(self, ids=None):
        """state_to_board planes (network.py:9-18) of the selected examples: float64 [n, 4, rows, cols]."""
        ids = slice(None) if ids is None else ids
        return boards_from_bitboards(self.game_id, self.rows, self.cols, self.bb[ids], self.ply[ids])

    def key(self, i):
        """The reference's info-state string of example i (the action history, ', '-joined); games that did not start at
        the initial position carry their start position in front (examplegenerator.start_key_prefix)."""
        from .examplegenerator import start_key_prefix
        return start_key_prefix(self.start[i, 0:2], self.start[i, 2]) + \
            ", ".join(str(int(a)) for a in self.hist[i, :self.hist_len[i]])

    def to_games(self):
        """Loss-less conversion to the reference's format: list of games of [key str, board ndarray, policy list, value]."""
        boards = self.boards()
        games = []
        for g in range(self.n_games):
            lo, hi = int(self.game_ptr[g]), int(self.game_ptr[g + 1])
            games.append([[self.key(i), boards[i], self.policy[i].tolist(), float(self.value[i])] for i in range(lo, hi)])
        return games

    # ------------------------------------------------------------------ Trainer.remove_duplicates on arrays
    def remove_duplicates(self):
        """train.py:156-201: examples with the same key (action history) are merged, policies and values averaged.

        Returns (first, policy, value): `first` = index of the first example of every key, in first-occurrence order (the
        reference's dict order), and that key's averaged targets.  Like the reference, whose accumulator IS the first
        example object of a key, the averaged targets are also written back into rows `first` of this batch."""
        n = len(self)
        if n == 0:
            return np.zeros(0, np.int64), self.policy[:0], self.value[:0]
        keyed = np.concatenate([self.hist_len[:, None].astype(np.int16), self.hist,
                                np.ascontiguousarray(self.start).view(np.int16).reshape(n, 12)], axis=1)
        _, first, inverse = np.unique(keyed, axis=0, return_index=True, return_inverse=True)
        inverse = inverse.reshape(-1)
        rank = np.empty(len(first), np.int64)                  # unique-order group -> first-occurrence order
        by_first = np.argsort(first, kind="stable")
        rank[by_first] = np.arange(len(first))
        grp = rank[inverse]
        first = first[by_first]
        count = np.bincount(grp, minlength=len(first)).astype(np.float64)
        # sums run in buffer order inside every group, exactly like the reference's sequential `acc + item`
        pol = np.zeros((len(first), self.policy.shape[1]), np.float64)
        val = np.zeros(len(first), np.float64)
        np.add.at(pol, grp, self.policy)
        np.add.at(val, grp, self.value)
        pol /= count[:, None]
        val /= count
        self.policy[first] = pol
        self.value[first] = val
        return first, pol, val
