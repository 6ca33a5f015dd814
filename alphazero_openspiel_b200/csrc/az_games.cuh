// az_games.cuh -- register-resident bitboard games for sm_100a.
//
// Replaces the pyspiel State calls on the reference's hot path (SURVEY B.1: clone / current_player /
// is_terminal / apply_action / legal_actions / player_return / information_state_as_normalized_vector,
// call sites mcts.py:138-149,178,184 and network.py:15-17).  Semantics follow OpenSpiel's
// connect_four.cc / breakthrough.cc as stated in SURVEY Appendix B.2/B.3.
//
// Canonical layout: bit i of b[p] = player p owns cell i, cell = row*cols + col.  Side to move = ply & 1.
// Every function here is thread-local (no shuffles), so the same code serves one-thread-per-game
// kernels and the lanes-per-tree search kernel (where all lanes of a tree hold the same state).
#pragma once
#include <stdint.h>

namespace az {

struct St {
  uint64_t b0, b1;  // player 0 / player 1 stones
  int ply;
};

struct Geo {
  int rows, cols, cells, n_actions;
  uint64_t notcol0, notcolL;  // cells not in the first / last column
  uint64_t row0, rowL;        // cells of row 0 / last row
  uint64_t all;
};

__device__ __forceinline__ uint64_t mix64(uint64_t x) {  // splitmix64 finaliser (oracle: oz_mix64)
  x += 0x9E3779B97F4A7C15ULL;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL;
  return x ^ (x >> 31);
}

__device__ __forceinline__ uint64_t counter(uint64_t seed, uint64_t tree, uint64_t game_seq, uint64_t ply,
                                            uint64_t idx, uint64_t stream) {  // oracle: oz_counter
  uint64_t x = mix64(seed ^ 0xA0761D3C5F2E8B49ULL);
  x = mix64(x + tree);
  x = mix64(x + game_seq);
  x = mix64(x + ply);
  x = mix64(x + idx);
  x = mix64(x + stream);
  return x;
}

// Left-right reflection of a cell mask: column c <-> column cols-1-c, rows unchanged.  Both games are symmetric under it
// (AZ_F_REFLECT); the host uses the same code (az_reflect_actions, tests).
__host__ __device__ __forceinline__ uint64_t mirror_columns(uint64_t x, const Geo& g) {
  const uint64_t col0 = g.all & ~g.notcol0;
  uint64_t y = 0;
  for (int c = 0; c < g.cols; ++c) y |= ((x >> c) & col0) << (g.cols - 1 - c);
  return y;
}
__host__ __device__ __forceinline__ St mirror_state(St s, const Geo& g) {
  s.b0 = mirror_columns(s.b0, g);
  s.b1 = mirror_columns(s.b1, g);
  return s;
}

// ------------------------------------------------------------------------------------------------
// Connect Four: 6 rows x 7 columns, action = column, row 0 = bottom (SURVEY B.2).
// ------------------------------------------------------------------------------------------------
struct C4 {
  static constexpr int G = 8;      // lanes per tree in the search kernel
  static constexpr int MAXC = 7;   // max children
  static constexpr int SLOTS = 1;  // children per lane
  static constexpr int MAXD = 48;  // max path length (42 plies + root)
  static constexpr int GAME_ID = 0;

  struct Legal {
    uint32_t mask;  // bit c = column c playable
  };

  static __device__ __forceinline__ Legal legal(const St& s, const Geo&) {
    const uint64_t occ = s.b0 | s.b1;
    Legal l;
    l.mask = (uint32_t)((~occ >> 35) & 0x7Fu);  // top row (row 5) empty
    return l;
  }
  static __device__ __forceinline__ int count(const Legal& l) { return __popc(l.mask); }
  // k-th legal action (ascending), k < count
  static __device__ __forceinline__ int action_of(const Legal& l, const St&, const Geo&, int k) {
    return (int)__fns(l.mask, 0, k + 1);
  }
  // index of `action` in the legal list, -1 if illegal
  static __device__ __forceinline__ int rank_of(const Legal& l, const St&, const Geo&, int action) {
    if (action < 0 || action > 6 || !((l.mask >> action) & 1u)) return -1;
    return __popc(l.mask & ((1u << action) - 1u));
  }
  static __device__ __forceinline__ St apply(St s, const Geo&, int a) {
    const uint64_t occ = s.b0 | s.b1;
    const int h = __popcll(occ & (0x0000000810204081ULL << a));  // stones already in column a
    const uint64_t bit = 1ULL << (h * 7 + a);
    if (s.ply & 1) s.b1 |= bit; else s.b0 |= bit;
    s.ply += 1;
    return s;
  }
  static __device__ __forceinline__ bool has4(uint64_t x) {
    const uint64_t NOT6 = ~0x0000020408102040ULL;  // not column 6
    const uint64_t NOT0 = ~0x0000000810204081ULL;  // not column 0
    uint64_t p = x & (x >> 1) & NOT6;              // horizontal pairs (c, c+1)
    if (p & (p >> 1) & (p >> 2)) return true;
    if (x & (x >> 7) & (x >> 14) & (x >> 21)) return true;  // vertical
    p = x & (x >> 8) & NOT6;                       // diagonal (r+1, c+1)
    if (p & (p >> 8) & (p >> 16)) return true;
    p = x & (x >> 6) & NOT0;                       // diagonal (r+1, c-1)
    if (p & (p >> 6) & (p >> 12)) return true;
    return false;
  }
  // -1 not terminal, 0 / 1 winner, 2 draw
  static __device__ __forceinline__ int outcome(const St& s, const Geo&) {
    if (has4(s.b0)) return 0;
    if (has4(s.b1)) return 1;
    if (__popcll(s.b0 | s.b1) == 42) return 2;
    return -1;
  }
  // observation plane ch (0..2) as a cell mask: empty, 'o' (player 1), 'x' (player 0)
  static __device__ __forceinline__ uint64_t plane(const St& s, const Geo& g, int ch) {
    return ch == 0 ? (~(s.b0 | s.b1) & g.all) : (ch == 1 ? s.b1 : s.b0);
  }
  // left-right reflection R(s) and the action map R(a): column a <-> 6 - a
  static __host__ __device__ __forceinline__ St reflect(const St& s, const Geo& g) { return mirror_state(s, g); }
  static __host__ __device__ __forceinline__ int reflect_action(int a, const Geo& g) { return g.cols - 1 - a; }
  static __device__ __forceinline__ St initial(const Geo&) {
    St s;
    s.b0 = s.b1 = 0;
    s.ply = 0;
    return s;
  }
};

// ------------------------------------------------------------------------------------------------
// Breakthrough R x C (<= 64 cells).  Player 0 (black) owns rows 0,1 and moves +row; player 1 (white)
// owns the last two rows and moves -row.  action = ((cell*6 + dir)*2 + capture), dir = dcol+1 (+3 for
// white); diagonal moves may capture, straight moves may not (SURVEY B.3).
// ------------------------------------------------------------------------------------------------
struct BT {
  static constexpr int G = 32;
  static constexpr int MAXC = 48;
  static constexpr int SLOTS = 2;
  static constexpr int MAXD = 160;
  static constexpr int GAME_ID = 1;

  struct Legal {
    uint64_t m[3];  // source cells that may move with dcol = -1, 0, +1
  };

  static __device__ __forceinline__ Legal legal(const St& s, const Geo& g) {
    const int C = g.cols;
    Legal l;
    if (!(s.ply & 1)) {
      const uint64_t me = s.b0, any = s.b0 | s.b1, src = me & ~g.rowL;
      l.m[0] = src & g.notcol0 & ~(me >> (C - 1));
      l.m[1] = src & ~(any >> C);
      l.m[2] = src & g.notcolL & ~(me >> (C + 1));
    } else {
      const uint64_t me = s.b1, any = s.b0 | s.b1, src = me & ~g.row0;
      l.m[0] = src & g.notcol0 & ~(me << (C + 1));
      l.m[1] = src & ~(any << C);
      l.m[2] = src & g.notcolL & ~(me << (C - 1));
    }
    return l;
  }
  static __device__ __forceinline__ int count(const Legal& l) {
    return __popcll(l.m[0]) + __popcll(l.m[1]) + __popcll(l.m[2]);
  }
  static __device__ __forceinline__ int below(const Legal& l, int cell) {  // legal moves from cells < cell
    const uint64_t lo = cell >= 64 ? ~0ULL : ((1ULL << cell) - 1ULL);
    return __popcll(l.m[0] & lo) + __popcll(l.m[1] & lo) + __popcll(l.m[2] & lo);
  }
  static __device__ __forceinline__ int encode(const St& s, const Geo& g, int cell, int d3) {
    const int pl = s.ply & 1;
    const int tgt = cell + (pl ? -g.cols : g.cols) + d3 - 1;
    const uint64_t opp = pl ? s.b0 : s.b1;
    const int cap = (d3 != 1) && ((opp >> tgt) & 1ULL);
    return ((cell * 6 + d3 + 3 * pl) * 2) + cap;
  }
  static __device__ __forceinline__ int action_of(const Legal& l, const St& s, const Geo& g, int k) {
    // smallest cell whose cumulative count (cells <= cell) exceeds k
    int lo = 0, hi = g.cells - 1;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (below(l, mid + 1) > k) hi = mid; else lo = mid + 1;
    }
    int r = k - below(l, lo);
    int d3 = 0;
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      if ((l.m[d] >> lo) & 1ULL) {
        if (r == 0) { d3 = d; break; }
        --r;
      }
    }
    return encode(s, g, lo, d3);
  }
  static __device__ __forceinline__ int rank_of(const Legal& l, const St& s, const Geo& g, int action) {
    if (action < 0 || action >= g.n_actions) return -1;
    const int pl = s.ply & 1;
    const int dir = (action >> 1) % 6, cell = (action >> 1) / 6;
    const int d3 = dir - 3 * pl;
    if (d3 < 0 || d3 > 2) return -1;
    if (!((l.m[d3] >> cell) & 1ULL)) return -1;
    if (encode(s, g, cell, d3) != action) return -1;
    int r = below(l, cell);
    for (int d = 0; d < d3; ++d) r += (int)((l.m[d] >> cell) & 1ULL);
    return r;
  }
  static __device__ __forceinline__ St apply(St s, const Geo& g, int a) {
    const int pl = s.ply & 1;
    const int dir = (a >> 1) % 6, cell = (a >> 1) / 6;
    const int tgt = cell + (dir < 3 ? g.cols : -g.cols) + (dir % 3) - 1;
    const uint64_t from = 1ULL << cell, to = 1ULL << tgt;
    if (pl) { s.b1 = (s.b1 & ~from) | to; s.b0 &= ~to; }
    else    { s.b0 = (s.b0 & ~from) | to; s.b1 &= ~to; }
    s.ply += 1;
    return s;
  }
  static __device__ __forceinline__ int outcome(const St& s, const Geo& g) {
    if ((s.b0 & g.rowL) || s.b1 == 0) return 0;
    if ((s.b1 & g.row0) || s.b0 == 0) return 1;
    return -1;
  }
  // planes: black (player 0), white (player 1), empty
  static __device__ __forceinline__ uint64_t plane(const St& s, const Geo& g, int ch) {
    return ch == 0 ? s.b0 : (ch == 1 ? s.b1 : (~(s.b0 | s.b1) & g.all));
  }
  // left-right reflection R(s) and the action map R(a): the move from (r, c) with column step dcol <-> the move from
  // (r, cols-1-c) with step -dcol (d3 <-> 2 - d3), same player, same capture bit
  static __host__ __device__ __forceinline__ St reflect(const St& s, const Geo& g) { return mirror_state(s, g); }
  static __host__ __device__ __forceinline__ int reflect_action(int a, const Geo& g) {
    const int dir = (a >> 1) % 6, cell = (a >> 1) / 6;
    const int r = cell / g.cols, c = cell - r * g.cols;
    const int d3 = dir % 3, pl = dir / 3;
    return ((r * g.cols + g.cols - 1 - c) * 6 + (2 - d3) + 3 * pl) * 2 + (a & 1);
  }
  static __device__ __forceinline__ St initial(const Geo& g) {
    St s;
    const uint64_t two = (g.cols * 2 >= 64) ? ~0ULL : ((1ULL << (2 * g.cols)) - 1ULL);
    s.b0 = two;
    s.b1 = two << ((g.rows - 2) * g.cols);
    s.ply = 0;
    return s;
  }
};

// return of the player who made the last move into terminal state `s` (== -leaf_value, mcts.py:149,152)
__device__ __forceinline__ double mover_return(int outcome, int ply) {
  const int mover = (ply - 1) & 1;
  return outcome == 2 ? 0.0 : (outcome == mover ? 1.0 : -1.0);
}

}  // namespace az
