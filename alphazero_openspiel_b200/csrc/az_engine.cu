// az_engine.cu -- B200 (sm_100a) self-play MCTS engine behind the C-ABI of include/az_b200.h.
//
// Replaces, for thousands of independent trees at once, the reference's per-game Python search:
//   Node.select/get_value  mcts.py:38-52,68-80     -> sim_select()   (fp64 PUCT, lanes-per-tree argmax)
//   Node.expand            mcts.py:54-66           -> expand_node()
//   Node.update_recursive  mcts.py:82-89           -> backup_path()
//   MCTS.playout/search    mcts.py:126-180         -> k_step main loop
//   expand_root_dirichlet  mcts.py:182-190         -> expand_root()
//   MCTS.update_root       mcts.py:192-203         -> finish_move() / k_command + k_compact
//   AlphaZeroBot.step      alphazerobot.py:42-93   -> finish_move()
//   play_game_self targets game_utils.py:168-204   -> emit_record()
//   state_to_board         network.py:9-18         -> write_obs()
//
// Data layout in HBM (per engine):
//   hdr   [n_trees]            64-byte tree header (root/pending positions, phase, arena cursor)
//   nodes [n_trees][2][cap]    24-byte records {uint2 {N, link}, double Q, double P}; link = first_child << 8 | n_children
//   path  [n_trees][MAXD]      node indices root..leaf of the in-flight simulation
//   cache [2^log2 entries]     AZ_F_EVAL_CACHE: evaluator outputs by position (CacheHead + float priors, see cache_find)
// The children of a node are ONE contiguous block in legal (ascending action) order, so a lane group
// reads a node's child statistics with three coalesced loads; the winning child's {N, link} comes back by
// shuffle, which makes one dependent load round per tree level.  Actions are never stored: child k of a
// node is the k-th legal move of the position, recomputed from the register-resident bitboards.
// The two arena halves double-buffer the re-root compaction (BFS copy of the kept subtree).
//
// All PUCT / backup arithmetic is fp64 with explicit round-to-nearest intrinsics in the reference's
// operation order (SURVEY A.1, A.4); the file is also compiled with -fmad=false.

#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <string.h>
#include <math.h>
#include <new>
#include <vector>

#include "../../include/az_b200.h"
#include "az_games.cuh"

namespace az {

constexpr int PH_BEGIN = 6;  // internal: a search must be started (root eval request or first simulation)
constexpr int PH_COMPACT = 7;  // internal: waiting for k_compact to re-root (pend_node = the child to promote)
constexpr int BLOCK = 128;
#ifndef K_STEP_MIN_BLOCKS
#define K_STEP_MIN_BLOCKS 7  // <= 73 registers: all 1024 CTAs of a 16,384-tree Connect Four launch are resident in one wave
#endif

struct __align__(16) TreeHdr {
  uint64_t root_b0, root_b1;
  uint64_t pend_b0, pend_b1;
  int32_t root_node;
  int32_t alloc;
  int32_t sims_done;
  int32_t pend_node;
  int32_t pend_depth;
  int32_t pend_ply;
  int32_t root_ply;
  int32_t game_seq;
  uint8_t phase, half, err, uct;  // uct: this tree scores with the use_puct=False formula (see fresh_tree)
  int32_t fast_sims;  // AZ_F_PLAYOUT_CAP: simulations of the current search if it is a fast one; 0 = a full search (a zeroed
                      // header never looks like a finished search)
  int32_t forced_lo, forced_hi;  // AZ_F_FORCED_PLAYOUTS: k of the current search if it is a forced one, 0 = not forced; the
                                 // halves of a double (forced_k / set_forced_k): a double member changes the register
                                 // allocation of the step kernels that never read it
};
static_assert(sizeof(TreeHdr) == 80, "TreeHdr size");

__device__ __forceinline__ double forced_k(const TreeHdr& h) { return __hiloint2double(h.forced_hi, h.forced_lo); }
__device__ __forceinline__ void set_forced_k(TreeHdr& h, double k) {
  h.forced_lo = __double2loint(k);
  h.forced_hi = __double2hiint(k);
}

__device__ __forceinline__ St root_state(const TreeHdr& h) {
  St s;
  s.b0 = h.root_b0;
  s.b1 = h.root_b1;
  s.ply = h.root_ply;
  return s;
}
__device__ __forceinline__ St pend_state(const TreeHdr& h) {
  St s;
  s.b0 = h.pend_b0;
  s.b1 = h.pend_b1;
  s.ply = h.pend_ply;
  return s;
}
__device__ __forceinline__ void set_root(TreeHdr& h, const St& s) {
  h.root_b0 = s.b0;
  h.root_b1 = s.b1;
  h.root_ply = s.ply;
}
// the evaluator request of node `node` at depth `depth` of the tree, at position s
__device__ __forceinline__ void set_pend(TreeHdr& h, const St& s, int node, int depth) {
  h.pend_b0 = s.b0;
  h.pend_b1 = s.b1;
  h.pend_ply = s.ply;
  h.pend_node = node;
  h.pend_depth = depth;
}

// one in-flight evaluator request of a tree in virtual-loss mode (AZ_F_VIRTUAL_LOSS)
struct __align__(16) VlPend {
  uint64_t b0, b1;
  int32_t node, depth, ply, valid;
};

// AZ_F_RESIGN: the values of az_set_resign, and per tree the state of its current game.  Kept out of TreeHdr, which k_step
// carries through its whole loop; only finish_move touches ResignTree.
struct ResignCfg {
  double threshold;
  int32_t permille;
  int32_t pad;
};
struct ResignTree {
  double rmin[2];   // calibration game: minimum r of player 0 / 1 so far (2.0: not moved yet)
  int32_t game_seq; // game this entry belongs to (-1 after az_reset: initialised at the game's first searched position)
  int32_t calib;    // no-resign calibration game
};

// AZ_F_PLAYOUT_CAP: the values of az_set_playout_cap
struct PlayoutCapCfg {
  int32_t fast_playouts;
  int32_t full_permille;
};

struct Node;
struct Params {
  TreeHdr* hdr;
  Node* nodes;
  int32_t* path;
  uint8_t* rec;
  unsigned long long* rec_count;
  unsigned long long* ctr;
  int* games_started;
  int* compact_list;   // trees waiting for re-root compaction (k_compact work list)
  int* compact_count;  // [0] = entries, [1] = CTAs done
  long long* dbg;      // optional [n_trees][4]: cycles, phase in, sims this step, flags (az_debug_timing)
  VlPend* vl_pend;     // AZ_F_VIRTUAL_LOSS: [n_trees][vl_k] in-flight requests
  int vl_k;            // leaves in flight per tree (evaluator rows per tree); 1 in the exact mode
  uint8_t* cache;            // AZ_F_EVAL_CACHE table, nullptr when off
  unsigned long long cache_mask;
  uint32_t* cache_epoch;     // [0] epoch of the current weights, [1] epoch of the rows the next k_cache_insert stores
  ResignCfg* resign_cfg;     // AZ_F_RESIGN, nullptr when off
  ResignTree* resign_tree;   // AZ_F_RESIGN: [n_trees]
  PlayoutCapCfg* pcap_cfg;   // AZ_F_PLAYOUT_CAP, nullptr when off
  const double* logtab;  // AZ_F_UCT: log(n) for n < LOGTAB_N, computed on the host with the C library's log() -- the same
                         // function CPython's math.log calls, so the UCT scores are bit-equal to the reference's
  long long rec_cap;
  int max_games;
  int rec_stride;
  int n_trees, cap;
  int n_playouts, num_prob, noise_mode, eval_mode, eval_shift, max_sims, start_mod;
  int cycle_budget;  // az_config.step_cycle_budget
  uint32_t flags;
  uint64_t seed;
  double c_puct, keep, noise_w, alpha, temperature;
  Geo geo;
  double* forced_cfg;  // AZ_F_FORCED_PLAYOUTS: k of az_set_forced_playouts, nullptr when off
};

// the simulations of the current search, fixed when it begins (begin_search; k_command for MCTS.playout)
__device__ __forceinline__ int search_target(const Params& p, const TreeHdr& h) {
  return h.fast_sims ? h.fast_sims : p.n_playouts;
}

struct StepIO {
  const void* priors;
  const void* values;
  const double* noise;
  void* obs;
  int obs_format;
};

// ---------------------------------------------------------------- lane-group helpers
template <int G>
__device__ __forceinline__ unsigned group_mask() {
  if constexpr (G >= 32) {
    return 0xffffffffu;
  } else {
    const unsigned lane = threadIdx.x & 31u;
    return ((1u << G) - 1u) << (lane & ~(unsigned)(G - 1));
  }
}
template <int G, class T>
__device__ __forceinline__ T gshfl(unsigned m, T v, int src) { return __shfl_sync(m, v, src, G); }
template <int G, class T>
__device__ __forceinline__ T gshfl_xor(unsigned m, T v, int off) { return __shfl_xor_sync(m, v, off, G); }
template <int G>
__device__ __forceinline__ int gsum(unsigned m, int v) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(m, v, o, G);
  return v;
}
template <int G>
__device__ __forceinline__ double gsumd(unsigned m, double v) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(m, v, o, G);
  return v;
}
template <int G>
__device__ __forceinline__ int gscan_incl(unsigned m, int v, int lane) {
#pragma unroll
  for (int o = 1; o < G; o <<= 1) {
    const int t = __shfl_up_sync(m, v, o, G);
    if (lane >= o) v += t;
  }
  return v;
}
// argmax with first-index tie-break over (value, index); index INT_MAX = no candidate
template <int G>
__device__ __forceinline__ void gargmax(unsigned m, double& v, int& i) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) {
    const double ov = __shfl_xor_sync(m, v, o, G);
    const int oi = __shfl_xor_sync(m, i, o, G);
    if (oi != 0x7fffffff && (i == 0x7fffffff || ov > v || (ov == v && oi < i))) { v = ov; i = oi; }
  }
}

__device__ __forceinline__ void ctr_add(unsigned long long* s_ctr, int which, unsigned long long v) {
  if (v) atomicAdd(&s_ctr[which], v);
}

// the counters one tree accumulates in registers during a step kernel; flush (lane 0) adds them to the block's
struct StepCtr {
  unsigned long long sims = 0, depth = 0, children = 0, exp = 0, legal = 0, term = 0;
  __device__ __forceinline__ void flush(unsigned long long* s_ctr, int alloc) const {
    atomicMax(&s_ctr[AZ_CTR_PEAK_NODES], (unsigned long long)alloc);
    ctr_add(s_ctr, AZ_CTR_SIMS, sims);
    ctr_add(s_ctr, AZ_CTR_DEPTH, depth);
    ctr_add(s_ctr, AZ_CTR_CHILDREN, children);
    ctr_add(s_ctr, AZ_CTR_EXPANSIONS, exp);
    ctr_add(s_ctr, AZ_CTR_LEGAL, legal);
    ctr_add(s_ctr, AZ_CTR_TERMINAL, term);
  }
};

// the block's counters into the engine's, once every thread of the block is done with s_ctr
__device__ __forceinline__ void flush_block_counters(const Params& p, const unsigned long long* s_ctr) {
  __syncthreads();
  if (threadIdx.x < AZ_CTR_COUNT && s_ctr[threadIdx.x]) {
    if (threadIdx.x == AZ_CTR_PEAK_NODES) atomicMax(&p.ctr[threadIdx.x], s_ctr[threadIdx.x]);
    else atomicAdd(&p.ctr[threadIdx.x], s_ctr[threadIdx.x]);
  }
}

// expand_node found no room for the children in the arena half: flag the tree and count the overflow
__device__ __forceinline__ void arena_overflow(TreeHdr& h, int lane, unsigned long long* s_ctr) {
  h.err = 1;
  if (lane == 0) ctr_add(s_ctr, AZ_CTR_OVERFLOW, 1);
}

// ---------------------------------------------------------------- evaluator inputs
struct EvalKey {
  uint64_t k;
};
__device__ __forceinline__ EvalKey eval_key(const Params& p, const St& s) {
  EvalKey e;
  e.k = mix64(s.b0 ^ mix64(s.b1 ^ mix64(p.seed + (uint64_t)(s.ply & 1))));
  return e;
}
__device__ __forceinline__ double eval_prior(const Params& p, const StepIO& io, int tree, const EvalKey& ek, int a) {
  if (p.eval_mode == AZ_EVAL_EXTERNAL) {
    const size_t idx = (size_t)tree * p.geo.n_actions + a;
    return (p.flags & AZ_F_PRIORS_F64) ? ((const double*)io.priors)[idx] : (double)((const float*)io.priors)[idx];
  }
  if (p.eval_mode == AZ_EVAL_UNIFORM) return 1.0 / (double)p.geo.n_actions;
  if (p.eval_mode == AZ_EVAL_ROLLOUT) return 1.0;   // np.ones(num_distinct_actions), mcts.py:222
  const uint64_t ha = mix64(ek.k + (uint64_t)(a + 1) * 0xD1B54A32D192ED03ULL);
  return (double)(1 + (int)((ha >> 40) & 0x3FF)) * exp2((double)-(10 + p.eval_shift));
}
// MCTS.random_rollout (mcts.py:205-223) on the device: one uniformly random playout from the position, scored for the player
// to move there.  The move stream is a pure function of (seed, position): r_j = mix64(key + (j+1) * golden), pick = r_j % L
// (oracle: oz_synth_eval kind 2), so the batched engine, the oracle and repeated runs agree bit for bit.
template <class GM>
__device__ double rollout_value(const Params& p, St s, const EvalKey& ek) {
  const int mover = s.ply & 1;
  for (uint64_t j = 0;; ++j) {
    const int out = GM::outcome(s, p.geo);
    if (out >= 0) return out == 2 ? 0.0 : (out == mover ? 1.0 : -1.0);
    const typename GM::Legal lg = GM::legal(s, p.geo);
    const int n = GM::count(lg);
    const uint64_t r = mix64(ek.k + (j + 1) * 0x9E3779B97F4A7C15ULL);
    s = GM::apply(s, p.geo, GM::action_of(lg, s, p.geo, (int)(r % (uint64_t)n)));
  }
}
template <class GM>
__device__ __forceinline__ double eval_value(const Params& p, const StepIO& io, int tree, const EvalKey& ek, const St& s) {
  if (p.eval_mode == AZ_EVAL_EXTERNAL)
    return (p.flags & AZ_F_PRIORS_F64) ? ((const double*)io.values)[tree] : (double)((const float*)io.values)[tree];
  if (p.eval_mode == AZ_EVAL_UNIFORM) return 0.0;
  if (p.eval_mode == AZ_EVAL_ROLLOUT) return rollout_value<GM>(p, s, ek);
  return (double)((int)((ek.k >> 20) & 31) - 16) / 16.0;
}

// ---------------------------------------------------------------- evaluator output cache (AZ_F_EVAL_CACHE)
// One direct-mapped entry per slot: CacheHead, float priors[MAXC] in legal order, and a 32-bit insertion lock in the last
// word; the stride is a power of two (64 B for Connect Four, 256 B for Breakthrough).  tag = epoch << 1 | (ply & 1), and the
// epoch starts at 1, so a zeroed slot never matches.  The evaluator's output is a function of (b0, b1, ply & 1) alone (the
// observation planes are built from exactly that), so a hit gives the float values a new evaluator row would give.
struct CacheHead {
  uint64_t b0, b1;
  uint32_t tag;
  float value;
};
static_assert(sizeof(CacheHead) == 24, "CacheHead size");
template <class GM>
__host__ __device__ constexpr int cache_stride() {
  int s = 1;
  while (s < (int)sizeof(CacheHead) + 4 * GM::MAXC + 4) s *= 2;
  return s;
}
template <class GM>
__device__ __forceinline__ uint8_t* cache_slot(const Params& p, const St& s) {
  return p.cache + (size_t)(eval_key(p, s).k & p.cache_mask) * cache_stride<GM>();
}
// The entry of position s under the current weights, or nullptr.  The full key is compared: a hash collision is a miss.
template <class GM>
__device__ __forceinline__ const CacheHead* cache_find(const Params& p, const St& s) {
  const CacheHead* e = reinterpret_cast<const CacheHead*>(cache_slot<GM>(p, s));
  const uint32_t tag = (p.cache_epoch[0] << 1) | (uint32_t)(s.ply & 1);
  return (e->b0 == s.b0 && e->b1 == s.b1 && e->tag == tag) ? e : nullptr;
}
__device__ __forceinline__ const float* cache_priors(const CacheHead* e) { return reinterpret_cast<const float*>(e + 1); }

// Gamma(alpha<1) by Marsaglia-Tsang on alpha+1 with the U^(1/alpha) boost; counter stream 5.
__device__ double gamma_draw(double alpha, uint64_t seed, uint64_t tree, uint64_t gseq, uint64_t ply, int child) {
  const double d = alpha + 1.0 - 1.0 / 3.0, c = 1.0 / sqrt(9.0 * d);
  for (int att = 0; att < 64; ++att) {
    // four draws per attempt, 64 attempts: 256 counter indices per child, no overlap between children or attempts
    const uint64_t base = (uint64_t)child * 256 + (uint64_t)att * 4;
    const uint64_t r0 = counter(seed, tree, gseq, ply, base + 0, 5);
    const uint64_t r1 = counter(seed, tree, gseq, ply, base + 1, 5);
    const uint64_t r2 = counter(seed, tree, gseq, ply, base + 2, 5);
    const double u0 = ((double)(r0 >> 11) + 1.0) * (1.0 / 9007199254740992.0);
    const double u1 = ((double)(r1 >> 11) + 0.5) * (1.0 / 9007199254740992.0);
    const double u2 = ((double)(r2 >> 11) + 1.0) * (1.0 / 9007199254740992.0);
    const double x = sqrt(-2.0 * log(u0)) * cospi(2.0 * u1);
    double v = 1.0 + c * x;
    if (v <= 0.0) continue;
    v = v * v * v;
    const uint64_t r3 = counter(seed, tree, gseq, ply, base + 3, 5);
    const double u3 = ((double)(r3 >> 11) + 1.0) * (1.0 / 9007199254740992.0);
    if (log(u3) < 0.5 * x * x + d - d * v + d * log(v)) return d * v * pow(u2, 1.0 / alpha);
  }
  return alpha;
}

// ---------------------------------------------------------------- observation (network.py:9-18)
template <class GM, int G>
__device__ __forceinline__ void write_obs(const Params& p, const StepIO& io, int tree, int lane, const St& s) {
  if (io.obs_format == AZ_OBS_NONE || io.obs == nullptr) return;
  const int n = p.geo.cells;
  const uint64_t pl0 = GM::plane(s, p.geo, 0), pl1 = GM::plane(s, p.geo, 1), pl2 = GM::plane(s, p.geo, 2);
  const int cur = s.ply & 1;
  if (io.obs_format == AZ_OBS_BF16_NHWC) {
    uint2* out = reinterpret_cast<uint2*>(io.obs) + (size_t)tree * n;
    const uint32_t one = 0x3F80u;  // bf16 1.0
    for (int c = lane; c < n; c += G) {
      uint2 v;
      v.x = (((pl0 >> c) & 1ULL) ? one : 0u) | ((((pl1 >> c) & 1ULL) ? one : 0u) << 16);
      v.y = (((pl2 >> c) & 1ULL) ? one : 0u) | ((cur ? one : 0u) << 16);
      out[c] = v;
    }
  } else {
    float* out = reinterpret_cast<float*>(io.obs) + (size_t)tree * 4 * n;
    for (int i = lane; i < 4 * n; i += G) {
      const int ch = i / n, c = i - ch * n;
      const uint64_t pm = ch == 0 ? pl0 : (ch == 1 ? pl1 : pl2);
      out[i] = ch == 3 ? (float)cur : (float)((pm >> c) & 1ULL);
    }
  }
}

// ---------------------------------------------------------------- tree primitives
// One 24-byte record per node: {N, link, Q, P}.  The children of a node are one contiguous run of records, so the three
// 8-byte fields that a lane group reads per child sit in the same one or two 128-byte lines (and the same DRAM page).
struct __align__(8) Node {
  uint2 nl;   // x = N (visit count), y = link = first_child << 8 | n_children
  double q;   // mean value
  double p;   // prior
};
static_assert(sizeof(Node) == 24, "Node size");
struct Arena {
  Node* nd;
  __device__ __forceinline__ uint2& nl(int i) const { return nd[i].nl; }
  __device__ __forceinline__ double& q(int i) const { return nd[i].q; }
  __device__ __forceinline__ double& p(int i) const { return nd[i].p; }
};
__device__ __forceinline__ Arena arena_of(const Params& p, int tree, int half) {
  Arena a;
  a.nd = p.nodes + ((size_t)tree * 2 + half) * (size_t)p.cap;
  return a;
}

// Node.update_recursive (mcts.py:82-89): node at path[j] receives v * (-1)^(depth-j); Q <- (N*Q + v)/(N+1).
template <int G>
__device__ __forceinline__ void backup_path(const Arena& a, const int32_t* path, int depth, double v_leaf, int lane) {
  for (int j = lane; j <= depth; j += G) {
    const int node = path[j];
    const double v = ((depth - j) & 1) ? -v_leaf : v_leaf;
    const uint2 nl = a.nl(node);
    const double q = a.q(node);
    a.q(node) = __ddiv_rn(__dadd_rn(__dmul_rn((double)nl.x, q), v), (double)(nl.x + 1u));
    a.nl(node).x = nl.x + 1u;
  }
}

// Node.expand (mcts.py:54-66).  noise != nullptr: root Dirichlet mix (mcts.py:186-189), eta indexed by legal position.
// cached != nullptr: the priors come from an AZ_F_EVAL_CACHE entry (float, legal order) instead of the evaluator row.
// Returns false on arena overflow (nothing written).
template <class GM, int G>
__device__ __forceinline__ bool expand_node(const Params& p, const StepIO& io, const Arena& a, TreeHdr& h, int tree,
                                            int node, const St& s, int lane, unsigned gm, bool root_mix,
                                            const double* eta_lane /* [SLOTS] per-lane eta values */, int* L_out,
                                            const float* cached = nullptr) {
  const typename GM::Legal lg = GM::legal(s, p.geo);
  const int L = GM::count(lg);
  *L_out = L;
  const uint2 nl = a.nl(node);
  int fc;
  bool fresh;
  if ((nl.y & 0xffu) != 0) {  // children exist (re-expanded root): overwrite P only
    fc = (int)(nl.y >> 8);
    fresh = false;
  } else {
    if (h.alloc + L > p.cap) return false;
    fc = h.alloc;
    h.alloc += L;
    fresh = true;
    if (lane == 0) a.nl(node).y = ((unsigned)fc << 8) | (unsigned)L;
  }
  const EvalKey ek = eval_key(p, s);
#pragma unroll
  for (int sl = 0; sl < GM::SLOTS; ++sl) {
    const int i = lane + sl * G;
    if (i < L) {
      double pr = cached ? (double)cached[i] : eval_prior(p, io, tree, ek, GM::action_of(lg, s, p.geo, i));
      if (root_mix) pr = __dadd_rn(__dmul_rn(p.keep, pr), __dmul_rn(p.noise_w, eta_lane[sl]));
      a.p(fc + i) = pr;
      if (fresh) {
        a.nl(fc + i) = make_uint2(0u, 0u);
        a.q(fc + i) = 0.0;
      }
    }
  }
  __syncwarp(gm);
  return true;
}

constexpr int LOGTAB_N = 1 << 20;  // parent visit counts covered by the AZ_F_UCT log table (a game has < 1e5 simulations)

// AZ_F_FORCED_PLAYOUTS: the forced-playout floor nf(c) = sqrt((k * P(c)) * N_root) of a root child
__device__ __forceinline__ double forced_floor(double k, double prior, unsigned n_root) {
  return __dsqrt_rn(__dmul_rn(__dmul_rn(k, prior), (double)n_root));
}

// One PUCT (or, UCT = true, use_puct=False) descent (mcts.py:139-142).  On return: node/depth/state of the childless node
// reached; path in spath.  FORCED (AZ_F_FORCED_PLAYOUTS) with forced_k > 0: at the root, a visited child below its floor
// (1 <= N(c) < nf(c)) scores +inf, so the first such child in legal order is taken.
template <class GM, int G, bool UCT, bool FORCED = false>
__device__ __forceinline__ void sim_select(const Params& p, const Arena& a, int root, St& s, int& node, int& depth,
                                           int32_t* spath, int lane, unsigned gm, unsigned long long& n_children,
                                           bool& depth_overflow, bool tree_uct, double forced_k = 0.0) {
  node = root;
  depth = 0;
  if (lane == 0) spath[0] = root;
  uint2 cur = a.nl(root);
  for (;;) {
    const int nc = (int)(cur.y & 0xffu);
    if (nc == 0) break;
    if (depth + 1 >= GM::MAXD) { depth_overflow = true; break; }
    const int fc = (int)(cur.y >> 8);
    const double sq = __dsqrt_rn((double)cur.x);
    // UCT: log(N_parent); a parent beyond the table (never in practice) is treated like the last entry and flagged
    const double lg_np = (UCT && tree_uct) ? p.logtab[cur.x < (unsigned)LOGTAB_N ? cur.x : (unsigned)(LOGTAB_N - 1)] : 0.0;
    if (UCT && tree_uct && cur.x >= (unsigned)LOGTAB_N) depth_overflow = true;
    const bool forced = FORCED && depth == 0 && forced_k > 0.0;
    double best = 0.0;
    int bi = 0x7fffffff;
    uint2 bnl = make_uint2(0u, 0u);
#pragma unroll
    for (int sl = 0; sl < GM::SLOTS; ++sl) {
      const int i = lane + sl * G;
      if (i < nc) {
        const uint2 nl = a.nl(fc + i);
        const double q = a.q(fc + i);
        const double pp = a.p(fc + i);
        double sc;
        if (UCT && tree_uct) {
          // inf if N == 0 else Q + ((c_puct * P) * sqrt(log(N_parent) / N))      mcts.py:80
          sc = nl.x == 0u ? __longlong_as_double(0x7ff0000000000000LL)
                          : __dadd_rn(q, __dmul_rn(__dmul_rn(p.c_puct, pp), __dsqrt_rn(__ddiv_rn(lg_np, (double)nl.x))));
        } else {
          // Q + (((c_puct * P) * sqrt(N_parent)) / (N + 1))      mcts.py:78
          const double u = __ddiv_rn(__dmul_rn(__dmul_rn(p.c_puct, pp), sq), (double)(nl.x + 1u));
          sc = __dadd_rn(q, u);
          if (forced && nl.x >= 1u && (double)nl.x < forced_floor(forced_k, pp, cur.x))
            sc = __longlong_as_double(0x7ff0000000000000LL);
        }
        if (bi == 0x7fffffff || sc > best) { best = sc; bi = i; bnl = nl; }
      }
    }
    int wi = bi;
    gargmax<G>(gm, best, wi);
    const int owner = wi % G;  // the owner lane's local best is the winner
    cur.x = gshfl<G>(gm, bnl.x, owner);
    cur.y = gshfl<G>(gm, bnl.y, owner);
    const typename GM::Legal lg = GM::legal(s, p.geo);
    s = GM::apply(s, p.geo, GM::action_of(lg, s, p.geo, wi));
    node = fc + wi;
    ++depth;
    if (lane == 0) spath[depth] = node;
    n_children += (unsigned long long)nc;
  }
  __syncwarp(gm);
}

// game_utils.py:182-194 -- greedy descent by N+P among visited children.
template <class GM, int G>
__device__ double offpolicy_value(const Arena& a, int root, int lane, unsigned gm) {
  int node = root;
  uint2 cur = a.nl(root);
  double value = 0.0, mult = 1.0;
  for (;;) {
    const int nc = (int)(cur.y & 0xffu);
    if (nc == 0) break;
    const int fc = (int)(cur.y >> 8);
    value = a.q(node);
    double best = 0.0;
    int bi = 0x7fffffff;
    uint2 bnl = make_uint2(0u, 0u);
#pragma unroll
    for (int sl = 0; sl < GM::SLOTS; ++sl) {
      const int i = lane + sl * G;
      if (i < nc) {
        const uint2 nl = a.nl(fc + i);
        const double sc = nl.x > 0 ? __dadd_rn((double)nl.x, a.p(fc + i)) : -99.0;
        if (bi == 0x7fffffff || sc > best) { best = sc; bi = i; bnl = nl; }
      }
    }
    int wi = bi;
    gargmax<G>(gm, best, wi);
    const int owner = wi % G;
    cur.x = gshfl<G>(gm, bnl.x, owner);
    cur.y = gshfl<G>(gm, bnl.y, owner);
    node = fc + wi;
    mult = -mult;
  }
  if (cur.x > 0) {
    value = a.q(node);
    mult = -mult;
  }
  return value * mult;
}

template <int G>
// uct_root: the reference keeps use_puct on every Node, children inherit it from their parent (mcts.py:64), and only the root
// that update_root creates for a leaf root (mcts.py:199-200) gets the MCTS object's flag -- the root of MCTS.__init__
// (mcts.py:122) is built without it.  So the formula is a property of the tree, decided when its root is created.
__device__ __forceinline__ void fresh_tree(const Params& p, TreeHdr& h, int tree, int lane, unsigned gm, bool uct_root = false) {
  h.uct = uct_root ? 1 : 0;
  const Arena a = arena_of(p, tree, h.half);
  if (lane == 0) {
    a.nl(0) = make_uint2(0u, 0u);  // Node(None, 0.0)  mcts.py:122
    a.q(0) = 0.0;
    a.p(0) = 0.0;
  }
  h.root_node = 0;
  h.alloc = 1;
  __syncwarp(gm);
}

template <class GM>
__device__ St start_position(const Params& p, int tree, int gseq) {
  St s = GM::initial(p.geo);
  if (!(p.flags & AZ_F_RANDOM_START) || p.start_mod <= 0) return s;
  const int k = (int)(counter(p.seed, tree, gseq, 0, 0, 4) % (uint64_t)p.start_mod);
  for (uint64_t attempt = 0;; ++attempt) {
    s = GM::initial(p.geo);
    bool ok = true;
    for (int j = 0; j < k; ++j) {
      const typename GM::Legal lg = GM::legal(s, p.geo);
      const int n = GM::count(lg);
      const int pick = (int)(counter(p.seed, tree, gseq, j, attempt, 3) % (uint64_t)n);
      s = GM::apply(s, p.geo, GM::action_of(lg, s, p.geo, pick));
      if (GM::outcome(s, p.geo) >= 0) { ok = false; break; }
    }
    if (ok) return s;
  }
}

// training record (game_utils.py:168-194); returns through *slot_out the record slot or -1
template <class GM, int G>
__device__ void emit_record(const Params& p, int tree, const TreeHdr& h, const St& s, int kind, int action, int n_legal,
                            int root_n, double root_q, double v_a0c, double v_off, int end, const int* counts_lane,
                            const typename GM::Legal* lg, int lane, unsigned gm, unsigned long long* s_ctr) {
  long long slot = 0;
  if (lane == 0) slot = (long long)atomicAdd(p.rec_count, 1ULL);
  slot = gshfl<G>(gm, slot, 0);
  if (slot >= p.rec_cap) {
    if (lane == 0) ctr_add(s_ctr, AZ_CTR_OVERFLOW, 1);
    return;
  }
  uint8_t* base = p.rec + (size_t)slot * p.rec_stride;
  if (lane == 0) {
    az_record r;
    r.tree = tree;
    r.game_seq = h.game_seq;
    r.ply = s.ply;
    r.action = action;
    r.n_legal = n_legal;
    r.kind = kind;
    r.root_n = root_n;
    r.end = end;
    r.bb[0] = s.b0;
    r.bb[1] = s.b1;
    r.root_q = root_q;
    r.v_a0c = v_a0c;
    r.v_offpolicy = v_off;
    *reinterpret_cast<az_record*>(base) = r;
  }
  int32_t* cnt = reinterpret_cast<int32_t*>(base + sizeof(az_record));
  int16_t* act = reinterpret_cast<int16_t*>(base + sizeof(az_record) + 4 * GM::MAXC);
#pragma unroll
  for (int sl = 0; sl < GM::SLOTS; ++sl) {
    const int i = lane + sl * G;
    if (i < GM::MAXC) {
      const bool have = counts_lane && lg && i < n_legal;
      cnt[i] = have ? counts_lane[sl] : 0;
      act[i] = have ? (int16_t)GM::action_of(*lg, s, p.geo, i) : (int16_t)-1;
    }
  }
}

// A game is over (terminal position or resignation): count it, then start the next game in the slot (AZ_F_AUTO_RESTART,
// within the max_games tickets) or leave the tree idle at the final position s_end.
template <class GM, int G>
__device__ void end_game(const Params& p, TreeHdr& h, int tree, int lane, unsigned gm, unsigned long long* s_ctr,
                         const St& s_end) {
  if (lane == 0) ctr_add(s_ctr, AZ_CTR_GAMES, 1);
  bool restart = (p.flags & AZ_F_AUTO_RESTART) != 0;
  if (restart && p.max_games > 0) {
    int ticket = 0;
    if (lane == 0) ticket = atomicAdd(p.games_started, 1);
    ticket = gshfl<G>(gm, ticket, 0);
    restart = ticket < p.max_games;
  }
  if (restart) {
    h.game_seq += 1;
    set_root(h, start_position<GM>(p, tree, h.game_seq));
    fresh_tree<G>(p, h, tree, lane, gm);
    h.phase = PH_BEGIN;
  } else {
    set_root(h, s_end);
    h.phase = AZ_PH_IDLE;
  }
}

// AZ_F_RESIGN at a searched root of the mover m = ply & 1 (see AZ_F_RESIGN in az_b200.h): starts the tree's ResignTree entry
// at the game's first searched position, keeps a calibration game's minimum r, and returns whether the game resigns here.
template <int G>
__device__ bool resign_check(const Params& p, const TreeHdr& h, int tree, int lane, unsigned gm, int ply, double root_q,
                             double a0c) {
  ResignTree* rp = p.resign_tree + tree;
  ResignTree t = *rp;
  const ResignCfg c = *p.resign_cfg;
  if (t.game_seq != h.game_seq) {
    t.game_seq = h.game_seq;
    t.calib = (int)(counter(p.seed, tree, h.game_seq, 0, 0, 6) % 1000ULL) < c.permille ? 1 : 0;
    t.rmin[0] = 2.0;
    t.rmin[1] = 2.0;
  }
  const double r = a0c > -root_q ? a0c : -root_q;
  if (t.calib) {
    if (ply & 1) {
      if (r < t.rmin[1]) t.rmin[1] = r;
    } else {
      if (r < t.rmin[0]) t.rmin[0] = r;
    }
  }
  __syncwarp(gm);  // every lane has read the entry before lane 0 overwrites it
  if (lane == 0) *rp = t;
  return !t.calib && r < c.threshold;
}

// AZ_F_RESIGN, game over at a terminal position: for a calibration game, count it and its would-be false resignations
// (players whose minimum r is below the current threshold and who did not lose; out = GM::outcome) and return end = 2 with
// the two minima, else end = 0.
template <int G>
__device__ int resign_game_over(const Params& p, int tree, int lane, unsigned gm, int out, unsigned long long* s_ctr,
                                double& rmin0, double& rmin1) {
  __syncwarp(gm);  // lane 0's write of the entry in resign_check is visible
  const ResignTree t = p.resign_tree[tree];
  if (!t.calib) return 0;
  rmin0 = t.rmin[0];
  rmin1 = t.rmin[1];
  if (lane == 0) {
    const double thr = p.resign_cfg->threshold;
    ctr_add(s_ctr, AZ_CTR_RESIGN_SAMPLES, 1);
    ctr_add(s_ctr, AZ_CTR_RESIGN_FALSE, (unsigned long long)((rmin0 < thr && out != 1) + (rmin1 < thr && out != 0)));
  }
  return 2;
}

// AZ_F_FORCED_PLAYOUTS policy target pruning (see az_b200.h) of the root child counts cnt (per lane, legal order; qv their
// Q) after a forced search with k = forced_k.  c* (the first maximal count) keeps its count; every other visited child drops
// to the smallest n >= N - nf whose PUCT score stays below c*'s (sim_select's expression), and a remainder of 1 to 0.  Changes
// no node.  Returns the new total.
template <class GM, int G>
__device__ int prune_counts(const Params& p, const Arena& a, int fc, int nc, unsigned n_root, double forced_k, int* cnt,
                            const double* qv, int lane, unsigned gm) {
  double bv = -1.0;
  int bi = 0x7fffffff;
#pragma unroll
  for (int sl = 0; sl < GM::SLOTS; ++sl) {
    const int i = lane + sl * G;
    if (i < nc && (bi == 0x7fffffff || (double)cnt[sl] > bv)) { bv = (double)cnt[sl]; bi = i; }
  }
  gargmax<G>(gm, bv, bi);
  const double sq = __dsqrt_rn((double)n_root);
  const double s_star =
      __dadd_rn(a.q(fc + bi), __ddiv_rn(__dmul_rn(__dmul_rn(p.c_puct, a.p(fc + bi)), sq), (double)((unsigned)bv + 1u)));
  int total = 0;
#pragma unroll
  for (int sl = 0; sl < GM::SLOTS; ++sl) {
    const int i = lane + sl * G;
    if (i < nc && i != bi && cnt[sl] > 0) {
      const double pp = a.p(fc + i);
      const double cps = __dmul_rn(__dmul_rn(p.c_puct, pp), sq);
      const double lo = __dsub_rn((double)cnt[sl], forced_floor(forced_k, pp, n_root));
      int n = cnt[sl];
      // score(n - 1) = Q + cps / n is non-increasing in n: step down while n - 1 is still allowed
      while (n > 0 && (double)(n - 1) >= lo && __dadd_rn(qv[sl], __ddiv_rn(cps, (double)n)) < s_star) --n;
      cnt[sl] = n == 1 ? 0 : n;
    }
    total += cnt[sl];
  }
  return gsum<G>(gm, total);
}

// AlphaZeroBot.step after the search (alphazerobot.py:72-93) + play_game_self bookkeeping (game_utils.py:156-204).
// Sets h.phase to PH_BEGIN / AZ_PH_IDLE / AZ_PH_SEARCH_DONE.  FORCED: after a forced search (AZ_F_FORCED_PLAYOUTS) the
// move choice and the ply record use the pruned counts (prune_counts); everything else uses the tree as it is.
template <class GM, int G, bool FORCED = false>
__device__ void finish_move(const Params& p, TreeHdr& h, int tree, int lane, unsigned gm, unsigned long long* s_ctr) {
  const Arena a = arena_of(p, tree, h.half);
  const St s = root_state(h);
  const typename GM::Legal lg = GM::legal(s, p.geo);
  const int L = GM::count(lg);
  const uint2 rnl = a.nl(h.root_node);
  const int fc = (int)(rnl.y >> 8);
  const int nc = (int)(rnl.y & 0xffu);  // == L once expanded
  int cnt[GM::SLOTS];
  double qv[GM::SLOTS];
  int total = 0;
  double a0c = -99.0;
  int a0c_i = 0x7fffffff;
#pragma unroll
  for (int sl = 0; sl < GM::SLOTS; ++sl) {
    const int i = lane + sl * G;
    cnt[sl] = 0;
    qv[sl] = 0.0;
    if (i < nc) {
      cnt[sl] = (int)a.nl(fc + i).x;
      qv[sl] = a.q(fc + i);
      const double v = cnt[sl] > 0 ? qv[sl] : -99.0;
      if (a0c_i == 0x7fffffff || v > a0c) { a0c = v; a0c_i = i; }
    }
    total += cnt[sl];
  }
  total = gsum<G>(gm, total);
  gargmax<G>(gm, a0c, a0c_i);
  const double root_q = a.q(h.root_node);
  double v_off = 0.0;
  if ((p.flags & AZ_F_RECORDS) && (p.flags & AZ_F_OFFPOLICY)) v_off = offpolicy_value<GM, G>(a, h.root_node, lane, gm);

  if (p.flags & AZ_F_MANUAL) {
    if (p.flags & AZ_F_RECORDS)
      emit_record<GM, G>(p, tree, h, s, 0, -1, L, (int)rnl.x, root_q, a0c, v_off, 0, cnt, &lg, lane, gm, s_ctr);
    h.phase = AZ_PH_SEARCH_DONE;
    return;
  }

  if (FORCED && forced_k(h) > 0.0 && nc > 0)
    total = prune_counts<GM, G>(p, a, fc, nc, rnl.x, forced_k(h), cnt, qv, lane, gm);
  const int ply_end = h.fast_sims ? 3 : 0;  // the ply record's end: 3 marks a fast search (AZ_F_PLAYOUT_CAP)
  if ((p.flags & AZ_F_RESIGN) && resign_check<G>(p, h, tree, lane, gm, s.ply, root_q, a0c)) {
    if (p.flags & AZ_F_RECORDS) {
      emit_record<GM, G>(p, tree, h, s, 0, -1, L, (int)rnl.x, root_q, a0c, v_off, ply_end, cnt, &lg, lane, gm, s_ctr);
      const double ret0 = (s.ply & 1) ? 1.0 : -1.0;  // the mover loses
      emit_record<GM, G>(p, tree, h, s, 1, -1, 0, 0, ret0, 0.0, 0.0, 1, nullptr, nullptr, lane, gm, s_ctr);
    }
    if (lane == 0) ctr_add(s_ctr, AZ_CTR_RESIGNS, 1);
    end_game<GM, G>(p, h, tree, lane, gm, s_ctr, s);
    return;
  }

  // ---- move choice
  int k = 0;
  if ((p.flags & AZ_F_SAMPLE_MOVES) && s.ply < p.num_prob && total > 0) {
    const uint64_t r64 = counter(p.seed, tree, h.game_seq, s.ply, 0, 2);
    if (p.temperature == 1.0) {
      // proportional to visit counts: r = floor(u32 * total / 2^32); first child with cumulative count > r
      const long long r = (long long)(((r64 >> 32) * (uint64_t)total) >> 32);
      int off = 0, pick = 0x7fffffff;
#pragma unroll
      for (int sl = 0; sl < GM::SLOTS; ++sl) {
        const int incl = gscan_incl<G>(gm, cnt[sl], lane) + off;
        if (incl > r && cnt[sl] > 0) pick = min(pick, lane + sl * G);
        off = gshfl<G>(gm, incl, G - 1);
      }
#pragma unroll
      for (int o = G / 2; o > 0; o >>= 1) pick = min(pick, __shfl_xor_sync(gm, pick, o, G));
      k = pick;
    } else {
      // p_i ~ count_i^(1/T)  (alphazerobot.py:78); serial inverse-CDF over children on every lane
      const double invT = 1.0 / p.temperature;
      double wsum = 0.0;
      for (int i = 0; i < nc; ++i) {
        const int c = gshfl<G>(gm, cnt[i / G], i % G);
        wsum += pow((double)c, invT);
      }
      const double u = ((double)(r64 >> 11)) * (1.0 / 9007199254740992.0) * wsum;
      double cum = 0.0;
      k = -1;
      int lastpos = 0;
      for (int i = 0; i < nc; ++i) {
        const int c = gshfl<G>(gm, cnt[i / G], i % G);
        if (c > 0) lastpos = i;
        cum += pow((double)c, invT);
        if (k < 0 && c > 0 && cum > u) k = i;
      }
      if (k < 0) k = lastpos;
    }
  } else {
    // np.argmax: first maximal visit count (alphazerobot.py:86)
    double bv = -1.0;
    int bi = 0x7fffffff;
#pragma unroll
    for (int sl = 0; sl < GM::SLOTS; ++sl) {
      const int i = lane + sl * G;
      if (i < nc && (bi == 0x7fffffff || (double)cnt[sl] > bv)) { bv = (double)cnt[sl]; bi = i; }
    }
    gargmax<G>(gm, bv, bi);
    k = bi;
  }
  const int action = GM::action_of(lg, s, p.geo, k);
  if (p.flags & AZ_F_RECORDS)
    emit_record<GM, G>(p, tree, h, s, 0, action, L, (int)rnl.x, root_q, a0c, v_off, ply_end, cnt, &lg, lane, gm, s_ctr);

  // ---- apply (game_utils.py:197)
  const St s2 = GM::apply(s, p.geo, action);
  if (lane == 0) ctr_add(s_ctr, AZ_CTR_MOVES, 1);
  const int out = GM::outcome(s2, p.geo);
  if (out >= 0) {
    double rmin0 = 0.0, rmin1 = 0.0;
    int end = 0;
    if (p.flags & AZ_F_RESIGN) end = resign_game_over<G>(p, tree, lane, gm, out, s_ctr, rmin0, rmin1);
    if (p.flags & AZ_F_RECORDS) {
      const double ret0 = out == 2 ? 0.0 : (out == 0 ? 1.0 : -1.0);
      emit_record<GM, G>(p, tree, h, s2, 1, -1, 0, 0, ret0, rmin0, rmin1, end, nullptr, nullptr, lane, gm, s_ctr);
    }
    end_game<GM, G>(p, h, tree, lane, gm, s_ctr, s2);
    return;
  }
  set_root(h, s2);
  if ((p.flags & AZ_F_KEEP_TREE) && nc > 0) {
    // MCTS.update_root (mcts.py:192-203).  While the arena half still has room for the worst case of one more search
    // (every simulation expands one leaf), the chosen child simply becomes the root in place and the discarded siblings
    // stay behind as garbage; the tree continues with its next root evaluation in this very launch.
    if (!(p.flags & AZ_F_EAGER_COMPACT) && (long long)h.alloc + (long long)(p.n_playouts + 1) * GM::MAXC <= (long long)p.cap) {
      h.root_node = fc + k;
      h.phase = PH_BEGIN;
      return;
    }
    // Otherwise the kept subtree is copied into the other half (hundreds of dependent loads): done by k_compact, off this
    // kernel's critical path, so that one moving tree does not set the duration of the whole lock-step launch.
    h.pend_node = fc + k;
    h.phase = PH_COMPACT;
    if (lane == 0) p.compact_list[atomicAdd(p.compact_count, 1)] = tree;
    return;
  }
  fresh_tree<G>(p, h, tree, lane, gm);
  h.phase = PH_BEGIN;
}

// expand_root_dirichlet (mcts.py:182-190): the root expansion with the noise mix, from evaluator row `row` (cached == nullptr)
// or from an AZ_F_EVAL_CACHE entry's priors.  The noise is the tree's.  Leaves the tree in AZ_PH_RUN.
template <class GM, int G>
__device__ __forceinline__ void expand_root(const Params& p, const StepIO& io, TreeHdr& h, int tree, int row, int lane,
                                            unsigned gm, unsigned long long* s_ctr, const float* cached) {
  const Arena a = arena_of(p, tree, h.half);
  const St s = root_state(h);
  const typename GM::Legal lg = GM::legal(s, p.geo);
  const int L = GM::count(lg);
  double eta[GM::SLOTS];
#pragma unroll
  for (int sl = 0; sl < GM::SLOTS; ++sl) eta[sl] = 0.0;
  if (p.noise_mode == AZ_NOISE_HOST) {
#pragma unroll
    for (int sl = 0; sl < GM::SLOTS; ++sl) {
      const int i = lane + sl * G;
      if (i < L) eta[sl] = io.noise[(size_t)tree * GM::MAXC + i];
    }
  } else if (p.noise_mode == AZ_NOISE_COUNTER) {
    double sum = 0.0;  // sequential sum in legal order, identical on every lane (oracle: oz_selfplay_game)
    for (int i = 0; i < L; ++i) {
      const double u = (double)((counter(p.seed, tree, h.game_seq, s.ply, i, 1) >> 11) + 1ULL) *
                       (1.0 / 9007199254740992.0);
      sum = __dadd_rn(sum, u);
#pragma unroll
      for (int sl = 0; sl < GM::SLOTS; ++sl)
        if (i == lane + sl * G) eta[sl] = u;
    }
#pragma unroll
    for (int sl = 0; sl < GM::SLOTS; ++sl) eta[sl] = __ddiv_rn(eta[sl], sum);
  } else if (p.noise_mode == AZ_NOISE_DIRICHLET) {
    double sum = 0.0;
#pragma unroll
    for (int sl = 0; sl < GM::SLOTS; ++sl) {
      const int i = lane + sl * G;
      if (i < L) eta[sl] = gamma_draw(p.alpha, p.seed, tree, h.game_seq, s.ply, i);
      sum += eta[sl];
    }
    sum = gsumd<G>(gm, sum);
#pragma unroll
    for (int sl = 0; sl < GM::SLOTS; ++sl) eta[sl] = sum > 0.0 ? eta[sl] / sum : 1.0 / (double)L;
  }
  int L2 = 0;
  if (!expand_node<GM, G>(p, io, a, h, row, h.root_node, s, lane, gm, true, eta, &L2, cached)) arena_overflow(h, lane, s_ctr);
  h.phase = AZ_PH_RUN;
  if (lane == 0) ctr_add(s_ctr, AZ_CTR_ROOT_EVALS, 1);
}

// ---------------------------------------------------------------- search operations of both step kernels
// MCTS.search (mcts.py:173-176) from PH_BEGIN.  Without root noise the simulations start at once (AZ_PH_RUN).  With it the root
// is expanded first: from an AZ_F_EVAL_CACHE hit, or through a root request to evaluator row `row` -- then the tree waits in
// AZ_PH_ROOT_EVAL and this returns true.  CACHE: the kernel looks up the cache (k_step_vl runs without one).
// AZ_F_PLAYOUT_CAP: a fast search (counter stream 7) runs fast_playouts simulations and starts like one without root noise.
// FORCED (AZ_F_FORCED_PLAYOUTS): a search with root noise takes the k of az_set_forced_playouts in force now (0: not forced).
template <class GM, int G, bool CACHE, bool FORCED = false>
__device__ __forceinline__ bool begin_search(const Params& p, const StepIO& io, TreeHdr& h, int tree, int row, int lane,
                                             unsigned gm, unsigned long long* s_ctr) {
  h.sims_done = 0;
  h.phase = AZ_PH_RUN;
  h.fast_sims = 0;
  if (FORCED) set_forced_k(h, 0.0);
  if (p.flags & AZ_F_PLAYOUT_CAP) {
    const PlayoutCapCfg c = *p.pcap_cfg;
    if ((int)(counter(p.seed, tree, h.game_seq, h.root_ply, 0, 7) % 1000ULL) >= c.full_permille) {
      h.fast_sims = c.fast_playouts;
      return false;
    }
  }
  if (p.noise_mode == AZ_NOISE_NONE) return false;
  if (FORCED) set_forced_k(h, *p.forced_cfg);
  const St s = root_state(h);
  const CacheHead* hit = CACHE && p.cache ? cache_find<GM>(p, s) : nullptr;
  if (hit) {
    expand_root<GM, G>(p, io, h, tree, row, lane, gm, s_ctr, cache_priors(hit));
    return false;
  }
  h.phase = AZ_PH_ROOT_EVAL;
  set_pend(h, s, h.root_node, 0);
  write_obs<GM, G>(p, io, row, lane, s);
  return true;
}

// Node.expand + node.update_recursive(-leaf_value) (mcts.py:146-152) of the non-terminal leaf `node` at position s, from
// evaluator row `row` or (cached != nullptr) from the AZ_F_EVAL_CACHE entry that holds the same values.  BACKUP is backup_path,
// or vl_backup for a path that carries a virtual loss.
template <class GM, int G, void (*BACKUP)(const Arena&, const int32_t*, int, double, int)>
__device__ __forceinline__ void apply_leaf(const Params& p, const StepIO& io, const Arena& a, TreeHdr& h, int row, int node,
                                           const St& s, const int32_t* path, int depth, const CacheHead* cached, int lane,
                                           unsigned gm, unsigned long long* s_ctr, StepCtr& c) {
  int L = 0;
  if (!expand_node<GM, G>(p, io, a, h, row, node, s, lane, gm, false, nullptr, &L, cached ? cache_priors(cached) : nullptr))
    arena_overflow(h, lane, s_ctr);
  const double v = cached ? (double)cached->value : eval_value<GM>(p, io, row, eval_key(p, s), s);
  BACKUP(a, path, depth, -v, lane);
  __syncwarp(gm);
  h.sims_done += 1;
  c.sims += 1;
  c.depth += depth;
  c.exp += 1;
  c.legal += L;
  if (cached && lane == 0) ctr_add(s_ctr, AZ_CTR_CACHE_HITS, 1);
}

// terminal leaf: leaf_value = -player_return(mover); node.update_recursive(-leaf_value)   mcts.py:148-152
template <int G>
__device__ __forceinline__ void terminal_leaf(const Arena& a, TreeHdr& h, const int32_t* path, int depth, int out, int ply,
                                              int lane, unsigned gm, StepCtr& c) {
  backup_path<G>(a, path, depth, mover_return(out, ply), lane);
  __syncwarp(gm);
  h.sims_done += 1;
  c.sims += 1;
  c.depth += depth;
  c.term += 1;
}

// ---------------------------------------------------------------- the step kernel
// FORCED: the instantiation of AZ_F_FORCED_PLAYOUTS engines (forced playouts in sim_select, pruning in finish_move)
template <class GM, bool UCT, bool FORCED = false>
__global__ void __launch_bounds__(BLOCK, K_STEP_MIN_BLOCKS) k_step(const Params p, const StepIO io) {
  constexpr int G = GM::G;
  __shared__ int32_t s_path[BLOCK / G][GM::MAXD];
  __shared__ unsigned long long s_ctr[AZ_CTR_COUNT];
  if (threadIdx.x < AZ_CTR_COUNT) s_ctr[threadIdx.x] = 0ULL;
  __syncthreads();
  const int tree = (int)((blockIdx.x * (unsigned)BLOCK + threadIdx.x) / G);
  const int lane = threadIdx.x % G;
  // the rows k_cache_insert stores next are evaluated (after this launch) with the current weights
  if (p.cache && blockIdx.x == 0 && threadIdx.x == 0) p.cache_epoch[1] = p.cache_epoch[0];
  if (tree < p.n_trees) {
    const unsigned gm = group_mask<G>();
    int32_t* spath = s_path[threadIdx.x / G];
    int32_t* gpath = p.path + (size_t)tree * GM::MAXD;
    const long long t_start = p.dbg ? clock64() : 0;
    const long long t_begin = p.cycle_budget > 0 ? clock64() : 0;
    TreeHdr h = p.hdr[tree];
    const int phase_in = h.phase;
    long long t_consume = 0;
    StepCtr c;

    // ---------------- 1. consume the evaluator outputs of the pending request
    if (h.phase == AZ_PH_LEAF_EVAL) {
      apply_leaf<GM, G, backup_path<G>>(p, io, arena_of(p, tree, h.half), h, tree, h.pend_node, pend_state(h), gpath,
                                        h.pend_depth, nullptr, lane, gm, s_ctr, c);
      h.phase = AZ_PH_RUN;
    } else if (h.phase == AZ_PH_ROOT_EVAL) {
      expand_root<GM, G>(p, io, h, tree, tree, lane, gm, s_ctr, nullptr);
    }

    if (p.dbg) t_consume = clock64() - t_start;
    // ---------------- 2. run until the next evaluator request
    int sims_this_step = 0;
    bool advanced = false;
    for (;;) {
      if (h.phase == PH_BEGIN && begin_search<GM, G, true, FORCED>(p, io, h, tree, tree, lane, gm, s_ctr)) break;
      if (h.phase != AZ_PH_RUN) {
        if (lane == 0) ctr_add(s_ctr, AZ_CTR_IDLE_SLOTS, 1);
        break;
      }
      if (h.sims_done >= search_target(p, h)) {
        if (advanced) {
          if (lane == 0) ctr_add(s_ctr, AZ_CTR_IDLE_SLOTS, 1);
          break;
        }
        finish_move<GM, G, FORCED>(p, h, tree, lane, gm, s_ctr);
        advanced = true;
        continue;
      }
      if (p.max_sims > 0 && sims_this_step >= p.max_sims) {
        if (lane == 0) ctr_add(s_ctr, AZ_CTR_IDLE_SLOTS, 1);
        break;
      }
      // step_cycle_budget: a tree whose simulations keep ending in terminal leaves stops once the launch has run this long
      // (the launch lasts as long as its slowest tree).  How the simulations of a search are spread over steps does not
      // change any result, only how many evaluator rows stay empty.
      if (p.cycle_budget > 0 && sims_this_step > 0) {
        const int over = gshfl<G>(gm, (int)(clock64() - t_begin > (long long)p.cycle_budget), 0);
        if (over) {
          if (lane == 0) ctr_add(s_ctr, AZ_CTR_IDLE_SLOTS, 1);
          break;
        }
      }
      // ---- one simulation (mcts.py:126-153)
      const Arena a = arena_of(p, tree, h.half);
      St s = root_state(h);
      int node, depth;
      bool dovf = false;
      sim_select<GM, G, UCT, FORCED>(p, a, h.root_node, s, node, depth, spath, lane, gm, c.children, dovf, h.uct != 0,
                                     FORCED ? forced_k(h) : 0.0);
      if (dovf) {
        h.err = 1;
        h.phase = AZ_PH_ERROR;
        if (lane == 0) ctr_add(s_ctr, AZ_CTR_OVERFLOW, 1);
        break;
      }
      const int out = depth > 0 ? GM::outcome(s, p.geo) : -1;
      ++sims_this_step;
      if (out >= 0) {
        terminal_leaf<G>(a, h, spath, depth, out, s.ply, lane, gm, c);
        if (p.flags & AZ_F_MANUAL) {  // MCTS.playout(state) leaves `state` at the leaf: keep the path for az_request_info
          for (int j = lane; j <= depth; j += G) gpath[j] = spath[j];
          h.pend_depth = depth;
        }
        continue;
      }
      // non-terminal leaf: its evaluation from the cache, exactly as the AZ_PH_LEAF_EVAL consume path would apply the row
      const CacheHead* hit = p.cache ? cache_find<GM>(p, s) : nullptr;
      if (hit) {
        apply_leaf<GM, G, backup_path<G>>(p, io, a, h, tree, node, s, spath, depth, hit, lane, gm, s_ctr, c);
        continue;
      }
      // otherwise request the evaluator (mcts.py:146)
      set_pend(h, s, node, depth);
      h.phase = AZ_PH_LEAF_EVAL;
      for (int j = lane; j <= depth; j += G) gpath[j] = spath[j];
      write_obs<GM, G>(p, io, tree, lane, s);
      break;
    }

    if (lane == 0) {
      p.hdr[tree] = h;
      if (p.dbg) {
        p.dbg[4 * tree + 0] = clock64() - t_start;
        p.dbg[4 * tree + 1] = phase_in;
        p.dbg[4 * tree + 2] = sims_this_step;
        p.dbg[4 * tree + 3] = t_consume * 2 + (advanced ? 1 : 0);
      }
      c.flush(s_ctr, h.alloc);
    }
  }
  flush_block_counters(p, s_ctr);
}

// ---------------------------------------------------------------- evaluator cache insertion (AZ_F_EVAL_CACHE)
// Runs right before k_step: stores the evaluator rows of every pending request (leaf or root) under the epoch of the weights
// that computed them.  Lookups happen only in the following k_step, so no reader sees a half-written entry.  Two writers of
// one launch may map to the same slot: the first to take the slot's lock writes the whole entry, the other skips its insert.
template <class GM>
__global__ void __launch_bounds__(BLOCK) k_cache_insert(const Params p, const StepIO io) {
  constexpr int G = GM::G;
  const int tree = (int)((blockIdx.x * (unsigned)BLOCK + threadIdx.x) / G);
  const int lane = threadIdx.x % G;
  if (tree >= p.n_trees) return;
  const TreeHdr& h = p.hdr[tree];
  if (h.phase != AZ_PH_LEAF_EVAL && h.phase != AZ_PH_ROOT_EVAL) return;
  const unsigned gm = group_mask<G>();
  const St s = pend_state(h);
  uint8_t* slot = cache_slot<GM>(p, s);
  unsigned* lock = reinterpret_cast<unsigned*>(slot + cache_stride<GM>() - 4);
  int got = 0;
  if (lane == 0) got = atomicCAS(lock, 0u, 1u) == 0u;
  if (!gshfl<G>(gm, got, 0)) return;
  const typename GM::Legal lg = GM::legal(s, p.geo);
  const int L = GM::count(lg);
  float* pri = reinterpret_cast<float*>(slot + sizeof(CacheHead));
  const float* row = (const float*)io.priors + (size_t)tree * p.geo.n_actions;
#pragma unroll
  for (int sl = 0; sl < GM::SLOTS; ++sl) {
    const int i = lane + sl * G;
    if (i < L) pri[i] = row[GM::action_of(lg, s, p.geo, i)];
  }
  if (lane == 0) {
    CacheHead e;
    e.b0 = s.b0;
    e.b1 = s.b1;
    e.tag = (p.cache_epoch[1] << 1) | (uint32_t)(s.ply & 1);
    e.value = ((const float*)io.values)[tree];
    *reinterpret_cast<CacheHead*>(slot) = e;
  }
  __threadfence();
  __syncwarp(gm);
  if (lane == 0) atomicExch(lock, 0u);
}

__global__ void k_cache_new_epoch(uint32_t* epoch) { epoch[0] += 1u; }

// ---------------------------------------------------------------- virtual-loss step kernel (AZ_F_VIRTUAL_LOSS)
// Throughput mode for SMALL pools (BASELINE configs[1]: 1,024 games cannot fill the evaluator with one row per tree): every
// tree keeps up to K leaves in flight, so the evaluator batch is n_trees * K rows (row = tree * K + slot).  The reference has
// no such mode (mcts.py:177-179 runs its playouts strictly one after the other); this is the usual virtual-loss scheme and is
// NOT bit-exact with the reference: while a leaf is in flight every node on its path carries one extra visit with value -1
// (Q <- (N*Q - 1)/(N + 1), N <- N + 1), which steers the following descents of the same step elsewhere; the real backup
// replaces that visit (Q <- (N*Q + 1 + v)/N).  A leaf that is already in flight ends the collection for this step (its
// link carries the marker 0xFFFFFF00).  Everything else is the exact kernel's code: sim_select, begin_search, expand_root
// (root noise), apply_leaf (with vl_backup), terminal_leaf and finish_move (move choice, records, re-rooting).  K = 1
// through this kernel is still not the exact path.
constexpr unsigned VL_MARK = 0xFFFFFF00u;

template <int G>
__device__ __forceinline__ void vl_apply(const Arena& a, const int32_t* path, int depth, int lane) {
  for (int j = lane; j <= depth; j += G) {
    const int node = path[j];
    const uint2 nl = a.nl(node);
    a.q(node) = ((double)nl.x * a.q(node) - 1.0) / (double)(nl.x + 1u);
    a.nl(node).x = nl.x + 1u;
  }
}
// real backup of a simulation whose path carries a virtual loss: the visit is already counted
template <int G>
__device__ __forceinline__ void vl_backup(const Arena& a, const int32_t* path, int depth, double v_leaf, int lane) {
  for (int j = lane; j <= depth; j += G) {
    const int node = path[j];
    const double v = ((depth - j) & 1) ? -v_leaf : v_leaf;
    const uint2 nl = a.nl(node);
    a.q(node) = ((double)nl.x * a.q(node) + 1.0 + v) / (double)nl.x;
  }
}

template <class GM, bool FORCED = false>
__global__ void __launch_bounds__(BLOCK, 4) k_step_vl(const Params p, const StepIO io) {
  constexpr int G = GM::G;
  __shared__ int32_t s_path[BLOCK / G][GM::MAXD];
  __shared__ unsigned long long s_ctr[AZ_CTR_COUNT];
  if (threadIdx.x < AZ_CTR_COUNT) s_ctr[threadIdx.x] = 0ULL;
  __syncthreads();
  const int tree = (int)((blockIdx.x * (unsigned)BLOCK + threadIdx.x) / G);
  const int lane = threadIdx.x % G;
  if (tree < p.n_trees) {
    const unsigned gm = group_mask<G>();
    const int K = p.vl_k;
    int32_t* spath = s_path[threadIdx.x / G];
    int32_t* gpaths = p.path + (size_t)tree * K * GM::MAXD;
    VlPend* pend = p.vl_pend + (size_t)tree * K;
    const int row0 = tree * K;
    TreeHdr h = p.hdr[tree];
    StepCtr c;

    // ---------------- 1. consume the evaluator rows of the requests in flight
    if (h.phase == AZ_PH_LEAF_EVAL) {
      const Arena a = arena_of(p, tree, h.half);
      for (int slot = 0; slot < K; ++slot) {
        const VlPend pe = pend[slot];
        if (!pe.valid) continue;
        St s;
        s.b0 = pe.b0;
        s.b1 = pe.b1;
        s.ply = pe.ply;
        if (lane == 0) a.nl(pe.node).y = 0u;   // drop the in-flight marker: expand_node sees a childless node
        __syncwarp(gm);
        apply_leaf<GM, G, vl_backup<G>>(p, io, a, h, row0 + slot, pe.node, s, gpaths + (size_t)slot * GM::MAXD, pe.depth,
                                        nullptr, lane, gm, s_ctr, c);
        if (lane == 0) pend[slot].valid = 0;
      }
      h.phase = AZ_PH_RUN;
    } else if (h.phase == AZ_PH_ROOT_EVAL) {
      expand_root<GM, G>(p, io, h, tree, row0, lane, gm, s_ctr, nullptr);
    }

    // ---------------- 2. collect up to K new leaves
    int n_pending = 0, sims_this_step = 0;
    bool advanced = false;
    for (;;) {
      if (h.phase == PH_BEGIN && begin_search<GM, G, false, FORCED>(p, io, h, tree, row0, lane, gm, s_ctr)) {
        n_pending = 1;   // (one evaluator row in use; not a leaf request)
        break;
      }
      if (h.phase != AZ_PH_RUN) break;
      if (h.sims_done + n_pending >= search_target(p, h)) {
        if (n_pending > 0 || advanced) break;
        finish_move<GM, G, FORCED>(p, h, tree, lane, gm, s_ctr);
        advanced = true;
        continue;
      }
      if (n_pending >= K) break;
      if (p.max_sims > 0 && sims_this_step >= p.max_sims + K) break;
      const Arena a = arena_of(p, tree, h.half);
      St s = root_state(h);
      int node, depth;
      bool dovf = false;
      sim_select<GM, G, false, FORCED>(p, a, h.root_node, s, node, depth, spath, lane, gm, c.children, dovf, false,
                                       FORCED ? forced_k(h) : 0.0);
      if (dovf) {
        h.err = 1;
        h.phase = AZ_PH_ERROR;
        if (lane == 0) ctr_add(s_ctr, AZ_CTR_OVERFLOW, 1);
        break;
      }
      const int out = depth > 0 ? GM::outcome(s, p.geo) : -1;
      ++sims_this_step;
      if (out >= 0) {   // terminal leaf: real backup at once, no virtual loss needed
        terminal_leaf<G>(a, h, spath, depth, out, s.ply, lane, gm, c);
        continue;
      }
      if (a.nl(node).y == VL_MARK) break;   // this leaf is already in flight: stop collecting for this step
      const int slot = n_pending++;
      if (lane == 0) {
        VlPend pe;
        pe.b0 = s.b0;
        pe.b1 = s.b1;
        pe.node = node;
        pe.depth = depth;
        pe.ply = s.ply;
        pe.valid = 1;
        pend[slot] = pe;
        a.nl(node).y = VL_MARK;
      }
      int32_t* gp = gpaths + (size_t)slot * GM::MAXD;
      for (int j = lane; j <= depth; j += G) gp[j] = spath[j];
      __syncwarp(gm);
      vl_apply<G>(a, spath, depth, lane);
      __syncwarp(gm);
      write_obs<GM, G>(p, io, row0 + slot, lane, s);
    }
    if (h.phase == AZ_PH_RUN && n_pending > 0) h.phase = AZ_PH_LEAF_EVAL;
    if (lane == 0) {
      p.hdr[tree] = h;
      ctr_add(s_ctr, AZ_CTR_IDLE_SLOTS, (unsigned long long)(K - n_pending));
      c.flush(s_ctr, h.alloc);
    }
  }
  flush_block_counters(p, s_ctr);
}

// ---------------------------------------------------------------- re-root compaction, one CTA per moving tree
// MCTS.update_root (mcts.py:192-203): BFS copy of the subtree of h.pend_node into the other arena half, for the trees queued
// by finish_move (they wait in PH_COMPACT and go on to their next search) and by k_command's update_root (they keep the phase
// k_command gave them).  The new arena is its own queue, 256 queue nodes per iteration: the copy is a chain of dependent
// global loads, so its duration is the number of iterations, not the number of nodes.
constexpr int COMPACT_BLOCK = 256;
__global__ void __launch_bounds__(COMPACT_BLOCK) k_compact(const Params p) {
  __shared__ int s_warp_sum[COMPACT_BLOCK / 32];
  __shared__ unsigned long long s_copied;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_copied = 0ULL;
  const int count = *p.compact_count;
  for (int i = blockIdx.x; i < count; i += gridDim.x) {
    const int tree = p.compact_list[i];
    TreeHdr h = p.hdr[tree];
    const Arena src = arena_of(p, tree, h.half);
    const Arena dst = arena_of(p, tree, h.half ^ 1);
    if (tid == 0) {
      dst.nl(0) = src.nl(h.pend_node);
      dst.q(0) = src.q(h.pend_node);
      dst.p(0) = src.p(h.pend_node);
    }
    __syncthreads();
    int head = 0, tail = 1;
    while (head < tail) {
      const int nb = min(COMPACT_BLOCK, tail - head);
      const int idx = head + tid;
      int mync = 0, oldfc = 0;
      if (tid < nb) {
        const uint2 nl = dst.nl(idx);
        mync = (int)(nl.y & 0xffu);
        oldfc = (int)(nl.y >> 8);
      }
      const int incl = gscan_incl<32>(0xffffffffu, mync, lane);
      if (lane == 31) s_warp_sum[warp] = incl;
      __syncthreads();
      int off = 0, total = 0;
#pragma unroll
      for (int w = 0; w < COMPACT_BLOCK / 32; ++w) {
        const int v = s_warp_sum[w];
        if (w < warp) off += v;
        total += v;
      }
      if (mync > 0) {
        const int newfc = tail + off + incl - mync;
        dst.nl(idx).y = ((unsigned)newfc << 8) | (unsigned)mync;
        for (int j = 0; j < mync; ++j) {
          dst.nl(newfc + j) = src.nl(oldfc + j);
          dst.q(newfc + j) = src.q(oldfc + j);
          dst.p(newfc + j) = src.p(oldfc + j);
        }
      }
      __syncthreads();
      tail += total;
      head += nb;
    }
    if (tid == 0) {
      h.half ^= 1;
      h.root_node = 0;
      h.alloc = tail;
      if (h.phase == PH_COMPACT) h.phase = PH_BEGIN;
      p.hdr[tree] = h;
      s_copied += (unsigned long long)tail;
    }
    __syncthreads();
  }
  __syncthreads();
  if (tid == 0) {
    if (s_copied) atomicAdd(&p.ctr[AZ_CTR_COMPACT_NODES], s_copied);
    __threadfence();
    const int done = atomicAdd(p.compact_count + 1, 1);
    if (done == (int)gridDim.x - 1) {  // last CTA: reset the work list for the next k_step
      p.compact_count[0] = 0;
      p.compact_count[1] = 0;
    }
  }
}

// ---------------------------------------------------------------- control kernels
template <class GM>
__global__ void k_reset(const Params p) {
  constexpr int G = GM::G;
  const int tree = (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) / G);
  const int lane = threadIdx.x % G;
  if (tree >= p.n_trees) return;
  const unsigned gm = group_mask<G>();
  TreeHdr h;
  memset(&h, 0, sizeof(h));
  set_root(h, start_position<GM>(p, tree, 0));
  h.game_seq = 0;
  h.half = 0;
  fresh_tree<G>(p, h, tree, lane, gm);
  h.phase = (p.flags & AZ_F_MANUAL) ? AZ_PH_IDLE : PH_BEGIN;
  if (lane == 0) p.hdr[tree] = h;
}

// set positions by replaying histories; tree nodes untouched
template <class GM>
__global__ void k_set_positions(const Params p, const int32_t* hist, const int32_t* len, int max_len, int32_t* bad) {
  const int tree = blockIdx.x * blockDim.x + threadIdx.x;
  if (tree >= p.n_trees) return;
  const int n = len[tree];
  if (n < 0) return;
  St s = GM::initial(p.geo);
  for (int j = 0; j < n; ++j) {
    const typename GM::Legal lg = GM::legal(s, p.geo);
    const int a = hist[(size_t)tree * max_len + j];
    if (GM::outcome(s, p.geo) >= 0 || GM::rank_of(lg, s, p.geo, a) < 0) {
      atomicAdd(bad, 1);
      return;
    }
    s = GM::apply(s, p.geo, a);
  }
  set_root(p.hdr[tree], s);
}

template <class GM>
__global__ void k_command(const Params p, const int32_t* upd, const int32_t* rst, const int32_t* beg, int32_t* bad) {
  constexpr int G = GM::G;
  const int tree = (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) / G);
  const int lane = threadIdx.x % G;
  if (tree < p.n_trees) {
    const unsigned gm = group_mask<G>();
    TreeHdr h = p.hdr[tree];
    bool dirty = false;
    if (rst && rst[tree]) {
      // 1: the root of MCTS.__init__ (mcts.py:122); 2: the root update_root builds for a leaf root (mcts.py:199-200)
      fresh_tree<G>(p, h, tree, lane, gm, rst[tree] == 2 && (p.flags & AZ_F_UCT) != 0);
      h.phase = AZ_PH_IDLE;
      dirty = true;
    }
    if (upd && upd[tree] >= 0) {
      const int action = upd[tree];
      const Arena a = arena_of(p, tree, h.half);
      const St s = root_state(h);
      const typename GM::Legal lg = GM::legal(s, p.geo);
      const int k = GM::outcome(s, p.geo) >= 0 ? -1 : GM::rank_of(lg, s, p.geo, action);
      const uint2 rnl = a.nl(h.root_node);
      if ((rnl.y & 0xffu) == 0) {
        // root is a leaf -> Node(None, 0.0, use_puct=self.use_puct)   mcts.py:198-200
        fresh_tree<G>(p, h, tree, lane, gm, (p.flags & AZ_F_UCT) != 0);
      } else if (k < 0) {
        if (lane == 0) atomicAdd(bad, 1);     // KeyError in the reference (mcts.py:202)
      } else {  // the chosen child becomes the root: k_compact, launched right after this kernel, copies its subtree
        h.pend_node = (int)(rnl.y >> 8) + k;
        if (lane == 0) p.compact_list[atomicAdd(p.compact_count, 1)] = tree;
      }
      if (k >= 0) set_root(h, GM::apply(s, p.geo, action));
      h.phase = AZ_PH_IDLE;
      dirty = true;
    }
    if (beg && beg[tree]) {
      if (beg[tree] == 2) {  // MCTS.playout (mcts.py:126-153): ONE simulation, no root Dirichlet expansion
        h.phase = AZ_PH_RUN;
        h.sims_done = p.n_playouts - 1;
        h.fast_sims = 0;
        set_forced_k(h, 0.0);
        h.pend_depth = 0;
      } else {
        h.phase = PH_BEGIN;
        h.sims_done = 0;
      }
      dirty = true;
    }
    if (dirty && lane == 0) p.hdr[tree] = h;
  }
}

template <class GM>
__global__ void k_status(const Params p, int32_t* phase, int32_t* sims, int32_t* ply, int32_t* req_legal) {
  const int tree = blockIdx.x * blockDim.x + threadIdx.x;
  if (tree >= p.n_trees) return;
  const TreeHdr h = p.hdr[tree];
  if (phase) phase[tree] = (h.phase == PH_BEGIN || h.phase == PH_COMPACT) ? AZ_PH_RUN : h.phase;
  if (sims) sims[tree] = h.sims_done;
  if (ply) ply[tree] = h.root_ply;
  if (req_legal) {
    int L = 0;
    if (h.phase == AZ_PH_LEAF_EVAL || h.phase == AZ_PH_ROOT_EVAL) {
      L = GM::count(GM::legal(pend_state(h), p.geo));
    }
    req_legal[tree] = L;
  }
}

template <class GM>
__global__ void k_request_info(const Params p, uint64_t* bb, int32_t* ply, int32_t* path_actions, int32_t* depth_out,
                               int max_depth) {
  const int tree = blockIdx.x * blockDim.x + threadIdx.x;
  if (tree >= p.n_trees) return;
  const TreeHdr h = p.hdr[tree];
  const bool pending = h.phase == AZ_PH_LEAF_EVAL || h.phase == AZ_PH_ROOT_EVAL;
  if (bb) {
    bb[2 * tree] = pending ? h.pend_b0 : 0;
    bb[2 * tree + 1] = pending ? h.pend_b1 : 0;
  }
  if (ply) ply[tree] = pending ? h.pend_ply : -1;
  const bool last_path = (p.flags & AZ_F_MANUAL) && h.phase == AZ_PH_SEARCH_DONE;   // path of the last simulation
  const int depth = (h.phase == AZ_PH_LEAF_EVAL || last_path) ? h.pend_depth : (pending ? 0 : -1);
  if (depth_out) depth_out[tree] = depth;
  if (path_actions && depth > 0) {
    const Arena a = arena_of(p, tree, h.half);
    const int32_t* gpath = p.path + (size_t)tree * GM::MAXD;
    St s = root_state(h);
    for (int j = 0; j < depth && j < max_depth; ++j) {
      const int fc = (int)(a.nl(gpath[j]).y >> 8);
      const int k = gpath[j + 1] - fc;
      const typename GM::Legal lg = GM::legal(s, p.geo);
      const int act = GM::action_of(lg, s, p.geo, k);
      path_actions[(size_t)tree * max_depth + j] = act;
      s = GM::apply(s, p.geo, act);
    }
  }
}

template <class GM>
__global__ void k_root_stats(const Params p, int32_t* root_n, double* root_q, int32_t* n_children, int32_t* child_action,
                             int32_t* child_n, double* child_q, double* child_p, double* v_a0c, double* v_off) {
  constexpr int G = GM::G;
  const int tree = (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) / G);
  const int lane = threadIdx.x % G;
  if (tree >= p.n_trees) return;
  const unsigned gm = group_mask<G>();
  const TreeHdr h = p.hdr[tree];
  const Arena a = arena_of(p, tree, h.half);
  const uint2 rnl = a.nl(h.root_node);
  const int nc = (int)(rnl.y & 0xffu), fc = (int)(rnl.y >> 8);
  const St s = root_state(h);
  const typename GM::Legal lg = GM::legal(s, p.geo);
  if (lane == 0) {
    if (root_n) root_n[tree] = (int)rnl.x;
    if (root_q) root_q[tree] = a.q(h.root_node);
    if (n_children) n_children[tree] = nc;
  }
  double a0c = -99.0;
  int a0c_i = 0x7fffffff;
#pragma unroll
  for (int sl = 0; sl < GM::SLOTS; ++sl) {
    const int i = lane + sl * G;
    if (i < GM::MAXC) {
      const size_t o = (size_t)tree * GM::MAXC + i;
      const bool have = i < nc;
      const uint2 nl = have ? a.nl(fc + i) : make_uint2(0u, 0u);
      const double q = have ? a.q(fc + i) : 0.0;
      if (child_action) child_action[o] = have ? GM::action_of(lg, s, p.geo, i) : -1;
      if (child_n) child_n[o] = have ? (int)nl.x : 0;
      if (child_q) child_q[o] = q;
      if (child_p) child_p[o] = have ? a.p(fc + i) : 0.0;
      if (have) {
        const double v = nl.x > 0 ? q : -99.0;
        if (a0c_i == 0x7fffffff || v > a0c) { a0c = v; a0c_i = i; }
      }
    }
  }
  gargmax<G>(gm, a0c, a0c_i);
  if (v_a0c && lane == 0) v_a0c[tree] = a0c;
  if (v_off) {
    const double v = offpolicy_value<GM, G>(a, h.root_node, lane, gm);
    if (lane == 0) v_off[tree] = v;
  }
}

template <class GM>
__global__ void k_positions(const Params p, uint64_t* bb, int32_t* ply, int32_t* terminal, double* ret0) {
  const int tree = blockIdx.x * blockDim.x + threadIdx.x;
  if (tree >= p.n_trees) return;
  const TreeHdr h = p.hdr[tree];
  const St s = root_state(h);
  const int out = GM::outcome(s, p.geo);
  if (bb) {
    bb[2 * tree] = s.b0;
    bb[2 * tree + 1] = s.b1;
  }
  if (ply) ply[tree] = s.ply;
  if (terminal) terminal[tree] = out >= 0;
  if (ret0) ret0[tree] = out == 0 ? 1.0 : (out == 1 ? -1.0 : 0.0);
}

// ---------------------------------------------------------------- stateless game kernels (parity tests)
template <class GM>
__global__ void k_game_replay(const Geo geo, int n, const int32_t* hist, const int32_t* len, int max_len, uint64_t* bb,
                              int32_t* status, double* ret0, int32_t* n_legal, int32_t* legal, void* obs,
                              int obs_format) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  St s = GM::initial(geo);
  int st = 0;
  for (int j = 0; j < len[i]; ++j) {
    const typename GM::Legal lg = GM::legal(s, geo);
    const int a = hist[(size_t)i * max_len + j];
    if (GM::outcome(s, geo) >= 0 || GM::rank_of(lg, s, geo, a) < 0) {
      st |= 2;
      break;
    }
    s = GM::apply(s, geo, a);
  }
  const int out = GM::outcome(s, geo);
  if (out >= 0) st |= 1;
  if (bb) {
    bb[2 * i] = s.b0;
    bb[2 * i + 1] = s.b1;
  }
  if (status) status[i] = st;
  if (ret0) ret0[i] = out == 0 ? 1.0 : (out == 1 ? -1.0 : 0.0);
  const typename GM::Legal lg = GM::legal(s, geo);
  const int L = out >= 0 ? 0 : GM::count(lg);
  if (n_legal) n_legal[i] = L;
  if (legal)
    for (int k = 0; k < GM::MAXC; ++k) legal[(size_t)i * GM::MAXC + k] = k < L ? GM::action_of(lg, s, geo, k) : -1;
  if (obs && obs_format != AZ_OBS_NONE) {
    Params p;
    p.geo = geo;
    StepIO io;
    io.obs = obs;
    io.obs_format = obs_format;
    write_obs<GM, 1>(p, io, i, 0, s);
  }
}

// state_to_board (network.py:9-18) for a gathered minibatch: example idx[i] (or i) of a replay buffer held as canonical
// bitboards + ply -> observation planes in obs_format.  The trainer's minibatch builder (train.py:108-112 builds the same
// planes from Python lists of numpy boards).
template <class GM>
__global__ void k_observations(const Geo geo, int n, const uint64_t* bb, const int32_t* ply, const int64_t* idx, void* obs,
                               int obs_format) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const long long src = idx ? idx[i] : (long long)i;
  St s;
  s.b0 = bb[2 * src];
  s.b1 = bb[2 * src + 1];
  s.ply = ply[src];
  Params p;
  p.geo = geo;
  StepIO io;
  io.obs = obs;
  io.obs_format = obs_format;
  write_obs<GM, 1>(p, io, i, 0, s);
}

template <class GM>
__global__ void k_game_random_playouts(const Geo geo, int n, uint64_t seed, int max_plies, int32_t* hist, int32_t* len) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  St s = GM::initial(geo);
  int j = 0;
  for (; j < max_plies; ++j) {
    if (GM::outcome(s, geo) >= 0) break;
    const typename GM::Legal lg = GM::legal(s, geo);
    const int L = GM::count(lg);
    const int a = GM::action_of(lg, s, geo, (int)(counter(seed, i, 0, j, 0, 3) % (uint64_t)L));
    hist[(size_t)i * max_plies + j] = a;
    s = GM::apply(s, geo, a);
  }
  len[i] = j;
}

}  // namespace az

// =====================================================================================================
// Host side: the C-ABI
// =====================================================================================================
using namespace az;

static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define CK(call)                                                                              \
  do {                                                                                        \
    cudaError_t _e = (call);                                                                  \
    if (_e != cudaSuccess) return fail(-2, "%s failed: %s", #call, cudaGetErrorString(_e));   \
  } while (0)

struct az_engine {
  az_config cfg;
  Params p;
  int max_children, maxd, group;
  int64_t bytes;
  int32_t* d_cmd;  // 3 * n_trees command staging + 1 error word
  int32_t* d_bad;
};

static Geo make_geo(int game_id, int rows, int cols) {
  Geo g;
  memset(&g, 0, sizeof(g));
  if (game_id == AZ_GAME_CONNECT_FOUR) {
    rows = 6;
    cols = 7;
  }
  g.rows = rows;
  g.cols = cols;
  g.cells = rows * cols;
  g.n_actions = game_id == AZ_GAME_CONNECT_FOUR ? 7 : rows * cols * 12;
  g.all = g.cells >= 64 ? ~0ULL : ((1ULL << g.cells) - 1ULL);
  uint64_t c0 = 0, cl = 0;
  for (int r = 0; r < rows; ++r) {
    c0 |= 1ULL << (r * cols);
    cl |= 1ULL << (r * cols + cols - 1);
  }
  g.notcol0 = g.all & ~c0;
  g.notcolL = g.all & ~cl;
  g.row0 = cols >= 64 ? ~0ULL : ((1ULL << cols) - 1ULL);
  g.rowL = g.row0 << ((rows - 1) * cols);
  return g;
}

static int check_game(int game_id, int rows, int cols) {
  if (game_id == AZ_GAME_CONNECT_FOUR) return 0;
  if (game_id != AZ_GAME_BREAKTHROUGH) return fail(-1, "unknown game_id %d", game_id);
  if (rows < 4 || cols < 2 || rows * cols > 64 || cols > 16)
    return fail(-1, "breakthrough %dx%d unsupported (need rows>=4, cols>=2, rows*cols<=64)", rows, cols);
  return 0;
}

template <class F>
static int dispatch_game(int game_id, F&& f) {
  if (game_id == AZ_GAME_CONNECT_FOUR) return f(C4());
  return f(BT());
}

static inline int compact_grid(int n_trees) {  // one CTA per moving tree; ~n_trees * e / n_playouts trees move per step
  int grid = n_trees / 128 + 4;
  return grid > 296 ? 296 : grid;
}
static inline int groups_grid(int n_trees, int G, int block) { return (int)(((long long)n_trees * G + block - 1) / block); }

extern "C" {

const char* az_last_error(void) { return g_err; }
int az_version(void) { return 1; }

int az_create(const az_config* cfg_in, az_engine** out) {
  if (!cfg_in || !out) return fail(-1, "null argument");
  az_config cfg = *cfg_in;
  if (check_game(cfg.game_id, cfg.rows, cfg.cols)) return -1;
  if (cfg.game_id == AZ_GAME_CONNECT_FOUR) {
    cfg.rows = 6;
    cfg.cols = 7;
  }
  if (cfg.n_trees <= 0) return fail(-1, "n_trees must be positive");
  if (cfg.n_playouts <= 0) return fail(-1, "n_playouts must be positive");
  if (cfg.temperature <= 0.0) cfg.temperature = 1.0;
  if (cfg.dirichlet_alpha <= 0.0) cfg.dirichlet_alpha = 0.3;
  if (cfg.noise_weight == 0.0) cfg.noise_weight = 0.25;
  if (cfg.num_probabilistic_actions <= 0) cfg.num_probabilistic_actions = 1000;
  if (cfg.noise_mode < 0 || cfg.noise_mode > 3) return fail(-1, "bad noise_mode");
  if (cfg.eval_mode < 0 || cfg.eval_mode > 3) return fail(-1, "bad eval_mode");
  const int maxc = cfg.game_id == AZ_GAME_CONNECT_FOUR ? C4::MAXC : BT::MAXC;
  const int maxd = cfg.game_id == AZ_GAME_CONNECT_FOUR ? C4::MAXD : BT::MAXD;
  const int group = cfg.game_id == AZ_GAME_CONNECT_FOUR ? C4::G : BT::G;
  if (cfg.node_capacity <= 0) {
    // Every playout expands at most one leaf (<= branch children) and a re-rooted tree keeps at most what it had, so the
    // worst case grows by (n_playouts+1)*branch per ply.  Measured high-water marks (AZ_CTR_PEAK_NODES, 25k-step soaks):
    // Connect Four @800: 26.7k nodes = 4.7 searches' worth -> default 8 searches' worth.  Overflow is counted and raised.
    const int branch = cfg.game_id == AZ_GAME_CONNECT_FOUR ? 7 : 3 * cfg.cols + 8;
    long long c = (long long)(cfg.n_playouts + 2) * branch * 8 + 64;
    if (c > (1 << 24) - 1) c = (1 << 24) - 1;
    cfg.node_capacity = (int)c;
  }
  if (cfg.node_capacity >= (1 << 24)) return fail(-1, "node_capacity must be < 2^24");
  if (cfg.leaves_per_tree <= 0 || !(cfg.flags & AZ_F_VIRTUAL_LOSS)) cfg.leaves_per_tree = 1;
  if (cfg.leaves_per_tree > 64) return fail(-1, "leaves_per_tree must be <= 64");
  if ((cfg.flags & AZ_F_VIRTUAL_LOSS) && (cfg.flags & (AZ_F_MANUAL | AZ_F_UCT)))
    return fail(-1, "AZ_F_VIRTUAL_LOSS is a batched self-play mode (no AZ_F_MANUAL / AZ_F_UCT)");
  if ((cfg.flags & AZ_F_RESIGN) && (cfg.flags & AZ_F_MANUAL))
    return fail(-1, "AZ_F_RESIGN is a batched self-play mode: with AZ_F_MANUAL the host decides the moves");
  if ((cfg.flags & AZ_F_PLAYOUT_CAP) && (cfg.flags & AZ_F_MANUAL))
    return fail(-1, "AZ_F_PLAYOUT_CAP is a batched self-play mode: with AZ_F_MANUAL the host starts the searches");
  if ((cfg.flags & AZ_F_FORCED_PLAYOUTS) && (cfg.flags & AZ_F_MANUAL))
    return fail(-1, "AZ_F_FORCED_PLAYOUTS is a batched self-play mode: with AZ_F_MANUAL the host decides the moves");
  if ((cfg.flags & AZ_F_FORCED_PLAYOUTS) && (cfg.flags & AZ_F_UCT))
    return fail(-1, "AZ_F_FORCED_PLAYOUTS is a PUCT rule: AZ_F_UCT scores with the use_puct=False formula");
  if ((cfg.flags & AZ_F_FORCED_PLAYOUTS) && cfg.noise_mode == AZ_NOISE_NONE)
    return fail(-1, "AZ_F_FORCED_PLAYOUTS forces only searches with root noise: AZ_NOISE_NONE has none");
  if (cfg.record_capacity <= 0) cfg.record_capacity = cfg.n_trees * 64 < (1 << 20) ? (1 << 20) : cfg.n_trees * 64;
  if (!(cfg.flags & AZ_F_RECORDS)) cfg.record_capacity = 1;
  if (cfg.flags & AZ_F_EVAL_CACHE) {
    if (cfg.eval_mode != AZ_EVAL_EXTERNAL || (cfg.flags & (AZ_F_PRIORS_F64 | AZ_F_MANUAL | AZ_F_VIRTUAL_LOSS)) ||
        cfg.noise_mode == AZ_NOISE_HOST)
      return fail(-1, "AZ_F_EVAL_CACHE needs AZ_EVAL_EXTERNAL float outputs, no AZ_F_MANUAL / AZ_F_VIRTUAL_LOSS / "
                      "AZ_NOISE_HOST");
    int lg = (int)AZ_EVAL_CACHE_LOG2(cfg.flags);
    if (lg == 0) {
      lg = AZ_EVAL_CACHE_EXTRA_LOG2;
      while ((1LL << lg) < (long long)cfg.n_trees * cfg.n_playouts << AZ_EVAL_CACHE_EXTRA_LOG2) ++lg;
      lg = lg < 16 ? 16 : (lg > 27 ? 27 : lg);
    }
    if (lg > 30) return fail(-1, "evaluator cache size 2^%d: at most 2^30 entries", lg);
    cfg.flags = (cfg.flags & ~(31u << AZ_EVAL_CACHE_LOG2_SHIFT)) | ((uint32_t)lg << AZ_EVAL_CACHE_LOG2_SHIFT);
  } else {
    cfg.flags &= ~(31u << AZ_EVAL_CACHE_LOG2_SHIFT);
  }

  CK(cudaSetDevice(cfg.device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, cfg.device));
  if (prop.major < 10) return fail(-3, "az_b200 needs an sm_100a GPU (found sm_%d%d)", prop.major, prop.minor);

  az_engine* e = new (std::nothrow) az_engine();
  if (!e) return fail(-4, "out of host memory");
  memset(e, 0, sizeof(*e));
  e->cfg = cfg;
  e->max_children = maxc;
  e->maxd = maxd;
  e->group = group;
  Params& p = e->p;
  p.n_trees = cfg.n_trees;
  p.cap = cfg.node_capacity;
  p.n_playouts = cfg.n_playouts;
  p.num_prob = cfg.num_probabilistic_actions;
  p.noise_mode = cfg.noise_mode;
  p.eval_mode = cfg.eval_mode;
  p.eval_shift = cfg.eval_shift;
  p.max_sims = cfg.max_sims_per_step;
  p.cycle_budget = cfg.step_cycle_budget > 0 ? cfg.step_cycle_budget : 0;
  p.start_mod = cfg.start_plies_mod;
  p.flags = cfg.flags;
  p.seed = cfg.seed;
  p.c_puct = cfg.c_puct;
  p.keep = 1.0 - cfg.dirichlet_ratio;
  p.noise_w = cfg.noise_weight;
  p.alpha = cfg.dirichlet_alpha;
  p.temperature = cfg.temperature;
  p.geo = make_geo(cfg.game_id, cfg.rows, cfg.cols);
  p.rec_stride = (int)((sizeof(az_record) + 6 * (size_t)maxc + 7) / 8 * 8);
  p.max_games = cfg.max_games;
  p.rec_cap = cfg.record_capacity;
  p.vl_k = cfg.leaves_per_tree;

  const size_t nodes = (size_t)cfg.n_trees * 2 * (size_t)cfg.node_capacity;
  size_t bytes = 0;
  auto alloc = [&](void** ptr, size_t n) -> cudaError_t {
    bytes += n;
    return cudaMalloc(ptr, n);
  };
  cudaError_t err = cudaSuccess;
  if ((err = alloc((void**)&p.hdr, sizeof(TreeHdr) * (size_t)cfg.n_trees)) != cudaSuccess ||
      (err = alloc((void**)&p.nodes, sizeof(Node) * nodes)) != cudaSuccess ||
      (err = alloc((void**)&p.path, sizeof(int32_t) * (size_t)cfg.n_trees * maxd * (size_t)cfg.leaves_per_tree)) != cudaSuccess ||
      (err = alloc((void**)&p.vl_pend, sizeof(VlPend) * (size_t)cfg.n_trees * (size_t)cfg.leaves_per_tree)) != cudaSuccess ||
      (err = alloc((void**)&p.rec, (size_t)p.rec_stride * (size_t)p.rec_cap)) != cudaSuccess ||
      (err = alloc((void**)&p.rec_count, sizeof(unsigned long long))) != cudaSuccess ||
      (err = alloc((void**)&p.ctr, sizeof(unsigned long long) * AZ_CTR_COUNT)) != cudaSuccess ||
      (err = alloc((void**)&p.games_started, sizeof(int))) != cudaSuccess ||
      (err = alloc((void**)&p.compact_list, sizeof(int) * (size_t)cfg.n_trees)) != cudaSuccess ||
      (err = alloc((void**)&p.compact_count, sizeof(int) * 2)) != cudaSuccess ||
      (err = alloc((void**)&e->d_cmd, sizeof(int32_t) * ((size_t)cfg.n_trees * 3))) != cudaSuccess ||
      (err = alloc((void**)&e->d_bad, sizeof(int32_t))) != cudaSuccess) {
    fail(-2, "cudaMalloc failed (%zu bytes requested so far): %s", bytes, cudaGetErrorString(err));
    az_destroy(e);
    return -2;
  }
  if (cfg.flags & AZ_F_EVAL_CACHE) {
    const size_t n = (size_t)1 << AZ_EVAL_CACHE_LOG2(cfg.flags);
    const size_t cbytes = n * (cfg.game_id == AZ_GAME_CONNECT_FOUR ? cache_stride<C4>() : cache_stride<BT>());
    if ((err = alloc((void**)&p.cache, cbytes)) != cudaSuccess ||
        (err = alloc((void**)&p.cache_epoch, 2 * sizeof(uint32_t))) != cudaSuccess) {
      fail(-2, "cudaMalloc failed (evaluator cache, %zu bytes): %s", cbytes, cudaGetErrorString(err));
      az_destroy(e);
      return -2;
    }
    p.cache_mask = n - 1;
    const uint32_t epoch0[2] = {1u, 1u};  // a zeroed entry (tag 0) never matches
    CK(cudaMemset(p.cache, 0, cbytes));
    CK(cudaMemcpy(p.cache_epoch, epoch0, sizeof(epoch0), cudaMemcpyHostToDevice));
  }
  if (cfg.flags & AZ_F_RESIGN) {
    if ((err = alloc((void**)&p.resign_cfg, sizeof(ResignCfg))) != cudaSuccess ||
        (err = alloc((void**)&p.resign_tree, sizeof(ResignTree) * (size_t)cfg.n_trees)) != cudaSuccess) {
      fail(-2, "cudaMalloc failed (resignation state): %s", cudaGetErrorString(err));
      az_destroy(e);
      return -2;
    }
    const ResignCfg rc0 = {-1.0, 0, 0};  // never resigns
    CK(cudaMemcpy(p.resign_cfg, &rc0, sizeof(rc0), cudaMemcpyHostToDevice));
  }
  if (cfg.flags & AZ_F_PLAYOUT_CAP) {
    if ((err = alloc((void**)&p.pcap_cfg, sizeof(PlayoutCapCfg))) != cudaSuccess) {
      fail(-2, "cudaMalloc failed (playout cap): %s", cudaGetErrorString(err));
      az_destroy(e);
      return -2;
    }
    const PlayoutCapCfg pc0 = {cfg.n_playouts, 1000};  // every search is full
    CK(cudaMemcpy(p.pcap_cfg, &pc0, sizeof(pc0), cudaMemcpyHostToDevice));
  }
  if (cfg.flags & AZ_F_FORCED_PLAYOUTS) {
    if ((err = alloc((void**)&p.forced_cfg, sizeof(double))) != cudaSuccess) {
      fail(-2, "cudaMalloc failed (forced playouts): %s", cudaGetErrorString(err));
      az_destroy(e);
      return -2;
    }
    const double k0 = 0.0;  // no search is forced
    CK(cudaMemcpy(p.forced_cfg, &k0, sizeof(k0), cudaMemcpyHostToDevice));
  }
  if (cfg.flags & AZ_F_UCT) {
    double* tab = nullptr;
    if ((err = alloc((void**)&tab, sizeof(double) * LOGTAB_N)) != cudaSuccess) {
      fail(-2, "cudaMalloc failed (log table): %s", cudaGetErrorString(err));
      az_destroy(e);
      return -2;
    }
    p.logtab = tab;
    std::vector<double> host(LOGTAB_N);
    for (int n = 0; n < LOGTAB_N; ++n) host[n] = log((double)n);  // log(0) = -inf is never used (a visited child has a visited parent)
    CK(cudaMemcpy(tab, host.data(), sizeof(double) * LOGTAB_N, cudaMemcpyHostToDevice));
  }
  e->bytes = (int64_t)bytes;
  CK(cudaMemset(p.rec_count, 0, sizeof(unsigned long long)));
  CK(cudaMemset(p.ctr, 0, sizeof(unsigned long long) * AZ_CTR_COUNT));
  CK(cudaMemset(e->d_bad, 0, sizeof(int32_t)));
  CK(cudaMemset(p.compact_count, 0, sizeof(int) * 2));
  CK(cudaMemset(p.vl_pend, 0, sizeof(VlPend) * (size_t)cfg.n_trees * (size_t)cfg.leaves_per_tree));
  *out = e;
  int rc = az_reset(e, nullptr);
  if (rc) return rc;
  CK(cudaDeviceSynchronize());
  return 0;
}

int az_destroy(az_engine* e) {
  if (!e) return 0;
  Params& p = e->p;
  cudaFree(p.hdr);
  cudaFree(p.nodes);
  cudaFree(p.path);
  cudaFree(p.vl_pend);
  cudaFree(p.rec);
  cudaFree(p.rec_count);
  cudaFree(p.ctr);
  cudaFree(p.games_started);
  cudaFree(p.compact_list);
  cudaFree(p.compact_count);
  if (p.dbg) cudaFree(p.dbg);
  if (p.logtab) cudaFree(const_cast<double*>(p.logtab));
  if (p.cache) cudaFree(p.cache);
  if (p.cache_epoch) cudaFree(p.cache_epoch);
  if (p.resign_cfg) cudaFree(p.resign_cfg);
  if (p.resign_tree) cudaFree(p.resign_tree);
  if (p.pcap_cfg) cudaFree(p.pcap_cfg);
  if (p.forced_cfg) cudaFree(p.forced_cfg);
  cudaFree(e->d_cmd);
  cudaFree(e->d_bad);
  delete e;
  return 0;
}

int az_config_get(const az_engine* e, az_config* out) {
  if (!e || !out) return fail(-1, "null argument");
  *out = e->cfg;
  return 0;
}
int az_max_children(const az_engine* e) { return e ? e->max_children : -1; }
int az_num_actions(const az_engine* e) { return e ? e->p.geo.n_actions : -1; }
int az_record_stride(const az_engine* e) { return e ? e->p.rec_stride : -1; }
int64_t az_device_bytes(const az_engine* e) { return e ? e->bytes : -1; }

int az_reset(az_engine* e, void* stream) {
  if (!e) return fail(-1, "null engine");
  cudaStream_t st = (cudaStream_t)stream;
  const Params p = e->p;
  CK(cudaMemcpyAsync(p.games_started, &e->cfg.n_trees, sizeof(int), cudaMemcpyHostToDevice, st));
  CK(cudaMemsetAsync(p.compact_count, 0, sizeof(int) * 2, st));
  // game_seq -1: every tree's entry is started afresh at its first searched position
  if (p.resign_tree) CK(cudaMemsetAsync(p.resign_tree, 0xff, sizeof(ResignTree) * (size_t)p.n_trees, st));
  dispatch_game(e->cfg.game_id, [&](auto gm) {
    using GM = decltype(gm);
    k_reset<GM><<<groups_grid(p.n_trees, GM::G, BLOCK), BLOCK, 0, st>>>(p);
    return 0;
  });
  CK(cudaGetLastError());
  return 0;
}

static int check_bad(az_engine* e, cudaStream_t st, const char* what) {
  int32_t bad = 0;
  CK(cudaMemcpyAsync(&bad, e->d_bad, sizeof(bad), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if (bad) {
    cudaMemsetAsync(e->d_bad, 0, sizeof(int32_t), st);
    return fail(-5, "%s: %d tree(s) got an illegal action", what, bad);
  }
  return 0;
}

int az_set_positions(az_engine* e, const int32_t* hist_host, const int32_t* len_host, int32_t max_len, void* stream) {
  if (!e || !len_host) return fail(-1, "null argument");
  cudaStream_t st = (cudaStream_t)stream;
  const Params p = e->p;
  const size_t hn = (size_t)p.n_trees * (size_t)(max_len > 0 ? max_len : 1);
  // one temporary holding lengths + histories; released on every path out of this function
  int32_t* d_tmp = nullptr;
  CK(cudaMalloc((void**)&d_tmp, sizeof(int32_t) * (hn + (size_t)p.n_trees)));
  int32_t *d_len = d_tmp, *d_hist = d_tmp + p.n_trees;
  struct Free {
    int32_t* ptr;
    ~Free() { cudaFree(ptr); }
  } guard{d_tmp};
  if (max_len > 0 && hist_host) CK(cudaMemcpyAsync(d_hist, hist_host, sizeof(int32_t) * hn, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d_len, len_host, sizeof(int32_t) * (size_t)p.n_trees, cudaMemcpyHostToDevice, st));
  dispatch_game(e->cfg.game_id, [&](auto gm) {
    using GM = decltype(gm);
    k_set_positions<GM><<<(p.n_trees + 127) / 128, 128, 0, st>>>(p, d_hist, d_len, max_len > 0 ? max_len : 1, e->d_bad);
    return 0;
  });
  CK(cudaGetLastError());
  return check_bad(e, st, "az_set_positions");   // synchronises the stream: the temporary is idle when the guard frees it
}

int az_command(az_engine* e, const int32_t* update_root_host, const int32_t* reset_tree_host, const int32_t* begin_host,
               void* stream) {
  if (!e) return fail(-1, "null engine");
  cudaStream_t st = (cudaStream_t)stream;
  const Params p = e->p;
  const size_t n = (size_t)p.n_trees;
  int32_t* d_upd = update_root_host ? e->d_cmd : nullptr;
  int32_t* d_rst = reset_tree_host ? e->d_cmd + n : nullptr;
  int32_t* d_beg = begin_host ? e->d_cmd + 2 * n : nullptr;
  if (d_upd) CK(cudaMemcpyAsync(d_upd, update_root_host, sizeof(int32_t) * n, cudaMemcpyHostToDevice, st));
  if (d_rst) CK(cudaMemcpyAsync(d_rst, reset_tree_host, sizeof(int32_t) * n, cudaMemcpyHostToDevice, st));
  if (d_beg) CK(cudaMemcpyAsync(d_beg, begin_host, sizeof(int32_t) * n, cudaMemcpyHostToDevice, st));
  dispatch_game(e->cfg.game_id, [&](auto gm) {
    using GM = decltype(gm);
    k_command<GM><<<groups_grid(p.n_trees, GM::G, BLOCK), BLOCK, 0, st>>>(p, d_upd, d_rst, d_beg, e->d_bad);
    return 0;
  });
  if (d_upd) k_compact<<<compact_grid(p.n_trees), 256, 0, st>>>(p);  // re-root the trees k_command queued
  CK(cudaGetLastError());
  return check_bad(e, st, "az_command(update_root)");
}

int az_step(az_engine* e, const void* priors_dev, const void* values_dev, const double* noise_dev, void* obs_dev,
            int32_t obs_format, void* stream) {
  if (!e) return fail(-1, "null engine");
  if (obs_format < 0 || obs_format > 2) return fail(-1, "bad obs_format");
  cudaStream_t st = (cudaStream_t)stream;
  const Params p = e->p;
  StepIO io;
  io.priors = priors_dev;
  io.values = values_dev;
  io.noise = noise_dev;
  io.obs = obs_dev;
  io.obs_format = obs_format;
  if (p.noise_mode == AZ_NOISE_HOST && !noise_dev) return fail(-1, "AZ_NOISE_HOST needs noise_dev");
  if ((p.flags & AZ_F_KEEP_TREE) && !(p.flags & AZ_F_MANUAL) && !(p.flags & AZ_F_ASYNC_COMPACT)) {
    k_compact<<<compact_grid(p.n_trees), 256, 0, st>>>(p);  // re-root the trees that moved in the previous step
    CK(cudaGetLastError());
  }
  dispatch_game(e->cfg.game_id, [&](auto gm) {
    using GM = decltype(gm);
    // k_step stays the last launch of az_step: the evaluator's first kernel waits on it with griddepcontrol.wait
    if (p.cache && priors_dev) k_cache_insert<GM><<<groups_grid(p.n_trees, GM::G, BLOCK), BLOCK, 0, st>>>(p, io);
    const dim3 grid = groups_grid(p.n_trees, GM::G, BLOCK);
    const bool forced = (p.flags & AZ_F_FORCED_PLAYOUTS) != 0;
    if (p.flags & AZ_F_VIRTUAL_LOSS) {
      if (forced) k_step_vl<GM, true><<<grid, BLOCK, 0, st>>>(p, io);
      else k_step_vl<GM><<<grid, BLOCK, 0, st>>>(p, io);
    } else if (p.flags & AZ_F_UCT) {
      k_step<GM, true><<<grid, BLOCK, 0, st>>>(p, io);
    } else if (forced) {
      k_step<GM, false, true><<<grid, BLOCK, 0, st>>>(p, io);
    } else {
      k_step<GM, false><<<grid, BLOCK, 0, st>>>(p, io);
    }
    return 0;
  });
  CK(cudaGetLastError());
  return 0;
}

int az_eval_cache_invalidate(az_engine* e, void* stream) {
  if (!e) return fail(-1, "null engine");
  if (!e->p.cache) return 0;
  k_cache_new_epoch<<<1, 1, 0, (cudaStream_t)stream>>>(e->p.cache_epoch);
  CK(cudaGetLastError());
  return 0;
}

int az_set_resign(az_engine* e, double threshold, int32_t disabled_permille, void* stream) {
  if (!e) return fail(-1, "null engine");
  if (!e->p.resign_cfg) return fail(-1, "az_set_resign: the engine was created without AZ_F_RESIGN");
  if (!isfinite(threshold)) return fail(-1, "az_set_resign: the threshold must be finite");
  if (disabled_permille < 0 || disabled_permille > 1000)
    return fail(-1, "az_set_resign: disabled_permille %d is outside [0, 1000]", disabled_permille);
  const ResignCfg rc = {threshold, disabled_permille, 0};
  // pageable source: the copy has been staged when the call returns
  CK(cudaMemcpyAsync(e->p.resign_cfg, &rc, sizeof(rc), cudaMemcpyHostToDevice, (cudaStream_t)stream));
  return 0;
}

int az_set_playout_cap(az_engine* e, int32_t fast_playouts, int32_t full_permille, void* stream) {
  if (!e) return fail(-1, "null engine");
  if (!e->p.pcap_cfg) return fail(-1, "az_set_playout_cap: the engine was created without AZ_F_PLAYOUT_CAP");
  if (fast_playouts < 1 || fast_playouts > e->p.n_playouts)
    return fail(-1, "az_set_playout_cap: fast_playouts %d is outside [1, n_playouts = %d]", fast_playouts, e->p.n_playouts);
  if (full_permille < 0 || full_permille > 1000)
    return fail(-1, "az_set_playout_cap: full_permille %d is outside [0, 1000]", full_permille);
  const PlayoutCapCfg pc = {fast_playouts, full_permille};
  // pageable source: the copy has been staged when the call returns
  CK(cudaMemcpyAsync(e->p.pcap_cfg, &pc, sizeof(pc), cudaMemcpyHostToDevice, (cudaStream_t)stream));
  return 0;
}

int az_set_forced_playouts(az_engine* e, double k, void* stream) {
  if (!e) return fail(-1, "null engine");
  if (!e->p.forced_cfg) return fail(-1, "az_set_forced_playouts: the engine was created without AZ_F_FORCED_PLAYOUTS");
  if (!isfinite(k) || k < 0.0) return fail(-1, "az_set_forced_playouts: k must be finite and >= 0 (got %g)", k);
  // pageable source: the copy has been staged when the call returns
  CK(cudaMemcpyAsync(e->p.forced_cfg, &k, sizeof(k), cudaMemcpyHostToDevice, (cudaStream_t)stream));
  return 0;
}

int az_compact(az_engine* e, void* stream) {
  if (!e) return fail(-1, "null engine");
  const Params p = e->p;
  k_compact<<<compact_grid(p.n_trees), 256, 0, (cudaStream_t)stream>>>(p);
  CK(cudaGetLastError());
  return 0;
}

int az_debug_timing(az_engine* e, long long* out_host) {
  /* Development aid: per-tree SM cycle counts of the LAST k_step ([n_trees][4]: total cycles, phase on entry, simulations
   * run, 2*consume_cycles + moved).  The first call only arms the instrumentation. */
  if (!e || !out_host) return fail(-1, "null argument");
  const size_t bytes = sizeof(long long) * 4 * (size_t)e->p.n_trees;
  if (!e->p.dbg) {
    CK(cudaMalloc((void**)&e->p.dbg, bytes));
    CK(cudaMemset(e->p.dbg, 0, bytes));
  }
  CK(cudaMemcpy(out_host, e->p.dbg, bytes, cudaMemcpyDeviceToHost));
  return 0;
}

int az_status(az_engine* e, int32_t* phase_dev, int32_t* sims_dev, int32_t* ply_dev, int32_t* req_legal_dev, void* stream) {
  if (!e) return fail(-1, "null engine");
  const Params p = e->p;
  dispatch_game(e->cfg.game_id, [&](auto gm) {
    using GM = decltype(gm);
    k_status<GM><<<(p.n_trees + 127) / 128, 128, 0, (cudaStream_t)stream>>>(p, phase_dev, sims_dev, ply_dev, req_legal_dev);
    return 0;
  });
  CK(cudaGetLastError());
  return 0;
}

int az_request_info(az_engine* e, uint64_t* bb_dev, int32_t* ply_dev, int32_t* path_actions_dev, int32_t* depth_dev,
                    int32_t max_depth, void* stream) {
  if (!e) return fail(-1, "null engine");
  const Params p = e->p;
  dispatch_game(e->cfg.game_id, [&](auto gm) {
    using GM = decltype(gm);
    k_request_info<GM><<<(p.n_trees + 127) / 128, 128, 0, (cudaStream_t)stream>>>(p, bb_dev, ply_dev, path_actions_dev,
                                                                                 depth_dev, max_depth);
    return 0;
  });
  CK(cudaGetLastError());
  return 0;
}

int az_root_stats(az_engine* e, int32_t* root_n_dev, double* root_q_dev, int32_t* n_children_dev, int32_t* child_action_dev,
                  int32_t* child_n_dev, double* child_q_dev, double* child_p_dev, double* v_a0c_dev,
                  double* v_offpolicy_dev, void* stream) {
  if (!e) return fail(-1, "null engine");
  const Params p = e->p;
  dispatch_game(e->cfg.game_id, [&](auto gm) {
    using GM = decltype(gm);
    k_root_stats<GM><<<groups_grid(p.n_trees, GM::G, BLOCK), BLOCK, 0, (cudaStream_t)stream>>>(
        p, root_n_dev, root_q_dev, n_children_dev, child_action_dev, child_n_dev, child_q_dev, child_p_dev, v_a0c_dev,
        v_offpolicy_dev);
    return 0;
  });
  CK(cudaGetLastError());
  return 0;
}

int az_positions(az_engine* e, uint64_t* bb_dev, int32_t* ply_dev, int32_t* terminal_dev, double* return0_dev, void* stream) {
  if (!e) return fail(-1, "null engine");
  const Params p = e->p;
  dispatch_game(e->cfg.game_id, [&](auto gm) {
    using GM = decltype(gm);
    k_positions<GM><<<(p.n_trees + 127) / 128, 128, 0, (cudaStream_t)stream>>>(p, bb_dev, ply_dev, terminal_dev, return0_dev);
    return 0;
  });
  CK(cudaGetLastError());
  return 0;
}

int az_drain_records(az_engine* e, void* host_buf, int64_t max_records, int64_t* n_out, void* stream) {
  if (!e || !n_out) return fail(-1, "null argument");
  cudaStream_t st = (cudaStream_t)stream;
  unsigned long long n = 0;
  CK(cudaMemcpyAsync(&n, e->p.rec_count, sizeof(n), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if ((long long)n > e->p.rec_cap) n = (unsigned long long)e->p.rec_cap;
  if ((int64_t)n > max_records) return fail(-6, "host buffer too small: %lld records buffered, room for %lld", (long long)n, (long long)max_records);
  if (n && host_buf) CK(cudaMemcpyAsync(host_buf, e->p.rec, (size_t)n * e->p.rec_stride, cudaMemcpyDeviceToHost, st));
  CK(cudaMemsetAsync(e->p.rec_count, 0, sizeof(unsigned long long), st));
  CK(cudaStreamSynchronize(st));
  *n_out = (int64_t)n;
  return 0;
}

int az_counters(az_engine* e, uint64_t* out_host, void* stream) {
  if (!e || !out_host) return fail(-1, "null argument");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaMemcpyAsync(out_host, e->p.ctr, sizeof(uint64_t) * AZ_CTR_COUNT, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return 0;
}

int az_game_replay(int32_t game_id, int32_t rows, int32_t cols, int32_t n, const int32_t* hist_dev, const int32_t* len_dev,
                   int32_t max_len, uint64_t* bb_dev, int32_t* status_dev, double* returns0_dev, int32_t* n_legal_dev,
                   int32_t* legal_dev, void* obs_dev, int32_t obs_format, void* stream) {
  if (check_game(game_id, rows, cols)) return -1;
  if (n <= 0) return 0;
  const Geo geo = make_geo(game_id, rows, cols);
  dispatch_game(game_id, [&](auto gm) {
    using GM = decltype(gm);
    k_game_replay<GM><<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(geo, n, hist_dev, len_dev, max_len, bb_dev, status_dev,
                                                                        returns0_dev, n_legal_dev, legal_dev, obs_dev,
                                                                        obs_format);
    return 0;
  });
  CK(cudaGetLastError());
  return 0;
}

int az_observations(int32_t game_id, int32_t rows, int32_t cols, int32_t n, const uint64_t* bb_dev, const int32_t* ply_dev,
                    const int64_t* idx_dev, void* obs_dev, int32_t obs_format, void* stream) {
  if (check_game(game_id, rows, cols)) return -1;
  if (n <= 0) return 0;
  if (!bb_dev || !ply_dev || !obs_dev || obs_format < 1 || obs_format > 2) return fail(-1, "az_observations: bad argument");
  const Geo geo = make_geo(game_id, rows, cols);
  dispatch_game(game_id, [&](auto gm) {
    using GM = decltype(gm);
    k_observations<GM><<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(geo, n, bb_dev, ply_dev, idx_dev, obs_dev, obs_format);
    return 0;
  });
  CK(cudaGetLastError());
  return 0;
}

int az_game_random_playouts(int32_t game_id, int32_t rows, int32_t cols, int32_t n, uint64_t seed, int32_t max_plies,
                            int32_t* hist_dev, int32_t* len_dev, void* stream) {
  if (check_game(game_id, rows, cols)) return -1;
  if (n <= 0) return 0;
  const Geo geo = make_geo(game_id, rows, cols);
  dispatch_game(game_id, [&](auto gm) {
    using GM = decltype(gm);
    k_game_random_playouts<GM><<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(geo, n, seed, max_plies, hist_dev, len_dev);
    return 0;
  });
  CK(cudaGetLastError());
  return 0;
}

}  // extern "C"
