/*
 * az_b200.h -- C-ABI of the B200-native AlphaZero self-play engine (libaz_b200.so).
 *
 * This is the drop-in boundary for the ONE hot path of danielwillemsen/alphazero-openspiel:
 * self-play MCTS.  The reference has no FFI of its own (it is pure Python over pyspiel); each entry
 * point below names the reference interface it replaces (file:line under /root/reference).  The
 * reference-side binding a maintainer would add is a ctypes stub -- see INTEGRATION.md.
 *
 * Conventions
 *   - plain C symbols, opaque handle, int return codes: 0 = ok, negative = error; the message of the
 *     last error on the calling thread is az_last_error().  No exceptions cross the boundary.
 *   - one engine per GPU; not thread-safe per handle; all work is stream-ordered on the caller's
 *     cudaStream_t (passed as void*; NULL = legacy default stream).
 *   - "dev" pointers are device (or host-mapped pinned) addresses the caller owns, e.g. torch
 *     tensor.data_ptr().  "host" pointers are ordinary host memory; calls taking them synchronise the stream.
 *   - there is NO CPU fallback: every entry point that computes launches sm_100a kernels.
 *
 * Engine model (replaces mcts.py:92-203, alphazerobot.py:42-93, game_utils.py:148-206,
 * examplegenerator.py:39-77): `n_trees` independent search trees live in HBM node arenas.  Every tree
 * always has at most ONE evaluator request in flight (the reference has no virtual loss: mcts.py:177-179),
 * so visit counts are bit-exact with the reference for the same evaluator outputs.  One az_step():
 *     consume the evaluator outputs of the previous request  (Node.expand + update_recursive, mcts.py:54-66,82-89;
 *                                                              expand_root_dirichlet, mcts.py:182-190)
 *     run PUCT simulations until the next non-terminal leaf    (MCTS.playout select loop, mcts.py:126-153;
 *                                                              terminal leaves are backed up in-kernel)
 *     when n_playouts are done: pick the move, emit the training record, apply it, re-root + compact
 *                                                             (alphazerobot.py:71-93, game_utils.py:156-204,
 *                                                              MCTS.update_root mcts.py:192-203)
 *     write the observation planes of the new request          (state_to_board, network.py:9-18)
 * so the evaluator batch is always one row per tree.
 *
 * Canonical bitboards: bit i of bb[p] = player p owns cell i, cell = row*cols+col (OpenSpiel cell order:
 * Connect Four row 0 = bottom; Breakthrough row 0 = black's home row).  Side to move = ply & 1.
 *
 * Deterministic counter streams (AZ_NOISE_COUNTER / AZ_F_SAMPLE_COUNTER / az_reset_random / AZ_EVAL_HASH):
 *   mix64 = splitmix64 finaliser; counter(seed,tree,game_seq,ply,idx,stream) = 6 chained mix64
 *   (oracle/az_oracle.c:oz_counter is the CPU restatement).  stream 1 = root noise, 2 = move sampling,
 *   3 = random start plies, 4 = number of random start plies, 5 = device Dirichlet gammas,
 *   6 = no-resign calibration games (AZ_F_RESIGN: counter(seed,tree,game_seq,0,0,6) % 1000 < disabled_permille),
 *   7 = fast searches (AZ_F_PLAYOUT_CAP: the search at root ply `ply` is fast iff
 *       counter(seed,tree,game_seq,ply,0,7) % 1000 >= full_permille).
 */
#ifndef AZ_B200_H
#define AZ_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AZ_GAME_CONNECT_FOUR 0 /* pyspiel.load_game("connect_four") */
#define AZ_GAME_BREAKTHROUGH 1 /* pyspiel.load_game("breakthrough(rows=R,columns=C)") */

/* flags */
#define AZ_F_KEEP_TREE      (1u << 0) /* AlphaZeroBot keep_search_tree (alphazerobot.py:53-64) */
#define AZ_F_AUTO_RESTART   (1u << 1) /* finished game -> new game in the same slot (keeps the batch full) */
#define AZ_F_MANUAL         (1u << 2) /* searches start/stop on host commands (MCTS / AlphaZeroBot drop-in) */
#define AZ_F_SAMPLE_MOVES   (1u << 3) /* self_play=True: sample while ply < num_probabilistic_actions (alphazerobot.py:81-86) */
#define AZ_F_RECORDS        (1u << 4) /* emit per-ply training records (game_utils.py:168-194) */
#define AZ_F_OFFPOLICY      (1u << 5) /* also compute the A0GB off-policy target per ply (game_utils.py:182-194) */
#define AZ_F_PRIORS_F64     (1u << 6) /* az_step priors/values are double (generic policy_fn), else float (Net outputs) */
#define AZ_F_RANDOM_START   (1u << 7) /* (re)started games begin after counter%start_plies_mod random plies (bench synthetic positions) */
#define AZ_F_ASYNC_COMPACT  (1u << 8) /* the caller runs az_compact() itself (e.g. on a side stream next to the evaluator) */
#define AZ_F_EAGER_COMPACT  (1u << 9) /* compact the kept subtree after EVERY move; default: re-root in place and compact
                                         only when the arena half cannot hold another worst-case search */
#define AZ_F_UCT            (1u << 10) /* use_puct=False (mcts.py:80): score = inf if N == 0 else
                                          Q + c_puct * P * sqrt(log(N_parent) / N); log() from a host-built table.  Exactly
                                          as in the reference the formula belongs to the nodes: only a tree whose root was
                                          created by update_root on a leaf root (mcts.py:199-200) uses it */

#define AZ_F_VIRTUAL_LOSS   (1u << 11) /* throughput mode for small pools, NOT bit-exact with the reference (which runs its
                                          playouts strictly in sequence, mcts.py:177-179): up to az_config.leaves_per_tree
                                          leaves in flight per tree, each path carrying a virtual loss until its evaluator
                                          row arrives.  The evaluator batch is n_trees * leaves_per_tree rows, row =
                                          tree * leaves_per_tree + slot, for priors, values and observations alike */
#define AZ_F_EVAL_CACHE     (1u << 12) /* reuse evaluator outputs of positions already evaluated: a direct-mapped device table of
                                          2^AZ_EVAL_CACHE_LOG2(flags) entries keyed by the full position (b0, b1, ply & 1) and a
                                          weights epoch (az_eval_cache_invalidate).  A leaf (or a root awaiting its Dirichlet
                                          expansion) whose position is in the table is expanded from the stored float priors and
                                          value in the same launch instead of requesting an evaluator row.  Bit-exact only if the
                                          evaluator's output for a row depends on that row's position alone (not on its place in the
                                          batch).  Needs AZ_EVAL_EXTERNAL with float priors; not with AZ_F_MANUAL,
                                          AZ_F_VIRTUAL_LOSS or AZ_NOISE_HOST */
/* AZ_F_EVAL_CACHE table size in bits 24-28 of az_config.flags (so that az_config keeps its layout): log2 of the number of
 * entries (64 B each for Connect Four, 256 B for Breakthrough), at most 30; 0 = default: 2^AZ_EVAL_CACHE_EXTRA_LOG2 entries
 * per simulation of one search of every tree (n_trees * n_playouts, rounded up to a power of two), within 2^16..2^27.
 * az_config_get reports the size in use. */
#define AZ_F_RESIGN         (1u << 13) /* resignation (AlphaGo Zero; an extension: the reference plays every game to its end).
                                          At a searched root the mover m = ply & 1 has r = max(-root_q, v_a0c) (the values of
                                          the ply record; v_a0c = -99 when no child was visited).  A game resigns at the first
                                          searched position with r < threshold (strict; threshold <= -1 never fires): the ply
                                          record is emitted with action -1, then the kind-1 record (end = 1) with the resign
                                          position and returns()[0] = -1 if player 0 resigned, else +1; no move is counted and
                                          the game ends like a terminal one.  A no-resign calibration game (counter stream 6,
                                          decided at its first searched position) never resigns and keeps each player's
                                          minimum r.  Threshold and permille: az_set_resign.  Not with AZ_F_MANUAL */
#define AZ_F_PLAYOUT_CAP    (1u << 14) /* playout cap randomization (KataGo; an extension: the reference runs every search with
                                          n_playouts).  A search is decided when it begins: fast with counter stream 7 (see
                                          above), else full.  A full search is the usual one.  A fast search runs fast_playouts
                                          simulations instead of n_playouts and has no root noise (it starts like AZ_NOISE_NONE:
                                          no root request, no AZ_CTR_ROOT_EVALS); the move choice and tree reuse are unchanged.
                                          Its ply record carries end = 3 so that it can be left out of the training examples
                                          (it stays in the record stream: later positions' action histories need its action).
                                          fast_playouts and full_permille: az_set_playout_cap.  Not with AZ_F_MANUAL */
#define AZ_F_FORCED_PLAYOUTS (1u << 15) /* forced playouts and policy target pruning (KataGo; an extension: the reference has
                                          neither).  A search is forced iff, when it begins, k (az_set_forced_playouts) is > 0
                                          and it has root noise (not an AZ_F_PLAYOUT_CAP fast search); it keeps that k.  All
                                          fp64, rounded to nearest; N_root = the root's visit count (the sqrt of the PUCT
                                          score), which differs from the paper's sum of child visits by at most 1.
                                          Selection, root only: nf(c) = sqrt((k * P(c)) * N_root) with P the noise-mixed
                                          prior; a child with 1 <= N(c) < nf(c) scores +inf, so the first one in legal order is
                                          taken; unvisited children are never forced.  Pruning, after the search: c* = the
                                          first child with the maximal count keeps it; every other child with N > 0 gets the
                                          smallest n with N - nf <= n <= N and (n == N or Q + ((c_puct * P) * sqrt(N_root)) /
                                          (n + 1) < the same score of c* at N(c*)); a pruned count of 1 becomes 0.  The
                                          pruned counts are the ones the move is sampled from (argmax cannot change) and the
                                          ply record's counts (root_n stays the raw visit count); root_q, v_a0c, v_offpolicy,
                                          resignation and tree reuse see the tree as it is.  k: az_set_forced_playouts (0 after
                                          az_create).  Not with AZ_F_MANUAL, AZ_F_UCT or AZ_NOISE_NONE */
#define AZ_EVAL_CACHE_LOG2_SHIFT 24
#define AZ_EVAL_CACHE_LOG2(flags) (((flags) >> AZ_EVAL_CACHE_LOG2_SHIFT) & 31u)
#define AZ_EVAL_CACHE_EXTRA_LOG2 1

/* root noise (mcts.py:182-190) */
#define AZ_NOISE_NONE      0 /* use_dirichlet=False */
#define AZ_NOISE_DIRICHLET 1 /* device Dirichlet(alpha) from the counter stream (throughput mode) */
#define AZ_NOISE_HOST      2 /* eta read from az_step(noise_dev): injected np.random.dirichlet draws */
#define AZ_NOISE_COUNTER   3 /* eta_i = u_i / sum(u): exact counter-uniform noise (CPU/GPU bit-identical parity mode) */

/* evaluator */
#define AZ_EVAL_EXTERNAL 0 /* priors/values come from the caller (the ResNet), az_step inputs */
#define AZ_EVAL_UNIFORM  1 /* in-kernel uniform 1/A priors, value 0 (tree-kernel-only throughput) */
#define AZ_EVAL_HASH     2 /* in-kernel hash evaluator (oracle oz_synth_eval kind 1) */
#define AZ_EVAL_ROLLOUT  3 /* MCTS.random_rollout (mcts.py:205-223) in the kernel: priors = 1 for every action, value = the result
                             of one uniformly random playout from the leaf for the player to move there; the move stream is
                             a counter hash of (seed, position) (oracle oz_synth_eval kind 2) */

/* observation formats written by az_step (network.py:9-18 planes + current-player plane) */
#define AZ_OBS_NONE      0
#define AZ_OBS_F32_NCHW  1 /* float32 [n_trees][4][rows][cols] -- the reference layout */
#define AZ_OBS_BF16_NHWC 2 /* bfloat16 [n_trees][rows][cols][4] -- channels-last for the bf16 evaluator */

/* tree phases reported by az_status */
#define AZ_PH_IDLE       0 /* nothing pending (manual mode, or game over without auto-restart) */
#define AZ_PH_ROOT_EVAL  1 /* waiting for the evaluator on the root (Dirichlet expansion) */
#define AZ_PH_LEAF_EVAL  2 /* waiting for the evaluator on a leaf */
#define AZ_PH_SEARCH_DONE 3 /* n_playouts finished; manual mode waits for a command */
#define AZ_PH_RUN        4 /* mid-search, no request this step (per-step simulation cap reached) */
#define AZ_PH_ERROR      5 /* arena / depth overflow: results of this tree are invalid */

typedef struct az_config {
  int32_t game_id, rows, cols;
  int32_t n_trees;
  int32_t node_capacity;       /* nodes per tree per arena half; 0 = default from n_playouts */
  int32_t n_playouts;          /* MCTS(n_playouts=...) mcts.py:99 */
  double c_puct;               /* mcts.py:98 */
  double dirichlet_ratio;      /* mcts.py:101: priors scaled by (1-ratio) */
  double dirichlet_alpha;      /* literal 0.3, mcts.py:187 */
  double noise_weight;         /* literal 0.25, mcts.py:189 */
  double temperature;          /* alphazerobot.py:39,78 */
  int32_t num_probabilistic_actions; /* alphazerobot.py:36 */
  int32_t noise_mode;          /* AZ_NOISE_* */
  int32_t eval_mode;           /* AZ_EVAL_* */
  int32_t eval_shift;          /* AZ_EVAL_HASH prior scale 2^-(10+shift) */
  int32_t max_sims_per_step;   /* cap on in-kernel (terminal-leaf) simulations per tree per step; 0 = unlimited */
  int32_t start_plies_mod;     /* AZ_F_RANDOM_START: k = counter % mod */
  int32_t record_capacity;     /* training records buffered on device; 0 = default */
  int32_t max_games;           /* AZ_F_AUTO_RESTART: total games to start over all trees; 0 = unlimited */
  int32_t device;              /* CUDA device ordinal */
  uint32_t flags;              /* AZ_F_* */
  uint64_t seed;
  int32_t leaves_per_tree;     /* AZ_F_VIRTUAL_LOSS: evaluator rows (leaves in flight) per tree; else 1 */
  int32_t step_cycle_budget;   /* > 0: a tree that already ran a simulation in this az_step starts no further in-kernel
                                  (terminal-leaf) simulation once the launch is this many SM cycles old; bounds the
                                  launch's tail like max_sims_per_step, but by time instead of count; results are
                                  unaffected (exact kernel only; ignored with AZ_F_VIRTUAL_LOSS) */
} az_config;

typedef struct az_engine az_engine;

/* training record (one per ply when AZ_F_RECORDS; kind 1 closes a game).  Stride = az_record_stride(). */
typedef struct az_record {
  int32_t tree, game_seq, ply, action; /* action chosen at this ply (-1 in manual mode) */
  int32_t n_legal, kind;               /* kind 0 = ply, 1 = game end */
  int32_t root_n;
  int32_t end;                         /* kind 1: 0 = terminal position, 1 = resigned, 2 = calibration game (AZ_F_RESIGN)
                                          that reached a terminal position; kind 0: 3 = a fast search (AZ_F_PLAYOUT_CAP),
                                          else 0 */
  uint64_t bb[2];                      /* position the search ran on (kind 1: final or resign position) */
  double root_q;                       /* soft-Z target is -root_q (game_utils.py:174); kind 1: returns()[0] */
  double v_a0c;                        /* game_utils.py:178; kind 1 with end 2: player 0's minimum r (2.0: never moved) */
  double v_offpolicy;                  /* game_utils.py:183-194 (AZ_F_OFFPOLICY); kind 1 with end 2: player 1's minimum r */
  /* followed by int32 counts[max_children]: root child visits in legal (ascending action) order,
   * then int16 actions[max_children]: the action id of each child (-1 beyond n_legal) */
} az_record;

/* counters (az_counters): the measured means SURVEY 8(d) needs for bytes/simulation */
enum {
  AZ_CTR_SIMS = 0,        /* completed simulations (MCTS.playout calls) */
  AZ_CTR_DEPTH,           /* sum of select depth */
  AZ_CTR_CHILDREN,        /* sum of children scored during select */
  AZ_CTR_EXPANSIONS,      /* leaf expansions (evaluator rows answered + AZ_CTR_CACHE_HITS) */
  AZ_CTR_LEGAL,           /* sum of legal moves at expansion */
  AZ_CTR_TERMINAL,        /* simulations that ended on a terminal leaf */
  AZ_CTR_ROOT_EVALS,      /* root (Dirichlet) expansions, from an evaluator row or the AZ_F_EVAL_CACHE table */
  AZ_CTR_MOVES,           /* plies played */
  AZ_CTR_GAMES,           /* games finished */
  AZ_CTR_COMPACT_NODES,   /* nodes copied by re-root compaction */
  AZ_CTR_OVERFLOW,        /* arena/depth/record overflows -- must stay 0 */
  AZ_CTR_IDLE_SLOTS,      /* evaluator rows wasted (no request from that tree this step) */
  AZ_CTR_PEAK_NODES,      /* high-water mark of nodes in use in one tree's arena half (size node_capacity from it) */
  AZ_CTR_CACHE_HITS,      /* leaf expansions served from the AZ_F_EVAL_CACHE table (no evaluator row) */
  AZ_CTR_RESIGNS,         /* AZ_F_RESIGN: games that ended by resignation */
  AZ_CTR_RESIGN_SAMPLES,  /* AZ_F_RESIGN: no-resign calibration games finished */
  AZ_CTR_RESIGN_FALSE,    /* AZ_F_RESIGN: players of finished calibration games whose minimum r was below the threshold in
                             force at the game's end and who did not lose (would-be false resignations) */
  AZ_CTR_COUNT
};

const char* az_last_error(void);
int az_version(void);

/* MCTS.__init__ / AlphaZeroBot.__init__ / ExampleGenerator.__init__ kwargs (mcts.py:96-124,
 * alphazerobot.py:26-40, examplegenerator.py:80-104) -> one engine. */
int az_create(const az_config* cfg, az_engine** out);
int az_destroy(az_engine* e);
int az_config_get(const az_engine* e, az_config* out); /* effective config (defaults filled) */
int az_max_children(const az_engine* e);               /* 7 / rows*cols... bound used for per-tree child arrays */
int az_num_actions(const az_engine* e);                /* game.num_distinct_actions() */
int az_record_stride(const az_engine* e);              /* bytes per az_record incl. counts[] */
int64_t az_device_bytes(const az_engine* e);           /* HBM held by the engine */

/* game.new_initial_state() for every tree + fresh roots (game_utils.py:150-154); begins the first search
 * unless AZ_F_MANUAL.  With AZ_F_RANDOM_START the synthetic start positions are used. */
int az_reset(az_engine* e, void* stream);

/* Manual mode: set tree positions by replaying action histories (state.history(), alphazerobot.py:55) on the
 * device.  hist_host: [n_trees][max_len] int32 actions, len_host[n_trees] (len -1 = leave tree untouched).
 * Tree nodes are left as they are (MCTS.search(state) trusts the caller, mcts.py:164). */
int az_set_positions(az_engine* e, const int32_t* hist_host, const int32_t* len_host, int32_t max_len, void* stream);

/* Manual mode commands, one per tree (host arrays, -1 / 0 = no-op):
 *   update_root_host[i] >= 0 : MCTS.update_root(action) mcts.py:192-203 (also advances the tree's position)
 *   reset_tree_host[i] != 0  : self.mcts = MCTS(...) (alphazerobot.py:66-68) -- fresh root; the value 2 builds the root that
 *                              update_root creates for a leaf root instead (it carries use_puct, see AZ_F_UCT)
 *   begin_host[i] != 0       : MCTS.search(state) mcts.py:164-180 -- start n_playouts simulations; the value 2 runs
 *                              MCTS.playout(state) mcts.py:126-153 instead: ONE simulation, no root Dirichlet expansion
 * Order applied: reset, update_root, begin. */
int az_command(az_engine* e, const int32_t* update_root_host, const int32_t* reset_tree_host,
               const int32_t* begin_host, void* stream);

/* One evaluator round trip.  priors_dev [n_trees][num_actions] and values_dev [n_trees] answer the requests
 * produced by the previous az_step/az_reset (ignored for trees without a request; may be NULL on the first
 * call or with an in-kernel evaluator; with AZ_F_VIRTUAL_LOSS the batch is n_trees * leaves_per_tree rows).  noise_dev [n_trees][max_children] doubles (AZ_NOISE_HOST).
 * obs_dev receives the next requests in obs_format.  policy_fn(state) of mcts.py:146,183 is thus batched as
 * eval_batch(obs) -> (priors, values). */
int az_step(az_engine* e, const void* priors_dev, const void* values_dev, const double* noise_dev,
            void* obs_dev, int32_t obs_format, void* stream);

/* AZ_F_EVAL_CACHE: the evaluator's weights change after this call.  Stream-ordered: evaluator rows that az_step consumes
 * next were computed before the change and are still stored under the old weights; from that az_step on, entries of the
 * old weights no longer match. */
int az_eval_cache_invalidate(az_engine* e, void* stream);

/* AZ_F_RESIGN: resign threshold and the share of no-resign calibration games, in per mille (0..1000).  A stream-ordered write
 * to device memory that the step kernels read there, so a captured CUDA graph of az_step sees the new values on its next
 * replay.  After az_create: threshold -1.0 (never resigns), permille 0.  A game's calibration status is drawn with the
 * permille in force at its first searched position.  Rejects a non-finite threshold, a permille outside [0, 1000] and an
 * engine created without AZ_F_RESIGN. */
int az_set_resign(az_engine* e, double threshold, int32_t disabled_permille, void* stream);

/* AZ_F_PLAYOUT_CAP: simulations of a fast search and the share of full searches, in per mille (0..1000).  A stream-ordered
 * write to device memory like az_set_resign: a captured CUDA graph of az_step uses the new values on its next replay.  A
 * search is decided with the values in force when it begins.  After az_create: fast_playouts = n_playouts, permille 1000
 * (every search is full).  Rejects fast_playouts outside [1, n_playouts], a permille outside [0, 1000] and an engine
 * created without AZ_F_PLAYOUT_CAP. */
int az_set_playout_cap(az_engine* e, int32_t fast_playouts, int32_t full_permille, void* stream);

/* AZ_F_FORCED_PLAYOUTS: the k of the forced-playout floor (the paper's value is 2; 0 forces no search).  A stream-ordered
 * write to device memory like az_set_playout_cap: a captured CUDA graph of az_step uses the new value on its next replay.
 * A search keeps the k in force when it begins.  After az_create: k = 0.  Rejects a non-finite or negative k and an engine
 * created without AZ_F_FORCED_PLAYOUTS. */
int az_set_forced_playouts(az_engine* e, double k, void* stream);

/* Re-root compaction (MCTS.update_root, mcts.py:192-203) of the trees that played a move in the last az_step: BFS-copies
 * the kept subtree into the other arena half, one warp per tree.  az_step runs it first by itself unless
 * AZ_F_ASYNC_COMPACT is set; then the caller must call it once between two az_step calls, on any stream ordered after
 * the first and before the second (typically a side stream, overlapping the evaluator). */
int az_compact(az_engine* e, void* stream);

/* Development aid: per-tree SM cycle counts of the last az_step into host memory [n_trees][4] (total cycles, phase on
 * entry, simulations run, 2*consume_cycles + moved).  The first call arms the instrumentation (returns zeros). */
int az_debug_timing(az_engine* e, long long* out_host);

/* Per-tree status into device arrays (any may be NULL): phase (AZ_PH_*), sims done in the current search,
 * ply of the root position, legal-move count of the pending request's position. */
int az_status(az_engine* e, int32_t* phase_dev, int32_t* sims_dev, int32_t* ply_dev, int32_t* req_legal_dev,
              void* stream);

/* Pending request positions: canonical bitboards [n_trees][2], ply [n_trees], and the action path from the
 * root to the requested leaf [n_trees][max_depth] with its length depth_dev[n_trees] -- lets a host policy_fn
 * rebuild the leaf state (root.clone() + apply_action along the path).  In manual mode a tree in AZ_PH_SEARCH_DONE reports
 * the path of its LAST simulation (depth >= 0, bitboards 0 / ply -1): MCTS.playout leaves the caller's state at the leaf. */
int az_request_info(az_engine* e, uint64_t* bb_dev, int32_t* ply_dev, int32_t* path_actions_dev,
                    int32_t* depth_dev, int32_t max_depth, void* stream);

/* Root statistics (MCTS.root.N/.Q, children N/Q/P: mcts.py:155-162, game_utils.py:174-194), per tree:
 * root_n[n], root_q[n], n_children[n], child_action/child_n/child_q/child_p [n][max_children] in legal order,
 * v_a0c[n], v_offpolicy[n].  Any pointer may be NULL. */
int az_root_stats(az_engine* e, int32_t* root_n_dev, double* root_q_dev, int32_t* n_children_dev,
                  int32_t* child_action_dev, int32_t* child_n_dev, double* child_q_dev, double* child_p_dev,
                  double* v_a0c_dev, double* v_offpolicy_dev, void* stream);

/* Root positions: bitboards [n_trees][2], ply [n_trees], terminal flag, returns()[0] (device arrays, NULL ok). */
int az_positions(az_engine* e, uint64_t* bb_dev, int32_t* ply_dev, int32_t* terminal_dev, double* return0_dev,
                 void* stream);

/* Copy buffered training records to host memory and clear the device buffer (synchronises the stream).
 * Returns the number of records through n_out. */
int az_drain_records(az_engine* e, void* host_buf, int64_t max_records, int64_t* n_out, void* stream);

/* Cumulative counters (AZ_CTR_COUNT uint64) to host (synchronises the stream). */
int az_counters(az_engine* e, uint64_t* out_host, void* stream);

/* ---- stateless batched game ops (pyspiel State subset, SURVEY B.1) -- used by the parity tests ----
 * Replays `len[i]` actions of hist[i][max_len] from the initial state of (game_id, rows, cols) and writes, for
 * the reached position: bitboards [n][2]; status [n]: bit0 terminal, bit1 an action was illegal;
 * returns0 [n]; legal mask as n_legal [n] + legal actions [n][max_children] ascending;
 * observation in obs_format.  All pointers are device pointers (NULL ok). */
int az_game_replay(int32_t game_id, int32_t rows, int32_t cols, int32_t n, const int32_t* hist_dev,
                   const int32_t* len_dev, int32_t max_len, uint64_t* bb_dev, int32_t* status_dev,
                   double* returns0_dev, int32_t* n_legal_dev, int32_t* legal_dev, void* obs_dev,
                   int32_t obs_format, void* stream);

/* state_to_board (network.py:9-18) for a gathered minibatch of a replay buffer held on the device as canonical bitboards
 * [.][2] + ply [.]: row i of obs_dev (obs_format AZ_OBS_F32_NCHW / AZ_OBS_BF16_NHWC) = the planes of example idx_dev[i]
 * (int64; NULL = example i).  The trainer's minibatch builder (train.py:108-112). */
int az_observations(int32_t game_id, int32_t rows, int32_t cols, int32_t n, const uint64_t* bb_dev, const int32_t* ply_dev,
                    const int64_t* idx_dev, void* obs_dev, int32_t obs_format, void* stream);

/* Random playouts entirely on the device from counter stream 3 (seed, i): plays up to max_plies uniformly
 * random legal moves per game and writes the action history (hist_dev [n][max_plies], len_dev [n]).  Used to
 * generate full-size property-test inputs without host work. */
int az_game_random_playouts(int32_t game_id, int32_t rows, int32_t cols, int32_t n, uint64_t seed,
                            int32_t max_plies, int32_t* hist_dev, int32_t* len_dev, void* stream);

/* ---- evaluator kernels (az_resnet.cu): the ResNet of network.py:21-104 for the batched evaluator ----
 * Activations are NHWC bf16 tensors [boards][H+1][W][64]: the 50 filters zero-padded to 64, and one extra board row (row H)
 * that must be zero when a tensor is first used and is kept zero by the kernels - it separates consecutive boards.  There
 * are no pad columns in global memory (TMA zero-fills / clips them).  All pointers are device pointers; 3 <= H <= 16,
 * 2 <= W <= 8.
 *
 * az_nn_conv3x3: out = conv3x3(in) + bias, optional LeakyReLU, optional + res; optional second output
 *   out2 = LeakyReLU(s2*out + t2) (the next block's BatchNorm, network.py:100).  The conv computes the network's 50 filters
 *   (network.py:22) from all 64 input channels; channels 50..63 of out / out2 are written as zeros.
 *   wpack is bf16 [3 ky][160][8][8]: per kernel row the three kx taps side by side without padding, row r = kx*50 + co =
 *   the 64 input channels (128 B) of output channel co, rows 150..159 zero, in the SWIZZLE_128B K-major UMMA image (16-byte
 *   chunk c stored at position c ^ (r & 7)).  tcgen05 implicit GEMM, 12 MMAs of M128 N160 K16 per 128-row tile, three
 *   TMEM accumulator stages; n_ctas <= 0 -> one CTA per SM.  res may alias out (in-place residual stream).  flags: AZ_NN_F_*.
 * az_nn_stem: the first conv of resblock1 on the 4 observation planes, slab built from the az_step AZ_OBS_BF16_NHWC batch
 *   [boards][H][W][4]: u[0..49] = LeakyReLU(conv1(LeakyReLU(s*x+t)) + b1) (network.py:99-100) and u[50..53] = x, the raw
 *   planes: the block's 1x1 skip projection (resblock1.conv3, network.py:101-103) is then four extra input channels of the
 *   centre tap of the following az_nn_conv3x3.  wpack is bf16 [9 taps = ky*3+kx][2 k-chunks][64 n][8],
 *   no-swizzle K-major, only k 0-3 of chunk 0 non-zero (BatchNorm 2 folded).  bn_st = device [8]: scale[4], shift[4].
 * az_nn_head: the FC head (fc1, network.py:48,61-66) for games with n_actions + 1 <= 8 outputs: priors [.][n_actions] =
 *   softmax(x_flat @ w[0..A-1]^T + bias), values = tanh(x_flat @ w[A]^T + bias[A]), fp32.  w is bf16 [8][H*W*64] over the
 *   H*W cells of one board (zero on pad channels / unused outputs; the pad row is not read), bias fp32 [8]. */
/* az_nn_block: one whole residual block without projection (network.py:99-104, blocks 2-5) in one launch:
 *   U = LeakyReLU(conv3x3(t_in; w1) + b1) (bn2 folded into w1 / b1), x <- conv3x3(U; w2) + b2 + x (in place),
 *   t_out = LeakyReLU(s2 * x + t2) when t_out != NULL (the next block's bn1 + LeakyReLU).  The intermediate U stays in shared
 *   memory (4 instead of 6 activation passes through HBM).  w1 / w2: the wpack images of az_nn_conv3x3; tensors as there;
 *   t_out and x must not alias t_in. */
int az_nn_block(const void* t_in, const void* w1, const float* b1, const void* w2, const float* b2, void* x, void* t_out,
                const float* s2, const float* t2, int32_t boards, int32_t H, int32_t W, int32_t n_ctas, void* stream);
#define AZ_NN_F_REVERSE 1 /* walk the 128-row tiles back to front (alternate per layer: the tail of the previous layer's
                             output is still in L2) */
const char* az_nn_last_error(void);
int az_nn_conv3x3(const void* in, const void* wpack, const float* bias, const void* res, void* out, void* out2,
                  const float* s2, const float* t2, int32_t boards, int32_t H, int32_t W, int32_t lrelu, int32_t flags,
                  int32_t n_ctas, void* stream);
int az_nn_stem(const void* obs, const void* wpack, const float* b1, const float* bn_st, void* u, int32_t boards, int32_t H,
               int32_t W, int32_t n_ctas, void* stream);
int az_nn_head(const void* x, const void* w, const float* bias, float* priors, float* values, int32_t boards, int32_t H,
               int32_t W, int32_t n_actions, int32_t n_ctas, void* stream);
/* az_nn_head_large: the same FC head (fc1 + softmax over ALL n_actions + tanh, network.py:48,60-64) for large action spaces
 *   (Breakthrough: 433 / 769 outputs) as a tcgen05 GEMM: M = boards, K = H*W*64 (the board cells of x; the pad row is
 *   skipped), N = n_actions + 1, fp32 accumulation and fp32 logits.  w is bf16 [n_actions + 1][(H+1)*W*64] (row n = the
 *   weights of output n in the NHWC cell order of x, zero on pad channels; the last (H+1)-th row group is never read),
 *   bias fp32 [n_actions + 1].  scratch: az_nn_head_large_scratch_bytes(boards, n_actions) bytes of device memory, zeroed
 *   once by the caller before the first use (chunk statistics + self-resetting tile counters). */
int64_t az_nn_head_large_scratch_bytes(int32_t boards, int32_t n_actions);
int az_nn_head_large(const void* x, const void* w, const float* bias, float* priors, float* values, void* scratch,
                     int32_t boards, int32_t H, int32_t W, int32_t n_actions, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AZ_B200_H */
