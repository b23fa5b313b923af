/*
 * azalea_b200.h -- C ABI of the B200-native Azalea self-play search engine.
 *
 * The reference (jseppanen/azalea) is pure Python + Numba and has no FFI for
 * this path; these entry points are what a binding for it would call, one
 * per reference function on the hot path (SURVEY.md section 8b).  Each cites
 * the reference file:line it replaces.  INTEGRATION.md shows the ctypes stub
 * a maintainer would add on the reference side.
 *
 * Conventions
 *  - plain pointers and sizes only; no torch / C++ types.
 *  - `*_dev` pointers are device pointers, everything else is host memory.
 *  - every op enqueues work on `stream` (a cudaStream_t passed as void*, NULL
 *    = legacy default stream) and returns without synchronising.
 *  - return value: 0 = ok, negative = AZ_E_* (az_strerror()).
 *  - one game per row: arrays are indexed [game][...]; G = num_games.
 *  - moves are 1-based tile ids (0 = padding / "no move"), move ids are
 *    ordinals in the ascending legal-move list, colours are 1 (X, first
 *    player) / 2 (O), results 0 ongoing / 1 O won / 3 X won -- all as in the
 *    reference (game/hex.py:151-179, typing/agent.py:34-41).
 *
 * Memory: the caller owns ONE device block of az_engine_device_bytes() bytes
 * (allocate it with the framework's allocator, e.g. a torch uint8 tensor);
 * az_engine_buffer() gives the offset/shape of the views the caller may read
 * or write directly (leaf boards for the network, value/prior inputs ...).
 */
#ifndef AZALEA_B200_H
#define AZALEA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AZ_ABI_VERSION 3

enum {
    AZ_OK = 0,
    AZ_E_INVALID = -1,      /* bad argument */
    AZ_E_CUDA = -2,         /* CUDA runtime error (az_last_cuda_error()) */
    AZ_E_NOMEM = -3,        /* device block too small */
    AZ_E_UNSUPPORTED = -4
};

/* per-game status bits (az_status) */
enum {
    AZ_ST_POOL_FULL = 1,    /* physical node pool exhausted */
    AZ_ST_TREE_FULL = 2,    /* reference MAX_NODES reached: SearchTreeFull,
                               search_tree.py:17-22,258-259 */
    AZ_ST_ILLEGAL = 4,      /* illegal move / inconsistent state (the
                               reference's AssertionError, hex.py:174-176) */
    AZ_ST_DISABLED = 8
};

/* leaf flags (leaf_info[..][1] & 0xff) */
enum {
    AZ_LEAF_TERMINAL_KNOWN = 1, /* re-visited terminal node, mcts.py:236-237 */
    AZ_LEAF_TERMINAL_NEW = 2    /* first visit found the game over */
};
/* leaf_info[..][1] bit 9: the leaf's network row is rotated (az_engine_set_reflect) */
#define AZ_LEAF_REFLECTED_BIT 9

typedef struct az_config {
    int32_t num_games;       /* G: games resident on this GPU */
    int32_t board_size;      /* n: 2..19 */
    int32_t max_batch;       /* search_batch_size upper bound, 1..32 */
    int32_t nodes_per_game;  /* capacity of each half of a game's node pool */
    int64_t max_nodes_ref;   /* search_tree.MAX_NODES emulation (1e7) */
    int32_t replay_rows;     /* capacity of the replay output buffer (rows) */
    int32_t max_plies;       /* play_game game_max_length (300) clipped to n*n */
    uint64_t seed;           /* Philox key; streams keyed by global game id */
    int64_t first_game_id;   /* global id of local game 0 (rank * G) */
    int64_t game_id_stride;  /* ids of successive games in one slot differ by this
                                (total games over all ranks) */
    int32_t flags;           /* AZ_CFG_* */
    int32_t reserved;
} az_config;

/* az_config.flags */
enum {
    /* When a game's physical node pool is exhausted, leave the leaf
     * unexpanded (it is still backed up, and expanded on a later visit once
     * the next re-root has compacted the pool) instead of flagging
     * AZ_ST_POOL_FULL and dropping the game.  The reference never gets there
     * (one 1e7-node pool per game, search_tree.py:17-18); skipped expansions
     * are counted in AZ_CNT_POOL_SKIPPED. */
    AZ_CFG_SOFT_POOL_FULL = 1,
    /* Packed leaves.  The reference evaluates only the unique, non-terminal
     * leaves of a batch (mcts.py:75,139-152,192-200); with this flag
     * az_mcts_select writes exactly those, densely: the boards of a window's
     * leaves go to rows [g0 * max_batch, g0 * max_batch + live) of
     * AZ_BUF_LEAF_BOARD (g0 = first game of the window), live is left in
     * AZ_BUF_LEAF_ROWS[g0], leaf_info[..][3] becomes depth | row << 10, and
     * az_mcts_expand_backup reads value / prior of a leaf at its row and
     * resets the count.  The evaluator (az_nn_*_live) then works on `live`
     * rows instead of num_games * max_batch: duplicates and terminal leaves
     * cost no network time.  Not for az_leaf_moves / host evaluators. */
    AZ_CFG_PACK_LEAVES = 2
};

typedef struct az_engine az_engine;

/* buffers the caller may view inside its device block */
enum {
    AZ_BUF_LEAF_BOARD = 0,  /* int8  [G][max_batch][cell_stride]  network-view cells 0/1/2 */
    AZ_BUF_LEAF_INFO = 1,   /* int32 [G][max_batch][4] node(-1 = none), flags|colour<<8|rotated<<9, num_moves, depth
                               (AZ_CFG_PACK_LEAVES: depth | row << 10) */
    AZ_BUF_VALUE = 2,       /* f32   [G][max_batch]           evaluator output */
    AZ_BUF_PRIOR = 3,       /* f32   [G][max_batch][n*n]      evaluator output (priors or logits) */
    AZ_BUF_META = 4,        /* int32 [G][16]; [14] = descent count when this move's search
                               began (az_engine_set_playout_cap) */
    AZ_BUF_REPLAY = 5,      /* uint8 [replay_rows][replay_row_bytes] */
    AZ_BUF_COUNTERS = 6,    /* int64 [G][16] per-game counters (sum over games on the host) */
    AZ_BUF_LEAF_MOVES = 7,  /* int32 [G][max_batch][n*n] network-view legal moves, 0-padded */
    AZ_BUF_GLOBALS = 8,     /* int64 [16]: [0] = replay append cursor (rows) */
    AZ_BUF_LEAF_ROWS = 9,   /* int32 [G]: [g0] = live leaf rows of the window starting at game g0
                               (AZ_CFG_PACK_LEAVES) */
    AZ_BUF_RESIGN = 10,     /* uint32 [G][72] per-slot resignation state (az_engine_set_resign;
                               sum the counts over games on the host): [0], [1] = f32 bits of
                               colour 1's / 2's lowest r in the current game (+inf at its start);
                               [2] = games that ended by resignation; [3] = calibration games that
                               ended with a winner; [4] = of those, games whose winner's lowest r
                               was below the threshold (false positives); [5..69] = histogram of
                               the winner's lowest r over [3]'s games, bin min(64, max(0,
                               floor((r + 1) * 64))) in f32; [70], [71] padding */
    AZ_BUF__COUNT = 11
};

/* counter columns (AZ_BUF_COUNTERS); each game's warp owns its row, so the
 * hot kernels never contend on an atomic */
enum {
    AZ_CNT_SIMULATIONS = 0,   /* root-to-leaf descents */
    AZ_CNT_SUM_CHILDREN = 1,  /* sum over descents and levels of k */
    AZ_CNT_SUM_DEPTH = 2,     /* sum over descents of depth */
    AZ_CNT_UNIQUE_LEAVES = 3,
    AZ_CNT_EXPANDED_CHILDREN = 4,
    AZ_CNT_PLIES = 5,         /* committed self-play moves */
    AZ_CNT_GAMES = 6,         /* finished self-play games */
    AZ_CNT_REPLAY_ROWS = 7,   /* rows appended to the replay buffer */
    AZ_CNT_REPLAY_DROPPED = 8,
    AZ_CNT_GAMES_FAILED = 9,  /* dropped on SearchTreeFull, parallel_player.py:71-76 */
    AZ_CNT_COMPACTED_NODES = 10,
    AZ_CNT_NN_ROWS = 11,      /* non-terminal unique leaves (rows the network must evaluate) */
    AZ_CNT_POOL_SKIPPED = 12, /* expansions skipped because the pool half was full (AZ_CFG_SOFT_POOL_FULL) */
    AZ_CNT_TERMINAL_LEAVES = 13, /* unique leaves that were terminal positions (value -1, mcts.py:192-195) */
    AZ_CNT_REFLECTED_ROWS = 14, /* network rows written rotated (az_engine_set_reflect) */
    AZ_CNT_FAST_PLIES = 15      /* committed moves of fast plies (az_engine_set_playout_cap);
                                   their rows are not flushed to the replay output */
};

typedef struct az_buffer_desc {
    size_t offset;          /* bytes from the start of the device block */
    size_t bytes;
    int32_t elem_bytes;
    int32_t ndim;
    int64_t shape[4];
} az_buffer_desc;

/* -------------------------------------------------------------- lifecycle */

int az_abi_version(void);
const char *az_strerror(int code);
const char *az_last_cuda_error(void);

/* SearchTree.__init__, search_tree.py:43-57: how much device memory a pool
 * of G trees + boards + scratch needs. */
size_t az_engine_device_bytes(const az_config *cfg);
int az_engine_create(az_engine **out, const az_config *cfg, void *mem_dev,
                     size_t mem_bytes, int device);
void az_engine_destroy(az_engine *e);
int az_engine_buffer(const az_engine *e, int which, az_buffer_desc *out);
int az_replay_row_bytes(const az_engine *e);

/* ------------------------------------------------------------------ games */

/* Restrict the per-game entry points below (everything that launches one warp
 * per game: reset, hex_*, mcts_*, leaf_moves, root_stats, tree_move, stub_eval,
 * play_commit) to the games [first_game, first_game + num_games); num_games <=
 * 0 restores the full range.  Per-game arrays owned by the engine or sized
 * [G] by the caller keep their absolute indexing; the value / prior arrays
 * handed to az_mcts_expand_backup hold the window's rows only.  The window is
 * read at launch time, so two halves of the games can be driven on two
 * streams: the tree kernels of one half run under the evaluator of the other
 * (selfplay.LockstepSelfPlay(streams=2)). */
int az_engine_set_window(az_engine *e, int first_game, int num_games);

/* Random orientation of the network rows (the reference's random_reflect
 * hook, mcts.py:179-186), off by default.  Hex has one symmetry that keeps
 * the rules: the 180-degree rotation tile t -> n*n-1-t.  With on != 0,
 * az_mcts_select and az_mcts_select_root draw one coin per leaf that goes to
 * the network from the game's Philox stream (counter: descent, ply) and, when
 * it is set, write the leaf's AZ_BUF_LEAF_BOARD row rotated and set
 * AZ_LEAF_REFLECTED in leaf_info[..][1]; the AZ_PRIOR_LOGITS path of
 * az_mcts_expand_backup / az_mcts_expand_root reads the logit of tile t of a
 * rotated row at n*n-1-t.  Coins do not depend on windows, streams or the
 * world size.  AZ_PRIOR_PROBS priors (by move ordinal), az_stub_eval and
 * az_leaf_moves refer to the true board and ignore the orientation: a host
 * evaluator leaves this off and rotates its own batch.  Read at launch time
 * like the window (set it before capturing a graph).  Off: every buffer is
 * byte for byte what it is without this call. */
int az_engine_set_reflect(az_engine *e, int on);

/* Playout cap randomization (Wu 2019, "Accelerating Self-Play Learning in
 * Go"), off by default.  At each ply every game draws one coin from its
 * Philox key (counter: ply), so the draw does not depend on windows, streams
 * or the world size; with probability full_search_prob the ply gets the full
 * search.  Otherwise it is a fast ply: az_mcts_select stops searching the
 * game once it has made fast_descents new descents in this move (counted from
 * az_mcts_select_root, which every move must begin with; visits reused from
 * the previous move do not count, and the check is made per launch, so
 * fast_descents should be a multiple of the batch size), a capped game emits
 * no leaves, and the root draws and mixes no Dirichlet noise.  az_play_commit
 * picks the move by the same rule on both kinds of ply, counts fast plies in
 * AZ_CNT_FAST_PLIES and flushes only the rows of full plies to the replay
 * output (game_len and result are still the whole game's).  The start of the
 * move's search is kept in meta slot 14.  full_search_prob >= 1 turns it off;
 * AZ_E_INVALID for a negative or NaN probability, or for fast_descents < 1
 * with the cap on.  Read at launch time like the window (set it before
 * capturing a graph).  Off: every buffer is byte for byte what it is without
 * this call. */
int az_engine_set_playout_cap(az_engine *e, float full_search_prob, int fast_descents);

/* Resignation with calibration games (AlphaGo Zero, Silver et al. 2017,
 * "Methods: Self-play"), off by default.  az_play_commit, after the search
 * and before the move is drawn, computes r = max(Q_root, Q_best) for the
 * player to move: Q_root = W/N of the root, Q_best = -W/N of the most-visited
 * root child (lowest ordinal on ties; r = Q_root if no child has a visit), in
 * f32 with round-to-nearest divisions.  Each game draws one coin from its
 * Philox key (counter: 0), so the draw does not depend on windows, streams or
 * the world size; with probability disable_prob the game is a calibration
 * game and never resigns.  In any other game, r < threshold makes the mover
 * resign: no move is drawn, no row is recorded for that ply and the tree is
 * not re-rooted; the opponent is the winner, chosen_dev gets (0, -1, result,
 * ply), and the game is finished like a won one (rows of plies 0..ply-1 are
 * flushed with game_len = ply, AZ_CNT_GAMES counts it, AZ_CNT_PLIES does not
 * count the resigning ply; then auto_reset).  The check comes before the
 * max_plies draw and runs on fast plies of the playout cap as well.  A
 * calibration game keeps each colour's lowest r and, when it ends with a
 * winner, counts itself, a false positive if the winner's lowest r is below
 * the threshold, and the winner's lowest r in a histogram (AZ_BUF_RESIGN).
 * The false positives bound the rate of wrong resignations from above: the
 * loser might have resigned first.  Draws and failed games are not counted.
 * threshold <= -1 turns it off; disable_prob = 1 measures without resigning.
 * AZ_E_INVALID for a NaN threshold or one above 1, or for disable_prob
 * outside [0, 1].  Read at launch time like the window (set it before
 * capturing a graph).  Off: every other buffer is byte for byte what it is
 * without this call. */
int az_engine_set_resign(az_engine *e, float threshold, float disable_prob);

/* Forced playouts and policy target pruning (Wu 2019, "Accelerating
 * Self-Play Learning in Go", section 3.2), off by default.  Forcing: on full
 * plies (every ply unless the playout cap is on), az_mcts_select gives a root
 * child with 0 < N < n_forced = sqrt(k * P * sum N) the score +inf, so the
 * lowest such ordinal is descended into; sum N is the children's visit sum
 * including the batch's virtual losses, and P is the child's stored prior, not
 * the noised one (the noise is drawn per simulation), in f32 with one rounding
 * per operation.  Root mode and fast plies never force.  Pruning: on full
 * plies az_play_commit, after the move has been drawn from the raw visits,
 * writes pruned visits into the ply's replay row: with c* the most-visited
 * child (lowest ordinal on ties) and score(c, n) = Q_c + (exploration_coef *
 * P_c) * (sqrt(sum N) / (1 + n)) in az_mcts_select's operation order (Q_c
 * from the child's real N), every other visited child keeps the fewest n that
 * still score below score(c*, N*), but at least N - floor(n_forced) and at
 * most N, and one left at 1 visit gets 0.  The tree, the move, chosen_dev,
 * resignation and every counter see the raw visits.  k == 0 turns it off;
 * AZ_E_INVALID for a negative or non-finite k or exploration_coef, which
 * should be the coefficient az_mcts_select is launched with.  Read at launch
 * time like the window (set it before capturing a graph).  Off: every buffer
 * is byte for byte what it is without this call. */
int az_engine_set_forced_playouts(az_engine *e, float k, float exploration_coef);

/* HexGame.reset + Policy.reset for the games whose mask byte is non-zero
 * (NULL = all), hex.py:47-49, policy.py:72-76, search_tree.py:59-71. */
int az_games_reset(az_engine *e, const uint8_t *mask_dev, void *stream);
/* HexGameImpl.step on each game's root position, hex.py:172-179.  moves 0 =
 * leave the game alone.  results_dev (nullable) receives 0/1/3. */
int az_hex_step(az_engine *e, const int32_t *moves_dev, int32_t *results_dev,
                void *stream);
/* HexGame.state, hex.py:55-60: board int8[G][n*n] (0/1/2, absolute view),
 * colour to move 0/1, result 0/1/3, ply.  Any pointer may be NULL. */
int az_hex_state(az_engine *e, int8_t *board_dev, int32_t *color_dev,
                 int32_t *result_dev, int32_t *ply_dev, void *stream);
/* HexGameImpl.legal_moves, hex.py:151-159: int32[G][n*n] ascending, 0-padded */
int az_hex_legal_moves(az_engine *e, int32_t *moves_dev, int32_t *count_dev,
                       void *stream);
/* Overwrite root positions (HexGame.__setstate__, hex.py:39-45): board
 * int8[G][n*n], colour to move 1/2.  The winner is recomputed from
 * `last_tile_dev` (nullable; -1 = none).  reset_trees != 0 also clears the
 * search trees (Policy.reset); 0 keeps them (the caller vouches that the
 * tree root is this position, as SearchTree.search does). */
int az_hex_set_state(az_engine *e, const int8_t *board_dev,
                     const int32_t *color_dev, const int32_t *last_tile_dev,
                     int reset_trees, void *stream);

/* ----------------------------------------------------------------- search */

typedef struct az_search_params {
    int32_t batch_size;         /* search_batch_size, mcts.py:62 */
    float exploration_coef;     /* c_puct, mcts.py:133 */
    double noise_scale;         /* Dirichlet epsilon (0 = off), mcts.py:126-131 */
    double noise_alpha;
} az_search_params;

/* evaluate_root's selection half, mcts.py:18-24: games with an unevaluated
 * root emit the root position as leaf slot 0; others emit nothing. */
int az_mcts_select_root(az_engine *e, void *stream);
/* select_batch + deduplicate_leaves, mcts.py:46-76,139-152: batch_size
 * sequential PUCT descents per game with virtual loss, undo, first-occurrence
 * dedup, leaf position + win check, network-view board planes
 * (mcts.py:176-181, hex.py:72-87). */
int az_mcts_select(az_engine *e, const az_search_params *p, void *stream);
/* Network-view legal moves of the current leaves into AZ_BUF_LEAF_MOVES
 * (prep.batch_games + flip_player_board_moves, prep.py:15-21, hex.py:89-122);
 * only the generic evaluator interface needs them. */
int az_leaf_moves(az_engine *e, void *stream);

enum {
    AZ_PRIOR_PROBS = 0,     /* prior[g][b][j] by move ordinal, stride n*n */
    AZ_PRIOR_LOGITS = 1     /* logits[g][b][tile] by network-view tile; the engine
                               gathers legal tiles, masked log-softmax, exp
                               (network.py:146-151, mcts.py:210) */
};
/* evaluate_batch's terminal rule + expand_batch + backup_batch,
 * mcts.py:192-200,226-255.  value_dev f32[G][max_batch], prior_dev
 * f32[G][max_batch][n*n]; NULL = the engine's own AZ_BUF_VALUE/PRIOR. */
int az_mcts_expand_backup(az_engine *e, const float *value_dev,
                          const float *prior_dev, int prior_kind,
                          void *stream);
/* evaluate_root's expansion half, mcts.py:25-26 (value discarded). */
int az_mcts_expand_root(az_engine *e, const float *prior_dev, int prior_kind,
                        void *stream);
/* root.move_stats + root node, search_tree.py:105-112,192-204:
 * visits/total_value/prior f32[G][n*n] (children in legal-move order,
 * total_value in the stored (child's own) sign), num_children int32[G]
 * (-1 = unevaluated root), root_nw f32[G][2] = (N, W) of the root,
 * num_nodes int64[G] = the reference's tree.num_nodes.  NULLs are skipped. */
int az_root_stats(az_engine *e, float *visits_dev, float *total_value_dev,
                  float *prior_dev, int32_t *num_children_dev,
                  float *root_nw_dev, int64_t *num_nodes_dev, void *stream);
/* RandomPolicy.choose_action (random_policy.py:25-41) for every game: puts
 * one visit on each child of the expanded root (az_mcts_select_root +
 * evaluator + az_mcts_expand_root first), so that az_play_commit with
 * temperature 1 and sampling draws the move uniformly and the replay row
 * records moves_prob = 1 / num_moves.  Used to fill the replay buffer before
 * training (policy_trainer.py:145-158). */
int az_mcts_root_uniform(az_engine *e, void *stream);

/* SearchTree.move, search_tree.py:115-132: re-root to child move_id (with
 * subtree compaction) or reset when it is unevaluated; move_id -1 = skip. */
int az_tree_move(az_engine *e, const int32_t *move_ids_dev, void *stream);
/* per-game AZ_ST_* bits */
int az_status(az_engine *e, int32_t *status_dev, void *stream);

/* Deterministic stub evaluator on the device (TEST / BENCH aid; the same
 * arithmetic as oracle/azalea_oracle.c:ostub_eval): fills AZ_BUF_VALUE and
 * AZ_BUF_PRIOR (AZ_PRIOR_PROBS layout) for the current leaves. */
int az_stub_eval(az_engine *e, int mode, void *stream);

/* ------------------------------------------------------- trainer feed */

/* prep.torch_batch_replays (prep.py:24-39) on device-resident replay rows:
 * for each of `count` row indices writes board int32[count][n*n], legal_moves
 * int32[count][n*n] (ascending, 0-padded), moves_prob f32[count][n*n]
 * (= as_distribution(visits, temperature), search_tree.py:327-344), reward
 * f32, colour int64 (0/1), result int64 (0: recorded before the move),
 * num_moves int32 (so the caller can trim the padding to the batch maximum
 * like prep.pad, prep.py:70-86). */
int az_replay_collate(const uint8_t *rows_dev, int row_bytes,
                      const int64_t *index_dev, int count, int board_size,
                      int32_t *board_dev, int32_t *moves_dev, float *probs_dev,
                      float *reward_dev, int64_t *color_dev, int64_t *result_dev,
                      int32_t *num_moves_dev, void *stream);

/* random_reflect for training samples: rotates the rows i of a collated batch
 * whose coins_dev[i] (uint8) is non-zero by 180 degrees, in place.  board
 * int32[count][n*n]; legal_moves int32 and moves_prob f32 rows of `ld`
 * elements, of which the first `width` hold the ascending, zero-padded moves
 * and their probabilities: the k non-zero moves m become n*n+1-m and, like
 * their probabilities, are reversed, so the list stays ascending; padding
 * stays zero.  Applying it twice with the same coins is the identity. */
int az_batch_reflect(int32_t *board_dev, int32_t *moves_dev, float *probs_dev,
                     const uint8_t *coins_dev, int count, int board_size, int width,
                     int ld, void *stream);

/* ------------------------------------------------------- evaluator glue */

/* HexNetwork input stage (network.py:138-142 + :71): Embedding(3,4) ->
 * conv3x3(4 -> channels) -> BatchNorm -> ReLU as one table lookup kernel.
 * cells int8 [num_boards][cell_stride] (network-view 0/1/2, what
 * az_mcts_select wrote), table bf16 [9][4][channels] = conv weights x
 * embedding with BN folded (row 3 of each tap = zeros = off board), bias
 * f32 [channels]; out bf16 [num_boards][n*n][channels] (NHWC). */
int az_nn_stem(const int8_t *cells_dev, int cell_stride, int board_size,
               int64_t num_boards, const void *table_dev, const float *bias_dev,
               void *out_dev, int channels, int padded_layout, void *stream);
/* Both 1x1 head convolutions + BN + ReLU (network.py:75-76,82-83) in one
 * pass: x bf16 [positions][channels] (NHWC), w f32 [heads][channels], b f32
 * [heads] -> out bf16 [positions][heads]; heads = 6 (2 value + 4 policy).
 * out_board_stride (slab layout only, else 0): elements between the rows of
 * two consecutive boards in out, >= n*n*heads and even (0 = dense) -- lets the
 * caller pad the row to a GEMM-friendly K; the padding is not written. */
int az_nn_heads(const void *x_dev, int64_t positions, const float *w_dev,
                const float *b_dev, void *out_dev, int64_t out_board_stride,
                int channels, int heads, int padded_board_size, void *stream);

/* Everything after the merged fully connected GEMM (network.py:78-80,145): y
 * bf16 [num_boards][ld] holds, WITHOUT bias, the value_fc2 pre-activations in
 * columns [0, nfc2) and the move_fc logits over tiles in [nfc2, nfc2 + n*n);
 * fc_bias f32 [>= nfc2 + n*n], w3 f32 [nfc2] and b3 f32 [1] = value_fc3.
 * value[b * value_stride] = tanh(w3 . relu(y[:nfc2] + bias) + b3) and
 * logits[b * logits_stride + tile] = y + bias, both fp32 and both nullable --
 * pass the engine's AZ_BUF_VALUE / AZ_BUF_PRIOR rows to hand the evaluation to
 * az_mcts_expand_backup(.., AZ_PRIOR_LOGITS) without any copy. */
int az_nn_tail(const void *y_dev, int64_t num_boards, int ld, int nfc2,
               int board_size, const float *fc_bias_dev, const float *w3_dev,
               const float *b3_dev, float *value_dev, int64_t value_stride,
               float *logits_dev, int64_t logits_stride, void *stream);

/* One tower convolution (Resblock.conv1/conv2 + BatchNorm + ReLU, with the
 * residual add for conv2; network.py:17-39) as a tcgen05 implicit GEMM, 64 ->
 * 64 channels (csrc/az_tower.cuh).  Activations use the tower's slab layout:
 * bf16 rows of 64 channels; one 128-row slab holds board row y of bpg =
 * az_nn_tower_group(n) = 128 / (n+1) boards:
 *     row = 8 + 128 * ((board / bpg) * n + y) + (board % bpg) * (n+1) + x
 * with one zero pad cell per board row (x == n), zero rows elsewhere, and
 * 16-byte chunk j of row R stored at chunk j ^ (R & 7).  A buffer holds az_nn_tower_rows(n, boards) rows; everything
 * that is not a real cell must be zero (the kernels keep it zero).
 * padded_layout = 1 makes az_nn_stem write this layout, padded_board_size = n
 * makes az_nn_heads read it.  w: bf16 [3 kx][3 ky][64 c_out][64 c_in] with the
 * same chunk swizzle (by c_out), bias f32 [64], resid (nullable) in the
 * activation layout (out may alias resid). */
int az_nn_tower_group(int board_size);
int az_nn_tower_halo(int board_size);     /* zero rows in front of the first slab (8) */
int64_t az_nn_tower_rows(int board_size, int64_t num_boards);   /* rows a buffer must hold */
int az_nn_conv3x3(const void *x_dev, const void *w_dev, const float *bias_dev,
                  const void *resid_dev, void *out_dev, int board_size,
                  int64_t num_boards, void *stream);

/* One whole residual block (network.py:17-39: conv1 + BN + ReLU, conv2 + BN,
 * + x, ReLU) in ONE launch and in place, x <- relu(conv2(relu(conv1(x))) + x),
 * reading the activations once and writing them once (csrc/az_block.cuh: a
 * cluster of two CTAs, conv1 on one SM streaming its output slabs through
 * distributed shared memory into conv2 on the other).  x: slab layout as for
 * az_nn_conv3x3; w: the two layers' packed weights back to back
 * [2][3 kx][3 ky][64][64] bf16; bias f32 [2][64]; scratch: unused, may be
 * NULL (the intermediate slabs travel through distributed shared memory;
 * az_nn_resblock_scratch_bytes() returns 0).
 * Bit-identical to az_nn_conv3x3(x, w1, b1, NULL, y) followed by
 * az_nn_conv3x3(y, w2, b2, x, x). */
size_t az_nn_resblock_scratch_bytes(void);
int az_nn_resblock(void *x_dev, const void *w_dev, const float *bias_dev,
                   void *scratch_dev, int board_size, int64_t num_boards,
                   void *stream);
/* The residual tower (network.py:73: nn.Sequential of num_blocks Resblocks):
 * num_blocks blocks applied one after the other, chained inside one launch
 * (eight per launch at most, then the next launch).  Every cluster owns a
 * range of board groups and runs block b + 1 over it as soon as it has
 * finished block b there -- a board's activations depend on no other board --
 * so the two-CTA pipeline is filled and drained once per launch, not once per
 * block; only the weights are exchanged in between.  w: [num_blocks][2]
 * packed layers, bias f32 [num_blocks][2][64].  Bit-identical to num_blocks
 * az_nn_resblock calls. */
int az_nn_resblocks(void *x_dev, const void *w_dev, const float *bias_dev,
                    void *scratch_dev, int board_size, int64_t num_boards,
                    int num_blocks, void *stream);
/* The same four evaluator stages over a batch whose size is only known on the
 * device (AZ_CFG_PACK_LEAVES): num_boards is the capacity the grids are sized
 * for, *live_rows_dev (int32, device; NULL = num_boards) the number of leading
 * rows that hold boards when the kernel runs.  Slab layout only.  The stem
 * writes the groups the live rows occupy whole (rows past the count as empty
 * boards), the tower and the heads run over those groups, the tail writes
 * value / logits of the live rows; nothing else is touched. */
int az_nn_stem_live(const int8_t *cells_dev, int cell_stride, int board_size,
                    int64_t num_boards, const void *table_dev, const float *bias_dev,
                    void *out_dev, int channels, int padded_layout,
                    const int32_t *live_rows_dev, void *stream);
int az_nn_resblocks_live(void *x_dev, const void *w_dev, const float *bias_dev,
                         void *scratch_dev, int board_size, int64_t num_boards,
                         int num_blocks, const int32_t *live_rows_dev, void *stream);
int az_nn_heads_live(const void *x_dev, int64_t positions, const float *w_dev,
                     const float *b_dev, void *out_dev, int64_t out_board_stride,
                     int channels, int heads, int padded_board_size,
                     const int32_t *live_rows_dev, void *stream);
int az_nn_tail_live(const void *y_dev, int64_t num_boards, int ld, int nfc2,
                    int board_size, const float *fc_bias_dev, const float *w3_dev,
                    const float *b3_dev, float *value_dev, int64_t value_stride,
                    float *logits_dev, int64_t logits_stride,
                    const int32_t *live_rows_dev, void *stream);
/* Diagnostic: how many two-CTA clusters az_nn_resblock sizes its grid for on
 * the current device (cudaOccupancyMaxActiveClusters; 74 on a B200), 0 before
 * the first launch. */
int az_nn_resblock_clusters(void);

/* Test aid for the root exploration noise (mcts.py:126-131), which only has
 * statistical parity with RandomState.dirichlet: writes the Dirichlet(alpha)
 * vector over k children that game g would draw for simulation `sim` of its
 * current ply into out_dev f32[G][k]. */
int az_noise_sample(az_engine *e, float alpha, int k, int sim, float *out_dev,
                    void *stream);

/* --------------------------------------------------------- lockstep play */

typedef struct az_play_params {
    float temperature;          /* exploration_temperature, policy.py:142-149 */
    int32_t exploration_depth;  /* temperature 0 from this ply on */
    int32_t move_sampling;      /* settings['move_sampling'] */
    int32_t collect_replay;     /* play_game collect_data, play_game.py:90-96 */
    int32_t auto_reset;         /* start a new game in a finished slot */
} az_play_params;

/* Policy.choose_action's tail + AzaleaAgent.execute_action + play_game's
 * bookkeeping for every game at once (policy.py:160-176,
 * azalea_agent.py:60-64, play_game.py:46-67): draw the move from the root
 * visit distribution (device Philox stream per game), record the replay row,
 * step the game, re-root the tree; finished games get their rewards, are
 * flushed to the replay buffer and (auto_reset) restarted.
 * chosen_dev (nullable) int32[G][4]: move, move_id, result, ply. */
int az_play_commit(az_engine *e, const az_play_params *p, int32_t *chosen_dev,
                   void *stream);
/* Reset the replay append counter after the host has harvested the rows. */
int az_replay_clear(az_engine *e, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* AZALEA_B200_H */
