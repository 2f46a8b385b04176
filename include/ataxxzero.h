/*
 * ataxxzero.h -- C ABI of libataxxzero.so, the B200-native self-play hot path.
 *
 * Plain pointers and sizes only (no torch / C++ types).  Every entry point cites the
 * reference interface it replaces (file:line relative to petersn/AtaxxZero).  All
 * functions return AZ_OK (0) or a negative az_status; az_last_error() gives the text.
 * There is NO CPU fallback: without a usable sm_100 device every compute call fails
 * with AZ_ERR_CUDA.  "Host" pointers are ordinary (ideally pinned) host memory;
 * "dev" pointers are device memory on the context's GPU (e.g. torch tensor data_ptr()).
 */
#ifndef ATAXXZERO_H
#define ATAXXZERO_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    AZ_OK = 0,
    AZ_ERR_ARG = -1,        /* bad argument (null pointer, size, FEN, ...)           */
    AZ_ERR_CUDA = -2,       /* CUDA runtime / no device / kernel failure             */
    AZ_ERR_STATE = -3,      /* call made in the wrong state (e.g. no weights loaded) */
    AZ_ERR_CAPACITY = -4,   /* a device pool overflowed (node pool, record buffer)   */
    AZ_ERR_IO = -5          /* output file could not be opened / written             */
} az_status;

/* cpp/ataxx.hpp:28-34 `struct Position` -- identical layout (32 bytes).
 * bit sq = rank*7 + file, a1 = 0 ... g7 = 48; turn 0 = x (CROSS), 1 = o (NOUGHT). */
typedef struct {
    int32_t  ply;
    int32_t  turn;
    uint64_t blockers;
    uint64_t pieces[2];
} az_position;

/* cpp/move.hpp:9-31 `struct Move{int from,to}` packed as from | to<<8; a single (clone)
 * move has from == to (move.cpp:100-103); AZ_NO_MOVE mirrors NO_MOVE={50,50} (move.hpp:33). */
typedef uint16_t az_move;
#define AZ_MOVE(from, to)  ((az_move)((from) | ((to) << 8)))
#define AZ_MOVE_FROM(m)    ((int)((m) & 0xff))
#define AZ_MOVE_TO(m)      ((int)((m) >> 8))
#define AZ_NO_MOVE         AZ_MOVE(50, 50)
#define AZ_MAX_MOVES       256          /* movegen.cpp:69 asserts n < 256 */
#define AZ_FEATURES        196          /* [7][7][4]  index 28x+4y+c  (self_play_client.cpp:174-202) */
#define AZ_LOGITS          833          /* [7][7][17] index 119x+17y+p (self_play_client.cpp:224-237) */

typedef struct az_context az_context;

/* ---------------- context ---------------- */
const char *az_last_error(void);                       /* thread-local message of the last failure */
const char *az_version(void);
int az_create(int device, uint64_t seed, az_context **out);   /* replaces the process-global state of
                                                                  self_play_client.cpp:591-602 */
void az_destroy(az_context *ctx);
int az_device_count(void);
int az_sync(az_context *ctx);                          /* cudaStreamSynchronize on the context stream */
/* raw handle of the context's stream (cudaStream_t) so callers can record CUDA events on it */
void *az_stream(az_context *ctx);

/* ---------------- rules: host-side helpers (no GPU) ---------------- */
/* cpp/ataxx.cpp:14-92 set_board: same FEN grammar, "startpos", same return codes 0..8 */
int az_set_board(az_position *pos, const char *fen);
/* cpp/move.cpp:11-21 move_string: "b6" for singles, "a7b5" for doubles; returns length */
int az_move_string(az_move m, char out[5]);
/* inverse of move_string (cpp/makemove.cpp:22-54 parser); returns AZ_NO_MOVE on bad text */
az_move az_parse_move(const char *text);
/* fen text of a position (rows rank 7..1, '-' blockers); returns length */
int az_fen(const az_position *pos, char *out, size_t cap);

/* ---------------- rules: batched device kernels (host buffers in/out) ---------------- */
/* cpp/movegen.cpp:10-79 movegen over n positions.  moves is [n][AZ_MAX_MOVES]; order is the
 * reference's (doubles by from/to ascending, then singles by destination ascending). */
int az_movegen_batch(az_context *ctx, const az_position *pos, int n, az_move *moves, int32_t *counts);
/* cpp/makemove.cpp:56-76 makemove, one move per position, in place */
int az_makemove_batch(az_context *ctx, az_position *pos, const az_move *moves, int n);
/* cpp/self_play_client.cpp:109-144 get_board_result: 0 ongoing, 1 x wins, 2 o wins */
int az_result_batch(az_context *ctx, const az_position *pos, int n, int32_t *result);
/* cpp/self_play_client.cpp:174-202 feature planes, float [n][7][7][4] */
int az_features_batch(az_context *ctx, const az_position *pos, int n, float *features);
/* cpp/bitboards.cpp:6-39 whole-board dilations */
int az_jump_bb_batch(az_context *ctx, const uint64_t *bb, int n, uint64_t *single_out, uint64_t *double_out);

/* ---------------- perft (perft.py:5-26; reference C++ has only movegen+makemove) ------------- */
/* nodes[i] = number of leaf nodes at `depth` below pos[i] (a stuck side has 0 children) */
int az_perft_batch(az_context *ctx, const az_position *pos, int n, int depth, uint64_t *nodes);
int az_perft(az_context *ctx, const az_position *root, int depth, uint64_t *nodes);
/* device-resident variant: d_pos / d_nodes are device pointers; runs on the context stream */
int az_perft_batch_dev(az_context *ctx, const void *d_pos, int n, int depth, void *d_nodes);
/* statistics of the last perft call: device-side counted parents ("count nodes") and kernel launches */
int az_perft_last_stats(az_context *ctx, uint64_t *count_nodes, int32_t *launches, int32_t *frontier_items);

/* ---------------- random play (generate_games.py --random-play, generate_games.py:20-24,50-57) ------------- */
/* n_games uniformly random games from `start`, played on the device (one move drawn uniformly from the legal moves per
 * ply, Philox stream keyed by seed and game).  plies_out: n_games x max_plies records of 24 bytes {uint64 x, uint64 o
 * (pieces BEFORE the move), uint32 move = from | to << 8, uint32 0}; n_plies_out[g] plies were played; result_out[g] is
 * 1 / 2, or 0 when max_plies was reached first (the reference skips such games).  All outputs are host memory. */
int az_random_playouts(az_context *ctx, const az_position *start, int n_games, int max_plies, uint64_t seed, void *plies_out,
                       int32_t *n_plies_out, int32_t *result_out);

/* ---------------- network (model.py:38-79 forward; .npy weights model.py:179-196) ------------- */
/* Precision modes of the forward pass. */
#define AZ_NET_FP32   0   /* CUDA-core fp32, reference-accurate (<= 1e-5 vs the fp32/fp64 restatement) */
#define AZ_NET_BF16   1   /* bf16 tcgen05 tensor-core implicit GEMM, fp32 accumulate (<= 2e-2 abs at the scale of the
                             reference's initialisation; 8-bit mantissa: ~1.4 % rms of the logit scale for a trained net) */
#define AZ_NET_F16    3   /* the same kernel with IEEE-half operands (11-bit mantissa, same tensor throughput): <= 2e-2 abs
                             also for trained-scale logits; operands must stay below 65504 (batch-normalised towers do)  */

/* Upload weights.  `packed` is float32, host memory, in model.py parameter order:
 *   W_in[3][3][4][F], then 2*blocks x W[3][3][F][F]   (TF layout [kh(x)][kw(y)][Cin][Cout]),
 *   W_policy[F][17], W_value[F][1], fc_w[49], fc_b[1],
 *   then for each of the 1+2*blocks batch-norm layers: moving_mean[F], moving_variance[F].
 * Batch-norm is applied in inference form with gamma=1, beta=0, eps=1e-3 (model.py:120-124; gamma/beta
 * are never stored in the .npy, SURVEY App. B-5).  F must be 128 in this build. */
int az_net_load(az_context *ctx, const float *packed, size_t count, int filters, int blocks);
size_t az_net_param_count(int filters, int blocks);   /* expected `count` */

/* sess.run([policy_output, value_output], {input_ph: features}) of accelerated_generate_games.py:57-63 /
 * engine.py:184-190: features float32 [n][7][7][4] -> logits float32 [n][7][7][17], values float32 [n]. */
int az_net_forward(az_context *ctx, const float *features, int n, int mode, float *logits, float *values);
/* gpu_server.py:52-56 wire form: int8 features [n][196] (rpc_client.py:16-19) */
int az_net_forward_i8(az_context *ctx, const int8_t *features, int n, int mode, float *logits, float *values);
/* nn_evals.py:48-62 evaluate(board): mean policy (rotated back spatially; direction planes are NOT permuted, as in the
 * reference) and mean value over the 8 dihedral images of each position, all 8n images in one batch */
int az_net_forward_sym8(az_context *ctx, const float *features, int n, int mode, float *logits, float *values);
/* device-resident: d_features float32 [n][196]; d_logits [n][833]; d_values [n]; context stream, no sync */
int az_net_forward_dev(az_context *ctx, const void *d_features, int n, int mode, void *d_logits, void *d_values);
/* fused leaf encoding (self_play_client.cpp:174-202) + forward: d_pos is az_position[n] on the device */
int az_net_forward_pos_dev(az_context *ctx, const void *d_pos, int n, int mode, void *d_logits, void *d_values);

/* ---------------- search / self-play over a pool of device-resident trees ------------------ */
/* One pool = G concurrent games, one PUCT tree each, all state in HBM (replaces the 2*buffer_size
 * std::threads + per-thread MCTS objects of self_play_client.cpp:369-493,608-646). */
#define AZ_EVAL_EXTERNAL 2      /* evaluations are supplied by the caller (legacy contract / parity hook) */

typedef struct az_pool az_pool;

typedef struct {
    int32_t games;          /* G: concurrent games (accelerated_generate_games.py: 2*buffer_size threads)      */
    int32_t visits;         /* search until root.all_edge_visits >= visits (self_play_client.cpp:522)       */
    int32_t max_plies;      /* maximum_game_plies = 400 (self_play_client.cpp:34)                            */
    int32_t noise;          /* 1: Dirichlet(0.15) x 0.25 at every root (self_play_client.cpp:250-271)        */
    int32_t auto_play;      /* 1: self-play (sample move ~ visits, record, re-root, restart finished games);
                               0: search only (MCTS::step / MCTS::play driven by the caller)                 */
    int32_t eval_mode;      /* AZ_NET_FP32, AZ_NET_BF16 or AZ_EVAL_EXTERNAL                                   */
    int32_t node_capacity;  /* nodes per tree; 0 = visits + 64                                               */
    int32_t steps_per_tick; /* max MCTS steps a game may take per tick without needing the net; 0 = 8       */
    uint64_t seed;          /* Philox stream for move sampling and Dirichlet noise                           */
    char start_fen[64];     /* "" = STARTING_GAME_POSITION (self_play_client.cpp:23)                         */
    int32_t speculate;      /* search pools (auto_play = 0) on the tensor-core net: every time a node's evaluation is consumed,
                               the evaluations of its `speculate` highest-prior children are requested in the same batch and
                               kept in a per-game cache (engine.py:387-392 queues likely children the same way); a leaf whose
                               position is cached links without waiting for the net.  Visit counts are unchanged.  0 = off */
    int32_t one_random_move;/* self-play: the reference's compile-time ONE_RANDOM_MOVE variant of generate_game
                               (self_play_client.cpp:24,515-552): ply random_ply ~ U{0..119} is played uniformly at random, the plies
                               before it are sampled ~ visits, the plies after it take the most visited move; records carry
                               "random_ply" and games that end at or before that ply are skipped (:632-637).  0 = off (as shipped) */
    int32_t reserved[2];
} az_pool_config;

typedef struct {
    uint64_t ticks;            /* tree-kernel launches                                            */
    uint64_t steps;            /* MCTS::step() equivalents                                        */
    uint64_t evals;            /* leaf evaluations requested from the net                         */
    uint64_t terminal_steps;   /* steps that ended in an adjudicated leaf (no evaluation)         */
    uint64_t positions;        /* plies recorded (len(entry["moves"]) summed over all games)     */
    uint64_t games_finished;   /* games with result 1 or 2                                        */
    uint64_t games_skipped;    /* games that hit max_plies with result 0 (self_play_client.cpp:628-631) */
    uint64_t max_depth;        /* deepest selection path seen                                     */
    uint64_t kernel_launches;  /* kernels launched by the pool                                    */
    uint64_t record_bytes;     /* game-record bytes copied device -> host                         */
    double   net_seconds;      /* device time in the net kernel: CUDA events around every launch of the timed ticks, summed    */
    double   tree_seconds;     /* ... and in the tree kernel                                                                  */
    uint64_t levels;           /* tree levels walked by completed selections (sum of path lengths)                            */
    double   tick_seconds;     /* tree + net of every self-play tick                                                          */
    uint64_t timed_ticks;      /* ticks behind the three sums (az_selfplay_* only; az_pool_run does not time its ticks): the   */
                               /* events sit on contiguous windows, the first 256 ticks of every 1024                          */
    uint64_t timed_evals;      /* evaluations served by the net launches of those ticks (counted on the device)                */
} az_pool_stats;

int az_pool_create(az_context *ctx, const az_pool_config *cfg, az_pool **out);
void az_pool_destroy(az_pool *pool);
int az_pool_stats_get(az_pool *pool, az_pool_stats *out);

/* MCTS(thread_id, board, use_dirichlet_noise) ctor (self_play_client.cpp:375-384): reset tree `game` to `root` */
int az_pool_set_root(az_pool *pool, int game, const az_position *root);
/* the same for every tree at once: roots is az_position[cfg.games] (host memory) */
int az_pool_set_roots(az_pool *pool, const az_position *roots);
/* change the visit target of every tree (MCTSEngine.MAX_STEPS / VISITS style control); must fit node_capacity */
int az_pool_set_visits(az_pool *pool, int visits);
/* Advance every tree with the internal net until each has root visits >= cfg.visits (search mode) or
 * `max_ticks` ticks have run.  *idle_out = 1 when no tree needs more work. */
int az_pool_run(az_pool *pool, int max_ticks, int32_t *idle_out);
/* External evaluator (the legacy contract): advance trees until each is blocked on an evaluation or done;
 * writes float features [n][7][7][4] for the n pending requests (n <= games). */
int az_pool_collect(az_pool *pool, float *features, int32_t *n_requests);
/* ... and hand back logits [n][833] / values [n] in the same order (complete_workload semantics). */
int az_pool_provide(az_pool *pool, const float *logits, const float *values);
/* the same with the row count of the caller's arrays stated: AZ_ERR_ARG unless n_rows == the n of az_pool_collect */
int az_pool_provide_n(az_pool *pool, const float *logits, const float *values, int32_t n_rows);
/* root statistics in reference movegen order (visits[i] = edge_visits or 0 when no edge exists) */
int az_pool_root(az_pool *pool, int game, az_position *pos, int32_t *n_moves, az_move *moves, int32_t *visits,
                 double *total_score, double *prior, int32_t *root_visits, double *root_value);
/* engine.py:331-336 select_principal_variation(best=True): the most-visited line below the root, at most max_len plies */
int az_pool_pv(az_pool *pool, int game, az_move *moves, int32_t *visits, int max_len, int32_t *len_out);
/* MCTS::play(move) (self_play_client.cpp:475-492): re-root on the child (subtree kept) or rebuild */
int az_pool_play(az_pool *pool, int game, az_move move);

/* Self-play generation (generate_game + Worker::thread_main, self_play_client.cpp:508-645): runs until
 * `target_games` finished games have been appended to `output_path` as reference-format JSON lines,
 * `target_positions` plies were recorded or `max_seconds` passed (0 = no limit on that axis).  The lines are formatted and
 * written by a background thread while the kernels run; every record of a finished game is in the file when the call returns. */
int az_selfplay_run(az_pool *pool, const char *output_path, int64_t target_games, int64_t target_positions,
                    double max_seconds, az_pool_stats *stats_out);

/* Fixed amount of work instead of a target: exactly `ticks` (tree kernel + net kernel) iterations.  With
 * output_path = NULL finished games are recycled on the device and their records are not copied out. */
int az_selfplay_ticks(az_pool *pool, const char *output_path, int64_t ticks, az_pool_stats *stats_out);

/* ---------------- arena: two networks play each other on the device ------------------ */
/* An arena pool holds 2*slots search trees: trees [0, slots) search for player A, trees [slots, 2*slots) for player B, and slot s
 * plays one game at a time between tree s and tree s + slots.  Only the tree whose player is to move searches (no noise, no
 * sampling); at its player's visit target it plays the most visited root edge (first created on equal counts: az_pool_pv,
 * engine.py:331-336 best=True) and both trees re-root on the move (az_pool_play).  A free slot takes the next game index. */
typedef struct {
    int32_t slots;          /* concurrent games; the pool holds 2*slots trees                                       */
    int32_t visits[2];      /* visit target per move of player A / player B (1 .. 2^22)                              */
    int32_t max_plies;      /* a game ends with result 0 when its ply count (from the opening) reaches it; 0 = 400   */
    int32_t eval_mode;      /* AZ_NET_FP32 / AZ_NET_BF16 / AZ_NET_F16, both players                                  */
    int32_t node_capacity;  /* nodes per tree; 0 = max(visits) + 64                                                  */
    int32_t reserved[2];
} az_arena_config;
/* Player A is evaluated with the network loaded in ctx_a, player B with the one in ctx_b (same device; ctx_b may be
 * ctx_a).  Every kernel runs on ctx_a's stream.  az_pool_destroy and az_pool_stats_get work on the pool; az_pool_run and
 * az_selfplay_* refuse it (AZ_ERR_STATE). */
int az_arena_create(az_context *ctx_a, az_context *ctx_b, const az_arena_config *cfg, az_pool **out);
/* Plays the 2*n games of n openings (host az_position[n], none already decided) to the end: game i starts from opening i >> 1,
 * A moves first in the even games and B in the odd ones.  Outputs are host arrays indexed by game: moves [2n][max_plies]
 * (az_move; the first plies[i] entries of row i are the game, the rest 0), plies [2n], result [2n] (1 x won, 2 o won, 0
 * max_plies reached).  stats_out may be NULL.  AZ_ERR_STATE on a pool that az_arena_create did not make. */
int az_arena_play(az_pool *pool, const az_position *openings, int n, az_move *moves, int32_t *plies, int32_t *result,
                  az_pool_stats *stats_out);

/* ---------------- training-sample extraction (train.py:43-77 get_sample_from_entries) ---------------- */
/* A minibatch of (features, policy target, value target) triples straight from ply records.
 *   plies:   table of ply records, uint32 words each: [0,1] x bitboard, [2,3] o bitboard, [4] played move | entries<<16,
 *            [5] N = sum of visit counts (0: pair values are float32 probabilities), then `entries` pairs (move, count|prob)
 *            -- the binary layout the self-play kernels record, or the same packed from JSON game files;
 *   offsets: word offset of each sample's ply record;   meta: bit 0 side to move (0 = x), bits 1-2 game result (1|2),
 *            bits 3-5 dihedral symmetry index (train.py:11-23), bit 6: 1 = use the visit distribution ("dists"),
 *            0 = one-hot on the played move (records without "dists", train.py:62-63).
 * Outputs: features int8 [n][7][7][4] (engine.board_to_features; plane 3 is 0, SURVEY App. B-1), policy float32
 * [n][7][7][17], value float32 [n] (+1 when the side to move won, else -1). */
int az_samples_extract(az_context *ctx, const uint32_t *plies, size_t ply_words, const uint64_t *offsets, const uint32_t *meta, int n,
                       int8_t *features, float *policy, float *value);
/* device-resident variant (all pointers on the context's GPU; runs on the context stream, no sync, no validation) */
int az_samples_extract_dev(az_context *ctx, const void *d_plies, const void *d_offsets, const void *d_meta, int n, void *d_features,
                           void *d_policy, void *d_value);

/* ---------------- training step (model.py:81-101 build_training, model.py:116-142 train / run_on_samples) ---------------- */
/* One optimisation step of the reference's network on the GPU: conv tower with batch-norm in TRAINING mode (batch
 * statistics, moving averages updated with decay 0.99), softmax cross-entropy on the 833 policy logits (mean over the
 * batch) + mean squared value error + 1e-4 * l2_loss of every trainable variable, MomentumOptimizer(lr, 0.9).
 * bf16 tensor-core operands, fp32 accumulation / master weights / momentum.  128 filters; any block count. */
typedef struct az_trainer az_trainer;
int az_trainer_create(az_context *ctx, int max_batch, int blocks, az_trainer **out);
void az_trainer_destroy(az_trainer *trainer);
/* `packed`: the vector az_net_load takes.  Like a fresh train.py process (train.py:112-120) the batch-norm gamma / beta
 * start at 1 / 0 and the momentum accumulators at 0. */
int az_trainer_load(az_trainer *trainer, const float *packed, size_t count);
/* network.train(minibatch, learning_rate) (train.py:154-155).  features int8 [n][7][7][4], policies float [n][7][7][17],
 * values float [n] -- az_samples_extract's outputs; 2 <= n <= max_batch.  losses (optional) = {policy, value,
 * regularisation} of this minibatch before the update. */
int az_trainer_step(az_trainer *trainer, const int8_t *features, const float *policies, const float *values, int n, float learning_rate,
                    float *losses);
/* The games of a training run as az_samples_extract's binary ply table, uploaded once and kept on the device (train.py:105-110
 * loads its games once); az_trainer_step_picks then runs one step on the samples (offsets, meta) -- az_samples_extract's sample
 * description, get_sample_from_entries (train.py:43-77) -- with no host round trip: the extraction kernel writes the minibatch
 * straight into the trainer's input buffers. */
int az_trainer_set_games(az_trainer *trainer, const uint32_t *plies, size_t ply_words);
int az_trainer_step_picks(az_trainer *trainer, const uint64_t *offsets, const uint32_t *meta, int n, float learning_rate, float *losses);
/* run_on_samples(policy_loss.eval / value_loss.eval) (train.py:141-142): is_training = False (moving statistics), any n.
 * losses = {policy, value}; logits [n][833] and values_out [n] are optional (NULL to skip). */
int az_trainer_eval(az_trainer *trainer, const int8_t *features, const float *policies, const float *values, int n, float *losses, float *logits,
                    float *values_out);
/* model.save_model (model.py:173-183): weights + moving statistics back in az_net_load's order (gamma / beta are not part
 * of the file format) */
int az_trainer_export(az_trainer *trainer, float *packed, size_t count);
unsigned long long az_trainer_launches(const az_trainer *trainer);
/* device time of the last step's kernels, CUDA events on the launching stream (the minibatch already in HBM) */
float az_trainer_last_step_ms(const az_trainer *trainer);
/* test hook: an internal tensor of the last step ("z", "act", "d_h", "grad_conv", "grad_gamma", "grad_beta", "gamma", "beta",
 * "conv", "moving", "grad_heads"), see az_train.cu */
int az_trainer_debug_read(az_trainer *trainer, const char *what, int layer, int n, float *out, size_t count);

/* ---------------- legacy 4-function ABI (link.py:8-32; self_play_client.cpp:683,708,723,740) -------- */
/* Same names, arguments and blocking behaviour.  The trees live on GPU 0 (or $AZ_DEVICE); the caller is
 * the evaluator: get_workload() fills fill_buffer{1,2} with `buffer_entries` feature planes and returns the
 * buffer index, complete_workload() takes the matching logits/values.  buffer_entries <= thread_count <= 2*buffer_entries
 * (self_play_client.cpp:683-706 accepts any count up to 2*entries and needs `entries` workers to ever fill a buffer); with
 * fewer than 2*buffer_entries threads only one workload can be outstanding at a time, as in the reference. */
void launch_threads(char *output_path, int visits, float *fill_buffer1, float *fill_buffer2, int buffer_entries,
                    int thread_count);
int get_workload(void);
void complete_workload(int workload, float *posteriors, float *values);
void shutdown(void);

#ifdef __cplusplus
}
#endif
#endif
