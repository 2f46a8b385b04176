// az_tree.cuh -- device-resident PUCT trees: memory layout shared by az_tree.cu (kernels)
// and az_pool.cu (host runtime).  Internal.
//
// One tree per game, one fixed-stride slot per node (no allocator metadata on the hot path).
//
// The reference's select_action (self_play_client.cpp:333-366) scores every legal move of a node on every visit.
// A move WITHOUT an edge scores fl(sqrt(1+N) * P) + 0 (:313-315,322), which is monotone in P, so among those moves only
// the one with the largest prior can win (exactly equal priors: the one that comes last in the reference's
// unordered_map iteration order).  A node therefore keeps
//   * a dense list of the moves that HAVE an edge, in order of creation ("entries": prior, total score, visits,
//     child), and
//   * one CANDIDATE among the others (its movegen index and prior) plus the next smaller prior value -- the latter
//     only to detect the rare case of two different priors rounding to the same product, which a full scan resolves.
// A descent touches the header and the k entries of a node, not its L moves: for the deep nodes of a tree (k of a
// handful, L around 50) that is one or two 128-byte lines instead of ~20, and the hot part of all trees fits the L2.
// oracle/tree_model.c restates this algorithm on the CPU and tests/test_tree_model.py checks it against the
// reference-order search (exact ties, re-rooting, adversarial priors).
//
//   node slot (kNodeStride bytes, 128-B aligned):
//     [   0,   64)  NodeHdr
//     [  64, 6184)  Entry[255]  24 B each: P f64, W f64 (edge_total_score :283), n u32 (edge_visits :282, bits 0..22;
//                               bits 23..31: how many entries the CHILD had when this edge was last extended below --
//                               a load hint), child u32 (node index bits 0..23, movegen index of the move bits 24..31)
//     [6208, 8256)  P[256]      f64  prior of every move in movegen order (:151 posterior)
//     [8256, 8768)  move[256]   u16  from | to<<8, reference movegen order (cpp/movegen.cpp:16-66)
//     [8768, 9024)  rank[256]   u8   position of the move in the reference's hash-map iteration order (select_action's
//                                    `>=` tie-break walks that order, :345-358); filled in lazily, the first time a
//                                    node actually sees an exact tie
//     [9024, 9056)  visited     256-bit set: move i has an edge
//
// Dead subtrees are recycled lazily: re-rooting pushes the discarded siblings on a per-game stack;
// allocating a node pops one entry and pushes that node's children.  The pool therefore never holds
// more than (live nodes + 1) slots and is never compacted or copied.
#pragma once
#include "az_common.h"

namespace aztree {

constexpr int kNodeStride = 9088;
constexpr int kOffEntry = 64, kEntryBytes = 24, kMaxEntries = 255;
constexpr int kOffP = 6208, kOffMove = 8256, kOffRank = 8768, kOffVisited = 9024;
constexpr int kMaxPath = 1024;
constexpr uint32_t kVisitMask = 0x007fffffu;     // Entry::n: visit count (pool visits are capped at 2^22)
constexpr int kHintShift = 23;
constexpr uint32_t kChildMask = 0x00ffffffu;     // Entry::child: node index
constexpr int kMoveIdxShift = 24;
constexpr int kNoCand = 0xff;
constexpr int kRecWordsPerPly = 6 + 2 * 256;    // worst-case record words per ply

enum : uint32_t {
    NF_TERMINAL = 1u,
    NF_POPULATED = 2u,
    NF_RANKED = 4u,      // rank[] is valid for the node's current population
    NF_REPOPULATED = 8u  // the node became a root: the reference re-inserted its posterior into a clear()ed map (:489-490)
};
enum : int32_t { ST_IDLE = 0, ST_WAIT = 1, ST_DONE = 2, ST_STALL = 3, ST_ERROR = 4, ST_DESCEND = 5,
                 ST_PARK = 6 };  // arena: the partner tree's player is to move; this tree waits for its move in the mailbox
enum : int32_t { ERR_NODES = 1, ERR_PATH = 2, ERR_MOVES = 3, ERR_MAIL = 4 };

struct __align__(16) NodeHdr {
    uint64_t own, opp;       // pieces of the side to move / of the opponent
    double value;            // evals.value: from the side to move's point of view
    double cand_p;           // prior of the candidate (0 when there is none)
    double cand2_p;          // largest prior below cand_p among the moves without an edge; < 0: none
    int32_t N;               // all_edge_visits
    uint16_t n_moves;        // L; 0 for adjudicated (terminal) nodes
    uint8_t k;               // moves with an edge = entries in use
    uint8_t cand;            // movegen index of the candidate, kNoCand: every move has an edge
    uint8_t turn;            // absolute side to move: 0 = x, 1 = o
    uint8_t flags;
    uint16_t pad0;
    uint32_t pad[3];
};
static_assert(sizeof(NodeHdr) == 64, "node header is 64 bytes");

struct Entry {
    double P, W;
    uint32_t n, child;
};
static_assert(sizeof(Entry) == kEntryBytes, "entry is 24 bytes");

struct __align__(16) Game {
    int32_t status;
    int32_t root;
    int32_t pending;         // node awaiting an evaluation (ST_WAIT)
    int32_t path_len;
    int32_t n_alloc;         // bump pointer of never-used node slots
    int32_t gsp;             // garbage stack pointer
    int32_t ply;
    int32_t req_slot;
    uint64_t blockers;
    uint32_t rec_words;      // words written to the current record buffer
    int32_t rec_buf;         // 0/1
    int32_t rec_plies;
    uint32_t games_started;  // RNG stream selector
    int32_t rec_busy[2];     // record buffer handed to the host and not yet released
    int32_t error;
    int32_t start_turn;
    uint64_t start_own, start_opp;    // starting position of this slot (side to move / opponent)
    // statistics (summed by the host on demand)
    unsigned long long steps, evals, terminal_steps, positions, finished, skipped, max_depth;
    unsigned long long levels;        // tree levels walked by completed selections (sum of path lengths)
    int32_t random_ply;               // ONE_RANDOM_MOVE games (self_play_client.cpp:515-518): the ply that is played uniformly at random
    int32_t pad3;
};
static_assert(sizeof(Game) == 160, "Game records are 160 bytes");

// Search pools on the tensor-core net may evaluate SPECULATIVELY (az_pool_config::speculate, engine.py:387-392 queues the
// likely children of a new node the same way): every game owns a small set-associative cache of evaluations keyed by the
// exact position.  Expanding a move first looks its position up; the children with the largest priors of every node whose
// evaluation is consumed are requested in the same batch.  An evaluation is a pure function of the position, so a hit
// changes WHEN a leaf is linked, never what the search computes.
struct __align__(16) CacheTag {
    uint64_t own, opp;       // position: pieces of the side to move / of the opponent (blockers are fixed per game)
    uint32_t turn;           // absolute side to move
    uint32_t tick;           // tick in which the evaluation was requested: usable from the next tick on
    uint32_t valid;
    uint32_t pad;
};
constexpr int kCacheWays = 4;   // tags of one set share a 128-byte line

struct DoneEntry {
    int32_t game, buf, words, plies, result;
    int32_t random_ply;               // + 1; 0: the record has no "random_ply" key
    int32_t pad[2];
};

struct PoolDev {
    uint8_t *nodes;          // [G][C][kNodeStride]
    Game *games;             // [G]
    uint32_t *path;          // [G][kMaxPath]  node << 8 | entry
    uint32_t *gstack;        // [G][C]
    az_position *req_pos;    // [G]
    int32_t *req_game;       // [G]
    az_position *req_stage;  // [G] a game's request of this tick, by game index (internal net, no cache)
    uint64_t *req_mark;      // [G] tick_id << 1 | 0 (request deferred last tick) / 1 (new request); k_order_requests lays
                             // the marked requests of this tick out in req_pos in an order that does not depend on timing
    int32_t *req_count;      // [3 slots][2]: {requests, games that still have work but made no request} of a tick.  Ticks
                             // rotate through the slots (tick_slot); a tick reads its predecessor's request count (of which
                             // the first `cap` were evaluated) and zeroes its successor's slot, so the host never memsets.
                             // Arena pools: player B's half has its own [3][2] at req_count + 6.
    float *logits;           // [G][833]
    float *values;           // [G]
    uint32_t *records;       // [G][2][rec_cap_words]
    DoneEntry *done;         // [2G]
    int32_t *done_count;     // [1]
    int32_t G, C, visits, max_plies, noise, auto_play, steps_per_tick;
    int32_t levels_per_tick; // bound on tree levels a game may descend per tick (tail latency of deep endgame lines)
    int32_t cap;             // evaluations served per tick: a whole number of net-kernel rounds; later requests are re-queued
    int32_t consume;         // 1: evaluations of the previous requests are in logits/values; 0: top-up tick, leave waiting games alone
    int32_t tick_slot;       // slot of req_count this tick appends its requests to
    uint32_t rec_cap_words;
    uint64_t seed;
    // speculative evaluation (search pools; all null / 0 otherwise)
    CacheTag *cache_tag;     // [G][cache_entries]
    double *cache_exps;      // [G * cache_entries + 1][833]  softmax numerators of a cached evaluation (last entry: trash)
    double *cache_tot;       // [G * cache_entries + 1]       their sequential sum
    float *cache_val;        // [G * cache_entries + 1]       value head
    int32_t *req_out;        // [req_cap] cache entry (global index) every request of this tick is evaluated into
    int32_t cache_entries;   // per game, a power of two >= kCacheWays
    int32_t spec_k;          // children requested per consumed node
    int32_t req_cap;         // requests the net kernel serves per tick
    uint32_t tick_id;        // increments with every tick
    int32_t one_random_move; // the reference's compile-time ONE_RANDOM_MOVE variant of generate_game (self_play_client.cpp:24,515-552)
    int32_t prefetch;        // a level pulls the children of a node with at most this many edges into L2 while it selects
                             // (default 8, AZ_TREE_PREFETCH=0 switches it off)
    int32_t force_slow;      // test knob (AZ_TREE_FORCE_SLOW=1): resolve every candidate by the full scan
    unsigned long long *timed_evals;   // non-null: the previous tick's net launch was event-timed -- add the evaluations it served
    unsigned long long *prof;   // AZ_POOL_PROFILE=1: [G][8] clock cycles per phase of the last tick (debug aid, normally nullptr)
    // arena pools (az_arena_create; all null / 0 otherwise): G = 2S trees, [0, S) play for A, [S, 2S) for B, slot s pairs tree s
    // with tree s + S.  Each half orders its requests on its own (k_order_requests, one block per half) into req_pos[half * S ...]
    // and is evaluated by its own network; `cap` applies to each half.
    int32_t *arena_slot_game;   // [S] game index slot s plays; -1: no game left
    uint4 *mailbox;             // [G] posts to a tree from its partner: {tick of a game-over post, 0, tick of a move post, move};
                                // a post is read from the tick after the one that stamped it, and cleared by the reader
    const az_position *openings;// [n] game i starts from openings[i >> 1]; A moves first when i is even
    uint16_t *arena_moves;      // [2n][max_plies] the moves of every game
    int32_t *arena_plies;       // [2n]
    int32_t *arena_result;      // [2n] 1 x won, 2 o won, 0 max_plies reached
    int32_t *arena_counters;    // [0] next game index, [1] games finished, [2] trees that hit an error
    int32_t arena_games;        // 2n
    int32_t visits_b;           // visit target of B's trees (A's: visits)
};

}  // namespace aztree
