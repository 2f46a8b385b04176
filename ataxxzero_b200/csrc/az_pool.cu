// az_pool.cu -- host runtime of the device-resident game pool: allocation, the tick loop
// (tree kernel <-> net kernel, no host round trip per evaluation), external-evaluator stepping,
// reference-format JSON game records, arena pools (two networks playing each other), and the legacy 4-function ABI of link.py.
//
// Replaces the thread pool / double-buffered request queue of cpp/self_play_client.cpp:588-749 and
// the Python feed loop of accelerated_generate_games.py:54-83.
#include "az_net.h"
#include "az_rules.cuh"
#include "az_tree.cuh"

#include <algorithm>
#include <condition_variable>
#include <deque>
#include <mutex>
#include <thread>
#include <charconv>
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <map>

using namespace aztree;

void aztree_launch_tick(const PoolDev &P, cudaStream_t s);
void aztree_launch_init_all(const PoolDev &P, const az_position &pos, cudaStream_t s);
void aztree_launch_set_root(const PoolDev &P, int g, const az_position &pos, cudaStream_t s);
void aztree_launch_set_roots(const PoolDev &P, const az_position *d_pos, cudaStream_t s);
void aztree_launch_play(const PoolDev &P, int g, int move, int *d_status, cudaStream_t s);
void aztree_launch_arena_start(const PoolDev &P, cudaStream_t s);
void aztree_launch_release(const PoolDev &P, const DoneEntry *d_done, int n, cudaStream_t s);
void aztree_launch_features(const az_position *d_pos, int n, float *d_out, cudaStream_t s);
void aztree_launch_gather(const PoolDev &P, const DoneEntry *d_done, const uint32_t *d_offsets, int n, uint32_t *d_out, cudaStream_t s);
void aztree_launch_debug_gamma(double alpha, uint64_t seed, int n, double *d_out, cudaStream_t s);
void aztree_launch_debug_exp(const float *d_x, int n, double *d_out, cudaStream_t s);
void aztree_launch_debug_div(const double *d_in, int n, int puct, double *d_out, cudaStream_t s);
void aztree_launch_debug_sample(const int32_t *d_visits, int L, int N, uint64_t seed, int n, int32_t *d_out, cudaStream_t s);

const int kTicksPerDrain = 32;
const int kEventPeriod = 1024, kEventWindow = 256;    // CUDA events on the first 256 ticks of every 1024 (run_ticks)

// Finished games leave the device as packed binary records; turning them into the reference's JSON lines (sorted-key
// objects, one std::map per ply) costs the host ~0.3 ms per game.  A writer thread does that, so the thread that launches
// kernels goes straight back to launching.  flush() returns once every queued record is in the file (and reports a write
// error); the entry points call it before they return or close the file.
struct RecordJob {
    FILE *out = nullptr;
    std::vector<uint32_t> words;          // the drained records, back to back
    std::vector<DoneEntry> done;
    std::vector<uint32_t> offsets;        // word offset of every record in `words`
};
struct RecordWriter {
    std::thread worker;
    std::mutex m;
    std::condition_variable cv, idle_cv;
    std::deque<RecordJob> jobs;
    bool busy = false, stop = false, failed = false;
    void push(RecordJob &&job);
    bool flush();                         // false: a write failed since the last flush
    void shutdown();
    void run();
};

// Every kernel and copy of a pool runs on the context stream.
struct az_pool {
    az_context *ctx = nullptr;
    az_context *ctx_b = nullptr;          // arena pools: the context whose network plays for B (trees [S, 2S)); null otherwise
    RecordWriter writer;
    az_pool_config cfg{};
    PoolDev dev{};
    int slot = 0;                         // req_count slot of the last tick
    int32_t *d_status = nullptr;
    float *d_features = nullptr;          // external mode: [G][196]
    DoneEntry *d_done_snapshot = nullptr; // copy of the done queue being drained
    uint32_t *d_offsets = nullptr;        // [2G] word offset of every drained record in d_stage
    uint32_t *d_stage = nullptr;          // finished records packed back to back (k_gather_records)
    size_t stage_words = 0;
    // pinned host mirrors
    int32_t *h_counts = nullptr;          // [0] req_count, [1] busy_count, [2] status, [3] done_count
    DoneEntry *h_done = nullptr;          // [2G]
    uint32_t *h_offsets = nullptr;        // [2G]
    uint32_t *h_stage = nullptr;          // [stage_words]
    std::vector<Game> h_games;
    // CUDA events around the tree and the net kernel of EVERY tick between two drains: tree_seconds / net_seconds are sums
    // of measured launches, not extrapolations
    // Two sets, used alternately: the set of the batch that just ran is read out AFTER the next batch has been launched,
    // so the ~100 cudaEventElapsedTime calls never sit between two batches with the GPU idle.
    std::vector<cudaEvent_t> ev[2];       // [1 + 2 * kTicksPerDrain] each
    int ev_ticks[2] = {0, 0};             // ticks recorded in the set and not yet read out
    int ev_cur = 0;
    unsigned long long *d_timed_evals = nullptr;      // evaluations served by the event-timed net launches (counted on the device)
    int pending_requests = 0;             // external mode: requests handed out by collect()
    uint64_t ticks = 0, launches = 0;
    double net_seconds = 0.0, tree_seconds = 0.0;     // sums over every launch of the self-play loop (CUDA events)
    double tick_seconds = 0.0;                        // every tick, first event to last
    uint64_t timed_ticks = 0;                         // ticks behind the three sums
    uint64_t timed_evals_host = 0;                    // evaluations of the timed launches that closed a batch (counted after its sync)
    uint64_t written_games = 0, written_positions = 0, d2h_bytes = 0;

    int G() const { return cfg.games; }
};

namespace {

void read_events(az_pool *pool, int set);

template <typename T>
int dev_alloc(T **p, size_t count, bool zero = true)
{
    AZ_CUDA(cudaMalloc(p, sizeof(T) * count));
    if (zero) AZ_CUDA(cudaMemset(*p, 0, sizeof(T) * count));
    return AZ_OK;
}

const char *kErrNames[] = {"", "node pool exhausted", "selection path longer than 1024 plies", ">= 256 legal moves",
                           "arena: the partner's move is not legal at this tree's root"};

int check_game_errors(az_pool *pool)
{
    // called after a sync: any game in ST_ERROR turns into AZ_ERR_CAPACITY
    AZ_CUDA(cudaMemcpy(pool->h_games.data(), pool->dev.games, sizeof(Game) * pool->dev.G, cudaMemcpyDeviceToHost));
    for (int g = 0; g < pool->dev.G; ++g)
        if (pool->h_games[g].status == ST_ERROR)
            return az_fail(AZ_ERR_CAPACITY, "game %d: %s", g, kErrNames[std::min(std::max(pool->h_games[g].error, 0), 4)]);
    return AZ_OK;
}

// ---- one tick: (previous evaluations ->) tree kernel -> requests ----
int launch_tree(az_pool *pool, bool consume = true)
{
    cudaStream_t s = pool->ctx->stream;
    if (consume) pool->slot = (pool->slot + 1) % 3;      // the kernel itself zeroes the slot after this one
    else AZ_CUDA(cudaMemsetAsync(pool->dev.req_count + 2 * pool->slot + 1, 0, sizeof(int32_t), s));   // top-up: same slot, fresh busy count
    pool->dev.consume = consume ? 1 : 0;
    pool->dev.tick_slot = pool->slot;
    pool->dev.tick_id++;
    aztree_launch_tick(pool->dev, s);
    const int kernels = pool->dev.cache_tag ? 1 : 2;      // + k_order_requests
    pool->launches += kernels;
    pool->ctx->launches += kernels;
    AZ_CUDA(cudaGetLastError());
    return AZ_OK;
}

int launch_net(az_pool *pool)
{
    const PoolDev &D = pool->dev;
    int rc;
    if (pool->ctx_b) {    // arena: each player's half of the requests with that player's network, both on the pool's stream
        const int S = D.G / 2;
        rc = az_net_forward_internal(pool->ctx, D.req_pos, AZ_IN_POS, D.cap, pool->cfg.eval_mode, D.logits, D.values,
                                     D.req_count + 2 * pool->slot, pool->ctx->stream);
        if (rc == AZ_OK)
            rc = az_net_forward_internal(pool->ctx_b, D.req_pos + S, AZ_IN_POS, D.cap, pool->cfg.eval_mode, D.logits + (size_t)S * AZ_LOGITS,
                                         D.values + S, D.req_count + 6 + 2 * pool->slot, pool->ctx->stream);
        pool->launches += 2;
        return rc;
    }
    if (D.cache_tag)      // speculative search pool: every evaluation of the batch lands in its cache entry
        rc = az_net_forward_internal(pool->ctx, D.req_pos, AZ_IN_POS, D.req_cap, pool->cfg.eval_mode, nullptr, D.cache_val,
                                     D.req_count + 2 * pool->slot, pool->ctx->stream, D.cache_exps, D.cache_tot, D.req_out);
    else
        rc = az_net_forward_internal(pool->ctx, D.req_pos, AZ_IN_POS, D.cap, pool->cfg.eval_mode, D.logits, D.values,
                                     D.req_count + 2 * pool->slot, pool->ctx->stream);
    pool->launches++;
    return rc;
}

// ---- JSON (nlohmann::json::dump() conventions: no spaces, keys sorted, shortest round-trip doubles) ----
void append_double(std::string &out, double v)
{
    char buf[40];
    auto r = std::to_chars(buf, buf + sizeof(buf), v);
    std::string s(buf, r.ptr);
    if (s.find_first_of(".en") == std::string::npos) s += ".0";     // 1 -> 1.0, like nlohmann
    out += s;
}

std::string record_to_json(const uint32_t *rec, int words, int plies, int result, int random_ply_plus_1 = 0)
{
    std::string boards = "[", dists = "[", moves = "[";
    int w = 0;
    char mvbuf[8];
    for (int p = 0; p < plies && w < words; ++p) {
        const uint64_t x = (uint64_t)rec[w] | ((uint64_t)rec[w + 1] << 32), o = (uint64_t)rec[w + 2] | ((uint64_t)rec[w + 3] << 32);
        const az_move mv = (az_move)(rec[w + 4] & 0xffff);
        const int entries = (int)(rec[w + 4] >> 16);
        const double total = (double)rec[w + 5];
        if (p) { boards += ","; dists += ","; moves += ","; }
        boards += "[";
        for (int y = 0; y < 7; ++y)                                  // serialize_board_for_json (:88-107): top row first
            for (int xx = 0; xx < 7; ++xx) {
                const uint64_t bit = 1ULL << (xx + 7 * (6 - y));
                if (y || xx) boards += ",";
                boards += (x & bit) ? "1" : (o & bit) ? "2" : "0";
            }
        boards += "]";
        az_move_string(mv, mvbuf);
        moves += "\"";
        moves += mvbuf;
        moves += "\"";
        std::map<std::string, double> dist;                           // nlohmann objects are std::map: keys sorted
        for (int e = 0; e < entries; ++e) {
            az_move_string((az_move)(rec[w + 6 + 2 * e] & 0xffff), mvbuf);
            dist[mvbuf] = (double)rec[w + 7 + 2 * e] / total;
        }
        dists += "{";
        bool first = true;
        for (auto &kv : dist) {
            if (!first) dists += ",";
            first = false;
            dists += "\"" + kv.first + "\":";
            append_double(dists, kv.second);
        }
        dists += "}";
        w += 6 + 2 * entries;
    }
    const std::string random_ply = random_ply_plus_1 > 0 ? ",\"random_ply\":" + std::to_string(random_ply_plus_1 - 1) : "";   // sorted keys
    return "{\"boards\":" + boards + "],\"dists\":" + dists + "],\"moves\":" + moves + "]" + random_ply + ",\"result\":" + std::to_string(result) + "}";
}

}  // namespace

void RecordWriter::run()
{
    std::unique_lock<std::mutex> lock(m);
    for (;;) {
        cv.wait(lock, [&] { return stop || !jobs.empty(); });
        if (jobs.empty()) return;                          // stop requested and nothing left
        RecordJob job = std::move(jobs.front());
        jobs.pop_front();
        busy = true;
        lock.unlock();
        bool ok = true;
        for (size_t i = 0; i < job.done.size() && ok; ++i) {
            const DoneEntry &d = job.done[i];
            const std::string line = record_to_json(job.words.data() + job.offsets[i], d.words, d.plies, d.result, d.random_ply);
            ok = fwrite(line.data(), 1, line.size(), job.out) == line.size() && fputc('\n', job.out) != EOF;
        }
        if (ok) ok = fflush(job.out) == 0;                 // whole lines only, flushed once per drain (:641-642 flushes per game)
        lock.lock();
        busy = false;
        if (!ok) failed = true;
        if (jobs.empty()) idle_cv.notify_all();
    }
}
void RecordWriter::push(RecordJob &&job)
{
    std::lock_guard<std::mutex> lock(m);
    if (!worker.joinable()) worker = std::thread([this] { run(); });
    jobs.push_back(std::move(job));
    cv.notify_one();
}
bool RecordWriter::flush()
{
    std::unique_lock<std::mutex> lock(m);
    idle_cv.wait(lock, [&] { return jobs.empty() && !busy; });
    const bool ok = !failed;
    failed = false;
    return ok;
}
void RecordWriter::shutdown()
{
    {
        std::lock_guard<std::mutex> lock(m);
        stop = true;
        cv.notify_all();
    }
    if (worker.joinable()) worker.join();
}

namespace {

// Copy out the pool's finished games, append them to `out` (may be null: records are dropped), release the buffers.
// The records are packed into one staging buffer on the device and cross PCIe in ONE copy per drain.
int drain_finished(az_pool *pool, FILE *out, int64_t *games_written, bool copy_payload = true)
{
    cudaStream_t s = pool->ctx->stream;
    AZ_CUDA(cudaMemcpyAsync(pool->h_counts + 3, pool->dev.done_count, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    AZ_CUDA(cudaStreamSynchronize(s));
    const int n = pool->h_counts[3];
    if (n == 0) return AZ_OK;
    AZ_CUDA(cudaMemcpyAsync(pool->h_done, pool->dev.done, sizeof(DoneEntry) * n, cudaMemcpyDeviceToHost, s));
    AZ_CUDA(cudaMemcpyAsync(pool->d_done_snapshot, pool->dev.done, sizeof(DoneEntry) * n, cudaMemcpyDeviceToDevice, s));
    AZ_CUDA(cudaMemsetAsync(pool->dev.done_count, 0, sizeof(int32_t), s));
    AZ_CUDA(cudaStreamSynchronize(s));
    if (copy_payload) {
        for (int first = 0; first < n;) {                 // normally one pass; more only if a drain exceeds the staging buffer
            size_t words = 0;
            int last = first;
            while (last < n && words + (size_t)pool->h_done[last].words <= pool->stage_words) {
                pool->h_offsets[last] = (uint32_t)words;
                words += (size_t)pool->h_done[last].words;
                ++last;
            }
            if (last == first) return az_fail(AZ_ERR_CAPACITY, "record of %d words exceeds the staging buffer", pool->h_done[first].words);
            const int m = last - first;
            AZ_CUDA(cudaMemcpyAsync(pool->d_offsets, pool->h_offsets + first, sizeof(uint32_t) * m, cudaMemcpyHostToDevice, s));
            aztree_launch_gather(pool->dev, pool->d_done_snapshot + first, pool->d_offsets, m, pool->d_stage, s);
            pool->launches++;
            AZ_CUDA(cudaMemcpyAsync(pool->h_stage, pool->d_stage, sizeof(uint32_t) * words, cudaMemcpyDeviceToHost, s));
            AZ_CUDA(cudaStreamSynchronize(s));
            pool->d2h_bytes += sizeof(uint32_t) * (uint64_t)words;
            if (out) {                                    // JSON and file I/O happen on the writer thread
                RecordJob job;
                job.out = out;
                job.words.assign(pool->h_stage, pool->h_stage + words);
                job.done.assign(pool->h_done + first, pool->h_done + last);
                job.offsets.assign(pool->h_offsets + first, pool->h_offsets + last);
                pool->writer.push(std::move(job));
            }
            first = last;
        }
    }
    for (int i = 0; i < n; ++i) {
        pool->written_games++;
        pool->written_positions += pool->h_done[i].plies;
        if (games_written) (*games_written)++;
    }
    aztree_launch_release(pool->dev, pool->d_done_snapshot, n, s);
    pool->launches++;
    return AZ_OK;
}

void free_buffers(az_pool *pool)
{
    PoolDev &D = pool->dev;
    void *ptrs[] = {D.nodes, D.games, D.path, D.gstack, D.req_pos, D.req_game, D.req_stage, D.req_mark, D.req_count, D.logits, D.values, D.cache_tag,
                    D.cache_exps, D.cache_tot, D.cache_val, D.req_out, D.records,
                    D.done, D.done_count, pool->d_done_snapshot, pool->d_status, pool->d_timed_evals, pool->d_features, pool->d_offsets, pool->d_stage,
                    D.arena_slot_game, D.mailbox, const_cast<az_position *>(D.openings), D.arena_moves, D.arena_plies, D.arena_result,
                    D.arena_counters};
    for (void *p : ptrs)
        if (p) cudaFree(p);
    if (pool->h_counts) cudaFreeHost(pool->h_counts);
    if (pool->h_done) cudaFreeHost(pool->h_done);
    if (pool->h_offsets) cudaFreeHost(pool->h_offsets);
    if (pool->h_stage) cudaFreeHost(pool->h_stage);
    for (auto &set : pool->ev)
      for (auto &e : set)
        if (e) cudaEventDestroy(e);
}

bool valid_position(const az_position &r)
{
    const uint64_t all = r.pieces[0] | r.pieces[1] | r.blockers;
    return !(r.pieces[0] & r.pieces[1]) && !((r.pieces[0] | r.pieces[1]) & r.blockers) && !(all >> 49) && (r.pieces[0] | r.pieces[1]);
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
extern "C" int az_pool_create(az_context *ctx, const az_pool_config *cfg, az_pool **out)
{
    AZ_REQUIRE(ctx && cfg && out, AZ_ERR_ARG, "az_pool_create: null argument");
    *out = nullptr;
    AZ_REQUIRE(cfg->games >= 1 && cfg->games <= (1 << 20), AZ_ERR_ARG, "az_pool_create: games=%d", cfg->games);
    AZ_REQUIRE(cfg->visits >= 1 && cfg->visits <= (1 << 22), AZ_ERR_ARG, "az_pool_create: visits=%d", cfg->visits);
    AZ_REQUIRE(cfg->eval_mode == AZ_NET_FP32 || cfg->eval_mode == AZ_NET_BF16 || cfg->eval_mode == AZ_NET_F16 || cfg->eval_mode == AZ_EVAL_EXTERNAL, AZ_ERR_ARG,
               "az_pool_create: eval_mode=%d", cfg->eval_mode);
    AZ_REQUIRE(cfg->eval_mode == AZ_EVAL_EXTERNAL || ctx->net, AZ_ERR_STATE, "az_pool_create: no weights loaded (az_net_load)");
    az_position start;
    const char *fen = cfg->start_fen[0] ? cfg->start_fen : "startpos";
    AZ_REQUIRE(az_set_board(&start, fen) == 0, AZ_ERR_ARG, "az_pool_create: bad start_fen '%s'", fen);

    az_pool *pool = new az_pool();
    pool->ctx = ctx;
    pool->cfg = *cfg;
    if (pool->cfg.max_plies <= 0) pool->cfg.max_plies = 400;
    if (pool->cfg.node_capacity <= 0) pool->cfg.node_capacity = cfg->visits + 64;
    if (pool->cfg.steps_per_tick <= 0) pool->cfg.steps_per_tick = 8;
    AZ_REQUIRE(pool->cfg.node_capacity < (1 << 24), AZ_ERR_ARG, "az_pool_create: node_capacity too large");

    const bool tensor_net = cfg->eval_mode == AZ_NET_BF16 || cfg->eval_mode == AZ_NET_F16;
    size_t free_b = 0, total_b = 0;
    AZ_CUDA(cudaMemGetInfo(&free_b, &total_b));
    const uint32_t rec_cap_words = cfg->auto_play ? (uint32_t)pool->cfg.max_plies * kRecWordsPerPly : 16;
    {
        const size_t G = (size_t)cfg->games, C = (size_t)pool->cfg.node_capacity;
        const size_t need = G * C * kNodeStride + G * 2 * rec_cap_words * 4 + G * (kMaxPath + C) * 4 + G * 4096;
        if (need > free_b) {
            delete pool;
            return az_fail(AZ_ERR_CAPACITY, "az_pool_create: needs %.1f GiB of HBM, %.1f GiB free", need / 1073741824.0, free_b / 1073741824.0);
        }
    }
    PoolDev &D = pool->dev;
    D.G = cfg->games;
    D.C = pool->cfg.node_capacity;
    D.visits = cfg->visits;
    D.max_plies = pool->cfg.max_plies;
    D.noise = cfg->noise ? 1 : 0;
    D.auto_play = cfg->auto_play ? 1 : 0;
    D.steps_per_tick = pool->cfg.steps_per_tick;
    // evaluations per tick: a whole number of rounds of the net kernel's persistent CTAs, so its last round is
    // never half empty; later requests are re-queued.  Self-play on the tensor-core net only (search pools serve every
    // request).  AZ_REQ_CAP=<n> sets the cap, 0 serves every request.
    D.cap = D.G;
    if (cfg->auto_play && tensor_net) {
        const int round = az_net_pair_boards_per_round(ctx);
        if (const char *env = getenv("AZ_REQ_CAP")) D.cap = atoi(env) > 0 ? std::min(atoi(env), D.G) : D.G;
        else if (D.G >= round) D.cap = D.G / round * round;
    }
    // the level budget trims the tail of a tick over thousands of games; a handful of trees has no tail to trim, and a
    // suspended descent would cost it a whole (empty) net launch
    // The budget is in levels, not in clock cycles: how far a game gets would then depend on timing, and the same seed
    // would not replay the same games.
    D.levels_per_tick = getenv("AZ_LEVELS_PER_TICK") ? atoi(getenv("AZ_LEVELS_PER_TICK")) : (cfg->games < 64 ? (1 << 20) : 48);
    D.seed = cfg->seed;
    D.prefetch = getenv("AZ_TREE_PREFETCH") ? atoi(getenv("AZ_TREE_PREFETCH")) : 8;
    D.force_slow = getenv("AZ_TREE_FORCE_SLOW") ? atoi(getenv("AZ_TREE_FORCE_SLOW")) : 0;
    D.one_random_move = (cfg->auto_play && cfg->one_random_move) ? 1 : 0;
    D.rec_cap_words = rec_cap_words;
    const size_t G = (size_t)D.G;
    int rc = 0;
    rc |= dev_alloc(&D.nodes, G * D.C * kNodeStride, false);
    rc |= dev_alloc(&D.games, G);
    rc |= dev_alloc(&D.path, G * kMaxPath, false);
    rc |= dev_alloc(&D.gstack, G * D.C, false);
    rc |= dev_alloc(&D.req_pos, G);
    rc |= dev_alloc(&D.req_game, G);
    rc |= dev_alloc(&D.req_stage, G);
    rc |= dev_alloc(&D.req_mark, G);          // zero: no tick 0 is ever launched
    rc |= dev_alloc(&D.req_count, 12);       // [3][2], and B's [3][2] of an arena pool
    rc |= dev_alloc(&D.logits, G * AZ_LOGITS);
    rc |= dev_alloc(&D.values, G);
    const int spec_k = (tensor_net && !cfg->auto_play) ? std::min(std::max(cfg->speculate, 0), 64) : 0;
    if (spec_k > 0) {
        // speculative evaluation: a per-game cache of evaluations + a request batch that can hold the extra requests
        int entries = 1024;
        while (entries < 2 * pool->cfg.node_capacity && entries < (1 << 18)) entries *= 2;    // 6.7 KB per entry
        D.cache_entries = entries;
        D.spec_k = spec_k;
        D.req_cap = std::max(2 * az_net_pair_boards_per_round(ctx), (int)G * (1 + spec_k));
        const size_t total = G * (size_t)entries + 1;        // + the trash entry
        rc |= dev_alloc(&D.cache_tag, total);
        rc |= dev_alloc(&D.cache_exps, total * AZ_LOGITS, false);
        rc |= dev_alloc(&D.cache_tot, total, false);
        rc |= dev_alloc(&D.cache_val, total, false);
        rc |= dev_alloc(&D.req_out, (size_t)D.req_cap);
        cudaFree(D.req_pos);
        D.req_pos = nullptr;
        rc |= dev_alloc(&D.req_pos, (size_t)std::max<int>(D.req_cap, (int)G));
    }
    rc |= dev_alloc(&D.records, G * 2 * D.rec_cap_words, false);
    rc |= dev_alloc(&D.done, 2 * G);
    rc |= dev_alloc(&D.done_count, 1);
    rc |= dev_alloc(&pool->d_done_snapshot, 2 * G);
    rc |= dev_alloc(&pool->d_offsets, 2 * G);
    // staging for one drain: every game can hand over at most its two record buffers; in practice a drain carries a few
    // dozen games, so the buffer is sized for 64 full-length records (a larger drain is fetched in several passes)
    pool->stage_words = (size_t)D.rec_cap_words * (cfg->auto_play ? std::min<size_t>(2 * G, 64) : 1);
    rc |= dev_alloc(&pool->d_stage, pool->stage_words, false);
    rc |= dev_alloc(&pool->d_status, 4);
    rc |= dev_alloc(&pool->d_timed_evals, 1);
    rc |= dev_alloc(&pool->d_features, G * AZ_FEATURES);
    if (rc == 0 && (cudaMallocHost(&pool->h_counts, 16 * sizeof(int32_t)) != cudaSuccess ||
                    cudaMallocHost(&pool->h_done, sizeof(DoneEntry) * 2 * G) != cudaSuccess ||
                    cudaMallocHost(&pool->h_offsets, sizeof(uint32_t) * 2 * G) != cudaSuccess ||
                    cudaMallocHost(&pool->h_stage, sizeof(uint32_t) * pool->stage_words) != cudaSuccess))
        rc = az_fail(AZ_ERR_CUDA, "az_pool_create: pinned host alloc");
    pool->h_games.resize(G);
    for (auto &set : pool->ev) {
        set.assign(1 + 2 * kTicksPerDrain, nullptr);
        for (auto &e : set)
            if (cudaEventCreate(&e) != cudaSuccess) rc = az_fail(AZ_ERR_CUDA, "az_pool_create: event");
    }
    if (getenv("AZ_POOL_PROFILE")) rc |= dev_alloc(&D.prof, G * 16);
    if (rc) { az_pool_destroy(pool); return rc; }
    aztree_launch_init_all(D, start, ctx->stream);
    pool->launches++;
    const cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { az_pool_destroy(pool); return az_fail(AZ_ERR_CUDA, "az_pool_create: %s", cudaGetErrorString(e)); }
    AZ_CUDA(cudaGetLastError());
    if ((rc = check_game_errors(pool))) { az_pool_destroy(pool); return rc; }
    *out = pool;
    return AZ_OK;
}

extern "C" void az_pool_destroy(az_pool *pool)
{
    if (!pool) return;
    cudaStreamSynchronize(pool->ctx->stream);
    pool->writer.flush();
    pool->writer.shutdown();
    if (pool->dev.prof) {              // per-phase cycles, accumulated over every tick: mean and worst game
        std::vector<unsigned long long> h((size_t)pool->dev.G * 16);
        cudaMemcpy(h.data(), pool->dev.prof, h.size() * 8, cudaMemcpyDeviceToHost);
        const char *names[6] = {"populate", "backup", "descent", "expand", "make_move", "total"};
        for (int ph = 0; ph < 6; ++ph) {
            double sum = 0, mx = 0;
            for (int g = 0; g < pool->dev.G; ++g) { sum += (double)h[(size_t)g * 16 + ph]; mx = std::max(mx, (double)h[(size_t)g * 16 + ph]); }
            fprintf(stderr, "[az_pool profile] %-9s mean %.1f kcycles/tick/game, worst game %.1f kcycles/tick (%llu ticks)\n", names[ph],
                    sum / pool->dev.G / std::max<uint64_t>(pool->ticks, 1) / 1e3, mx / std::max<uint64_t>(pool->ticks, 1) / 1e3,
                    (unsigned long long)pool->ticks);
        }
        // the last tick on the wall clock: when did each game start and finish inside the kernel?
        std::vector<double> start, finish;
        unsigned long long t0 = ~0ull;
        for (int g = 0; g < pool->dev.G; ++g)
            if (h[(size_t)g * 16 + 6]) t0 = std::min(t0, h[(size_t)g * 16 + 6]);
        std::vector<std::pair<double, int>> order;
        for (int g = 0; g < pool->dev.G; ++g)
            if (h[(size_t)g * 16 + 6]) {
                start.push_back((double)(h[(size_t)g * 16 + 6] - t0) * 1e-3);
                finish.push_back((double)(h[(size_t)g * 16 + 7] - t0) * 1e-3);
                order.push_back({finish.back(), g});
            }
        // what the games of each finish-time band did in that tick (cycles per phase, steps, tree levels)
        std::sort(order.begin(), order.end());
        const double bands[6] = {0.0, 0.25, 0.5, 0.75, 0.9, 0.97};
        for (int b = 0; b < 6 && !order.empty(); ++b) {
            const size_t lo = (size_t)(bands[b] * order.size()), hi = b == 5 ? order.size() : (size_t)(bands[b + 1] * order.size());
            if (hi <= lo) continue;                    // pools of a few games: not every band has one
            double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, waiting = 0;
            for (size_t i = lo; i < hi; ++i) {
                const unsigned long long *q = &h[(size_t)order[i].second * 16 + 8];
                for (int j = 0; j < 7; ++j) acc[j] += (double)q[j];
                waiting += q[7] == 1 ? 1 : 0;
            }
            const double n = (double)std::max<size_t>(hi - lo, 1);
            fprintf(stderr, "[az_pool profile] last tick, finish %5.1f..%5.1f us (%4zu games): populate %5.1f backup %4.1f descent %5.1f expand %4.1f "
                            "sum of all %5.1f kcycles | steps %.2f levels %.1f | requested an evaluation %.0f%%\n",
                    order[lo].first, order[hi - 1].first, hi - lo, acc[0] / n / 1e3, acc[1] / n / 1e3, acc[2] / n / 1e3, acc[3] / n / 1e3,
                    acc[4] / n / 1e3, acc[5] / n, acc[6] / n, 100.0 * waiting / n);
        }
        // the stragglers one by one: the tick ends with the last of them
        for (size_t i = order.size() > 12 ? order.size() - 12 : 0; i < order.size(); ++i) {
            const unsigned long long *q = &h[(size_t)order[i].second * 16 + 8];
            fprintf(stderr, "[az_pool profile] straggler game %5d finished %5.1f us: populate %5.1f backup %4.1f descent %5.1f expand %4.1f "
                            "all %5.1f kcycles | steps %llu levels %llu status %llu\n",
                    order[i].second, order[i].first, q[0] / 1e3, q[1] / 1e3, q[2] / 1e3, q[3] / 1e3, q[4] / 1e3, q[5], q[6], q[7]);
        }
        if (!finish.empty()) {
            std::sort(start.begin(), start.end());
            std::sort(finish.begin(), finish.end());
            auto pct = [](const std::vector<double> &v, double q) { return v[std::min(v.size() - 1, (size_t)(q * v.size()))]; };
            fprintf(stderr, "[az_pool profile] last tick, us after the first warp started: starts p50 %.1f p99 %.1f max %.1f | finishes p10 %.1f "
                            "p50 %.1f p75 %.1f p87 %.1f p95 %.1f p99 %.1f max %.1f\n",
                    pct(start, 0.5), pct(start, 0.99), start.back(), pct(finish, 0.10), pct(finish, 0.5), pct(finish, 0.75), pct(finish, 0.87),
                    pct(finish, 0.95), pct(finish, 0.99), finish.back());
        }
        cudaFree(pool->dev.prof);
        pool->dev.prof = nullptr;
    }
    free_buffers(pool);
    delete pool;
}

extern "C" int az_pool_stats_get(az_pool *pool, az_pool_stats *out)
{
    AZ_REQUIRE(pool && out, AZ_ERR_ARG, "az_pool_stats_get: null argument");
    AZ_CUDA(cudaStreamSynchronize(pool->ctx->stream));
    read_events(pool, 0);                          // every batch has completed: bring the timing sums up to date
    read_events(pool, 1);
    az_pool_stats s{};
    AZ_CUDA(cudaMemcpy(pool->h_games.data(), pool->dev.games, sizeof(Game) * pool->dev.G, cudaMemcpyDeviceToHost));
    for (const Game &g : pool->h_games) {
        s.steps += g.steps;
        s.evals += g.evals;
        s.terminal_steps += g.terminal_steps;
        s.positions += g.positions;
        s.games_finished += g.finished;
        s.games_skipped += g.skipped;
        s.max_depth = std::max<uint64_t>(s.max_depth, g.max_depth);
        s.levels += g.levels;
    }
    s.ticks = pool->ticks;
    s.kernel_launches = pool->launches;
    s.record_bytes = pool->d2h_bytes;
    s.net_seconds = pool->net_seconds;
    s.tree_seconds = pool->tree_seconds;
    s.tick_seconds = pool->tick_seconds;
    s.timed_ticks = pool->timed_ticks;
    unsigned long long device_timed_evals = 0;
    AZ_CUDA(cudaMemcpy(&device_timed_evals, pool->d_timed_evals, sizeof(device_timed_evals), cudaMemcpyDeviceToHost));
    s.timed_evals = pool->timed_evals_host + device_timed_evals;
    *out = s;
    return AZ_OK;
}

extern "C" int az_pool_set_root(az_pool *pool, int game, const az_position *root)
{
    AZ_REQUIRE(pool && root, AZ_ERR_ARG, "az_pool_set_root: null argument");
    AZ_REQUIRE(game >= 0 && game < pool->G(), AZ_ERR_ARG, "az_pool_set_root: game %d out of range", game);
    AZ_REQUIRE(pool->pending_requests == 0, AZ_ERR_STATE, "az_pool_set_root: evaluations are outstanding (az_pool_provide first)");
    AZ_REQUIRE(valid_position(*root), AZ_ERR_ARG, "az_pool_set_root: invalid position");
    aztree_launch_set_root(pool->dev, game, *root, pool->ctx->stream);
    pool->launches++;
    AZ_CUDA(cudaStreamSynchronize(pool->ctx->stream));
    AZ_CUDA(cudaGetLastError());
    return AZ_OK;
}

extern "C" int az_pool_set_roots(az_pool *pool, const az_position *roots)
{
    AZ_REQUIRE(pool && roots, AZ_ERR_ARG, "az_pool_set_roots: null argument");
    AZ_REQUIRE(pool->pending_requests == 0, AZ_ERR_STATE, "az_pool_set_roots: evaluations are outstanding (az_pool_provide first)");
    for (int g = 0; g < pool->G(); ++g)
        AZ_REQUIRE(valid_position(roots[g]), AZ_ERR_ARG, "az_pool_set_roots: invalid position for game %d", g);
    cudaStream_t s = pool->ctx->stream;
    AZ_CUDA(cudaMemcpyAsync(pool->dev.req_pos, roots, sizeof(az_position) * pool->dev.G, cudaMemcpyHostToDevice, s));
    aztree_launch_set_roots(pool->dev, pool->dev.req_pos, s);     // req_pos is free between ticks: reuse it as staging
    pool->launches++;
    AZ_CUDA(cudaStreamSynchronize(s));
    AZ_CUDA(cudaGetLastError());
    return check_game_errors(pool);
}

extern "C" int az_pool_set_visits(az_pool *pool, int visits)
{
    AZ_REQUIRE(pool, AZ_ERR_ARG, "az_pool_set_visits: null pool");
    AZ_REQUIRE(visits >= 1 && visits + 2 <= pool->cfg.node_capacity, AZ_ERR_ARG, "az_pool_set_visits: visits=%d does not fit node_capacity=%d",
               visits, pool->cfg.node_capacity);
    AZ_CUDA(cudaStreamSynchronize(pool->ctx->stream));
    pool->cfg.visits = visits;
    pool->dev.visits = visits;
    // trees that were parked as "done" under the old target may have work again
    AZ_CUDA(cudaMemcpy(pool->h_games.data(), pool->dev.games, sizeof(Game) * pool->dev.G, cudaMemcpyDeviceToHost));
    for (Game &g : pool->h_games)
        if (g.status == ST_DONE) g.status = ST_IDLE;
    AZ_CUDA(cudaMemcpy(pool->dev.games, pool->h_games.data(), sizeof(Game) * pool->dev.G, cudaMemcpyHostToDevice));
    return AZ_OK;
}

extern "C" int az_pool_run(az_pool *pool, int max_ticks, int32_t *idle_out)
{
    AZ_REQUIRE(pool, AZ_ERR_ARG, "az_pool_run: null pool");
    AZ_REQUIRE(!pool->ctx_b, AZ_ERR_STATE, "az_pool_run: arena pools are driven by az_arena_play");
    AZ_REQUIRE(pool->cfg.eval_mode != AZ_EVAL_EXTERNAL, AZ_ERR_STATE, "az_pool_run: pool uses an external evaluator (collect/provide)");
    if (idle_out) *idle_out = 0;
    // Ticks are launched in bursts and the "anything left to do?" counters are read back once per burst: a tick of an
    // idle pool is two empty kernels, far cheaper than a host round trip per tick (single-tree searches are
    // latency-bound: one leaf per tick).  The burst doubles up to 16 while the pool stays busy.
    int burst = 1;
    for (int t = 0; t < max_ticks;) {
        const int n = std::min(burst, max_ticks - t);
        for (int k = 0; k < n; ++k) {
            int rc = launch_tree(pool);
            if (rc) return rc;
            if (k == n - 1)
                AZ_CUDA(cudaMemcpyAsync(pool->h_counts, pool->dev.req_count + 2 * pool->slot, 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, pool->ctx->stream));
            if ((rc = launch_net(pool))) return rc;
            pool->ticks++;
        }
        t += n;
        AZ_CUDA(cudaStreamSynchronize(pool->ctx->stream));
        if (pool->h_counts[0] == 0 && pool->h_counts[1] == 0) {    // no requests, nobody mid-step: every tree is done (or stalled)
            if (idle_out) *idle_out = 1;
            break;
        }
        burst = std::min(2 * burst, 16);
    }
    AZ_CUDA(cudaGetLastError());
    return check_game_errors(pool);
}

extern "C" int az_pool_collect(az_pool *pool, float *features, int32_t *n_requests)
{
    AZ_REQUIRE(pool && features && n_requests, AZ_ERR_ARG, "az_pool_collect: null argument");
    AZ_REQUIRE(pool->cfg.eval_mode == AZ_EVAL_EXTERNAL, AZ_ERR_STATE, "az_pool_collect: pool uses the internal net");
    AZ_REQUIRE(pool->pending_requests == 0, AZ_ERR_STATE, "az_pool_collect: previous requests not answered (az_pool_provide)");
    cudaStream_t s = pool->ctx->stream;
    *n_requests = 0;
    // The first tick consumes the evaluations handed in by az_pool_provide.  A tree may burn its step budget
    // on adjudicated leaves without reaching a leaf that needs the net, so "top-up" ticks (which leave the
    // already-waiting games alone and append to the request list) run until no tree can make progress.
    for (int attempt = 0; attempt < 65536; ++attempt) {
        int rc = launch_tree(pool, attempt == 0);
        if (rc) return rc;
        if (attempt == 0) pool->ticks++;
        AZ_CUDA(cudaMemcpyAsync(pool->h_counts, pool->dev.req_count + 2 * pool->slot, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
        AZ_CUDA(cudaStreamSynchronize(s));
        if ((rc = check_game_errors(pool))) return rc;
        bool busy = false;
        for (int g = 0; g < pool->dev.G; ++g) busy |= pool->h_games[g].status == ST_IDLE || pool->h_games[g].status == ST_DESCEND;
        if (!busy) break;                       // every tree is waiting, done or stalled
    }
    const int n = std::min(pool->h_counts[0], pool->dev.cap);   // requests beyond the cap stay queued (the tree kernel re-issues them)
    if (n > 0) {
        aztree_launch_features(pool->dev.req_pos, n, pool->d_features, s);
        pool->launches++;
        AZ_CUDA(cudaMemcpyAsync(features, pool->d_features, sizeof(float) * AZ_FEATURES * n, cudaMemcpyDeviceToHost, s));
        AZ_CUDA(cudaStreamSynchronize(s));
    }
    AZ_CUDA(cudaGetLastError());
    pool->pending_requests = n;
    *n_requests = n;
    return AZ_OK;
}

extern "C" int az_pool_provide_n(az_pool *pool, const float *logits, const float *values, int32_t n_rows)
{
    AZ_REQUIRE(pool && logits && values, AZ_ERR_ARG, "az_pool_provide: null argument");
    AZ_REQUIRE(pool->pending_requests > 0, AZ_ERR_STATE, "az_pool_provide: no outstanding requests");
    const int n = pool->pending_requests;
    AZ_REQUIRE(n_rows == n, AZ_ERR_ARG, "az_pool_provide: %d evaluations handed in for %d outstanding requests", n_rows, n);
    cudaStream_t s = pool->ctx->stream;
    AZ_CUDA(cudaMemcpyAsync(pool->dev.logits, logits, sizeof(float) * AZ_LOGITS * n, cudaMemcpyHostToDevice, s));
    AZ_CUDA(cudaMemcpyAsync(pool->dev.values, values, sizeof(float) * n, cudaMemcpyHostToDevice, s));
    AZ_CUDA(cudaStreamSynchronize(s));      // the caller may free its arrays right away (complete_workload copies too)
    pool->pending_requests = 0;
    return AZ_OK;
}

// complete_workload() semantics: the caller's arrays are trusted to hold one row per outstanding request
extern "C" int az_pool_provide(az_pool *pool, const float *logits, const float *values)
{
    AZ_REQUIRE(pool, AZ_ERR_ARG, "az_pool_provide: null argument");
    return az_pool_provide_n(pool, logits, values, pool->pending_requests);
}

extern "C" int az_pool_root(az_pool *pool, int game, az_position *pos, int32_t *n_moves, az_move *moves, int32_t *visits,
                            double *total_score, double *prior, int32_t *root_visits, double *root_value)
{
    AZ_REQUIRE(pool, AZ_ERR_ARG, "az_pool_root: null pool");
    AZ_REQUIRE(game >= 0 && game < pool->G(), AZ_ERR_ARG, "az_pool_root: game %d out of range", game);
    AZ_CUDA(cudaStreamSynchronize(pool->ctx->stream));
    Game gm;
    AZ_CUDA(cudaMemcpy(&gm, pool->dev.games + game, sizeof(Game), cudaMemcpyDeviceToHost));
    AZ_REQUIRE(gm.status != ST_ERROR, AZ_ERR_CAPACITY, "game %d: %s", game, kErrNames[std::min(std::max(gm.error, 0), 4)]);
    std::vector<uint8_t> slot(kNodeStride);
    AZ_CUDA(cudaMemcpy(slot.data(), pool->dev.nodes + ((size_t)game * pool->dev.C + gm.root) * kNodeStride, kNodeStride,
                       cudaMemcpyDeviceToHost));
    const NodeHdr *h = reinterpret_cast<const NodeHdr *>(slot.data());
    if (pos) {
        pos->ply = gm.ply;
        pos->turn = h->turn;
        pos->blockers = gm.blockers;
        pos->pieces[h->turn] = h->own;
        pos->pieces[h->turn ^ 1] = h->opp;
    }
    if (n_moves) *n_moves = h->n_moves;
    if (root_visits) *root_visits = h->N;
    if (root_value) *root_value = h->value;
    for (int i = 0; i < h->n_moves; ++i) {
        if (moves) moves[i] = reinterpret_cast<const uint16_t *>(slot.data() + kOffMove)[i];
        if (visits) visits[i] = 0;
        if (total_score) total_score[i] = 0.0;
        if (prior) prior[i] = reinterpret_cast<const double *>(slot.data() + kOffP)[i];
    }
    const Entry *ent = reinterpret_cast<const Entry *>(slot.data() + kOffEntry);
    for (int e = 0; e < h->k; ++e) {                      // edges live in a dense list; report them by movegen index
        const int i = (int)(ent[e].child >> kMoveIdxShift);
        if (visits) visits[i] = (int32_t)(ent[e].n & kVisitMask);
        if (total_score) total_score[i] = ent[e].W;
    }
    return AZ_OK;
}

extern "C" int az_pool_pv(az_pool *pool, int game, az_move *moves, int32_t *visits, int max_len, int32_t *len_out)
{
    AZ_REQUIRE(pool && moves && len_out && max_len >= 0, AZ_ERR_ARG, "az_pool_pv: bad argument");
    AZ_REQUIRE(game >= 0 && game < pool->G(), AZ_ERR_ARG, "az_pool_pv: game %d out of range", game);
    AZ_CUDA(cudaStreamSynchronize(pool->ctx->stream));
    Game gm;
    AZ_CUDA(cudaMemcpy(&gm, pool->dev.games + game, sizeof(Game), cudaMemcpyDeviceToHost));
    std::vector<uint8_t> slot(kNodeStride);
    int node = gm.root, n = 0;
    while (n < max_len && node >= 0) {                      // select_principal_variation(best=True), engine.py:331-336
        AZ_CUDA(cudaMemcpy(slot.data(), pool->dev.nodes + ((size_t)game * pool->dev.C + node) * kNodeStride, kNodeStride, cudaMemcpyDeviceToHost));
        const NodeHdr *h = reinterpret_cast<const NodeHdr *>(slot.data());
        const Entry *ent = reinterpret_cast<const Entry *>(slot.data() + kOffEntry);
        int best = -1;
        for (int e = 0; e < h->k; ++e)                     // max(): first of the most visited edges, in order of creation
            if (best < 0 || (ent[e].n & kVisitMask) > (ent[best].n & kVisitMask)) best = e;   // (engine.py's dict order)
        if (best < 0) break;
        moves[n] = reinterpret_cast<const uint16_t *>(slot.data() + kOffMove)[ent[best].child >> kMoveIdxShift];
        if (visits) visits[n] = (int32_t)(ent[best].n & kVisitMask);
        ++n;
        node = (int)(ent[best].child & kChildMask);
    }
    *len_out = n;
    return AZ_OK;
}

// Debug / analysis hook (not in the public header): positions (own, opp, turn) of every node reachable from the root
// of `game`, breadth first.  Used to measure how many leaves of a search are transpositions of each other.
extern "C" int az_pool_debug_nodes(az_pool *pool, int game, uint64_t *own, uint64_t *opp, int32_t *turn, int32_t *visits, int max_nodes,
                                   int32_t *n_out)
{
    AZ_REQUIRE(pool && own && opp && turn && n_out, AZ_ERR_ARG, "az_pool_debug_nodes: bad argument");
    AZ_CUDA(cudaStreamSynchronize(pool->ctx->stream));
    Game gm;
    AZ_CUDA(cudaMemcpy(&gm, pool->dev.games + game, sizeof(Game), cudaMemcpyDeviceToHost));
    std::vector<uint8_t> arena((size_t)pool->dev.C * kNodeStride);
    AZ_CUDA(cudaMemcpy(arena.data(), pool->dev.nodes + (size_t)game * pool->dev.C * kNodeStride, arena.size(), cudaMemcpyDeviceToHost));
    std::vector<int> queue{gm.root};
    int n = 0;
    for (size_t q = 0; q < queue.size() && n < max_nodes; ++q) {
        const uint8_t *nd = arena.data() + (size_t)queue[q] * kNodeStride;
        const NodeHdr *h = reinterpret_cast<const NodeHdr *>(nd);
        own[n] = h->own; opp[n] = h->opp; turn[n] = h->turn;
        if (visits) visits[n] = h->N;
        ++n;
        const Entry *ent = reinterpret_cast<const Entry *>(nd + kOffEntry);
        for (int e = 0; e < h->k; ++e) queue.push_back((int)(ent[e].child & kChildMask));
    }
    *n_out = n;
    return AZ_OK;
}

extern "C" int az_pool_play(az_pool *pool, int game, az_move move)
{
    AZ_REQUIRE(pool, AZ_ERR_ARG, "az_pool_play: null pool");
    AZ_REQUIRE(game >= 0 && game < pool->G(), AZ_ERR_ARG, "az_pool_play: game %d out of range", game);
    AZ_REQUIRE(pool->pending_requests == 0, AZ_ERR_STATE, "az_pool_play: evaluations are outstanding");
    cudaStream_t s = pool->ctx->stream;
    aztree_launch_play(pool->dev, game, (int)move, pool->d_status, s);
    pool->launches++;
    AZ_CUDA(cudaMemcpyAsync(pool->h_counts + 2, pool->d_status, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    AZ_CUDA(cudaStreamSynchronize(s));
    AZ_CUDA(cudaGetLastError());
    const int st = pool->h_counts[2];
    AZ_REQUIRE(st != -1, AZ_ERR_ARG, "az_pool_play: move is not legal at the root of game %d", game);
    AZ_REQUIRE(st != -2, AZ_ERR_STATE, "az_pool_play: game %d is waiting for an evaluation", game);
    AZ_REQUIRE(st == 0, AZ_ERR_CAPACITY, "az_pool_play: node pool exhausted");
    return AZ_OK;
}

namespace {

// `ticks` (<= kTicksPerDrain) iterations of (tree kernel, net kernel), then one drain of finished games.  Every tick is
// bracketed by CUDA events on the context stream; after the drain's synchronisation the per-launch times are summed into
// tree_seconds / net_seconds / tick_seconds -- every launch is measured, nothing is extrapolated.
//
// Measured and rejected (r02, profiles/r02_early_launch_trace.txt): launching the net kernel PROGRAMMATICALLY behind the tree
// kernel (griddepcontrol.launch_dependents + request-slot stamps) so that the tree's tail -- its slowest game takes twice as
// long as the median one -- hides behind the net's first tower pass.  The overlap happens (net CTAs start 49..178 us into
// the tick instead of ~105), but a net CTA can only move onto an SM once most of that SM's games are done, the games still
// running next to it slow down 1.8x (last finish 173 us instead of 97), and the SMs hosting them start their two CTAs last
// -- with three 170-us unit passes per CTA nothing can be rebalanced at that granularity, so the kernel ends when it did.
// read out the event set `set` (its batch has completed) into the pool's timing sums
void read_events(az_pool *pool, int set)
{
    // ev[0]: before the batch; ev[1 + 2t] / ev[2 + 2t]: behind the tree / the net kernel of tick t.  A kernel's time runs from the
    // event behind its predecessor, so the launch gap in front of it is part of it.
    const std::vector<cudaEvent_t> &ev = pool->ev[set];
    for (int t = 0; t < pool->ev_ticks[set]; ++t) {
        float a = 0.f, b = 0.f;
        if (cudaEventElapsedTime(&a, ev[2 * t], ev[2 * t + 1]) != cudaSuccess || cudaEventElapsedTime(&b, ev[2 * t + 1], ev[2 * t + 2]) != cudaSuccess) continue;
        pool->tree_seconds += a * 1e-3;
        pool->net_seconds += b * 1e-3;
        pool->tick_seconds += (a + b) * 1e-3;
        pool->timed_ticks++;
    }
    pool->ev_ticks[set] = 0;
}

// everything a caller may look at after an entry point returns: timing sums complete, every record in its file
int finish_batches(az_pool *pool)
{
    read_events(pool, 0);
    read_events(pool, 1);
    if (!pool->writer.flush()) return az_fail(AZ_ERR_IO, "short write to the game file");
    return AZ_OK;
}

int run_ticks(az_pool *pool, FILE *out, bool copy_records, int ticks, int64_t *games)
{
    int rc = AZ_OK;
    cudaStream_t s = pool->ctx->stream;
    const int set = pool->ev_cur;
    // Which launches carry events: a timing event between two kernels costs ~3 us of GPU time (the front end cannot prepare
    // the next launch behind it: 0.579 against 0.572 ms per tick with and without them), so the events sit on a CONTIGUOUS
    // window of kEventWindow ticks out of every kEventPeriod -- every tree and net launch inside a window is bracketed, and
    // the evaluations those net launches served are counted on the device (PoolDev::timed_evals), nothing is extrapolated.
    // AZ_POOL_EVENT_WINDOW=<ticks> changes the window (>= the period: every tick, 0: none).
    static const int window = getenv("AZ_POOL_EVENT_WINDOW") ? atoi(getenv("AZ_POOL_EVENT_WINDOW")) : kEventWindow;
    const bool timed = (int)(pool->ticks % kEventPeriod) < window;
    if (timed) cudaEventRecord(pool->ev[set][0], s);
    for (int t = 0; t < ticks && rc == AZ_OK; ++t) {
        pool->dev.timed_evals = (timed && t > 0) ? pool->d_timed_evals : nullptr;      // tick t's tree kernel counts tick t-1's net launch
        rc = launch_tree(pool);
        pool->dev.timed_evals = nullptr;
        if (timed) cudaEventRecord(pool->ev[set][2 * t + 1], s);
        if (rc == AZ_OK) rc = launch_net(pool);
        if (timed) cudaEventRecord(pool->ev[set][2 * t + 2], s);
        pool->ticks++;
    }
    if (rc) return rc;
    if (timed)                                    // the batch's last net launch: its request count is read behind the batch
        AZ_CUDA(cudaMemcpyAsync(pool->h_counts + 4, pool->dev.req_count + 2 * pool->slot, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    pool->ev_ticks[set] = timed ? ticks : 0;
    pool->ev_cur = set ^ 1;
    // the previous batch finished before this one was launched: its events are read while the GPU works on this one
    read_events(pool, set ^ 1);
    if ((rc = drain_finished(pool, out, games, copy_records))) return rc;
    AZ_CUDA(cudaStreamSynchronize(s));
    if (timed) pool->timed_evals_host += (uint64_t)std::min(pool->h_counts[4], pool->dev.cap);
    return AZ_OK;
}
}  // namespace

extern "C" int az_selfplay_run(az_pool *pool, const char *output_path, int64_t target_games, int64_t target_positions,
                               double max_seconds, az_pool_stats *stats_out)
{
    AZ_REQUIRE(pool, AZ_ERR_ARG, "az_selfplay_run: null pool");
    AZ_REQUIRE(!pool->ctx_b, AZ_ERR_STATE, "az_selfplay_run: arena pools are driven by az_arena_play");
    AZ_REQUIRE(pool->cfg.auto_play, AZ_ERR_STATE, "az_selfplay_run: pool was created with auto_play = 0");
    AZ_REQUIRE(pool->cfg.eval_mode != AZ_EVAL_EXTERNAL, AZ_ERR_STATE, "az_selfplay_run: external evaluator pools are driven by collect/provide");
    AZ_REQUIRE(target_games > 0 || target_positions > 0 || max_seconds > 0, AZ_ERR_ARG, "az_selfplay_run: no stop condition");
    FILE *out = nullptr;
    if (output_path && output_path[0]) {
        out = fopen(output_path, "a");            // append mode, like std::ios_base::app (:691)
        if (!out) return az_fail(AZ_ERR_IO, "az_selfplay_run: cannot open '%s' for appending", output_path);
    }
    const auto t0 = std::chrono::steady_clock::now();
    const uint64_t pos0 = pool->written_positions;
    int64_t games = 0;
    int rc = AZ_OK;
    for (;;) {
        if ((rc = run_ticks(pool, out, true, kTicksPerDrain, &games))) break;
        const double elapsed = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        if (target_games > 0 && games >= target_games) break;
        if (target_positions > 0 && (int64_t)(pool->written_positions - pos0) >= target_positions) break;
        if (max_seconds > 0 && elapsed >= max_seconds) break;
        if ((pool->ticks & 1023) < (uint64_t)kTicksPerDrain && (rc = check_game_errors(pool))) break;
    }
    const int frc = finish_batches(pool);         // before the file is closed: the writer thread may still hold records
    if (out) fclose(out);
    if (rc) return rc;
    if (frc) return frc;
    if ((rc = check_game_errors(pool))) return rc;
    if (stats_out) return az_pool_stats_get(pool, stats_out);
    return AZ_OK;
}

extern "C" int az_selfplay_ticks(az_pool *pool, const char *output_path, int64_t ticks, az_pool_stats *stats_out)
{
    AZ_REQUIRE(pool && ticks >= 0, AZ_ERR_ARG, "az_selfplay_ticks: bad argument");
    AZ_REQUIRE(!pool->ctx_b, AZ_ERR_STATE, "az_selfplay_ticks: arena pools are driven by az_arena_play");
    AZ_REQUIRE(pool->cfg.auto_play, AZ_ERR_STATE, "az_selfplay_ticks: pool was created with auto_play = 0");
    AZ_REQUIRE(pool->cfg.eval_mode != AZ_EVAL_EXTERNAL, AZ_ERR_STATE, "az_selfplay_ticks: external evaluator pools are driven by collect/provide");
    FILE *out = nullptr;
    if (output_path && output_path[0]) {
        out = fopen(output_path, "a");
        if (!out) return az_fail(AZ_ERR_IO, "az_selfplay_ticks: cannot open '%s' for appending", output_path);
    }
    int rc = AZ_OK;
    int64_t games = 0;
    for (int64_t done = 0; done < ticks && rc == AZ_OK;) {
        const int chunk = (int)std::min<int64_t>(kTicksPerDrain, ticks - done);
        rc = run_ticks(pool, out, out != nullptr, chunk, &games);
        done += chunk;
    }
    const int frc = finish_batches(pool);         // before the file is closed: the writer thread may still hold records
    if (out) fclose(out);
    if (rc) return rc;
    if (frc) return frc;
    if ((rc = check_game_errors(pool))) return rc;
    if (stats_out) return az_pool_stats_get(pool, stats_out);
    return AZ_OK;
}

// ---------------------------------------------------------------------------------------------
// arena: two networks play each other, `slots` games at a time (az_tree.cu, arena_move / arena_receive)
// ---------------------------------------------------------------------------------------------
extern "C" int az_arena_create(az_context *ctx_a, az_context *ctx_b, const az_arena_config *cfg, az_pool **out)
{
    AZ_REQUIRE(ctx_a && ctx_b && cfg && out, AZ_ERR_ARG, "az_arena_create: null argument");
    *out = nullptr;
    AZ_REQUIRE(ctx_a->device == ctx_b->device, AZ_ERR_ARG, "az_arena_create: contexts on devices %d and %d", ctx_a->device, ctx_b->device);
    AZ_REQUIRE(cfg->slots >= 1 && cfg->slots <= (1 << 19), AZ_ERR_ARG, "az_arena_create: slots=%d", cfg->slots);
    for (int k = 0; k < 2; ++k)
        AZ_REQUIRE(cfg->visits[k] >= 1 && cfg->visits[k] <= (1 << 22), AZ_ERR_ARG, "az_arena_create: visits[%d]=%d", k, cfg->visits[k]);
    AZ_REQUIRE(cfg->eval_mode == AZ_NET_FP32 || cfg->eval_mode == AZ_NET_BF16 || cfg->eval_mode == AZ_NET_F16, AZ_ERR_ARG,
               "az_arena_create: eval_mode=%d", cfg->eval_mode);
    AZ_REQUIRE(ctx_a->net && ctx_b->net, AZ_ERR_STATE, "az_arena_create: no weights loaded in context %s (az_net_load)", ctx_a->net ? "b" : "a");
    az_pool_config pc{};
    pc.games = 2 * cfg->slots;
    pc.visits = cfg->visits[0];
    pc.max_plies = cfg->max_plies;
    pc.eval_mode = cfg->eval_mode;
    pc.node_capacity = cfg->node_capacity > 0 ? cfg->node_capacity : std::max(cfg->visits[0], cfg->visits[1]) + 64;
    az_pool *pool = nullptr;
    int rc = az_pool_create(ctx_a, &pc, &pool);
    if (rc) return rc;
    pool->ctx_b = ctx_b;
    PoolDev &D = pool->dev;
    const int S = cfg->slots;
    D.visits_b = cfg->visits[1];
    // each half is served in whole net rounds, as a self-play pool is (az_pool_create); both halves hold S trees on one
    // device, so they share the cap
    D.cap = S;
    if (cfg->eval_mode != AZ_NET_FP32) {
        const int round = az_net_pair_boards_per_round(ctx_a);
        if (S >= round) D.cap = S / round * round;
    }
    rc |= dev_alloc(&D.arena_slot_game, (size_t)S);
    rc |= dev_alloc(&D.mailbox, (size_t)D.G);
    rc |= dev_alloc(&D.arena_counters, 4);
    if (rc) { az_pool_destroy(pool); return rc; }
    *out = pool;
    return AZ_OK;
}

extern "C" int az_arena_play(az_pool *pool, const az_position *openings, int n, az_move *moves, int32_t *plies, int32_t *result,
                             az_pool_stats *stats_out)
{
    AZ_REQUIRE(pool && openings && moves && plies && result, AZ_ERR_ARG, "az_arena_play: null argument");
    AZ_REQUIRE(pool->ctx_b, AZ_ERR_STATE, "az_arena_play: not an arena pool (az_arena_create)");
    AZ_REQUIRE(n >= 1 && n <= (1 << 24), AZ_ERR_ARG, "az_arena_play: n=%d", n);
    std::vector<az_position> start(openings, openings + n);
    for (int j = 0; j < n; ++j) {
        AZ_REQUIRE(valid_position(start[j]) && (start[j].turn == 0 || start[j].turn == 1), AZ_ERR_ARG, "az_arena_play: opening %d is invalid", j);
        AZ_REQUIRE(az::board_result(start[j], nullptr) == 0, AZ_ERR_ARG, "az_arena_play: opening %d is already decided", j);
        start[j].ply = 0;                         // plies are counted from the opening
    }
    PoolDev &D = pool->dev;
    cudaStream_t s = pool->ctx->stream;
    const int S = D.G / 2, games = 2 * n, max_plies = D.max_plies;
    int rc = 0;
    az_position *d_openings = nullptr;
    rc |= dev_alloc(&d_openings, (size_t)n, false);
    D.openings = d_openings;
    rc |= dev_alloc(&D.arena_moves, (size_t)games * max_plies);
    rc |= dev_alloc(&D.arena_plies, (size_t)games);
    rc |= dev_alloc(&D.arena_result, (size_t)games);
    auto release = [&] {
        for (void *p : {(void *)d_openings, (void *)D.arena_moves, (void *)D.arena_plies, (void *)D.arena_result})
            if (p) cudaFree(p);
        D.openings = nullptr;
        D.arena_moves = nullptr;
        D.arena_plies = D.arena_result = nullptr;
    };
    if (rc) { release(); return rc; }
    D.arena_games = games;
    const int32_t counters[4] = {std::min(S, games), 0, 0, 0};
    cudaError_t e = cudaMemcpyAsync(d_openings, start.data(), sizeof(az_position) * n, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(D.arena_counters, counters, sizeof(counters), cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemsetAsync(D.mailbox, 0, sizeof(uint4) * D.G, s);
    if (e == cudaSuccess) {
        aztree_launch_arena_start(D, s);
        pool->launches++;
        e = cudaGetLastError();
    }
    // Ticks run in bursts (as in az_pool_run) and the finished-game counter is read once per burst.  A game lasts at most
    // max_plies moves of at most max(visits) evaluations each, and a request waits at most S / cap ticks for the net: the
    // bound on ticks only stops a pool that cannot make progress.
    const int64_t games_per_slot = (games + S - 1) / S;
    const int64_t max_ticks = 4 * games_per_slot * max_plies * (int64_t)(std::max(D.visits, D.visits_b) + 2) * ((S + D.cap - 1) / D.cap);
    int64_t ticks = 0;
    int burst = 1;
    while (e == cudaSuccess && rc == AZ_OK) {
        for (int k = 0; k < burst && rc == AZ_OK; ++k) {
            rc = launch_tree(pool);
            if (rc == AZ_OK) rc = launch_net(pool);
            pool->ticks++;
        }
        ticks += burst;
        if (rc) break;
        e = cudaMemcpyAsync(pool->h_counts, D.arena_counters, 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        if (e != cudaSuccess || pool->h_counts[1] >= games || pool->h_counts[2] > 0) break;
        if (ticks >= max_ticks) { rc = az_fail(AZ_ERR_STATE, "az_arena_play: %d of %d games finished after %lld ticks", pool->h_counts[1], games, (long long)ticks); break; }
        burst = std::min(2 * burst, 16);
    }
    if (e == cudaSuccess && rc == AZ_OK) e = cudaMemcpyAsync(moves, D.arena_moves, sizeof(az_move) * games * max_plies, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess && rc == AZ_OK) e = cudaMemcpyAsync(plies, D.arena_plies, sizeof(int32_t) * games, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess && rc == AZ_OK) e = cudaMemcpyAsync(result, D.arena_result, sizeof(int32_t) * games, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    release();
    if (e != cudaSuccess) return az_fail(AZ_ERR_CUDA, "az_arena_play: %s", cudaGetErrorString(e));
    if (rc) return rc;
    if ((rc = check_game_errors(pool))) return rc;
    if (stats_out) return az_pool_stats_get(pool, stats_out);
    return AZ_OK;
}

// ---------------------------------------------------------------------------------------------
// legacy ABI (link.py:8-32).  Process-global like the reference (self_play_client.cpp:591-602).
// thread_count == 2*buffer_entries (what accelerated_generate_games.py:70-77 passes): two halves of the pool play the
// role of the two fill buffers; get_workload() alternates between them, so while the caller evaluates buffer i the other
// half's answers can already be applied.  buffer_entries <= thread_count < 2*buffer_entries (the reference accepts any
// count up to 2*entries, :683-706, and needs at least `entries` workers to ever fill a buffer): ONE pool of thread_count
// games whose first buffer_entries requests are handed out per workload, the rest stay queued -- as in the reference,
// only one workload can then be outstanding at a time.
// ---------------------------------------------------------------------------------------------
namespace {
struct Legacy {
    az_context *ctx = nullptr;
    az_pool *half[2] = {nullptr, nullptr};       // single-pool mode: both point at the same pool
    bool single = false;
    float *fill[2] = {nullptr, nullptr};
    int entries = 0;
    int next = 0;
    FILE *out = nullptr;
    bool waiting[2] = {false, false};
    std::vector<float> staging;
} g_legacy;

void legacy_die(const char *what)
{
    // the reference aborts on failed asserts / exceptions; so do we, loudly
    fprintf(stderr, "libataxxzero legacy ABI: %s: %s\n", what, az_last_error());
    abort();
}
}  // namespace

extern "C" void launch_threads(char *output_path, int visits, float *fill_buffer1, float *fill_buffer2, int buffer_entries,
                               int thread_count)
{
    if (g_legacy.ctx) legacy_die("launch_threads called twice without shutdown");
    if (!fill_buffer1 || !fill_buffer2 || buffer_entries < 1 || thread_count < buffer_entries || thread_count > 2 * buffer_entries) {
        az_fail(AZ_ERR_ARG, "need two fill buffers and buffer_entries <= thread_count <= 2*buffer_entries (got %d entries, %d threads)",
                buffer_entries, thread_count);
        legacy_die("launch_threads");
    }
    const char *dev_env = getenv("AZ_DEVICE");
    if (az_create(dev_env ? atoi(dev_env) : 0, (uint64_t)std::chrono::steady_clock::now().time_since_epoch().count(), &g_legacy.ctx))
        legacy_die("az_create");
    printf("Launching into %p, %p with %d entries and %d threads.\n", (void *)fill_buffer1, (void *)fill_buffer2, buffer_entries,
           thread_count);
    printf("Writing to: %s\n", output_path);
    g_legacy.out = fopen(output_path, "a");
    if (!g_legacy.out) { az_fail(AZ_ERR_IO, "cannot open '%s'", output_path); legacy_die("launch_threads"); }
    g_legacy.fill[0] = fill_buffer1;
    g_legacy.fill[1] = fill_buffer2;
    g_legacy.entries = buffer_entries;
    g_legacy.next = 0;
    g_legacy.single = thread_count != 2 * buffer_entries;
    g_legacy.staging.resize((size_t)buffer_entries * AZ_FEATURES);
    for (int h = 0; h < (g_legacy.single ? 1 : 2); ++h) {
        az_pool_config cfg{};
        cfg.games = g_legacy.single ? thread_count : buffer_entries;
        cfg.visits = visits;
        cfg.max_plies = 400;
        cfg.noise = 1;
        cfg.auto_play = 1;
        cfg.eval_mode = AZ_EVAL_EXTERNAL;
        cfg.steps_per_tick = 64;
        cfg.seed = g_legacy.ctx->seed + 0x9E3779B97F4A7C15ULL * (h + 1);
        if (az_pool_create(g_legacy.ctx, &cfg, &g_legacy.half[h])) legacy_die("az_pool_create");
        g_legacy.half[h]->dev.cap = buffer_entries;      // a workload is exactly one fill buffer
        g_legacy.waiting[h] = false;
    }
    if (g_legacy.single) { g_legacy.half[1] = g_legacy.half[0]; g_legacy.waiting[1] = false; }
}

extern "C" int get_workload(void)
{
    if (!g_legacy.ctx) { az_fail(AZ_ERR_STATE, "launch_threads not called"); legacy_die("get_workload"); }
    const int h = g_legacy.next;
    if (g_legacy.waiting[h] || (g_legacy.single && g_legacy.waiting[h ^ 1])) {
        az_fail(AZ_ERR_STATE, g_legacy.single ? "thread_count < 2*buffer_entries: only one workload can be outstanding (the reference would block here)"
                                              : "buffer %d was handed out and not completed", h);
        legacy_die("get_workload");
    }
    az_pool *pool = g_legacy.half[h];
    // the reference hands out a buffer only when all `buffer_entries` slots are filled: every game of this
    // half must be blocked on an evaluation.  Games that end are restarted inside the tick, so this terminates.
    std::vector<float> &st = g_legacy.staging;
    int32_t have = 0;
    if (az_pool_collect(pool, st.data(), &have)) legacy_die("az_pool_collect");
    if (have != g_legacy.entries) {
        az_fail(AZ_ERR_STATE, "only %d of %d games requested an evaluation", have, g_legacy.entries);
        legacy_die("get_workload");
    }
    std::memcpy(g_legacy.fill[h], st.data(), sizeof(float) * AZ_FEATURES * (size_t)have);
    int64_t dummy = 0;
    if (drain_finished(pool, g_legacy.out, &dummy) || !pool->writer.flush()) legacy_die("drain");
    g_legacy.waiting[h] = true;
    g_legacy.next ^= 1;
    return h;
}

extern "C" void complete_workload(int workload, float *posteriors, float *values)
{
    if (!g_legacy.ctx || workload < 0 || workload > 1 || !g_legacy.waiting[workload]) {
        az_fail(AZ_ERR_STATE, "complete_workload(%d) without a matching get_workload", workload);
        legacy_die("complete_workload");
    }
    if (az_pool_provide(g_legacy.half[workload], posteriors, values)) legacy_die("az_pool_provide");
    g_legacy.waiting[workload] = false;
}

extern "C" void shutdown(void)
{
    if (!g_legacy.ctx) return;
    for (int h = 0; h < 2; ++h) {
        if (h == 0 || !g_legacy.single) az_pool_destroy(g_legacy.half[h]);
        g_legacy.half[h] = nullptr;
        g_legacy.waiting[h] = false;
    }
    if (g_legacy.out) fclose(g_legacy.out);
    g_legacy.out = nullptr;
    az_destroy(g_legacy.ctx);
    g_legacy.ctx = nullptr;                    // cleared so launch_threads may be called again (:744-748)
}

// ---------------------------------------------------------------------------------------------
// statistical test hooks (not in the public header; tests/test_rng_gpu.py): run the tick kernel's own Gamma sampler and
// its visit-proportional move sampler n times with independent counter-based streams.  Host pointers in and out.
// ---------------------------------------------------------------------------------------------
extern "C" int az_debug_gamma(az_context *ctx, double alpha, uint64_t seed, int n, double *out)
{
    AZ_REQUIRE(ctx && out && n > 0 && alpha > 0.0 && alpha < 1.0, AZ_ERR_ARG, "az_debug_gamma: bad argument");
    AZ_REQUIRE(ctx->scratch[0].reserve(sizeof(double) * (size_t)n) == 0, AZ_ERR_CUDA, "scratch alloc");
    aztree_launch_debug_gamma(alpha, seed, n, ctx->scratch[0].as<double>(), ctx->stream);
    ctx->launches++;
    AZ_CUDA(cudaMemcpyAsync(out, ctx->scratch[0].ptr, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    AZ_CUDA(cudaStreamSynchronize(ctx->stream));
    AZ_CUDA(cudaGetLastError());
    return AZ_OK;
}

// out[2i] = the tick kernel's straight-line exponential of x[i], out[2i+1] = exp((double)x[i]) (must be bit-identical)
extern "C" int az_debug_exp(az_context *ctx, const float *x, int n, double *out)
{
    AZ_REQUIRE(ctx && x && out && n > 0, AZ_ERR_ARG, "az_debug_exp: bad argument");
    AZ_REQUIRE(ctx->scratch[0].reserve(sizeof(float) * (size_t)n) == 0 && ctx->scratch[1].reserve(2 * sizeof(double) * (size_t)n) == 0,
               AZ_ERR_CUDA, "scratch alloc");
    AZ_CUDA(cudaMemcpyAsync(ctx->scratch[0].ptr, x, sizeof(float) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    aztree_launch_debug_exp(ctx->scratch[0].as<float>(), n, ctx->scratch[1].as<double>(), ctx->stream);
    ctx->launches++;
    AZ_CUDA(cudaMemcpyAsync(out, ctx->scratch[1].ptr, 2 * sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    AZ_CUDA(cudaStreamSynchronize(ctx->stream));
    AZ_CUDA(cudaGetLastError());
    return AZ_OK;
}

// in[4i..4i+3] = a1, b1, a2, b2; out[4i..4i+3] = the tick kernel's paired division (q1, q2), then a1/b1 and a2/b2 by the library
// puct != 0: the variant select_action runs (operands must be PUCT-shaped: a1 in [1, 2^12], b counts, a2 a score sum or 0)
extern "C" int az_debug_div(az_context *ctx, const double *in, int n, int puct, double *out)
{
    AZ_REQUIRE(ctx && in && out && n > 0, AZ_ERR_ARG, "az_debug_div: bad argument");
    const size_t bytes = 4 * sizeof(double) * (size_t)n;
    AZ_REQUIRE(ctx->scratch[0].reserve(bytes) == 0 && ctx->scratch[1].reserve(bytes) == 0, AZ_ERR_CUDA, "scratch alloc");
    AZ_CUDA(cudaMemcpyAsync(ctx->scratch[0].ptr, in, bytes, cudaMemcpyHostToDevice, ctx->stream));
    aztree_launch_debug_div(ctx->scratch[0].as<double>(), n, puct, ctx->scratch[1].as<double>(), ctx->stream);
    ctx->launches++;
    AZ_CUDA(cudaMemcpyAsync(out, ctx->scratch[1].ptr, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    AZ_CUDA(cudaStreamSynchronize(ctx->stream));
    AZ_CUDA(cudaGetLastError());
    return AZ_OK;
}

extern "C" int az_debug_sample_moves(az_context *ctx, const int32_t *visits, int n_moves, uint64_t seed, int n, int32_t *out)
{
    AZ_REQUIRE(ctx && visits && out && n > 0 && n_moves > 0 && n_moves < AZ_MAX_MOVES, AZ_ERR_ARG, "az_debug_sample_moves: bad argument");
    int64_t total = 0;
    for (int i = 0; i < n_moves; ++i) {
        AZ_REQUIRE(visits[i] >= 0, AZ_ERR_ARG, "az_debug_sample_moves: negative visit count");
        total += visits[i];
    }
    AZ_REQUIRE(total > 0 && total < (1 << 30), AZ_ERR_ARG, "az_debug_sample_moves: visit counts must sum to 1..2^30");
    AZ_REQUIRE(ctx->scratch[0].reserve(sizeof(int32_t) * (size_t)n_moves) == 0 && ctx->scratch[1].reserve(sizeof(int32_t) * (size_t)n) == 0,
               AZ_ERR_CUDA, "scratch alloc");
    AZ_CUDA(cudaMemcpyAsync(ctx->scratch[0].ptr, visits, sizeof(int32_t) * (size_t)n_moves, cudaMemcpyHostToDevice, ctx->stream));
    aztree_launch_debug_sample(ctx->scratch[0].as<int32_t>(), n_moves, (int)total, seed, n, ctx->scratch[1].as<int32_t>(), ctx->stream);
    ctx->launches++;
    AZ_CUDA(cudaMemcpyAsync(out, ctx->scratch[1].ptr, sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    AZ_CUDA(cudaStreamSynchronize(ctx->stream));
    AZ_CUDA(cudaGetLastError());
    return AZ_OK;
}
