// AZ_NVCC_FLAGS: -fmad=false
// az_net_pair.cu -- the bf16/f16 conv tower as tcgen05 implicit GEMMs on CTA PAIRS (cta_group::2), whole network in ONE
// persistent kernel (sm_100a).  Replaces TF1's sess.run of model.py:38-79 on the self-play hot path.
//
// Why pairs: a single-CTA kernel is paced by weight INGEST, not by the tensor pipe -- every CTA streams the whole 16-KiB
// weight stage of a (tap, 64 input channels) chunk into its own shared memory for 4 MMAs of 64 clocks, two CTAs per SM,
// and an SM takes in ~45 B/clk (DESIGN.md 3c).  Here the two CTAs of a cluster sit on the two SMs of a TPC and issue ONE
// M=256 MMA per step: each CTA holds its own 128 rows of activations (2 boards) and only HALF of the weight tile -- 64 of
// the 128 output channels, 8 KiB per stage; the tensor cores read the other half from the peer's shared memory.
//
// Geometry: a board is 64 GEMM rows (row 8 + 8x + y holds cell (x, y); y == 7 and rows 0..7 are zero padding), so a 3x3
// tap is a CONSTANT ROW SHIFT of the same activation buffer and im2col is never built.  Activations stay in shared memory
// for all 25 layers in the no-swizzle K-major UMMA layout; the fp32 accumulator and the fp32 residual stream live in TMEM
// (the second conv of a block accumulates on top of the residual); weights (BN scale folded) are pre-tiled in HBM as the
// exact shared-memory image of a stage and streamed by 1-D bulk TMA copies; a layer starts on the first input-channel
// half while the previous epilogue still writes the second.  Roles per CTA: warp 0 = TMA producer (its own half of every
// stage), warp 1 = MMA issuer in the LEADER (cluster rank 0) / relay in the peer, warps 2-5 = epilogue, and in the
// speculative cache pass warp 6 = softmax helper.
// The peer's relay warp (one lane per barrier) forwards completions: whenever one of the peer's own barriers completes
// (weights landed, activations written, input staged) it arrives on the leader's barrier of the same name, so the one
// issuing thread sees "both halves ready" as a single barrier phase.  tcgen05.commit multicasts completions back to both CTAs.
#include "az_net.h"
#include "az_rules.cuh"

#include <algorithm>
#include <cstdlib>
#include <type_traits>

namespace {

constexpr int F = AZ_F;
constexpr int KG = F / 8;                // 16 k-groups of 8 channels
constexpr int TILE_M = 128;              // GEMM rows per CTA (2 boards x 64)
constexpr int MARGIN = 16;
constexpr int ROW_BYTES = 16;
constexpr int SPLIT = 2;                 // input-channel parts per layer (early release after the first)
constexpr int PART_KG = KG / SPLIT;      // 8 k-groups per chunk
constexpr int PART_MMAS = PART_KG / 2;   // 4 K=16 steps per chunk
constexpr int HALF_N = F / 2;            // output channels whose weights live in THIS CTA
constexpr int STAGE_BYTES = PART_KG * HALF_N * ROW_BYTES;      // 8 KiB: one tap x 64 input channels x 64 output channels
constexpr int CHUNK_BYTES = 2 * STAGE_BYTES;                   // both halves of a chunk, as laid out in HBM
constexpr int CHUNKS = SPLIT * 9;
constexpr int W_LBO = HALF_N * ROW_BYTES;                      // 1024: bytes between k-groups of this CTA's B half
constexpr int WIN_KSTEP_BYTES = 2 * HALF_N * ROW_BYTES;        // one K=16 step of the input conv (two taps), this half: 2 KiB
constexpr int WIN_HALF_BYTES = 5 * WIN_KSTEP_BYTES;            // 10 KiB
constexpr int WIN_KSTEPS_PER_STAGE = STAGE_BYTES / WIN_KSTEP_BYTES;     // 4
constexpr int HEAD_N = 32;               // 17 policy planes + 1 value plane, padded
constexpr int HEAD_HALF = HEAD_N / 2;
constexpr int WHEAD_HALF_BYTES = KG * HEAD_HALF * ROW_BYTES;   // 4 KiB
constexpr int HEAD_LBO = HEAD_HALF * ROW_BYTES;

constexpr int ACT_ROWS = MARGIN + TILE_M + MARGIN;
constexpr int ACT_LBO = ACT_ROWS * ROW_BYTES;
constexpr int ACT_BYTES = KG * ACT_LBO;  // one tile's activations; its input planes are staged in k-group 0
constexpr uint32_t TM_ACC = 0, TM_RES = 128, TM_TILE = 256;    // per tile: accumulator + residual columns
constexpr int ACC = 0, ACT = 1, IN = 1 + SPLIT, TILE_BARS = 2 + SPLIT;   // per-tile barriers: accumulator, activation parts, input

// Pass kinds.  PLAIN: logits and values of a batch of boards; PROF: the same, with the issuer's wait records
// (az_net_pair_profile).  The other three run the one-tile schedule only:
//   CACHE: the speculative search's pass -- no logits; the values, the softmax numerators exp((double)logit) and their
//          strictly sequential sum, all through an output map.  The head epilogue writes the numerators and a helper warp
//          adds them up while the epilogue already works on the CTA's next unit: 833 double exponentials and an 833-long
//          chain of double additions per leaf would otherwise saturate the fp64 pipes of the latency-bound tree kernel.
//   SYM8:  the symmetry ensemble (nn_evals.py:48-62): each CTA evaluates one position at a time, its 8 dihedral images in
//          4 passes of 2, generated while the input is staged and averaged in the head epilogue.
//   TOWER: the first P.layers convs only, no heads; the last one's fp32 activations go to P.debug_act (az_net_debug_tower).
enum : int { K_PLAIN = 0, K_PROF = 1, K_CACHE = 2, K_SYM8 = 3, K_TOWER = 4 };
constexpr int SYM_BYTES = 3392;          // CACHE: the helper warp's staging; SYM8: float[833] policy sum + float[8] values

// TILES = 1: two CTAs (two unrelated pairs) per SM, one 128-row tile each.  TILES = 2: one CTA per SM with two tiles that
// consume every weight stage one after the other, so that each tile's epilogue runs behind the other tile's MMAs (see the issuer).
template <int TILES, int KIND = K_PLAIN>
struct PairCfg {
    static constexpr int STAGES = 8 * TILES;                    // TILES = 2: a stage stays live for 9 chunks of tile 0
    static constexpr int OFF_ACT = 0;                           // one activation buffer per tile
    static constexpr int OFF_RING = OFF_ACT + TILES * ACT_BYTES;
    static constexpr int OFF_SHIFT = OFF_RING + STAGES * STAGE_BYTES;   // float[TILES][2][F]
    static constexpr int OFF_VPART = OFF_SHIFT + TILES * 2 * F * 4;     // float[TILES][16]
    static constexpr int OFF_BAR = OFF_VPART + TILES * 64;
    static constexpr int B_FULL = 0, B_EMPTY = STAGES, B_TILE = 2 * STAGES;
    static constexpr int NUM_BARS = B_TILE + TILES * TILE_BARS;
    static constexpr int OFF_TMEM = OFF_BAR + NUM_BARS * 8;
    static constexpr int OFF_SYM = OFF_TMEM + 16;               // CACHE, SYM8 and TOWER only
    static constexpr int SMEM_BYTES = OFF_SYM + (KIND >= K_CACHE ? SYM_BYTES : 0);
    static constexpr int NUM_WARPS = 2 + 4 * TILES + (KIND == K_CACHE ? 1 : 0);   // producer, issuer / relay, 4 epilogue warps per tile, helper
    static constexpr int HELPER_WARP = 2 + 4 * TILES;
    static constexpr int NUM_THREADS = NUM_WARPS * 32;
    static constexpr int UNIT_BOARDS = 2 * TILES;
    static constexpr int CTAS_PER_SM = TILES == 1 ? 2 : 1;
    static constexpr uint32_t TMEM_COLS = TM_TILE * TILES;
};
static_assert(PairCfg<1>::SMEM_BYTES * 2 + 2048 <= 228 * 1024, "two CTAs per SM");
static_assert(PairCfg<1, K_CACHE>::SMEM_BYTES * 2 + 2048 <= 228 * 1024, "two CTAs per SM with the staging / sym8 area");
static_assert(PairCfg<1>::OFF_SYM % 16 == 0, "the staging area holds doubles");
static_assert(PairCfg<2>::SMEM_BYTES + 1024 <= 228 * 1024, "one two-tile CTA per SM");
static_assert(PairCfg<2>::STAGES - 9 >= 4, "the ring must prefetch while a part's nine stages wait for the second tile");

// instruction descriptor: D=f32, A/B bf16 (bits 7, 10; cleared for IEEE half), K-major both, N >> 3 at bit 17, M >> 4 at bit 24.
// M is the PAIR's: 256.
constexpr uint32_t make_idesc(int n, bool f16) { return (1u << 4) | (f16 ? 0u : ((1u << 7) | (1u << 10))) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(256 >> 4) << 24); }

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count)); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// arrive on the barrier at the same shared-memory offset in CTA `rank` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint32_t bar, uint32_t rank)
{
    uint32_t remote;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(bar), "r"(rank));
    asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    uint32_t done;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    } while (!done);
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank()
{
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all()
{
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t cols)
{
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols)
{
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// no-swizzle K-major shared-memory matrix descriptor (SBO = 128 B: 8-row core matrices are contiguous)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes)
{
    return (uint64_t)((saddr >> 4) & 0x3fff) | ((uint64_t)((lbo_bytes >> 4) & 0x3fff) << 16) | ((uint64_t)(128 >> 4) << 32) | (1ULL << 46);
}
__device__ __forceinline__ void umma2(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem), "l"(adesc),
                 "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma2_lo(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc, uint32_t accumulate)
{
    asm volatile("{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tmov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\tsetp.ne.b32 p, %6, 0;\n\t"
                 "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %5, p;\n\t}" ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc),
                 "r"(accumulate) : "memory");
}
__device__ __forceinline__ bool elect_one()
{
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
// arrive on the barrier at this offset in BOTH CTAs of the pair once the MMAs issued so far have completed
__device__ __forceinline__ void umma2_commit(uint32_t bar)
{
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32])
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
                   "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
                   "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]),
                   "=r"(r[31])
                 : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32])
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
                 "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
                 "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
                 "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]),
                 "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]),
                 "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
                 : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ uint32_t pack_op(float lo, float hi, int f16)
{
    if (f16) { __half2 v = __floats2half2_rn(lo, hi); return *reinterpret_cast<uint32_t *>(&v); }
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t *>(&v);
}
// the 128 epilogue threads of one tile (immediate barrier ids: a register operand would reserve all 16 barriers)
__device__ __forceinline__ void group_sync(int tile)
{
    if (tile == 0) asm volatile("bar.sync 1, 128;" ::: "memory");
    else asm volatile("bar.sync 2, 128;" ::: "memory");
}
// CACHE: the 128 epilogue threads -> the softmax helper warp, "the numerators of this unit are written"
__device__ __forceinline__ void helper_arrive() { asm volatile("bar.arrive 3, 160;" ::: "memory"); }
__device__ __forceinline__ void helper_wait() { asm volatile("bar.sync 3, 160;" ::: "memory"); }

// exp((double)logit) exactly as the tree kernel computes it (az_tree.cu populate_from_eval): same libdevice routine, same
// compiler flags (no fused multiply-add contraction in either file).  Not inlined: 17 calls per epilogue thread and unit.
__device__ __noinline__ double exp_d(float x) { return exp((double)x); }

// nn_evals.apply_symmetry (nn_evals.py:7-15): image[i][j] = board[a'][b'] with (a, b) = sym&4 ? (j, i) : (i, j),
// b' = sym&2 ? 6-b : b, a' = sym&1 ? 6-a : a.  The same map takes an image cell to the board cell its policy belongs to
// when the image was made with `sym` (applying inverse_symmetry[sym] to the output, nn_evals.py:27,58-61, undoes it).
__device__ __forceinline__ int sym_cell(int sym, int i, int j)
{
    int a = (sym & 4) ? j : i, b = (sym & 4) ? i : j;
    if (sym & 2) b = 6 - b;
    if (sym & 1) a = 6 - a;
    return a * 7 + b;
}

struct PairParams {
    const void *input;                 // float[n][196] or az_position[n]
    int n;
    const int *n_ptr;                  // when non-null the board count is read from device memory
    int layers;                        // 1 + 2*blocks (TOWER: the conv layers to run)
    const uint8_t *w_stream;           // pair tiling: [input conv 2 x 10 KiB][2*blocks x 18 chunks x 2 x 8 KiB][heads 2 x 4 KiB]
    const float *shift;                // [layers][128]
    const float *fc_w, *fc_b;
    float *logits, *values;
    int f16;
    long long *prof;                   // issuer wait records (K_PROF only, see az_net_pair_profile)
    int prof_max;                      // records per CTA
};
// the parameters of CACHE, SYM8 and TOWER (PLAIN and PROF keep the smaller block: its size alone changes their code)
struct PairParamsX : PairParams {
    const int *out_map;                // CACHE: when non-null, the outputs of board b go to row out_map[b] of values / exps / totals
    double *exps;                      // CACHE: [rows][833] exp((double)logit)
    double *totals;                    // CACHE: [rows] their strictly sequential sum
    float *debug_act;                  // TOWER: [n][49][128] the last conv layer's fp32 activations
};
template <int KIND>
using PairParamsOf = std::conditional_t<(KIND >= K_CACHE), PairParamsX, PairParams>;

// Issuer wait records of the profiling instantiation: per CTA a header {smid, clock at start, clock at end, records} and records
// {kind + 256 * layer, t0, t1} in clock64() cycles.  Layer 0 is the input conv, 1..nl the tower, nl + 1 the heads.
enum : int { PROF_GAP = 0, PROF_ACT0 = 1, PROF_ACT1 = 2, PROF_FULL = 3, PROF_IN = 4, PROF_UNIT_GAP = 5 };
constexpr int PROF_HDR = 4;

__device__ __forceinline__ bool row_is_real(int r, int &board_in_tile, int &cell)
{
    board_in_tile = r >> 6;
    const int w = r & 63;
    const int x = (w >> 3) - 1, y = w & 7;
    cell = x * 7 + y;
    return w >= 8 && y != 7;
}

template <int TILES, int IN_KIND, int KIND>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(PairCfg<TILES, KIND>::NUM_THREADS, PairCfg<TILES, KIND>::CTAS_PER_SM) k_net_pair(const PairParamsOf<KIND> P)
{
    using C = PairCfg<TILES, KIND>;
    constexpr int STAGES = C::STAGES, NUM_THREADS = C::NUM_THREADS, UNIT_BOARDS = C::UNIT_BOARDS;
    constexpr int OFF_ACT = C::OFF_ACT, OFF_RING = C::OFF_RING, B_FULL = C::B_FULL, B_EMPTY = C::B_EMPTY;
    constexpr bool PROF = KIND == K_PROF, HEADS = KIND != K_TOWER;
    static_assert(KIND == K_PLAIN || TILES == 1, "wait records and the other pass kinds are taken for the one-tile schedule");
    // SYM8: a work item is one position, 4 passes of 2 images; every other kind: one unit of UNIT_BOARDS boards, one pass.
    // Producer, issuer and relay walk the chunk sequence once per pass.
    constexpr int PASSES = KIND == K_SYM8 ? 8 / UNIT_BOARDS : 1;
    const uint32_t crank = cluster_ctarank();
    const bool leader = crank == 0;
    extern __shared__ __align__(1024) uint8_t smem[];
    const uint32_t sbase = smem_u32(smem);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    auto bar = [&](int i) { return sbase + C::OFF_BAR + 8 * i; };
    auto tbar = [&](int tile, int i) { return bar(C::B_TILE + tile * TILE_BARS + i); };     // per-tile barrier i (ACC, ACT + part, IN)

    const int n_boards = P.n_ptr ? min(*P.n_ptr, P.n) : P.n;
    const int items = KIND == K_SYM8 ? n_boards : (n_boards + UNIT_BOARDS - 1) / UNIT_BOARDS;
    const int num_units = (items + 1) / 2 * 2;      // both CTAs of a pair run the same passes
    const int nl = P.layers - 1;                    // 128 -> 128 convs
    const uint32_t idesc_128 = make_idesc(128, P.f16 != 0), idesc_head = make_idesc(HEAD_N, P.f16 != 0);

    // ---- one-time setup ----
    for (int i = threadIdx.x; i < TILES * ACT_BYTES / 16; i += NUM_THREADS) reinterpret_cast<uint4 *>(smem + OFF_ACT)[i] = make_uint4(0, 0, 0, 0);
    if (threadIdx.x == 0) {
        // barriers the issuing thread waits on count the peer's relay as one more arrival (leader only)
        const uint32_t extra = leader ? 1u : 0u;
        for (int s = 0; s < STAGES; ++s) { mbar_init(bar(B_FULL + s), 1 + extra); mbar_init(bar(B_EMPTY + s), 1); }
        for (int t = 0; t < TILES; ++t) {
            mbar_init(tbar(t, ACC), 1);
            for (int p = 0; p < SPLIT; ++p) mbar_init(tbar(t, ACT + p), 128 + extra);
            mbar_init(tbar(t, IN), 128 + extra);
        }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(sbase + C::OFF_TMEM, C::TMEM_COLS);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                  // the peer's barriers and zero-filled activations exist before anything refers to them
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t *>(smem + C::OFF_TMEM);

    // chunk sequence of one unit (identical in producer, issuer and relay): input conv (2 stages), nl x 18 tower chunks, heads
    if (warp == 0) {
        // =============================== TMA producer: this CTA's half of every stage ===============================
        if (lane == 0) {
            uint32_t it = 0;
            auto push = [&](const uint8_t *src, uint32_t bytes) {
                const int s = it % STAGES;
                mbar_wait(bar(B_EMPTY + s), ((it / STAGES) & 1) ^ 1);
                mbar_expect_tx(bar(B_FULL + s), bytes);
                bulk_g2s(sbase + OFF_RING + s * STAGE_BYTES, src, bytes, bar(B_FULL + s));
                ++it;
            };
            const uint8_t *win = P.w_stream + crank * WIN_HALF_BYTES;
            const uint8_t *tower = P.w_stream + 2 * WIN_HALF_BYTES + crank * STAGE_BYTES;
            const uint8_t *head_w = P.w_stream + 2 * WIN_HALF_BYTES + (size_t)nl * CHUNKS * CHUNK_BYTES + crank * WHEAD_HALF_BYTES;
            for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x)
            for (int pass = 0; pass < PASSES; ++pass) {
                for (int j0 = 0; j0 < 5; j0 += WIN_KSTEPS_PER_STAGE)
                    push(win + j0 * WIN_KSTEP_BYTES, min(WIN_KSTEPS_PER_STAGE, 5 - j0) * WIN_KSTEP_BYTES);
                for (int c = 0; c < nl * CHUNKS; ++c) push(tower + (size_t)c * CHUNK_BYTES, STAGE_BYTES);
                if (HEADS) push(head_w, WHEAD_HALF_BYTES);
            }
        }
    } else if (warp == 1 && !leader) {
        // =============================== relay (peer): forward "my half is ready" to the leader ===============================
        int my_units = 0;
        for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) my_units += PASSES;      // counts passes
        const int pushes_per_unit = (5 + WIN_KSTEPS_PER_STAGE - 1) / WIN_KSTEPS_PER_STAGE + nl * CHUNKS + (HEADS ? 1 : 0);
        // every barrier is its own event stream with self-consistent phases: one lane per stream, so that a slow hop on one
        // of them never delays the others (the weight stages; per tile the two activation parts and the staged input)
        static_assert(STAGES + TILES * (SPLIT + 1) <= 32, "one relay lane per event stream");
        if (lane < STAGES) {
            const uint32_t total = (uint32_t)my_units * (uint32_t)pushes_per_unit;
            for (uint32_t it = lane; it < total; it += STAGES) {
                mbar_wait(bar(B_FULL + lane), (it / STAGES) & 1);
                mbar_arrive_remote(bar(B_FULL + lane), 0);
            }
        } else if (lane < STAGES + TILES * (SPLIT + 1)) {
            const int tile = (lane - STAGES) / (SPLIT + 1), k = (lane - STAGES) % (SPLIT + 1);     // k < SPLIT: part k, else input
            const uint32_t b = tbar(tile, k < SPLIT ? ACT + k : IN);
            const uint32_t total = (uint32_t)my_units * (uint32_t)(k < SPLIT ? nl + 1 : 1);
            for (uint32_t e = 0; e < total; ++e) {
                mbar_wait(b, e & 1);
                mbar_arrive_remote(b, 0);
            }
        }
    } else if (warp == 1) {
        // =============================== MMA issuer (leader): one M=256 MMA per step for the pair ===============================
        // TILES = 2: the tiles take every weight stage one after the other -- per layer t0.part0, t1.part0, t0.part1, t1.part1 --
        // so tile 1 runs half a layer behind tile 0.  Tile 0's epilogue of layer l then runs behind t1.part1(l), and t0.part0(l+1)
        // needs only its first half; tile 1's epilogue runs behind t0.part0(l+1) in the same way.  A stage is freed after the last
        // tile's MMAs on it (9 chunks after the first tile's), hence the 16-stage ring.  Per tile, the operands, the chunk order
        // and the accumulation are those of TILES = 1: the results are identical bit for bit.
        if (elect_one()) {
            uint32_t it = 0, in_phase = 0, act_phase = 0;
            // PROF: the issuer also waits for each accumulator commit before the wait that follows it anyway, to time the
            // stretch in which this pair has no MMA queued ("gap": accumulator done -> next layer's first input part ready)
            long long *rec = PROF ? P.prof + (size_t)blockIdx.x * (PROF_HDR + 3 * P.prof_max) : nullptr;
            int nrec = 0;
            uint32_t acc_ph = 0;
            long long t_acc = 0, full_sum = 0;
            auto note = [&](int kind, int layer, long long t0, long long t1) {
                if (PROF && nrec < P.prof_max) {
                    rec[PROF_HDR + 3 * nrec] = kind + 256 * layer; rec[PROF_HDR + 3 * nrec + 1] = t0; rec[PROF_HDR + 3 * nrec + 2] = t1;
                    ++nrec;
                }
            };
            auto acc_done = [&]() {
                if (PROF) { mbar_wait(tbar(0, ACC), acc_ph); acc_ph ^= 1; t_acc = clock64(); }
            };
            auto full_wait = [&](int s, uint32_t parity) {
                const long long t0 = PROF ? clock64() : 0;
                mbar_wait(bar(B_FULL + s), parity);
                if (PROF) full_sum += clock64() - t0;
            };
            if (PROF) { uint32_t smid; asm volatile("mov.u32 %0, %%smid;" : "=r"(smid)); rec[0] = smid; rec[1] = clock64(); t_acc = rec[1]; }
            auto acquire = [&]() {
                const int s = it % STAGES;
                full_wait(s, (it / STAGES) & 1);
                tc_fence_after();
                return sbase + OFF_RING + s * STAGE_BYTES;
            };
            auto release = [&]() { umma2_commit(bar(B_EMPTY + it % STAGES)); ++it; };
            const uint32_t a_hi = (uint32_t)(make_desc(0, ACT_LBO) >> 32), b_hi = (uint32_t)(make_desc(0, W_LBO) >> 32);
            const uint32_t a_lo0 = (uint32_t)make_desc(sbase + OFF_ACT + MARGIN * ROW_BYTES, ACT_LBO);
            const uint32_t b_lo0 = (uint32_t)make_desc(sbase + OFF_RING, W_LBO);
            constexpr uint32_t A_KSTEP = (2 * ACT_LBO) >> 4, B_KSTEP = (2 * W_LBO) >> 4, A_PART = (PART_KG * ACT_LBO) >> 4, A_TILE = ACT_BYTES >> 4;
            // every pass of every unit of this CTA as one loop: nothing below depends on the pass, and a nested loop over
            // PASSES = 1 would change how the plain kinds are scheduled
            for (int unit = blockIdx.x, pass = 0; unit < num_units; pass = pass + 1 < PASSES ? pass + 1 : 0, unit += pass ? 0 : gridDim.x) {
                // ---- input conv: 9 taps x 8 (4 real) channels, two taps per K=16 step ----
                for (int j0 = 0; j0 < 5; j0 += WIN_KSTEPS_PER_STAGE) {
                    const uint32_t b_rows = acquire();
                    const int j1 = min(j0 + WIN_KSTEPS_PER_STAGE, 5);
#pragma unroll
                    for (int t = 0; t < TILES; ++t) {
                        if (j0 == 0) {
                            const long long t0 = PROF ? clock64() : 0;
                            mbar_wait(tbar(t, IN), in_phase);
                            if (PROF) { const long long t1 = clock64(); note(PROF_IN, 0, t0, t1); note(PROF_UNIT_GAP, 0, t_acc, t1); }
                            tc_fence_after();
                        }
                        const uint32_t in_rows = sbase + OFF_ACT + t * ACT_BYTES + MARGIN * ROW_BYTES;
                        for (int j = j0; j < j1; ++j) {
                            const int tap0 = 2 * j, tap1 = 2 * j + 1;
                            const uint32_t a0 = in_rows + ((tap0 / 3 - 1) * 8 + (tap0 % 3 - 1)) * ROW_BYTES;
                            const uint32_t a1 = tap1 < 9 ? in_rows + ((tap1 / 3 - 1) * 8 + (tap1 % 3 - 1)) * ROW_BYTES : a0 + ROW_BYTES;   // 10th tap: zero weights
                            umma2(tmem_base + t * TM_TILE + TM_ACC, make_desc(a0, a1 - a0), make_desc(b_rows + (j - j0) * 2 * W_LBO, W_LBO), idesc_128, j > 0);
                        }
                        if (j1 == 5) umma2_commit(tbar(t, ACC));
                    }
                    release();
                }
                in_phase ^= 1;
                // ---- tower ----
                for (int l = 0; l < nl; ++l) {
                    const uint32_t onto_res = (uint32_t)(l & 1);        // second conv of a block: on top of the residual columns
                    if (PROF) { note(PROF_FULL, l, 0, full_sum); full_sum = 0; acc_done(); }
#pragma unroll 1
                    for (int part = 0; part < SPLIT; ++part) {
#pragma unroll
                        for (int t = 0; t < TILES; ++t) {
                            const uint32_t d_col = tmem_base + t * TM_TILE + (onto_res ? TM_RES : TM_ACC);
                            {
                                const long long t0 = PROF ? clock64() : 0;
                                mbar_wait(tbar(t, ACT + part), act_phase);
                                if (PROF) {
                                    const long long t1 = clock64();
                                    note(part ? PROF_ACT1 : PROF_ACT0, l + 1, t0, t1);
                                    if (part == 0) note(PROF_GAP, l + 1, t_acc, t1);
                                }
                            }
                            tc_fence_after();
#pragma unroll
                            for (int tap = 0; tap < 9; ++tap) {
                                const int s = (it + tap) % STAGES;
                                if (t == 0) {           // the later tiles find the stage landed
                                    full_wait(s, ((it + tap) / STAGES) & 1);
                                    tc_fence_after();
                                }
                                const uint32_t b_lo = b_lo0 + s * (STAGE_BYTES >> 4);
                                const uint32_t a_lo = a_lo0 + t * A_TILE + part * A_PART + (uint32_t)((tap / 3 - 1) * 8 + (tap % 3 - 1));
#pragma unroll
                                for (int j = 0; j < PART_MMAS; ++j)
                                    umma2_lo(d_col, a_lo + j * A_KSTEP, a_hi, b_lo + j * B_KSTEP, b_hi, idesc_128, onto_res | (uint32_t)((part | tap | j) != 0));
                                if (part == SPLIT - 1 && tap == 8) umma2_commit(tbar(t, ACC));
                                if (t == TILES - 1) umma2_commit(bar(B_EMPTY + s));
                            }
                        }
                        it += 9;
                    }
                    act_phase ^= 1;
                }
                // ---- heads: [256 rows x 128 ch] x [128 ch x 32] ----
                if (PROF) { note(PROF_FULL, nl, 0, full_sum); full_sum = 0; acc_done(); }
                if (!HEADS) {
                    // TOWER: no heads; the last layer's activations are still awaited, which keeps act_phase in step
                    for (int p = 0; p < SPLIT; ++p) mbar_wait(tbar(0, ACT + p), act_phase);
                } else {
                    uint32_t b_rows = 0;
#pragma unroll
                    for (int t = 0; t < TILES; ++t) {
                        {
                            const long long t0 = PROF ? clock64() : 0;
                            for (int p = 0; p < SPLIT; ++p) mbar_wait(tbar(t, ACT + p), act_phase);
                            if (PROF) { const long long t1 = clock64(); note(PROF_ACT0, nl + 1, t0, t1); note(PROF_GAP, nl + 1, t_acc, t1); }
                        }
                        tc_fence_after();
                        if (t == 0) b_rows = acquire();
                        const uint32_t a_rows = sbase + OFF_ACT + t * ACT_BYTES + MARGIN * ROW_BYTES;
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                            umma2(tmem_base + t * TM_TILE + TM_ACC, make_desc(a_rows + 2 * j * ACT_LBO, ACT_LBO), make_desc(b_rows + 2 * j * HEAD_LBO, HEAD_LBO),
                                  idesc_head, j > 0);
                        umma2_commit(tbar(t, ACC));
                    }
                    release();
                }
                act_phase ^= 1;
                if (PROF) { note(PROF_FULL, nl + 1, 0, full_sum); full_sum = 0; acc_done(); }
            }
            if (PROF) { rec[2] = clock64(); rec[3] = nrec; }
        }
    } else if (KIND == K_CACHE && warp == C::HELPER_WARP) {
        if constexpr (KIND == K_CACHE) {
            // =============================== softmax helper (CACHE) ===============================
            // total = sum_i exp(logit_i), i ascending, added one by one in double (self_play_client.cpp:212-214): one lane per
            // board of the unit the epilogue warps have just finished; they are already working on the next one.
            // All 32 lanes fetch the numerators chunk by chunk (coalesced, the next chunk in flight while the current one is
            // being added) into a small shared-memory stage; lane b then walks board b's chunk in order.
            constexpr int CH = 96;                                  // doubles per board and chunk: 3 per lane
            constexpr int NCH = (AZ_LOGITS + CH - 1) / CH;
            double *stage = reinterpret_cast<double *>(smem + C::OFF_SYM);       // [UNIT_BOARDS][CH]
            static_assert(UNIT_BOARDS * CH * 8 <= SYM_BYTES, "softmax stage fits the staging area");
            for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
                helper_wait();
                const double *e[UNIT_BOARDS];
                int ob[UNIT_BOARDS];
#pragma unroll
                for (int b = 0; b < UNIT_BOARDS; ++b) {
                    const int board = unit * UNIT_BOARDS + b;
                    ob[b] = board < n_boards ? (P.out_map ? __ldg(P.out_map + board) : board) : -1;
                    e[b] = P.exps + (size_t)max(ob[b], 0) * AZ_LOGITS;
                }
                double v[UNIT_BOARDS][3];
                auto fetch = [&](int c) {
#pragma unroll
                    for (int b = 0; b < UNIT_BOARDS; ++b)
#pragma unroll
                        for (int j = 0; j < 3; ++j) {
                            const int i = c * CH + lane + 32 * j;
                            v[b][j] = (ob[b] >= 0 && i < AZ_LOGITS) ? __ldcg(e[b] + i) : 0.0;
                        }
                };
                double total = 0.0;
                fetch(0);
#pragma unroll 1
                for (int c = 0; c < NCH; ++c) {
#pragma unroll
                    for (int b = 0; b < UNIT_BOARDS; ++b)
#pragma unroll
                        for (int j = 0; j < 3; ++j) stage[b * CH + lane + 32 * j] = v[b][j];
                    __syncwarp();
                    if (c + 1 < NCH) fetch(c + 1);
                    if (lane < UNIT_BOARDS) {
                        const double *row = stage + lane * CH;
                        const int count = min(CH, AZ_LOGITS - c * CH);
                        int i = 0;
                        for (; i + 8 <= count; i += 8) {
                            const double2 a = *reinterpret_cast<const double2 *>(row + i), b2 = *reinterpret_cast<const double2 *>(row + i + 2);
                            const double2 c2 = *reinterpret_cast<const double2 *>(row + i + 4), d2 = *reinterpret_cast<const double2 *>(row + i + 6);
                            total = __dadd_rn(total, a.x); total = __dadd_rn(total, a.y);
                            total = __dadd_rn(total, b2.x); total = __dadd_rn(total, b2.y);
                            total = __dadd_rn(total, c2.x); total = __dadd_rn(total, c2.y);
                            total = __dadd_rn(total, d2.x); total = __dadd_rn(total, d2.y);
                        }
                        for (; i < count; ++i) total = __dadd_rn(total, row[i]);
                    }
                    __syncwarp();
                }
                if (lane < UNIT_BOARDS) {
                    int mine = -1;
#pragma unroll
                    for (int b = 0; b < UNIT_BOARDS; ++b) mine = lane == b ? ob[b] : mine;
                    if (mine >= 0) P.totals[mine] = total;
                }
            }
        }
    } else {
        // =============================== epilogue warps (both CTAs, each on its own 128 TMEM lanes of its tile) ===============================
        const int tile = TILES == 1 ? 0 : (warp - 2) >> 2;
        const int quad = warp & 3;               // a warp reaches TMEM lanes 32 * (warp % 4) ..
        const int r = quad * 32 + lane;
        const int gtid = ((warp - 2) & 3) * 32 + lane;
        int bit, cell;
        const bool real = row_is_real(r, bit, cell);
        float *shift_base = reinterpret_cast<float *>(smem + C::OFF_SHIFT) + tile * 2 * F;
        float *vpart = reinterpret_cast<float *>(smem + C::OFF_VPART) + tile * 16;
        const uint32_t lane_addr = tmem_base + tile * TM_TILE + ((uint32_t)(quad * 32) << 16);
        uint8_t *act_row = smem + OFF_ACT + tile * ACT_BYTES + (MARGIN + r) * ROW_BYTES;
        uint32_t acc_phase = 0;
        // "this row's part of the activations is written": locally, and -- in the leader -- that is all; the peer's relay
        // thread forwards the completed phase
        float *sym_acc = reinterpret_cast<float *>(smem + C::OFF_SYM);      // SYM8: policy sum [833], then the 8 values
        for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x)
        for (int pass = 0; pass < PASSES; ++pass) {
            // SYM8: position `unit`, image sym = pass * UNIT_BOARDS + (row's board in the unit); otherwise the unit's boards
            const int sym = KIND == K_SYM8 ? pass * UNIT_BOARDS + tile * 2 + bit : 0;
            const int board = KIND == K_SYM8 ? unit : unit * UNIT_BOARDS + tile * 2 + bit;
            const bool live = real && board < n_boards;
            {
                uint4 v = make_uint4(0, 0, 0, 0);
                if (live) {
                    float f[4];
                    const int src_cell = KIND == K_SYM8 ? sym_cell(sym, cell / 7, cell % 7) : cell;   // the image's cell shows this board cell
                    if (IN_KIND == AZ_IN_F32) {
                        const float4 q = reinterpret_cast<const float4 *>(P.input)[(size_t)board * 49 + src_cell];
                        f[0] = q.x; f[1] = q.y; f[2] = q.z; f[3] = q.w;
                    } else {
                        az_position p = reinterpret_cast<const az_position *>(P.input)[board];
                        p.turn &= 1;
                        az::feature_cell(p, src_cell / 7, src_cell % 7, f);
                    }
                    v.x = pack_op(f[0], f[1], P.f16);
                    v.y = pack_op(f[2], f[3], P.f16);
                }
                *reinterpret_cast<uint4 *>(act_row) = v;         // k-group 0 of the tile's activations
                fence_proxy_async();
                mbar_arrive(tbar(tile, IN));
            }
            for (int l = 0; l < P.layers; ++l) {
                const bool second = l > 0 && (l & 1) == 0;
                const bool writes_res = l == 0 || second;
                float *shift_s = shift_base + (l & 1) * F;
                shift_s[gtid] = __ldg(P.shift + l * F + gtid);
                group_sync(tile);
                mbar_wait(tbar(tile, ACC), acc_phase);
                acc_phase ^= 1;
                tc_fence_after();
                const uint32_t src = lane_addr + (second ? TM_RES : TM_ACC);
                uint32_t acc[2][32];
                tmem_ld32(src, acc[0]);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    uint32_t (&a)[32] = acc[q & 1];
                    tmem_wait_ld();
                    if (q < 3) tmem_ld32(src + (q + 1) * 32, acc[(q + 1) & 1]);
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        float v = __uint_as_float(a[i]) + shift_s[q * 32 + i];
                        v = live ? fmaxf(v, 0.f) : 0.f;
                        a[i] = __float_as_uint(v);
                    }
                    if (writes_res) tmem_st32(lane_addr + TM_RES + q * 32, a);
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        uint4 o;
                        o.x = pack_op(__uint_as_float(a[8 * g + 0]), __uint_as_float(a[8 * g + 1]), P.f16);
                        o.y = pack_op(__uint_as_float(a[8 * g + 2]), __uint_as_float(a[8 * g + 3]), P.f16);
                        o.z = pack_op(__uint_as_float(a[8 * g + 4]), __uint_as_float(a[8 * g + 5]), P.f16);
                        o.w = pack_op(__uint_as_float(a[8 * g + 6]), __uint_as_float(a[8 * g + 7]), P.f16);
                        *reinterpret_cast<uint4 *>(act_row + (q * 4 + g) * ACT_LBO) = o;
                    }
                    if constexpr (KIND == K_TOWER) if (l == P.layers - 1 && live) {
                        float *dst = P.debug_act + ((size_t)board * 49 + cell) * F + q * 32;
                        for (int i = 0; i < 32; ++i) dst[i] = __uint_as_float(a[i]);
                    }
                    if (l > 0 && q == 1) {
                        // channels 0..63 of this row are in shared memory: the next layer may start on them (not after the input
                        // conv: layer 1 reuses the accumulator this epilogue is still reading)
                        fence_proxy_async();
                        tc_fence_before();
                        mbar_arrive(tbar(tile, ACT + 0));
                    }
                }
                if (writes_res) tmem_wait_st();
                fence_proxy_async();
                tc_fence_before();
                if (l == 0) mbar_arrive(tbar(tile, ACT + 0));
                mbar_arrive(tbar(tile, ACT + 1));
            }
            if (HEADS) {
                mbar_wait(tbar(tile, ACC), acc_phase);
                acc_phase ^= 1;
                tc_fence_after();
                uint32_t a[32];
                tmem_ld32(lane_addr + TM_ACC, a);
                tmem_wait_ld();
                float vterm = 0.f;
                if (live) {
                    if (KIND == K_PLAIN || KIND == K_PROF) {
                        float *dst = P.logits + (size_t)board * AZ_LOGITS + cell * 17;
#pragma unroll
                        for (int i = 0; i < 17; ++i) dst[i] = __uint_as_float(a[i]);
                    }
                    vterm = __uint_as_float(a[17]) * __ldg(P.fc_w + cell);
                }
#pragma unroll
                for (int s = 16; s; s >>= 1) vterm += __shfl_xor_sync(0xffffffffu, vterm, s);
                if (lane == 0) vpart[quad] = vterm;
                tc_fence_before();
                group_sync(tile);
                if (gtid < 2) {
                    const int b = unit * UNIT_BOARDS + tile * 2 + gtid;
                    if constexpr (KIND == K_SYM8) sym_acc[AZ_LOGITS + pass * UNIT_BOARDS + tile * 2 + gtid] = tanhf(vpart[2 * gtid] + vpart[2 * gtid + 1] + __ldg(P.fc_b));
                    else if (b < n_boards) {
                        if constexpr (KIND == K_CACHE) P.values[P.out_map ? __ldg(P.out_map + b) : b] = tanhf(vpart[2 * gtid] + vpart[2 * gtid + 1] + __ldg(P.fc_b));
                        else P.values[b] = tanhf(vpart[2 * gtid] + vpart[2 * gtid + 1] + __ldg(P.fc_b));
                    }
                }
                if constexpr (KIND == K_SYM8) {
                    // mean over the 8 images, each rotated back onto the board (spatially only: the 16 direction planes are
                    // not permuted, nn_evals.py:58-62).  Images are added in ascending order (np.mean's order for axis 0), one
                    // image at a time: an image is a permutation of the cells, so its rows never collide.
                    const int dst_cell = sym_cell(sym, cell / 7, cell % 7);
                    for (int im = 0; im < UNIT_BOARDS; ++im) {
                        if (im == bit && live) {
                            float *dst = sym_acc + dst_cell * 17;
#pragma unroll
                            for (int i = 0; i < 17; ++i) dst[i] = sym == 0 ? __uint_as_float(a[i]) : dst[i] + __uint_as_float(a[i]);
                        }
                        group_sync(tile);
                    }
                    if (pass == PASSES - 1) {
                        if (board < n_boards) {
                            for (int i = gtid; i < AZ_LOGITS; i += 128) P.logits[(size_t)board * AZ_LOGITS + i] = sym_acc[i] * 0.125f;
                            if (gtid == 0) {
                                const float *v = sym_acc + AZ_LOGITS;       // np.mean of 8 floats: numpy's pairwise tree
                                P.values[board] = (((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]))) * 0.125f;
                            }
                        }
                        group_sync(tile);           // the sum is read before the next position overwrites it
                    }
                } else if constexpr (KIND == K_CACHE) {
                    // softmax numerators in double for the tree kernel; the helper warp adds them up
                    if (live) {
                        double *e = P.exps + (size_t)(P.out_map ? __ldg(P.out_map + board) : board) * AZ_LOGITS + cell * 17;
#pragma unroll
                        for (int i = 0; i < 17; ++i) e[i] = exp_d(__uint_as_float(a[i]));
                    }
                    __threadfence_block();
                    helper_arrive();
                    group_sync(tile);
                } else {
                    group_sync(tile);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                  // nobody leaves (or frees tensor memory) while the pair's MMAs may still touch it
    if (warp == 1) tmem_dealloc(tmem_base, C::TMEM_COLS);
}

// ---- weight tiling for the pair layout ----
__device__ __forceinline__ uint16_t to_operand(float w, int f16)
{
    if (f16) { const __half h = __float2half_rn(w); return *reinterpret_cast<const uint16_t *>(&h); }
    const __nv_bfloat16 b = __float2bfloat16_rn(w);
    return *reinterpret_cast<const uint16_t *>(&b);
}

// tower: out index ((((l*18 + chunk)*2 + half)*8 + kg)*64 + co)*8 + i, chunk = part*9 + tap, cout = half*64 + co
__global__ void k_tile_tower_pair(const float *__restrict__ w_tower, const float *__restrict__ scale, int tower_layers, uint16_t *__restrict__ out, int f16)
{
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t total = (size_t)tower_layers * CHUNKS * 2 * PART_KG * HALF_N * 8;
    if (idx >= total) return;
    const int i = (int)(idx & 7);
    const int co = (int)((idx >> 3) & 63);
    size_t rest = idx >> 9;
    const int kg = (int)(rest % PART_KG); rest /= PART_KG;
    const int half = (int)(rest & 1); rest >>= 1;
    const int chunk = (int)(rest % CHUNKS);
    const int l = (int)(rest / CHUNKS);
    const int part = chunk / 9, tap = chunk % 9;
    const int cin = (part * PART_KG + kg) * 8 + i, cout = half * HALF_N + co;
    out[idx] = to_operand(w_tower[(((size_t)l * 9 + tap) * F + cin) * F + cout] * scale[(size_t)(l + 1) * F + cout], f16);
}

__global__ void k_tile_small_pair(const float *__restrict__ w_in, const float *__restrict__ w_policy, const float *__restrict__ w_value,
                                  const float *__restrict__ bn_raw, const float *__restrict__ scale, int layers, uint16_t *__restrict__ out_in,
                                  uint16_t *__restrict__ out_heads, float *__restrict__ shift, int f16)
{
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < 2 * 5 * 2 * HALF_N * 8) {          // input conv: [half][kstep j][g][co 64][i], tap = 2j+g (tap 9 = zero), 4 real channels
        const int i = idx & 7, co = (idx >> 3) & 63, g = (idx >> 9) & 1, j = (idx >> 10) % 5, half = idx / (5 * 2 * HALF_N * 8);
        const int tap = 2 * j + g, cout = half * HALF_N + co;
        float w = 0.f;
        if (tap < 9 && i < 4) w = w_in[((size_t)tap * 4 + i) * F + cout] * scale[cout];
        out_in[idx] = to_operand(w, f16);
    }
    if (idx < 2 * KG * HEAD_HALF * 8) {          // heads: [half][kg][row 16][i]: head row = half*16 + row; rows 0..16 policy, 17 value
        const int i = idx & 7, row = (idx >> 3) & 15, kg = (idx >> 7) % KG, half = idx / (KG * HEAD_HALF * 8);
        const int cin = kg * 8 + i, hrow = half * HEAD_HALF + row;
        float w = 0.f;
        if (hrow < 17) w = w_policy[(size_t)cin * 17 + hrow];
        else if (hrow == 17) w = w_value[cin];
        out_heads[idx] = to_operand(w, f16);
    }
    if (idx < layers * F) {                      // epilogue shift = -mean * scale, in double like the reference's BN
        const int l = idx / F, c = idx % F;
        const double sc = 1.0 / sqrt((double)bn_raw[(size_t)(2 * l + 1) * F + c] + (double)AZ_BN_EPS);
        shift[idx] = (float)(-(double)bn_raw[(size_t)(2 * l) * F + c] * sc);
    }
}

}  // namespace

// ------------------------------------------------------------------------------------------
// host side (called from az_net.cu)
// ------------------------------------------------------------------------------------------
size_t az_net_pair_stream_bytes(const AzNet *net)
{
    return 2 * (size_t)WIN_HALF_BYTES + (size_t)2 * net->blocks * CHUNKS * CHUNK_BYTES + 2 * (size_t)WHEAD_HALF_BYTES;
}

int az_net_pair_alloc(AzNet *net)
{
    const size_t bytes = az_net_pair_stream_bytes(net);
    AZ_CUDA(cudaMalloc(&net->pair_stream, bytes));
    AZ_CUDA(cudaMalloc(&net->pair_stream16, bytes));
    AZ_CUDA(cudaMalloc(&net->pair_shift, (size_t)net->layers * F * 4));
#define AZ_PAIR_ATTR(T, K, KIND) AZ_CUDA(cudaFuncSetAttribute(k_net_pair<T, K, KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize, PairCfg<T, KIND>::SMEM_BYTES))
    AZ_PAIR_ATTR(1, AZ_IN_F32, K_PLAIN); AZ_PAIR_ATTR(1, AZ_IN_POS, K_PLAIN); AZ_PAIR_ATTR(1, AZ_IN_F32, K_PROF); AZ_PAIR_ATTR(1, AZ_IN_POS, K_PROF);
    AZ_PAIR_ATTR(2, AZ_IN_F32, K_PLAIN); AZ_PAIR_ATTR(2, AZ_IN_POS, K_PLAIN);
    AZ_PAIR_ATTR(1, AZ_IN_POS, K_CACHE); AZ_PAIR_ATTR(1, AZ_IN_F32, K_SYM8); AZ_PAIR_ATTR(1, AZ_IN_F32, K_TOWER);
#undef AZ_PAIR_ATTR
    const char *env = getenv("AZ_NET_PAIR_TILES");     // forces one variant; by default the batch size picks it
    net->pair_tiles = (env && (atoi(env) == 1 || atoi(env) == 2)) ? atoi(env) : 0;
    return AZ_OK;
}

// Re-tile the fp32 TF-layout parameters into the operand images the kernel streams, folding the batch-norm scale
// 1/sqrt(var+eps) of the conv's own BN layer into its output channels, and compute the epilogue's BN shifts.
int az_net_pair_prepare(az_context *ctx, AzNet *net)
{
    cudaStream_t s = ctx->stream;
    const size_t tower = (size_t)2 * net->blocks * CHUNKS * 2 * PART_KG * HALF_N * 8;
    const size_t tower_bytes = (size_t)2 * net->blocks * CHUNKS * CHUNK_BYTES;
    const int small = std::max(2 * 5 * 2 * HALF_N * 8, net->layers * F);
    for (int f16 = 0; f16 < 2; ++f16) {
        uint8_t *base = f16 ? net->pair_stream16 : net->pair_stream;
        k_tile_tower_pair<<<(unsigned)((tower + 255) / 256), 256, 0, s>>>(net->w_tower, net->bn_scale, 2 * net->blocks,
                                                                          reinterpret_cast<uint16_t *>(base + 2 * WIN_HALF_BYTES), f16);
        k_tile_small_pair<<<(small + 255) / 256, 256, 0, s>>>(net->w_in, net->w_policy, net->w_value, net->bn_raw, net->bn_scale, net->layers,
                                                              reinterpret_cast<uint16_t *>(base),
                                                              reinterpret_cast<uint16_t *>(base + 2 * WIN_HALF_BYTES + tower_bytes), net->pair_shift, f16);
    }
    AZ_CUDA(cudaGetLastError());
    return AZ_OK;
}

void az_net_pair_release(AzNet *net)
{
    if (net->pair_stream) cudaFree(net->pair_stream);
    if (net->pair_stream16) cudaFree(net->pair_stream16);
    if (net->pair_shift) cudaFree(net->pair_shift);
    net->pair_stream = net->pair_stream16 = nullptr;
    net->pair_shift = nullptr;
}

int az_net_pair_boards_per_round(az_context *ctx)
{
    return ctx->sm_count * PairCfg<1>::CTAS_PER_SM * PairCfg<1>::UNIT_BOARDS;
}

// Profiling hook (not part of the public header, used by tools/net_pair_waits.py): while `d_buf` is non-null, every plain
// k_net_pair launch of this context's loaded net runs the one-tile instantiation that writes issuer wait records
// (PairParams::prof) -- (4 + 3 * max_records) int64 per CTA.  It stays set for this context until cleared with a null buffer.
extern "C" int az_net_pair_profile(az_context *ctx, long long *d_buf, int max_records)
{
    AZ_REQUIRE(ctx && ctx->net, AZ_ERR_STATE, "az_net_pair_profile: no weights loaded");
    AZ_REQUIRE(!d_buf || max_records > 0, AZ_ERR_ARG, "az_net_pair_profile: max_records=%d", max_records);
    ctx->net->pair_prof = d_buf;
    ctx->net->pair_prof_max = max_records;
    return AZ_OK;
}

static PairParamsX pair_params(const AzNet *net, const void *d_in, int n, float *d_logits, float *d_values, int f16)
{
    PairParamsX P{};
    P.input = d_in;
    P.n = n;
    P.layers = net->layers;
    P.w_stream = f16 ? net->pair_stream16 : net->pair_stream;
    P.shift = net->pair_shift;
    P.fc_w = net->fc_w;
    P.fc_b = net->fc_b;
    P.logits = d_logits;
    P.values = d_values;
    P.f16 = f16;
    return P;
}

// `units` work items (units of UNIT_BOARDS boards, or SYM8 positions) over at most one wave of CTAs
template <int T, int IN_KIND, int KIND>
static int pair_launch(az_context *ctx, const PairParamsX &P, int units, cudaStream_t stream)
{
    using C = PairCfg<T, KIND>;
    int grid = std::min(units, ctx->sm_count * C::CTAS_PER_SM);
    grid = (grid + 1) / 2 * 2;                                  // whole pairs; a surplus CTA runs an all-padding pass
    k_net_pair<T, IN_KIND, KIND><<<grid, C::NUM_THREADS, C::SMEM_BYTES, stream>>>(P);     // PLAIN and PROF take P's PairParams part
    ctx->launches++;
    AZ_CUDA(cudaGetLastError());
    return AZ_OK;
}

int az_net_pair_forward(az_context *ctx, AzNet *net, const void *d_in, int in_kind, int n, float *d_logits, float *d_values, const int *d_count,
                        cudaStream_t stream, int f16, double *d_exps, double *d_totals, const int *d_out_map, int tiles)
{
    if (!stream) stream = ctx->stream;
    PairParamsX P = pair_params(net, d_in, n, d_logits, d_values, f16);
    P.n_ptr = d_count;
    if (d_exps) {                       // the speculative cache pass (az_pool.cu launch_net)
        AZ_REQUIRE(in_kind == AZ_IN_POS, AZ_ERR_ARG, "az_net_forward: softmax numerators are produced from position input only");
        P.exps = d_exps;
        P.totals = d_totals;
        P.out_map = d_out_map;
        return pair_launch<1, AZ_IN_POS, K_CACHE>(ctx, P, (n + 1) / 2, stream);
    }
    P.prof = net->pair_prof;
    P.prof_max = net->pair_prof_max;
    // Two tiles per CTA keep the tensor pipe fed across epilogues, but one CTA per SM only fills the GPU from a full round of
    // 4 boards per SM on; smaller batches (single trees, latency-bound callers) run one-tile CTAs, two per SM.  The wait
    // records are taken for the one-tile schedule.
    if (P.prof) tiles = 1;
    else if (!tiles) tiles = net->pair_tiles ? net->pair_tiles : n >= 4 * ctx->sm_count ? 2 : 1;
    const int units = (n + 2 * tiles - 1) / (2 * tiles);
    if (P.prof)
        return in_kind == AZ_IN_F32 ? pair_launch<1, AZ_IN_F32, K_PROF>(ctx, P, units, stream) : pair_launch<1, AZ_IN_POS, K_PROF>(ctx, P, units, stream);
    if (tiles == 1)
        return in_kind == AZ_IN_F32 ? pair_launch<1, AZ_IN_F32, K_PLAIN>(ctx, P, units, stream) : pair_launch<1, AZ_IN_POS, K_PLAIN>(ctx, P, units, stream);
    return in_kind == AZ_IN_F32 ? pair_launch<2, AZ_IN_F32, K_PLAIN>(ctx, P, units, stream) : pair_launch<2, AZ_IN_POS, K_PLAIN>(ctx, P, units, stream);
}

// nn_evals.evaluate for n positions in ONE launch: images generated in the input staging, averaged in the head epilogue
int az_net_pair_forward_sym8(az_context *ctx, AzNet *net, const float *d_features, int n, float *d_logits, float *d_values, int f16)
{
    const PairParamsX P = pair_params(net, d_features, n, d_logits, d_values, f16);
    return pair_launch<1, AZ_IN_F32, K_SYM8>(ctx, P, n, ctx->stream);
}

// the first `conv_layers` convolutions of the tower in bf16; the last one's fp32 activations (before the bf16 rounding) to d_act
int az_net_pair_tower(az_context *ctx, AzNet *net, const float *d_features, int n, int conv_layers, float *d_act)
{
    PairParamsX P = pair_params(net, d_features, n, nullptr, nullptr, 0);
    P.layers = conv_layers;
    P.debug_act = d_act;
    return pair_launch<1, AZ_IN_F32, K_TOWER>(ctx, P, (n + 1) / 2, ctx->stream);
}
