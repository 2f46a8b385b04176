// AZ_NVCC_FLAGS: -fmad=false
// az_net_tc.cu -- the conv tower as bf16 tcgen05 implicit GEMMs, whole network in ONE persistent
// kernel (sm_100a).  Replaces TF1's sess.run of model.py:38-79 on the self-play hot path
// (accelerated_generate_games.py:57-63) and the dead cuDNN stub cpp/fast_eval.cpp:37-126.
//
// Mapping (DESIGN.md "net kernel"):
//   * A CTA owns a "unit" of 4 boards = 2 M-tiles of 128 GEMM rows.  A board is 64 rows: row
//     8 + 8x + y holds cell (x, y), y == 7 and rows 0..7 are zero padding, so each 3x3 tap is a
//     CONSTANT ROW SHIFT (8*dx + dy) of the same activation buffer -> the im2col matrix is never
//     built; the A-operand descriptor of a tap just starts `shift` rows earlier/later.
//   * Activations stay in shared memory for all 25 layers as bf16 in the no-swizzle K-major UMMA
//     layout [k-group of 8 channels][row][8 channels] (16-byte rows, so any row shift is a legal
//     descriptor start address).  Outputs overwrite inputs in place: an epilogue only runs after
//     every MMA of its layer has completed.
//   * Accumulators (128 lanes x 128 fp32 columns per tile) and the fp32 residual stream live in
//     TMEM: 2 tiles x (128 + 128) columns = all 512.
//   * Weights (BN scale folded, bf16) are pre-tiled in HBM in exactly the shared-memory image of a
//     pipeline stage (one tap x 64 input channels = 16 KiB) and streamed through a 4-stage ring by
//     1-D bulk TMA copies (cp.async.bulk + mbarrier complete_tx); each stage feeds both tiles.
//   * Warp roles: warp 0 = TMA producer, warp 1 = MMA issuer (single elected lane), warps 2-5 /
//     6-9 = epilogue of tile 0 / tile 1 (TMEM -> +shift, +residual, ReLU -> bf16 -> smem, and the
//     heads' logits/value to HBM), last warp = softmax helper.
//   * Softmax front half for the tree kernel (self_play_client.cpp:208-214), when the caller asks for it: the head
//     epilogue also writes exp((double)logit) of all 833 logits, and the helper warp adds them up strictly left to
//     right -- the reference's sequential `total +=` -- one lane per board, while the CTA is already busy with its
//     next boards.  833 double exponentials and an 833-long dependent chain of double additions per leaf would
//     otherwise saturate the fp64 pipes of the latency-bound tree kernel (16 games per SM start on them at once).
//     This file is compiled without fused multiply-add contraction like az_tree.cu, so both produce the same bits.
//   * Symmetry ensemble (nn_evals.py:48-62): in sym8 mode a CTA runs the 8 dihedral images of one position through the
//     tower in four consecutive passes -- the images are generated while the input planes are staged and averaged
//     (policies rotated back spatially, direction planes not permuted, as in the reference) in the head epilogue.
#include "az_net.h"
#include "az_rules.cuh"

#include <algorithm>
#include <cstdlib>

namespace {

constexpr int F = AZ_F;                  // channels
constexpr int KG = F / 8;                // 16 k-groups of 8 channels
constexpr int TILE_M = 128;              // GEMM rows per tile (2 boards x 64)
constexpr int MARGIN = 16;               // zero rows before/after the tiles (shifts reach +-9)
constexpr int ROW_BYTES = 16;            // 8 bf16
#ifndef AZ_NET_SPLIT
#define AZ_NET_SPLIT 2
#endif
// A layer's weights travel as SPLIT x 9 chunks: input-channel part (128 / SPLIT channels) major, tap minor.  A layer can start
// on part p as soon as the previous epilogue has produced that part's channels, so SPLIT sets how early the MMAs -- and with
// them the weight stream -- restart after a layer (SPLIT = 2: half way through the epilogue, 4: after its first quarter).
// Measured (B200, 2048 games x 800 visits): SPLIT 2 -> 0.507 ms per net launch, SPLIT 4 -> 0.541 ms (8-KiB stages double the
// per-stage hand-offs of the single issuing thread); the 2-tile variant is indifferent (0.517 / 0.516 ms).
constexpr int SPLIT = AZ_NET_SPLIT;
constexpr int PART_KG = KG / SPLIT;      // k-groups (of 8 channels) per chunk
constexpr int PART_MMAS = PART_KG / 2;   // K = 16 steps per chunk
constexpr int STAGE_BYTES = PART_KG * F * ROW_BYTES;           // one tap x 128/SPLIT input channels x 128 cout (SPLIT 4: 8 KiB)
constexpr int CHUNKS = SPLIT * 9;
static_assert(SPLIT == 2 || SPLIT == 4, "input channels per chunk: 64 or 32");
constexpr int W_LBO = F * ROW_BYTES;     // 2048: bytes between k-groups of the B operand
constexpr int ZERO_BYTES = TILE_M * ROW_BYTES;                 // zero k-group for the padded 10th tap
constexpr int WIN_BYTES = 5 * 2 * F * ROW_BYTES;               // input conv: 5 k-steps x 2 k-groups x 128 cout = 20480
constexpr int WIN_KSTEP_BYTES = 2 * F * ROW_BYTES;             // one K = 16 step of the input conv (two taps): 4 KiB
constexpr int WIN_KSTEPS_PER_STAGE = STAGE_BYTES / WIN_KSTEP_BYTES;     // the 5 k-steps travel in stages of this many
constexpr int HEAD_N = 32;               // 17 policy planes + 1 value plane, padded to a legal UMMA N
constexpr int WHEAD_BYTES = KG * HEAD_N * ROW_BYTES;           // 8192
constexpr int HEAD_LBO = HEAD_N * ROW_BYTES;

// Per-variant geometry: TILES tiles (2 boards each) per CTA.  TILES = 2 -> one CTA per SM, each weight stage feeds
// two tiles; TILES = 1 -> two independent CTAs per SM whose epilogues and MMAs interleave on the tensor pipe.
template <int TILES>
struct Cfg {
    static constexpr int UNIT_BOARDS = 2 * TILES;
    static constexpr int STAGES = (TILES == 1 ? 4 : 8) * (16384 / STAGE_BYTES);   // 64 / 128 KiB of weight stages in flight
    static constexpr int ACT_ROWS = MARGIN + TILES * TILE_M + MARGIN;
    static constexpr int ACT_LBO = ACT_ROWS * ROW_BYTES;           // bytes between k-groups of the A operand
    static constexpr int ACT_BYTES = KG * ACT_LBO;
    static constexpr int IN_BYTES = ACT_ROWS * ROW_BYTES;          // input planes: one k-group (4 real + 4 zero channels)
    static constexpr int OFF_ACT = 0;
    static constexpr int OFF_RING = OFF_ACT + ACT_BYTES;
    // The input planes are staged in k-group 0 of the activation buffer itself: it is dead between the heads of one unit
    // and the layer-0 epilogue of the next (which overwrites it only after the input-conv MMAs have completed).
    static constexpr int OFF_IN = OFF_ACT;
    static constexpr int OFF_SHIFT = OFF_RING + STAGES * STAGE_BYTES;   // float[TILES][2][F]: per-layer BN shifts, double-buffered
    static constexpr int OFF_VPART = OFF_SHIFT + TILES * 2 * F * 4;
    static constexpr int OFF_SYM = OFF_VPART + 64;                   // sym8 mode: float[833] policy sum + float[8] values (+ pad)
    static constexpr int SYM_BYTES = 3392;
    static constexpr int OFF_BAR = OFF_SYM + SYM_BYTES;
    static constexpr int NUM_BARS = 2 * STAGES + (1 + SPLIT) * TILES + 1;   // full/empty ring, acc_full + SPLIT x act_ready per tile, input staged
    static constexpr int OFF_TMEM = OFF_BAR + NUM_BARS * 8;
    static constexpr int SMEM_BYTES = OFF_TMEM + 16;
    static constexpr int NUM_WARPS = 3 + 4 * TILES;                 // producer, MMA issuer, 4 epilogue warps per tile, softmax helper
    static constexpr int HELPER_WARP = 2 + 4 * TILES;
    static constexpr int EPI_THREADS = 128 * TILES;
    static constexpr int NUM_THREADS = NUM_WARPS * 32;
    static constexpr int CTAS_PER_SM = TILES == 1 ? 2 : 1;
    static constexpr uint32_t TMEM_COLS = TILES * 256;             // per tile: 128 accumulator + 128 residual columns
    static constexpr uint32_t TM_ACC = 0;                          // + tile*128
    static constexpr uint32_t TM_RES = TILES * 128;                // + tile*128
    static_assert(SMEM_BYTES * CTAS_PER_SM + 1024 * CTAS_PER_SM <= 228 * 1024, "shared memory budget");
};

// instruction descriptor: D=f32, A=B=bf16, K-major both, M=128, N
// (A / B format fields, bits 7-9 / 10-12: 1 = bf16, 0 = f16 -- the AZ_NET_F16 mode clears both)
constexpr uint32_t make_idesc(int n) { return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(TILE_M >> 4) << 24); }
constexpr uint32_t IDESC_128 = make_idesc(128);
constexpr uint32_t IDESC_HEAD = make_idesc(HEAD_N);
constexpr uint32_t IDESC_FMT_BF16 = (1u << 7) | (1u << 10);

// ------------------------------------------------------------------------------------------
// PTX helpers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    uint32_t done;
    do {
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
    } while (!done);
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
// the same copy, delivered to the same shared-memory offset (and signalling the same mbarrier offset) of every CTA in
// `cta_mask` of the cluster: one L2 read feeds several SMs
__device__ __forceinline__ void bulk_g2s_multicast(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar, uint16_t cta_mask)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%3], %4;" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar), "h"(cta_mask)
                 : "memory");
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
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols)
{
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}

// no-swizzle K-major shared-memory matrix descriptor (SBO = 128 B: 8-row core matrices are contiguous)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes)
{
    return (uint64_t)((saddr >> 4) & 0x3fff) | ((uint64_t)((lbo_bytes >> 4) & 0x3fff) << 16) |
           ((uint64_t)(128 >> 4) << 32) | (1ULL << 46);
}

__device__ __forceinline__ void umma(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// same, with the 64-bit descriptors assembled from a running low word (start address field) and a constant high word:
// stepping through taps / k-groups / stages is then ONE integer add per operand on the issuing thread
__device__ __forceinline__ void umma_lo(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                        uint32_t accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        ".reg .b64 da, db;\n\t"
        "mov.b64 da, {%1, %2};\n\t"
        "mov.b64 db, {%3, %4};\n\t"
        "setp.ne.b32 p, %6, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t"
        "}" ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ bool elect_one()
{
    uint32_t pred;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void umma_commit(uint32_t bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// arrive on the barrier at this offset in every CTA of `cta_mask` once the MMAs issued so far have completed
__device__ __forceinline__ void umma_commit_multicast(uint32_t bar, uint16_t cta_mask)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"(cta_mask)
                 : "memory");
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32])
{
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
        "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),
        "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),
        "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi)
{
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t *>(&v);
}
__device__ __forceinline__ uint32_t pack_f16(float lo, float hi)
{
    __half2 v = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<uint32_t *>(&v);
}
template <bool F16>
__device__ __forceinline__ uint32_t pack_op(float lo, float hi) { return F16 ? pack_f16(lo, hi) : pack_bf16(lo, hi); }

// 32 channels of one GEMM row -> four 16-byte k-group rows of the activation buffer, in the operand format
template <bool F16>
__device__ __forceinline__ void store_row(const uint32_t (&a)[32], uint8_t *dst, int lbo)
{
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        uint4 o;
        o.x = pack_op<F16>(__uint_as_float(a[8 * g + 0]), __uint_as_float(a[8 * g + 1]));
        o.y = pack_op<F16>(__uint_as_float(a[8 * g + 2]), __uint_as_float(a[8 * g + 3]));
        o.z = pack_op<F16>(__uint_as_float(a[8 * g + 4]), __uint_as_float(a[8 * g + 5]));
        o.w = pack_op<F16>(__uint_as_float(a[8 * g + 6]), __uint_as_float(a[8 * g + 7]));
        *reinterpret_cast<uint4 *>(dst + g * lbo) = o;
    }
}

// named barrier among the 4 epilogue warps of one tile
__device__ __forceinline__ void group_sync(int tile)
{
    // literal barrier ids so ptxas reserves 3 barriers, not all 16 (two CTAs share an SM in the 1-tile variant)
    if (tile == 0) asm volatile("bar.sync 1, 128;" ::: "memory");
    else asm volatile("bar.sync 2, 128;" ::: "memory");
}

// exp((double)logit) exactly as the tree kernel computes it (az_tree.cu populate_from_eval): same libdevice routine, same
// compiler flags.  Not inlined: 17 calls per epilogue thread and unit, off the layer-to-layer critical path.
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

template <int TILES>
__device__ __forceinline__ void epilogue_sync_all()       // all epilogue threads of the CTA (both tiles)
{
    if (TILES == 1) asm volatile("bar.sync 1, 128;" ::: "memory");
    else asm volatile("bar.sync 4, 256;" ::: "memory");
}
template <int TILES>
__device__ __forceinline__ void helper_arrive()           // epilogue threads -> softmax helper warp: "the exps of this unit are written"
{
    if (TILES == 1) asm volatile("bar.arrive 3, 160;" ::: "memory");
    else asm volatile("bar.arrive 3, 288;" ::: "memory");
}
template <int TILES>
__device__ __forceinline__ void helper_wait()
{
    if (TILES == 1) asm volatile("bar.sync 3, 160;" ::: "memory");
    else asm volatile("bar.sync 3, 288;" ::: "memory");
}

struct TcParams {
    const void *input;                 // float[n][196] or az_position[n]
    int n;                             // boards
    const int *n_ptr;                  // when non-null the board count is read from device memory
    int layers;                        // 1 + 2*blocks
    int debug_layers;                  // >= 0: stop after this many conv layers and dump activations
    const uint8_t *w_stream;           // [input conv 20480 B][2*blocks x 18 chunks x 16384 B][heads 8192 B]
    const float *shift;                // [layers][128]
    const float *fc_w;                 // [49]
    const float *fc_b;                 // [1]
    float *logits;                     // [n][833]
    float *values;                     // [n]
    float *debug_act;                  // [n][49][128] (debug only)
    const int *out_map;                // when non-null: the outputs of board b go to row out_map[b] of values / exps / totals (logits too)
    double *exps;                      // when non-null: [n][833] exp((double)logit), the softmax numerators of :210-211
    double *totals;                    // [n] their strictly sequential sum (:212-214)
    int f16;                           // operands (weights, activations) are IEEE half instead of bf16: 3 more mantissa bits, 5-bit exponent
    int sym8;                          // 1: `n` positions, each evaluated as the mean over its 8 dihedral images (nn_evals.py:48-62)
};

// row r of a tile -> board within tile / cell; real rows carry data, the rest are zero padding
__device__ __forceinline__ bool row_is_real(int r, int &board_in_tile, int &cell)
{
    board_in_tile = r >> 6;
    const int w = r & 63;
    const int x = (w >> 3) - 1, y = w & 7;
    cell = x * 7 + y;
    return w >= 8 && y != 7;
}

// CS = thread-block cluster size.  The CS CTAs of a cluster walk the same weight stream in lockstep: each fetches 1/CS of
// every pipeline stage from L2 and multicasts it into the shared memory of all of them, so the L2 -> SM weight traffic
// (the kernel's real bottleneck: ~12 TB/s without it) drops by CS.  A stage slot is free once the MMA issuers of ALL the
// cluster's CTAs have committed it (empty barriers count CS multicast arrivals).
template <int TILES, int IN_KIND, int CS>
__global__ void __launch_bounds__(Cfg<TILES>::NUM_THREADS, Cfg<TILES>::CTAS_PER_SM) k_net_tc(const TcParams P)
{
    using C = Cfg<TILES>;
    constexpr uint16_t CMASK = (uint16_t)((1u << CS) - 1);
    const uint32_t crank = CS > 1 ? cluster_ctarank() : 0;
    extern __shared__ __align__(1024) uint8_t smem[];
    const uint32_t sbase = smem_u32(smem);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    auto bar = [&](int i) { return sbase + C::OFF_BAR + 8 * i; };
    // barrier indices
    constexpr int STAGES = C::STAGES;
    // B_ACT + SPLIT*tile + p: channels [128/SPLIT * p, 128/SPLIT * (p+1)) of the tile's new activations are in shared memory
    constexpr int B_FULL = 0, B_EMPTY = STAGES, B_ACC = 2 * STAGES, B_ACT = 2 * STAGES + TILES, B_IN = 2 * STAGES + (1 + SPLIT) * TILES;

    const int n_boards = P.n_ptr ? min(*P.n_ptr, P.n) : P.n;
    // work items of a CTA: units of UNIT_BOARDS boards, or (sym8) whole positions, each `passes` trips through the tower
    const int passes = P.sym8 ? 8 / C::UNIT_BOARDS : 1;
    const int items = P.sym8 ? n_boards : (n_boards + C::UNIT_BOARDS - 1) / C::UNIT_BOARDS;
    const int num_units = (items + CS - 1) / CS * CS;              // cluster peers run the same number of passes
    const int tower_layers = P.layers - 1;          // tensor-core 128->128 convs
    const int run_layers = P.debug_layers >= 0 ? min(P.debug_layers, P.layers) : P.layers;   // conv layers executed (incl. input conv)
    const int nl = min(tower_layers, run_layers - 1);
    const bool heads = P.debug_layers < 0;

    // ---- one-time setup ----
    for (int i = threadIdx.x; i < C::ACT_BYTES / 16; i += C::NUM_THREADS) reinterpret_cast<uint4 *>(smem + C::OFF_ACT)[i] = make_uint4(0, 0, 0, 0);
    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(bar(B_FULL + s), 1); mbar_init(bar(B_EMPTY + s), CS); }
        for (int t = 0; t < TILES; ++t) {
            mbar_init(bar(B_ACC + t), 1);
            for (int p = 0; p < SPLIT; ++p) mbar_init(bar(B_ACT + SPLIT * t + p), 128);
        }
        mbar_init(bar(B_IN), 128 * TILES);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(sbase + C::OFF_TMEM, C::TMEM_COLS);
    fence_proxy_async();                 // zero-fills above must be visible to the tensor core's async proxy
    tc_fence_before();
    __syncthreads();
    if (CS > 1) cluster_sync_all();      // every peer's barriers exist before anything is multicast at them
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t *>(smem + C::OFF_TMEM);

    if (warp == 0) {
        // =============================== TMA producer ===============================
        // per unit the weight stream is: input conv (16 KiB + 4 KiB), 18 chunks per tower layer, heads (8 KiB)
        if (lane == 0) {
            uint32_t it = 0;
            auto push = [&](const uint8_t *src, uint32_t bytes) {
                const int s = it % STAGES;
                mbar_wait(bar(B_EMPTY + s), ((it / STAGES) & 1) ^ 1);
                mbar_expect_tx(bar(B_FULL + s), bytes);           // the whole stage: own slice + the peers' slices
                if (CS == 1) {
                    bulk_g2s(sbase + C::OFF_RING + s * STAGE_BYTES, src, bytes, bar(B_FULL + s));
                } else {
                    const uint32_t slice = bytes / CS;
                    bulk_g2s_multicast(sbase + C::OFF_RING + s * STAGE_BYTES + crank * slice, src + crank * slice, slice, bar(B_FULL + s), CMASK);
                }
                ++it;
            };
            const uint8_t *tower = P.w_stream + WIN_BYTES;
            const uint8_t *head_w = tower + (size_t)tower_layers * CHUNKS * STAGE_BYTES;
            for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x)
                for (int pass = 0; pass < passes; ++pass) {
                    for (int j0 = 0; j0 < 5; j0 += WIN_KSTEPS_PER_STAGE)
                        push(P.w_stream + j0 * WIN_KSTEP_BYTES, min(WIN_KSTEPS_PER_STAGE, 5 - j0) * WIN_KSTEP_BYTES);
                    for (int c = 0; c < nl * CHUNKS; ++c) push(tower + (size_t)c * STAGE_BYTES, STAGE_BYTES);
                    if (heads) push(head_w, WHEAD_BYTES);
                }
        }
    } else if (warp == 1) {
        // =============================== MMA issuer ===============================
        if (elect_one()) {
            uint32_t it = 0, in_phase = 0, act_phase = 0;
            const uint32_t idesc_128 = P.f16 ? (IDESC_128 & ~IDESC_FMT_BF16) : IDESC_128;
            const uint32_t idesc_head = P.f16 ? (IDESC_HEAD & ~IDESC_FMT_BF16) : IDESC_HEAD;
            auto acquire = [&]() {               // wait for the next stage of the weight stream
                const int s = it % STAGES;
                mbar_wait(bar(B_FULL + s), (it / STAGES) & 1);
                tc_fence_after();
                return sbase + C::OFF_RING + s * STAGE_BYTES;
            };
            auto free_stage = [&](int s) {
                if (CS == 1) umma_commit(bar(B_EMPTY + s));
                else umma_commit_multicast(bar(B_EMPTY + s), CMASK);
            };
            auto release = [&]() { free_stage(it % STAGES); ++it; };
            for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x)
            for (int pass = 0; pass < passes; ++pass) {
                // ---- input conv: 9 taps x 8 (4 real) channels, two taps per K=16 step ----
                mbar_wait(bar(B_IN), in_phase);
                in_phase ^= 1;
                tc_fence_after();
                for (int j0 = 0; j0 < 5; j0 += WIN_KSTEPS_PER_STAGE) {
                    const uint32_t b_rows = acquire();
                    const int j1 = min(j0 + WIN_KSTEPS_PER_STAGE, 5);
                    for (int t = 0; t < TILES; ++t) {
                        const uint32_t in_rows = sbase + C::OFF_IN + (MARGIN + t * TILE_M) * ROW_BYTES;
                        for (int j = j0; j < j1; ++j) {
                            const int tap0 = 2 * j, tap1 = 2 * j + 1;
                            const uint32_t a0 = in_rows + ((tap0 / 3 - 1) * 8 + (tap0 % 3 - 1)) * ROW_BYTES;
                            // the 10th "tap" has all-zero weights: any finite rows will do, take the next row
                            const uint32_t a1 = tap1 < 9 ? in_rows + ((tap1 / 3 - 1) * 8 + (tap1 % 3 - 1)) * ROW_BYTES : a0 + ROW_BYTES;
                            umma(tmem_base + C::TM_ACC + t * 128, make_desc(a0, a1 - a0), make_desc(b_rows + (j - j0) * 2 * W_LBO, W_LBO),
                                 idesc_128, j > 0);
                        }
                        if (j1 == 5) umma_commit(bar(B_ACC + t));
                    }
                    release();
                }
                // ---- tower ----
                // descriptor words: [0,14) start address >> 4, [16,30) LBO >> 4 | hi word: SBO >> 4, version
                const uint32_t a_hi = (uint32_t)(make_desc(0, C::ACT_LBO) >> 32), b_hi = (uint32_t)(make_desc(0, W_LBO) >> 32);
                const uint32_t a_lo0 = (uint32_t)make_desc(sbase + C::OFF_ACT + MARGIN * ROW_BYTES, C::ACT_LBO);
                const uint32_t b_lo0 = (uint32_t)make_desc(sbase + C::OFF_RING, W_LBO);
                constexpr uint32_t A_KSTEP = (2 * C::ACT_LBO) >> 4, B_KSTEP = (2 * W_LBO) >> 4, A_PART = (PART_KG * C::ACT_LBO) >> 4;
                for (int l = 0; l < nl; ++l) {
                    // tower layer l is conv layer l+1.  The second conv of a block accumulates straight ON TOP of the
                    // block's input (the fp32 residual stream kept in TMEM): the skip connection costs no TMEM read, and
                    // consecutive layers never share an accumulator -- which is what lets a layer START on its first input-
                    // channel part (its first nine chunks) while the previous layer's epilogue is still producing the rest.
                    const uint32_t onto_res = (uint32_t)(l & 1);
                    const uint32_t d_col = tmem_base + (onto_res ? C::TM_RES : C::TM_ACC);
#pragma unroll 1
                    for (int part = 0; part < SPLIT; ++part) {
                        for (int t = 0; t < TILES; ++t) mbar_wait(bar(B_ACT + SPLIT * t + part), act_phase);
                        tc_fence_after();
#pragma unroll
                        for (int tap = 0; tap < 9; ++tap) {
                            const int s = it % STAGES;
                            mbar_wait(bar(B_FULL + s), (it / STAGES) & 1);
                            tc_fence_after();
                            const uint32_t b_lo = b_lo0 + s * (STAGE_BYTES >> 4);
                            // tap shift in rows == shift in 16-byte units of the start-address field
                            const uint32_t a_lo = a_lo0 + part * A_PART + (uint32_t)((tap / 3 - 1) * 8 + (tap % 3 - 1));
#pragma unroll
                            for (int t = 0; t < TILES; ++t) {           // every weight stage feeds all of the CTA's tiles
#pragma unroll
                                for (int j = 0; j < PART_MMAS; ++j)
                                    umma_lo(d_col + t * 128, a_lo + t * TILE_M + j * A_KSTEP, a_hi, b_lo + j * B_KSTEP, b_hi, idesc_128,
                                            onto_res | (uint32_t)((part | tap | j) != 0));
                                if (part == SPLIT - 1 && tap == 8) umma_commit(bar(B_ACC + t));
                            }
                            free_stage(s);
                            ++it;
                        }
                    }
                    act_phase ^= 1;
                }
                // ---- heads: [128 rows x 128 ch] x [128 ch x 32] ----
                for (int t = 0; t < TILES; ++t)
                    for (int p = 0; p < SPLIT; ++p) mbar_wait(bar(B_ACT + SPLIT * t + p), act_phase);
                act_phase ^= 1;
                tc_fence_after();
                if (heads) {
                    const uint32_t b_rows = acquire();
                    for (int t = 0; t < TILES; ++t) {
                        const uint32_t a_rows = sbase + C::OFF_ACT + (MARGIN + t * TILE_M) * ROW_BYTES;
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                            umma(tmem_base + C::TM_ACC + t * 128, make_desc(a_rows + 2 * j * C::ACT_LBO, C::ACT_LBO),
                                 make_desc(b_rows + 2 * j * HEAD_LBO, HEAD_LBO), idesc_head, j > 0);
                        umma_commit(bar(B_ACC + t));
                    }
                    release();
                }
            }
        }
    } else if (warp == C::HELPER_WARP) {
        // =============================== softmax helper ===============================
        // total = sum_i exp(logit_i), i ascending, added one by one in double (self_play_client.cpp:212-214): one lane per
        // board of the unit the epilogue warps have just finished; they are already working on the next one.
        // All 32 lanes fetch the numerators chunk by chunk (coalesced, the next chunk in flight while the current one is
        // being added) into a small shared-memory stage; lane b then walks board b's chunk in order.  The chain of 833
        // dependent additions per board (~8 clocks each) is all that remains on the kernel's tail after the last unit.
        if (heads && P.exps && !P.sym8) {
            constexpr int CH = 96;                                  // doubles per board and chunk: 3 per lane
            constexpr int NCH = (AZ_LOGITS + CH - 1) / CH;
            double *stage = reinterpret_cast<double *>(smem + C::OFF_SYM);       // [UNIT_BOARDS][CH] (the sym8 area is free here)
            static_assert(C::UNIT_BOARDS * CH * 8 <= C::SYM_BYTES, "softmax stage fits the sym8 area");
            for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
                helper_wait<TILES>();
                const double *e[C::UNIT_BOARDS];
                int ob[C::UNIT_BOARDS];
#pragma unroll
                for (int b = 0; b < C::UNIT_BOARDS; ++b) {
                    const int board = unit * C::UNIT_BOARDS + b;
                    ob[b] = board < n_boards ? (P.out_map ? __ldg(P.out_map + board) : board) : -1;
                    e[b] = P.exps + (size_t)max(ob[b], 0) * AZ_LOGITS;
                }
                double v[C::UNIT_BOARDS][3];
                auto fetch = [&](int c) {
#pragma unroll
                    for (int b = 0; b < C::UNIT_BOARDS; ++b)
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
                    for (int b = 0; b < C::UNIT_BOARDS; ++b)
#pragma unroll
                        for (int j = 0; j < 3; ++j) stage[b * CH + lane + 32 * j] = v[b][j];
                    __syncwarp();
                    if (c + 1 < NCH) fetch(c + 1);
                    if (lane < C::UNIT_BOARDS) {
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
                if (lane < C::UNIT_BOARDS) {
                    int mine = -1;
#pragma unroll
                    for (int b = 0; b < C::UNIT_BOARDS; ++b) mine = lane == b ? ob[b] : mine;
                    if (mine >= 0) P.totals[mine] = total;
                }
            }
        }
    } else {
        // =============================== epilogue warps ===============================
        const int tile = (warp - 2) >> 2;
        const int quad = warp & 3;                    // TMEM lane quadrant this warp may touch
        const int r = quad * 32 + lane;               // row within the tile == TMEM lane
        const int gtid = (warp - 2 - tile * 4) * 32 + lane;   // 0..127 within the tile's epilogue group
        int bit, cell;
        const bool real = row_is_real(r, bit, cell);
        float *shift_base = reinterpret_cast<float *>(smem + C::OFF_SHIFT) + tile * 2 * F;
        float *vpart = reinterpret_cast<float *>(smem + C::OFF_VPART) + tile * 4;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(quad * 32) << 16);
        uint8_t *act_row = smem + C::OFF_ACT + (MARGIN + tile * TILE_M + r) * ROW_BYTES;
        uint32_t acc_phase = 0;

        float *sym_acc = reinterpret_cast<float *>(smem + C::OFF_SYM);       // sym8 mode: policy sum [833], then the 8 values
        for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x)
        for (int pass = 0; pass < passes; ++pass) {
            // normal mode: the unit's boards; sym8 mode: position `unit`, image sym = pass * UNIT_BOARDS + (row's board in the unit)
            const int sym = P.sym8 ? pass * C::UNIT_BOARDS + tile * 2 + bit : 0;
            const int board = P.sym8 ? unit : unit * C::UNIT_BOARDS + tile * 2 + bit;
            const bool live = real && board < n_boards;
            // ---- stage the input planes of this row: 4 feature channels + 4 zeros, bf16 ----
            {
                uint4 v = make_uint4(0, 0, 0, 0);
                if (live) {
                    float f[4];
                    const int src_cell = P.sym8 ? sym_cell(sym, cell / 7, cell % 7) : cell;    // the image's cell shows this board cell
                    if (IN_KIND == AZ_IN_F32) {
                        const float4 q = reinterpret_cast<const float4 *>(P.input)[(size_t)board * 49 + src_cell];
                        f[0] = q.x; f[1] = q.y; f[2] = q.z; f[3] = q.w;
                    } else {
                        az_position p = reinterpret_cast<const az_position *>(P.input)[board];
                        p.turn &= 1;
                        az::feature_cell(p, src_cell / 7, src_cell % 7, f);
                    }
                    v.x = P.f16 ? pack_f16(f[0], f[1]) : pack_bf16(f[0], f[1]);
                    v.y = P.f16 ? pack_f16(f[2], f[3]) : pack_bf16(f[2], f[3]);
                }
                *reinterpret_cast<uint4 *>(smem + C::OFF_IN + (MARGIN + tile * TILE_M + r) * ROW_BYTES) = v;
                fence_proxy_async();
                mbar_arrive(bar(B_IN));
            }
            for (int l = 0; l < run_layers; ++l) {
                // layer l: 0 = input conv, odd = first conv of a block, even (>0) = second conv (+residual)
                const bool second = l > 0 && (l & 1) == 0;
                const bool writes_res = l == 0 || second;
                float *shift_s = shift_base + (l & 1) * F;     // double-buffered: a fast thread may run one layer ahead
                shift_s[gtid] = __ldg(P.shift + l * F + gtid);
                group_sync(tile);
                mbar_wait(bar(B_ACC + tile), acc_phase);
                acc_phase ^= 1;
                tc_fence_after();
                // 32 channels at a time, TMEM loads software-pipelined one step ahead of the arithmetic.  For the second
                // conv of a block the accumulator already contains the residual (see the MMA issuer).
                const uint32_t src = lane_addr + (second ? C::TM_RES : C::TM_ACC) + tile * 128;
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
                    if (writes_res) tmem_st32(lane_addr + C::TM_RES + tile * 128 + q * 32, a);
                    if (P.f16) store_row<true>(a, act_row + q * 4 * C::ACT_LBO, C::ACT_LBO);
                    else store_row<false>(a, act_row + q * 4 * C::ACT_LBO, C::ACT_LBO);
                    if (P.debug_layers >= 0 && l == run_layers - 1 && live) {
                        float *dst = P.debug_act + ((size_t)board * 49 + cell) * F + q * 32;
                        for (int i = 0; i < 32; ++i) dst[i] = __uint_as_float(a[i]);
                    }
                    if (l > 0 && q < 3 && ((q + 1) % (4 / SPLIT)) == 0) {
                        // a part of this row's channels is in shared memory: the next layer may start on it.  Not after the
                        // input conv: layer 1 reuses the accumulator this epilogue is still reading.
                        fence_proxy_async();
                        tc_fence_before();
                        mbar_arrive(bar(B_ACT + SPLIT * tile + q / (4 / SPLIT)));
                    }
                }
                if (writes_res) tmem_wait_st();
                fence_proxy_async();
                tc_fence_before();
                if (l == 0)
                    for (int p = 0; p < SPLIT - 1; ++p) mbar_arrive(bar(B_ACT + SPLIT * tile + p));
                mbar_arrive(bar(B_ACT + SPLIT * tile + SPLIT - 1));
            }
            if (heads) {
                mbar_wait(bar(B_ACC + tile), acc_phase);
                acc_phase ^= 1;
                tc_fence_after();
                uint32_t a[32];
                tmem_ld32(lane_addr + C::TM_ACC + tile * 128, a);
                tmem_wait_ld();
                float vterm = 0.f;
                const int ob = (P.out_map && board < n_boards) ? __ldg(P.out_map + board) : board;     // output row of this board
                if (live) {
                    if (!P.sym8 && P.logits) {
                        float *dst = P.logits + (size_t)ob * AZ_LOGITS + cell * 17;
#pragma unroll
                        for (int i = 0; i < 17; ++i) dst[i] = __uint_as_float(a[i]);
                    }
                    vterm = __uint_as_float(a[17]) * __ldg(P.fc_w + cell);
                }
                // value head: sum over the board's 49 cells (one board = 2 warps), then tanh
#pragma unroll
                for (int s = 16; s; s >>= 1) vterm += __shfl_xor_sync(0xffffffffu, vterm, s);
                if (lane == 0) vpart[quad] = vterm;
                tc_fence_before();
                group_sync(tile);
                if (gtid < 2) {
                    const float value = tanhf(vpart[2 * gtid] + vpart[2 * gtid + 1] + __ldg(P.fc_b));
                    if (P.sym8) {
                        sym_acc[AZ_LOGITS + pass * C::UNIT_BOARDS + tile * 2 + gtid] = value;
                    } else {
                        const int b = unit * C::UNIT_BOARDS + tile * 2 + gtid;
                        if (b < n_boards) P.values[P.out_map ? __ldg(P.out_map + b) : b] = value;
                    }
                }
                if (P.sym8) {
                    // mean over the 8 images, each rotated back onto the board (spatially only: the 16 direction planes are
                    // not permuted, nn_evals.py:58-62).  Images are added in ascending order (np.mean's order for axis 0), one
                    // image at a time: an image is a permutation of the cells, so its rows never collide.
                    const int my_image = tile * 2 + bit;
                    const int dst_cell = sym_cell(sym, cell / 7, cell % 7);
                    for (int im = 0; im < C::UNIT_BOARDS; ++im) {
                        if (im == my_image && live) {
                            float *dst = sym_acc + dst_cell * 17;
#pragma unroll
                            for (int i = 0; i < 17; ++i) dst[i] = sym == 0 ? __uint_as_float(a[i]) : dst[i] + __uint_as_float(a[i]);
                        }
                        epilogue_sync_all<TILES>();
                    }
                    if (pass == passes - 1) {
                        const int t_all = tile * 128 + gtid;
                        if (board < n_boards) {
                            for (int i = t_all; i < AZ_LOGITS; i += C::EPI_THREADS) P.logits[(size_t)board * AZ_LOGITS + i] = sym_acc[i] * 0.125f;
                            if (t_all == 0) {
                                const float *v = sym_acc + AZ_LOGITS;       // np.mean of 8 floats: numpy's pairwise tree
                                P.values[board] = (((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]))) * 0.125f;
                            }
                        }
                        epilogue_sync_all<TILES>();      // the sum is read before the next position overwrites it
                    }
                } else if (P.exps) {
                    // softmax numerators in double for the tree kernel; the helper warp adds them up
                    if (live) {
                        double *e = P.exps + (size_t)ob * AZ_LOGITS + cell * 17;
#pragma unroll
                        for (int i = 0; i < 17; ++i) e[i] = exp_d(__uint_as_float(a[i]));
                    }
                    __threadfence_block();
                    helper_arrive<TILES>();
                    group_sync(tile);
                } else {
                    group_sync(tile);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (CS > 1) cluster_sync_all();      // no CTA leaves while a peer may still multicast into it
    if (warp == 1) tmem_dealloc(tmem_base, C::TMEM_COLS);
}

}  // namespace

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------

namespace {
// Re-tile the fp32 TF-layout parameters into the UMMA operand images the kernel streams, folding the
// batch-norm scale 1/sqrt(var+eps) of the conv's own BN layer into its output channels.
__device__ __forceinline__ uint16_t to_operand(float w, int f16)
{
    if (f16) { const __half h = __float2half_rn(w); return *reinterpret_cast<const uint16_t *>(&h); }
    const __nv_bfloat16 b = __float2bfloat16_rn(w);
    return *reinterpret_cast<const uint16_t *>(&b);
}

__global__ void k_tile_tower(const float *__restrict__ w_tower, const float *__restrict__ scale, int tower_layers,
                             uint16_t *__restrict__ out, int f16)
{
    // out index: ((((l*CHUNKS + chunk)*PART_KG + kg)*128 + co)*8 + i), chunk = part*9 + tap
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t total = (size_t)tower_layers * CHUNKS * PART_KG * F * 8;
    if (idx >= total) return;
    const int i = (int)(idx & 7);
    const int co = (int)((idx >> 3) & 127);
    const size_t rest = idx >> 10;
    const int kg = (int)(rest % PART_KG);
    const int chunk = (int)((rest / PART_KG) % CHUNKS);
    const int l = (int)(rest / PART_KG / CHUNKS);
    const int part = chunk / 9, tap = chunk % 9;
    const int cin = (part * PART_KG + kg) * 8 + i;
    const float w = w_tower[(((size_t)l * 9 + tap) * F + cin) * F + co] * scale[(size_t)(l + 1) * F + co];
    out[idx] = to_operand(w, f16);
}

__global__ void k_tile_small(const float *__restrict__ w_in, const float *__restrict__ w_policy, const float *__restrict__ w_value,
                             const float *__restrict__ bn_raw, const float *__restrict__ scale, int layers,
                             uint16_t *__restrict__ out_in, uint16_t *__restrict__ out_heads, float *__restrict__ shift, int f16)
{
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < 5 * 2 * F * 8) {                   // input conv: [kstep j][g][cout][i], tap = 2j+g (tap 9 = zero), 4 real channels
        const int i = idx & 7, co = (idx >> 3) & 127, g = (idx >> 10) & 1, j = idx >> 11;
        const int tap = 2 * j + g;
        float w = 0.f;
        if (tap < 9 && i < 4) w = w_in[((size_t)tap * 4 + i) * F + co] * scale[co];
        out_in[idx] = to_operand(w, f16);
    }
    if (idx < KG * HEAD_N * 8) {                 // heads: [kg][row 0..31][i]: rows 0..16 policy planes, row 17 value plane
        const int i = idx & 7, row = (idx >> 3) & 31, kg = idx >> 8;
        const int cin = kg * 8 + i;
        float w = 0.f;
        if (row < 17) w = w_policy[(size_t)cin * 17 + row];
        else if (row == 17) w = w_value[cin];
        out_heads[idx] = to_operand(w, f16);
    }
    if (idx < layers * F) {                      // epilogue shift = -mean * scale, in double like the reference's BN
        const int l = idx / F, c = idx % F;
        const double sc = 1.0 / sqrt((double)bn_raw[(size_t)(2 * l + 1) * F + c] + (double)AZ_BN_EPS);
        shift[idx] = (float)(-(double)bn_raw[(size_t)(2 * l) * F + c] * sc);
    }
}
}  // namespace

int az_net_tc_alloc(AzNet *net)
{
    // one contiguous weight stream per operand format: [input conv][tower][heads], exactly the order the producer walks
    const size_t tower = (size_t)2 * net->blocks * CHUNKS * STAGE_BYTES;
    AZ_CUDA(cudaMalloc(&net->tc_stream, WIN_BYTES + tower + WHEAD_BYTES));
    AZ_CUDA(cudaMalloc(&net->tc_stream16, WIN_BYTES + tower + WHEAD_BYTES));
    net->tc_w_in = reinterpret_cast<__nv_bfloat16 *>(net->tc_stream);
    net->tc_w = reinterpret_cast<__nv_bfloat16 *>(net->tc_stream + WIN_BYTES);
    net->tc_w_heads = reinterpret_cast<__nv_bfloat16 *>(net->tc_stream + WIN_BYTES + tower);
    AZ_CUDA(cudaMalloc(&net->tc_shift, (size_t)net->layers * F * 4));
#define AZ_TC_ATTR(T, K, CSZ) AZ_CUDA(cudaFuncSetAttribute(k_net_tc<T, K, CSZ>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<T>::SMEM_BYTES))
    AZ_TC_ATTR(1, AZ_IN_F32, 1); AZ_TC_ATTR(1, AZ_IN_POS, 1); AZ_TC_ATTR(2, AZ_IN_F32, 1); AZ_TC_ATTR(2, AZ_IN_POS, 1);
    AZ_TC_ATTR(1, AZ_IN_F32, 2); AZ_TC_ATTR(1, AZ_IN_POS, 2); AZ_TC_ATTR(2, AZ_IN_F32, 2); AZ_TC_ATTR(2, AZ_IN_POS, 2);
    AZ_TC_ATTR(1, AZ_IN_F32, 4); AZ_TC_ATTR(1, AZ_IN_POS, 4); AZ_TC_ATTR(2, AZ_IN_F32, 4); AZ_TC_ATTR(2, AZ_IN_POS, 4);
#undef AZ_TC_ATTR
    int rc = az_net_pair_alloc(net);
    if (rc) return rc;
    const char *penv = getenv("AZ_NET_PAIR");
    net->tc_pair = penv ? (atoi(penv) != 0) : AZ_NET_PAIR_DEFAULT;
    const char *cenv = getenv("AZ_NET_CLUSTER");       // CTAs sharing one weight stream by multicast: 1, 2 or 4
    net->tc_cluster = cenv ? (atoi(cenv) == 4 ? 4 : atoi(cenv) == 2 ? 2 : 1) : AZ_NET_CLUSTER_DEFAULT;
    const char *env = getenv("AZ_NET_TILES");          // tuning knob: 1 = two single-tile CTAs per SM, 2 = one two-tile CTA per SM
    net->tc_tiles = (env && atoi(env) == 2) ? 2 : (env && atoi(env) == 1) ? 1 : AZ_NET_TILES_DEFAULT;
    return AZ_OK;
}

int az_net_tc_prepare(az_context *ctx, AzNet *net)
{
    cudaStream_t s = ctx->stream;
    const size_t tower = (size_t)2 * net->blocks * CHUNKS * PART_KG * F * 8;
    const size_t tower_bytes = (size_t)2 * net->blocks * CHUNKS * STAGE_BYTES;
    const int small = std::max(std::max(5 * 2 * F * 8, KG * HEAD_N * 8), net->layers * F);
    for (int f16 = 0; f16 < 2; ++f16) {              // the same tiling in both operand formats (bf16: AZ_NET_BF16, half: AZ_NET_F16)
        uint8_t *base = f16 ? net->tc_stream16 : net->tc_stream;
        k_tile_tower<<<(unsigned)((tower + 255) / 256), 256, 0, s>>>(net->w_tower, net->bn_scale, 2 * net->blocks,
                                                                     reinterpret_cast<uint16_t *>(base + WIN_BYTES), f16);
        k_tile_small<<<(small + 255) / 256, 256, 0, s>>>(net->w_in, net->w_policy, net->w_value, net->bn_raw, net->bn_scale, net->layers,
                                                         reinterpret_cast<uint16_t *>(base), reinterpret_cast<uint16_t *>(base + WIN_BYTES + tower_bytes),
                                                         net->tc_shift, f16);
    }
    AZ_CUDA(cudaGetLastError());
    return az_net_pair_prepare(ctx, net);
}

void az_net_tc_release(AzNet *net)
{
    az_net_pair_release(net);
    if (net->tc_stream) cudaFree(net->tc_stream);
    if (net->tc_stream16) cudaFree(net->tc_stream16);
    net->tc_stream16 = nullptr;
    if (net->tc_shift) cudaFree(net->tc_shift);
    net->tc_stream = nullptr;
    net->tc_w = net->tc_w_in = net->tc_w_heads = nullptr;
    net->tc_shift = nullptr;
}

template <int TILES, int CS>
static cudaError_t tc_launch_cluster(const TcParams &P, int in_kind, int grid, cudaStream_t stream)
{
    using C = Cfg<TILES>;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(C::NUM_THREADS);
    cfg.dynamicSmemBytes = C::SMEM_BYTES;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CS;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (in_kind == AZ_IN_F32) return cudaLaunchKernelEx(&cfg, k_net_tc<TILES, AZ_IN_F32, CS>, P);
    return cudaLaunchKernelEx(&cfg, k_net_tc<TILES, AZ_IN_POS, CS>, P);
}

template <int TILES>
static void tc_launch_variant(az_context *ctx, const TcParams &P, int in_kind, int n, cudaStream_t stream, int cluster)
{
    using C = Cfg<TILES>;
    const int units = P.sym8 ? n : (n + C::UNIT_BOARDS - 1) / C::UNIT_BOARDS;     // sym8: one work item per position
    const int slots = ctx->sm_count * C::CTAS_PER_SM;
    int grid = units < slots ? units : slots;
    if (cluster > 1) {
        grid = (grid + cluster - 1) / cluster * cluster;          // whole clusters; surplus CTAs run an all-padding pass
        if (cluster == 2) tc_launch_cluster<TILES, 2>(P, in_kind, grid, stream);
        else tc_launch_cluster<TILES, 4>(P, in_kind, grid, stream);
        return;
    }
    if (in_kind == AZ_IN_F32)
        k_net_tc<TILES, AZ_IN_F32, 1><<<grid, C::NUM_THREADS, C::SMEM_BYTES, stream>>>(P);
    else
        k_net_tc<TILES, AZ_IN_POS, 1><<<grid, C::NUM_THREADS, C::SMEM_BYTES, stream>>>(P);
}

int az_net_tc_boards_per_round(az_context *ctx)
{
    const int tiles = ctx->net ? ctx->net->tc_tiles : AZ_NET_TILES_DEFAULT;
    const int slots = tiles == 1 ? ctx->sm_count * Cfg<1>::CTAS_PER_SM : ctx->sm_count * Cfg<2>::CTAS_PER_SM;
    return slots * (tiles == 1 ? Cfg<1>::UNIT_BOARDS : Cfg<2>::UNIT_BOARDS);
}

static int tc_launch(az_context *ctx, AzNet *net, const void *d_in, int in_kind, int n, float *d_logits, float *d_values,
                     int debug_layers, float *d_debug, const int *d_count = nullptr, cudaStream_t stream = nullptr, int tiles = 0,
                     double *d_exps = nullptr, double *d_totals = nullptr, int sym8 = 0, int f16 = 0, const int *d_out_map = nullptr)
{
    if (!stream) stream = ctx->stream;
    if (tiles == 0) tiles = net->tc_tiles;
    // plain forward passes can run on CTA pairs (az_net_pair.cu): half the weight ingest per SM for the same arithmetic
    if (net->tc_pair && debug_layers < 0 && !d_exps && !d_out_map && !sym8)
        return az_net_pair_forward(ctx, net, d_in, in_kind, n, d_logits, d_values, d_count, stream, f16);
    TcParams P;
    P.input = d_in;
    P.n = n;
    P.n_ptr = d_count;
    P.layers = net->layers;
    P.debug_layers = debug_layers;
    P.w_stream = f16 ? net->tc_stream16 : net->tc_stream;
    P.f16 = f16;
    P.shift = net->tc_shift;
    P.fc_w = net->fc_w;
    P.fc_b = net->fc_b;
    P.logits = d_logits;
    P.values = d_values;
    P.debug_act = d_debug;
    P.out_map = d_out_map;
    P.exps = d_exps;
    P.totals = d_totals;
    P.sym8 = sym8;
    if (tiles == 1) tc_launch_variant<1>(ctx, P, in_kind, n, stream, net->tc_cluster);
    else tc_launch_variant<2>(ctx, P, in_kind, n, stream, net->tc_cluster);
    ctx->launches++;
    AZ_CUDA(cudaGetLastError());
    return AZ_OK;
}

int az_net_tc_forward(az_context *ctx, AzNet *net, const void *d_in, int in_kind, int n, float *d_logits, float *d_values,
                      const int *d_count, cudaStream_t stream, int tiles, double *d_exps, double *d_totals, int f16, const int *d_out_map)
{
    return tc_launch(ctx, net, d_in, in_kind, n, d_logits, d_values, -1, nullptr, d_count, stream, tiles, d_exps, d_totals, 0, f16, d_out_map);
}

// nn_evals.evaluate for n positions in ONE launch: images generated in the input staging, averaged in the head epilogue
int az_net_tc_forward_sym8(az_context *ctx, AzNet *net, const void *d_in, int in_kind, int n, float *d_logits, float *d_values, int f16)
{
    return tc_launch(ctx, net, d_in, in_kind, n, d_logits, d_values, -1, nullptr, nullptr, nullptr, 0, nullptr, nullptr, 1, f16);
}

// Debug/validation hook (not part of the public header): run the first `conv_layers` convolutions of the
// tensor-core tower and return the fp32 (pre-bf16-rounding) activations [n][49][128] of the last one.
extern "C" int az_net_debug_tower(az_context *ctx, const float *features, int n, int conv_layers, float *act_out)
{
    AZ_REQUIRE(ctx && ctx->net && features && act_out && n > 0, AZ_ERR_ARG, "az_net_debug_tower: bad argument");
    AZ_REQUIRE(conv_layers >= 1 && conv_layers <= ctx->net->layers, AZ_ERR_ARG, "conv_layers out of range");
    const size_t fb = sizeof(float) * AZ_FEATURES * (size_t)n, ab = sizeof(float) * 49 * F * (size_t)n;
    AZ_REQUIRE(ctx->scratch[0].reserve(fb) == 0 && ctx->scratch[1].reserve(ab) == 0, AZ_ERR_CUDA, "scratch alloc");
    AZ_CUDA(cudaMemcpyAsync(ctx->scratch[0].ptr, features, fb, cudaMemcpyHostToDevice, ctx->stream));
    AZ_CUDA(cudaMemsetAsync(ctx->scratch[1].ptr, 0, ab, ctx->stream));
    int rc = tc_launch(ctx, ctx->net, ctx->scratch[0].ptr, AZ_IN_F32, n, nullptr, nullptr, conv_layers, ctx->scratch[1].as<float>());
    if (rc) return rc;
    AZ_CUDA(cudaMemcpyAsync(act_out, ctx->scratch[1].ptr, ab, cudaMemcpyDeviceToHost, ctx->stream));
    AZ_CUDA(cudaStreamSynchronize(ctx->stream));
    AZ_CUDA(cudaGetLastError());
    return AZ_OK;
}
