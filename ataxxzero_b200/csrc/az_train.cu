// az_train.cu -- one optimisation step of the reference's network, hand-written for sm_100a (SURVEY 8f-4).
//
// Replaces model.py:81-101 (Network.build_training: softmax cross-entropy on the 833 policy logits + squared value error +
// 1e-4 * l2_loss of every trainable variable, MomentumOptimizer(lr, 0.9), batch-norm update ops) and the session calls of
// train.py:140-157 (network.train / run_on_samples).  The network is model.py:35-79,116-142: conv3x3 + batch-norm + ReLU
// tower with residual blocks, 1x1 policy conv, 1x1 value conv + 49 -> 1 dense + tanh.
//
// Data layout.  A minibatch of B boards is B*64 GEMM rows: a board is an 8x8 frame whose first row and last column are
// zero padding (row = 8*(x+1) + y), so a 3x3 tap is a constant row shift and the padding cells double as the conv's zero
// border between boards (the geometry of az_net_tc.cu).  Two boards form a TILE of 128 rows.  Tensors live in HBM in
// "tile-blocked" form, which is exactly the shared-memory image the tensor cores read:
//   TB16 (bf16 operands):  [tile][channel group of 8][row 0..127][8]   32 KiB per tile -- activations, dz
//   TB32 (fp32 values):    [tile][channel group of 4][row 0..127][4]   64 KiB per tile -- conv outputs z, gradients
// One bulk copy per 2-KiB channel-group slice brings a tile into shared memory; epilogue threads (one per row) write
// 16-byte pieces that are contiguous across a warp.
//
// Kernels (one launch each per layer; batch statistics need a grid-wide reduction between conv and normalisation):
//   k_conv      forward conv AND data gradient: out[r][n] = sum_tap sum_k in[r + shift(tap)][k] * W[tap][k][n] as 72
//               tcgen05 MMAs (M 128 x N 128 x K 16, fp32 accumulator in TMEM) per tile; the weight image is streamed
//               through a 4-stage ring of 16-KiB bulk copies.  dgrad is the same kernel on the image with taps mirrored
//               and input / output channels swapped.
//   k_wgrad     weight gradient dW[tap][ci][co] = sum_r in[r + shift(tap)][ci] * dz[r][co]: the contraction runs over ROWS,
//               so both operands are read MN-major straight from the same tile-blocked images (no transposes anywhere);
//               a CTA owns three taps (three 128-column accumulators) and a range of tiles and writes its partial sums;
//               k_wgrad_reduce adds the ranges up in a fixed order.
//   k_bn_*      normalise + residual + ReLU, and the second pass of the batch-norm backward.  The batch statistics themselves
//               (sum z, sum z^2 forward; sum g, sum g*xhat backward; fp64 sums) are taken in the conv epilogues.
//   k_heads     per board: policy / value heads, losses, their gradients, the gradient flowing into the tower.
//   k_sgd       L2 term + momentum update, then k_images re-tiles the new weights into the two bf16 operand images.
// Operands are bf16, accumulation and every statistic / master weight / momentum is fp32 (sums in fp64): the step agrees
// with an fp32 PyTorch restatement to bf16 rounding (tests/test_train_gpu.py states the bounds).  The statistics and the head
// gradients are summed with atomics, so like the reference's TensorFlow step the result is not bit-reproducible from run to
// run.  The launches of a step are chained with programmatic dependent launch (pdl_trigger / pdl_wait).
#include "az_net.h"
#include "az_umma.cuh"

#include <algorithm>
#include <cmath>
#include <cstring>

using namespace azumma;

namespace {

constexpr int F = AZ_F;
constexpr int KG = F / 8;                  // 16 channel groups of 8 (bf16 operands)
constexpr int CG = F / 4;                  // 32 channel groups of 4 (fp32 values)
constexpr int TILE_M = 128;
constexpr int MARGIN = 16;                 // zero rows before / after a tile in shared memory (shifts reach +-9)
constexpr int ROW_BYTES = 16;
constexpr int ACT_ROWS = MARGIN + TILE_M + MARGIN;
constexpr int ACT_LBO = ACT_ROWS * ROW_BYTES;          // 2560: distance between channel groups of the staged input tile
constexpr int ACT_BYTES = KG * ACT_LBO;                // 40960
constexpr int SLICE_BYTES = TILE_M * ROW_BYTES;        // 2048: one channel group of a tile in HBM
constexpr int TB16_TILE = KG * SLICE_BYTES;            // 32768 bytes
constexpr int TB32_TILE_F = CG * TILE_M * 4;           // 16384 floats
constexpr int W_LBO = F * ROW_BYTES;                   // 2048: distance between k-groups of the weight operand
constexpr int PART_KG = 8;                             // k-groups per weight stage (64 input channels)
constexpr int STAGE_BYTES = PART_KG * W_LBO;           // 16 KiB: one tap x 64 input channels x 128 output channels
constexpr int CHUNKS = 18;                             // 2 input-channel halves x 9 taps
constexpr int LAYER_IMG_BYTES = CHUNKS * STAGE_BYTES;  // 288 KiB
constexpr int LAYER_W = 9 * F * F;                     // fp32 weights of a layer, TF order [tap][cin][cout]
constexpr int POLICY_PLANES = 17;
constexpr int HEAD_OUT = 18;                           // 17 policy planes + the value plane
constexpr float L2_SCALE = 1e-4f;                      // model.py:90
constexpr float MOMENTUM = 0.9f;                       // model.py:100
constexpr float BN_DECAY = 0.99f;                      // tf.layers.batch_normalization default momentum

__device__ __forceinline__ bool row_is_real(int r, int &board_in_tile, int &cell)
{
    board_in_tile = r >> 6;
    const int w = r & 63;
    const int x = (w >> 3) - 1, y = w & 7;
    cell = x * 7 + y;
    return w >= 8 && y != 7;
}
// Programmatic dependent launch: every kernel of a step lets its successor start at once (its CTAs move in as this kernel's
// drain, and run their prologue -- barrier init, TMEM allocation, zero fills, parameter loads) and itself waits for its
// predecessor's memory before it touches global memory.  No-ops when the launch carries no such dependency.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

__host__ __device__ __forceinline__ int tap_shift(int tap) { return (tap / 3 - 1) * 8 + (tap % 3 - 1); }
__device__ __forceinline__ uint4 load_bf8(const uint8_t *tb16, int tile, int kg, int row)
{
    return *reinterpret_cast<const uint4 *>(tb16 + (size_t)tile * TB16_TILE + kg * SLICE_BYTES + row * ROW_BYTES);
}

// ------------------------------------------------------------------------------------------
// k_conv: forward convolution / data gradient of one layer, one CTA per tile
// ------------------------------------------------------------------------------------------
constexpr int CONV_STAGES = 4;
constexpr int CONV_BARS = 2 * CONV_STAGES + 2;         // full[4], empty[4], input, accumulator
// TILES tiles per CTA share every weight stage: 1 -> two CTAs per SM; 2 -> one CTA per SM whose 16-KiB stages each feed 8 MMAs
// (an SM takes in ~45 B/clk, so with one tile per CTA the 288-KiB weight image, not the tensor pipe, paces the kernel)
template <int TILES>
struct ConvCfg {
    static constexpr int OFF_RING = TILES * ACT_BYTES;
    static constexpr int OFF_BAR = OFF_RING + CONV_STAGES * STAGE_BYTES;
    static constexpr int OFF_TMEM = OFF_BAR + CONV_BARS * 8;
    static constexpr int SMEM = OFF_TMEM + 16;
    static constexpr int THREADS = 64 + TILES * 128;   // warp 0 copies, warp 1 issues MMAs, 4 epilogue warps per tile
    static constexpr int CTAS_PER_SM = TILES == 1 ? 2 : 1;
    static constexpr uint32_t TMEM_COLS = TILES * 128;
};
static_assert(2 * (ConvCfg<1>::SMEM + 1024) <= 228 * 1024, "two 1-tile conv CTAs per SM");
static_assert(ConvCfg<2>::SMEM + 1024 <= 227 * 1024, "one 2-tile conv CTA per SM");

struct ConvParams {
    const uint8_t *in;       // TB16
    const uint8_t *w;        // weight image of the layer
    float *out;              // TB32
    int tiles;               // tiles of the batch (a CTA of the 2-tile variant may own a tile beyond the end)
    int accumulate;          // 1: out += result (the skip connection's gradient is already there)
    double *stats;           // optional [2][F]: per-channel sum / sum of squares of the result are added (batch-norm statistics)
    // data-gradient launches: the result is the gradient w.r.t. the OUTPUT of the layer below; the first pass of that
    // layer's batch-norm backward (sum g, sum g * xhat with g = result masked by the ReLU) is taken here, in registers
    const uint8_t *below_act;      // TB16 output activation of the layer below (ReLU mask); nullptr: no fused statistics
    const float *below_z;          // TB32 its conv output
    const float *below_mean_rstd;  // [2][F]
    double *below_sums;            // [2][F]
};

// column sums of a 32 x 32 block held one row per lane: after five exchange-and-add steps lane c holds the sum of column c
__device__ __forceinline__ float warp_column_sums(float (&v)[32], int lane)
{
#pragma unroll
    for (int half = 16; half; half >>= 1) {
        const bool upper = lane & half;
#pragma unroll
        for (int i = 0; i < half; ++i) {
            const float keep = upper ? v[i + half] : v[i], send = upper ? v[i] : v[i + half];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, half);
        }
    }
    return v[0];
}

template <int TILES>
__global__ void __launch_bounds__(ConvCfg<TILES>::THREADS, ConvCfg<TILES>::CTAS_PER_SM) k_conv(const ConvParams P)
{
    using C = ConvCfg<TILES>;
    extern __shared__ __align__(1024) uint8_t smem[];
    const uint32_t sbase = smem_u32(smem);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tile0 = blockIdx.x * TILES;
    auto bar = [&](int i) { return sbase + C::OFF_BAR + 8 * i; };
    constexpr int B_FULL = 0, B_EMPTY = CONV_STAGES, B_IN = 2 * CONV_STAGES, B_ACC = 2 * CONV_STAGES + 1;
    pdl_trigger();

    for (int i = threadIdx.x; i < TILES * KG * 2 * MARGIN; i += C::THREADS) {    // zero the margins of every channel group
        const int kg = i / (2 * MARGIN), j = i % (2 * MARGIN);                   // (kg runs over the tiles' groups: ACT_BYTES = KG * ACT_LBO)
        const int row = j < MARGIN ? j : TILE_M + j;
        *reinterpret_cast<uint4 *>(smem + kg * ACT_LBO + row * ROW_BYTES) = make_uint4(0, 0, 0, 0);
    }
    if (threadIdx.x == 0) {
        for (int i = 0; i < CONV_BARS; ++i) mbar_init(bar(i), 1);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(sbase + C::OFF_TMEM, C::TMEM_COLS);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t *>(smem + C::OFF_TMEM);
    pdl_wait();

    if (warp == 0) {
        if (lane == 0) {
            int have = 0;
            for (int t = 0; t < TILES; ++t) have += tile0 + t < P.tiles;
            mbar_expect_tx(bar(B_IN), have * TB16_TILE);
            for (int t = 0; t < have; ++t) {
                const uint8_t *src = P.in + (size_t)(tile0 + t) * TB16_TILE;
                for (int kg = 0; kg < KG; ++kg)
                    bulk_g2s(sbase + t * ACT_BYTES + kg * ACT_LBO + MARGIN * ROW_BYTES, src + kg * SLICE_BYTES, SLICE_BYTES, bar(B_IN));
            }
            for (int c = 0; c < CHUNKS; ++c) {
                const int s = c % CONV_STAGES;
                mbar_wait(bar(B_EMPTY + s), ((c / CONV_STAGES) & 1) ^ 1);
                mbar_expect_tx(bar(B_FULL + s), STAGE_BYTES);
                bulk_g2s(sbase + C::OFF_RING + s * STAGE_BYTES, P.w + (size_t)c * STAGE_BYTES, STAGE_BYTES, bar(B_FULL + s));
            }
        }
    } else if (warp == 1) {
        if (elect_one()) {
            constexpr uint32_t IDESC = make_idesc(128, 128, false, false);
            mbar_wait(bar(B_IN), 0);
            tc_fence_after();
            for (int c = 0; c < CHUNKS; ++c) {
                const int s = c % CONV_STAGES, part = c / 9, tap = c % 9;
                mbar_wait(bar(B_FULL + s), (c / CONV_STAGES) & 1);
                tc_fence_after();
                const uint32_t b0 = sbase + C::OFF_RING + s * STAGE_BYTES;
#pragma unroll
                for (int t = 0; t < TILES; ++t) {       // a tile beyond the end multiplies stale shared memory into an accumulator nobody reads
                    const uint32_t a0 = sbase + t * ACT_BYTES + part * PART_KG * ACT_LBO + (MARGIN + tap_shift(tap)) * ROW_BYTES;
#pragma unroll
                    for (int j = 0; j < PART_KG / 2; ++j)
                        umma(tmem_base + t * 128, make_desc(a0 + 2 * j * ACT_LBO, ACT_LBO, 128), make_desc(b0 + 2 * j * W_LBO, W_LBO, 128), IDESC,
                             (uint32_t)((c | j) != 0));
                }
                umma_commit(bar(B_EMPTY + s));
            }
            umma_commit(bar(B_ACC));
        }
    } else {
        const int et = (warp - 2) >> 2;                 // tile of this epilogue warp
        const int quad = warp & 3;                      // TMEM lane quadrant this warp may read
        const int r = quad * 32 + lane;
        const int tile = tile0 + et;
        const bool have_tile = tile < P.tiles;
        int bit, cell;
        const bool real = row_is_real(r, bit, cell);
        float *dst = P.out + (size_t)tile * TB32_TILE_F + r * 4;
        mbar_wait(bar(B_ACC), 0);
        tc_fence_after();
        const uint32_t lane_addr = tmem_base + ((uint32_t)(quad * 32) << 16) + et * 128;
        float *part = reinterpret_cast<float *>(smem);  // [TILES * 4 warps][2][F] column sums; the staged input is dead by now
        const bool sums = P.stats || P.below_act;
        const int pw = et * 4 + quad;
#pragma unroll 1
        for (int q = 0; q < 4; ++q) {
            float v[32];
            if (have_tile) {
                uint32_t a[32];
                tmem_ld32(lane_addr + q * 32, a);
                tmem_wait_ld();
#pragma unroll
                for (int g = 0; g < 8; ++g) {
                    float4 o = real ? make_float4(__uint_as_float(a[4 * g]), __uint_as_float(a[4 * g + 1]), __uint_as_float(a[4 * g + 2]), __uint_as_float(a[4 * g + 3]))
                                    : make_float4(0.f, 0.f, 0.f, 0.f);
                    float4 *p = reinterpret_cast<float4 *>(dst + (q * 8 + g) * TILE_M * 4);
                    if (P.accumulate) { const float4 old = *p; o.x += old.x; o.y += old.y; o.z += old.z; o.w += old.w; }
                    *p = o;
                    v[4 * g] = o.x; v[4 * g + 1] = o.y; v[4 * g + 2] = o.z; v[4 * g + 3] = o.w;
                }
            } else {
#pragma unroll
                for (int i = 0; i < 32; ++i) v[i] = 0.f;
            }
            if (sums) {
                float w[32];
                if (P.stats || !have_tile) {
#pragma unroll
                    for (int i = 0; i < 32; ++i) w[i] = v[i] * v[i];
                } else {
                    // g = gradient where the layer below was active; w = g * xhat of the layer below
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        const uint4 m = load_bf8(P.below_act, tile, q * 4 + g, r);
                        const uint32_t mw[4] = {m.x, m.y, m.z, m.w};
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            if (!(bf16_lo(mw[i]) > 0.f)) v[8 * g + 2 * i] = 0.f;
                            if (!(bf16_hi(mw[i]) > 0.f)) v[8 * g + 2 * i + 1] = 0.f;
                        }
                    }
#pragma unroll
                    for (int g = 0; g < 8; ++g) {
                        const float4 z = *reinterpret_cast<const float4 *>(P.below_z + (size_t)tile * TB32_TILE_F + ((q * 8 + g) * TILE_M + r) * 4);
                        const float zz[4] = {z.x, z.y, z.z, z.w};
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const int c = q * 32 + 4 * g + i;
                            w[4 * g + i] = v[4 * g + i] * ((zz[i] - __ldg(P.below_mean_rstd + c)) * __ldg(P.below_mean_rstd + F + c));
                        }
                    }
                }
                part[(pw * 2 + 0) * F + q * 32 + lane] = warp_column_sums(v, lane);
                part[(pw * 2 + 1) * F + q * 32 + lane] = warp_column_sums(w, lane);
            }
        }
        if (sums) {
            if (TILES == 1) asm volatile("bar.sync 1, 128;" ::: "memory");
            else asm volatile("bar.sync 1, 256;" ::: "memory");
            if (et == 0) {
                double *dst_sums = P.stats ? P.stats : P.below_sums;
                const int c = (warp - 2) * 32 + lane;
#pragma unroll
                for (int k = 0; k < 2; ++k) {
                    double s = 0.0;
#pragma unroll
                    for (int w8 = 0; w8 < TILES * 4; ++w8) s += (double)part[(w8 * 2 + k) * F + c];
                    atomicAdd(dst_sums + k * F + c, s);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, C::TMEM_COLS);
}

// ------------------------------------------------------------------------------------------
// k_wgrad: weight gradient of one layer.  grid = (row ranges, 3 tap groups)
// ------------------------------------------------------------------------------------------
constexpr int WG_STAGES = 3;
constexpr int WG_STAGE_BYTES = ACT_BYTES + TB16_TILE;                // staged input tile (with margins) + dz tile
constexpr int WG_OFF_BAR = WG_STAGES * WG_STAGE_BYTES;
constexpr int WG_BARS = 2 * WG_STAGES + 1;
constexpr int WG_OFF_TMEM = WG_OFF_BAR + WG_BARS * 8;
constexpr int WG_SMEM = WG_OFF_TMEM + 16;
constexpr int WG_THREADS = 192;
constexpr int WG_TAPS = 3;
constexpr int WG_RANGES = 48;                                        // 48 x 3 = 144 CTAs <= 148 SMs

struct WgradParams {
    const uint8_t *in;       // TB16: the layer's input activations
    const uint8_t *dz;       // TB16: gradient w.r.t. the layer's conv output
    float *partial;          // [ranges][9][F][F] fp32: every CTA writes the sums over its own tiles (k_wgrad_reduce adds them up)
    int tiles;
};

__global__ void __launch_bounds__(WG_THREADS, 1) k_wgrad(const WgradParams P)
{
    extern __shared__ __align__(1024) uint8_t smem[];
    const uint32_t sbase = smem_u32(smem);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int t0 = (int)((long long)P.tiles * blockIdx.x / gridDim.x), t1 = (int)((long long)P.tiles * (blockIdx.x + 1) / gridDim.x);
    if (t0 >= t1) return;                               // (the host launches at most one range per tile)
    const int tap0 = blockIdx.y * WG_TAPS;
    auto bar = [&](int i) { return sbase + WG_OFF_BAR + 8 * i; };
    constexpr int B_FULL = 0, B_EMPTY = WG_STAGES, B_ACC = 2 * WG_STAGES;
    pdl_trigger();

    for (int i = threadIdx.x; i < WG_STAGES * KG * 2 * MARGIN; i += WG_THREADS) {
        const int s = i / (KG * 2 * MARGIN), rest = i % (KG * 2 * MARGIN);
        const int kg = rest / (2 * MARGIN), j = rest % (2 * MARGIN);
        const int row = j < MARGIN ? j : TILE_M + j;
        *reinterpret_cast<uint4 *>(smem + s * WG_STAGE_BYTES + kg * ACT_LBO + row * ROW_BYTES) = make_uint4(0, 0, 0, 0);
    }
    if (threadIdx.x == 0) {
        for (int i = 0; i < WG_BARS; ++i) mbar_init(bar(i), 1);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(sbase + WG_OFF_TMEM, 512);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t *>(smem + WG_OFF_TMEM);
    pdl_wait();

    if (warp == 0) {
        if (lane == 0) {
            for (int t = t0; t < t1; ++t) {
                const int it = t - t0, s = it % WG_STAGES;
                mbar_wait(bar(B_EMPTY + s), ((it / WG_STAGES) & 1) ^ 1);
                mbar_expect_tx(bar(B_FULL + s), 2 * TB16_TILE);
                const uint32_t a_dst = sbase + s * WG_STAGE_BYTES;
                const uint8_t *src = P.in + (size_t)t * TB16_TILE;
                for (int kg = 0; kg < KG; ++kg) bulk_g2s(a_dst + kg * ACT_LBO + MARGIN * ROW_BYTES, src + kg * SLICE_BYTES, SLICE_BYTES, bar(B_FULL + s));
                bulk_g2s(a_dst + ACT_BYTES, P.dz + (size_t)t * TB16_TILE, TB16_TILE, bar(B_FULL + s));
            }
        }
    } else if (warp == 1) {
        if (elect_one()) {
            // D[ci][co] += sum over 16 rows of A[ci][row] * B[co][row]: both operands MN-major (rows of 16 B hold 8 channels of
            // one GEMM row); K groups of 8 rows are 128 B apart, channel groups ACT_LBO (input) / SLICE_BYTES (dz) apart
            constexpr uint32_t IDESC = make_idesc(128, 128, true, true);
            for (int t = t0; t < t1; ++t) {
                const int it = t - t0, s = it % WG_STAGES;
                mbar_wait(bar(B_FULL + s), (it / WG_STAGES) & 1);
                tc_fence_after();
                const uint32_t a_base = sbase + s * WG_STAGE_BYTES, b_base = a_base + ACT_BYTES;
#pragma unroll
                for (int j = 0; j < WG_TAPS; ++j) {
                    const uint32_t a0 = a_base + (MARGIN + tap_shift(tap0 + j)) * ROW_BYTES;
#pragma unroll
                    for (int k = 0; k < TILE_M / 16; ++k)
                        umma(tmem_base + j * 128, make_desc(a0 + k * 16 * ROW_BYTES, 128, ACT_LBO), make_desc(b_base + k * 16 * ROW_BYTES, 128, SLICE_BYTES), IDESC,
                             (uint32_t)((it | k) != 0));
                }
                umma_commit(bar(B_EMPTY + s));
            }
            umma_commit(bar(B_ACC));
        }
    } else {
        const int quad = warp & 3;
        const int ci = quad * 32 + lane;                // accumulator row = input channel
        mbar_wait(bar(B_ACC), 0);
        tc_fence_after();
        const uint32_t lane_addr = tmem_base + ((uint32_t)(quad * 32) << 16);
        // partial sums are stored [tap][group of 4 output channels][input channel][4]: the 32 lanes of a warp (consecutive
        // input channels) write 512 contiguous bytes per store
#pragma unroll 1
        for (int j = 0; j < WG_TAPS; ++j) {
            float *dst = P.partial + (size_t)blockIdx.x * LAYER_W + (size_t)(tap0 + j) * F * F + ci * 4;
#pragma unroll 1
            for (int q = 0; q < 4; ++q) {
                uint32_t a[32];
                tmem_ld32(lane_addr + j * 128 + q * 32, a);
                tmem_wait_ld();
#pragma unroll
                for (int i = 0; i < 8; ++i)
                    *reinterpret_cast<float4 *>(dst + (q * 8 + i) * F * 4) =
                        make_float4(__uint_as_float(a[4 * i]), __uint_as_float(a[4 * i + 1]), __uint_as_float(a[4 * i + 2]), __uint_as_float(a[4 * i + 3]));
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// dw[i] = sum over the row ranges of partial[range][i], always in the same order (deterministic).  A block covers 64 float4
// columns; its four thread rows each add a quarter of the ranges, all loads of a quarter in flight together.
constexpr int WGR_COLS = 64, WGR_SPLIT = 4, WGR_PER = WG_RANGES / WGR_SPLIT;
static_assert(WG_RANGES % WGR_SPLIT == 0, "ranges split evenly");
__global__ void __launch_bounds__(WGR_COLS * WGR_SPLIT) k_wgrad_reduce(const float *__restrict__ partial, float *__restrict__ dw, int ranges)
{
    __shared__ float4 part[WGR_SPLIT][WGR_COLS];
    const int col = threadIdx.x % WGR_COLS, quarter = threadIdx.x / WGR_COLS;
    const int i = blockIdx.x * WGR_COLS + col;                    // float4 index
    pdl_trigger();
    pdl_wait();
    float4 v[WGR_PER];
#pragma unroll
    for (int k = 0; k < WGR_PER; ++k) {
        const int r = quarter * WGR_PER + k;
        v[k] = r < ranges ? __ldcg(reinterpret_cast<const float4 *>(partial + (size_t)r * LAYER_W) + i) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    float4 acc = v[0];
#pragma unroll
    for (int k = 1; k < WGR_PER; ++k) { acc.x += v[k].x; acc.y += v[k].y; acc.z += v[k].z; acc.w += v[k].w; }
    part[quarter][col] = acc;
    __syncthreads();
    if (quarter == 0) {
#pragma unroll
        for (int k = 1; k < WGR_SPLIT; ++k) { acc.x += part[k][col].x; acc.y += part[k][col].y; acc.z += part[k][col].z; acc.w += part[k][col].w; }
        // partial layout [tap][cout / 4][cin][4] -> TF layout [tap][cin][cout]
        const int ci = i % F, cg = (i / F) % CG, tap = i / (F * CG);
        reinterpret_cast<float4 *>(dw)[((size_t)tap * F + ci) * CG + cg] = acc;
    }
}

// ------------------------------------------------------------------------------------------
// elementwise / reduction kernels on tile-blocked tensors.  grid = (16 channel groups of 8, tile chunks), 128 threads = rows
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void load8(const float *tb32, int tile, int kg, int row, float (&v)[8])
{
    const float4 a = *reinterpret_cast<const float4 *>(tb32 + (size_t)tile * TB32_TILE_F + ((2 * kg) * TILE_M + row) * 4);
    const float4 b = *reinterpret_cast<const float4 *>(tb32 + (size_t)tile * TB32_TILE_F + ((2 * kg + 1) * TILE_M + row) * 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void store8(float *tb32, int tile, int kg, int row, const float (&v)[8])
{
    *reinterpret_cast<float4 *>(tb32 + (size_t)tile * TB32_TILE_F + ((2 * kg) * TILE_M + row) * 4) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4 *>(tb32 + (size_t)tile * TB32_TILE_F + ((2 * kg + 1) * TILE_M + row) * 4) = make_float4(v[4], v[5], v[6], v[7]);
}
__device__ __forceinline__ void store_bf8(uint8_t *tb16, int tile, int kg, int row, const float (&v)[8])
{
    *reinterpret_cast<uint4 *>(tb16 + (size_t)tile * TB16_TILE + kg * SLICE_BYTES + row * ROW_BYTES) =
        make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
}
// sums of 16 per-thread values over the 128 threads of the block, added to 16 doubles in global memory
__device__ __forceinline__ void block_sum16_to_global(float (&v)[16], double *dst0, double *dst1, int kg)
{
    __shared__ float part[4][16];
#pragma unroll
    for (int i = 0; i < 16; ++i)
#pragma unroll
        for (int s = 16; s; s >>= 1) v[i] += __shfl_xor_sync(0xffffffffu, v[i], s);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0)
#pragma unroll
        for (int i = 0; i < 16; ++i) part[warp][i] = v[i];
    __syncthreads();
    if (threadIdx.x < 16) {
        const int i = threadIdx.x;
        const double s = (double)part[0][i] + (double)part[1][i] + (double)part[2][i] + (double)part[3][i];
        atomicAdd((i < 8 ? dst0 : dst1) + kg * 8 + (i & 7), s);
    }
}

__global__ void __launch_bounds__(128) k_stage_input(const int8_t *__restrict__ feats, uint8_t *__restrict__ act0, int n)
{
    const int tile = blockIdx.x, row = threadIdx.x;
    int bit, cell;
    const bool real = row_is_real(row, bit, cell);
    const int board = tile * 2 + bit;
    pdl_trigger();
    pdl_wait();
    float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (real && board < n) {
        const char4 f = *reinterpret_cast<const char4 *>(feats + ((size_t)board * 49 + cell) * 4);
        v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w;
    }
    store_bf8(act0, tile, 0, row, v);
}

struct BnApplyParams {
    const float *z;          // TB32 conv output
    const double *sums;      // [2][F] batch sum / sum of squares (training)
    const float *gamma, *beta;
    float *mean_rstd;        // [2][F] written for the backward pass
    float *moving;           // [2][F] moving mean / variance: updated in training, used when use_moving
    float *h32;              // TB32 fp32 residual stream
    uint8_t *act_out;        // TB16
    int res_mode;            // 0: plain, 1: h32 = out, 2: out = relu(bn + h32), h32 = out
    int tiles, n, use_moving;
};

__global__ void __launch_bounds__(128) k_bn_apply(const BnApplyParams P)
{
    const int kg = blockIdx.x, row = threadIdx.x;
    const double cnt = (double)P.n * 49.0;
    pdl_trigger();
    pdl_wait();
    // per-channel scale / shift: the mean and the E[z^2] - mean^2 subtraction in double, the rest in float
    const double inv_cnt = 1.0 / cnt;
    float sc[8], sh[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int c = kg * 8 + i;
        float mean, var;
        if (P.use_moving) { mean = P.moving[c]; var = P.moving[F + c]; }
        else {
            const double m = P.sums[c] * inv_cnt;
            mean = (float)m;
            var = fmaxf((float)(P.sums[F + c] * inv_cnt - m * m), 0.f);
        }
        const float rstd = 1.f / sqrtf(var + AZ_BN_EPS);
        sc[i] = P.gamma[c] * rstd;
        sh[i] = P.beta[c] - mean * sc[i];
        if (blockIdx.y == 0 && row == i && !P.use_moving) {
            P.mean_rstd[c] = mean;
            P.mean_rstd[F + c] = rstd;
            // tf.layers.batch_normalization update ops (fused kernel: the moving variance takes the unbiased estimate)
            P.moving[c] = BN_DECAY * P.moving[c] + (1.f - BN_DECAY) * mean;
            P.moving[F + c] = BN_DECAY * P.moving[F + c] + (1.f - BN_DECAY) * (var * (float)(cnt / fmax(cnt - 1.0, 1.0)));
        }
    }
    int bit, cell;
    const bool real = row_is_real(row, bit, cell);
    for (int tile = blockIdx.y; tile < P.tiles; tile += gridDim.y) {
        const bool live = real && tile * 2 + bit < P.n;
        float v[8];
        load8(P.z, tile, kg, row, v);
        if (P.res_mode == 2) {
            float h[8];
            load8(P.h32, tile, kg, row, h);
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = v[i] * sc[i] + sh[i] + h[i];
        } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = v[i] * sc[i] + sh[i];
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = live ? fmaxf(v[i], 0.f) : 0.f;
        if (P.res_mode) store8(P.h32, tile, kg, row, v);
        store_bf8(P.act_out, tile, kg, row, v);
    }
}

struct BnBwdParams {
    float *d_out;            // TB32 gradient w.r.t. the layer's output (after ReLU); write_g: replaced by the masked gradient
    const uint8_t *act_out;  // TB16 the layer's output (ReLU mask)
    const float *z;          // TB32 conv output
    const float *mean_rstd;  // [2][F]
    const float *gamma;
    double *sums;            // [2][F]: sum g, sum g * xhat
    uint8_t *dz;             // TB16 gradient w.r.t. the conv output
    float *g_gamma, *g_beta; // [F] each
    int write_g, tiles, n;
};

__device__ __forceinline__ void masked_grad(const BnBwdParams &P, int tile, int kg, int row, const float (&mean)[8], const float (&rstd)[8], float (&g)[8],
                                            float (&xh)[8])
{
    float z[8];
    load8(P.d_out, tile, kg, row, g);
    load8(P.z, tile, kg, row, z);
    const uint4 a = load_bf8(P.act_out, tile, kg, row);
    const uint32_t w[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        if (!(bf16_lo(w[i]) > 0.f)) g[2 * i] = 0.f;
        if (!(bf16_hi(w[i]) > 0.f)) g[2 * i + 1] = 0.f;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) xh[i] = (z[i] - mean[i]) * rstd[i];
}

__global__ void __launch_bounds__(128) k_bn_bwd_stats(const BnBwdParams P)
{
    const int kg = blockIdx.x, row = threadIdx.x;
    pdl_trigger();
    pdl_wait();
    float mean[8], rstd[8], acc[16];
#pragma unroll
    for (int i = 0; i < 8; ++i) { mean[i] = P.mean_rstd[kg * 8 + i]; rstd[i] = P.mean_rstd[F + kg * 8 + i]; acc[i] = 0.f; acc[8 + i] = 0.f; }
    for (int tile = blockIdx.y; tile < P.tiles; tile += gridDim.y) {
        float g[8], xh[8];
        masked_grad(P, tile, kg, row, mean, rstd, g, xh);           // padding rows: activation 0 -> g = 0
#pragma unroll
        for (int i = 0; i < 8; ++i) { acc[i] += g[i]; acc[8 + i] += g[i] * xh[i]; }
    }
    block_sum16_to_global(acc, P.sums, P.sums + F, kg);
}

__global__ void __launch_bounds__(128) k_bn_bwd_apply(const BnBwdParams P)
{
    const int kg = blockIdx.x, row = threadIdx.x;
    const float inv = 1.f / ((float)P.n * 49.f);
    pdl_trigger();
    pdl_wait();
    float mean[8], rstd[8], sg[8], sgx[8], k[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int c = kg * 8 + i;
        mean[i] = P.mean_rstd[c];
        rstd[i] = P.mean_rstd[F + c];
        sg[i] = (float)P.sums[c];
        sgx[i] = (float)P.sums[F + c];
        k[i] = P.gamma[c] * rstd[i];
        if (blockIdx.y == 0 && row == i) { P.g_beta[c] = sg[i]; P.g_gamma[c] = sgx[i]; }
    }
    int bit, cell;
    const bool real = row_is_real(row, bit, cell);
    for (int tile = blockIdx.y; tile < P.tiles; tile += gridDim.y) {
        const bool live = real && tile * 2 + bit < P.n;
        float g[8], xh[8], d[8];
        masked_grad(P, tile, kg, row, mean, rstd, g, xh);
#pragma unroll
        for (int i = 0; i < 8; ++i) d[i] = live ? k[i] * (g[i] - sg[i] * inv - xh[i] * sgx[i] * inv) : 0.f;
        store_bf8(P.dz, tile, kg, row, d);
        if (P.write_g) store8(P.d_out, tile, kg, row, g);
    }
}

// ------------------------------------------------------------------------------------------
// k_heads: one block per board
// ------------------------------------------------------------------------------------------
struct HeadsParams {
    const float *h32;        // TB32 tower output (fp32)
    const float *w_policy;   // [F][17]
    const float *w_value;    // [F]
    const float *fc_w;       // [49]
    const float *fc_b;       // [1]
    const float *policies;   // [n][833] desired policy
    const float *values;     // [n] desired value
    double *loss;            // [0] += policy loss / n, [1] += value loss / n
    float *logits_out;       // optional [n][833]
    float *values_out;       // optional [n]
    float *d_h;              // TB32 gradient w.r.t. the tower output (training)
    float *g_policy, *g_value, *g_fc_w, *g_fc_b;
    int n, train;
};

__device__ __forceinline__ float block_reduce(float v, float *scratch, bool is_max)
{
#pragma unroll
    for (int s = 16; s; s >>= 1) {
        const float o = __shfl_xor_sync(0xffffffffu, v, s);
        v = is_max ? fmaxf(v, o) : v + o;
    }
    __syncthreads();
    if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
    __syncthreads();
    return is_max ? fmaxf(fmaxf(scratch[0], scratch[1]), fmaxf(scratch[2], scratch[3])) : (scratch[0] + scratch[1]) + (scratch[2] + scratch[3]);
}

// A block walks boards blockIdx.x, blockIdx.x + gridDim.x, ...; the weight gradients of the heads are summed in registers over
// its boards and added to global memory once (one atomic per weight and block instead of one per weight and board).
__global__ void __launch_bounds__(128) k_heads(const HeadsParams P, int boards)
{
    __shared__ __align__(16) float h[49][F + 4];         // rows 16-byte aligned: read four channels at a time
    __shared__ float wp[F][HEAD_OUT];
    __shared__ float out[49][HEAD_OUT];
    __shared__ __align__(8) float dl[49][HEAD_OUT];
    __shared__ float scratch[4];
    const int tid = threadIdx.x;
    pdl_trigger();
    pdl_wait();
    for (int i = tid; i < F * HEAD_OUT; i += 128) {
        const int c = i / HEAD_OUT, p = i % HEAD_OUT;
        wp[c][p] = p < POLICY_PLANES ? P.w_policy[c * POLICY_PLANES + p] : P.w_value[c];
    }
    float gw[HEAD_OUT];                                  // thread = channel: d loss / d (policy | value conv weights of this channel)
    float wreg[HEAD_OUT];                                // ... and those weights themselves
#pragma unroll
    for (int p = 0; p < HEAD_OUT; ++p) {
        gw[p] = 0.f;
        wreg[p] = p < POLICY_PLANES ? P.w_policy[tid * POLICY_PLANES + p] : P.w_value[tid];
    }
    float g_fc = 0.f, g_bias = 0.f;                      // threads 0..48: d loss / d fc_w[tid]; thread 0: d loss / d fc_b
    double loss_p = 0.0, loss_v = 0.0;
    const float inv_n = 1.f / (float)P.n;

    for (int board = blockIdx.x; board < boards; board += gridDim.x) {
        const int tile = board >> 1, row0 = (board & 1) * 64;
        if (board >= P.n) {                              // the empty half of the last tile: no gradient
            if (P.train)
                for (int i = tid; i < CG * 64; i += 128) {
                    const int cg = i / 64, r = i % 64;
                    *reinterpret_cast<float4 *>(P.d_h + (size_t)tile * TB32_TILE_F + (cg * TILE_M + row0 + r) * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
                }
            continue;
        }
        __syncthreads();                                 // the previous board's h / dl are no longer read
        for (int i = tid; i < CG * 49; i += 128) {
            const int cg = i / 49, cell = i % 49;
            const int r = row0 + 8 + (cell / 7) * 8 + cell % 7;
            const float4 v = *reinterpret_cast<const float4 *>(P.h32 + (size_t)tile * TB32_TILE_F + (cg * TILE_M + r) * 4);
            h[cell][cg * 4] = v.x; h[cell][cg * 4 + 1] = v.y; h[cell][cg * 4 + 2] = v.z; h[cell][cg * 4 + 3] = v.w;
        }
        __syncthreads();
        if (tid < 7 * HEAD_OUT) {                        // thread = (row of 7 cells, output plane): 7 dot products over the channels
            const int p = tid % HEAD_OUT, c0 = tid / HEAD_OUT * 7;
            float acc[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll 2
            for (int c = 0; c < F; c += 4) {
                const float w0 = wp[c][p], w1 = wp[c + 1][p], w2 = wp[c + 2][p], w3 = wp[c + 3][p];
#pragma unroll
                for (int j = 0; j < 7; ++j) {
                    const float4 hv = *reinterpret_cast<const float4 *>(&h[c0 + j][c]);
                    acc[j] += hv.x * w0 + hv.y * w1 + hv.z * w2 + hv.w * w3;
                }
            }
#pragma unroll
            for (int j = 0; j < 7; ++j) out[c0 + j][p] = acc[j];
        }
        __syncthreads();
        // value head: tanh(sum_cell v[cell] * fc_w[cell] + fc_b)   (model.py:70-76; cells in x-major order like tf.reshape of NHWC)
        const float vterm = tid < 49 ? out[tid][POLICY_PLANES] * P.fc_w[tid] : 0.f;
        const float pre = block_reduce(vterm, scratch, false) + P.fc_b[0];
        const float val = tanhf(pre);
        // policy: softmax cross-entropy with soft labels over the 833 logits (model.py:83-86)
        float mx = -INFINITY;
        for (int i = tid; i < AZ_LOGITS; i += 128) mx = fmaxf(mx, out[i / POLICY_PLANES][i % POLICY_PLANES]);
        mx = block_reduce(mx, scratch, true);
        float se = 0.f, st = 0.f, stx = 0.f;
        const float *target = P.policies + (size_t)board * AZ_LOGITS;
        for (int i = tid; i < AZ_LOGITS; i += 128) {
            const float x = out[i / POLICY_PLANES][i % POLICY_PLANES] - mx, t = target[i];
            se += expf(x);
            st += t;
            stx += t * x;
        }
        se = block_reduce(se, scratch, false);
        st = block_reduce(st, scratch, false);
        stx = block_reduce(stx, scratch, false);
        const float lse = logf(se);
        const float want = P.values[board];
        if (tid == 0) {
            loss_p += (double)(st * lse - stx) * (double)inv_n;                      // -sum t * (x - lse)
            loss_v += (double)((want - val) * (want - val)) * (double)inv_n;
            if (P.values_out) P.values_out[board] = val;
        }
        if (P.logits_out)
            for (int i = tid; i < AZ_LOGITS; i += 128) P.logits_out[(size_t)board * AZ_LOGITS + i] = out[i / POLICY_PLANES][i % POLICY_PLANES];
        if (!P.train) continue;

        // gradients of the (mean over the batch) losses w.r.t. the head outputs
        const float dpre = 2.f * (val - want) * inv_n * (1.f - val * val);
        for (int i = tid; i < AZ_LOGITS; i += 128) {
            const int cell = i / POLICY_PLANES, p = i % POLICY_PLANES;
            dl[cell][p] = (expf(out[cell][p] - mx - lse) * st - target[i]) * inv_n;
        }
        if (tid < 49) {
            dl[tid][POLICY_PLANES] = dpre * P.fc_w[tid];
            g_fc += dpre * out[tid][POLICY_PLANES];
        }
        if (tid == 0) g_bias += dpre;
        __syncthreads();
        // thread = channel: weight gradients of the two 1x1 convs, and the gradient flowing into the tower (which replaces
        // this thread's own column of h[][])
        for (int cell = 0; cell < 49; ++cell) {
            const float hv = h[cell][tid];
            float acc = 0.f;
#pragma unroll
            for (int p = 0; p < HEAD_OUT; p += 2) {
                const float2 d = *reinterpret_cast<const float2 *>(&dl[cell][p]);
                gw[p] += hv * d.x;
                gw[p + 1] += hv * d.y;
                acc += d.x * wreg[p] + d.y * wreg[p + 1];
            }
            h[cell][tid] = acc;
        }
        __syncthreads();
        for (int i = tid; i < CG * 64; i += 128) {
            const int cg = i / 64, r = i % 64;
            const int x = (r >> 3) - 1, y = r & 7;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r >= 8 && y != 7) {
                const int cell = x * 7 + y;
                v = make_float4(h[cell][cg * 4], h[cell][cg * 4 + 1], h[cell][cg * 4 + 2], h[cell][cg * 4 + 3]);
            }
            *reinterpret_cast<float4 *>(P.d_h + (size_t)tile * TB32_TILE_F + (cg * TILE_M + row0 + r) * 4) = v;
        }
    }
    if (tid == 0) {
        atomicAdd(P.loss + 0, loss_p);
        atomicAdd(P.loss + 1, loss_v);
    }
    if (P.train) {
#pragma unroll
        for (int p = 0; p < POLICY_PLANES; ++p) atomicAdd(P.g_policy + tid * POLICY_PLANES + p, gw[p]);
        atomicAdd(P.g_value + tid, gw[POLICY_PLANES]);
        if (tid < 49) atomicAdd(P.g_fc_w + tid, g_fc);
        if (tid == 0) atomicAdd(P.g_fc_b, g_bias);
    }
}

// ------------------------------------------------------------------------------------------
// optimiser + operand images
// ------------------------------------------------------------------------------------------
// model.py:88-100: loss += 1e-4 * sum(w^2)/2 over every trainable variable; accum = 0.9 * accum + grad; w -= lr * accum
__global__ void __launch_bounds__(256) k_sgd(float *__restrict__ theta, float *__restrict__ mom, const float *__restrict__ grad, size_t count, float lr,
                                             double *__restrict__ reg_loss)
{
    __shared__ float part[8];
    float sq = 0.f;
    pdl_trigger();
    pdl_wait();
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x) {
        const float w = theta[i];
        const float m = MOMENTUM * mom[i] + (grad[i] + L2_SCALE * w);
        mom[i] = m;
        theta[i] = w - lr * m;
        sq += w * w;
    }
#pragma unroll
    for (int s = 16; s; s >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, s);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = sq;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int i = 0; i < 8; ++i) s += (double)part[i];
        atomicAdd(reg_loss, 0.5 * (double)L2_SCALE * s);
    }
}

// fp32 weights [layer][tap][cin][cout] -> the two bf16 operand images of every layer:
//   forward:  chunk = (cin / 64) * 9 + tap,        k-group (cin % 64) / 8,  row cout, element cin % 8
//   dgrad:    chunk = (cout / 64) * 9 + (8 - tap), k-group (cout % 64) / 8, row cin,  element cout % 8
__global__ void __launch_bounds__(256) k_images(const float *__restrict__ theta, __nv_bfloat16 *__restrict__ img_f, __nv_bfloat16 *__restrict__ img_b, size_t count)
{
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    pdl_wait();
    if (idx >= count) return;
    const int co = (int)(idx % F), ci = (int)((idx / F) % F), tap = (int)((idx / (F * F)) % 9);
    const size_t l = idx / LAYER_W;
    const __nv_bfloat16 w = __float2bfloat16_rn(theta[idx]);
    const size_t base = l * (size_t)(LAYER_IMG_BYTES / 2);
    img_f[base + ((size_t)(((ci / 64) * 9 + tap) * PART_KG + (ci % 64) / 8) * F + co) * 8 + ci % 8] = w;
    img_b[base + ((size_t)(((co / 64) * 9 + (8 - tap)) * PART_KG + (co % 64) / 8) * F + ci) * 8 + co % 8] = w;
}

// launch with the programmatic-stream-serialisation attribute (see pdl_trigger); AZ_TRAIN_PDL=0 launches plainly
template <typename... KArgs, typename... Args>
void launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args... args)
{
    static const bool pdl = !(getenv("AZ_TRAIN_PDL") && atoi(getenv("AZ_TRAIN_PDL")) == 0);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

template <typename T>
int dev_alloc(T **p, size_t count, bool zero = true)
{
    if (cudaMalloc(reinterpret_cast<void **>(p), std::max<size_t>(count, 1) * sizeof(T)) != cudaSuccess) return az_fail(AZ_ERR_CUDA, "az_trainer: device allocation of %zu bytes failed", count * sizeof(T));
    if (zero && cudaMemset(*p, 0, std::max<size_t>(count, 1) * sizeof(T)) != cudaSuccess) return az_fail(AZ_ERR_CUDA, "az_trainer: memset failed");
    return AZ_OK;
}

}  // namespace

struct az_trainer {
    az_context *ctx = nullptr;
    int max_batch = 0, max_tiles = 0, blocks = 0, layers = 0;
    size_t count = 0;                                   // trainable parameters (layer 0 padded to 128 input channels)
    size_t off_gamma = 0, off_beta = 0, off_policy = 0, off_value = 0, off_fcw = 0, off_fcb = 0;
    float *theta = nullptr, *mom = nullptr, *grad = nullptr, *moving = nullptr, *mean_rstd = nullptr;
    uint8_t *img_f = nullptr, *img_b = nullptr, *act = nullptr, *dz = nullptr;
    float *z = nullptr, *h32 = nullptr, *d_h = nullptr, *d_y = nullptr, *wg_partial = nullptr;
    double *fsum = nullptr, *bsum = nullptr, *loss = nullptr;
    uint32_t *d_plies = nullptr;                        // resident ply table (az_trainer_set_games)
    std::vector<uint32_t> h_plies;                      // host copy: the picks of every step are validated against it
    unsigned long long *d_offsets = nullptr;
    uint32_t *d_meta = nullptr;
    int8_t *d_feats = nullptr;
    float *d_pol = nullptr, *d_val = nullptr, *d_logits = nullptr, *d_values_out = nullptr;
    double *h_loss = nullptr;                           // pinned
    cudaEvent_t ev[2] = {nullptr, nullptr};             // around the kernels of a step (inputs already on the device)
    float last_step_ms = 0.f;
    int ew_chunks = 64;                                 // blocks per channel group in the elementwise kernels
    int conv_tiles = 0;                                 // 0: by batch size
    int skip = 0;                                       // AZ_TRAIN_SKIP bits (timing studies only, results are wrong): 1 forward conv, 2 data
                                                        // gradient, 4 weight gradient + reduce, 8 k_bn_apply, 16 k_bn_bwd_apply, 32 heads
    bool loaded = false;
    unsigned long long steps = 0, launches = 0;

    uint8_t *act_at(int l) const { return act + (size_t)l * max_tiles * TB16_TILE; }
    float *z_at(int l) const { return z + (size_t)l * max_tiles * TB32_TILE_F; }
};

namespace {

// batches that fill the GPU more than once with one tile per CTA run the 2-tile variant (AZ_TRAIN_CONV_TILES=1|2 forces one)
void launch_conv(az_trainer *t, int tiles, cudaStream_t s, const ConvParams &C)
{
    const int variant = t->conv_tiles ? t->conv_tiles : (tiles > t->ctx->sm_count ? 2 : 1);
    if (variant == 2) launch(k_conv<2>, dim3((tiles + 1) / 2), dim3(ConvCfg<2>::THREADS), ConvCfg<2>::SMEM, s, C);
    else launch(k_conv<1>, dim3(tiles), dim3(ConvCfg<1>::THREADS), ConvCfg<1>::SMEM, s, C);
}

int refresh_images(az_trainer *t)
{
    const size_t n = (size_t)t->layers * LAYER_W;
    launch(k_images, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, t->ctx->stream, t->theta, reinterpret_cast<__nv_bfloat16 *>(t->img_f), reinterpret_cast<__nv_bfloat16 *>(t->img_b), n);
    t->launches++;
    AZ_CUDA(cudaGetLastError());
    return AZ_OK;
}

int stage_batch(az_trainer *t, const int8_t *features, const float *policies, const float *values, int n)
{
    cudaStream_t s = t->ctx->stream;
    AZ_CUDA(cudaMemcpyAsync(t->d_feats, features, (size_t)n * AZ_FEATURES, cudaMemcpyHostToDevice, s));
    AZ_CUDA(cudaMemcpyAsync(t->d_pol, policies, (size_t)n * AZ_LOGITS * sizeof(float), cudaMemcpyHostToDevice, s));
    AZ_CUDA(cudaMemcpyAsync(t->d_val, values, (size_t)n * sizeof(float), cudaMemcpyHostToDevice, s));
    return AZ_OK;
}

// forward pass over the staged batch; training: batch statistics (+ moving-average update), else the moving statistics
int forward(az_trainer *t, int n, bool train, bool want_outputs)
{
    cudaStream_t s = t->ctx->stream;
    const int tiles = (n + 1) / 2;
    const dim3 ew(KG, std::min(tiles, t->ew_chunks));
    launch(k_stage_input, dim3(tiles), dim3(128), 0, s, t->d_feats, t->act_at(0), n);
    t->launches++;
    for (int l = 0; l < t->layers; ++l) {
        // training: the conv epilogue also adds up the batch statistics of its output
        ConvParams C{t->act_at(l), t->img_f + (size_t)l * LAYER_IMG_BYTES, t->z_at(l), tiles, 0, train ? t->fsum + (size_t)l * 2 * F : nullptr, nullptr, nullptr, nullptr, nullptr};
        if (!(t->skip & 1)) launch_conv(t, tiles, s, C);
        BnApplyParams B{};
        B.z = t->z_at(l);
        B.sums = t->fsum + (size_t)l * 2 * F;
        B.gamma = t->theta + t->off_gamma + (size_t)l * F;
        B.beta = t->theta + t->off_beta + (size_t)l * F;
        B.mean_rstd = t->mean_rstd + (size_t)l * 2 * F;
        B.moving = t->moving + (size_t)l * 2 * F;
        B.h32 = t->h32;
        B.act_out = t->act_at(l + 1);
        B.res_mode = l == 0 ? 1 : (l & 1) ? 0 : 2;
        B.tiles = tiles;
        B.n = n;
        B.use_moving = train ? 0 : 1;
        if (!(t->skip & 8)) launch(k_bn_apply, dim3(ew), dim3(128), 0, s, B);
        t->launches += 2;
    }
    HeadsParams H{};
    H.h32 = t->h32;
    H.w_policy = t->theta + t->off_policy;
    H.w_value = t->theta + t->off_value;
    H.fc_w = t->theta + t->off_fcw;
    H.fc_b = t->theta + t->off_fcb;
    H.policies = t->d_pol;
    H.values = t->d_val;
    H.loss = t->loss;
    H.logits_out = want_outputs ? t->d_logits : nullptr;
    H.values_out = want_outputs ? t->d_values_out : nullptr;
    H.d_h = t->d_h;
    H.g_policy = t->grad + t->off_policy;
    H.g_value = t->grad + t->off_value;
    H.g_fc_w = t->grad + t->off_fcw;
    H.g_fc_b = t->grad + t->off_fcb;
    H.n = n;
    H.train = train ? 1 : 0;
    if (!(t->skip & 32)) launch(k_heads, dim3(std::min(2 * tiles, 2 * t->ctx->sm_count)), dim3(128), 0, s, H, 2 * tiles);
    t->launches++;
    AZ_CUDA(cudaGetLastError());
    return AZ_OK;
}

int backward(az_trainer *t, int n)
{
    cudaStream_t s = t->ctx->stream;
    const int tiles = (n + 1) / 2;
    const dim3 ew(KG, std::min(tiles, t->ew_chunks));
    for (int l = t->layers - 1; l >= 0; --l) {
        const bool second = l > 0 && (l & 1) == 0;      // second conv of a block: its output gradient is the block's (d_h)
        const bool first = (l & 1) == 1;
        BnBwdParams B{};
        B.d_out = (l == 0 || second) ? t->d_h : t->d_y;
        B.act_out = t->act_at(l + 1);
        B.z = t->z_at(l);
        B.mean_rstd = t->mean_rstd + (size_t)l * 2 * F;
        B.gamma = t->theta + t->off_gamma + (size_t)l * F;
        B.sums = t->bsum + (size_t)l * 2 * F;
        B.dz = t->dz;
        B.g_gamma = t->grad + t->off_gamma + (size_t)l * F;
        B.g_beta = t->grad + t->off_beta + (size_t)l * F;
        B.write_g = second ? 1 : 0;                     // the masked gradient also flows down the skip connection
        B.tiles = tiles;
        B.n = n;
        if (l == t->layers - 1) {                       // every other layer's sums come out of the data-gradient epilogue above it
            launch(k_bn_bwd_stats, dim3(ew), dim3(128), 0, s, B);
            t->launches++;
        }
        if (!(t->skip & 16)) launch(k_bn_bwd_apply, dim3(ew), dim3(128), 0, s, B);
        const int ranges = std::min(WG_RANGES, tiles);       // every range owns at least one tile
        WgradParams W{t->act_at(l), t->dz, t->wg_partial, tiles};
        if (!(t->skip & 4)) launch(k_wgrad, dim3(dim3(ranges, 9 / WG_TAPS)), dim3(WG_THREADS), WG_SMEM, s, W);
        if (!(t->skip & 4)) launch(k_wgrad_reduce, dim3(LAYER_W / 4 / WGR_COLS), dim3(WGR_COLS * WGR_SPLIT), 0, s, t->wg_partial, t->grad + (size_t)l * LAYER_W, ranges);
        t->launches += 3;
        if (l > 0) {
            // data gradient: into d_y for the second conv of a block, ON TOP of the skip gradient in d_h for the first
            ConvParams C{t->dz, t->img_b + (size_t)l * LAYER_IMG_BYTES, first ? t->d_h : t->d_y, tiles, first ? 1 : 0, nullptr,
                         t->act_at(l), t->z_at(l - 1), t->mean_rstd + (size_t)(l - 1) * 2 * F, t->bsum + (size_t)(l - 1) * 2 * F};
            if (!(t->skip & 2)) launch_conv(t, tiles, s, C);
            t->launches++;
        }
    }
    AZ_CUDA(cudaGetLastError());
    return AZ_OK;
}

int check_batch(az_trainer *t, const void *a, const void *b, const void *c, int n, const char *who)
{
    AZ_REQUIRE(t && a && b && c, AZ_ERR_ARG, "%s: null argument", who);
    AZ_REQUIRE(t->loaded, AZ_ERR_STATE, "%s: no weights loaded (az_trainer_load)", who);
    AZ_REQUIRE(n >= 2 && n <= t->max_batch, AZ_ERR_ARG, "%s: batch of %d boards, this trainer takes 2..%d", who, n, t->max_batch);
    return AZ_OK;
}

}  // namespace

extern "C" int az_trainer_create(az_context *ctx, int max_batch, int blocks, az_trainer **out)
{
    AZ_REQUIRE(ctx && out, AZ_ERR_ARG, "az_trainer_create: null argument");
    AZ_REQUIRE(max_batch >= 2 && max_batch <= (1 << 16), AZ_ERR_ARG, "az_trainer_create: max_batch %d out of range", max_batch);
    AZ_REQUIRE(blocks >= 0 && blocks <= 64, AZ_ERR_ARG, "az_trainer_create: blocks %d out of range", blocks);
    AZ_CUDA(cudaSetDevice(ctx->device));
    az_trainer *t = new az_trainer();
    t->ctx = ctx;
    t->max_batch = max_batch;
    t->max_tiles = (max_batch + 1) / 2;
    t->blocks = blocks;
    t->layers = 1 + 2 * blocks;
    if (getenv("AZ_TRAIN_SKIP")) t->skip = atoi(getenv("AZ_TRAIN_SKIP"));
    if (getenv("AZ_TRAIN_CONV_TILES")) t->conv_tiles = atoi(getenv("AZ_TRAIN_CONV_TILES")) == 2 ? 2 : 1;
    if (getenv("AZ_TRAIN_EW_CHUNKS")) t->ew_chunks = std::max(1, atoi(getenv("AZ_TRAIN_EW_CHUNKS")));
    const size_t L = (size_t)t->layers, T = (size_t)t->max_tiles;
    t->off_gamma = L * LAYER_W;
    t->off_beta = t->off_gamma + L * F;
    t->off_policy = t->off_beta + L * F;
    t->off_value = t->off_policy + (size_t)F * POLICY_PLANES;
    t->off_fcw = t->off_value + F;
    t->off_fcb = t->off_fcw + 49;
    t->count = t->off_fcb + 1;
    int rc = 0;
    rc |= dev_alloc(&t->theta, t->count);
    rc |= dev_alloc(&t->mom, t->count);
    rc |= dev_alloc(&t->grad, t->count);
    rc |= dev_alloc(&t->moving, L * 2 * F);
    rc |= dev_alloc(&t->mean_rstd, L * 2 * F);
    rc |= dev_alloc(&t->img_f, L * LAYER_IMG_BYTES);
    rc |= dev_alloc(&t->img_b, L * LAYER_IMG_BYTES);
    rc |= dev_alloc(&t->act, (L + 1) * T * TB16_TILE);          // zero: channel groups 1..15 of the input layer stay zero
    rc |= dev_alloc(&t->dz, T * TB16_TILE);
    rc |= dev_alloc(&t->z, L * T * TB32_TILE_F);
    rc |= dev_alloc(&t->h32, T * TB32_TILE_F);
    rc |= dev_alloc(&t->d_h, T * TB32_TILE_F);
    rc |= dev_alloc(&t->d_y, T * TB32_TILE_F);
    rc |= dev_alloc(&t->wg_partial, (size_t)WG_RANGES * LAYER_W);
    rc |= dev_alloc(&t->fsum, L * 2 * F);
    rc |= dev_alloc(&t->bsum, L * 2 * F);
    rc |= dev_alloc(&t->loss, 4);
    rc |= dev_alloc(&t->d_offsets, (size_t)max_batch);
    rc |= dev_alloc(&t->d_meta, (size_t)max_batch);
    rc |= dev_alloc(&t->d_feats, (size_t)max_batch * AZ_FEATURES);
    rc |= dev_alloc(&t->d_pol, (size_t)max_batch * AZ_LOGITS);
    rc |= dev_alloc(&t->d_val, (size_t)max_batch);
    rc |= dev_alloc(&t->d_logits, (size_t)max_batch * AZ_LOGITS);
    rc |= dev_alloc(&t->d_values_out, (size_t)max_batch);
    if (!rc && cudaMallocHost(&t->h_loss, 4 * sizeof(double)) != cudaSuccess) rc = az_fail(AZ_ERR_CUDA, "az_trainer_create: pinned host alloc");
    if (!rc && (cudaEventCreate(&t->ev[0]) != cudaSuccess || cudaEventCreate(&t->ev[1]) != cudaSuccess)) rc = az_fail(AZ_ERR_CUDA, "az_trainer_create: event");
    if (!rc && (cudaFuncSetAttribute(k_conv<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvCfg<1>::SMEM) != cudaSuccess ||
                cudaFuncSetAttribute(k_conv<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvCfg<2>::SMEM) != cudaSuccess ||
                cudaFuncSetAttribute(k_wgrad, cudaFuncAttributeMaxDynamicSharedMemorySize, WG_SMEM) != cudaSuccess))
        rc = az_fail(AZ_ERR_CUDA, "az_trainer_create: cudaFuncSetAttribute: %s", cudaGetErrorString(cudaGetLastError()));
    if (rc) { az_trainer_destroy(t); return rc; }
    *out = t;
    return AZ_OK;
}

extern "C" void az_trainer_destroy(az_trainer *t)
{
    if (!t) return;
    cudaStreamSynchronize(t->ctx->stream);
    void *bufs[] = {t->theta, t->mom, t->grad, t->moving, t->mean_rstd, t->img_f, t->img_b, t->act, t->dz, t->z, t->h32, t->d_h, t->d_y,
                    t->fsum, t->bsum, t->loss, t->wg_partial, t->d_plies, t->d_offsets, t->d_meta, t->d_feats, t->d_pol, t->d_val, t->d_logits, t->d_values_out};
    for (void *p : bufs) cudaFree(p);
    if (t->h_loss) cudaFreeHost(t->h_loss);
    for (cudaEvent_t e : t->ev)
        if (e) cudaEventDestroy(e);
    delete t;
}

// `packed`: the vector az_net_load takes (model.Network.packed()): conv list, then the moving mean / variance pairs.
// Like a fresh train.py run (train.py:112-120: initialize_all_variables, then load_model assigns the saved tensors), the
// batch-norm gamma / beta start at 1 / 0 and the momentum accumulators at 0.
extern "C" int az_trainer_load(az_trainer *t, const float *packed, size_t count)
{
    AZ_REQUIRE(t && packed, AZ_ERR_ARG, "az_trainer_load: null argument");
    const size_t L = (size_t)t->layers;
    const size_t want = 9 * 4 * F + (L - 1) * LAYER_W + (size_t)F * POLICY_PLANES + F + 49 + 1 + L * 2 * F;
    AZ_REQUIRE(count == want, AZ_ERR_ARG, "az_trainer_load: %zu values, a %d-filter %d-block network has %zu", count, F, t->blocks, want);
    std::vector<float> theta(t->count, 0.f), moving(L * 2 * F);
    const float *p = packed;
    for (int tap = 0; tap < 9; ++tap)
        for (int ci = 0; ci < 4; ++ci)
            for (int co = 0; co < F; ++co) theta[((size_t)tap * F + ci) * F + co] = *p++;
    std::memcpy(theta.data() + LAYER_W, p, (L - 1) * LAYER_W * sizeof(float));
    p += (L - 1) * LAYER_W;
    for (size_t i = 0; i < L * F; ++i) theta[t->off_gamma + i] = 1.f;
    std::memcpy(theta.data() + t->off_policy, p, ((size_t)F * POLICY_PLANES + F + 49 + 1) * sizeof(float));
    p += (size_t)F * POLICY_PLANES + F + 49 + 1;
    std::memcpy(moving.data(), p, L * 2 * F * sizeof(float));
    for (float v : theta) AZ_REQUIRE(std::isfinite(v), AZ_ERR_ARG, "az_trainer_load: non-finite weight");
    cudaStream_t s = t->ctx->stream;
    AZ_CUDA(cudaMemcpyAsync(t->theta, theta.data(), t->count * sizeof(float), cudaMemcpyHostToDevice, s));
    AZ_CUDA(cudaMemcpyAsync(t->moving, moving.data(), moving.size() * sizeof(float), cudaMemcpyHostToDevice, s));
    AZ_CUDA(cudaMemsetAsync(t->mom, 0, t->count * sizeof(float), s));
    int rc = refresh_images(t);
    if (rc) return rc;
    AZ_CUDA(cudaStreamSynchronize(s));
    t->loaded = true;
    t->steps = 0;
    return AZ_OK;
}

namespace {
// everything of a step after the minibatch has been staged in d_feats / d_pol / d_val (stream-ordered)
int step_staged(az_trainer *t, int n, float learning_rate, float *losses, const char *who)
{
    cudaStream_t s = t->ctx->stream;
    int rc;
    AZ_CUDA(cudaEventRecord(t->ev[0], s));
    if ((rc = forward(t, n, true, false))) return rc;
    if ((rc = backward(t, n))) return rc;
    launch(k_sgd, dim3(592), dim3(256), 0, s, t->theta, t->mom, t->grad, t->count, learning_rate, t->loss + 2);
    t->launches++;
    if ((rc = refresh_images(t))) return rc;
    AZ_CUDA(cudaEventRecord(t->ev[1], s));
    AZ_CUDA(cudaMemcpyAsync(t->h_loss, t->loss, 4 * sizeof(double), cudaMemcpyDeviceToHost, s));
    AZ_CUDA(cudaStreamSynchronize(s));
    AZ_CUDA(cudaGetLastError());
    AZ_CUDA(cudaEventElapsedTime(&t->last_step_ms, t->ev[0], t->ev[1]));
    t->steps++;
    if (losses) { losses[0] = (float)t->h_loss[0]; losses[1] = (float)t->h_loss[1]; losses[2] = (float)t->h_loss[2]; }
    for (int i = 0; i < 3 && !t->skip; ++i) AZ_REQUIRE(std::isfinite(t->h_loss[i]), AZ_ERR_STATE, "%s: loss term %d is not finite (diverged)", who, i);
    return AZ_OK;
}

int zero_step_accumulators(az_trainer *t)
{
    cudaStream_t s = t->ctx->stream;
    const size_t L = (size_t)t->layers;
    AZ_CUDA(cudaMemsetAsync(t->grad, 0, t->count * sizeof(float), s));
    AZ_CUDA(cudaMemsetAsync(t->fsum, 0, L * 2 * F * sizeof(double), s));
    AZ_CUDA(cudaMemsetAsync(t->bsum, 0, L * 2 * F * sizeof(double), s));
    AZ_CUDA(cudaMemsetAsync(t->loss, 0, 4 * sizeof(double), s));
    return AZ_OK;
}
}  // namespace

// network.train(minibatch, learning_rate) (model.py:116-127, train.py:154-155).  losses = {policy, value, regularisation} of
// THIS minibatch before the update, as the reference's loss tensors would evaluate in the same session call.
extern "C" int az_trainer_step(az_trainer *t, const int8_t *features, const float *policies, const float *values, int n, float learning_rate, float *losses)
{
    int rc = check_batch(t, features, policies, values, n, "az_trainer_step");
    if (rc) return rc;
    AZ_REQUIRE(std::isfinite(learning_rate) && learning_rate >= 0.f, AZ_ERR_ARG, "az_trainer_step: learning rate %g", (double)learning_rate);
    if ((rc = zero_step_accumulators(t))) return rc;
    if ((rc = stage_batch(t, features, policies, values, n))) return rc;
    return step_staged(t, n, learning_rate, losses, "az_trainer_step");
}

// The games a run trains on, as the binary ply table of az_samples_extract (train_data.pack_entries): uploaded ONCE and kept
// on the device (train.py:105-110 loads its games once, too).
extern "C" int az_trainer_set_games(az_trainer *t, const uint32_t *plies, size_t ply_words)
{
    AZ_REQUIRE(t && plies && ply_words >= 6, AZ_ERR_ARG, "az_trainer_set_games: bad argument");
    AZ_CUDA(cudaStreamSynchronize(t->ctx->stream));
    if (t->d_plies) cudaFree(t->d_plies);
    t->d_plies = nullptr;
    int rc = dev_alloc(&t->d_plies, ply_words, false);
    if (rc) return rc;
    t->h_plies.assign(plies, plies + ply_words);
    AZ_CUDA(cudaMemcpy(t->d_plies, plies, ply_words * sizeof(uint32_t), cudaMemcpyHostToDevice));
    return AZ_OK;
}

// One training step on the samples (offsets, meta) of the resident games -- az_samples_extract's sample description
// (get_sample_from_entries, train.py:43-77) -- without a host round trip: the extraction kernel writes the minibatch
// straight into the trainer's input buffers.
extern "C" int az_trainer_step_picks(az_trainer *t, const uint64_t *offsets, const uint32_t *meta, int n, float learning_rate, float *losses)
{
    AZ_REQUIRE(t && offsets && meta, AZ_ERR_ARG, "az_trainer_step_picks: null argument");
    AZ_REQUIRE(t->loaded, AZ_ERR_STATE, "az_trainer_step_picks: no weights loaded (az_trainer_load)");
    AZ_REQUIRE(t->d_plies, AZ_ERR_STATE, "az_trainer_step_picks: no games loaded (az_trainer_set_games)");
    AZ_REQUIRE(n >= 2 && n <= t->max_batch, AZ_ERR_ARG, "az_trainer_step_picks: batch of %d boards, this trainer takes 2..%d", n, t->max_batch);
    AZ_REQUIRE(std::isfinite(learning_rate) && learning_rate >= 0.f, AZ_ERR_ARG, "az_trainer_step_picks: learning rate %g", (double)learning_rate);
    const size_t words = t->h_plies.size();
    for (int i = 0; i < n; ++i) {               // a record must lie inside the table, entries included (as in az_samples_extract)
        AZ_REQUIRE(offsets[i] + 6 <= words, AZ_ERR_ARG, "az_trainer_step_picks: sample %d points outside the ply table", i);
        const size_t need = ((meta[i] >> 6) & 1u) ? 6 + 2 * (size_t)(t->h_plies[offsets[i] + 4] >> 16) : 6;
        AZ_REQUIRE(offsets[i] + need <= words, AZ_ERR_ARG, "az_trainer_step_picks: sample %d has a truncated record", i);
        const int result = (int)((meta[i] >> 1) & 3u);
        AZ_REQUIRE(result == 1 || result == 2, AZ_ERR_ARG, "az_trainer_step_picks: sample %d has result %d", i, result);
    }
    cudaStream_t s = t->ctx->stream;
    int rc;
    if ((rc = zero_step_accumulators(t))) return rc;
    AZ_CUDA(cudaMemcpyAsync(t->d_offsets, offsets, (size_t)n * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
    AZ_CUDA(cudaMemcpyAsync(t->d_meta, meta, (size_t)n * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
    if ((rc = az_samples_extract_dev(t->ctx, t->d_plies, t->d_offsets, t->d_meta, n, t->d_feats, t->d_pol, t->d_val))) return rc;
    t->launches++;
    return step_staged(t, n, learning_rate, losses, "az_trainer_step_picks");
}

// run_on_samples(policy_loss.eval / value_loss.eval) (model.py:129-142, train.py:141-142): is_training = False, so the
// batch-norm layers use their moving statistics; any n (evaluated in slices of max_batch, weighted mean).
// logits [n][833] / values_out [n] are optional.
extern "C" int az_trainer_eval(az_trainer *t, const int8_t *features, const float *policies, const float *values, int n, float *losses, float *logits,
                               float *values_out)
{
    AZ_REQUIRE(t && features && policies && values, AZ_ERR_ARG, "az_trainer_eval: null argument");
    AZ_REQUIRE(t->loaded, AZ_ERR_STATE, "az_trainer_eval: no weights loaded (az_trainer_load)");
    AZ_REQUIRE(n >= 1, AZ_ERR_ARG, "az_trainer_eval: empty batch");
    cudaStream_t s = t->ctx->stream;
    double sum_p = 0.0, sum_v = 0.0;
    for (int base = 0; base < n; base += t->max_batch) {
        const int m = std::min(t->max_batch, n - base);
        AZ_CUDA(cudaMemsetAsync(t->loss, 0, 4 * sizeof(double), s));
        int rc = stage_batch(t, features + (size_t)base * AZ_FEATURES, policies + (size_t)base * AZ_LOGITS, values + base, m);
        if (rc) return rc;
        if ((rc = forward(t, m, false, logits || values_out))) return rc;
        AZ_CUDA(cudaMemcpyAsync(t->h_loss, t->loss, 4 * sizeof(double), cudaMemcpyDeviceToHost, s));
        if (logits) AZ_CUDA(cudaMemcpyAsync(logits + (size_t)base * AZ_LOGITS, t->d_logits, (size_t)m * AZ_LOGITS * sizeof(float), cudaMemcpyDeviceToHost, s));
        if (values_out) AZ_CUDA(cudaMemcpyAsync(values_out + base, t->d_values_out, (size_t)m * sizeof(float), cudaMemcpyDeviceToHost, s));
        AZ_CUDA(cudaStreamSynchronize(s));
        sum_p += t->h_loss[0] * m;
        sum_v += t->h_loss[1] * m;
    }
    if (losses) { losses[0] = (float)(sum_p / n); losses[1] = (float)(sum_v / n); }
    return AZ_OK;
}

// model.save_model (model.py:173-183): conv / dense weights and the batch-norm MOVING statistics, in az_net_load's order.
// The learned gamma / beta are not part of the file format (SURVEY App. B-5).
extern "C" int az_trainer_export(az_trainer *t, float *packed, size_t count)
{
    AZ_REQUIRE(t && packed, AZ_ERR_ARG, "az_trainer_export: null argument");
    AZ_REQUIRE(t->loaded, AZ_ERR_STATE, "az_trainer_export: no weights loaded");
    const size_t L = (size_t)t->layers;
    const size_t want = 9 * 4 * F + (L - 1) * LAYER_W + (size_t)F * POLICY_PLANES + F + 49 + 1 + L * 2 * F;
    AZ_REQUIRE(count == want, AZ_ERR_ARG, "az_trainer_export: room for %zu values, the network has %zu", count, want);
    std::vector<float> theta(t->count), moving(L * 2 * F);
    AZ_CUDA(cudaStreamSynchronize(t->ctx->stream));
    AZ_CUDA(cudaMemcpy(theta.data(), t->theta, t->count * sizeof(float), cudaMemcpyDeviceToHost));
    AZ_CUDA(cudaMemcpy(moving.data(), t->moving, moving.size() * sizeof(float), cudaMemcpyDeviceToHost));
    float *p = packed;
    for (int tap = 0; tap < 9; ++tap)
        for (int ci = 0; ci < 4; ++ci)
            for (int co = 0; co < F; ++co) *p++ = theta[((size_t)tap * F + ci) * F + co];
    std::memcpy(p, theta.data() + LAYER_W, (L - 1) * LAYER_W * sizeof(float));
    p += (L - 1) * LAYER_W;
    std::memcpy(p, theta.data() + t->off_policy, ((size_t)F * POLICY_PLANES + F + 49 + 1) * sizeof(float));
    p += (size_t)F * POLICY_PLANES + F + 49 + 1;
    std::memcpy(p, moving.data(), L * 2 * F * sizeof(float));
    return AZ_OK;
}

extern "C" unsigned long long az_trainer_launches(const az_trainer *t) { return t ? t->launches : 0; }
// device time of the last step's kernels (CUDA events on the launching stream; the batch was already in HBM)
extern "C" float az_trainer_last_step_ms(const az_trainer *t) { return t ? t->last_step_ms : 0.f; }

// Test hook (not in the public header's stable part): copies an internal tensor of the LAST step to the host.
//   what = "z" / "act": conv output / activation of `layer` as float [n][7][7][F]      (act: layer 0 = input .. layers = tower output)
//          "grad_conv": float [9][F][F] of `layer`; "grad_gamma" / "grad_beta" / "gamma" / "beta": float [F] of `layer`;
//          "grad_heads": float [F*17 + F + 49 + 1]; "moving": float [2][F] of `layer`
//          "d_h": float [n][7][7][F] (`layer` 0): after a step, the gradient of the loss with respect to layer 0's output.  k_heads
//          writes the tower output's gradient there, each block's skip and data gradient replace / add to it on the way down,
//          and layer 0's batch-norm backward reads it without overwriting it (write_g = 0).  After an eval call: unchanged.
extern "C" int az_trainer_debug_read(az_trainer *t, const char *what, int layer, int n, float *out, size_t count)
{
    AZ_REQUIRE(t && what && out, AZ_ERR_ARG, "az_trainer_debug_read: null argument");
    AZ_CUDA(cudaStreamSynchronize(t->ctx->stream));
    const std::string w(what);
    auto flat = [&](const float *src, size_t m) -> int {
        AZ_REQUIRE(count == m, AZ_ERR_ARG, "az_trainer_debug_read(%s): %zu values expected, room for %zu", what, m, count);
        AZ_CUDA(cudaMemcpy(out, src, m * sizeof(float), cudaMemcpyDeviceToHost));
        return AZ_OK;
    };
    if (w == "z" || w == "act" || w == "d_h") {
        const int max_layer = w == "act" ? t->layers : t->layers - 1;
        AZ_REQUIRE(layer >= 0 && layer <= max_layer && n >= 1 && n <= t->max_batch, AZ_ERR_ARG, "az_trainer_debug_read(%s): layer %d / n %d out of range", what, layer, n);
        AZ_REQUIRE(count == (size_t)n * 49 * F, AZ_ERR_ARG, "az_trainer_debug_read(%s): %zu values expected", what, (size_t)n * 49 * F);
        const size_t tiles = (size_t)(n + 1) / 2;
        if (w == "act") {
            std::vector<uint16_t> buf(tiles * TB16_TILE / 2);
            AZ_CUDA(cudaMemcpy(buf.data(), t->act_at(layer), buf.size() * 2, cudaMemcpyDeviceToHost));
            for (int b = 0; b < n; ++b)
                for (int cell = 0; cell < 49; ++cell)
                    for (int c = 0; c < F; ++c) {
                        const int row = (b & 1) * 64 + 8 + (cell / 7) * 8 + cell % 7;
                        const uint32_t bits = (uint32_t)buf[(size_t)(b / 2) * (TB16_TILE / 2) + ((size_t)(c / 8) * TILE_M + row) * 8 + c % 8] << 16;
                        float f;
                        std::memcpy(&f, &bits, 4);
                        out[((size_t)b * 49 + cell) * F + c] = f;
                    }
        } else {
            std::vector<float> buf(tiles * TB32_TILE_F);
            AZ_CUDA(cudaMemcpy(buf.data(), w == "z" ? t->z_at(layer) : t->d_h, buf.size() * 4, cudaMemcpyDeviceToHost));
            for (int b = 0; b < n; ++b)
                for (int cell = 0; cell < 49; ++cell)
                    for (int c = 0; c < F; ++c) {
                        const int row = (b & 1) * 64 + 8 + (cell / 7) * 8 + cell % 7;
                        out[((size_t)b * 49 + cell) * F + c] = buf[(size_t)(b / 2) * TB32_TILE_F + ((size_t)(c / 4) * TILE_M + row) * 4 + c % 4];
                    }
        }
        return AZ_OK;
    }
    AZ_REQUIRE(layer >= 0 && layer < t->layers, AZ_ERR_ARG, "az_trainer_debug_read(%s): layer %d out of range", what, layer);
    if (w == "grad_conv") return flat(t->grad + (size_t)layer * LAYER_W, LAYER_W);
    if (w == "conv") return flat(t->theta + (size_t)layer * LAYER_W, LAYER_W);
    if (w == "grad_gamma") return flat(t->grad + t->off_gamma + (size_t)layer * F, F);
    if (w == "grad_beta") return flat(t->grad + t->off_beta + (size_t)layer * F, F);
    if (w == "gamma") return flat(t->theta + t->off_gamma + (size_t)layer * F, F);
    if (w == "beta") return flat(t->theta + t->off_beta + (size_t)layer * F, F);
    if (w == "moving") return flat(t->moving + (size_t)layer * 2 * F, 2 * F);
    if (w == "grad_heads") return flat(t->grad + t->off_policy, (size_t)F * POLICY_PLANES + F + 49 + 1);
    return az_fail(AZ_ERR_ARG, "az_trainer_debug_read: unknown tensor '%s'", what);
}
