// az_net.cu -- policy/value network forward pass: weight upload, the fp32 reference-accurate
// kernel, and the C-ABI entry points.  (The bf16 tcgen05 path lives in az_net_tc.cu.)
//
// Network (model.py:38-79): conv3x3(4->128)+BN+ReLU; 12 x [conv3x3+BN+ReLU, conv3x3+BN, +skip, ReLU];
// policy = conv1x1(128->17); value = conv1x1(128->1) -> reshape 49 (x-major) -> fc(49->1)+b -> tanh.
// Spatial axes: first = x (file), second = y (top-down); features/logits are [x][y][c].
#include "az_net.h"
#include "az_rules.cuh"

#include <cmath>
#include <cstring>

namespace {

constexpr int F = AZ_F;
constexpr int NB = 2;                 // boards per CTA
constexpr int PW = 9, PPB = 81;       // zero-haloed 9x9 board -> a tap is a constant row shift
constexpr int ROWS = NB * PPB;        // 162 padded rows per buffer
constexpr int THREADS = 256;
constexpr int POS_PER_THREAD = 13;    // ceil(98 real positions / 8 position groups)
constexpr size_t SMEM_FP32 = sizeof(float) * (2 * ROWS * F + 2 * 49 + 8);

__device__ __forceinline__ int padded_row(int r)   // r in [0, 98): real position index over the CTA's boards
{
    const int b = r / 49, cell = r % 49;
    return b * PPB + (cell / 7 + 1) * PW + (cell % 7 + 1);
}

// out[pr][c] = epilogue( sum_{tap, cin} in[pr + shift(tap)][cin] * w[tap][cin][c] )
template <bool RESIDUAL>
__device__ __forceinline__ void conv3x3(const float *__restrict__ in, float *__restrict__ out,
                                        const float *__restrict__ w, int cin_count,
                                        const float *__restrict__ mean, const float *__restrict__ scale)
{
    const int cg = threadIdx.x & 31;          // 4 output channels 4cg..4cg+3
    const int pg = threadIdx.x >> 5;          // position group (warp-uniform -> smem broadcast)
    float4 acc[POS_PER_THREAD];
    int rows[POS_PER_THREAD];
#pragma unroll
    for (int k = 0; k < POS_PER_THREAD; ++k) {
        acc[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        const int r = pg + 8 * k;
        rows[k] = padded_row(r < NB * 49 ? r : 0);
    }
    for (int tap = 0; tap < 9; ++tap) {
        const int shift = (tap / 3 - 1) * PW + (tap % 3 - 1);
        const float *wt = w + (size_t)tap * cin_count * F + 4 * cg;
        for (int c = 0; c < cin_count; c += 4) {
            const float4 w0 = __ldg(reinterpret_cast<const float4 *>(wt + (size_t)(c + 0) * F));
            const float4 w1 = __ldg(reinterpret_cast<const float4 *>(wt + (size_t)(c + 1) * F));
            const float4 w2 = __ldg(reinterpret_cast<const float4 *>(wt + (size_t)(c + 2) * F));
            const float4 w3 = __ldg(reinterpret_cast<const float4 *>(wt + (size_t)(c + 3) * F));
#pragma unroll
            for (int k = 0; k < POS_PER_THREAD; ++k) {
                const float4 a = *reinterpret_cast<const float4 *>(in + (rows[k] + shift) * F + c);
                acc[k].x = fmaf(a.x, w0.x, acc[k].x); acc[k].y = fmaf(a.x, w0.y, acc[k].y);
                acc[k].z = fmaf(a.x, w0.z, acc[k].z); acc[k].w = fmaf(a.x, w0.w, acc[k].w);
                acc[k].x = fmaf(a.y, w1.x, acc[k].x); acc[k].y = fmaf(a.y, w1.y, acc[k].y);
                acc[k].z = fmaf(a.y, w1.z, acc[k].z); acc[k].w = fmaf(a.y, w1.w, acc[k].w);
                acc[k].x = fmaf(a.z, w2.x, acc[k].x); acc[k].y = fmaf(a.z, w2.y, acc[k].y);
                acc[k].z = fmaf(a.z, w2.z, acc[k].z); acc[k].w = fmaf(a.z, w2.w, acc[k].w);
                acc[k].x = fmaf(a.w, w3.x, acc[k].x); acc[k].y = fmaf(a.w, w3.y, acc[k].y);
                acc[k].z = fmaf(a.w, w3.z, acc[k].z); acc[k].w = fmaf(a.w, w3.w, acc[k].w);
            }
        }
    }
    const float4 m = *reinterpret_cast<const float4 *>(mean + 4 * cg);
    const float4 s = *reinterpret_cast<const float4 *>(scale + 4 * cg);
    __syncthreads();            // everyone finished reading `in` (out may alias the residual buffer only)
#pragma unroll
    for (int k = 0; k < POS_PER_THREAD; ++k) {
        if (pg + 8 * k >= NB * 49) continue;
        float4 v;
        v.x = (acc[k].x - m.x) * s.x; v.y = (acc[k].y - m.y) * s.y;
        v.z = (acc[k].z - m.z) * s.z; v.w = (acc[k].w - m.w) * s.w;
        float4 *dst = reinterpret_cast<float4 *>(out + rows[k] * F + 4 * cg);
        if (RESIDUAL) {
            const float4 r = *dst;
            v.x += r.x; v.y += r.y; v.z += r.z; v.w += r.w;
        }
        v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f);
        *dst = v;
    }
    __syncthreads();
}

template <int IN_KIND>
__global__ void __launch_bounds__(THREADS, 1)
k_net_fp32(const void *__restrict__ input, int n_max, const int *__restrict__ n_ptr, AzNet net, float *__restrict__ logits,
           float *__restrict__ values)
{
    const int n = n_ptr ? min(*n_ptr, n_max) : n_max;
    if (blockIdx.x * NB >= n) return;
    extern __shared__ __align__(16) float smem[];
    float *bufX = smem;
    float *bufY = smem + ROWS * F;
    float *vbuf = smem + 2 * ROWS * F;           // [NB][49] value-head conv outputs
    const int board0 = blockIdx.x * NB;
    for (int i = threadIdx.x; i < 2 * ROWS * F; i += THREADS) smem[i] = 0.f;
    __syncthreads();
    // stage the input planes into bufY (channels 0..3 of each real position)
    for (int i = threadIdx.x; i < NB * 49; i += THREADS) {
        const int b = board0 + i / 49, cell = i % 49;
        if (b >= n) continue;
        float4 v;
        if (IN_KIND == AZ_IN_F32) {
            v = reinterpret_cast<const float4 *>(input)[(size_t)b * 49 + cell];
        } else {
            az_position p = reinterpret_cast<const az_position *>(input)[b];
            p.turn &= 1;
            float f[4];
            az::feature_cell(p, cell / 7, cell % 7, f);
            v = make_float4(f[0], f[1], f[2], f[3]);
        }
        *reinterpret_cast<float4 *>(bufY + padded_row(i) * F) = v;
    }
    __syncthreads();
    conv3x3<false>(bufY, bufX, net.w_in, 4, net.bn_mean, net.bn_scale);
    for (int b = 0; b < net.blocks; ++b) {
        const float *w1 = net.w_tower + (size_t)(2 * b) * 9 * F * F;
        const float *w2 = w1 + (size_t)9 * F * F;
        conv3x3<false>(bufX, bufY, w1, F, net.bn_mean + (1 + 2 * b) * F, net.bn_scale + (1 + 2 * b) * F);
        conv3x3<true>(bufY, bufX, w2, F, net.bn_mean + (2 + 2 * b) * F, net.bn_scale + (2 + 2 * b) * F);
    }
    // heads: 17 policy planes + 1 value plane per real position
    for (int o = threadIdx.x; o < NB * 49 * 18; o += THREADS) {
        const int r = o / 18, plane = o % 18;
        const int b = board0 + r / 49;
        if (b >= n) continue;
        const float *a = bufX + padded_row(r) * F;
        float acc = 0.f;
        if (plane < 17) {
            for (int c = 0; c < F; ++c) acc = fmaf(a[c], __ldg(net.w_policy + c * 17 + plane), acc);
            logits[(size_t)b * AZ_LOGITS + (r % 49) * 17 + plane] = acc;
        } else {
            for (int c = 0; c < F; ++c) acc = fmaf(a[c], __ldg(net.w_value + c), acc);
            vbuf[r] = acc;
        }
    }
    __syncthreads();
    if (threadIdx.x < NB && board0 + threadIdx.x < n) {
        float acc = 0.f;
        for (int cell = 0; cell < 49; ++cell) acc = fmaf(vbuf[threadIdx.x * 49 + cell], __ldg(net.fc_w + cell), acc);
        values[board0 + threadIdx.x] = tanhf(acc + __ldg(net.fc_b));
    }
}

__global__ void k_i8_to_f32(const int8_t *in, float *out, size_t n)
{
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (float)in[i];
}

}  // namespace

extern "C" size_t az_net_param_count(int filters, int blocks)
{
    const size_t f = (size_t)filters;
    return 9 * 4 * f + (size_t)2 * blocks * 9 * f * f + f * 17 + f + 49 + 1 + (size_t)(1 + 2 * blocks) * 2 * f;
}

void az_net_release(az_context *ctx)
{
    AzNet *n = ctx->net;
    if (!n) return;
    az_net_tc_release(n);
    for (float *p : {n->packed, n->bn_mean, n->bn_scale})
        if (p) cudaFree(p);
    if (n->d_flag) cudaFree(n->d_flag);
    delete n;
    ctx->net = nullptr;
}

namespace {
// inference batch-norm constants: scale = 1/sqrt(var + eps) (computed in double), and a finiteness check of
// every parameter (a NaN/Inf weight is an argument error, not something to discover 25 layers later)
__global__ void k_prepare_bn(const float *__restrict__ packed, size_t count, const float *__restrict__ bn, int layers, int f,
                             float *__restrict__ mean, float *__restrict__ scale, int *__restrict__ flag)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count && !isfinite(packed[i])) atomicOr(flag, 1);
    if (i < (size_t)layers * f) {
        const int l = (int)(i / f), c = (int)(i % f);
        const float var = bn[(size_t)(2 * l + 1) * f + c];
        if (!(var + AZ_BN_EPS > 0.f)) atomicOr(flag, 2);
        mean[i] = bn[(size_t)(2 * l) * f + c];
        scale[i] = (float)(1.0 / sqrt((double)var + (double)AZ_BN_EPS));
    }
}
}  // namespace

extern "C" int az_net_load(az_context *ctx, const float *packed, size_t count, int filters, int blocks)
{
    AZ_REQUIRE(ctx && packed, AZ_ERR_ARG, "az_net_load: null argument");
    AZ_REQUIRE(filters == AZ_F, AZ_ERR_ARG, "az_net_load: this build supports filters=128 only (got %d)", filters);
    AZ_REQUIRE(blocks >= 1 && blocks <= 64, AZ_ERR_ARG, "az_net_load: blocks=%d out of range", blocks);
    AZ_REQUIRE(count == az_net_param_count(filters, blocks), AZ_ERR_ARG,
               "az_net_load: expected %zu floats for filters=%d blocks=%d, got %zu", az_net_param_count(filters, blocks),
               filters, blocks, count);
    AzNet *net = ctx->net;
    if (net && (net->filters != filters || net->blocks != blocks)) {
        AZ_CUDA(cudaStreamSynchronize(ctx->stream));
        az_net_release(ctx);
        net = nullptr;
    }
    const size_t f = (size_t)filters;
    if (!net) {                                  // first load of this shape: allocate once, reuse on every reload
        net = new AzNet();
        ctx->net = net;
        net->filters = filters;
        net->blocks = blocks;
        net->layers = 1 + 2 * blocks;
        AZ_CUDA(cudaMalloc(&net->packed, sizeof(float) * count));
        AZ_CUDA(cudaMalloc(&net->bn_mean, sizeof(float) * net->layers * f));
        AZ_CUDA(cudaMalloc(&net->bn_scale, sizeof(float) * net->layers * f));
        AZ_CUDA(cudaMalloc(&net->d_flag, sizeof(int)));
        float *p = net->packed;
        net->w_in = p;                      p += 9 * 4 * f;
        net->w_tower = p;                   p += (size_t)2 * blocks * 9 * f * f;
        net->w_policy = p;                  p += f * 17;
        net->w_value = p;                   p += f;
        net->fc_w = p;                      p += 49;
        net->fc_b = p;                      p += 1;
        net->bn_raw = p;
        int rc = az_net_tc_alloc(net);
        if (rc) return rc;
        AZ_CUDA(cudaFuncSetAttribute(k_net_fp32<AZ_IN_F32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_FP32));
        AZ_CUDA(cudaFuncSetAttribute(k_net_fp32<AZ_IN_POS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_FP32));
    }
    cudaStream_t s = ctx->stream;
    AZ_CUDA(cudaMemcpyAsync(net->packed, packed, sizeof(float) * count, cudaMemcpyHostToDevice, s));
    AZ_CUDA(cudaMemsetAsync(net->d_flag, 0, sizeof(int), s));
    k_prepare_bn<<<(unsigned)((count + 255) / 256), 256, 0, s>>>(net->packed, count, net->bn_raw, net->layers, filters, net->bn_mean,
                                                                 net->bn_scale, net->d_flag);
    int rc = az_net_tc_prepare(ctx, net);        // bf16 re-tiling with the BN scale folded in, on the device
    if (rc) return rc;
    ctx->launches += 4;
    int flag = 0;
    AZ_CUDA(cudaMemcpyAsync(&flag, net->d_flag, sizeof(int), cudaMemcpyDeviceToHost, s));
    AZ_CUDA(cudaStreamSynchronize(s));
    AZ_CUDA(cudaGetLastError());
    if (flag) {
        az_net_release(ctx);
        return az_fail(AZ_ERR_ARG, flag & 1 ? "az_net_load: non-finite weight" : "az_net_load: batch-norm variance + eps <= 0");
    }
    return AZ_OK;
}

static int net_forward_dev(az_context *ctx, const void *d_in, int in_kind, int n, int mode, void *d_logits, void *d_values,
                           const int *d_count = nullptr, cudaStream_t stream = nullptr, int tiles = 0, double *d_exps = nullptr,
                           double *d_totals = nullptr, const int *d_out_map = nullptr)
{
    if (!stream && ctx) stream = ctx->stream;
    AZ_REQUIRE(ctx && (n == 0 || (d_in && (d_logits || d_exps) && d_values)), AZ_ERR_ARG, "az_net_forward: null argument");
    AZ_REQUIRE(ctx->net, AZ_ERR_STATE, "az_net_forward: no weights loaded (call az_net_load first)");
    AZ_REQUIRE(n >= 0, AZ_ERR_ARG, "az_net_forward: n=%d", n);
    AZ_REQUIRE(mode == AZ_NET_FP32 || mode == AZ_NET_BF16 || mode == AZ_NET_F16, AZ_ERR_ARG, "az_net_forward: unknown mode %d", mode);
    if (n == 0) return AZ_OK;
    if (mode == AZ_NET_BF16 || mode == AZ_NET_F16)
        return az_net_tc_forward(ctx, ctx->net, d_in, in_kind, n, static_cast<float *>(d_logits), static_cast<float *>(d_values), d_count, stream, tiles,
                                 d_exps, d_totals, mode == AZ_NET_F16, d_out_map);
    AZ_REQUIRE(!d_exps && !d_out_map, AZ_ERR_ARG, "az_net_forward: softmax numerators are produced by the tensor-core kernel only");
    const int grid = (n + NB - 1) / NB;
    if (in_kind == AZ_IN_F32)
        k_net_fp32<AZ_IN_F32><<<grid, THREADS, SMEM_FP32, stream>>>(d_in, n, d_count, *ctx->net, static_cast<float *>(d_logits),
                                                                       static_cast<float *>(d_values));
    else
        k_net_fp32<AZ_IN_POS><<<grid, THREADS, SMEM_FP32, stream>>>(d_in, n, d_count, *ctx->net, static_cast<float *>(d_logits),
                                                                       static_cast<float *>(d_values));
    ctx->launches++;
    AZ_CUDA(cudaGetLastError());
    return AZ_OK;
}

int az_net_forward_internal(az_context *ctx, const void *d_in, int in_kind, int n, int mode, float *d_logits, float *d_values,
                            const int *d_count, cudaStream_t stream, int tiles, double *d_exps, double *d_totals, const int *d_out_map)
{
    return net_forward_dev(ctx, d_in, in_kind, n, mode, d_logits, d_values, d_count, stream, tiles, d_exps, d_totals, d_out_map);
}

extern "C" int az_net_forward_dev(az_context *ctx, const void *d_features, int n, int mode, void *d_logits, void *d_values)
{
    return net_forward_dev(ctx, d_features, AZ_IN_F32, n, mode, d_logits, d_values);
}

// Test hook (not part of the public header): a forward pass over min(*d_count, n) boards, the count read from device memory
// when the kernel starts -- the way the self-play pool launches the net behind the tree kernel.
extern "C" int az_net_forward_counted_dev(az_context *ctx, const void *d_features, int n, const int *d_count, int mode, void *d_logits, void *d_values)
{
    AZ_REQUIRE(d_count, AZ_ERR_ARG, "az_net_forward_counted_dev: no count");
    return net_forward_dev(ctx, d_features, AZ_IN_F32, n, mode, d_logits, d_values, d_count);
}

// Test hook (not part of the public header): the forward pass exactly as the self-play pool launches it (launch_net in
// az_pool.cu) -- az_position[] input, board count read from device memory when d_count is non-null, and for a speculative
// cache pool the softmax numerators, their sequential sums and the values scattered through d_out_map with d_logits null.
extern "C" int az_net_forward_pool_dev(az_context *ctx, const void *d_pos, int n, const int *d_count, int mode, int tiles, void *d_logits,
                                       void *d_values, double *d_exps, double *d_totals, const int *d_out_map)
{
    return net_forward_dev(ctx, d_pos, AZ_IN_POS, n, mode, d_logits, d_values, d_count, nullptr, tiles, d_exps, d_totals, d_out_map);
}

extern "C" int az_net_forward_pos_dev(az_context *ctx, const void *d_pos, int n, int mode, void *d_logits, void *d_values)
{
    return net_forward_dev(ctx, d_pos, AZ_IN_POS, n, mode, d_logits, d_values);
}

extern "C" int az_net_forward(az_context *ctx, const float *features, int n, int mode, float *logits, float *values)
{
    AZ_REQUIRE(ctx && n >= 0 && (n == 0 || (features && logits && values)), AZ_ERR_ARG, "az_net_forward: bad argument");
    if (n == 0) return AZ_OK;
    const size_t fb = sizeof(float) * AZ_FEATURES * (size_t)n, lb = sizeof(float) * AZ_LOGITS * (size_t)n;
    AZ_REQUIRE(ctx->scratch[0].reserve(fb) == 0 && ctx->scratch[1].reserve(lb) == 0 &&
                   ctx->scratch[2].reserve(sizeof(float) * (size_t)n) == 0,
               AZ_ERR_CUDA, "az_net_forward: device scratch alloc");
    AZ_CUDA(cudaMemcpyAsync(ctx->scratch[0].ptr, features, fb, cudaMemcpyHostToDevice, ctx->stream));
    int rc = net_forward_dev(ctx, ctx->scratch[0].ptr, AZ_IN_F32, n, mode, ctx->scratch[1].ptr, ctx->scratch[2].ptr);
    if (rc) return rc;
    AZ_CUDA(cudaMemcpyAsync(logits, ctx->scratch[1].ptr, lb, cudaMemcpyDeviceToHost, ctx->stream));
    AZ_CUDA(cudaMemcpyAsync(values, ctx->scratch[2].ptr, sizeof(float) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    AZ_CUDA(cudaStreamSynchronize(ctx->stream));
    AZ_CUDA(cudaGetLastError());
    return AZ_OK;
}

// ---------------------------------------------------------------------------------------------
// symmetry-ensembled evaluation (nn_evals.py:48-62): the 8 dihedral images of a position go through the net as one
// batch; the policies are rotated back SPATIALLY only (the reference does not permute the 16 direction planes,
// SURVEY App. B-9 -- kept) and averaged, the values are averaged.
// ---------------------------------------------------------------------------------------------
namespace {
// nn_evals.apply_symmetry (:7-15): out[i][j] = in[a'][b'] with (a, b) = sym&4 ? (j, i) : (i, j), b' = sym&2 ? 6-b : b, a' = sym&1 ? 6-a : a
__device__ __forceinline__ int sym_source_cell(int sym, int i, int j)
{
    int a = (sym & 4) ? j : i, b = (sym & 4) ? i : j;
    if (sym & 2) b = 6 - b;
    if (sym & 1) a = 6 - a;
    return a * 7 + b;
}
__constant__ int kInverseSymmetry[8] = {0, 1, 2, 3, 4, 6, 5, 7};      // nn_evals.py:27

__global__ void k_sym8_expand(const float4 *__restrict__ in, int n, float4 *__restrict__ out)
{
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;            // (board, sym, cell)
    if (idx >= n * 8 * 49) return;
    const int cell = idx % 49, sym = (idx / 49) & 7, b = idx / (49 * 8);
    out[idx] = in[b * 49 + sym_source_cell(sym, cell / 7, cell % 7)];
}

__global__ void k_sym8_reduce(const float *__restrict__ logits8, const float *__restrict__ values8, int n, float *__restrict__ logits,
                              float *__restrict__ values)
{
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;            // (board, cell, plane)
    if (idx < n * AZ_LOGITS) {
        const int b = idx / AZ_LOGITS, r = idx % AZ_LOGITS, cell = r / 17, plane = r % 17;
        float acc = 0.f;
        for (int sym = 0; sym < 8; ++sym) {                           // np.mean(axis=0): images added in order, then / 8
            const int src = sym_source_cell(kInverseSymmetry[sym], cell / 7, cell % 7);
            const float v = logits8[((size_t)(b * 8 + sym) * 49 + src) * 17 + plane];
            acc = sym ? acc + v : v;
        }
        logits[idx] = acc * 0.125f;
    }
    if (idx < n) {
        const float *v = values8 + (size_t)idx * 8;                   // np.mean of 8 floats: numpy's pairwise tree
        values[idx] = (((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]))) * 0.125f;
    }
}
}  // namespace

extern "C" int az_net_forward_sym8(az_context *ctx, const float *features, int n, int mode, float *logits, float *values)
{
    AZ_REQUIRE(ctx && n >= 0 && (n == 0 || (features && logits && values)), AZ_ERR_ARG, "az_net_forward_sym8: bad argument");
    AZ_REQUIRE(ctx->net, AZ_ERR_STATE, "az_net_forward_sym8: no weights loaded (call az_net_load first)");
    if (n == 0) return AZ_OK;
    const size_t nn = (size_t)n, fb = sizeof(float) * AZ_FEATURES * nn, lb = sizeof(float) * AZ_LOGITS * nn;
    AzBuffer *b = ctx->scratch;
    AZ_REQUIRE(b[0].reserve(fb) == 0 && b[1].reserve(8 * fb) == 0 && b[2].reserve(8 * lb) == 0 && b[3].reserve(8 * 4 * nn) == 0 &&
                   b[4].reserve(lb) == 0 && b[5].reserve(4 * nn) == 0,
               AZ_ERR_CUDA, "az_net_forward_sym8: device scratch alloc");
    cudaStream_t s = ctx->stream;
    AZ_CUDA(cudaMemcpyAsync(b[0].ptr, features, fb, cudaMemcpyHostToDevice, s));
    if (mode == AZ_NET_BF16 || mode == AZ_NET_F16) {
        // fused: the tensor-core kernel generates the 8 images while it stages its input and averages in its head epilogue
        int rc = az_net_tc_forward_sym8(ctx, ctx->net, b[0].ptr, AZ_IN_F32, n, b[4].as<float>(), b[5].as<float>(), mode == AZ_NET_F16);
        if (rc) return rc;
        AZ_CUDA(cudaMemcpyAsync(logits, b[4].ptr, lb, cudaMemcpyDeviceToHost, s));
        AZ_CUDA(cudaMemcpyAsync(values, b[5].ptr, 4 * nn, cudaMemcpyDeviceToHost, s));
        AZ_CUDA(cudaStreamSynchronize(s));
        AZ_CUDA(cudaGetLastError());
        return AZ_OK;
    }
    AZ_REQUIRE(mode == AZ_NET_FP32, AZ_ERR_ARG, "az_net_forward_sym8: unknown mode %d", mode);
    k_sym8_expand<<<(n * 8 * 49 + 255) / 256, 256, 0, s>>>(b[0].as<float4>(), n, b[1].as<float4>());
    int rc = net_forward_dev(ctx, b[1].ptr, AZ_IN_F32, 8 * n, mode, b[2].ptr, b[3].ptr);
    if (rc) return rc;
    k_sym8_reduce<<<(n * AZ_LOGITS + 255) / 256, 256, 0, s>>>(b[2].as<float>(), b[3].as<float>(), n, b[4].as<float>(), b[5].as<float>());
    ctx->launches += 2;
    AZ_CUDA(cudaMemcpyAsync(logits, b[4].ptr, lb, cudaMemcpyDeviceToHost, s));
    AZ_CUDA(cudaMemcpyAsync(values, b[5].ptr, 4 * nn, cudaMemcpyDeviceToHost, s));
    AZ_CUDA(cudaStreamSynchronize(s));
    AZ_CUDA(cudaGetLastError());
    return AZ_OK;
}

extern "C" int az_net_forward_i8(az_context *ctx, const int8_t *features, int n, int mode, float *logits, float *values)
{
    AZ_REQUIRE(ctx && n >= 0 && (n == 0 || (features && logits && values)), AZ_ERR_ARG, "az_net_forward_i8: bad argument");
    if (n == 0) return AZ_OK;
    const size_t cnt = (size_t)AZ_FEATURES * n;
    AZ_REQUIRE(ctx->scratch[3].reserve(cnt) == 0 && ctx->scratch[0].reserve(sizeof(float) * cnt) == 0 &&
                   ctx->scratch[1].reserve(sizeof(float) * AZ_LOGITS * (size_t)n) == 0 &&
                   ctx->scratch[2].reserve(sizeof(float) * (size_t)n) == 0,
               AZ_ERR_CUDA, "az_net_forward_i8: device scratch alloc");
    AZ_CUDA(cudaMemcpyAsync(ctx->scratch[3].ptr, features, cnt, cudaMemcpyHostToDevice, ctx->stream));
    k_i8_to_f32<<<(unsigned)((cnt + 255) / 256), 256, 0, ctx->stream>>>(ctx->scratch[3].as<int8_t>(), ctx->scratch[0].as<float>(), cnt);
    ctx->launches++;
    int rc = net_forward_dev(ctx, ctx->scratch[0].ptr, AZ_IN_F32, n, mode, ctx->scratch[1].ptr, ctx->scratch[2].ptr);
    if (rc) return rc;
    AZ_CUDA(cudaMemcpyAsync(logits, ctx->scratch[1].ptr, sizeof(float) * AZ_LOGITS * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    AZ_CUDA(cudaMemcpyAsync(values, ctx->scratch[2].ptr, sizeof(float) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    AZ_CUDA(cudaStreamSynchronize(ctx->stream));
    AZ_CUDA(cudaGetLastError());
    return AZ_OK;
}
