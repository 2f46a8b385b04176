// az_net.h -- device-resident network weights (internal).
#pragma once
#include "az_common.h"
#include <cuda_bf16.h>
#include <cuda_fp16.h>

constexpr int AZ_F = 128;            // filters (model.py:16)
constexpr float AZ_BN_EPS = 1e-3f;   // tf.layers.batch_normalization default epsilon

struct AzNet {
    int filters = 0, blocks = 0, layers = 0;   // layers = 1 + 2*blocks convolutions with batch-norm
    float *packed = nullptr;     // the caller's parameter vector, verbatim (everything below points into it)
    float *bn_raw = nullptr;     // [layers][2][F] moving mean / variance as stored in the .npy
    int *d_flag = nullptr;       // validation flag written by the prepare kernels
    // fp32 mode: weights in TF order [layer][tap = kh*3+kw][cin][cout]; layer 0 has cin = 4
    float *w_in = nullptr;       // [9][4][F]
    float *w_tower = nullptr;    // [2*blocks][9][F][F]
    float *bn_mean = nullptr;    // [layers][F]
    float *bn_scale = nullptr;   // [layers][F]   1/sqrt(var + eps)
    float *w_policy = nullptr;   // [F][17]
    float *w_value = nullptr;    // [F]
    float *fc_w = nullptr;       // [49]
    float *fc_b = nullptr;       // [1]
    // bf16 / f16 tensor-core modes (az_net_pair.cu): BN scale folded into the weights, UMMA operand layout
    uint8_t *pair_stream = nullptr;    // [input conv | tower | heads] in the order the TMA producer streams them, every stage
                                       // split into the two CTAs' output-channel halves
    uint8_t *pair_stream16 = nullptr;  // the same stream with IEEE-half operands (AZ_NET_F16)
    float *pair_shift = nullptr;       // [layers][F]   -mean * scale
    int pair_tiles = 0;                // tiles per CTA of the pair kernel: 1, 2, or 0 = 2 for batches of a full round, else 1
    long long *pair_prof = nullptr;    // issuer wait records of k_net_pair (az_net_pair_profile; profiling only)
    int pair_prof_max = 0;
};

// az_net.cu: forward over up to `n` boards; when d_count != nullptr the actual count is read on the device.  `stream` =
// nullptr: the context stream.  d_exps / d_totals (bf16 / f16 only): instead of logits, exp((double)logit) [n][833] and their
// sequential sum [n], with the values, through d_out_map when it is non-null
int az_net_forward_internal(az_context *ctx, const void *d_in, int in_kind, int n, int mode, float *d_logits, float *d_values,
                            const int *d_count, cudaStream_t stream = nullptr, double *d_exps = nullptr, double *d_totals = nullptr,
                            const int *d_out_map = nullptr);

// az_net_pair.cu
int az_net_pair_alloc(AzNet *net);
int az_net_pair_prepare(az_context *ctx, AzNet *net);
void az_net_pair_release(AzNet *net);
int az_net_pair_boards_per_round(az_context *ctx);   // boards one wave of one-tile CTA pairs evaluates: 4 per SM
int az_net_pair_forward(az_context *ctx, AzNet *net, const void *d_in, int in_kind, int n, float *d_logits, float *d_values, const int *d_count,
                        cudaStream_t stream, int f16, double *d_exps = nullptr, double *d_totals = nullptr, const int *d_out_map = nullptr,
                        int tiles = 0);       // tiles: 1 or 2 forces the plain pass's tiles per CTA, 0 = AZ_NET_PAIR_TILES or by batch size
// mean over the 8 dihedral images of each of the n positions, one launch (nn_evals.py:48-62)
int az_net_pair_forward_sym8(az_context *ctx, AzNet *net, const float *d_features, int n, float *d_logits, float *d_values, int f16);
int az_net_pair_tower(az_context *ctx, AzNet *net, const float *d_features, int n, int conv_layers, float *d_act);

enum { AZ_IN_F32 = 0, AZ_IN_POS = 1 };
