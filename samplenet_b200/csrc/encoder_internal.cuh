// encoder_internal.cuh -- declarations shared by encoder.cu (CUDA-core path), encoder_tc.cu (tcgen05 path), conv_stack.cu and generator.cu.
#pragma once
#include "common.cuh"

namespace snb {

struct TcLayerParams {
    // FIRST mode (x != nullptr): the A operand is layer 1 (3 -> c_in, weights w1/b1) evaluated on the fly from the cloud,
    // its BatchNorm statistics having been derived analytically from the input moments (x_moments_kernel).
    const float *x;             // cloud (b, n, 3) BNC or (b, 3, n) BCN, or nullptr
    int x_layout;
    const float *w1, *b1;       // (c_in, 3), (c_in)
    const float *in;            // previous layer's raw output (b*n, c_in) row-major (x == nullptr)
    int c_in, c_out;
    int b, n, tiles_per_cloud;
    const double *in_stats;
    const float *in_gamma, *in_beta, *in_run_mean, *in_run_var;
    float in_eps;
    int in_relu, in_has_bn, in_training;
    const float *weight, *bias;
    float *out;                 // raw output or nullptr (last layer)
    double *out_stats;          // or nullptr
    float *tile_max, *tile_min; // or nullptr
    // debug / bring-up knobs (see snb200_debug_tc_gemm): descriptor high word template and K-advance in 16-byte units
    unsigned desc_hi;
    int k_adv16;
    int swizzle;                // 1 = XOR-128B data placement, 0 = plain rows
};

int launch_tc_layer(const TcLayerParams &P, cudaStream_t stream);
bool tc_layer_supported(int c_in, int c_out);
int tc_tiles_per_cloud(int n);
int launch_x_moments(int b, int n, int layout, const float *x, double *mom, unsigned *counter, const float *w1, const float *b1, int c1,
                     double *stats0, cudaStream_t stream);
// CUDA-core conv stack: writes per-tile extrema of the last layer and (training) per-layer statistics
int launch_simt_conv_stack(int b, int n, int layout, const float *x, int num_layers, const snb200_layer *layers, int training, float *act0,
                           float *act1, double *const *stats, float *tile_max, float *tile_min, int *tiles_per_cloud_out, cudaStream_t stream);

// pool + FC head description (generator.cu builds it; the cluster kernel and the fused tail of the conv-stack kernel consume it)
struct HeadLayer {
    int c_in, c_out;
    const float *weight, *bias, *gamma, *beta;
    float *run_mean, *run_var;
    float eps, momentum;
    int has_bn, relu;
};

struct HeadParams {
    int b, training;
    // pooling of the last conv layer
    int c_feat, tiles_per_cloud;
    const float *tile_max, *tile_min;
    const double *last_stats;
    int stat_rep;                // 0: (sum, sumsq) of every conv layer are the plain [2][C] block; 1: the accumulators the conv-stack kernel adds into
                                 // are spread one per 128-byte line behind that block: accumulator idx at stats[2C + idx * kStatStride]
    const float *last_gamma, *last_beta, *last_run_mean, *last_run_var;
    float last_eps;
    int last_has_bn, last_relu;
    double count;
    float *feat;                 // (b, c_feat) global: pooled feature (also an API output)
    // running-statistics updates of the conv layers
    int ru_num;
    const double *ru_stats[SNB200_MAX_CONV_LAYERS];
    int ru_rep[SNB200_MAX_CONV_LAYERS];   // replicas behind each of them (see stat_rep)
    float *ru_mean[SNB200_MAX_CONV_LAYERS];
    float *ru_var[SNB200_MAX_CONV_LAYERS];
    float ru_momentum[SNB200_MAX_CONV_LAYERS];
    int ru_c[SNB200_MAX_CONV_LAYERS];
    // FC layers
    int num_fc;
    HeadLayer fc[SNB200_MAX_FC_LAYERS];
    float *act[2];               // (b, max width) scratch
    float *out;                  // (b, c_out_last)
    int out_inner;
    // torch BatchNorm bookkeeping: int64 counters incremented once per training forward
    int num_counters;
    long long *counters[SNB200_MAX_CONV_LAYERS + SNB200_MAX_FC_LAYERS];
    int dbg;                     // bring-up switches (always 0 in the product): 1 = stop after pooling, 2 = no TMA weight prefetch
    float *ll[SNB200_MAX_FC_LAYERS + 1];   // fused head: self-validating exchange buffers, zero at launch: [0] pooled feature (b, c_feat),
                                           // [l+1] output of FC layer l (b, c_out); a word of 0 means "not stored yet"
};

// persistent cooperative conv-stack kernel (conv_stack.cu); head != nullptr fuses the pool + FC head into the same launch
bool conv_stack_supported(int b, int n, int nconv, const snb200_layer *conv);
int conv_stack_slots_per_cloud(int b, int n);   // pool partials per cloud written by the conv-stack kernel (its `tiles_per_cloud`)
int launch_conv_stack(int b, int n, int layout, const float *x, int nconv, const snb200_layer *conv, int training, double *const *stats,
                      double *mom, unsigned *barrier, float *tile_max, float *tile_min, int *tiles_per_cloud_out, const HeadParams *head,
                      char *clean_ptr, size_t clean_bytes, cudaStream_t stream, float *const *zsave = nullptr, float *const *act = nullptr);

#ifdef __CUDACC__
// scale/shift of a BatchNorm given either batch statistics or running statistics
__device__ __forceinline__ void bn_scale_shift(const double *stats, int c_total, int c, double count, const float *gamma, const float *beta,
                                               const float *run_mean, const float *run_var, float eps, int training, float &scale, float &shift)
{
    float mean, var;
    if (training) {
        const double m = stats[c] / count;
        double v = stats[c_total + c] / count - m * m;
        if (v < 0) v = 0;
        mean = (float)m;
        var = (float)v;
    } else {
        mean = run_mean[c];
        var = run_var[c];
    }
    const float invstd = 1.0f / sqrtf(var + eps);
    scale = gamma[c] * invstd;
    shift = beta[c] - mean * scale;
}
#endif  // __CUDACC__

}  // namespace snb
