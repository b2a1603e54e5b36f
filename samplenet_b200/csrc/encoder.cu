// encoder.cu -- SampleNet generator: per-point MLP (1x1 conv + BatchNorm + ReLU stack), global max-pool, FC head.
//
// Reference behaviour restated (not ported): registration/src/samplenet.py:90-104 runs, per layer, a cuDNN/cuBLAS conv,
// a BatchNorm kernel and a ReLU kernel, each round-tripping the (B,C,N) activation tensor; then torch.max and four
// Linear+BN+ReLU triples.  reconstruction/src/samplers.py:22-36 and classification/models/samplenet_model.py:31-108 are the
// same stack with other widths / BN epsilon.
//
// This file is the exact-fp32 CUDA-core path (every product and sum in fp32, like the reference's CPU path):
//   * one launch per conv layer.  The layer kernel applies the PREVIOUS layer's BatchNorm + ReLU while it loads its input
//     tile (so normalised activations never exist in memory), multiplies by the weight tile out of shared memory with an
//     8x8 register tile per thread, adds the bias, writes the raw (pre-BN) output once, and accumulates the per-channel
//     sum / sum-of-squares that training-mode BatchNorm needs (fp32 inside the tile, fp64 atomics across tiles);
//   * the last conv layer never writes its activation: it only emits per-tile max / min of the raw output, from which
//     max_n relu(bn(y)) follows exactly because the BN affine map is monotone per channel;
//   * a pool-finalise kernel turns statistics into the pooled feature; the FC head keeps each output channel inside one
//     warp so that BatchNorm over the batch needs no cross-CTA traffic.
// The tcgen05 tensor-core variant of the conv stack lives in encoder_tc.cu.
#include "encoder_internal.cuh"

namespace snb {

constexpr int kEncThreads = 256;
constexpr int kEncKC = 32;  // K chunk staged in shared memory per step

struct ConvLayerParams {
    // input: either the cloud itself (first layer) or the previous layer's raw output (points-major, `c_in` wide)
    const float *in;
    long long in_cloud_stride;  // floats between consecutive clouds
    int in_stride_p, in_stride_c;
    int c_in, c_out;
    int b, n, tiles_per_cloud;
    // BatchNorm + ReLU of the PREVIOUS layer, applied on load (nullptrs => identity)
    const double *in_stats;        // [2][c_in] sum, sumsq over b*n positions (training) or nullptr
    const float *in_gamma, *in_beta, *in_run_mean, *in_run_var;
    float in_eps;
    int in_relu, in_has_bn, in_training;
    // this layer
    const float *weight, *bias;    // (c_out, c_in), (c_out)
    float *out;                    // raw output (b*n, c_out) or nullptr for the last layer
    double *out_stats;             // [2][c_out] or nullptr (no BN after this layer / eval mode)
    float *tile_max, *tile_min;    // (b*tiles_per_cloud, c_out) or nullptr
};

// CC = output channels per CTA (64 or 128); thread tile 8 points x 8 channels; TP = points per CTA.
template <int CC>
__global__ void __launch_bounds__(kEncThreads) conv_layer_kernel(const __grid_constant__ ConvLayerParams P)
{
    constexpr int TXN = CC / 8;             // threads along channels
    constexpr int TYN = kEncThreads / TXN;  // threads along points
    constexpr int TP = TYN * 8;             // points per CTA: 256 (CC=64) or 128 (CC=128)
    extern __shared__ __align__(16) float smem[];
    float *sA = smem;                        // [kEncKC][TP]
    float *sW = sA + kEncKC * TP;            // [kEncKC][CC]
    float *sScale = sW + kEncKC * CC;        // [c_in]
    float *sShift = sScale + P.c_in;         // [c_in]
    float *sRed = sShift + P.c_in;           // [TYN][CC] (epilogue reductions)

    const int tid = threadIdx.x;
    const int tx = tid % TXN, ty = tid / TXN;
    const int tile = blockIdx.x;
    const int cloud = tile / P.tiles_per_cloud;
    const int p0 = (tile % P.tiles_per_cloud) * TP;
    const int np = min(TP, P.n - p0);
    const int c0 = blockIdx.y * CC;
    const int c_in = P.c_in;

    // ---- prologue: BatchNorm(+ReLU) of the previous layer as a per-channel affine map
    for (int c = tid; c < c_in; c += kEncThreads) {
        float sc = 1.f, sh = 0.f;
        if (P.in_has_bn)
            bn_scale_shift(P.in_stats, c_in, c, (double)P.b * (double)P.n, P.in_gamma, P.in_beta, P.in_run_mean, P.in_run_var, P.in_eps,
                           P.in_training, sc, sh);
        sScale[c] = sc;
        sShift[c] = sh;
    }
    __syncthreads();

    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; i++)
#pragma unroll
        for (int j = 0; j < 8; j++) acc[i][j] = 0.f;

    const float *in_cloud = P.in + (size_t)cloud * P.in_cloud_stride;
    for (int k0 = 0; k0 < c_in; k0 += kEncKC) {
        const int kn = min(kEncKC, c_in - k0);
        // A tile: sA[k][p] = relu(bn(in[p][k0+k])), zero for p >= np.  lane -> point (conflict-free stores).
        for (int e = tid; e < kEncKC * TP; e += kEncThreads) {
            const int p = e % TP, k = e / TP;
            float v = 0.f;
            if (p < np && k < kn) {
                v = __ldg(in_cloud + (size_t)(p0 + p) * P.in_stride_p + (size_t)(k0 + k) * P.in_stride_c);
                v = fmaf(v, sScale[k0 + k], sShift[k0 + k]);
                if (P.in_relu) v = fmaxf(v, 0.f);
            }
            sA[k * TP + p] = v;
        }
        // W tile: sW[k][c] = W[c0+c][k0+k] (row-major (c_out, c_in)).  Lanes run along c so the transposed store is
        // bank-conflict free; the strided global reads stay in L1/L2 (the whole weight matrix is <= 128 KB).
        for (int e = tid; e < kEncKC * CC; e += kEncThreads) {
            const int c = e % CC, k = e / CC;
            float v = 0.f;
            if (k < kn && c0 + c < P.c_out) v = __ldg(P.weight + (size_t)(c0 + c) * c_in + k0 + k);
            sW[k * CC + c] = v;
        }
        __syncthreads();
#pragma unroll 4
        for (int k = 0; k < kn; k++) {
            const float4 a0 = *reinterpret_cast<const float4 *>(sA + k * TP + ty * 8);
            const float4 a1 = *reinterpret_cast<const float4 *>(sA + k * TP + ty * 8 + 4);
            const float4 w0 = *reinterpret_cast<const float4 *>(sW + k * CC + tx * 8);
            const float4 w1 = *reinterpret_cast<const float4 *>(sW + k * CC + tx * 8 + 4);
            const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float w[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
            for (int i = 0; i < 8; i++)
#pragma unroll
                for (int j = 0; j < 8; j++) acc[i][j] = fmaf(a[i], w[j], acc[i][j]);
        }
        __syncthreads();
    }

    // ---- epilogue: bias, raw store, statistics, per-tile extrema
    float bias[8];
#pragma unroll
    for (int j = 0; j < 8; j++) {
        const int c = c0 + tx * 8 + j;
        bias[j] = (c < P.c_out) ? __ldg(P.bias + c) : 0.f;
    }
    float s[8], ss[8], mx[8], mn[8];
#pragma unroll
    for (int j = 0; j < 8; j++) { s[j] = 0.f; ss[j] = 0.f; mx[j] = -INFINITY; mn[j] = INFINITY; }
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const int p = ty * 8 + i;
        const bool pv = p < np;
#pragma unroll
        for (int j = 0; j < 8; j++) {
            const float v = acc[i][j] + bias[j];
            acc[i][j] = v;
            if (pv) { s[j] += v; ss[j] = fmaf(v, v, ss[j]); mx[j] = fmaxf(mx[j], v); mn[j] = fminf(mn[j], v); }
        }
        if (P.out && pv) {
            float *o = P.out + ((size_t)cloud * P.n + p0 + p) * P.c_out + c0 + tx * 8;
            if (c0 + tx * 8 + 8 <= P.c_out && (P.c_out & 3) == 0) {
                *reinterpret_cast<float4 *>(o) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
                *reinterpret_cast<float4 *>(o + 4) = make_float4(acc[i][4], acc[i][5], acc[i][6], acc[i][7]);
            } else {
#pragma unroll
                for (int j = 0; j < 8; j++)
                    if (c0 + tx * 8 + j < P.c_out) o[j] = acc[i][j];
            }
        }
    }
    // cross-thread reductions over the TYN point groups, fixed order
    if (P.out_stats) {
#pragma unroll
        for (int j = 0; j < 8; j++) sRed[ty * CC + tx * 8 + j] = s[j];
        __syncthreads();
        if (tid < CC && c0 + tid < P.c_out) {
            float t = 0.f;
            for (int r = 0; r < TYN; r++) t += sRed[r * CC + tid];
            atomicAdd(P.out_stats + c0 + tid, (double)t);
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 8; j++) sRed[ty * CC + tx * 8 + j] = ss[j];
        __syncthreads();
        if (tid < CC && c0 + tid < P.c_out) {
            float t = 0.f;
            for (int r = 0; r < TYN; r++) t += sRed[r * CC + tid];
            atomicAdd(P.out_stats + P.c_out + c0 + tid, (double)t);
        }
        __syncthreads();
    }
    if (P.tile_max) {
#pragma unroll
        for (int j = 0; j < 8; j++) sRed[ty * CC + tx * 8 + j] = mx[j];
        __syncthreads();
        if (tid < CC && c0 + tid < P.c_out) {
            float t = -INFINITY;
            for (int r = 0; r < TYN; r++) t = fmaxf(t, sRed[r * CC + tid]);
            P.tile_max[(size_t)tile * P.c_out + c0 + tid] = t;
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 8; j++) sRed[ty * CC + tx * 8 + j] = mn[j];
        __syncthreads();
        if (tid < CC && c0 + tid < P.c_out) {
            float t = INFINITY;
            for (int r = 0; r < TYN; r++) t = fminf(t, sRed[r * CC + tid]);
            P.tile_min[(size_t)tile * P.c_out + c0 + tid] = t;
        }
    }
}

// ---- running-statistics update (PyTorch semantics: momentum mix with the UNBIASED batch variance)
__device__ __forceinline__ void update_running(const double *stats, int c_total, int c, double count, float momentum, float *run_mean,
                                               float *run_var)
{
    const double m = stats[c] / count;
    double v = stats[c_total + c] / count - m * m;
    if (v < 0) v = 0;
    const double unb = count > 1 ? v * count / (count - 1) : v;
    if (run_mean) run_mean[c] = (1.f - momentum) * run_mean[c] + momentum * (float)m;
    if (run_var) run_var[c] = (1.f - momentum) * run_var[c] + momentum * (float)unb;
}

struct RunUpdateParams {
    int num;
    const double *stats[SNB200_MAX_CONV_LAYERS];
    float *run_mean[SNB200_MAX_CONV_LAYERS];
    float *run_var[SNB200_MAX_CONV_LAYERS];
    float momentum[SNB200_MAX_CONV_LAYERS];
    int c[SNB200_MAX_CONV_LAYERS];
    double count;
    int num_counters;
    long long *counters[SNB200_MAX_CONV_LAYERS];
};

struct PoolParams {
    int b, c, tiles_per_cloud;
    const float *tile_max, *tile_min;
    const double *stats;
    const float *gamma, *beta, *run_mean, *run_var;
    float eps;
    int has_bn, relu, training;
    double count;
    float *feat;  // (b, c)
    RunUpdateParams ru;
};

// feat[b][c] = max_n act(bn(y[b][n][c])) from per-tile extrema; block (0) also applies all running-stat updates once.
__global__ void __launch_bounds__(256) pool_finalize_kernel(const __grid_constant__ PoolParams P)
{
    const int e = blockIdx.x * 256 + threadIdx.x;
    if (e < P.b * P.c) {
        const int bi = e / P.c, c = e % P.c;
        float mx = -INFINITY, mn = INFINITY;
        for (int t = 0; t < P.tiles_per_cloud; t++) {
            mx = fmaxf(mx, P.tile_max[((size_t)bi * P.tiles_per_cloud + t) * P.c + c]);
            mn = fminf(mn, P.tile_min[((size_t)bi * P.tiles_per_cloud + t) * P.c + c]);
        }
        float v = mx;
        if (P.has_bn) {
            float sc, sh;
            bn_scale_shift(P.stats, P.c, c, P.count, P.gamma, P.beta, P.run_mean, P.run_var, P.eps, P.training, sc, sh);
            v = sc >= 0.f ? fmaf(mx, sc, sh) : fmaf(mn, sc, sh);
        }
        if (P.relu) v = fmaxf(v, 0.f);
        P.feat[e] = v;
    }
    if (blockIdx.x == gridDim.x - 1) {
        if ((int)threadIdx.x < P.ru.num_counters) *P.ru.counters[threadIdx.x] += 1;
        // the last block applies the running-stat updates after every read of run_mean/run_var that other blocks
        // of THIS kernel could make is irrelevant: in training mode bn_scale_shift never reads the running buffers.
        for (int l = 0; l < P.ru.num; l++)
            for (int c = threadIdx.x; c < P.ru.c[l]; c += 256)
                update_running(P.ru.stats[l], P.ru.c[l], c, P.ru.count, P.ru.momentum[l], P.ru.run_mean[l], P.ru.run_var[l]);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// FC head: one warp per output channel, all batch rows; BatchNorm over the batch stays inside the warp.
// in (b, c_in) row-major, weight (c_out, c_in), out (b, c_out).  b <= 256.
// ------------------------------------------------------------------------------------------------------------------
constexpr int kFcWarps = 8;
constexpr int kFcMaxRowsPerLane = 8;  // b <= 256
constexpr int kFcRowChunk = 32;       // batch rows staged in shared memory per step

struct FcParams {
    int b, c_in, c_out;
    const float *in, *weight, *bias, *gamma, *beta;
    float *run_mean, *run_var;
    float eps, momentum;
    int has_bn, relu, training;
    int out_inner;  // > 0: store row (c_out/out_inner, out_inner) transposed
    float *out;
    long long *counter;  // BatchNorm num_batches_tracked of this layer (training) or nullptr
};

__global__ void __launch_bounds__(kFcWarps * 32) fc_layer_kernel(const __grid_constant__ FcParams P)
{
    extern __shared__ __align__(16) float s_in[];  // (kFcRowChunk, c_in)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int co = blockIdx.x * kFcWarps + warp;
    const bool active = co < P.c_out;  // warp-uniform
    if (blockIdx.x == 0 && threadIdx.x == 0 && P.counter) *P.counter += 1;
    const float *w = P.weight + (size_t)(active ? co : 0) * P.c_in;
    float y[kFcMaxRowsPerLane];  // lane holds rows lane, lane+32, ...
#pragma unroll
    for (int r = 0; r < kFcMaxRowsPerLane; r++) y[r] = 0.f;
    const float bias = (P.bias && active) ? P.bias[co] : 0.f;
    for (int r0 = 0; r0 < P.b; r0 += kFcRowChunk) {
        const int rn = min(kFcRowChunk, P.b - r0);
        __syncthreads();
        for (int i = threadIdx.x; i < rn * P.c_in; i += kFcWarps * 32) s_in[i] = P.in[(size_t)r0 * P.c_in + i];
        __syncthreads();
        if (!active) continue;
        for (int rr = 0; rr < rn; rr++) {
            const int row = r0 + rr;
            float part = 0.f;
            for (int k = lane; k < P.c_in; k += 32) part = fmaf(s_in[rr * P.c_in + k], __ldg(w + k), part);
            part = warp_sum(part) + bias;
#pragma unroll
            for (int r = 0; r < kFcMaxRowsPerLane; r++)
                if ((row >> 5) == r && (row & 31) == lane) y[r] = part;
        }
    }
    if (!active) return;
    float scale = 1.f, shift = 0.f;
    if (P.has_bn) {
        float mean, var;
        if (P.training) {
            float s = 0.f;
#pragma unroll
            for (int r = 0; r < kFcMaxRowsPerLane; r++)
                if (r * 32 + lane < P.b) s += y[r];
            mean = warp_sum(s) / (float)P.b;
            float q = 0.f;
#pragma unroll
            for (int r = 0; r < kFcMaxRowsPerLane; r++)
                if (r * 32 + lane < P.b) { const float d = y[r] - mean; q = fmaf(d, d, q); }
            q = warp_sum(q);
            var = q / (float)P.b;
            if (lane == 0) {
                const float unb = P.b > 1 ? q / (float)(P.b - 1) : var;
                if (P.run_mean) P.run_mean[co] = (1.f - P.momentum) * P.run_mean[co] + P.momentum * mean;
                if (P.run_var) P.run_var[co] = (1.f - P.momentum) * P.run_var[co] + P.momentum * unb;
            }
        } else {
            mean = P.run_mean[co];
            var = P.run_var[co];
        }
        const float invstd = 1.0f / sqrtf(var + P.eps);
        scale = P.gamma[co] * invstd;
        shift = P.beta[co] - mean * scale;
    }
#pragma unroll
    for (int r = 0; r < kFcMaxRowsPerLane; r++) {
        const int row = r * 32 + lane;
        if (row < P.b) {
            float v = P.has_bn ? fmaf(y[r], scale, shift) : y[r];
            if (P.relu) v = fmaxf(v, 0.f);
            const int oc = P.out_inner > 0 ? (co % P.out_inner) * (P.c_out / P.out_inner) + co / P.out_inner : co;
            P.out[(size_t)row * P.c_out + oc] = v;
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------------------
static int enc_tp(int c_out) { return c_out > 64 ? 128 : 256; }

struct EncWorkspace {
    float *act[2];
    double *stats[SNB200_MAX_CONV_LAYERS];
    float *tile_max, *tile_min;
    size_t stats_bytes;
    char *stats_base;
    size_t total;
};

static EncWorkspace carve_encoder_ws(void *base, int b, int n, int num_layers, const snb200_layer *layers)
{
    EncWorkspace W;
    char *p = reinterpret_cast<char *>(base);
    size_t off = 0;
    int maxc = 0;
    for (int l = 0; l + 1 < num_layers; l++) maxc = max(maxc, layers[l].c_out);
    const size_t act_bytes = align_up((size_t)b * n * maxc * sizeof(float), 256);
    W.act[0] = reinterpret_cast<float *>(p + off); off += act_bytes;
    W.act[1] = reinterpret_cast<float *>(p + off); off += act_bytes;
    W.stats_base = p + off;
    size_t sb = 0;
    for (int l = 0; l < num_layers; l++) {
        W.stats[l] = reinterpret_cast<double *>(p + off + sb);
        sb += align_up((size_t)2 * layers[l].c_out * sizeof(double), 256);
    }
    W.stats_bytes = sb;
    off += sb;
    const int c_last = layers[num_layers - 1].c_out;
    const int tpc = (n + enc_tp(c_last) - 1) / enc_tp(c_last);
    const size_t tb = align_up((size_t)b * tpc * c_last * sizeof(float), 256);
    W.tile_max = reinterpret_cast<float *>(p + off); off += tb;
    W.tile_min = reinterpret_cast<float *>(p + off); off += tb;
    W.total = off;
    return W;
}

size_t encoder_workspace_bytes(int b, int n, int num_layers, const snb200_layer *layers)
{
    return carve_encoder_ws(nullptr, b, n, num_layers, layers).total;
}

int launch_simt_conv_stack(int b, int n, int layout, const float *x, int num_layers, const snb200_layer *layers, int training, float *act0,
                           float *act1, double *const *stats, float *tile_max, float *tile_min, int *tiles_per_cloud_out, cudaStream_t stream)
{
    float *act[2] = {act0, act1};
    for (int l = 0; l < num_layers; l++) {
        const snb200_layer &L = layers[l];
        ConvLayerParams P;
        memset(&P, 0, sizeof(P));
        P.b = b; P.n = n; P.c_in = L.c_in; P.c_out = L.c_out;
        if (l == 0) {
            P.in = x;
            P.in_cloud_stride = (long long)n * 3;
            P.in_stride_p = layout == SNB200_BNC ? 3 : 1;
            P.in_stride_c = layout == SNB200_BNC ? 1 : n;
            P.in_has_bn = 0; P.in_relu = 0;
        } else {
            const snb200_layer &Lp = layers[l - 1];
            P.in = act[(l - 1) & 1];
            P.in_cloud_stride = (long long)n * Lp.c_out;
            P.in_stride_p = Lp.c_out; P.in_stride_c = 1;
            P.in_has_bn = Lp.bn_weight != nullptr;
            P.in_stats = stats[l - 1];
            P.in_gamma = Lp.bn_weight; P.in_beta = Lp.bn_bias; P.in_run_mean = Lp.bn_running_mean; P.in_run_var = Lp.bn_running_var;
            P.in_eps = Lp.bn_eps; P.in_relu = Lp.relu; P.in_training = training;
        }
        P.weight = L.weight; P.bias = L.bias;
        const bool last = (l == num_layers - 1);
        P.out = last ? nullptr : act[l & 1];
        P.out_stats = (training && L.bn_weight) ? stats[l] : nullptr;
        P.tile_max = last ? tile_max : nullptr;
        P.tile_min = last ? tile_min : nullptr;
        const int CC = L.c_out > 64 ? 128 : 64;
        const int TP = enc_tp(L.c_out);
        P.tiles_per_cloud = (n + TP - 1) / TP;
        if (last && tiles_per_cloud_out) *tiles_per_cloud_out = P.tiles_per_cloud;
        dim3 grid(b * P.tiles_per_cloud, (L.c_out + CC - 1) / CC);
        const int TYN = kEncThreads / (CC / 8);
        const size_t smem = ((size_t)kEncKC * TP + (size_t)kEncKC * CC + 2 * (size_t)L.c_in + (size_t)TYN * CC) * sizeof(float);
        static PerDeviceOnce attr_once;
        if (attr_once.first()) {
            cudaFuncSetAttribute(conv_layer_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
            cudaFuncSetAttribute(conv_layer_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
        }
        if (smem > 100 * 1024) { set_error("encoder: layer %d too wide for the shared-memory tile (c_in=%d)", l, L.c_in); return SNB200_EUNSUPPORTED; }
        if (CC == 64) conv_layer_kernel<64><<<grid, kEncThreads, smem, stream>>>(P);
        else conv_layer_kernel<128><<<grid, kEncThreads, smem, stream>>>(P);
        int rc = check_launch("encoder conv layer");
        if (rc) return rc;
    }
    return SNB200_OK;
}

int launch_encoder_forward(int b, int n, int layout, const float *x, int num_layers, const snb200_layer *layers, int training, float *feat,
                           void *workspace, cudaStream_t stream)
{
    EncWorkspace W = carve_encoder_ws(workspace, b, n, num_layers, layers);
    if (training) cudaMemsetAsync(W.stats_base, 0, W.stats_bytes, stream);
    int tpc_last = 0;
    int rc0 = launch_simt_conv_stack(b, n, layout, x, num_layers, layers, training, W.act[0], W.act[1], W.stats, W.tile_max, W.tile_min, &tpc_last, stream);
    if (rc0) return rc0;
    const snb200_layer &LL = layers[num_layers - 1];
    PoolParams Q;
    memset(&Q, 0, sizeof(Q));
    Q.b = b; Q.c = LL.c_out;
    Q.tiles_per_cloud = (n + enc_tp(LL.c_out) - 1) / enc_tp(LL.c_out);
    Q.tile_max = W.tile_max; Q.tile_min = W.tile_min; Q.stats = W.stats[num_layers - 1];
    Q.gamma = LL.bn_weight; Q.beta = LL.bn_bias; Q.run_mean = LL.bn_running_mean; Q.run_var = LL.bn_running_var;
    Q.eps = LL.bn_eps; Q.has_bn = LL.bn_weight != nullptr; Q.relu = LL.relu; Q.training = training;
    Q.count = (double)b * (double)n;
    Q.feat = feat;
    Q.ru.num = 0;
    Q.ru.count = Q.count;
    if (training) {
        for (int l = 0; l < num_layers; l++) {
            if (!layers[l].bn_weight || (!layers[l].bn_running_mean && !layers[l].bn_running_var)) continue;
            const int i = Q.ru.num++;
            Q.ru.stats[i] = W.stats[l]; Q.ru.run_mean[i] = layers[l].bn_running_mean; Q.ru.run_var[i] = layers[l].bn_running_var;
            Q.ru.momentum[i] = layers[l].bn_momentum; Q.ru.c[i] = layers[l].c_out;
        }
        for (int l = 0; l < num_layers; l++)
            if (layers[l].bn_weight && layers[l].bn_num_batches_tracked) Q.ru.counters[Q.ru.num_counters++] = layers[l].bn_num_batches_tracked;
    }
    pool_finalize_kernel<<<(b * LL.c_out + 255) / 256, 256, 0, stream>>>(Q);
    return check_launch("encoder pool finalize");
}

size_t fc_head_workspace_bytes(int b, int num_layers, const snb200_layer *layers)
{
    int maxc = 0;
    for (int l = 0; l + 1 < num_layers; l++) maxc = max(maxc, layers[l].c_out);
    return 2 * align_up((size_t)b * max(maxc, 1) * sizeof(float), 256);
}

int launch_fc_head_forward(int b, const float *in, int num_layers, const snb200_layer *layers, int training, float *out, int out_transpose_inner,
                           void *workspace, cudaStream_t stream)
{
    int maxc = 0;
    for (int l = 0; l + 1 < num_layers; l++) maxc = max(maxc, layers[l].c_out);
    float *buf[2];
    buf[0] = reinterpret_cast<float *>(workspace);
    buf[1] = reinterpret_cast<float *>(reinterpret_cast<char *>(workspace) + align_up((size_t)b * max(maxc, 1) * sizeof(float), 256));
    const float *cur = in;
    for (int l = 0; l < num_layers; l++) {
        const snb200_layer &L = layers[l];
        FcParams P;
        P.b = b; P.c_in = L.c_in; P.c_out = L.c_out;
        P.in = cur; P.weight = L.weight; P.bias = L.bias; P.gamma = L.bn_weight; P.beta = L.bn_bias;
        P.run_mean = L.bn_running_mean; P.run_var = L.bn_running_var; P.eps = L.bn_eps; P.momentum = L.bn_momentum;
        P.has_bn = L.bn_weight != nullptr; P.relu = L.relu; P.training = training;
        P.out = (l == num_layers - 1) ? out : buf[l & 1];
        P.out_inner = (l == num_layers - 1) ? out_transpose_inner : 0;
        P.counter = (training && L.bn_weight) ? L.bn_num_batches_tracked : nullptr;
        const size_t smem = (size_t)min(b, kFcRowChunk) * L.c_in * sizeof(float);
        static PerDeviceOnce fc_once;
        if (fc_once.first()) cudaFuncSetAttribute(fc_layer_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
        if (smem > 96 * 1024) { set_error("fc head: layer %d too wide (c_in=%d)", l, L.c_in); return SNB200_EUNSUPPORTED; }
        fc_layer_kernel<<<(L.c_out + kFcWarps - 1) / kFcWarps, kFcWarps * 32, smem, stream>>>(P);
        int rc = check_launch("fc layer");
        if (rc) return rc;
        cur = P.out;
    }
    return SNB200_OK;
}

}  // namespace snb
