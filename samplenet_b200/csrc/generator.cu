// generator.cu -- orchestration of the whole SampleNet generator (samplenet.py:90-104): path selection, workspace layout, and the
// stand-alone FC-head kernel of the non-fused paths.
//
//   path (training step at the headline size)                                          launches
//   default        cudaMemsetAsync(statistics, barrier word, FC exchange buffers)         (memset node)
//                  conv_stack_kernel   conv 1..5 + pool + fc1..fc4, persistent cooperative   1      (conv_stack.cu)
//   per-layer      memset; x_moments_kernel; tc_layer_kernel x4; fc_head_cluster_kernel      6      (encoder_tc.cu, here)
//   exact fp32     memset; conv_layer_kernel x5; fc_head_cluster_kernel                      6      (encoder.cu, here)
//   The default applies when the conv widths are 32/64/128 and the batch has at most 16 slices of 256 points per SM
//   (conv_stack_supported: one slice per SM keeps activations in registers, more than one parks them in L2 between layers -- still one
//   launch); everything else falls through to the per-layer tensor-core path, then to exact fp32.
//
// fc_head_cluster_kernel: the FC head (samplenet.py:99-104: 128->256->256->256->3M on B rows, BatchNorm over the batch) is tiny
// (7 MFLOP, 0.86 MB of weights) but has four layer-to-layer dependencies.  ONE thread-block cluster of 16 CTAs runs all of it:
// every CTA owns a slice of the output channels of each layer (so BatchNorm over the batch never leaves a warp: lane = batch
// row), activations are exchanged through a 32 KB global scratch that stays in L2, and layers are separated by cluster
// barriers.  The same kernel first turns the last conv layer's per-tile extrema into the pooled feature and applies every
// BatchNorm running-statistics update exactly once.  (The default path runs the head inside conv_stack_kernel instead.)
#include "encoder_internal.cuh"
#include <cooperative_groups.h>
#include <string.h>
namespace cg = cooperative_groups;

namespace snb {

constexpr int kHeadThreads = 256;      // 8 warps = 8 K slices; lanes = 8 row quads x 4 channel quads
constexpr int kHeadChPerCta = 16;
constexpr int kHeadMaxCluster = 16;

// bring-up instrumentation: SM-clock timestamps of CTA 0 / thread 0 at phase boundaries (read with snb200_debug_head_timestamps)
__device__ long long g_head_ts[64];
#define HEAD_TS(i) do { if (blockIdx.x == 0 && threadIdx.x == 0 && (i) < 64) g_head_ts[(i)] = clock64(); } while (0)

// RG = number of 32-row groups of the batch (b <= 32*RG).  256 threads = 8 warps.
// Everything here is a latency chain (4 dependent layers on <= 256 rows), so the kernel is organised around keeping loads
// off that chain and shared-memory wavefronts low:
//   * the weight slices of ALL layers do not depend on activations: they are fetched by TMA bulk copies (one mbarrier per
//     layer, one row per issuing thread) the moment the kernel starts;
//   * per-channel parameters (bias, gamma, beta, running stats) are read into registers before the layer's math;
//   * the per-CTA product [32 rows x c_in] x [c_in x 16 channels] is register-tiled 4 rows x 4 channels per thread with the
//     K range split over the 8 warps (2 LDS.128 wavefronts per 16 FMAs), partial sums are combined through shared memory in a
//     fixed order, and the combine leaves lane = batch row, warp = channel so BatchNorm over the batch is two warp shuffles.
template <int RG>
__global__ void __launch_bounds__(kHeadThreads) fc_head_cluster_kernel(const __grid_constant__ HeadParams P)
{
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = cluster.block_rank(), csize = cluster.num_blocks();
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    extern __shared__ __align__(16) float smem[];
    __shared__ uint64_t wbar[SNB200_MAX_FC_LAYERS];
    __shared__ float *s_wptr[SNB200_MAX_FC_LAYERS];
    // s_in  : [c_in_max][36]          one row group of the input, transposed (k-major), 4-row float4 reads
    // s_w   : per layer [16][c_in+4]  this CTA's first 16-channel weight slice, row-major like in HBM
    // s_part: [8 warps][32 rows][17]  partial dot products of the K slices
    int cmax = P.c_feat;
    for (int l = 0; l < P.num_fc; l++) cmax = max(cmax, P.fc[l].c_in);
    float *s_in = smem;
    float *s_part;
    HEAD_TS(0);
    if (tid == 0) {
        float *p = smem + (size_t)cmax * 36;
        for (int l = 0; l < P.num_fc; l++) { s_wptr[l] = p; p += (size_t)kHeadChPerCta * (P.fc[l].c_in + 4); }
        for (int l = 0; l < P.num_fc; l++) mbar_init(&wbar[l], 1);
        fence_mbar_init();
        if (!(P.dbg & 2))
            for (int l = 0; l < P.num_fc; l++) {   // arm every layer's barrier with the bytes its slice will deliver
                const HeadLayer &L = P.fc[l];
                const int per_cta = (L.c_out + csize - 1) / csize;
                const int c_lo = rank * per_cta, c_hi = min(L.c_out, c_lo + per_cta);
                const int nch = max(0, min(kHeadChPerCta, c_hi - c_lo));
                const bool tma_ok = (L.c_in & 3) == 0 && (reinterpret_cast<uintptr_t>(L.weight) & 15) == 0;
                if (tma_ok && nch > 0) mbar_expect_tx(&wbar[l], (uint32_t)nch * L.c_in * 4u);
            }
    }
    __syncthreads();
    {
        float *p = smem + (size_t)cmax * 36;
        for (int l = 0; l < P.num_fc; l++) p += (size_t)kHeadChPerCta * (P.fc[l].c_in + 4);
        s_part = p;
    }
    // ---- weight prefetch: thread t issues row (t % 16) of layer (t / 16)
    if (!(P.dbg & 2) && tid < P.num_fc * kHeadChPerCta) {
        const int l = tid / kHeadChPerCta, jrow = tid % kHeadChPerCta;
        const HeadLayer &L = P.fc[l];
        const int per_cta = (L.c_out + csize - 1) / csize;
        const int c_lo = rank * per_cta, c_hi = min(L.c_out, c_lo + per_cta);
        const int nch = max(0, min(kHeadChPerCta, c_hi - c_lo));
        const bool tma_ok = (L.c_in & 3) == 0 && (reinterpret_cast<uintptr_t>(L.weight) & 15) == 0;
        if (tma_ok && jrow < nch)
            tma_load_1d(s_wptr[l] + (size_t)jrow * (L.c_in + 4), L.weight + (size_t)(c_lo + jrow) * L.c_in, (uint32_t)L.c_in * 4u, &wbar[l]);
    }
    HEAD_TS(1);

    // ---- phase 0: pooled feature (this CTA's share) and the conv stack's running statistics (spread over the cluster)
    {
        const int total = P.b * P.c_feat;
        const double inv = 1.0 / P.count;
        for (int e = rank * kHeadThreads + tid; e < total; e += csize * kHeadThreads) {
            const int bi = e / P.c_feat, c = e % P.c_feat;
            float mx = -INFINITY, mn = INFINITY;
            const float *tm = P.tile_max + (size_t)bi * P.tiles_per_cloud * P.c_feat + c;
            const float *tn = P.tile_min + (size_t)bi * P.tiles_per_cloud * P.c_feat + c;
#pragma unroll 8
            for (int t = 0; t < P.tiles_per_cloud; t++) {
                mx = fmaxf(mx, __ldg(tm + (size_t)t * P.c_feat));
                mn = fminf(mn, __ldg(tn + (size_t)t * P.c_feat));
            }
            float v = mx;
            if (P.last_has_bn) {
                float mean, var;
                if (P.training) {
                    const double m = P.last_stats[c] * inv;
                    double vv = P.last_stats[P.c_feat + c] * inv - m * m;
                    if (vv < 0) vv = 0;
                    mean = (float)m; var = (float)vv;
                } else {
                    mean = P.last_run_mean[c]; var = P.last_run_var[c];
                }
                const float sc = P.last_gamma[c] * (1.0f / sqrtf(var + P.last_eps));
                const float sh = P.last_beta[c] - mean * sc;
                v = sc >= 0.f ? fmaf(mx, sc, sh) : fmaf(mn, sc, sh);  // max over points of a monotone map
            }
            if (P.last_relu) v = fmaxf(v, 0.f);
            P.feat[e] = v;
        }
        if (P.training) {   // training mode never reads the running buffers, so the update can go anywhere in the kernel
            int base = 0;
            const int gt = rank * kHeadThreads + tid, gn = csize * kHeadThreads;
            for (int l = 0; l < P.ru_num; l++) {
                for (int c = gt - base; c < P.ru_c[l]; c += gn) {
                    if (c < 0) continue;
                    const double m = P.ru_stats[l][c] * inv;
                    double v = P.ru_stats[l][P.ru_c[l] + c] * inv - m * m;
                    if (v < 0) v = 0;
                    const double unb = P.count > 1 ? v * (P.count / (P.count - 1)) : v;
                    const float mom = P.ru_momentum[l];
                    if (P.ru_mean[l]) P.ru_mean[l][c] = (1.f - mom) * P.ru_mean[l][c] + mom * (float)m;
                    if (P.ru_var[l]) P.ru_var[l][c] = (1.f - mom) * P.ru_var[l][c] + mom * (float)unb;
                }
                base = (base + P.ru_c[l]) % gn;
            }
        }
    }
    if (rank == csize - 1 && tid < P.num_counters) *P.counters[tid] += 1;
    HEAD_TS(2);
    cluster.sync();
    HEAD_TS(3);
    if (P.dbg & 1) return;

    // ---- FC layers
    const float *cur = P.feat;
    for (int l = 0; l < P.num_fc; l++) {
        const HeadLayer &L = P.fc[l];
        const bool last = (l == P.num_fc - 1);
        float *dst = last ? P.out : P.act[l & 1];
        const int c_in = L.c_in, ldw = c_in + 4;
        const int per_cta = (L.c_out + csize - 1) / csize;
        const int c_lo = rank * per_cta, c_hi = min(L.c_out, c_lo + per_cta);
        const bool vec = (c_in & 3) == 0;
        const bool tma_ok = vec && (reinterpret_cast<uintptr_t>(L.weight) & 15) == 0 && !(P.dbg & 2);
        float *sw = s_wptr[l];
        for (int cb = c_lo; cb < c_hi; cb += kHeadChPerCta) {      // passes of 16 channels (one pass unless c_out > 16*cluster)
            const int nch = min(kHeadChPerCta, c_hi - cb);
            HEAD_TS(4 + l * 8 + 0);
            // per-channel parameters of the two channels this warp finishes (warp, warp+8): loads start now
            float pb[2], pg[2], pbe[2], prm[2], prv[2];
#pragma unroll
            for (int j = 0; j < 2; j++) {
                const int c = cb + warp + 8 * j;
                const bool cv = (warp + 8 * j) < nch;
                pb[j] = (cv && L.bias) ? __ldg(L.bias + c) : 0.f;
                pg[j] = (cv && L.has_bn) ? __ldg(L.gamma + c) : 1.f;
                pbe[j] = (cv && L.has_bn) ? __ldg(L.beta + c) : 0.f;
                prm[j] = (cv && L.has_bn && L.run_mean) ? L.run_mean[c] : 0.f;
                prv[j] = (cv && L.has_bn && L.run_var) ? L.run_var[c] : 1.f;
            }
            if (cb == c_lo && tma_ok) {
                mbar_wait(&wbar[l], 0);                           // prefetched slice has landed
            } else {
                __syncthreads();
                for (int e = tid; e < kHeadChPerCta * c_in; e += kHeadThreads) {
                    const int jr = e / c_in, k = e % c_in;
                    sw[jr * ldw + k] = (jr < nch) ? __ldg(L.weight + (size_t)(cb + jr) * c_in + k) : 0.f;
                }
            }
            float y[RG][2];   // finished pre-activation of (row = g*32 + lane, channel = warp + 8*j)
#pragma unroll
            for (int g = 0; g < RG; g++) {
                y[g][0] = 0.f; y[g][1] = 0.f;
                const int r0 = g * 32;
                if (r0 < P.b) {   // uniform
                    const int rn = min(32, P.b - r0);
                    HEAD_TS(4 + l * 8 + 1);
                    __syncthreads();
                    HEAD_TS(4 + l * 8 + 2);
                    // input rows r0..r0+rn-1, transposed into s_in[k][r]; written by other CTAs of this kernel: plain loads,
                    // all of a thread's loads in flight before the first store
                    if (vec) {
                        // lane = batch row (conflict-free transposed stores), warps stride over the 16-byte k groups;
                        // up to 8 loads per thread in flight before the first store
                        const int q = c_in >> 2;
                        const float *src = cur + (size_t)(r0 + min(lane, rn - 1)) * c_in;
                        for (int q0 = warp; q0 < q; q0 += 8 * 8) {
                            float4 v[8];
#pragma unroll
                            for (int u = 0; u < 8; u++) {
                                const int kq = q0 + 8 * u;
                                v[u] = (kq < q) ? *(reinterpret_cast<const float4 *>(src) + kq) : make_float4(0, 0, 0, 0);
                            }
#pragma unroll
                            for (int u = 0; u < 8; u++) {
                                const int kq = q0 + 8 * u;
                                if (kq < q) {
                                    const float4 t = (lane < rn) ? v[u] : make_float4(0, 0, 0, 0);
                                    s_in[(kq * 4 + 0) * 36 + lane] = t.x; s_in[(kq * 4 + 1) * 36 + lane] = t.y;
                                    s_in[(kq * 4 + 2) * 36 + lane] = t.z; s_in[(kq * 4 + 3) * 36 + lane] = t.w;
                                }
                            }
                        }
                    } else {
                        for (int e = tid; e < 32 * c_in; e += kHeadThreads) {
                            const int r = e & 31, k = e >> 5;
                            s_in[k * 36 + r] = (r < rn) ? cur[(size_t)(r0 + r) * c_in + k] : 0.f;
                        }
                    }
                    __syncthreads();
                    HEAD_TS(4 + l * 8 + 3);
                    // register-tiled partial product: lane -> rows 4*rg..+3, channels cgp, cgp+4, cgp+8, cgp+12 (bank-conflict-free weight reads);
                    // warp -> K slice
                    const int rg = lane & 7, cgp = lane >> 3;
                    const int kr = ((c_in + 31) / 32) * 4;                    // K per warp, multiple of 4
                    const int k_lo = warp * kr, k_hi = min(c_in, k_lo + kr);
                    float acc[4][4];
#pragma unroll
                    for (int r = 0; r < 4; r++)
#pragma unroll
                        for (int j = 0; j < 4; j++) acc[r][j] = 0.f;
                    int k = k_lo;
                    for (; k + 4 <= k_hi; k += 4) {
                        float4 a[4], wv[4];
#pragma unroll
                        for (int i = 0; i < 4; i++) a[i] = *reinterpret_cast<const float4 *>(s_in + (k + i) * 36 + rg * 4);
#pragma unroll
                        for (int j = 0; j < 4; j++) wv[j] = *reinterpret_cast<const float4 *>(sw + (cgp + 4 * j) * ldw + k);
#pragma unroll
                        for (int j = 0; j < 4; j++) {
                            acc[0][j] = fmaf(a[3].x, wv[j].w, fmaf(a[2].x, wv[j].z, fmaf(a[1].x, wv[j].y, fmaf(a[0].x, wv[j].x, acc[0][j]))));
                            acc[1][j] = fmaf(a[3].y, wv[j].w, fmaf(a[2].y, wv[j].z, fmaf(a[1].y, wv[j].y, fmaf(a[0].y, wv[j].x, acc[1][j]))));
                            acc[2][j] = fmaf(a[3].z, wv[j].w, fmaf(a[2].z, wv[j].z, fmaf(a[1].z, wv[j].y, fmaf(a[0].z, wv[j].x, acc[2][j]))));
                            acc[3][j] = fmaf(a[3].w, wv[j].w, fmaf(a[2].w, wv[j].z, fmaf(a[1].w, wv[j].y, fmaf(a[0].w, wv[j].x, acc[3][j]))));
                        }
                    }
                    for (; k < k_hi; k++) {
                        const float4 a = *reinterpret_cast<const float4 *>(s_in + k * 36 + rg * 4);
#pragma unroll
                        for (int j = 0; j < 4; j++) {
                            const float wj = sw[(cgp + 4 * j) * ldw + k];
                            acc[0][j] = fmaf(a.x, wj, acc[0][j]); acc[1][j] = fmaf(a.y, wj, acc[1][j]);
                            acc[2][j] = fmaf(a.z, wj, acc[2][j]); acc[3][j] = fmaf(a.w, wj, acc[3][j]);
                        }
                    }
#pragma unroll
                    for (int r = 0; r < 4; r++)
#pragma unroll
                        for (int j = 0; j < 4; j++) s_part[(warp * 32 + rg * 4 + r) * 17 + cgp + 4 * j] = acc[r][j];
                    HEAD_TS(4 + l * 8 + 4);
                    __syncthreads();
                    HEAD_TS(4 + l * 8 + 5);
#pragma unroll
                    for (int j = 0; j < 2; j++) {   // fixed-order combination of the 8 K slices: lane = row, warp (+8) = channel
                        float t = 0.f;
#pragma unroll
                        for (int w8 = 0; w8 < 8; w8++) t += s_part[(w8 * 32 + lane) * 17 + warp + 8 * j];
                        y[g][j] = t;
                    }
                }
            }
            // bias, BatchNorm over the batch (rows live in lanes x row groups), activation, store
#pragma unroll
            for (int j = 0; j < 2; j++) {
                const int c = cb + warp + 8 * j;
                const bool cv = (warp + 8 * j) < nch;   // warp-uniform
                float scale = 1.f, shift = 0.f;
#pragma unroll
                for (int g = 0; g < RG; g++) y[g][j] += pb[j];
                if (L.has_bn && cv) {
                    float mean, var;
                    if (P.training) {
                        float sm = 0.f;
#pragma unroll
                        for (int g = 0; g < RG; g++)
                            if (g * 32 + lane < P.b) sm += y[g][j];
                        mean = warp_sum(sm) / (float)P.b;
                        float q = 0.f;
#pragma unroll
                        for (int g = 0; g < RG; g++)
                            if (g * 32 + lane < P.b) { const float d = y[g][j] - mean; q = fmaf(d, d, q); }
                        q = warp_sum(q);
                        var = q / (float)P.b;
                        if (lane == 0) {
                            const float unb = P.b > 1 ? q / (float)(P.b - 1) : var;
                            if (L.run_mean) L.run_mean[c] = (1.f - L.momentum) * prm[j] + L.momentum * mean;
                            if (L.run_var) L.run_var[c] = (1.f - L.momentum) * prv[j] + L.momentum * unb;
                        }
                    } else {
                        mean = prm[j]; var = prv[j];
                    }
                    const float invstd = 1.0f / sqrtf(var + L.eps);
                    scale = pg[j] * invstd;
                    shift = pbe[j] - mean * scale;
                }
                if (cv) {
#pragma unroll
                    for (int g = 0; g < RG; g++) {
                        const int row = g * 32 + lane;
                        if (row < P.b) {
                            float v = L.has_bn ? fmaf(y[g][j], scale, shift) : y[g][j];
                            if (L.relu) v = fmaxf(v, 0.f);
                            const int oc = (last && P.out_inner > 0) ? (c % P.out_inner) * (L.c_out / P.out_inner) + c / P.out_inner : c;
                            dst[(size_t)row * L.c_out + oc] = v;
                        }
                    }
                }
            }
        }
        cur = dst;
        HEAD_TS(4 + l * 8 + 6);
        cluster.sync();   // the next layer reads every CTA's slice
        HEAD_TS(4 + l * 8 + 7);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------------------
struct GenWorkspace {
    float *act[2];
    char *stats_base; size_t stats_bytes;
    double *mom; unsigned *counter; float *ll[SNB200_MAX_FC_LAYERS + 1];
    double *stats[SNB200_MAX_CONV_LAYERS];
    float *tile_max, *tile_min;
    float *feat;
    float *head_act[2];
    size_t total;
};

static GenWorkspace carve_gen_ws(void *base, int b, int n, int nconv, const snb200_layer *conv, int nfc, const snb200_layer *fc)
{
    GenWorkspace W;
    char *p = reinterpret_cast<char *>(base);
    size_t off = 0;
    int maxc = 8;
    for (int l = 0; l + 1 < nconv; l++) maxc = max(maxc, conv[l].c_out);
    const size_t act_bytes = align_up((size_t)b * n * maxc * sizeof(float), 256);
    W.act[0] = reinterpret_cast<float *>(p + off); off += act_bytes;
    W.act[1] = reinterpret_cast<float *>(p + off); off += act_bytes;
    W.stats_base = p + off;
    size_t sb = 0;
    W.mom = reinterpret_cast<double *>(p + off + sb); sb += 16 * sizeof(double);
    W.counter = reinterpret_cast<unsigned *>(p + off + sb); sb += 256 - 16 * sizeof(double);
    for (int l = 0; l < nconv; l++) {
        W.stats[l] = reinterpret_cast<double *>(p + off + sb);
        sb += align_up((size_t)(1 + kStatStride) * 2 * conv[l].c_out * sizeof(double), 256);   // canonical [2C] block + one line per accumulator
    }
    for (int l = 0; l <= SNB200_MAX_FC_LAYERS; l++) W.ll[l] = nullptr;
    for (int l = 0; l < nfc; l++) {   // exchange buffers of the fused head (zeroed with the statistics): the input of FC layer l
        const int width = (l == 0) ? conv[nconv - 1].c_out : fc[l - 1].c_out;
        W.ll[l] = reinterpret_cast<float *>(p + off + sb);
        sb += align_up((size_t)b * width * sizeof(float), 256);
    }
    W.stats_bytes = sb;
    off += sb;
    const int c_last = conv[nconv - 1].c_out;
    const int tpc = max((n + 127) / 128, (n + 63) / 64 + 1);  // upper bound over all paths (128- / 256-point tiles; conv-stack (cloud, CTA) slots)
    const size_t tb = align_up((size_t)b * tpc * c_last * sizeof(float), 256);
    W.tile_max = reinterpret_cast<float *>(p + off); off += tb;
    W.tile_min = reinterpret_cast<float *>(p + off); off += tb;
    W.feat = reinterpret_cast<float *>(p + off); off += align_up((size_t)b * c_last * sizeof(float), 256);
    int maxf = 8;
    for (int l = 0; l < nfc; l++) maxf = max(maxf, fc[l].c_out);
    const size_t hb = align_up((size_t)b * maxf * sizeof(float), 256);
    W.head_act[0] = reinterpret_cast<float *>(p + off); off += hb;
    W.head_act[1] = reinterpret_cast<float *>(p + off); off += hb;
    W.total = off;
    return W;
}

int debug_head_timestamps(long long *host_out64)
{
    return cudaMemcpyFromSymbol(host_out64, g_head_ts, sizeof(long long) * 64) == cudaSuccess ? SNB200_OK : SNB200_ECUDA;
}

size_t generator_workspace_bytes(int b, int n, int nconv, const snb200_layer *conv, int nfc, const snb200_layer *fc)
{
    return carve_gen_ws(nullptr, b, n, nconv, conv, nfc, fc).total;
}

static void fill_head_params(HeadParams &H, int b, int n, int tpc, int nconv, const snb200_layer *conv, int nfc, const snb200_layer *fc, int training,
                             float *out, int out_transpose_inner, float *feat_out, const GenWorkspace &W)
{
    memset(&H, 0, sizeof(H));
    const snb200_layer &LL = conv[nconv - 1];
    H.b = b; H.training = training; H.c_feat = LL.c_out; H.tiles_per_cloud = tpc;
    H.tile_max = W.tile_max; H.tile_min = W.tile_min; H.last_stats = W.stats[nconv - 1];
    H.last_gamma = LL.bn_weight; H.last_beta = LL.bn_bias; H.last_run_mean = LL.bn_running_mean; H.last_run_var = LL.bn_running_var;
    H.last_eps = LL.bn_eps; H.last_has_bn = LL.bn_weight != nullptr; H.last_relu = LL.relu;
    H.count = (double)b * (double)n;
    H.feat = feat_out ? feat_out : W.feat;
    if (training)
        for (int l = 0; l < nconv; l++) {
            if (!conv[l].bn_weight || (!conv[l].bn_running_mean && !conv[l].bn_running_var)) continue;
            const int i = H.ru_num++;
            H.ru_stats[i] = W.stats[l]; H.ru_mean[i] = conv[l].bn_running_mean; H.ru_var[i] = conv[l].bn_running_var;
            H.ru_momentum[i] = conv[l].bn_momentum; H.ru_c[i] = conv[l].c_out;
        }
    H.num_fc = nfc;
    for (int l = 0; l < nfc; l++) {
        HeadLayer &D = H.fc[l];
        D.c_in = fc[l].c_in; D.c_out = fc[l].c_out; D.weight = fc[l].weight; D.bias = fc[l].bias; D.gamma = fc[l].bn_weight; D.beta = fc[l].bn_bias;
        D.run_mean = fc[l].bn_running_mean; D.run_var = fc[l].bn_running_var; D.eps = fc[l].bn_eps; D.momentum = fc[l].bn_momentum;
        D.has_bn = fc[l].bn_weight != nullptr; D.relu = fc[l].relu;
    }
    H.act[0] = W.head_act[0]; H.act[1] = W.head_act[1];
    H.out = out; H.out_inner = out_transpose_inner;
    H.dbg = 0;
    H.stat_rep = 0;
    for (int l = 0; l <= SNB200_MAX_FC_LAYERS; l++) H.ll[l] = W.ll[l];
    if (training) {
        for (int l = 0; l < nconv; l++)
            if (conv[l].bn_weight && conv[l].bn_num_batches_tracked) H.counters[H.num_counters++] = conv[l].bn_num_batches_tracked;
        for (int l = 0; l < nfc; l++)
            if (fc[l].bn_weight && fc[l].bn_num_batches_tracked) H.counters[H.num_counters++] = fc[l].bn_num_batches_tracked;
    }
}

static bool tc_stack_supported(int nconv, const snb200_layer *conv)
{
    if (nconv < 2 || conv[0].c_in != 3) return false;
    if (conv[0].c_out % 8 != 0 || conv[0].c_out > 256) return false;
    for (int l = 1; l < nconv; l++)
        if (!tc_layer_supported(conv[l].c_in, conv[l].c_out)) return false;
    return true;
}

struct GenWorkspaceView {
    const double *stats[SNB200_MAX_CONV_LAYERS];
    const float *ll[SNB200_MAX_FC_LAYERS + 1];
};
GenWorkspaceView generator_workspace_view(void *fwd_workspace, int b, int n, int nconv, const snb200_layer *conv, int nfc, const snb200_layer *fc)
{
    GenWorkspace W = carve_gen_ws(fwd_workspace, b, n, nconv, conv, nfc, fc);
    GenWorkspaceView V;
    for (int l = 0; l < SNB200_MAX_CONV_LAYERS; l++) V.stats[l] = l < nconv ? W.stats[l] : nullptr;
    for (int l = 0; l <= SNB200_MAX_FC_LAYERS; l++) V.ll[l] = W.ll[l];
    return V;
}

int launch_generator_forward(int b, int n, int layout, const float *x, int nconv, const snb200_layer *conv, int nfc, const snb200_layer *fc,
                             int training, float *out, int out_transpose_inner, float *feat_out, int flags, void *workspace, cudaStream_t stream,
                             float *const *zsave)
{
    GenWorkspace W = carve_gen_ws(workspace, b, n, nconv, conv, nfc, fc);
    const bool cs_ok = conv_stack_supported(b, n, nconv, conv);
    const bool coop = !(flags & (SNB200_GEN_EXACT_FP32 | SNB200_GEN_PER_LAYER_KERNELS | SNB200_GEN_PROFILE_SKIP_CONV)) && tc_stack_supported(nconv, conv) && cs_ok;
    // SNB200_GEN_WORKSPACE_PRIMED: the caller keeps this workspace for this call sequence and its first 256 bytes (moments, barrier
    // and exit words) are zero -- freshly zeroed, or as the previous PRIMED call left them.  The persistent kernel then cleans the
    // rest itself (no memset node in front of it); every other path memsets as usual and re-zeroes those 256 bytes at the end.
    bool fuse_head_pre = !(flags & (SNB200_GEN_PROFILE_SKIP_HEAD | SNB200_GEN_SEPARATE_HEAD)) && b <= 256;
    for (int l = 0; l < nfc; l++) fuse_head_pre = fuse_head_pre && fc[l].c_in <= 1024;
    const bool primed = (flags & SNB200_GEN_WORKSPACE_PRIMED) != 0;
    const bool self_clean = primed && coop && fuse_head_pre;
    if ((training || coop) && !self_clean) cudaMemsetAsync(W.stats_base, 0, W.stats_bytes, stream);   // statistics, moments, grid-barrier counter
    struct Rezero {   // non-self-cleaning paths leave the head of a PRIMED workspace as they found it
        bool on; char *p; cudaStream_t s;
        ~Rezero() { if (on) cudaMemsetAsync(p, 0, 256, s); }
    } rezero{primed && !self_clean, W.stats_base, stream};
    const bool use_tc = !(flags & SNB200_GEN_EXACT_FP32) && tc_stack_supported(nconv, conv);
    int tpc = 0;
    if (flags & SNB200_GEN_PROFILE_SKIP_CONV) {
        tpc = (use_tc && cs_ok) ? conv_stack_slots_per_cloud(b, n) : use_tc ? tc_tiles_per_cloud(n) : (n + (conv[nconv - 1].c_out > 64 ? 128 : 256) - 1) / (conv[nconv - 1].c_out > 64 ? 128 : 256);
    } else if (use_tc && !(flags & SNB200_GEN_PER_LAYER_KERNELS) && cs_ok) {
        // one persistent cooperative launch for the conv stack AND (unless profiling flags split them) the pool + FC head
        HeadParams H;
        bool fuse_head = !(flags & (SNB200_GEN_PROFILE_SKIP_HEAD | SNB200_GEN_SEPARATE_HEAD)) && b <= 256;
        for (int l = 0; l < nfc; l++) fuse_head = fuse_head && fc[l].c_in <= 1024;
        if (fuse_head) fill_head_params(H, b, n, conv_stack_slots_per_cloud(b, n), nconv, conv, nfc, fc, training, out, out_transpose_inner, feat_out, W);
        int rc = launch_conv_stack(b, n, layout, x, nconv, conv, training, W.stats, W.mom, W.counter, W.tile_max, W.tile_min, &tpc,
                                   fuse_head ? &H : nullptr, (self_clean && fuse_head) ? W.stats_base + 256 : nullptr, W.stats_bytes - 256, stream, zsave, W.act);
        if (rc) return rc;
        if (fuse_head) return SNB200_OK;
    } else if (use_tc) {
        tpc = tc_tiles_per_cloud(n);
        const snb200_layer &L0 = conv[0];
        if (training && L0.bn_weight) {
            int rc = launch_x_moments(b, n, layout, x, W.mom, W.counter, L0.weight, L0.bias, L0.c_out, W.stats[0], stream);
            if (rc) return rc;
        }
        for (int l = 1; l < nconv; l++) {
            const snb200_layer &L = conv[l], &Lp = conv[l - 1];
            TcLayerParams P;
            memset(&P, 0, sizeof(P));
            P.b = b; P.n = n; P.tiles_per_cloud = tpc; P.c_in = L.c_in; P.c_out = L.c_out;
            if (l == 1) { P.x = x; P.x_layout = layout; P.w1 = L0.weight; P.b1 = L0.bias; }
            else P.in = W.act[(l - 1) & 1];
            P.in_has_bn = Lp.bn_weight != nullptr; P.in_stats = W.stats[l - 1];
            P.in_gamma = Lp.bn_weight; P.in_beta = Lp.bn_bias; P.in_run_mean = Lp.bn_running_mean; P.in_run_var = Lp.bn_running_var;
            P.in_eps = Lp.bn_eps; P.in_relu = Lp.relu; P.in_training = training;
            P.weight = L.weight; P.bias = L.bias;
            const bool last = (l == nconv - 1);
            P.out = last ? nullptr : W.act[l & 1];
            P.out_stats = (training && L.bn_weight) ? W.stats[l] : nullptr;
            P.tile_max = last ? W.tile_max : nullptr;
            P.tile_min = last ? W.tile_min : nullptr;
            int rc = launch_tc_layer(P, stream);
            if (rc) return rc;
        }
    } else {
        int rc = launch_simt_conv_stack(b, n, layout, x, nconv, conv, training, W.act[0], W.act[1], W.stats, W.tile_max, W.tile_min, &tpc, stream);
        if (rc) return rc;
    }

    if (flags & SNB200_GEN_PROFILE_SKIP_HEAD) return SNB200_OK;
    // ---- pool + FC head as its own cluster launch
    HeadParams H;
    fill_head_params(H, b, n, tpc, nconv, conv, nfc, fc, training, out, out_transpose_inner, feat_out, W);
    int cmax = conv[nconv - 1].c_out, max_out = 0;
    for (int l = 0; l < nfc; l++) { cmax = max(cmax, fc[l].c_in); max_out = max(max_out, fc[l].c_out); }
    // cluster size: enough CTAs that the widest layer is a single 16-channel pass per CTA, capped at 16 (non-portable size)
    int csize = 1;
    while (csize < kHeadMaxCluster && csize * kHeadChPerCta < max_out) csize *= 2;
    H.dbg = 0;
    size_t wfloats = 0;
    for (int l = 0; l < nfc; l++) wfloats += (size_t)kHeadChPerCta * (fc[l].c_in + 4);
    const size_t smem = ((size_t)cmax * 36 + wfloats + (size_t)8 * 32 * 17) * sizeof(float);
    const int rg = (b + 31) / 32;
    if (rg > 8) { set_error("generator: batch %d exceeds the FC head limit of 256 rows", b); return SNB200_EUNSUPPORTED; }
    if (smem > 200 * 1024) { set_error("generator: FC width %d too large for the shared-memory tile", cmax); return SNB200_EUNSUPPORTED; }
    static PerDeviceOnce once;
    if (once.first()) {
cudaFuncSetAttribute(fc_head_cluster_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        cudaFuncSetAttribute(fc_head_cluster_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        cudaFuncSetAttribute(fc_head_cluster_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        cudaFuncSetAttribute(fc_head_cluster_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        cudaFuncSetAttribute(fc_head_cluster_kernel<1>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
        cudaFuncSetAttribute(fc_head_cluster_kernel<2>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
        cudaFuncSetAttribute(fc_head_cluster_kernel<4>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
        cudaFuncSetAttribute(fc_head_cluster_kernel<8>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    }
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(csize); cfg.blockDim = dim3(kHeadThreads); cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = csize; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    cudaError_t e;
    if (rg == 1) e = cudaLaunchKernelEx(&cfg, fc_head_cluster_kernel<1>, H);
    else if (rg == 2) e = cudaLaunchKernelEx(&cfg, fc_head_cluster_kernel<2>, H);
    else if (rg <= 4) e = cudaLaunchKernelEx(&cfg, fc_head_cluster_kernel<4>, H);
    else e = cudaLaunchKernelEx(&cfg, fc_head_cluster_kernel<8>, H);
    if (e != cudaSuccess) { set_error("generator: FC head launch failed: %s", cudaGetErrorString(e)); cudaGetLastError(); return SNB200_ECUDA; }
    return check_launch("generator FC head");
}

}  // namespace snb
