// encoder_tc.cu -- the per-point MLP layers of the SampleNet generator on the 5th-generation tensor cores.
//
// Why tensor cores here and nowhere else: the conv stack (samplenet.py:90-94: 64->64->64->128->128 per point, 32 768
// points per step) is the one genuine dense contraction on the hot path (2.1 GFLOP of the step's 2.2).  Why 3xTF32: the
// reference computes these layers in fp32 and SampleNet's loss parity bar is 1e-5, which a single TF32/BF16 pass cannot
// hold.  Each fp32 operand is split exactly into hi = x & 0xffffe000 (representable in TF32) and lo = x - hi; the tile
// product is accumulated in fp32 TMEM as  A_hi*W_hi + A_hi*W_lo + A_lo*W_hi  (the dropped lo*lo term is < 2^-22 relative),
// i.e. three tcgen05.mma.kind::tf32 per K-step into the same accumulator.
//
// Kernel shape (one launch per layer, CTA = 128 points x all output channels):
//   prologue  all 256 threads: load the previous layer's RAW output tile, apply its BatchNorm+ReLU, split hi/lo and write
//             both into shared memory in the canonical K-major SWIZZLE_128B operand layout (rows of 128 B = 32 fp32 along K,
//             16-byte chunks XOR-swizzled with row%8, 8-row groups 1024 B apart); same for the weight tile (N rows);
//   MMA       one elected thread issues 3 x (KC/8) tcgen05.mma (M=128, N=c_out, K=8) per 64-wide K chunk, then
//             tcgen05.commit -> mbarrier;  accumulators live in TMEM (c_out columns x 128 lanes);
//   epilogue  tcgen05.ld 32x32b (thread = point row), + bias, raw store to HBM, and the tile is parked in shared memory
//             once more so that column sums / sums of squares (BatchNorm statistics) or column max/min (last layer, for the
//             max-pool) are reduced by one thread per channel in a fixed order.
// The layer's interface (workspace, statistics, extrema) is the one of the CUDA-core path in encoder.cu.
#include "encoder_internal.cuh"
#include "tcgen05.cuh"

namespace snb {

constexpr int kTcThreads = 256;
constexpr int kTcM = 128;   // points per CTA == UMMA M
constexpr int kTcKC = 32;   // K chunk resident in shared memory: one swizzle atom of 32 fp32 (128 B rows)

// byte offset of the 16-byte chunk `chunk` (0..7) of row `row` inside one [rows x 128 B] swizzle atom
__device__ __forceinline__ uint32_t sw128_off(int row, int chunk, int swizzle) { return (uint32_t)row * 128u + (uint32_t)((swizzle ? (chunk ^ (row & 7)) : chunk) << 4); }

__device__ __forceinline__ void split_store(unsigned char *hi_base, unsigned char *lo_base, uint32_t off, float4 v)
{
    float4 h, l;
    h.x = __uint_as_float(__float_as_uint(v.x) & 0xffffe000u); l.x = v.x - h.x;
    h.y = __uint_as_float(__float_as_uint(v.y) & 0xffffe000u); l.y = v.y - h.y;
    h.z = __uint_as_float(__float_as_uint(v.z) & 0xffffe000u); l.z = v.z - h.z;
    h.w = __uint_as_float(__float_as_uint(v.w) & 0xffffe000u); l.w = v.w - h.w;
    *reinterpret_cast<float4 *>(hi_base + off) = h;
    *reinterpret_cast<float4 *>(lo_base + off) = l;
}

template <int NOUT>  // padded output width: 64, 128 or 256 (UMMA N and TMEM columns)
__global__ void __launch_bounds__(kTcThreads, (NOUT <= 128 ? 2 : 1)) tc_layer_kernel(const __grid_constant__ TcLayerParams P)
{
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    // operand buffers, one 32-wide K atom each: [rows][128 B]
    constexpr uint32_t kAtomA = kTcM * 128, kAtomB = NOUT * 128;
    constexpr int NA = (kTcM * 8) / kTcThreads;   // float4 loads per thread for the A atom (4)
    constexpr int NB = (NOUT * 8) / kTcThreads;   // ... for the B atom (2 / 4 / 8)
    constexpr int LD = NOUT + 1;
    constexpr int H = kTcThreads / NOUT;          // row ranges in the epilogue reduction (4 / 2 / 1)
    unsigned char *sAhi = smem_raw;
    unsigned char *sAlo = sAhi + kAtomA;
    unsigned char *sBhi = sAlo + kAtomA;
    unsigned char *sBlo = sBhi + kAtomB;
    float *sStage = reinterpret_cast<float *>(smem_raw);  // epilogue: [128][NOUT+1] floats, aliases the operand buffers
    float *sPart = sStage + kTcM * LD;                    // [H][NOUT][4] partial reductions
    __shared__ float sScale[256], sShift[256];
    __shared__ float sX[kTcM * 3], sW1[256 * 3], sB1[256];
    __shared__ uint64_t mma_bar;
    __shared__ uint32_t tmem_base_smem;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int tile = blockIdx.x;
    const int cloud = tile / P.tiles_per_cloud;
    const int p0 = (tile % P.tiles_per_cloud) * kTcM;
    const int np = min(kTcM, P.n - p0);
    const int c_in = P.c_in, c_out = P.c_out;

    if (warp == 0) tmem_alloc(&tmem_base_smem, NOUT);
    if (tid == 32) {
        mbar_init(&mma_bar, 1);
        fence_mbar_init();
    }
    for (int c = tid; c < c_in; c += kTcThreads) {
        float sc = 1.f, sh = 0.f;
        if (P.in_has_bn)
            bn_scale_shift(P.in_stats, c_in, c, (double)P.b * (double)P.n, P.in_gamma, P.in_beta, P.in_run_mean, P.in_run_var, P.in_eps,
                           P.in_training, sc, sh);
        sScale[c] = sc;
        sShift[c] = sh;
    }
    if (P.x) {  // stage the 128 points of this tile and the first layer's weights
        const float *xc = P.x + (size_t)cloud * P.n * 3;
        for (int e = tid; e < kTcM * 3; e += kTcThreads) {
            const int r = e / 3, c = e % 3;
            sX[e] = (r < np) ? (P.x_layout == SNB200_BNC ? xc[(size_t)(p0 + r) * 3 + c] : xc[(size_t)c * P.n + p0 + r]) : 0.f;
        }
        for (int e = tid; e < c_in * 3; e += kTcThreads) sW1[e] = P.w1[e];
        for (int e = tid; e < c_in; e += kTcThreads) sB1[e] = P.b1 ? P.b1[e] : 0.f;
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_d = tmem_base_smem;
    const uint32_t idesc = make_idesc_tf32(kTcM, NOUT);

    const float *in_tile = P.x ? nullptr : P.in + ((size_t)cloud * P.n + p0) * c_in;
    uint32_t phase = 0;
    const int nchunks = (c_in + kTcKC - 1) / kTcKC;
    for (int kc = 0; kc < nchunks; kc++) {
        const int k0 = kc * kTcKC;
        // ---- 1. all global loads of this K chunk go out first (NA + NB independent 16-byte loads per thread) ...
        float4 av[NA], wv[NB];
#pragma unroll
        for (int u = 0; u < NA; u++) {
            const int e = tid + u * kTcThreads, row = e >> 3, k = k0 + (e & 7) * 4;
            av[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (!P.x && row < np && k < c_in) av[u] = __ldg(reinterpret_cast<const float4 *>(in_tile + (size_t)row * c_in + k));
        }
#pragma unroll
        for (int u = 0; u < NB; u++) {
            const int e = tid + u * kTcThreads, row = e >> 3, k = k0 + (e & 7) * 4;
            wv[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (row < c_out && k < c_in) wv[u] = __ldg(reinterpret_cast<const float4 *>(P.weight + (size_t)row * c_in + k));
        }
        // ---- 2. ... and fly while the tensor core finishes the previous chunk (its operands live in the same buffers)
        if (kc > 0) {
            mbar_wait(&mma_bar, phase);
            phase ^= 1;
            tc_fence_after();
        }
        // ---- 3. BatchNorm + ReLU of the previous layer, hi/lo split, swizzled store
#pragma unroll
        for (int u = 0; u < NA; u++) {
            const int e = tid + u * kTcThreads, row = e >> 3, ch = e & 7, k = k0 + ch * 4;
            float4 v = av[u];
            if (row < np && k < c_in) {
                if (P.x) {  // layer 1 on the fly: y = (w0*x + w1*y + w2*z) + b
                    const float px = sX[row * 3 + 0], py = sX[row * 3 + 1], pz = sX[row * 3 + 2];
                    v.x = fmaf(sW1[(k + 0) * 3 + 2], pz, fmaf(sW1[(k + 0) * 3 + 1], py, sW1[(k + 0) * 3 + 0] * px)) + sB1[k + 0];
                    v.y = fmaf(sW1[(k + 1) * 3 + 2], pz, fmaf(sW1[(k + 1) * 3 + 1], py, sW1[(k + 1) * 3 + 0] * px)) + sB1[k + 1];
                    v.z = fmaf(sW1[(k + 2) * 3 + 2], pz, fmaf(sW1[(k + 2) * 3 + 1], py, sW1[(k + 2) * 3 + 0] * px)) + sB1[k + 2];
                    v.w = fmaf(sW1[(k + 3) * 3 + 2], pz, fmaf(sW1[(k + 3) * 3 + 1], py, sW1[(k + 3) * 3 + 0] * px)) + sB1[k + 3];
                }
                v.x = fmaf(v.x, sScale[k + 0], sShift[k + 0]); v.y = fmaf(v.y, sScale[k + 1], sShift[k + 1]);
                v.z = fmaf(v.z, sScale[k + 2], sShift[k + 2]); v.w = fmaf(v.w, sScale[k + 3], sShift[k + 3]);
                if (P.in_relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
            }
            split_store(sAhi, sAlo, sw128_off(row, ch, P.swizzle), v);
        }
#pragma unroll
        for (int u = 0; u < NB; u++) {
            const int e = tid + u * kTcThreads, row = e >> 3, ch = e & 7;
            split_store(sBhi, sBlo, sw128_off(row, ch, P.swizzle), wv[u]);
        }
        fence_proxy_async();  // generic-proxy smem writes -> visible to the tensor core (async proxy)
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            const int ksteps = min(kTcKC, c_in - k0) / 8;
#pragma unroll 1
            for (int ks = 0; ks < ksteps; ks++) {
                const uint32_t kin = (uint32_t)ks * P.k_adv16 * 16u;  // byte advance inside the atom (32 B per K=8 step)
                const uint64_t a_hi = make_sdesc(smem_u32(sAhi) + kin, P.desc_hi);
                const uint64_t a_lo = make_sdesc(smem_u32(sAlo) + kin, P.desc_hi);
                const uint64_t b_hi = make_sdesc(smem_u32(sBhi) + kin, P.desc_hi);
                const uint64_t b_lo = make_sdesc(smem_u32(sBlo) + kin, P.desc_hi);
                const uint32_t acc = (kc > 0 || ks > 0) ? 1u : 0u;
                umma_tf32(tmem_d, a_lo, b_hi, idesc, acc);   // small terms first, the dominant hi*hi last
                umma_tf32(tmem_d, a_hi, b_lo, idesc, 1u);
                umma_tf32(tmem_d, a_hi, b_hi, idesc, 1u);
            }
            umma_commit(&mma_bar);  // arrives when every MMA issued so far has finished reading smem / writing TMEM
        }
    }
    mbar_wait(&mma_bar, phase);
    tc_fence_after();

    // ---- epilogue: TMEM -> registers (+bias) -> HBM raw store and a padded shared-memory copy of the tile
    {
        const int q = warp & 3;                 // TMEM lane quarter this warp may read
        const int row = q * 32 + lane;
        const int half = warp >> 2;             // warps 0-3 take the low half of the columns, 4-7 the high half
        const bool pv = row < np;
        float *orow = P.out ? P.out + ((size_t)cloud * P.n + p0 + row) * c_out : nullptr;
#pragma unroll 1
        for (int cb = half * (NOUT / 2); cb < (half + 1) * (NOUT / 2); cb += 32) {
            float v[32];
            tmem_ld32(tmem_d + ((uint32_t)(q * 32) << 16) + (uint32_t)cb, v);
#pragma unroll
            for (int j = 0; j < 32; j++) {
                const int c = cb + j;
                v[j] += (c < c_out) ? __ldg(P.bias + c) : 0.f;
                sStage[row * LD + c] = v[j];
            }
            if (orow && pv) {
                if (cb + 32 <= c_out && (c_out & 3) == 0) {
#pragma unroll
                    for (int j = 0; j < 32; j += 4) *reinterpret_cast<float4 *>(orow + cb + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                } else {
                    for (int j = 0; j < 32; j++)
                        if (cb + j < c_out) orow[cb + j] = v[j];
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    // ---- per-channel reductions over the tile's valid rows: H row ranges in parallel, combined in fixed order
    {
        const int c = tid % NOUT, h = tid / NOUT;
        const int r_lo = h * (kTcM / H), r_hi = min(np, (h + 1) * (kTcM / H));
        float sm = 0.f, ss = 0.f, mx = -INFINITY, mn = INFINITY;
        for (int r = r_lo; r < r_hi; r++) {
            const float v = sStage[r * LD + c];
            sm += v; ss = fmaf(v, v, ss); mx = fmaxf(mx, v); mn = fminf(mn, v);
        }
        float *pp = sPart + ((size_t)h * NOUT + c) * 4;
        pp[0] = sm; pp[1] = ss; pp[2] = mx; pp[3] = mn;
        __syncthreads();
        if (h == 0 && c < c_out) {
            for (int g = 1; g < H; g++) {
                const float *o = sPart + ((size_t)g * NOUT + c) * 4;
                sm += o[0]; ss += o[1]; mx = fmaxf(mx, o[2]); mn = fminf(mn, o[3]);
            }
            if (P.out_stats) {
                atomicAdd(P.out_stats + c, (double)sm);
                atomicAdd(P.out_stats + c_out + c, (double)ss);
            }
            if (P.tile_max) {
                P.tile_max[(size_t)tile * c_out + c] = mx;
                P.tile_min[(size_t)tile * c_out + c] = mn;
            }
        }
    }
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_d, NOUT);
}

// ------------------------------------------------------------------------------------------------------------------
// Input moments -> BatchNorm statistics of the first layer, analytically.  Layer 1 is affine in the point (y = W1 p + b1),
// so sum_y[c] = cnt*(w_c.mu + b_c) and sum_y2[c] = cnt*(var_c + mean_c^2) with var_c = w_c^T Cov(p) w_c.  Twelve sums over the
// cloud (fp32 per thread, fp64 across threads) replace an 8.4 MB activation write + read and a full pass of statistics.
// The last CTA to arrive converts the moments into the (sum, sumsq) layout every other layer uses.
// mom: [0..2] sum p, [3..8] sum xx,xy,xz,yy,yz,zz ; counter: arrival count (both zeroed by the caller's memset)
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) x_moments_kernel(int b, int n, int layout, const float *__restrict__ x, double *mom, unsigned *counter,
                                                        const float *__restrict__ w1, const float *__restrict__ b1, int c1, double *stats0)
{
    __shared__ double s_red[9][8];
    __shared__ bool s_last;
    const long long total = (long long)b * n;
    float acc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
        const long long bi = i / n, p = i % n;
        float px, py, pz;
        if (layout == SNB200_BNC) { const float *q = x + (bi * n + p) * 3; px = q[0]; py = q[1]; pz = q[2]; }
        else { const float *q = x + bi * n * 3 + p; px = q[0]; py = q[n]; pz = q[2 * (size_t)n]; }
        acc[0] += px; acc[1] += py; acc[2] += pz;
        acc[3] = fmaf(px, px, acc[3]); acc[4] = fmaf(px, py, acc[4]); acc[5] = fmaf(px, pz, acc[5]);
        acc[6] = fmaf(py, py, acc[6]); acc[7] = fmaf(py, pz, acc[7]); acc[8] = fmaf(pz, pz, acc[8]);
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int j = 0; j < 9; j++) {
        double v = (double)acc[j];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFullMask, v, o);
        if (lane == 0) s_red[j][warp] = v;
    }
    __syncthreads();
    if (threadIdx.x < 9) {
        double v = 0;
        for (int w = 0; w < 8; w++) v += s_red[threadIdx.x][w];
        atomicAdd(mom + threadIdx.x, v);
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(counter, 1u) == gridDim.x - 1);
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    const double cnt = (double)total;
    volatile double *vm = mom;
    const double mx = vm[0] / cnt, my = vm[1] / cnt, mz = vm[2] / cnt;
    const double cxx = vm[3] / cnt - mx * mx, cxy = vm[4] / cnt - mx * my, cxz = vm[5] / cnt - mx * mz;
    const double cyy = vm[6] / cnt - my * my, cyz = vm[7] / cnt - my * mz, czz = vm[8] / cnt - mz * mz;
    for (int c = threadIdx.x; c < c1; c += 256) {
        const double a0 = w1[c * 3 + 0], a1 = w1[c * 3 + 1], a2 = w1[c * 3 + 2];
        const double mean = a0 * mx + a1 * my + a2 * mz + (b1 ? (double)b1[c] : 0.0);
        double var = a0 * a0 * cxx + a1 * a1 * cyy + a2 * a2 * czz + 2.0 * (a0 * a1 * cxy + a0 * a2 * cxz + a1 * a2 * cyz);
        if (var < 0) var = 0;
        stats0[c] = cnt * mean;
        stats0[c1 + c] = cnt * (var + mean * mean);
    }
}

int launch_x_moments(int b, int n, int layout, const float *x, double *mom, unsigned *counter, const float *w1, const float *b1, int c1,
                     double *stats0, cudaStream_t stream)
{
    const long long total = (long long)b * n;
    int blocks = (int)((total + 255) / 256);
    if (blocks > kNumSMs) blocks = kNumSMs;
    x_moments_kernel<<<blocks, 256, 0, stream>>>(b, n, layout, x, mom, counter, w1, b1, c1, stats0);
    return check_launch("encoder input moments");
}

static size_t tc_smem_bytes(int nout)
{
    const size_t operands = 2 * (size_t)kTcM * 128 + 2 * (size_t)nout * 128;
    const size_t stage = (size_t)kTcM * (nout + 1) * sizeof(float) + (size_t)kTcThreads * 4 * sizeof(float);
    return (operands > stage ? operands : stage) + 1024;  // + alignment slack
}

bool tc_layer_supported(int c_in, int c_out) { return c_in % 8 == 0 && c_in >= 8 && c_in <= 256 && c_out >= 8 && c_out <= 256; }
int tc_tiles_per_cloud(int n) { return (n + kTcM - 1) / kTcM; }

int launch_tc_layer(const TcLayerParams &P0, cudaStream_t stream)
{
    TcLayerParams P = P0;
    if (P.desc_hi == 0) { P.desc_hi = kDescHiSw128; P.k_adv16 = 2; P.swizzle = 1; }
    const int nout = P.c_out <= 64 ? 64 : (P.c_out <= 128 ? 128 : 256);
    const size_t smem = tc_smem_bytes(nout);
    static PerDeviceOnce once;
    if (once.first()) {
        cudaFuncSetAttribute(tc_layer_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc_smem_bytes(64));
        cudaFuncSetAttribute(tc_layer_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc_smem_bytes(128));
        cudaFuncSetAttribute(tc_layer_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc_smem_bytes(256));
    }
    dim3 grid(P.b * P.tiles_per_cloud);
    if (nout == 64) tc_layer_kernel<64><<<grid, kTcThreads, smem, stream>>>(P);
    else if (nout == 128) tc_layer_kernel<128><<<grid, kTcThreads, smem, stream>>>(P);
    else tc_layer_kernel<256><<<grid, kTcThreads, smem, stream>>>(P);
    return check_launch("encoder tensor-core layer");
}

// Bring-up / unit-test entry: D (rows, c_out) = A (rows, c_in) * W (c_out, c_in)^T + bias through the tensor-core layer
// kernel with no BatchNorm, rows = b*n points.  desc_hi / k_adv16 / swizzle override the descriptor encoding (0 = defaults).
int launch_tc_gemm_debug(int rows, int c_in, int c_out, const float *A, const float *W, const float *bias, float *D, unsigned desc_hi,
                         int k_adv16, int swizzle, cudaStream_t stream)
{
    TcLayerParams P;
    memset(&P, 0, sizeof(P));
    P.in = A; P.c_in = c_in; P.c_out = c_out; P.b = 1; P.n = rows; P.tiles_per_cloud = tc_tiles_per_cloud(rows);
    P.weight = W; P.bias = bias; P.out = D;
    P.desc_hi = desc_hi; P.k_adv16 = k_adv16; P.swizzle = swizzle;
    return launch_tc_layer(P, stream);
}

}  // namespace snb
