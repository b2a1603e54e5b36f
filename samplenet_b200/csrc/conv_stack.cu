// conv_stack.cu -- the whole per-point MLP (conv layers 1..L, samplenet.py:90-94), the max-pool and the FC head as ONE persistent
// cooperative kernel whose activations never leave the SM.
//
// Round-2 design: the GEMMs are TRANSPOSED.  Every CTA (one per SM) owns `ppc` consecutive points of the flattened batch
// (ppc = ceil(B*N / #SMs) rounded up to 32: 224 at the headline size, so all 148 SMs carry the same load) for the whole stack and
// computes, per layer,            D^T[c_out x ppc] = W[c_out x K] . A^T[K x ppc]
//   * MMA A operand = the layer's weights, exact hi/lo TF32 split, held in TENSOR MEMORY (A-from-TMEM form of tcgen05.mma, columns
//     256..511: no shared-memory traffic for the weights during the MMAs), M = 128 rows (zero rows above c_out);
//   * MMA B operand = the activations: "N x K, K-major" SWIZZLE_128B tiles in shared memory, one 32-wide K chunk (hi + lo) per ring
//     slot, ring of three slots; N = ppc: ONE instruction covers all of the CTA's points (3 MMAs per K step of 8: lo*hi, hi*lo, hi*hi);
//   * the accumulator has TMEM lane = output channel, column = point.  A thread therefore owns ONE channel and ppc/4 points: the
//     BatchNorm batch statistics, the pool's max / min and the BatchNorm scale / shift are plain per-thread register loops -- no
//     shuffle networks, no per-channel tables in shared memory; the raw outputs of a layer are read from tensor memory ONCE
//     (tcgen05.ld, bias added) and stay in registers across the statistics grid barrier until they are normalised, split and stored
//     as the next layer's B operand (a warp's 32 lanes are the 32 consecutive k of one swizzled 128-byte row: conflict-free STS.32);
//   * training-mode BatchNorm needs the batch statistics of layer l before layer l+1 can start: per-CTA partial sums are added as
//     fixed-point words that carry their own arrival count (cs_fx_*: one 64-bit integer reduction per word, exact and order-
//     independent; a consumer that reads "count == grid size" holds the total -- no flag, no fence, no grid barrier between the
//     layers); only the last layer keeps fp64 accumulators and the one remaining grid barrier (the head needs every CTA's extrema
//     anyway).  Layer 1 (3 -> C) is evaluated on CUDA cores and its statistics follow analytically from the batch's 9 input
//     moments (phase 0);
//   * the last layer never materialises: only per-(CTA, cloud) max / min leave the SM (the max-pool commutes with the monotone
//     BN+ReLU map);
//   * the max-pool finalise and the FC head (fc1..fc4 with BatchNorm over the batch) run as the tail of the same launch, 8 output
//     channels per CTA; the 32 KB activation matrix of a layer travels between CTAs as self-validating words (a zeroed buffer,
//     producers never store the bit pattern 0, consumers spin on the data itself): no grid barrier in the head.
//   * batches beyond one 256-point slice per SM: the <kMulti = true> instantiation gives every CTA several slices and walks them inside
//     every layer, parking the raw layer outputs in global memory (L2) between layers; the <false> instantiation (the headline size)
//     keeps them in registers.
// Applicable to widths <= 128 with K in {32, 64, 128} and up to 16 slices per CTA; otherwise the per-layer kernels are used.
#include "encoder_internal.cuh"
#include "tcgen05.cuh"
#include <cooperative_groups.h>
#include <string.h>
#include <stdlib.h>

namespace snb {

constexpr int kCsMaxLayers = SNB200_MAX_CONV_LAYERS;
constexpr int kCsMaxSlicesPerCta = 16; // 256-point slices one CTA may walk per layer (batches beyond one slice per SM)
constexpr int kCsProducers = 512;     // 16 producer warps: warp & 3 = TMEM lane quarter (32 channels), warp >> 2 = column (point) group
constexpr int kCsThreadsAll = kCsProducers;        // (17 warps would cap the kernel at 96 registers: 5 warps on one scheduler)
constexpr int kCsIssuerWarp = 15;     // the producer warp whose lane 0 also issues the MMAs (q = 3: it owns a K chunk only in 128-wide layers)
constexpr int kCsMaxPts = 256;        // points per CTA = MMA N
constexpr int kCsMinPts = 64;
constexpr int kCsNPT = kCsMaxPts / 4; // points per thread (register array)
constexpr int kCsRing = 3;            // ring slots of one 32-wide K chunk (hi + lo)
constexpr int kCsMaxSeg = 8;          // clouds a CTA's point range may touch
constexpr uint32_t kCsColWhi = 256, kCsColWlo = 384;
constexpr int kCsLoPlane = kCsMaxPts * 128;          // a ring slot = hi plane (kCsMaxPts rows x 128 B) + lo plane, fixed size
constexpr uint32_t kCsSlotBytes = 2u * kCsLoPlane;   // tensor-memory columns of the weight operand (D occupies 0..255)

struct CsLayer {
    int c_in, c_out;
    const float *weight, *bias;
    // BatchNorm (+ReLU) applied to THIS layer's output when it is consumed by the next layer / the pool
    const float *gamma, *beta, *run_mean, *run_var;
    float eps;
    int has_bn, relu;
    double *stats;                      // [2][c_out] sum, sumsq (training) -- written here, read by the next layer and the head
    float *zsave;                       // optional (total points, c_out): this layer's raw output (with bias) kept for the backward pass
};

struct CsParams {
    const float *x; int layout;
    int b, n;
    long long total;                    // b * n points
    int ppc, npt;                       // points per CTA (multiple of 32), points per thread = ppc / 4
    int slots_per_cloud;                // pool partials: (cloud, slot) with slot = CTA index - first CTA touching the cloud
    int num_layers;                     // including layer 1
    CsLayer L[kCsMaxLayers];
    int training;
    double *mom;                        // [9] input moments (zeroed by the caller)
    unsigned *barrier;                  // grid barrier counter (zeroed by the caller)
    float *tile_max, *tile_min;         // (b, slots_per_cloud, c_last)
    int fuse_head;                      // run the pool + FC head as the tail of this launch
    HeadParams H;
    // self-cleaning workspace (SNB200_GEN_WORKSPACE_PRIMED): the caller guarantees moments / barrier word / exit word are zero; the
    // kernel zeroes [clean_ptr, clean_ptr + clean_bytes) itself before its first grid barrier and leaves the three words zero again
    int self_clean;
    char *clean_ptr;
    unsigned clean_bytes;
    // batches beyond one slice per SM: every CTA walks slices_per_cta slices (slice index = CTA + t * grid) layer by layer; the raw layer outputs
    // of its own slices travel through act[l & 1] (or the layer's zsave) -- thread-private round trips, no cross-CTA dependency
    int slices_per_cta, num_slices;
    float *act[2];
    int act_ld;                         // row stride (floats) of act[]: the widest parked layer, the SAME for every layer -- a slice's rows then occupy
                                        // the same bytes whatever the layer, so CTAs that drift layers apart (eval mode: nothing synchronises the grid
                                        // between layers) never touch each other's rows.  0 = each layer's own width (training: the statistics
                                        // exchange keeps the grid within one layer)
    int head_rows;                      // batch rows the FC head stages per pass (32 ... 128, a multiple of 32)
    int dbg;                            // bring-up switches (env SNB200_CS_DEBUG; 0 in the product): 1 = skip the statistics atomics (timing experiments only)
};

// bounded waits: a protocol bug must not hang the GPU box -- trap instead (surfaces as a launch failure in the next API call)
__device__ __forceinline__ void cs_mbar_wait(uint64_t *bar, uint32_t parity)
{
    uint32_t done = 0;
    for (unsigned spin = 0; !done; spin++) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
        if (spin > (1u << 24)) __trap();
    }
}
__device__ __forceinline__ void cs_grid_arrive(unsigned *counter)
{
    // release is cumulative over everything ordered before it by the preceding CTA barrier (the other threads' statistics atomics)
    asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(counter) : "memory");
}
__device__ __forceinline__ void cs_grid_wait(unsigned *counter, unsigned target)
{
    unsigned v, spin = 0;
    do {
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");
        if (++spin > (1u << 26)) __trap();
    } while (v < target);
}
__device__ __forceinline__ void cs_grid_barrier(unsigned *counter, unsigned target)
{
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(counter, 1u);
        unsigned v, spin = 0;
        do {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");
            if (++spin > (1u << 26)) __trap();
        } while (v < target);
    }
    __syncthreads();
}

// Self-validating exchange words: the exchange buffers are zeroed by the launch's memset and a producer never stores the bit
// pattern 0 (+0.0f travels as -0.0f, which is the same number to every consumer), so "word != 0" means "value present": a
// 4-byte store is atomic, a consumer spins on the data itself, and a value is usable one L2 round trip after it was stored -- no
// fence, no flag word, no grid barrier.  Loads bypass L1 (volatile).
__device__ __forceinline__ void cs_xchg_store(float *p, float v)
{
    unsigned u = __float_as_uint(v);
    if (u == 0u) u = 0x80000000u;
    asm volatile("st.volatile.global.u32 [%0], %1;" ::"l"(p), "r"(u) : "memory");
}
__device__ __forceinline__ unsigned cs_xchg_load1(const float *p)
{
    unsigned v;
    asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint4 cs_xchg_load4(const float *p)   // four consecutive words, 16-byte aligned
{
    uint4 v;
    asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
    return v;
}

// 8 weight rows (output channels cb..cb+nch-1) of an FC layer into shared memory, row-major as in HBM
__device__ __forceinline__ void cs_head_stage_weights(const HeadLayer &L, int cb, int nch, float *s_wh, int tid, bool producer)
{
    if (!producer) return;
    const int c_in = L.c_in;
    if ((c_in & 3) == 0) {
        const int q4 = c_in >> 2, total = 8 * q4;
        for (int e0 = tid; e0 < total; e0 += kCsProducers * 4) {
            float4 v[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int e = e0 + u * kCsProducers;
                const int jr = e / q4, kq = e - jr * q4;
                v[u] = (e < total && jr < nch) ? __ldg(reinterpret_cast<const float4 *>(L.weight + (size_t)(cb + jr) * c_in) + kq) : make_float4(0, 0, 0, 0);
            }
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int e = e0 + u * kCsProducers;
                if (e < total) *reinterpret_cast<float4 *>(s_wh + (size_t)e * 4) = v[u];
            }
        }
    } else {
        for (int e = tid; e < 8 * c_in; e += kCsProducers) {
            const int jr = e / c_in, k = e - jr * c_in;
            s_wh[e] = (jr < nch) ? __ldg(L.weight + (size_t)(cb + jr) * c_in + k) : 0.f;
        }
    }
}


__device__ __forceinline__ float cs_ld_now(const float *p)   // a load that is issued where it is written
{
    float v;
    asm volatile("ld.global.cg.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
    return v;
}

// one thread's share of an FC layer: 4 output channels x KR inputs of its batch row; x = the row's inputs (stride 1), w = 4 weight rows (stride c_in)
template <int KR>
__device__ __forceinline__ void cs_head_dot(const float *x, const float *w, int c_in, float (&a4)[4])
{
    float xr[KR];
#pragma unroll
    for (int i = 0; i < KR; i++) xr[i] = x[i];
#pragma unroll
    for (int i = 0; i < KR; i += 4) {
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const float4 wv = *reinterpret_cast<const float4 *>(w + j * c_in + i);
            a4[j] = fmaf(xr[i + 3], wv.w, fmaf(xr[i + 2], wv.z, fmaf(xr[i + 1], wv.y, fmaf(xr[i], wv.x, a4[j]))));
        }
    }
}

// (sum, sumsq) accumulator idx of a layer: the dense [2C] block, or (spread != 0) the padded accumulators behind it
__device__ __forceinline__ double cs_stat(const double *base, int c2, int idx, int spread)
{
    return __ldcg(spread ? base + c2 + (size_t)idx * kStatStride : base + idx);
}

// ---- BatchNorm statistics between the conv layers: fixed-point words that carry their own arrival count --------------------------
// Every CTA contributes one partial (sum, sum of squares) per channel and layer; the next layer cannot start before the totals are
// known.  A floating-point accumulator needs a separate "everybody has added" signal, ordered after the adds (release -> acquire:
// three dependent L2 round trips plus the fences).  Here each partial is converted to fixed point and added, together with a 1 in
// the top byte, by ONE 64-bit integer reduction: the word is its own arrival counter, a consumer that reads "count == grid size"
// holds the final total -- no fence, no flag, no barrier, one L2 round trip after the last add -- and integer addition is exact and
// order-independent, so the statistics are bit-reproducible by construction.
//   sum      : units of 2^-24, offset 2^47 per partial (non-negative fields cannot borrow from the count)   |partial| < 2^23
//   sumsq hi : units of 2^-9 (floor)                                                                          partial  < 2^38
//   sumsq lo : the remainder in units of 2^-48
// Absolute resolution of a total: 148 * 2^-25 = 4.4e-6 on a sum of b*n values and 5e-13 on a sum of squares -- far below what the
// eps of the BatchNorm lets through.  A partial outside the range (per-point pre-activations beyond ~3e4, or NaN / Inf input)
// contributes zero and poisons the CTA's pooled extrema (+-Inf), so the launch returns NaN rows instead of wrong numbers.
// Word placement: sum and sumsq-lo in the line of accumulator ch, sumsq-hi in the line of accumulator C + ch (two adds per line).
constexpr unsigned long long kFxCountOne = 1ull << 56, kFxFieldMask = kFxCountOne - 1;
constexpr long long kFxSumOffset = 1ll << 47;
__device__ __forceinline__ unsigned long long *cs_fx_line(double *stats, int C, int idx)
{
    return reinterpret_cast<unsigned long long *>(stats + 2 * C + (size_t)idx * kStatStride);
}
__device__ __forceinline__ void cs_fx_add(unsigned long long *p, unsigned long long v)
{
    asm volatile("red.relaxed.gpu.global.add.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long cs_fx_load(const unsigned long long *p)
{
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
// returns false when the partial is outside the fixed-point range (nothing but the arrival counts is added then)
__device__ __forceinline__ bool cs_fx_contribute(double *stats, int C, int ch, float sum, float sumsq)
{
    const bool ok = fabsf(sum) < 8388608.f && sumsq < 274877906944.f;   // (false for NaN)
    if (!ok) { sum = 0.f; sumsq = 0.f; }
    const long long ps = __double2ll_rn((double)sum * 16777216.0) + kFxSumOffset;
    const double qd = (double)sumsq, qh = floor(qd * 512.0);
    const long long hi = (long long)qh, lo = __double2ll_rn((qd - qh * (1.0 / 512.0)) * 281474976710656.0);
    unsigned long long *la = cs_fx_line(stats, C, ch), *lb = cs_fx_line(stats, C, C + ch);
    cs_fx_add(la, kFxCountOne + (unsigned long long)ps);
    cs_fx_add(lb, kFxCountOne + (unsigned long long)hi);
    cs_fx_add(la + 1, kFxCountOne + (unsigned long long)lo);
    return ok;
}
// spins until all G partials of channel ch are in, then decodes the totals
__device__ __forceinline__ void cs_fx_collect(double *stats, int C, int ch, unsigned G, double &sum, double &sumsq)
{
    const unsigned long long *la = cs_fx_line(stats, C, ch), *lb = cs_fx_line(stats, C, C + ch);
    unsigned long long a, b, c;
    unsigned spin = 0;
    do {
        a = cs_fx_load(la); c = cs_fx_load(la + 1); b = cs_fx_load(lb);
        if (++spin > (1u << 24)) __trap();
    } while ((unsigned)(a >> 56) != G || (unsigned)(b >> 56) != G || (unsigned)(c >> 56) != G);
    sum = (double)((long long)(a & kFxFieldMask) - (long long)G * kFxSumOffset) * (1.0 / 16777216.0);
    sumsq = (double)(long long)(b & kFxFieldMask) * (1.0 / 512.0) + (double)(long long)(c & kFxFieldMask) * (1.0 / 281474976710656.0);
}

__device__ long long g_cs_ts[64];
#define CS_TS(i) do { if (blockIdx.x == 0 && threadIdx.x == 0 && (i) < 64) g_cs_ts[(i)] = clock64(); } while (0)

__device__ __forceinline__ void cs_named_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }
__device__ __forceinline__ void cs_mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// One layer's weight row `ch`, columns [g*K/4, (g+1)*K/4), global -> registers (zero rows above c_out).  w holds up to 32 values.
__device__ __forceinline__ void cs_load_w(const CsLayer &L, int ch, int g, float *w)
{
    const int K4 = L.c_in >> 2;
    const bool valid = ch < L.c_out;
    const float4 *src = reinterpret_cast<const float4 *>(L.weight + (size_t)(valid ? ch : 0) * L.c_in + g * K4);
#pragma unroll
    for (int i4 = 0; i4 < 8; i4++) {
        if (i4 * 4 < K4) {
            const float4 t = valid ? __ldg(src + i4) : make_float4(0.f, 0.f, 0.f, 0.f);
            w[i4 * 4 + 0] = t.x; w[i4 * 4 + 1] = t.y; w[i4 * 4 + 2] = t.z; w[i4 * 4 + 3] = t.w;
        }
    }
}
// ... registers -> tensor memory (hi at kCsColWhi + k, lo at kCsColWlo + k; lane = output channel), exact hi/lo TF32 split
__device__ __forceinline__ void cs_store_w(uint32_t tmem_lane_base, int g, int K4, const float *w)
{
#pragma unroll
    for (int i8 = 0; i8 < 4; i8++) {
        if (i8 * 8 < K4) {
            uint32_t hi[8], lo[8];
#pragma unroll
            for (int i = 0; i < 8; i++) {
                const float v = w[i8 * 8 + i];
                const float h = __uint_as_float(__float_as_uint(v) & 0xffffe000u);
                hi[i] = __float_as_uint(h);
                lo[i] = __float_as_uint(v - h);
            }
            tmem_st8(tmem_lane_base + kCsColWhi + (uint32_t)(g * K4 + i8 * 8), hi);
            tmem_st8(tmem_lane_base + kCsColWlo + (uint32_t)(g * K4 + i8 * 8), lo);
        }
    }
    tmem_st_wait();
}

// (B) of the layer loop: this thread's channel = column k of the B operand: normalise, split and store its npt points into a ring slot.
// adr[i] = shared-space address of (row col0 + i, this thread's swizzled 4-byte cell) of the slot's hi plane; row col0 + 8 jb + i lies
// jb * 1024 bytes further (same swizzle phase: col0 and 8 jb are multiples of 8) and the lo plane kCsLoPlane bytes further: every store
// is [register + immediate].  One warp-uniform branch per 8 points; columns beyond the CTA's last point carry don't-care values (each
// accumulator column depends on its own operand row only, and those columns are excluded from every statistic).
template <int JB>
__device__ __forceinline__ void cs_write_block(const uint32_t (&v)[kCsNPT], float sc, float sh, float floor_v, const uint32_t (&adr)[8])
{
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const float t = fmaxf(fmaf(__uint_as_float(v[JB * 8 + i]), sc, sh), floor_v);   // floor_v = 0 (ReLU) or -inf
        const float h = __uint_as_float(__float_as_uint(t) & 0xffffe000u);
        asm volatile("st.shared.f32 [%0+%1], %2;" ::"r"(adr[i]), "n"(JB * 1024), "f"(h) : "memory");
        asm volatile("st.shared.f32 [%0+%1], %2;" ::"r"(adr[i]), "n"(JB * 1024 + kCsLoPlane), "f"(t - h) : "memory");
    }
}
__device__ __forceinline__ void cs_write_chunk(const uint32_t (&v)[kCsNPT], float sc, float sh, float floor_v, int npt, const uint32_t (&adr)[8])
{
    if (0 < npt) cs_write_block<0>(v, sc, sh, floor_v, adr);
    if (8 < npt) cs_write_block<1>(v, sc, sh, floor_v, adr);
    if (16 < npt) cs_write_block<2>(v, sc, sh, floor_v, adr);
    if (24 < npt) cs_write_block<3>(v, sc, sh, floor_v, adr);
    if (32 < npt) cs_write_block<4>(v, sc, sh, floor_v, adr);
    if (40 < npt) cs_write_block<5>(v, sc, sh, floor_v, adr);
    if (48 < npt) cs_write_block<6>(v, sc, sh, floor_v, adr);
    if (56 < npt) cs_write_block<7>(v, sc, sh, floor_v, adr);
}

// raw outputs of this thread's channel at its points -> global (points x channels): lanes = 32 consecutive channels of one point = 128
// contiguous bytes per warp store
__device__ __forceinline__ void cs_save_rows(float *dst, int ld, const uint32_t (&v)[kCsNPT], int npt, int nvalid)
{
    if (nvalid == npt) {
#pragma unroll
        for (int jb = 0; jb < kCsNPT / 8; jb++) {
            if (jb * 8 < npt) {
#pragma unroll
                for (int i = 0; i < 8; i++) dst[(size_t)(jb * 8 + i) * ld] = __uint_as_float(v[jb * 8 + i]);
            }
        }
    } else {
#pragma unroll
        for (int j = 0; j < kCsNPT; j++)
            if (j < nvalid) dst[(size_t)j * ld] = __uint_as_float(v[j]);
    }
}

// ... and back: this thread's channel at its points from a (points x channels) buffer (columns beyond the valid ones read as zero)
__device__ __forceinline__ void cs_load_rows(const float *src, int ld, uint32_t (&v)[kCsNPT], int npt, int nvalid)
{
#pragma unroll
    for (int jb = 0; jb < kCsNPT / 8; jb++) {
        if (jb * 8 < npt) {
#pragma unroll
            for (int i = 0; i < 8; i++) v[jb * 8 + i] = (jb * 8 + i < nvalid) ? __float_as_uint(__ldcg(src + (size_t)(jb * 8 + i) * ld)) : 0u;
        }
    }
}

// MMA issue for K chunk c of the current layer (whole warp waits, lane 0 issues): 4 K steps x 3 MMAs (3xTF32), then the commits
__device__ __forceinline__ void cs_issue_chunk(unsigned char *smem_raw, uint32_t slot_bytes, int ppc, uint32_t tmem0, uint32_t idesc, uint32_t gchunk,
                                               int c, int nchunks, uint64_t *bar_full, uint64_t *bar_ring, uint64_t *bar_acc, int lane)
{
    const uint32_t gi = gchunk + (uint32_t)c, slot = gi % kCsRing, use = gi / kCsRing;
    cs_mbar_wait(&bar_full[slot], use & 1u);
    tc_fence_after();
    if (lane == 0) {
        const uint32_t sb = smem_u32(smem_raw) + slot * slot_bytes;
        const uint64_t b_hi = make_sdesc(sb, kDescHiSw128), b_lo = make_sdesc(sb + (uint32_t)kCsLoPlane, kDescHiSw128);
        const uint32_t a_hi = tmem0 + kCsColWhi + (uint32_t)(c * 32), a_lo = tmem0 + kCsColWlo + (uint32_t)(c * 32);
#pragma unroll
        for (int ks = 0; ks < 4; ks++) {   // K = 8 tf32 per step: +8 TMEM columns (A), +32 bytes = +2 in the 16-byte address field (B)
            const uint64_t o = (uint64_t)(ks * 2);
            const uint32_t ka = (uint32_t)(ks * 8);
            umma_tf32_ts(tmem0, a_lo + ka, b_hi + o, idesc, (c > 0 || ks > 0) ? 1u : 0u);
            umma_tf32_ts(tmem0, a_hi + ka, b_lo + o, idesc, 1u);
            umma_tf32_ts(tmem0, a_hi + ka, b_hi + o, idesc, 1u);
        }
        umma_commit(&bar_ring[slot]);
        if (c == nchunks - 1) umma_commit(bar_acc);
    }
    __syncwarp();
}

// Thread roles: warps 0..15 (512 threads) are PRODUCERS: warp & 3 = q selects the TMEM lane quarter = 32 output channels (thread: channel
// ch = 32 q + lane), warp >> 2 = g selects npt = ppc/4 consecutive points (accumulator columns).  Warp 15 is ALSO the MMA ISSUER: lane 0 issues
// tcgen05.mma / tcgen05.commit for the K chunks in order (its own chunk, number 3, exists only in 128-wide layers and is prepared after
// chunks 0..2 have been issued -- the tensor pipe is busy with them for thousands of cycles by then).  Everything meets through mbarriers:
//   bar_w          producers -> issuer : the layer's weights are in tensor memory                          (512 arrivals)
//   bar_full[s]    producers -> issuer : ring slot s holds a prepared 32-wide K chunk of the B operand      (128 arrivals: one quarter)
//   bar_ring[s]    tensor core -> producers : the MMAs that read ring slot s have completed (tcgen05.commit)
//   bar_acc        tensor core -> producers : every MMA of this layer has completed
// kMulti: more than one 256-point slice per SM (large batches).  The single-slice instantiation keeps a layer's output in registers from
// one layer to the next; the multi-slice one walks its slices inside every layer and parks the raw outputs in global memory (L2) in between.
template <bool kMulti>
__global__ void __launch_bounds__(kCsThreadsAll, 1) conv_stack_kernel(const __grid_constant__ CsParams P)
{
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    // dynamic shared memory: ring of kCsRing slots x [hi: ppc x 128 B | lo: ppc x 128 B]; reused by the pool partials and by the head
    __shared__ __align__(16) float sX[kCsMaxPts * 3];
    __shared__ float sW1[128 * 3], sB1[128];
    __shared__ float sRedS[4][128], sRedQ[4][128];
    __shared__ uint64_t bar_full[kCsRing], bar_ring[kCsRing], bar_acc, bar_w;
    __shared__ uint32_t tmem_base_smem;
    __shared__ double sMom[9];
    __shared__ float sMomW[kCsProducers / 32][9];
    __shared__ int sBad;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const bool producer = true;                          // every warp prepares operands; warp kCsIssuerWarp also issues the MMAs
    const bool issuer = warp == kCsIssuerWarp;
    const int q = warp & 3, g = (warp >> 2) & 3;
    const int ch = q * 32 + lane;                       // the channel (TMEM lane) this producer thread owns in every layer
    const int G = gridDim.x;
    const int ppc = P.ppc, npt = P.npt, n = P.n;
    const long long P0 = (long long)blockIdx.x * ppc;   // first point (flattened batch) of this CTA
    const int npts = (int)min((long long)ppc, P.total - P0);
    const int col0 = g * npt;                           // first accumulator column of this thread
    const int nvalid = max(0, min(npt, npts - col0));   // its columns [0, nvalid) are real points
    const uint32_t slot_bytes = kCsSlotBytes;

    CS_TS(0);
    if (warp == 0) tmem_alloc(&tmem_base_smem, 512);
    if (tid == 0) {
        for (int s = 0; s < kCsRing; s++) { mbar_init(&bar_full[s], 128); mbar_init(&bar_ring[s], 1); }
        mbar_init(&bar_acc, 1);
        mbar_init(&bar_w, kCsProducers);
        fence_mbar_init();
    }
    if (tid < 9) sMom[tid] = 0.0;
    if (tid == 0) sBad = 0;
    // the points of this CTA and layer 1's weights
    const CsLayer &L1 = P.L[0];
    // slices of this CTA: slice index = CTA + t * grid (one slice, t = 0, unless kMulti)
    const int nslices = kMulti ? (P.num_slices - (int)blockIdx.x + G - 1) / G : 1;
    auto load_x_slice = [&](const long long P0s, const int nptss) {   // the slice's points -> sX (point-major xyz), zero beyond the batch
        if (P.layout == SNB200_BNC) {   // (b, n, 3): the flattened batch is contiguous
            const float *src = P.x + P0s * 3;
            const int nf = nptss * 3;
            for (int e = tid; e < ppc * 3; e += kCsProducers) sX[e] = (e < nf) ? __ldg(src + e) : 0.f;
        } else {
            for (int e = tid; e < ppc * 3; e += kCsProducers) {
                const int c = e / ppc, r = e - c * ppc;    // coalesced along points
                float xv = 0.f;
                if (r < nptss) {
                    const long long gp = P0s + r;
                    const int cloud = (int)(gp / n), pi = (int)(gp - (long long)cloud * n);
                    xv = __ldg(P.x + ((size_t)cloud * 3 + c) * n + pi);
                }
                sX[r * 3 + c] = xv;
            }
        }
    };
    if (producer) {
        if (!kMulti) load_x_slice(P0, npts);
        for (int e = tid; e < L1.c_out * 3; e += kCsProducers) sW1[e] = __ldg(L1.weight + e);
        for (int e = tid; e < L1.c_out; e += kCsProducers) sB1[e] = L1.bias ? __ldg(L1.bias + e) : 0.f;
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem0 = tmem_base_smem;
    const uint32_t tmem_lane = tmem0 + ((uint32_t)(q * 32) << 16);
    unsigned barrier_epoch = 0;
    const double cnt = (double)P.total, inv_cnt = 1.0 / cnt;
    CS_TS(1);
    const bool need_stats = P.training != 0;
    if (P.self_clean) {   // statistics accumulators and FC exchange words: zero before anybody adds to them (ordered by the first grid barrier)
        float4 *z = reinterpret_cast<float4 *>(P.clean_ptr);
        const unsigned n16 = P.clean_bytes >> 4;
        for (unsigned e = blockIdx.x * kCsThreadsAll + tid; e < n16; e += G * kCsThreadsAll) z[e] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (!(need_stats && L1.has_bn)) cs_grid_barrier(P.barrier, ++barrier_epoch * G);   // (no phase-0 barrier on this path)
    }

    // ---- the first tensor layer's weights: global -> registers now, tensor memory below (overlaps the phase-0 barrier)
    float wreg[32];
    if (producer) cs_load_w(P.L[1], ch, g, wreg);

    // ---- phase 0: input moments (training + BN after layer 1): 9 sums over this CTA's points, fp64 atomics, grid barrier
    if (need_stats && L1.has_bn) {
        const int mom_pts = kMulti ? ppc : npts;   // threads that hold a point (of some slice)
        if (producer) {
            float a9[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
            for (int t = 0; t < nslices; t++) {
                int nptss = npts;
                if (kMulti) {
                    const long long P0s = (long long)((int)blockIdx.x + t * G) * ppc;
                    nptss = (int)min((long long)ppc, P.total - P0s);
                    __syncthreads();
                    load_x_slice(P0s, nptss);
                    __syncthreads();
                }
                if (tid < nptss) {
                    const float px = sX[tid * 3 + 0], py = sX[tid * 3 + 1], pz = sX[tid * 3 + 2];
                    a9[0] += px; a9[1] += py; a9[2] += pz;
                    a9[3] = fmaf(px, px, a9[3]); a9[4] = fmaf(px, py, a9[4]); a9[5] = fmaf(px, pz, a9[5]);
                    a9[6] = fmaf(py, py, a9[6]); a9[7] = fmaf(py, pz, a9[7]); a9[8] = fmaf(pz, pz, a9[8]);
                }
            }
            if (warp * 32 < mom_pts) {
#pragma unroll
                for (int j = 0; j < 9; j++) {
                    float v = a9[j];
                    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFullMask, v, o);
                    if (lane == 0) sMomW[warp][j] = v;
                }
            }
        }
        __syncthreads();
        if (tid < 9) {   // one thread per moment: this CTA's sum, the grid's accumulator, then the arrival word (release: after the add, and --
            double t = 0.0;   // through the CTA barrier above -- after every thread's share of the self-clean stores)
            for (int w = 0; w * 32 < mom_pts && w < kCsProducers / 32; w++) t += (double)sMomW[w][tid];
            atomicAdd(P.mom + tid, t);
            cs_grid_arrive(reinterpret_cast<unsigned *>(P.mom + 9));
        }
    }
    if (producer) {   // weights of the first tensor layer into tensor memory
        cs_store_w(tmem_lane, g, P.L[1].c_in >> 2, wreg);
        tc_fence_before();
        cs_mbar_arrive(&bar_w);
    }
    if (need_stats && L1.has_bn) {
        if (tid < 9) {
            cs_grid_wait(reinterpret_cast<unsigned *>(P.mom + 9), 9u * G);
            sMom[tid] = __ldcg(P.mom + tid);
        }
        __syncthreads();
    }
    CS_TS(2);

    // ---- layer 1 (3 -> C1) on CUDA cores: this thread's channel at its npt points (raw, with bias), kept in registers
    uint32_t v[kCsNPT];   // (float bit patterns: tcgen05.ld writes straight into this array)
    auto layer1_eval = [&](const long long P0s, const int nvalids) {   // from the slice staged in sX
        if (producer && q * 32 < L1.c_out) {
            const bool cv = ch < L1.c_out;
            const float w0 = cv ? sW1[ch * 3 + 0] : 0.f, w1 = cv ? sW1[ch * 3 + 1] : 0.f, w2 = cv ? sW1[ch * 3 + 2] : 0.f, b1 = cv ? sB1[ch] : 0.f;
#pragma unroll
            for (int jb = 0; jb < kCsNPT / 8; jb++) {
                if (jb * 8 < npt) {
                    // 8 points = 24 consecutive floats = six 16-byte broadcast reads (col0 and 8 jb are multiples of 8: 96-byte aligned)
                    const float4 *xq = reinterpret_cast<const float4 *>(sX + (col0 + jb * 8) * 3);
                    float xr[24];
#pragma unroll
                    for (int u = 0; u < 6; u++) { const float4 t4 = xq[u]; xr[u * 4 + 0] = t4.x; xr[u * 4 + 1] = t4.y; xr[u * 4 + 2] = t4.z; xr[u * 4 + 3] = t4.w; }
#pragma unroll
                    for (int i = 0; i < 8; i++) v[jb * 8 + i] = __float_as_uint(fmaf(w2, xr[i * 3 + 2], fmaf(w1, xr[i * 3 + 1], w0 * xr[i * 3 + 0])) + b1);
                }
            }
            if (L1.zsave && cv) cs_save_rows(L1.zsave + (size_t)(P0s + col0) * L1.c_out + ch, L1.c_out, v, npt, nvalids);
        }
    };
    if (!kMulti) layer1_eval(P0, nvalid);

    uint32_t acc_uses = 0;              // completed accumulator phases (bar_acc parity)
    uint32_t gchunk = 0;                // global K-chunk counter (same sequence in producers and issuer): slot = gchunk % kCsRing
    // swizzle: point p's 128-byte row holds its 16-byte group c at position c ^ (p & 7); col0 is a multiple of 8, so p & 7 = j & 7.
    // toff[i]: byte offset inside a ring slot's hi plane of (row col0 + i, this thread's k = lane)
    uint32_t toff[8];
#pragma unroll
    for (int i = 0; i < 8; i++) toff[i] = (uint32_t)(col0 + i) * 128u + (uint32_t)(((lane >> 2) ^ i) << 4) + (uint32_t)((lane & 3) << 2);

    for (int l = 1; l < P.num_layers; l++) {
        const CsLayer &Lp = P.L[l - 1];   // producer of this layer's input (its BN+ReLU is applied when the registers are stored)
        const CsLayer &Lc = P.L[l];
        const int K = Lc.c_in, N = Lc.c_out;
        const int nchunks = K >> 5;
        const bool last = (l == P.num_layers - 1);
        const bool want_stats = need_stats && Lc.has_bn;

        {
            // =============================== producer warps ===============================
            CS_TS(3 + (l - 1) * 8 + 0);
            // (A) BatchNorm (+ReLU) of the producer layer for this thread's channel: two registers
            float sc = 1.f, sh = 0.f;
            if (Lp.has_bn && ch < K && g == 0) {   // one column group reads the statistics (hot L2 lines) and shares the result
                const float pgamma = cs_ld_now(Lp.gamma + ch), pbeta = cs_ld_now(Lp.beta + ch);   // in flight while the statistics are collected

                float mean, var;
                if (P.training) {
                    double m, vv;
                    if (l == 1) {   // analytic statistics of layer 1 from the input moments
                        const double mx = sMom[0] * inv_cnt, my = sMom[1] * inv_cnt, mz = sMom[2] * inv_cnt;
                        const double cxx = sMom[3] * inv_cnt - mx * mx, cxy = sMom[4] * inv_cnt - mx * my, cxz = sMom[5] * inv_cnt - mx * mz;
                        const double cyy = sMom[6] * inv_cnt - my * my, cyz = sMom[7] * inv_cnt - my * mz, czz = sMom[8] * inv_cnt - mz * mz;
                        const double a0 = sW1[ch * 3 + 0], a1 = sW1[ch * 3 + 1], a2 = sW1[ch * 3 + 2];
                        m = a0 * mx + a1 * my + a2 * mz + (double)sB1[ch];
                        vv = a0 * a0 * cxx + a1 * a1 * cyy + a2 * a2 * czz + 2.0 * (a0 * a1 * cxy + a0 * a2 * cxz + a1 * a2 * cyz);
                        if (vv < 0) vv = 0;
                        if (blockIdx.x == 0) {   // the (sum, sumsq) form every consumer of the statistics uses
                            Lp.stats[ch] = cnt * m;
                            Lp.stats[K + ch] = cnt * (vv + m * m);
                        }
                    } else {
                        double s1, s2;   // the grid's totals for this channel (see cs_fx_*: the words carry their own arrival count)
                        cs_fx_collect(Lp.stats, K, ch, (unsigned)G, s1, s2);
                        if (blockIdx.x == 0) { Lp.stats[ch] = s1; Lp.stats[K + ch] = s2; }   // the canonical block (head, backward pass)
                        m = s1 * inv_cnt;
                        vv = s2 * inv_cnt - m * m;
                        if (vv < 0) vv = 0;
                    }
                    mean = (float)m; var = (float)vv;
                } else {
                    mean = Lp.run_mean[ch]; var = Lp.run_var[ch];
                }
                const float invstd = 1.0f / sqrtf(var + Lp.eps);
                sc = pgamma * invstd;
                sh = pbeta - mean * sc;
            }
            if (Lp.has_bn) {
                if (g == 0 && ch < K) { sRedS[0][ch] = sc; sRedQ[0][ch] = sh; }   // (the partial-sum arrays are free between the layers)
                cs_named_sync(1, kCsProducers);
                if (ch < K) { sc = sRedS[0][ch]; sh = sRedQ[0][ch]; }
                cs_named_sync(1, kCsProducers);   // ... and must not be overwritten by this layer's partial sums before everybody has read them
            }
            CS_TS(3 + (l - 1) * 8 + 1);
            // (B) MMA issue (warp kCsIssuerWarp, chunks in order) around the operand preparation (every warp that owns a K chunk)
            const uint32_t idesc = make_idesc_tf32(128, ppc);
            if (issuer) {
                cs_mbar_wait(&bar_w, (uint32_t)(l - 1) & 1u);   // every thread's slice of this layer's weights is in tensor memory
                tc_fence_after();
            }
            const float bias = (ch < N && Lc.bias) ? __ldg(Lc.bias + ch) : 0.f;
            float sumL = 0.f, sqL = 0.f;                                     // (kMulti) this thread's statistics over all of its slices
            const float *act_in = kMulti && l > 1 ? (Lp.zsave ? Lp.zsave : P.act[(l - 1) & 1]) : nullptr;
            float *act_out = kMulti && !last ? (Lc.zsave ? Lc.zsave : P.act[l & 1]) : Lc.zsave;
            const int ld_in = (kMulti && !Lp.zsave && P.act_ld) ? P.act_ld : K, ld_out = (kMulti && !last && !Lc.zsave && P.act_ld) ? P.act_ld : N;
            // (cloud, slot) partial extrema of one slice (last layer); slot = the slice's rank among the slices that touch the cloud
            auto write_tiles = [&](const int sl, const int cl_first, const int nseg, const float *sPmax, const float *sPmin) {
                const int S = P.slots_per_cloud;
                for (int e = tid; e < nseg * N; e += kCsProducers) {
                    const int s = e / N, c = e - s * N;
                    const int cl = cl_first + s;
                    const int slot = sl - (int)(((long long)cl * n) / ppc);
                    float mx = -INFINITY, mn = INFINITY;
#pragma unroll
                    for (int gg = 0; gg < 4; gg++) {
                        mx = fmaxf(mx, sPmax[(gg * kCsMaxSeg + s) * 128 + c]);
                        mn = fminf(mn, sPmin[(gg * kCsMaxSeg + s) * 128 + c]);
                    }
                    if (sBad) { mx = INFINITY; mn = -INFINITY; }   // a statistics partial left the fixed-point range: the pooled feature becomes +-Inf
                                                                     // (fmaxf would drop a NaN) and the head's BatchNorm turns that into NaN rows
                    P.tile_max[((size_t)cl * S + slot) * N + c] = mx;
                    P.tile_min[((size_t)cl * S + slot) * N + c] = mn;
                    // the slice that holds a cloud's last point also fills the slots no slice owns
                    if ((int)((((long long)cl + 1) * n - 1) / ppc) == sl)
                        for (int s2 = slot + 1; s2 < S; s2++) {
                            P.tile_max[((size_t)cl * S + s2) * N + c] = -INFINITY;
                            P.tile_min[((size_t)cl * S + s2) * N + c] = INFINITY;
                        }
                }
            };
            int cl_first = 0, nseg = 0;
            float *sPmax = reinterpret_cast<float *>(smem_raw);                       // [4 groups][kCsMaxSeg][128]
            float *sPmin = sPmax + 4 * kCsMaxSeg * 128;
            for (int t = 0; t < nslices; t++) {
                // ---- this slice's geometry (kMulti: shadows the single-slice values of the kernel scope)
                const int sl = kMulti ? (int)blockIdx.x + t * G : (int)blockIdx.x;
                const long long P0 = (long long)sl * ppc;
                const int npts = (int)min((long long)ppc, P.total - P0);
                const int nvalid = max(0, min(npt, npts - col0));
                const bool lastslice = !kMulti || t == nslices - 1;
                if (kMulti) {   // the slice's input: layer 1 from the points, deeper layers from the raw outputs this thread parked a layer ago
                    if (l == 1) {
                        __syncthreads();
                        load_x_slice(P0, npts);
                        __syncthreads();
                        layer1_eval(P0, nvalid);
                    } else if (ch < K) {
                        cs_load_rows(act_in + (size_t)(P0 + col0) * ld_in + ch, ld_in, v, npt, nvalid);
                    }
                }
                if (issuer) {
                    for (int c = 0; c < min(nchunks, 3); c++)        // (this warp owns chunk 3)
                        cs_issue_chunk(smem_raw, slot_bytes, ppc, tmem0, idesc, gchunk, c, nchunks, bar_full, bar_ring, &bar_acc, lane);
                }
                if (q < nchunks) {
                    const uint32_t gi = gchunk + (uint32_t)q, slot = gi % kCsRing, use = gi / kCsRing;
                    if (use > 0) {   // the MMAs that read this ring slot last time must have completed
                        cs_mbar_wait(&bar_ring[slot], (use - 1) & 1u);
                        tc_fence_after();
                    }
                    uint32_t adr[8];
                    const uint32_t sbase = smem_u32(smem_raw) + slot * slot_bytes;
#pragma unroll
                    for (int i = 0; i < 8; i++) adr[i] = sbase + toff[i];
                    if (!last) CS_TS(3 + (l - 1) * 8 + 7);
                    cs_write_chunk(v, sc, sh, Lp.relu ? 0.f : -INFINITY, npt, adr);
                    tc_fence_before();     // this thread's tcgen05.ld of the previous accumulator are complete (wait::ld) and ordered
                    fence_proxy_async();   // generic-proxy writes -> visible to the tensor core
                    cs_mbar_arrive(&bar_full[slot]);
                }
                if (issuer && nchunks > 3) cs_issue_chunk(smem_raw, slot_bytes, ppc, tmem0, idesc, gchunk, 3, nchunks, bar_full, bar_ring, &bar_acc, lane);
                gchunk += (uint32_t)nchunks;
                CS_TS(3 + (l - 1) * 8 + 2);
                // (C) while the tensor core works: the NEXT layer's weight row into registers
                if (!last && lastslice) cs_load_w(P.L[l + 1], ch, g, wreg);
                // (D) every MMA of this slice has completed
                cs_mbar_wait(&bar_acc, acc_uses & 1u);
                acc_uses++;
                tc_fence_after();
                CS_TS(3 + (l - 1) * 8 + 3);
                // (E) the next layer's weights replace this layer's in tensor memory
                if (!last && lastslice) {
                    cs_store_w(tmem_lane, g, P.L[l + 1].c_in >> 2, wreg);
                    tc_fence_before();
                    cs_mbar_arrive(&bar_w);
                }
                // (F) the accumulator: lane = channel, this thread's npt columns -> registers (+bias); statistics / extrema on the way
                cl_first = (int)(P0 / n);
                nseg = (int)((P0 + npts - 1) / n) - cl_first + 1;
                if (q * 32 < N) {
#pragma unroll
                    for (int jb = 0; jb < kCsNPT / 8; jb++)
                        if (jb * 8 < npt) tmem_ld8(tmem_lane + (uint32_t)(col0 + jb * 8), v + jb * 8);
                    tmem_ld_wait();
                    tc_fence_before();   // the next MMA into this accumulator overwrites these columns: ordered through a CTA barrier below
                    float sum = 0.f, sq = 0.f;
                    if (nvalid == npt) {   // (every slice but the last: all columns are real points)
#pragma unroll
                        for (int jb = 0; jb < kCsNPT / 8; jb++) {
                            if (jb * 8 < npt) {
#pragma unroll
                                for (int i = 0; i < 8; i++) {
                                    const float u = __uint_as_float(v[jb * 8 + i]) + bias;
                                    v[jb * 8 + i] = __float_as_uint(u);
                                    sum += u; sq = fmaf(u, u, sq);
                                }
                            }
                        }
                    } else {
#pragma unroll
                        for (int j = 0; j < kCsNPT; j++) {
                            const float u = __uint_as_float(v[j]) + bias;
                            v[j] = __float_as_uint(u);
                            const float uu = j < nvalid ? u : 0.f;
                            sum += uu; sq = fmaf(uu, uu, sq);
                        }
                    }
                    if (kMulti) { sumL += sum; sqL += sq; }
                    else if (want_stats) { sRedS[g][ch] = sum; sRedQ[g][ch] = sq; }
                    // training with gradients (and kMulti: the next layer's input): the raw outputs go to HBM / L2 as well (a warp stores 32
                    // consecutive channels of a point)
                    if (act_out && ch < N) cs_save_rows(act_out + (size_t)(P0 + col0) * ld_out + ch, ld_out, v, npt, nvalid);
                    if (last) {   // per-cloud extrema of this thread's columns (the ring is dead: every MMA has completed)
                        for (int sgi = 0; sgi < nseg; sgi++) { sPmax[(g * kCsMaxSeg + sgi) * 128 + ch] = -INFINITY; sPmin[(g * kCsMaxSeg + sgi) * 128 + ch] = INFINITY; }
                        const long long gp0 = P0 + col0;
                        const int cl = (int)(gp0 / n);
                        const int first_nb = (int)((long long)(cl + 1) * n - gp0);   // column at which the next cloud starts
                        if (nvalid == npt && first_nb >= npt) {   // the common case: all of this thread's columns belong to one cloud
                            float mx = -INFINITY, mn = INFINITY;
#pragma unroll
                            for (int jb = 0; jb < kCsNPT / 8; jb++) {
                                if (jb * 8 < npt) {
#pragma unroll
                                    for (int i = 0; i < 8; i++) { mx = fmaxf(mx, __uint_as_float(v[jb * 8 + i])); mn = fminf(mn, __uint_as_float(v[jb * 8 + i])); }
                                }
                            }
                            sPmax[(g * kCsMaxSeg + cl - cl_first) * 128 + ch] = mx; sPmin[(g * kCsMaxSeg + cl - cl_first) * 128 + ch] = mn;
                        } else {   // columns straddle cloud boundaries (or the batch ends inside them): one masked pass per cloud segment
                            int jlo = 0;
                            for (int c2 = cl; jlo < nvalid; c2++) {
                                const int jhi = min(nvalid, (int)((long long)(c2 + 1) * n - gp0));
                                float mx = -INFINITY, mn = INFINITY;
#pragma unroll
                                for (int j = 0; j < kCsNPT; j++) {
                                    const bool in = j >= jlo && j < jhi;
                                    mx = in ? fmaxf(mx, __uint_as_float(v[j])) : mx;
                                    mn = in ? fminf(mn, __uint_as_float(v[j])) : mn;
                                }
                                sPmax[(g * kCsMaxSeg + c2 - cl_first) * 128 + ch] = mx; sPmin[(g * kCsMaxSeg + c2 - cl_first) * 128 + ch] = mn;
                                jlo = jhi;
                            }
                        }
                    }
                }
                if (kMulti) {   // every warp has read the accumulator (and written its extrema) before the next slice's MMAs / operand stores
                    cs_named_sync(1, kCsProducers);
                    if (last) {
                        write_tiles(sl, cl_first, nseg, sPmax, sPmin);
                        cs_named_sync(1, kCsProducers);   // ... and the extrema have been consumed
                    }
                }
            }
            if (kMulti && want_stats && q * 32 < N) { sRedS[g][ch] = sumL; sRedQ[g][ch] = sqL; }
            CS_TS(3 + (l - 1) * 8 + 4);
            if (want_stats || last) cs_named_sync(1, kCsProducers);
            if (want_stats && g == 0 && ch < N) {
                const float sm = (sRedS[0][ch] + sRedS[1][ch]) + (sRedS[2][ch] + sRedS[3][ch]);
                const float sqq = (sRedQ[0][ch] + sRedQ[1][ch]) + (sRedQ[2][ch] + sRedQ[3][ch]);
                if (last) {   // the head reads these behind the grid barrier below: plain fp64 accumulators, one 128-byte line each
                    double *acc = Lc.stats + 2 * N;
                    atomicAdd(acc + (size_t)ch * kStatStride, (double)sm);
                    atomicAdd(acc + (size_t)(N + ch) * kStatStride, (double)sqq);
                } else if (!cs_fx_contribute(Lc.stats, N, ch, (P.dbg & 1) ? 0.f : sm, (P.dbg & 1) ? 0.f : sqq)) {
                    sBad = 1;
                }
            }
            if (last && !kMulti) write_tiles((int)blockIdx.x, cl_first, nseg, sPmax, sPmin);
            CS_TS(3 + (l - 1) * 8 + 5);
            if (want_stats && last) {   // grid barrier: every CTA's statistics and extrema are in (the head reads both)
                cs_named_sync(1, kCsProducers);
                if (tid == 0) {
                    cs_grid_arrive(P.barrier);
                    CS_TS(3 + (l - 1) * 8 + 7);
                    cs_grid_wait(P.barrier, (barrier_epoch + 1) * G);
                }
                cs_named_sync(1, kCsProducers);
            } else if (!last && !want_stats) {
                // eval mode / no BatchNorm: still, every warp must have read its accumulator columns before the next layer's MMAs (which need
                // only K chunk 0) start overwriting them.  (With statistics, the CTA barrier in front of the atomics above already orders that.)
                cs_named_sync(1, kCsProducers);
            }
            CS_TS(3 + (l - 1) * 8 + 6);
        }
        if (want_stats && last) barrier_epoch++;
    }

    // every commit has been observed through bar_acc; tensor memory is released at the end of the kernel (off the head's critical path)
    tc_fence_before();
    __syncthreads();
    CS_TS(35);

    // ================================================================================================================
    // Fused tail: max-pool finalise + FC head (samplenet.py:97-104) on the CTAs of the grid.  Each FC layer's output channels
    // are spread over the CTAs, 8 per CTA (BatchNorm over the batch stays inside one warp: lane = batch row); activations go
    // through a few-KB global scratch that lives in L2 as self-validating words (cs_xchg_*), so the layers need no barrier.
    // Versus the 16-CTA cluster kernel this removes a launch and spreads each layer's latency chain over more SMs.
    // ================================================================================================================
    // Programmatic dependent launch: a kernel queued behind this one with the PDL attribute (the fused tail) may be scheduled onto
    // SMs as this grid's CTAs exit; it synchronises on this grid's completion itself (griddepcontrol.wait) before touching our output.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (!P.fuse_head) {   // stand-alone conv stack: the consumers (cluster head kernel, backward pass) read the canonical statistics block
        const CsLayer &LL = P.L[P.num_layers - 1];
        if (blockIdx.x == 0 && need_stats && LL.has_bn && tid < 2 * LL.c_out) LL.stats[tid] = cs_stat(LL.stats, 2 * LL.c_out, tid, 1);
        if (warp == 0) tmem_dealloc(tmem0, 512);
        return;
    }
    const HeadParams &H = P.H;
    // shared memory of the head (the conv stack's buffers are dead): input row group | partial sums | first weight rows of every layer
    float *s_in = reinterpret_cast<float *>(smem_raw);                 // [head_rows][c_in + 1] up to four row groups of the input
    int hcmax = H.c_feat, hcsum = 0;
    for (int l = 0; l < H.num_fc; l++) { hcmax = max(hcmax, H.fc[l].c_in); hcsum += H.fc[l].c_in; }
    const int RS = P.head_rows, gpb = RS >> 5;                                  // rows / row groups staged per pass
    float *s_part = reinterpret_cast<float *>(smem_raw) + (size_t)RS * (hcmax + 1);   // [8 K slices][8 channels][32 rows]
    float *s_wall = s_part + 8 * 8 * 32;                                       // per layer [8 channels][c_in] weight rows
    __shared__ uint64_t hbar[SNB200_MAX_FC_LAYERS];
    const double inv_cnt_h = 1.0 / H.count;
    const float inv_b = 1.0f / (float)H.b;
    CS_TS(36);
    // ---- weights do not depend on activations: the first 8-channel group of EVERY layer is fetched now, one TMA bulk copy per
    //      layer (the 8 rows are contiguous in HBM), completion on one mbarrier per layer; nobody touches them before the layer's math
    if (tid == 0) {
        for (int l = 0; l < H.num_fc; l++) mbar_init(&hbar[l], 1);
        fence_mbar_init();
        fence_proxy_async();   // the smem region was written through the generic proxy by the conv stack (every thread is past the CTA barrier above)
        int woff = 0;
        for (int l = 0; l < H.num_fc; l++) {
            const HeadLayer &L = H.fc[l];
            const int cpc = max(8, (((L.c_out + G - 1) / G + 7) / 8) * 8);
            const int lo = blockIdx.x * cpc, hi = min(L.c_out, lo + cpc);
            const bool tma_ok = (L.c_in & 3) == 0 && (hcmax & 3) == 0 && (reinterpret_cast<uintptr_t>(L.weight) & 15) == 0;
            if (lo < hi && tma_ok) {
                const uint32_t bytes = (uint32_t)min(8, hi - lo) * L.c_in * 4u;
                mbar_expect_tx(&hbar[l], bytes);
                tma_load_1d(s_wall + woff, L.weight + (size_t)lo * L.c_in, bytes, &hbar[l]);
            }
            woff += 8 * L.c_in;
        }
    }
    // (the pooled feature below is computed by the CTAs at the TOP of the grid, the FC layers by the CTAs at the bottom: the thread that issues
    //  these requests has no pooled element to wait for at the headline size)
    // In training mode the last layer's statistics barrier already ordered every CTA's extrema before this point; in eval mode
    // no grid barrier has been crossed yet.
    if (!(need_stats && P.L[P.num_layers - 1].has_bn)) cs_grid_barrier(P.barrier, ++barrier_epoch * G);
    // From here on CTAs exchange activations point to point through self-validating words (cs_xchg_*): consumers spin on the data
    // itself -- no fence, no flag word, no grid barrier.  The exchange buffers are zeroed by the launch's memset.
    //   stage 0 = the pooled feature, stage l+1 = the output of FC layer l
    // ---- phase P: pooled feature, spread over the grid
    {
        const int total = H.b * H.c_feat;
        const int gt = (G - 1 - (int)blockIdx.x) * kCsThreadsAll + tid, gn = G * kCsThreadsAll;
        float *ll0 = H.ll[0];
        for (int e = gt; e < total; e += gn) {
            const int bi = e / H.c_feat, c = e % H.c_feat;
            float mx = -INFINITY, mn = INFINITY;
            const float *tm = H.tile_max + (size_t)bi * H.tiles_per_cloud * H.c_feat + c;
            const float *tn = H.tile_min + (size_t)bi * H.tiles_per_cloud * H.c_feat + c;
            // every load of this element is issued before the first use
            const double st0 = (H.last_has_bn && H.training) ? cs_stat(H.last_stats, 2 * H.c_feat, c, H.stat_rep) : 0.0;
            const double st1 = (H.last_has_bn && H.training) ? cs_stat(H.last_stats, 2 * H.c_feat, H.c_feat + c, H.stat_rep) : 0.0;
            if (H.stat_rep && bi == 0 && H.last_has_bn && H.training) {   // canonical block of the last layer (read by the backward pass)
                double *canon = const_cast<double *>(H.last_stats);
                canon[c] = st0; canon[H.c_feat + c] = st1;
            }
            const float lg = H.last_has_bn ? __ldg(H.last_gamma + c) : 1.f, lb = H.last_has_bn ? __ldg(H.last_beta + c) : 0.f;
            for (int t0 = 0; t0 < H.tiles_per_cloud; t0 += 8) {   // 8 slots at a time, all 16 loads in flight before the first max / min
                float a8[8], b8[8];                                  // (a run-time trip count would serialise one L2 round trip per slot)
#pragma unroll
                for (int u = 0; u < 8; u++) {
                    const bool in = t0 + u < H.tiles_per_cloud;
                    a8[u] = in ? __ldcg(tm + (size_t)(t0 + u) * H.c_feat) : -INFINITY;
                    b8[u] = in ? __ldcg(tn + (size_t)(t0 + u) * H.c_feat) : INFINITY;
                }
#pragma unroll
                for (int u = 0; u < 8; u++) { mx = fmaxf(mx, a8[u]); mn = fminf(mn, b8[u]); }
            }
            float v = mx;
            if (H.last_has_bn) {
                float mean, var;
                if (H.training) {
                    const double m = st0 * inv_cnt_h;
                    double vv = st1 * inv_cnt_h - m * m;
                    if (vv < 0) vv = 0;
                    mean = (float)m; var = (float)vv;
                } else {
                    mean = H.last_run_mean[c]; var = H.last_run_var[c];
                }
                const float sc = lg * (1.0f / sqrtf(var + H.last_eps));
                const float sh = lb - mean * sc;
                v = sc >= 0.f ? fmaf(mx, sc, sh) : fmaf(mn, sc, sh);
            }
            if (H.last_relu) v = (v < 0.f) ? 0.f : v;
            cs_xchg_store(ll0 + e, v);
            H.feat[e] = v;
        }
    }
    CS_TS(37);
    __syncthreads();   // mbarrier inits visible; every thread of this CTA is done with the conv stack's shared memory
    CS_TS(38);

    int woff = 0;
    for (int l = 0; l < H.num_fc; l++) {
        const HeadLayer &L = H.fc[l];
        const bool lastfc = (l == H.num_fc - 1);
        float *dst = lastfc ? H.out : H.act[l & 1];
        float *lldst = lastfc ? nullptr : H.ll[l + 1];
        const float *llsrc = H.ll[l];
        const int c_in = L.c_in;
        float *s_wh = s_wall + woff;
        woff += 8 * c_in;
        // 8 output channels per pass and per CTA: few enough CTAs read the (shared) input that L2 does not serialise on it
        const int cpc = max(8, (((L.c_out + G - 1) / G + 7) / 8) * 8);
        const int c_lo = blockIdx.x * cpc, c_hi = min(L.c_out, c_lo + cpc);
        const int nrg = (H.b + 31) >> 5;
        const bool w_tma = (c_in & 3) == 0 && (hcmax & 3) == 0 && (reinterpret_cast<uintptr_t>(L.weight) & 15) == 0;
        CS_TS(39 + l * 6 + 0);
        for (int cb = c_lo; cb < c_hi; cb += 8) {                     // one group of 8 channels at a time
            const int nch = min(8, c_hi - cb);
            // per-channel parameters of the channel this warp will finish (warps 0..7): loads start now
            const int cw = cb + (warp & 7);
            const bool cvw = warp < 8 && (warp & 7) < nch;
            // (volatile loads: the compiler would otherwise sink them to their first use, behind the layer's math, and put an L2 round trip
            //  on the chain between two layers)
            const float pbias = (cvw && L.bias) ? cs_ld_now(L.bias + cw) : 0.f;
            const float pgam = (cvw && L.has_bn) ? cs_ld_now(L.gamma + cw) : 1.f;
            const float pbet = (cvw && L.has_bn) ? cs_ld_now(L.beta + cw) : 0.f;
            const float prm = (cvw && L.has_bn && L.run_mean) ? cs_ld_now(L.run_mean + cw) : 0.f;
            const float prv = (cvw && L.has_bn && L.run_var) ? cs_ld_now(L.run_var + cw) : 1.f;
            if (cb != c_lo || !w_tma) {   // (the first group of every layer was fetched by TMA at the start of the head)
                __syncthreads();
                cs_head_stage_weights(L, cb, nch, s_wh, tid, producer);
            }
            float yv[8];                                              // finished pre-activation: row group g, lane = row, warp = channel
#pragma unroll
            for (int gq = 0; gq < 8; gq++) yv[gq] = 0.f;
            // one row group (32 batch rows) of this channel group: stage the rows, partial products, fixed-order combine.  The common case (a batch
            // of at most 32 rows) runs ONE compact copy of this code; the 8-way unrolled form exists only for larger batches.  This kernel executes
            // every instruction of the head once per launch, so its pace is set by instruction fetch (ncu: 17 % of the warp samples are
            // "no instruction", almost all at branch targets), and seven skipped copies per FC layer are seven jumps to cold cache lines
            // Batch rows are staged up to head_rows (<= 128) at a time -- ONE polling pass over the exchange words for up to four row groups
            // (staging every group of 32 rows separately put four exchange latencies in sequence per layer for a batch of 128) -- and then
            // multiplied group by group: partial products, fixed-order combine.
            auto stage_rows = [&](const int r0) {
                const int rn = min(RS, H.b - r0), nr32 = (rn + 31) & ~31;   // live rows / rows written (dead rows are zero)
                if (producer) {   // stage rows r0..r0+rn-1 row-major with an odd row stride (conflict-free lane = row reads).  Lanes run
                                  // along k (coalesced 16-byte loads), a thread's loads are requested together and re-requested
                                  // until every word is present.
                    const int ldi = c_in + 1;
                    if ((c_in & 3) == 0) {
                        const int q4 = c_in >> 2, items = nr32 * q4;           // item = (row, 4 channels) = one 16-byte load
                        for (int i0 = tid; i0 < items; i0 += kCsProducers * 4) {
                            uint4 v[4];
                            unsigned spin = 0;
                            bool ok;
                            do {
                                ok = true;
#pragma unroll
                                for (int u = 0; u < 4; u++) {
                                    const int i = i0 + u * kCsProducers;
                                    const int r = i / q4, kq = i - r * q4;
                                    if (i < items && r < rn) v[u] = cs_xchg_load4(llsrc + (size_t)(r0 + r) * c_in + 4 * kq);
                                    else v[u] = make_uint4(1u, 1u, 1u, 1u);
                                }
#pragma unroll
                                for (int u = 0; u < 4; u++) ok = ok && v[u].x != 0u && v[u].y != 0u && v[u].z != 0u && v[u].w != 0u;
                                if (++spin > (1u << 24)) __trap();
                            } while (!ok);
#pragma unroll
                            for (int u = 0; u < 4; u++) {
                                const int i = i0 + u * kCsProducers;
                                if (i < items) {
                                    const int r = i / q4, kq = i - r * q4;
                                    float *d = s_in + r * ldi + 4 * kq;
                                    const bool live = r < rn;
                                    d[0] = live ? __uint_as_float(v[u].x) : 0.f; d[1] = live ? __uint_as_float(v[u].y) : 0.f;
                                    d[2] = live ? __uint_as_float(v[u].z) : 0.f; d[3] = live ? __uint_as_float(v[u].w) : 0.f;
                                }
                            }
                        }
                    } else {
                        for (int e = tid; e < nr32 * c_in; e += kCsProducers) {
                            const int r = e / c_in, k = e - r * c_in;
                            float xv = 0.f;
                            if (r < rn) {
                                unsigned q, spin = 0;
                                do {
                                    q = cs_xchg_load1(llsrc + (size_t)(r0 + r) * c_in + k);
                                    if (++spin > (1u << 24)) __trap();
                                } while (q == 0u);
                                xv = __uint_as_float(q);
                            }
                            s_in[r * ldi + k] = xv;
                        }
                    }
                }
            };
            auto group_math = [&](const int rl0, float &yout) {   // rows rl0 .. rl0 + 31 of the staged block
                if (producer) {   // warp -> (channel quad = warp & 1, K eighth = warp >> 1); lane = row
                    const int cq = (warp & 1) * 4, k8 = warp >> 1;
                    const int kr = ((c_in + 31) / 32) * 4;            // K per eighth, multiple of 4
                    const int k_lo = min(c_in, k8 * kr), k_hi = min(c_in, k_lo + kr);
                    const float *wq = s_wh + cq * c_in;
                    float a4[4] = {0.f, 0.f, 0.f, 0.f};
                    int k = k_lo;
                    if ((c_in & 3) == 0 && k_hi - k_lo == kr && (kr == 32 || kr == 16)) {   // the common widths (256, 128): fully unrolled, every
                        if (kr == 32) cs_head_dot<32>(s_in + (rl0 + lane) * (c_in + 1) + k_lo, wq + k_lo, c_in, a4);   // load in flight before the first FMA
                        else cs_head_dot<16>(s_in + (rl0 + lane) * (c_in + 1) + k_lo, wq + k_lo, c_in, a4);            // (same summation order as the loop below)
                        k = k_hi;
                    } else if ((c_in & 3) == 0) {
                        for (; k + 4 <= k_hi; k += 4) {
                            const float *xr = s_in + (rl0 + lane) * (c_in + 1) + k;
                            const float x0 = xr[0], x1 = xr[1], x2 = xr[2], x3 = xr[3];
#pragma unroll
                            for (int j = 0; j < 4; j++) {
                                const float4 wv = *reinterpret_cast<const float4 *>(wq + j * c_in + k);
                                a4[j] = fmaf(x3, wv.w, fmaf(x2, wv.z, fmaf(x1, wv.y, fmaf(x0, wv.x, a4[j]))));
                            }
                        }
                    }
                    for (; k < k_hi; k++) {
                        const float xv = s_in[(rl0 + lane) * (c_in + 1) + k];
#pragma unroll
                        for (int j = 0; j < 4; j++) a4[j] = fmaf(xv, wq[j * c_in + k], a4[j]);
                    }
#pragma unroll
                    for (int j = 0; j < 4; j++) s_part[(k8 * 8 + cq + j) * 32 + lane] = a4[j];
                }
                __syncthreads();
                CS_TS(39 + l * 6 + 2);
                if (warp < 8)   // fixed-order combination of the 8 K eighths: warp = channel, lane = row
                {
                    float t = 0.f;
#pragma unroll
                    for (int e8 = 0; e8 < 8; e8++) t += s_part[(e8 * 8 + warp) * 32 + lane];
                    yout = t;
                }
            };
            auto row_group = [&](const int gq, float &yout) {
                const bool first_of_block = gq % gpb == 0;
                if (gq > 0 || cb != c_lo || l > 0) __syncthreads();   // the previous user of s_in / s_part is done
                if (first_of_block) {
                    stage_rows(gq * 32);
                    if (cb == c_lo && gq == 0 && w_tma) mbar_wait(&hbar[l], 0);   // this layer's first weight rows have landed
                    __syncthreads();
                    CS_TS(39 + l * 6 + 1);
                }
                group_math((gq % gpb) * 32, yout);
            };
            if (nrg == 1) {
                row_group(0, yv[0]);
            } else {
#pragma unroll
                for (int gq = 0; gq < 8; gq++)
                    if (gq < nrg) row_group(gq, yv[gq]);
            }
            CS_TS(39 + l * 6 + 3);
            if (cvw) {
                float scale = 1.f, shift = 0.f;
#pragma unroll
                for (int gq = 0; gq < 8; gq++) yv[gq] += pbias;
                float bn_mean = 0.f, bn_q = 0.f;
                if (L.has_bn) {
                    float mean, var;
                    if (H.training) {
                        // batch statistics in one shuffle tree: deviations from a pivot sample (row 0), sum and sum of squares reduced
                        // together; var = (S2 - S1^2/n)/n is well conditioned because the pivot lies inside the data
                        const float pivot = __shfl_sync(kFullMask, yv[0], 0);
                        float s1 = 0.f, s2 = 0.f;
#pragma unroll
                        for (int gq = 0; gq < 8; gq++)
                            if (gq * 32 + lane < H.b) { const float d = yv[gq] - pivot; s1 += d; s2 = fmaf(d, d, s2); }
#pragma unroll
                        for (int o = 16; o > 0; o >>= 1) {
                            s1 += __shfl_xor_sync(kFullMask, s1, o);
                            s2 += __shfl_xor_sync(kFullMask, s2, o);
                        }
                        mean = fmaf(s1, inv_b, pivot);
                        bn_q = fmaxf(fmaf(-s1 * inv_b, s1, s2), 0.f);        // sum of squared deviations from the mean
                        var = bn_q * inv_b;
                        bn_mean = mean;
                    } else {
                        mean = prm; var = prv;
                    }
                    const float invstd = rsqrtf(var + L.eps);
                    scale = pgam * invstd;
                    shift = pbet - mean * scale;
                }
                CS_TS(39 + l * 6 + 4);
                auto store_group = [&](const int gq, const float y) {   // normalise + activate + hand over one row group of this channel
                    const int r = gq * 32 + lane;
                    if (r < H.b) {
                        float v = L.has_bn ? fmaf(y, scale, shift) : y;
                        if (L.relu) v = (v < 0.f) ? 0.f : v;   // (not fmaxf: a NaN must stay a NaN, as in torch -- and the statistics range guard relies on it)
                        if (lastfc) {
                            const int oc = (H.out_inner > 0) ? (cw % H.out_inner) * (L.c_out / H.out_inner) + cw / H.out_inner : cw;
                            dst[(size_t)r * L.c_out + oc] = v;
                        } else {
                            cs_xchg_store(lldst + (size_t)r * L.c_out + cw, v);   // the next layer's consumers spin on these words
                        }
                    }
                };
                if (nrg == 1) {   // (one compact copy on the common path, see row_group above)
                    store_group(0, yv[0]);
                } else {
#pragma unroll
                    for (int gq = 0; gq < 8; gq++)
                        if (gq < nrg) store_group(gq, yv[gq]);
                }
                if (L.has_bn && H.training && lane == 0) {   // running statistics: off the critical path
                    const float unb = H.b > 1 ? bn_q / (float)(H.b - 1) : bn_q * inv_b;
                    if (L.run_mean) L.run_mean[cw] = (1.f - L.momentum) * prm + L.momentum * bn_mean;
                    if (L.run_var) L.run_var[cw] = (1.f - L.momentum) * prv + L.momentum * unb;
                }
            }
        }
        CS_TS(39 + l * 6 + 5);
    }
    if (blockIdx.x == G - 1 && tid < H.num_counters) *H.counters[tid] += 1;
    // ---- running statistics of the conv stack: off the critical path, taken by the CTAs from the top of the grid (idle in the
    //      last FC layer); training mode never reads these buffers inside the kernel
    if (H.training) {
        const int gt = (G - 1 - (int)blockIdx.x) * kCsThreadsAll + tid, gn = G * kCsThreadsAll;
        int base = 0;
        for (int l = 0; l < H.ru_num; l++) {
            for (int c = gt - base; c < H.ru_c[l]; c += gn) {
                if (c < 0) continue;
                const double m = cs_stat(H.ru_stats[l], 2 * H.ru_c[l], c, H.ru_rep[l]) * inv_cnt_h;
                double v = cs_stat(H.ru_stats[l], 2 * H.ru_c[l], H.ru_c[l] + c, H.ru_rep[l]) * inv_cnt_h - m * m;
                if (v < 0) v = 0;
                const double unb = H.count > 1 ? v * (H.count / (H.count - 1)) : v;
                const float mom = H.ru_momentum[l];
                if (H.ru_mean[l]) H.ru_mean[l][c] = (1.f - mom) * H.ru_mean[l][c] + mom * (float)m;
                if (H.ru_var[l]) H.ru_var[l][c] = (1.f - mom) * H.ru_var[l][c] + mom * (float)unb;
            }
            base = (base + H.ru_c[l]) % gn;
        }
    }
    if (warp == 0) tmem_dealloc(tmem0, 512);
    if (P.self_clean) {   // the last CTA to leave puts the moments, the barrier word and the exit word back to zero for the next launch
        __syncthreads();
        if (tid == 0) {
            __threadfence();
            if (atomicAdd(P.barrier + 1, 1u) == G - 1) {
                for (int j = 0; j < 16; j++) P.mom[j] = 0.0;
                P.barrier[0] = 0u;
                P.barrier[1] = 0u;
            }
        }
    }
}

int debug_conv_stack_timestamps(long long *host_out64)
{
    return cudaMemcpyFromSymbol(host_out64, g_cs_ts, sizeof(long long) * 64) == cudaSuccess ? SNB200_OK : SNB200_ECUDA;
}

// ------------------------------------------------------------------------------------------------------------------
static int cs_num_sms()
{
    static int sms[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return kNumSMs;
    if (!sms[dev]) {
        int v = 0;
        sms[dev] = (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && v > 0) ? v : kNumSMs;
    }
    return sms[dev];
}

// Partition of the flattened batch: slices of ppc points (a multiple of 32: 4 column groups x 8-column tensor-memory loads; at most kCsMaxPts),
// spread evenly over the SMs; batches beyond one slice per SM give every CTA several slices (slice = CTA + t * grid).
struct CsPartition { int ppc, slices, grid, per_cta; };
static CsPartition cs_partition(long long total)
{
    const int sms = cs_num_sms();
    const long long rounds = max(1ll, (total + (long long)sms * kCsMaxPts - 1) / ((long long)sms * kCsMaxPts));
    long long ppc = (total + sms * rounds - 1) / (sms * rounds);
    ppc = (ppc + 31) / 32 * 32;
    if (ppc < kCsMinPts) ppc = kCsMinPts;
    if (ppc > kCsMaxPts) ppc = kCsMaxPts;
    CsPartition R;
    R.ppc = (int)ppc;
    R.slices = (int)((total + ppc - 1) / ppc);
    R.grid = min(sms, R.slices);
    R.per_cta = (R.slices + R.grid - 1) / R.grid;
    return R;
}
static int cs_points_per_cta(long long total) { return cs_partition(total).ppc; }

int conv_stack_slots_per_cloud(int b, int n)
{
    const int ppc = cs_points_per_cta((long long)b * n);
    return (n - 1) / ppc + 2;
}

bool conv_stack_supported(int b, int n, int nconv, const snb200_layer *conv)
{
    if (nconv < 2 || nconv > kCsMaxLayers || conv[0].c_in != 3) return false;
    if (conv[0].c_out % 32 != 0 || conv[0].c_out > 128) return false;
    for (int l = 1; l < nconv; l++) {
        if ((conv[l].c_in != 32 && conv[l].c_in != 64 && conv[l].c_in != 128) || conv[l].c_out > 128 || conv[l].c_out < 8) return false;
        if (reinterpret_cast<uintptr_t>(conv[l].weight) & 15) return false;   // 16-byte row loads
    }
    const long long total = (long long)b * n;
    const CsPartition R = cs_partition(total);
    if (R.per_cta > kCsMaxSlicesPerCta) return false;
    if ((R.ppc - 1) / n + 2 > kCsMaxSeg) return false;   // clouds one slice may touch
    if (R.grid > 255) return false;                      // the statistics words count arrivals in one byte
    return true;
}

int launch_conv_stack(int b, int n, int layout, const float *x, int nconv, const snb200_layer *conv, int training, double *const *stats,
                      double *mom, unsigned *barrier, float *tile_max, float *tile_min, int *tiles_per_cloud_out, const HeadParams *head,
                      char *clean_ptr, size_t clean_bytes, cudaStream_t stream, float *const *zsave, float *const *act)
{
    CsParams P;
    memset(&P, 0, sizeof(P));
    if (head) { P.fuse_head = 1; P.H = *head; }
    if (head && clean_ptr) { P.self_clean = 1; P.clean_ptr = clean_ptr; P.clean_bytes = (unsigned)clean_bytes; }
    P.x = x; P.layout = layout; P.b = b; P.n = n;
    P.total = (long long)b * n;
    const CsPartition R = cs_partition(P.total);
    P.ppc = R.ppc; P.slices_per_cta = R.per_cta; P.num_slices = R.slices;
    const bool multi = R.per_cta > 1;
    if (multi && !(act && act[0] && act[1])) { set_error("conv stack: %d slices per CTA need the activation workspace", R.per_cta); return SNB200_EINVAL; }
    if (act) { P.act[0] = act[0]; P.act[1] = act[1]; }
    // Training with BatchNorm on every layer: the statistics exchange orders the layers grid-wide (nobody starts layer l+1 before everybody has
    // finished layer l), so the parked rows may use each layer's natural stride (half the L2 footprint for the 64-wide layers).  Otherwise one
    // stride for all layers (the width carve_gen_ws sizes the two buffers for).
    bool layers_ordered = training != 0;
    for (int l = 0; l < nconv; l++) layers_ordered = layers_ordered && conv[l].bn_weight != nullptr;
    P.act_ld = 0;
    if (!layers_ordered) { P.act_ld = 8; for (int l = 0; l + 1 < nconv; l++) P.act_ld = max(P.act_ld, conv[l].c_out); }
    P.npt = P.ppc / 4;
    P.slots_per_cloud = (n - 1) / P.ppc + 2;
    P.num_layers = nconv; P.training = training;
    P.mom = mom; P.barrier = barrier; P.tile_max = tile_max; P.tile_min = tile_min;
    for (int l = 0; l < nconv; l++) {
        CsLayer &D = P.L[l];
        D.c_in = conv[l].c_in; D.c_out = conv[l].c_out; D.weight = conv[l].weight; D.bias = conv[l].bias;
        D.gamma = conv[l].bn_weight; D.beta = conv[l].bn_bias; D.run_mean = conv[l].bn_running_mean; D.run_var = conv[l].bn_running_var;
        D.eps = conv[l].bn_eps; D.has_bn = conv[l].bn_weight != nullptr; D.relu = conv[l].relu; D.stats = stats[l];
        D.zsave = zsave ? zsave[l] : nullptr;
    }
    { const char *e = getenv("SNB200_CS_DEBUG"); P.dbg = e ? atoi(e) : 0; }
    if (tiles_per_cloud_out) *tiles_per_cloud_out = P.slots_per_cloud;
    if (head) {
        P.H.tiles_per_cloud = P.slots_per_cloud;
        P.H.stat_rep = 1;
        // running statistics at the end of the head: the canonical [2C] blocks CTA 0 wrote on the way (ordered by the last layer's grid barrier),
        // except for the last layer, whose accumulators are read in place
        for (int i = 0; i < P.H.ru_num; i++) P.H.ru_rep[i] = (P.H.ru_stats[i] == stats[nconv - 1]) ? 1 : 0;
    }
    size_t smem = (size_t)kCsRing * kCsSlotBytes + 1024;
    if (head) {   // the fused tail reuses the same dynamic shared memory: input tile + partial sums + 8 weight rows
        int hcmax = head->c_feat;
        for (int l = 0; l < head->num_fc; l++) hcmax = max(hcmax, head->fc[l].c_in);
        size_t hcsum = 0;
        for (int l = 0; l < head->num_fc; l++) hcsum += head->fc[l].c_in;
        int rs = min(128, (b + 31) / 32 * 32);   // rows staged per pass: as many row groups as fit next to the partial sums and the weight rows
        size_t hs = 0;
        for (;; rs -= 32) {
            hs = ((size_t)rs * (hcmax + 1) + 2048 + (size_t)8 * hcsum) * sizeof(float) + 1024;
            if (hs <= 200 * 1024 || rs == 32) break;
        }
        if (hs > 200 * 1024) { set_error("conv stack: FC width %d too large for the fused head", hcmax); return SNB200_EUNSUPPORTED; }
        P.head_rows = rs;
        smem = max(smem, hs);
    }
    static PerDeviceOnce once;
    if (once.first()) {
        cudaFuncSetAttribute(conv_stack_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 204 * 1024);
        cudaFuncSetAttribute(conv_stack_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 204 * 1024);
    }
    const int grid = R.grid;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(kCsThreadsAll); cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative;
    attr[0].val.cooperative = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    cudaError_t e = multi ? cudaLaunchKernelEx(&cfg, conv_stack_kernel<true>, P) : cudaLaunchKernelEx(&cfg, conv_stack_kernel<false>, P);
    if (e != cudaSuccess) { set_error("conv stack: cooperative launch failed: %s", cudaGetErrorString(e)); cudaGetLastError(); return SNB200_ECUDA; }
    return check_launch("conv stack");
}

}  // namespace snb
