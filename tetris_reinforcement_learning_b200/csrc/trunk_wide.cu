// trunk_wide.cu — fused convolutional trunk for the WIDE nets (32 or 64 filters) on tcgen05:
//   * AlphaSame(blocks, filters = 32 | 64)  (reference architectures.py:60-126, pre-activation blocks :27-57;
//     BASELINE config 5 is AlphaSame(20, 64))
//   * BaseResNet / AuxBaseResNet            (reference architectures.py:159-271 / :279-353, post-activation
//     blocks :159-171; AuxBaseResNet(8, 32) is the Config default, ai.py:83)
// in eval mode with BatchNorm folded on the host (trunk.py).
//
// Same row-Toeplitz implicit GEMM as trunk_rows.cu — an MMA row is a BOARD ROW of a group of three
// images (128 slots incl. halo rows), the horizontal taps are folded into N:
//     D[row r, (x_out, oc)] += A[row r + dy - 1, (x_in, ic)] * B_dy[(x_out - x_in + 1, oc), ic]
// so ONE tcgen05.mma M=128 N=3F K=16 per (input column, vertical tap, 16 input channels).  At F = 64 that is
// N = 192: 96 clk of tensor math against 80 clk of shared-memory operand fetch per MMA (math bound), at
// F = 32 N = 96: 48 clk against 56 clk.
//
// What is different from the 16-filter kernel: nothing fits on chip any more.  A group's activations are
// 164 KB (F = 64) and a layer's weights 74 KB, the fp32 accumulator of a whole layer is 640 TMEM columns.  So
//   * activations live in a per-CTA scratch in global memory (two buffers per group: X and T/U, written in
//     place; 0.7 MB per CTA, i.e. L2 resident for all 148 CTAs) in exactly the UMMA operand layout
//     [x 10][k chunk F/8][row 136] x 16 B, and are STREAMED: one input column = one contiguous
//     cp.async.bulk (UBLKCP) into a ring of shared-memory column buffers;
//   * the accumulator is a RING of output columns in TMEM (512 / F slots): the MMAs of input column c
//     accumulate onto output columns c-1, c, c+1; column c-1 is final when they retire and an epilogue warp
//     set drains it (tcgen05.ld -> bias / residual / ReLU -> bf16 -> global scratch), re-zeroes the slot and
//     hands it back.  An MMA whose three slots wrap around the ring is issued as two;
//   * a layer's weights are double buffered in shared memory and prefetched one layer ahead;
//   * one CTA takes a PAIR of groups through all layers, alternating between them layer by layer, so the
//     write -> read-back latency of one group's layer boundary is covered by the other group's columns.
// Roles: 16 epilogue warps (4 sets x 128 TMEM lanes), one MMA warp, one copy warp; everything is handed
// over through mbarriers.  Every wait is bounded (status word + early exit) so that a protocol bug cannot
// hang the GPU.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "trl_common.cuh"

namespace {

constexpr int kSets = 4;                          // epilogue warp sets; set e drains output columns q = e (mod 4)
constexpr int kEpiWarps = 4 * kSets;
constexpr int kWarpMma = kEpiWarps, kWarpCopy = kEpiWarps + 1;
constexpr int kThreads = (kEpiWarps + 2) * 32;    // 576
constexpr int kImgs = 3;                          // images per group
constexpr int kSlotStride = 42;                   // image j row y -> slot 2 + 42 j + y (as trunk_rows.cu)
constexpr int kRowsBuf = 136;                     // operand rows per plane (slot s -> row s + 1)
constexpr int kPlaneBytes = kRowsBuf * 16;        // 2176: 8 channels x 136 rows
constexpr int kTmemCols = 512;
constexpr int kMaxOut = 5;                        // head channels: 1 (AlphaSame) or 4 own + 1 opponent (BaseResNet)

template <int F>
struct Geo {
    static constexpr int kKc = F / 8;                       // 8-channel planes per column
    static constexpr int kColBytes = kKc * kPlaneBytes;     // one input column of a group
    static constexpr int kBufBytes = 10 * kColBytes;        // one activation buffer of a group
    static constexpr int kLaneBytes = 2 * kBufBytes;        // X and T/U
    static constexpr int kLbo = 3 * F / 8 * 128;            // B: stride between 8-channel K chunks
    static constexpr int kWDyBytes = kKc * kLbo;            // 3F x F bf16: B matrix of one vertical tap
    static constexpr int kWLayerBytes = 3 * kWDyBytes;
    static constexpr int kRing = (F == 64) ? 4 : 8;         // input columns in flight
    static constexpr int kSlots = kTmemCols / F;            // output-column ring in TMEM
    static constexpr int kKSteps = F / 16;
    static constexpr int kBars = 2 * kRing + 2 * kSlots + 4 + 20;
    static constexpr int kOffIn = 2 * kWLayerBytes;
    static constexpr int kOffBar = kOffIn + kRing * kColBytes;
    static constexpr int kSmem = kOffBar + kBars * 8;
};

struct WideArgs {
    const __nv_bfloat16* grids;   // [n_images][400] 0/1 cells
    int n_images;
    int n_blocks;
    int stem_taps;                // 5 (AlphaSame) or 3 (BaseResNet)
    int pad_;
    int32_t* n_images_dev;        // optional device-side count (reset to 0 when consumed)
    const int32_t* out_row;       // optional output row of image k
    const uint4* w_packed;        // [2 n_blocks][3 dy][F/8][3F/8][8][8] bf16
    const float* consts;          // [(2 n_blocks + 1)][3][F] (bias, next scale, next bias), then head: W[n_out][F], scale, bias
    const float* stem_lut;        // [taps][1 << taps][F]
    __nv_bfloat16* out;           // [rows][n_out][400]
    uint8_t* scratch;             // [grid][2 lanes][2 buffers][10][F/8][136][16 B], zero initialised (pad rows stay zero)
    int32_t* counters;            // [0] work counter, [1] finished CTAs, [2] resident CTAs
    int32_t* status;              // [8]: [0] != 0 -> a wait timed out: tag, block, warp, parity, stream index
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}

// kind::f16 instruction descriptor: D = f32, A = B = bf16, both K-major, M = 128
__device__ __forceinline__ uint32_t idesc(uint32_t n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((n >> 3) << 17) | ((128u >> 4) << 24);
}

// issued by the whole (converged) MMA warp; elect.sync picks the lane (operands stay warp-uniform)
__device__ __forceinline__ void umma(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t id) {
    asm volatile(
        "{\n\t.reg .pred p, e;\n\t.reg .b64 da, db;\n\telect.sync _|e, 0xffffffff;\n\t"
        "mov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\tsetp.ne.b32 p, %6, 0;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, {%7, %7, %7, %7}, p;\n\t}\n"
        :: "r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(id), "r"(1u), "r"(0u) : "memory");
}

__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile(
        "{\n\t.reg .pred e;\n\telect.sync _|e, 0xffffffff;\n\t"
        "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}\n" :: "r"(bar) : "memory");
}

__device__ __forceinline__ bool mbar_try(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred q;\n\tmbarrier.try_wait.parity.shared::cta.b64 q, [%1], %2;\n\tselp.u32 %0, 1, 0, q;\n\t}\n"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}

// Bounded wait.  After ~2 s without progress the first waiter records where it stood in status[] and every
// wait of the launch returns at once from then on: the kernel ends (with garbage) instead of hanging the GPU.
__device__ __noinline__ void mbar_wait_slow(uint32_t bar, uint32_t parity, int tag, int idx, int32_t* status) {
    unsigned long long t0, t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (int spin = 0;; ++spin) {
        if (mbar_try(bar, parity)) return;
        if ((spin & 63) == 63) {
            if (*(volatile int32_t*)status != 0) return;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            if (t - t0 > 2000000000ull) {
                if (atomicCAS(status, 0, 1) == 0) {
                    status[1] = tag; status[2] = (int)blockIdx.x; status[3] = (int)(threadIdx.x >> 5);
                    status[4] = (int)parity; status[5] = idx;
                    __threadfence();
                }
                return;
            }
        }
    }
}

__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int tag, int idx, int32_t* status) {
    if (mbar_try(bar, parity)) return;
    mbar_wait_slow(bar, parity, tag, idx, status);
}

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(bar) : "memory");
}

__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
}

// contiguous global -> shared copy by the bulk-copy engine (async proxy), completion on an mbarrier
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&d)[16]) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n\t"
        "tcgen05.wait::ld.sync.aligned;\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr) : "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) d[i] = __uint_as_float(r[i]);
}

// issue only: the registers are valid after tmem_wait_ld()
__device__ __forceinline__ void tmem_ld16_issue(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ void tmem_st16_zero(uint32_t taddr) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1};\n"
        :: "r"(taddr), "r"(0u) : "memory");
}

__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ uint32_t pack_relu_bf16x2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
__device__ __forceinline__ float bf_lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf_hi(uint32_t w) { return __uint_as_float(w & 0xFFFF0000u); }

// 16 channels of one (column, row) as two 16-byte stores, one per 8-channel plane; relu optional
template <bool RELU>
__device__ __forceinline__ void store16(uint8_t* p, const float (&v)[16]) {
    uint4 a, b;
    if (RELU) {
        a.x = pack_relu_bf16x2(v[0], v[1]);   a.y = pack_relu_bf16x2(v[2], v[3]);
        a.z = pack_relu_bf16x2(v[4], v[5]);   a.w = pack_relu_bf16x2(v[6], v[7]);
        b.x = pack_relu_bf16x2(v[8], v[9]);   b.y = pack_relu_bf16x2(v[10], v[11]);
        b.z = pack_relu_bf16x2(v[12], v[13]); b.w = pack_relu_bf16x2(v[14], v[15]);
    } else {
        a.x = pack_bf16x2(v[0], v[1]);   a.y = pack_bf16x2(v[2], v[3]);
        a.z = pack_bf16x2(v[4], v[5]);   a.w = pack_bf16x2(v[6], v[7]);
        b.x = pack_bf16x2(v[8], v[9]);   b.y = pack_bf16x2(v[10], v[11]);
        b.z = pack_bf16x2(v[12], v[13]); b.w = pack_bf16x2(v[14], v[15]);
    }
    *reinterpret_cast<uint4*>(p) = a;
    *reinterpret_cast<uint4*>(p + kPlaneBytes) = b;
}

__device__ __forceinline__ void load16g(const float* __restrict__ p, float (&r)[16]) {   // warp-uniform address
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(p) + q);
        r[4 * q] = v.x; r[4 * q + 1] = v.y; r[4 * q + 2] = v.z; r[4 * q + 3] = v.w;
    }
}

// global writes of this thread (generic proxy) -> visible to the bulk-copy engine (async proxy) of this
// CTA, then one arrival per warp
__device__ __forceinline__ void publish_global(uint32_t bar) {
    asm volatile("fence.proxy.async;" ::: "memory");
    __syncwarp();
    if ((threadIdx.x & 31) == 0) mbar_arrive(bar);
}

enum { kTagColReady = 1, kTagInFree, kTagInFull, kTagOutFree, kTagOutDone, kTagWFree, kTagWFull };

// POST = false: AlphaSame (pre-activation blocks, 5x5 stem without BN, head = BN-ReLU-conv1x1(1)-BN-ReLU)
// POST = true : BaseResNet (post-activation blocks, 3x3 stem with BN-ReLU, head = 4 own-collapse sums + opponent collapse)
template <int F, bool POST>
__global__ void __launch_bounds__(kThreads, 1) trunk_wide_kernel(const __grid_constant__ WideArgs a) {
    using G = Geo<F>;
    constexpr int NOUT = POST ? 5 : 1;
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint32_t s_tmem_base;
    __shared__ int s_pair;
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int L = 2 * a.n_blocks;
    int32_t* status = a.status;
    const uint32_t bars = smem_u32(smem + G::kOffBar);
    // barrier map
    auto in_full = [&](int k) { return bars + 8u * (uint32_t)k; };
    auto in_free = [&](int k) { return bars + 8u * (uint32_t)(G::kRing + k); };
    auto out_done = [&](int r) { return bars + 8u * (uint32_t)(2 * G::kRing + r); };
    auto out_free = [&](int r) { return bars + 8u * (uint32_t)(2 * G::kRing + G::kSlots + r); };
    auto w_full = [&](int b) { return bars + 8u * (uint32_t)(2 * G::kRing + 2 * G::kSlots + b); };
    auto w_free = [&](int b) { return bars + 8u * (uint32_t)(2 * G::kRing + 2 * G::kSlots + 2 + b); };
    auto col_ready = [&](int ln, int c) { return bars + 8u * (uint32_t)(2 * G::kRing + 2 * G::kSlots + 4 + ln * 10 + c); };
    if (tid == 0) atomicAdd(a.counters + 2, 1);

    if (tid == 0) {
        for (int k = 0; k < G::kRing; ++k) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(in_full(k)));
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(in_free(k)));
        }
        for (int r = 0; r < G::kSlots; ++r) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(out_done(r)));
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 4;" :: "r"(out_free(r)));
        }
        for (int b = 0; b < 2; ++b) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(w_full(b)));
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(w_free(b)));
        }
        for (int i = 0; i < 20; ++i) asm volatile("mbarrier.init.shared::cta.b64 [%0], 4;" :: "r"(col_ready(i / 10, i % 10)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == kWarpMma) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(&s_tmem_base)), "r"(kTmemCols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, s_tmem_base, 0);

    trl_grid_dep_wait();
    int n_images = a.n_images;
    if (a.n_images_dev) n_images = min(n_images, *a.n_images_dev);
    const int n_groups = (n_images + kImgs - 1) / kImgs;
    const int n_pairs = (n_groups + 1) / 2;
    uint8_t* const scratch = a.scratch + (size_t)blockIdx.x * 2 * G::kLaneBytes;

    // epilogue geometry
    const int set = warp >> 2;
    const int slot = (warp & 3) * 32 + lane;
    const uint32_t tmem_lane = tmem_base + ((uint32_t)((warp & 3) * 32) << 16);
    const int sj = (slot >= 2) ? (slot - 2) / kSlotStride : 0;
    const int sy = (slot >= 2) ? (slot - 2) % kSlotStride : 40;
    if (warp < kEpiWarps) {   // the accumulator ring starts zeroed: every MMA accumulates
        for (int r = set; r < G::kSlots; r += kSets)
#pragma unroll
            for (int ch = 0; ch < F / 16; ++ch) tmem_st16_zero(tmem_lane + (uint32_t)(r * F + 16 * ch));
        tmem_wait_st();
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    }
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

    // running stream positions (every role counts the same sequence)
    int q = 0;          // column stream: unit * 10 + c, for input columns and output columns alike
    int wl = 0;         // layer stream
    int crc[2] = {0, 0};  // completions of col_ready consumed (copy warp) per lane
    const float* const head = a.consts + (size_t)(L + 1) * 3 * F;

    while (true) {
        if (tid == 0) s_pair = atomicAdd(a.counters, 1);
        __syncthreads();
        const int pair = s_pair;
        if (pair >= n_pairs) break;
        const int g0 = 2 * pair;
        const int nl = (g0 + 1 < n_groups) ? 2 : 1;

        if (warp == kWarpCopy) {
            // ============ copy warp: weights and input columns (one thread) ============
            if (lane == 0) {
                for (int l = 0; l < L; ++l, ++wl) {
                    if (l == 0) {   // first layer of the pair: its buffer was released by the previous pair's layer L-2
                        mbar_wait(w_free(wl & 1), ((wl >> 1) & 1) ^ 1, kTagWFree, wl, status);
                        mbar_expect_tx(w_full(wl & 1), G::kWLayerBytes);
                        bulk_g2s(smem_u32(smem + (wl & 1) * G::kWLayerBytes), reinterpret_cast<const uint8_t*>(a.w_packed) + (size_t)l * G::kWLayerBytes,
                                 G::kWLayerBytes, w_full(wl & 1));
                    }
                    const int in_buf = POST ? (l & 1) : 1;
                    for (int ln = 0; ln < nl; ++ln) {
                        const uint8_t* src = scratch + ln * G::kLaneBytes + in_buf * G::kBufBytes;
                        for (int c = 0; c < 10; ++c, ++q) {
                            mbar_wait(col_ready(ln, c), crc[ln] & 1, kTagColReady, q, status);
                            const int k = q % G::kRing;
                            mbar_wait(in_free(k), ((q / G::kRing) & 1) ^ 1, kTagInFree, q, status);
                            mbar_expect_tx(in_full(k), G::kColBytes);
                            bulk_g2s(smem_u32(smem + G::kOffIn + k * G::kColBytes), src + c * G::kColBytes, G::kColBytes, in_full(k));
                            if (ln == 0 && c == G::kRing && l + 1 < L) {
                                // the MMAs of column 0 of this layer have retired (its ring slot was just re-used), hence all
                                // of layer l-1: the other weight buffer is free -> prefetch layer l+1
                                const int nw = wl + 1;
                                mbar_wait(w_free(nw & 1), ((nw >> 1) & 1) ^ 1, kTagWFree, nw, status);
                                mbar_expect_tx(w_full(nw & 1), G::kWLayerBytes);
                                bulk_g2s(smem_u32(smem + (nw & 1) * G::kWLayerBytes),
                                         reinterpret_cast<const uint8_t*>(a.w_packed) + (size_t)(l + 1) * G::kWLayerBytes, G::kWLayerBytes, w_full(nw & 1));
                            }
                        }
                        ++crc[ln];
                    }
                }
            }
            __syncwarp();
        } else if (warp == kWarpMma) {
            // ============ MMA issuer (warp-uniform; elect.sync inside umma / umma_commit) ============
            const uint64_t ad = umma_desc(smem_u32(smem + G::kOffIn), kPlaneBytes, 128u);
            const uint32_t a_lo0 = (uint32_t)ad, a_hi = (uint32_t)(ad >> 32);
            const uint64_t bd = umma_desc(smem_u32(smem), G::kLbo, 128u);
            const uint32_t b_lo0 = (uint32_t)bd, b_hi = (uint32_t)(bd >> 32);
            for (int l = 0; l < L; ++l, ++wl) {
                mbar_wait(w_full(wl & 1), (wl >> 1) & 1, kTagWFull, wl, status);
                const uint32_t b_lo = b_lo0 + (uint32_t)((wl & 1) * (G::kWLayerBytes / 16));
                for (int ln = 0; ln < nl; ++ln) {
                    for (int c = 0; c < 10; ++c, ++q) {
                        const int k = q % G::kRing;
                        mbar_wait(in_full(k), (q / G::kRing) & 1, kTagInFull, q, status);
                        // output slots touched for the first time: they must have been drained and re-zeroed
                        if (c == 0) mbar_wait(out_free(q % G::kSlots), ((q / G::kSlots) & 1) ^ 1, kTagOutFree, q, status);
                        if (c < 9) mbar_wait(out_free((q + 1) % G::kSlots), (((q + 1) / G::kSlots) & 1) ^ 1, kTagOutFree, q + 1, status);
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                        // outputs j = 0..2 -> output columns q-1+j; the run of ring slots may wrap once
                        const int j_lo = (c == 0) ? 1 : 0, j_hi = (c == 9) ? 1 : 2;
                        const int s_lo = (q - 1 + j_lo) % G::kSlots;
                        const int n_j = j_hi - j_lo + 1;
                        const int n_first = min(n_j, G::kSlots - s_lo);      // slots before the wrap
                        const uint32_t a_col = a_lo0 + (uint32_t)(k * (G::kColBytes / 16));
#pragma unroll
                        for (int dy = 0; dy < 3; ++dy) {
#pragma unroll
                            for (int t = 0; t < G::kKSteps; ++t) {
                                const uint32_t aa = a_col + (uint32_t)(t * 2 * (kPlaneBytes / 16) + dy);
                                const uint32_t bb = b_lo + (uint32_t)(dy * (G::kWDyBytes / 16) + t * 2 * (G::kLbo / 16) + j_lo * (F / 8) * 8);
                                umma(tmem_base + (uint32_t)(s_lo * F), aa, a_hi, bb, b_hi, idesc((uint32_t)(n_first * F)));
                                if (n_first < n_j)
                                    umma(tmem_base, aa, a_hi, bb + (uint32_t)(n_first * (F / 8) * 8), b_hi, idesc((uint32_t)((n_j - n_first) * F)));
                            }
                        }
                        umma_commit(in_free(k));
                        if (c >= 1) umma_commit(out_done((q - 1) % G::kSlots));
                        if (c == 9) umma_commit(out_done(q % G::kSlots));
                    }
                }
                umma_commit(w_free(wl & 1));
            }
            __syncwarp();
        } else {
            // ============ epilogue warps: stem, then the output columns of every layer ============
            bool inside[2];
            int img[2];
#pragma unroll
            for (int ln = 0; ln < 2; ++ln) {
                img[ln] = (g0 + ln) * kImgs + sj;
                inside[ln] = ln < nl && sy < 40 && sj < kImgs && img[ln] < n_images;
            }
            // ---- stem: thread = board row; every set computes the columns c = set (mod 4) ----
            for (int ln = 0; ln < nl; ++ln) {
                uint32_t m[5] = {0u, 0u, 0u, 0u, 0u};   // bit x + 2 = cell x of board row sy + dy - taps / 2
                const int taps = a.stem_taps, half = taps >> 1;
                if (inside[ln]) {
                    for (int dy = 0; dy < taps; ++dy) {
                        const int yy = sy + dy - half;
                        if (yy < 0 || yy >= 40) continue;
                        const uint32_t* src = reinterpret_cast<const uint32_t*>(a.grids + ((size_t)img[ln] * 400 + yy * 10));
                        uint32_t bits = 0u;
#pragma unroll
                        for (int w = 0; w < 5; ++w) {
                            const uint32_t v = src[w];
                            bits |= ((v & 0x7FFFu) ? 1u : 0u) << (2 * w) | ((v & 0x7FFF0000u) ? 1u : 0u) << (2 * w + 1);
                        }
                        m[dy] = bits << 2;
                    }
                }
                uint8_t* bx = scratch + ln * G::kLaneBytes;          // X
                uint8_t* bt = bx + G::kBufBytes;                     // T/U
                const float* c0 = a.consts;                          // slot 0: stem bias, next scale, next bias
                for (int c = set; c < 10; c += kSets) {
                    const int sh = c + 2 - half;
#pragma unroll
                    for (int ch = 0; ch < F / 16; ++ch) {
                        float acc[16];
#pragma unroll
                        for (int i = 0; i < 16; ++i) acc[i] = 0.f;
                        for (int dy = 0; dy < taps; ++dy) {
                            const uint32_t pat = (m[dy] >> sh) & ((1u << taps) - 1u);
                            const float4* lp = reinterpret_cast<const float4*>(a.stem_lut + ((size_t)(dy << taps) + pat) * F + 16 * ch);
#pragma unroll
                            for (int v4 = 0; v4 < 4; ++v4) {
                                const float4 v = __ldg(lp + v4);
                                acc[4 * v4] += v.x; acc[4 * v4 + 1] += v.y; acc[4 * v4 + 2] += v.z; acc[4 * v4 + 3] += v.w;
                            }
                        }
                        float k0[16], k1[16], t[16];
                        const size_t off = ((size_t)(c * G::kKc + 2 * ch) * kRowsBuf + slot + 1) * 16;
                        if (POST) {      // X0 = relu(bn(conv)) (scale folded into the table)
                            load16g(c0 + 16 * ch, k0);
#pragma unroll
                            for (int i = 0; i < 16; ++i) t[i] = inside[ln] ? acc[i] + k0[i] : 0.f;
                            store16<true>(bx + off, t);
                        } else {         // X0 = conv;  T0 = relu(bn1_0(X0))
                            load16g(c0 + F + 16 * ch, k0);
                            load16g(c0 + 2 * F + 16 * ch, k1);
#pragma unroll
                            for (int i = 0; i < 16; ++i) {
                                t[i] = inside[ln] ? fmaf(k0[i], acc[i], k1[i]) : 0.f;
                                acc[i] = inside[ln] ? acc[i] : 0.f;
                            }
                            store16<false>(bx + off, acc);
                            store16<true>(bt + off, t);
                        }
                    }
                    publish_global(col_ready(ln, c));
                }
            }
            // ---- layers ----
            // An output column is published (fence.proxy.async + arrival on col_ready) when this warp has been woken for
            // its NEXT column: by then the stores are old and the fence does not wait for them.  The next column's
            // out_done never depends on the pending publication (it needs inputs of earlier columns only).
            uint32_t pending_bar = 0u;
            for (int l = 0; l < L; ++l) {
                const bool conv2 = (l & 1) != 0;
                const bool last = (l == L - 1);
                const float* cl = a.consts + (size_t)(l + 1) * 3 * F;
                for (int ln = 0; ln < nl; ++ln) {
                    uint8_t* bx = scratch + ln * G::kLaneBytes;
                    uint8_t* bt = bx + G::kBufBytes;
                    for (int c = 0; c < 10; ++c, ++q) {
                        if ((q & (kSets - 1)) != set) continue;
                        const int r = q % G::kSlots;
                        const size_t off0 = ((size_t)(c * G::kKc) * kRowsBuf + slot + 1) * 16;
                        mbar_wait(out_done(r), (q / G::kSlots) & 1, kTagOutDone, q, status);
                        if (pending_bar) { publish_global(pending_bar); pending_bar = 0u; }
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                        float hacc[NOUT];
#pragma unroll
                        for (int o = 0; o < NOUT; ++o) hacc[o] = 0.f;
                        uint32_t acc_raw[2][16];     // two 16-channel chunks of the accumulator in flight per wait
#pragma unroll
                        for (int ch = 0; ch < F / 16; ++ch) {
                            const size_t off = off0 + (size_t)(2 * ch) * kPlaneBytes;
                            uint4 ra = make_uint4(0, 0, 0, 0), rb = ra;
                            if (conv2) {   // residual: this thread's own earlier write (or the stem's)
                                ra = __ldcg(reinterpret_cast<const uint4*>(bx + off));
                                rb = __ldcg(reinterpret_cast<const uint4*>(bx + off + kPlaneBytes));
                            }
                            float d[16], kb[16];
                            const uint32_t ta = tmem_lane + (uint32_t)(r * F + 16 * ch);
                            if (!(ch & 1)) {
                                tmem_ld16_issue(ta, acc_raw[0]);
                                tmem_ld16_issue(ta + 16u, acc_raw[1]);
                                tmem_wait_ld();
                                tmem_st16_zero(ta);
                                tmem_st16_zero(ta + 16u);
                            }
#pragma unroll
                            for (int i = 0; i < 16; ++i) d[i] = __uint_as_float(acc_raw[ch & 1][i]);
                            load16g(cl + 16 * ch, kb);
#pragma unroll
                            for (int i = 0; i < 16; ++i) d[i] += kb[i];
                            if (conv2) {
                                d[0] += bf_lo(ra.x); d[1] += bf_hi(ra.x); d[2] += bf_lo(ra.y); d[3] += bf_hi(ra.y);
                                d[4] += bf_lo(ra.z); d[5] += bf_hi(ra.z); d[6] += bf_lo(ra.w); d[7] += bf_hi(ra.w);
                                d[8] += bf_lo(rb.x); d[9] += bf_hi(rb.x); d[10] += bf_lo(rb.y); d[11] += bf_hi(rb.y);
                                d[12] += bf_lo(rb.z); d[13] += bf_hi(rb.z); d[14] += bf_lo(rb.w); d[15] += bf_hi(rb.w);
                            }
                            if (!inside[ln]) {
#pragma unroll
                                for (int i = 0; i < 16; ++i) d[i] = 0.f;
                            }
                            float t[16];
                            if (!POST && conv2) {
                                // X' = X + conv2(U);  T' = relu(bn_next(X'))
                                float ks[16];
                                load16g(cl + F + 16 * ch, ks);
                                load16g(cl + 2 * F + 16 * ch, kb);
#pragma unroll
                                for (int i = 0; i < 16; ++i) t[i] = inside[ln] ? fmaxf(fmaf(ks[i], d[i], kb[i]), 0.f) : 0.f;
                                if (!last) {
                                    store16<false>(bx + off, d);
                                    store16<true>(bt + off, t);
                                }
                            } else {
#pragma unroll
                                for (int i = 0; i < 16; ++i) t[i] = fmaxf(d[i], 0.f);
                                if (!last) store16<true>((conv2 ? bx : bt) + off, t);
                            }
                            if (last) {
#pragma unroll
                                for (int o = 0; o < NOUT; ++o) {
                                    float hw[16];
                                    load16g(head + o * F + 16 * ch, hw);
#pragma unroll
                                    for (int i = 0; i < 16; ++i) hacc[o] = fmaf(hw[i], t[i], hacc[o]);
                                }
                            }
                        }
                        tmem_wait_st();
                        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                        __syncwarp();
                        if (lane == 0) mbar_arrive(out_free(r));
                        if (!last) {
                            pending_bar = col_ready(ln, c);
                        } else if (inside[ln]) {
                            const int orow = a.out_row ? a.out_row[img[ln]] : img[ln];
#pragma unroll
                            for (int o = 0; o < NOUT; ++o) {
                                float v = fmaf(__ldg(head + NOUT * F + o), hacc[o], __ldg(head + NOUT * F + NOUT + o));
                                if (!POST || o == NOUT - 1) v = fmaxf(v, 0.f);
                                a.out[((size_t)orow * NOUT + o) * 400 + sy * 10 + c] = __float2bfloat16(v);
                            }
                        }
                    }
                }
            }
            if (pending_bar) publish_global(pending_bar);   // (none is left: the last layer publishes nothing)
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        }
        __syncthreads();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    }

    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == kWarpMma) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"(kTmemCols));
    }
    if (tid == 0) {   // the last CTA leaves the counters at zero for the next launch on this slot
        __threadfence();
        if (atomicAdd(a.counters + 1, 1) == (int)gridDim.x - 1) {
            a.counters[0] = 0;
            a.counters[1] = 0;
            a.counters[2] = 0;
            if (a.n_images_dev) *a.n_images_dev = 0;
            __threadfence();
        }
    }
}

int* next_counter() {
    static int slot = 0;
    int* base = (int*)trl_workspace(TRL_WS_TRUNK_COUNTER_WIDE, 64 * 64);
    if (!base) return nullptr;
    int* c = base + 16 * slot;
    slot = (slot + 1) & 63;
    return c;
}

// The activation scratch (two buffers per group, 0.7 MB per CTA at 64 filters: 97 MB for 148 CTAs) is meant to live in
// L2, but under the default policy 70 % of its traffic went to DRAM (ncu: 12.4 GB per 4096-board launch).  The launch
// therefore carries an access-policy window over the scratch: as much of it as the device lets a context pin
// (persistingL2CacheMaxSize) is marked persisting, the rest streaming.  g_wide_l2_window = 0 switches it off (A/B).
int g_wide_l2_window = 1;

template <int F, bool POST>
int launch(const WideArgs& a, int grid, cudaStream_t stream, bool pdl) {
    int rc = trl_check(cudaFuncSetAttribute(trunk_wide_kernel<F, POST>, cudaFuncAttributeMaxDynamicSharedMemorySize, Geo<F>::kSmem));
    if (rc) return rc;
    // the persisting-L2 limit is set, and its size probed, once per device
    static size_t persist_of[TRL_MAX_DEVICES] = {}, window_of[TRL_MAX_DEVICES] = {};
    static bool probed[TRL_MAX_DEVICES] = {};
    const int dev = trl_device();
    if (dev < 0) return TRL_E_CUDA;
    if (!probed[dev]) {
        probed[dev] = true;
        int pmax = 0, wmax = 0;
        if (cudaDeviceGetAttribute(&pmax, cudaDevAttrMaxPersistingL2CacheSize, dev) == cudaSuccess &&
            cudaDeviceGetAttribute(&wmax, cudaDevAttrMaxAccessPolicyWindowSize, dev) == cudaSuccess && pmax > 0 && wmax > 0 &&
            cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, (size_t)pmax) == cudaSuccess) {
            persist_of[dev] = (size_t)pmax;
            window_of[dev] = (size_t)wmax;
        }
        cudaGetLastError();
    }
    const size_t persist_bytes = persist_of[dev], window_max = window_of[dev];
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(kThreads); cfg.dynamicSmemBytes = (size_t)Geo<F>::kSmem; cfg.stream = stream;
    cudaLaunchAttribute attr[3];
    unsigned n = 0;
    if (pdl && g_trl_pdl) {
        attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[n].val.programmaticStreamSerializationAllowed = 1;
        ++n;
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        attr[n].id = cudaLaunchAttributePriority;
        attr[n].val.priority = hi;
        ++n;
    }
    if (g_wide_l2_window && persist_bytes) {
        size_t bytes = (size_t)grid * 2 * Geo<F>::kLaneBytes;     // the part of the scratch this launch uses
        if (bytes > window_max) bytes = window_max;
        attr[n].id = cudaLaunchAttributeAccessPolicyWindow;
        attr[n].val.accessPolicyWindow.base_ptr = a.scratch;
        attr[n].val.accessPolicyWindow.num_bytes = bytes;
        attr[n].val.accessPolicyWindow.hitRatio = bytes <= persist_bytes ? 1.0f : (float)((double)persist_bytes / (double)bytes);
        attr[n].val.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        attr[n].val.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
        ++n;
    }
    cfg.attrs = attr; cfg.numAttrs = n;
    return trl_check(cudaLaunchKernelEx(&cfg, trunk_wide_kernel<F, POST>, a));
}

}  // namespace

extern "C" void trl_debug_trunk_wide_l2_window(int on) { g_wide_l2_window = on ? 1 : 0; }

extern "C" long long trl_trunk_wide_scratch_bytes(int filters) {
    if (filters != 32 && filters != 64) return 0;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long lane = filters == 64 ? Geo<64>::kLaneBytes : Geo<32>::kLaneBytes;
    return (long long)sms * 2 * lane;
}

extern "C" int trl_trunk_wide(const void* grids_bf16, int n_images, int32_t* n_images_dev, const int32_t* out_row,
                              int filters, int n_blocks, int post_act, int stem_taps, const void* w_packed,
                              const float* consts, const float* stem_lut, void* out_bf16, void* scratch,
                              long long scratch_bytes, int32_t* status, int pdl, void* stream) {
    if (n_images < 0 || n_blocks < 1 || (filters != 32 && filters != 64) || (stem_taps != 3 && stem_taps != 5) || !grids_bf16 ||
        !w_packed || !consts || !stem_lut || !out_bf16 || !scratch || !status || (n_images_dev && !out_row))
        return TRL_E_ARG;
    if (scratch_bytes < trl_trunk_wide_scratch_bytes(filters)) return TRL_E_ARG;
    if (n_images == 0) return TRL_OK;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int n_pairs = ((n_images + kImgs - 1) / kImgs + 1) / 2;
    const int grid = sms < n_pairs ? sms : n_pairs;
    WideArgs a;
    a.grids = (const __nv_bfloat16*)grids_bf16; a.n_images = n_images; a.n_blocks = n_blocks; a.stem_taps = stem_taps; a.pad_ = 0;
    a.n_images_dev = n_images_dev; a.out_row = out_row; a.w_packed = (const uint4*)w_packed; a.consts = consts;
    a.stem_lut = stem_lut; a.out = (__nv_bfloat16*)out_bf16; a.scratch = (uint8_t*)scratch; a.status = status;
    a.counters = next_counter();
    if (!a.counters) return TRL_E_NOMEM;
    cudaStream_t st = (cudaStream_t)stream;
    if (filters == 64) return post_act ? launch<64, true>(a, grid, st, pdl != 0) : launch<64, false>(a, grid, st, pdl != 0);
    return post_act ? launch<32, true>(a, grid, st, pdl != 0) : launch<32, false>(a, grid, st, pdl != 0);
}
