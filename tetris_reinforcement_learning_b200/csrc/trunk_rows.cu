// trunk_rows.cu — fused convolutional trunk of AlphaSame (filters = 16, kernels = 1), third
// formulation: ROW-TOEPLITZ implicit GEMM on tcgen05 with a column-wavefront software pipeline.
//
// Replaces AlphaSame.process_grid (reference architectures.py:120-126, ResidualBlock :27-57) in
// eval mode: conv5x5 (1->16) -> blocks x [BN-ReLU-Conv3x3, BN-ReLU-Conv3x3, +skip] -> BN-ReLU ->
// Conv1x1 (16->1) -> BN-ReLU -> flatten(400).  BatchNorm is folded on the host (trunk.py).
//
// Why a third formulation.  With M = pixels, N = 16 output channels and one MMA per 3x3 tap
// (trunk.cu) every activation byte is fetched from shared memory NINE times by the tensor core and
// the kernel sits on the 128 B/clk/SM shared-memory operand bandwidth (measured with
// tools/ubench/umma_rate.cu: M128 N16 K16 SS costs 36 clk of operand fetch against an 8 clk math
// floor).  Here an MMA row is a BOARD ROW and the horizontal taps are folded into N:
//
//     D[row r, (x_out, oc)] += A[row r + dy - 1, (x_in, ic)] * B_dy[(x_out - x_in + 1, oc), ic]
//
// For one input column x_in the three output columns x_in-1, x_in, x_in+1 are adjacent accumulator
// columns, so ONE tcgen05.mma M=128 N=48 K=16 per (x_in, dy) does the work of three taps for 128
// board rows; the B matrix (48 x 16) does not depend on x_in.  Operand fetch per image and
// convolution drops from 9 to 3 reads of the activations (432 clk instead of 1296 clk at 128 B/clk).
//
// Mapping (one persistent CTA per SM, 21 warps):
//   * group = 3 images = 128 MMA rows ("slots"): image j row y -> slot 2 + 42 j + y, two zero halo
//     slots around every image (2 + 40 + 2 + 40 + 2 + 40 + 2 = 128).  TMEM lane = slot.
//   * operand buffer in shared memory: [x_in 10][k half 2][row 136] x 16 B (8 channels bf16);
//     slot s lives at row s+1, so the vertical tap dy is the same buffer with the UMMA descriptor
//     start moved by dy rows (no im2col copy).  This is the canonical K-major no-swizzle layout.
//   * TMEM: X (fp32 residual stream) columns [0,160) = (x_out, oc); D1 columns [160,320).  The
//     second convolution of a block accumulates straight onto X (free skip connection); D1 is
//     zeroed by the epilogue after it is read so every MMA accumulates.
//   * the MMA warp (warp-uniform code, elect.sync) issues the MMAs column by column and commits one
//     mbarrier per column; 20 epilogue warps (5 sets x 128 lanes, set p owns columns 2p, 2p+1)
//     turn finished accumulator columns into the next layer's operand columns IN PLACE and signal
//     them back: the tensor pipe starts layer L+1 on column 0 while the epilogue still drains L.
//   * the binary 5x5 stem is 5 more MMAs (M=128 N=160 K=16: K = the 14 board columns incl. halo).
//   * all 2*blocks weight matrices stay resident in shared memory for the CTA's lifetime.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "trl_common.cuh"

namespace {

constexpr int kEpiWarps = 20;                    // 5 sets x 4 warps; set p owns the column pair (2p, 2p+1)
constexpr int kEpiThreads = kEpiWarps * 32;      // 640
constexpr int kThreads = kEpiThreads + 32;       // + the MMA warp
constexpr int kImgs = 3;                         // images per group
constexpr int kSlotStride = 42;                  // 40 rows + two halo slots (the 5x5 stem needs two)
constexpr int kRowsBuf = 136;                    // operand rows per plane
constexpr int kPlaneBytes = kRowsBuf * 16;       // 2176
constexpr int kColBytes = 2 * kPlaneBytes;       // 4352: one x_in column, two 8-channel planes
constexpr int kActBytes = 10 * kColBytes;        // 43520  (slot s -> row s + 1)
constexpr int kStemInBytes = kColBytes;          // 4352: board cells as a K=16 operand (slot s -> row s + 2)
constexpr int kStemWDyBytes = 160 * 16 * 2;      // 5120: Toeplitz matrix of one stem kernel row
constexpr int kStemWBytes = 5 * kStemWDyBytes;   // 25600
constexpr int kWDyBytes = 48 * 16 * 2;           // 1536: B matrix of one vertical tap
constexpr int kWLayerBytes = 3 * kWDyBytes;      // 4608
constexpr int kTmemCols = 512;
constexpr int kColX = 0, kColD = 320;            // X of lane 0 / lane 1 at columns 0 / 160, shared D1 at 320
constexpr int kMaxBlocks = 16;                   // resident weights: 32 x 4608 B (one lane); two lanes up to 11 blocks
constexpr int kBarsPerLane = 16;                 // I, M[10], O[5]
constexpr int kSmemLimit = 232448 - 1024;

// shared-memory bytes for n_lanes image groups in flight
__host__ __device__ inline int smem_bytes(int n_blocks, int n_lanes) {
    return n_lanes * (kActBytes + kStemInBytes) + kStemWBytes + 2 * kBarsPerLane * 8 +
           ((n_blocks * 48 + 50 + 3) / 4) * 16 + 2 * n_blocks * kWLayerBytes;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// K-major, SWIZZLE_NONE shared-memory matrix descriptor: start>>4 [0,14) | LBO>>4 [16,30) (stride
// between the two 8-element K chunks) | SBO>>4 [32,46) (stride between 8-row core matrices) | version 1
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}

// kind::f16 instruction descriptor: D = f32, A = B = bf16, both K-major, M = 128
__host__ __device__ constexpr uint32_t idesc(uint32_t n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((n >> 3) << 17) | ((128u >> 4) << 24);
}

// D[tmem] += A[smem] * B[smem], executed by the WHOLE (converged) MMA warp: elect.sync picks the
// issuing lane inside the asm, so every operand stays warp-uniform and ptxas keeps descriptors,
// addresses and the loop in uniform registers (back-to-back UTCHMMA, no per-lane replay loop).
// The descriptors are passed as (lo, hi) words: the start-address field is the low 14 bits, so
// moving an operand is one 32-bit add.
__device__ __forceinline__ void umma(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                     uint32_t id, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p, e;\n\t.reg .b64 da, db;\n\telect.sync _|e, 0xffffffff;\n\t"
        "mov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\tsetp.ne.b32 p, %6, 0;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, {%7, %7, %7, %7}, p;\n\t}\n"
        :: "r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(id), "r"(accumulate), "r"(0u) : "memory");
}

__device__ __forceinline__ void umma_commit(uint32_t bar) {   // whole warp, one elected lane commits
    asm volatile(
        "{\n\t.reg .pred e;\n\telect.sync _|e, 0xffffffff;\n\t"
        "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}\n" :: "r"(bar) : "memory");
}

__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 q, [%0], %1;\n\t"   // usually already complete: no suspend
        "@q bra DONE_%=;\n\tWAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 q, [%0], %1;\n\t"
        "@q bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}\n" :: "r"(bar), "r"(parity) : "memory");
}

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(bar) : "memory");
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

__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float (&d)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};\n"
        :: "r"(taddr), "r"(__float_as_uint(d[0])), "r"(__float_as_uint(d[1])), "r"(__float_as_uint(d[2])),
           "r"(__float_as_uint(d[3])), "r"(__float_as_uint(d[4])), "r"(__float_as_uint(d[5])), "r"(__float_as_uint(d[6])),
           "r"(__float_as_uint(d[7])), "r"(__float_as_uint(d[8])), "r"(__float_as_uint(d[9])), "r"(__float_as_uint(d[10])),
           "r"(__float_as_uint(d[11])), "r"(__float_as_uint(d[12])), "r"(__float_as_uint(d[13])), "r"(__float_as_uint(d[14])),
           "r"(__float_as_uint(d[15])) : "memory");
}

__device__ __forceinline__ void tmem_st16_zero(uint32_t taddr) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1};\n"
        :: "r"(taddr), "r"(0u) : "memory");
}

__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// relu + round to bf16 of two floats in ONE instruction (F2FP.RELU.BF16.PACK_AB)
__device__ __forceinline__ uint32_t pack_relu_bf16x2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}

// relu(v[0..16)) of (column x, slot) -> two 16-byte stores (one per 8-channel plane)
__device__ __forceinline__ void store_operand_relu(uint8_t* act, int x, int slot, const float (&v)[16]) {
    uint4 a, b;
    a.x = pack_relu_bf16x2(v[0], v[1]);   a.y = pack_relu_bf16x2(v[2], v[3]);
    a.z = pack_relu_bf16x2(v[4], v[5]);   a.w = pack_relu_bf16x2(v[6], v[7]);
    b.x = pack_relu_bf16x2(v[8], v[9]);   b.y = pack_relu_bf16x2(v[10], v[11]);
    b.z = pack_relu_bf16x2(v[12], v[13]); b.w = pack_relu_bf16x2(v[14], v[15]);
    uint8_t* p = act + x * kColBytes + (slot + 1) * 16;
    *reinterpret_cast<uint4*>(p) = a;
    *reinterpret_cast<uint4*>(p + kPlaneBytes) = b;
}

// operand column written (generic proxy) -> visible to the tensor core (async proxy); TMEM traffic
// of this thread ordered before the hand-off; one arrival per warp.
__device__ __forceinline__ void publish_column(uint32_t bar_o) {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncwarp();
    if ((threadIdx.x & 31) == 0) mbar_arrive(bar_o);
}

// 16 per-channel constants of the running layer in registers (shared-memory bandwidth belongs to
// the tensor core: at the operand-fetch bound every LDS in the epilogue is a stolen MMA cycle).
__device__ __forceinline__ void load16(const float* p, float (&r)[16]) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const float4 v = reinterpret_cast<const float4*>(p)[q];
        r[4 * q] = v.x; r[4 * q + 1] = v.y; r[4 * q + 2] = v.z; r[4 * q + 3] = v.w;
    }
}

// Folded BatchNorm constants travel as a by-value kernel parameter: they are warp-uniform, so they
// come through the constant bank (LDC/ULDC) and cost no shared-memory bandwidth.
struct TrunkConsts { float v[kMaxBlocks * 48 + 52]; };

__device__ __forceinline__ void load16c(const float* p, float (&r)[16]) {
#pragma unroll
    for (int q = 0; q < 16; ++q) r[q] = p[q];
}

__global__ void __launch_bounds__(kThreads, 1)
alphasame_trunk_rows_kernel(const __nv_bfloat16* __restrict__ grids, int n_images, int n_blocks, int n_lanes,
                            const uint4* __restrict__ w_packed,   // [2*n_blocks][3][2][6][8][8] bf16
                            const __grid_constant__ TrunkConsts consts,   // [n_blocks*48 + 50]
                            const uint4* __restrict__ stem_w,     // [5][2][20][8][8] bf16
                            __nv_bfloat16* __restrict__ out,      // [n_images][400]
                            int* __restrict__ next_group,         // [0] work counter, [1] finished CTAs; both zero on entry,
                                                                  // re-zeroed by the last CTA (no memset node per launch)
                            int* __restrict__ n_images_dev,       // optional: device-side image count (<= n_images); reset to 0 at the end
                            const int* __restrict__ out_row,      // optional: output row of image k (default k)
                            long long* __restrict__ trace) {      // optional [pseudo-layer][column][4] clock stamps (CTA 0, first group, lane 0)
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint32_t s_tmem_base;
    __shared__ int s_group;
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // provably warp-uniform
    const int n_layers = 2 * n_blocks;
    // shared memory: per lane [operand buffer | stem input], then stem weights, barriers, constants, weights
    const int lane_bytes = kActBytes + kStemInBytes;
    const int off_stem_w = n_lanes * lane_bytes, off_bar = off_stem_w + kStemWBytes, off_const = off_bar + 2 * kBarsPerLane * 8;
    const int off_w = off_const + ((n_blocks * 48 + 50 + 3) / 4) * 16;
    const float* s_const = consts.v;
    // per lane: I (cells staged), M[10] (MMAs of input column c complete), O[5] (operand columns 2p, 2p+1 written)
    const uint32_t bars = smem_u32(smem + off_bar);
    if (tid == 0) atomicAdd(next_group + 2, 1);   // resident CTAs (trl_alphasame_trunk_rows_gate polls this)

    // ---- one-time setup ----
    for (int i = tid; i < n_lanes * lane_bytes / 16; i += kThreads) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
    for (int i = tid; i < kStemWBytes / 16; i += kThreads) reinterpret_cast<uint4*>(smem + off_stem_w)[i] = stem_w[i];
    for (int i = tid; i < n_layers * (kWLayerBytes / 16); i += kThreads)
        reinterpret_cast<uint4*>(smem + off_w)[i] = w_packed[i];
    if (tid == 0) {
        for (int ln = 0; ln < 2; ++ln) {
            const uint32_t b = bars + ln * kBarsPerLane * 8;
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 4;" :: "r"(b));
            for (int c = 0; c < 10; ++c) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(b + 8 + 8 * c));
            for (int c = 0; c < 5; ++c) asm volatile("mbarrier.init.shared::cta.b64 [%0], 4;" :: "r"(b + 88 + 8 * c));
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == kEpiWarps) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(&s_tmem_base)), "r"(kTmemCols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, s_tmem_base, 0);
    // Everything above (weights, barriers, TMEM) is independent of the kernel before this one in the stream:
    // with a programmatic dependent launch it overlapped that kernel's tail.  Its outputs (image list, count)
    // are read only from here on.
    trl_grid_dep_wait();
    if (n_images_dev) n_images = min(n_images, *n_images_dev);
    const int n_groups = (n_images + kImgs - 1) / kImgs;

    // epilogue thread geometry: slot = MMA row = TMEM lane; image j row y lives in slot 2 + 42 j + y
    const int set = warp >> 2;                              // owns columns 2*set, 2*set + 1
    const int slot = (warp & 3) * 32 + lane;
    const uint32_t tmem_lane = tmem_base + ((uint32_t)((warp & 3) * 32) << 16);
    const int sj = (slot >= 2) ? (slot - 2) / kSlotStride : 0;
    const int sy = (slot >= 2) ? (slot - 2) % kSlotStride : 40;     // 40, 41: halo
    if (warp < kEpiWarps) {   // D1 starts zeroed: every MMA of a first convolution accumulates
        tmem_st16_zero(tmem_lane + (uint32_t)(kColD + 32 * set));
        tmem_st16_zero(tmem_lane + (uint32_t)(kColD + 32 * set + 16));
        tmem_wait_st();
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    }

    // running mbarrier parities per lane (every barrier of a lane completes once per pseudo-layer of that lane)
    uint32_t ph_i[2] = {0, 0}, ph[2] = {0, 0};
    int group_iter = 0;
    while (true) {
        if (tid == 0) s_group = atomicAdd(next_group, n_lanes);
        __syncthreads();
        const int g0 = s_group;
        if (g0 >= n_groups) break;
        // lane ln works on group g0 + ln; the two lanes alternate layer by layer on the tensor pipe, so the
        // epilogue of one lane's layer overlaps the MMAs of the other lane's layer
        const bool act1 = (n_lanes > 1) && (g0 + 1 < n_groups);
        const bool first_group = (group_iter++ == 0);

        if (warp == kEpiWarps) {
            // ============ MMA issuer (warp-uniform; elect.sync inside umma / umma_commit) ============
            const uint64_t bd = umma_desc(smem_u32(smem + off_w), 768u, 128u);
            const uint32_t b_hi = (uint32_t)(bd >> 32);
            uint32_t b_lo = (uint32_t)bd;
            const uint64_t sb = umma_desc(smem_u32(smem + off_stem_w), 20u * 128u, 128u);
#pragma unroll
            for (int ln = 0; ln < 2; ++ln) {
                if (ln == 1 && !act1) break;
                // stem: X = conv5x5(cells) as 5 MMAs M=128 N=160 K=16 (K = 14 board columns incl. halo)
                const uint32_t lb = bars + ln * kBarsPerLane * 8;
                const uint64_t sa = umma_desc(smem_u32(smem + ln * lane_bytes + kActBytes), kPlaneBytes, 128u);
                mbar_wait(lb, ph_i[ln]);
                ph_i[ln] ^= 1u;
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                if (trace && blockIdx.x == 0 && first_group && lane == 0 && ln == 0) trace[0] = clock64();
#pragma unroll
                for (int dy = 0; dy < 5; ++dy)
                    umma(tmem_base + (uint32_t)(kColX + 160 * ln), (uint32_t)sa + (uint32_t)dy, (uint32_t)(sa >> 32),
                         (uint32_t)sb + (uint32_t)(dy * (kStemWDyBytes / 16)), (uint32_t)(sb >> 32), idesc(160), dy > 0 ? 1u : 0u);
#pragma unroll
                for (int c = 0; c < 10; ++c) umma_commit(lb + 8 + 8 * c);
            }
            for (int layer = 0; layer < n_layers; ++layer, b_lo += kWLayerBytes / 16) {
                const bool first_conv = !(layer & 1);
#pragma unroll
                for (int ln = 0; ln < 2; ++ln) {
                    if (ln == 1 && !act1) break;
                    const uint32_t lb = bars + ln * kBarsPerLane * 8;
                    const uint64_t ad = umma_desc(smem_u32(smem + ln * lane_bytes), kPlaneBytes, 128u);
                    const uint32_t a_lo = (uint32_t)ad, a_hi = (uint32_t)(ad >> 32);
                    const uint32_t dst = tmem_base + (first_conv ? kColD : (uint32_t)(kColX + 160 * ln));
#pragma unroll
                    for (int c = 0; c < 10; ++c) {
                        if (!(c & 1)) mbar_wait(lb + 88 + 8 * (c >> 1), ph[ln]);
                        // D1 is shared by the lanes: lane 1's first convolution follows lane 0's, so its MMAs on
                        // columns c-1..c+1 wait until lane 0's epilogue has drained (and re-zeroed) them, i.e. until
                        // lane 0 has published the operand pair holding column c+1 for ITS next layer
                        if (first_conv && ln == 1) mbar_wait(bars + 88 + 8 * ((c < 9 ? c + 1 : 9) >> 1), ph[0]);
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                        if (trace && blockIdx.x == 0 && first_group && lane == 0 && ln == 0) trace[((layer + 1) * 10 + c) * 4] = clock64();
#pragma unroll
                        for (int dy = 0; dy < 3; ++dy) {
                            const uint32_t a = a_lo + (uint32_t)(c * (kColBytes / 16) + dy);   // column c, rows shifted by dy
                            const uint32_t b = b_lo + (uint32_t)(dy * (kWDyBytes / 16));
                            if (c == 0)        // x_out = 0, 1 (skip the x_out = -1 rows of B)
                                umma(dst, a, a_hi, b + 16u, b_hi, idesc(32), 1u);
                            else if (c == 9)   // x_out = 8, 9
                                umma(dst + 128u, a, a_hi, b, b_hi, idesc(32), 1u);
                            else
                                umma(dst + (uint32_t)(16 * (c - 1)), a, a_hi, b, b_hi, idesc(48), 1u);
                        }
                        umma_commit(lb + 8 + 8 * c);
                    }
                    ph[ln] ^= 1u;
                }
            }
            __syncwarp();
        } else {
            // ============ input staging, epilogues ============
            bool inside[2];
#pragma unroll
            for (int ln = 0; ln < 2; ++ln)
                inside[ln] = (ln == 0 || act1) && sy < 40 && sj < kImgs && (g0 + ln) * kImgs + sj < n_images;
            if (set < 2 && (set == 0 || act1)) {
                // set `ln` stages lane ln: board cells of this slot's row as one K=16 operand row, k = x + 2
                const int ln = set;
                uint32_t cells[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) cells[q] = 0u;
                if (inside[ln]) {
                    const uint32_t* src = reinterpret_cast<const uint32_t*>(grids + ((size_t)((g0 + ln) * kImgs + sj) * 400 + sy * 10));
#pragma unroll
                    for (int q = 0; q < 5; ++q) cells[q + 1] = src[q];   // 10 bf16 cells = 5 words, k = 2..11
                }
                uint8_t* p = smem + ln * lane_bytes + kActBytes + (slot + 2) * 16;
                *reinterpret_cast<uint4*>(p) = make_uint4(cells[0], cells[1], cells[2], cells[3]);
                *reinterpret_cast<uint4*>(p + kPlaneBytes) = make_uint4(cells[4], cells[5], cells[6], cells[7]);
                publish_column(bars + ln * kBarsPerLane * 8);
            }

            // pseudo-layer 0 = stem, then the 2 * n_blocks convolutions, column pair by column pair behind the tensor pipe
            for (int pl = 0; pl <= n_layers; ++pl) {
                const int layer = pl - 1;
                const bool first_conv = (pl > 0) && !(layer & 1);
                const bool last = (layer == n_layers - 1);
#pragma unroll
                for (int ln = 0; ln < 2; ++ln) {
                    if (ln == 1 && !act1) break;
                    const uint32_t lb = bars + ln * kBarsPerLane * 8;
                    uint8_t* act = smem + ln * lane_bytes;
                    // next operand = relu(ka * acc + kb) per channel, with the halo mask folded into the
                    // constants (halo slots and missing images get ka = kb = 0 -> exact zeros)
                    float ka[16], kb[16];
                    if (first_conv) {
                        load16c(s_const + (layer >> 1) * 48 + 32, kb);             // bn2 bias (scale folded into the weights)
#pragma unroll
                        for (int c = 0; c < 16; ++c) ka[c] = 1.f;
                    } else if (!last) {
                        const float* nb = s_const + (pl == 0 ? 0 : (layer >> 1) + 1) * 48;
                        load16c(nb, ka);                                           // next block's bn1 scale, bias
                        load16c(nb + 16, kb);
                    } else {
                        const float* fc = s_const + n_blocks * 48;
                        load16c(fc, ka);
                        load16c(fc + 16, kb);
                    }
                    if (!inside[ln]) {
#pragma unroll
                        for (int c = 0; c < 16; ++c) { ka[c] = 0.f; kb[c] = 0.f; }
                    }
                    // columns 2p-1..2p+2 of this layer are final.  Only the set's first warp polls the mbarrier;
                    // the other three sleep on a hardware barrier.
                    if ((warp & 3) == 0) mbar_wait(lb + 8 + 8 * (set < 4 ? 2 * set + 2 : 9), ph[ln]);
                    asm volatile("bar.sync %0, 128;" :: "r"(1 + set) : "memory");
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const bool tr = trace && blockIdx.x == 0 && first_group && (tid & 127) == 0 && ln == 0;
                    if (tr) trace[(pl * 10 + 2 * set) * 4 + 1] = clock64();
                    const int orow = !inside[ln] ? 0 : (out_row ? out_row[(g0 + ln) * kImgs + sj] : (g0 + ln) * kImgs + sj);
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const int x = 2 * set + h;
                        float d[16], v[16];
                        const uint32_t ta = tmem_lane + (uint32_t)((first_conv ? kColD : kColX + 160 * ln) + 16 * x);
                        tmem_ld16(ta, d);
                        if (first_conv) tmem_st16_zero(ta);      // D1 is accumulate-only: leave it zeroed
                        if (!last) {
                            // first conv: U = relu(conv1'(T) + c2);  else T = relu(bn1_next(X)), X = stem / X + conv2(U)
#pragma unroll
                            for (int c = 0; c < 16; ++c) v[c] = fmaf(ka[c], d[c], kb[c]);
                            store_operand_relu(act, x, slot, v);
                        } else if (inside[ln]) {
                            // head of the trunk: BN-ReLU, 1x1 conv to one channel, BN-ReLU, flatten
                            const float* fc = s_const + n_blocks * 48;
                            float acc = 0.f;
#pragma unroll
                            for (int c = 0; c < 16; ++c) acc = fmaf(fc[32 + c], fmaxf(fmaf(ka[c], d[c], kb[c]), 0.f), acc);
                            out[(size_t)orow * 400 + sy * 10 + x] = __float2bfloat16(fmaxf(fmaf(fc[48], acc, fc[49]), 0.f));
                        }
                        if (tr && h == 0) trace[(pl * 10 + 2 * set) * 4 + 2] = clock64();
                    }
                    if (!last) {
                        if (first_conv) tmem_wait_st();
                        publish_column(lb + 88 + 8 * set);
                        if (tr) trace[(pl * 10 + 2 * set) * 4 + 3] = clock64();
                    }
                    ph[ln] ^= 1u;
                }
            }
            // the next group's stem overwrites X in TMEM: order this group's TMEM reads before it
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        }
        __syncthreads();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    }

    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == kEpiWarps) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"(kTmemCols));
    }
    if (tid == 0) {   // the last CTA to finish leaves the counters at zero for the next launch that uses this slot
        __threadfence();
        if (atomicAdd(next_group + 1, 1) == (int)gridDim.x - 1) {
            next_group[0] = 0;
            next_group[1] = 0;
            next_group[2] = 0;
            if (n_images_dev) *n_images_dev = 0;   // consumed: the next step's feature encoder appends from zero
            __threadfence();
        }
    }
}

// Holds a forked stream back until every CTA of a trunk launch is resident (or a time-out): one thread.
__global__ void trunk_gate_kernel(const int* __restrict__ counter, int expected, unsigned long long max_ns) {
    unsigned long long t0, t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    while (true) {
        int v;
        asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(counter + 2) : "memory");
        if (v >= expected) break;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        if (t - t0 > max_ns) break;
        __nanosleep(200);
    }
}

}  // namespace

extern "C" int trl_alphasame_trunk_rows_max_blocks(void) { return kMaxBlocks; }

// Two image groups in flight per CTA when the resident weights leave room for two operand buffers.
static int g_force_lanes = 0;
extern "C" void trl_debug_trunk_rows_lanes(int n_lanes) { g_force_lanes = n_lanes; }
static int lanes_for(int n_blocks) {
    const int fit = smem_bytes(n_blocks, 2) <= kSmemLimit ? 2 : 1;
    return (g_force_lanes == 1 || g_force_lanes == 2) ? (g_force_lanes < fit ? g_force_lanes : fit) : fit;
}

// Work counter of one launch.  Launches on different streams (two engines pipelined against each
// other) must not share a counter, so every launch takes the next of 64 slots.
static int* next_counter() {
    static int slot = 0;
    int* base = (int*)trl_workspace(TRL_WS_TRUNK_COUNTER, 64 * 64);
    if (!base) return nullptr;
    int* c = base + 16 * slot;
    slot = (slot + 1) & 63;
    return c;
}

// Profiling aid (tools/trunk_trace.py): device buffer of 2*n_blocks*10*4 int64 clock stamps written
// by CTA 0 for its first group; nullptr (default) disables tracing.
static long long* g_trace = nullptr;
extern "C" void trl_debug_trunk_rows_trace(void* device_buffer) { g_trace = (long long*)device_buffer; }

static TrunkConsts host_consts(const float* consts_host, int n_blocks) {
    TrunkConsts c;
    for (int i = 0; i < kMaxBlocks * 48 + 52; ++i) c.v[i] = (i < n_blocks * 48 + 50) ? consts_host[i] : 0.f;
    return c;
}

extern "C" int trl_alphasame_trunk_rows(const void* grids_bf16, int n_images, int n_blocks, const void* w_packed,
                                        const float* consts, const void* stem_w, void* out_bf16, void* stream) {
    if (n_images < 0 || n_blocks < 1 || n_blocks > kMaxBlocks || !grids_bf16 || !w_packed || !consts || !stem_w || !out_bf16)
        return TRL_E_ARG;
    if (n_images == 0) return TRL_OK;
    const int n_lanes = lanes_for(n_blocks);
    const int smem = smem_bytes(n_blocks, n_lanes);
    int rc0 = trl_check(cudaFuncSetAttribute(alphasame_trunk_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    if (rc0) return rc0;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int n_units = ((n_images + kImgs - 1) / kImgs + n_lanes - 1) / n_lanes;
    int grid = sms < n_units ? sms : n_units;   // one persistent CTA per SM (it owns all 512 TMEM columns)
    int* counter = next_counter();   // zero on entry: the previous launch on this slot reset it
    if (!counter) return TRL_E_NOMEM;
    alphasame_trunk_rows_kernel<<<grid, kThreads, smem, (cudaStream_t)stream>>>(
        (const __nv_bfloat16*)grids_bf16, n_images, n_blocks, n_lanes, (const uint4*)w_packed, host_consts(consts, n_blocks), (const uint4*)stem_w,
        (__nv_bfloat16*)out_bf16, counter, nullptr, nullptr, g_trace);
    return trl_check(cudaGetLastError());
}

// the most recent trl_alphasame_trunk_rows_indexed launch of each device
static int* g_last_counter[TRL_MAX_DEVICES] = {};
static int g_last_grid[TRL_MAX_DEVICES] = {};

// Work submitted to `stream` after this call starts only when all CTAs of the most recent
// trl_alphasame_trunk_rows_indexed launch on the current device are resident on their SMs (or after 100 us).
extern "C" int trl_alphasame_trunk_rows_gate(void* stream) {
    const int dev = trl_device();
    if (dev < 0) return TRL_E_CUDA;
    if (!g_last_counter[dev]) return TRL_E_ARG;
    trunk_gate_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(g_last_counter[dev], g_last_grid[dev], 100000ull);
    return trl_check(cudaGetLastError());
}

extern "C" int trl_alphasame_trunk_rows_indexed(const void* images_bf16, int32_t* n_images_dev, int max_images,
                                                const int32_t* out_row, int n_blocks, const void* w_packed,
                                                const float* consts, const void* stem_w, void* out_bf16, void* stream) {
    if (max_images < 0 || n_blocks < 1 || n_blocks > kMaxBlocks || !images_bf16 || !n_images_dev || !out_row || !w_packed ||
        !consts || !stem_w || !out_bf16)
        return TRL_E_ARG;
    if (max_images == 0) return TRL_OK;
    const int n_lanes = lanes_for(n_blocks);
    const int smem = smem_bytes(n_blocks, n_lanes);
    const int dev = trl_device();
    if (dev < 0) return TRL_E_CUDA;
    int rc = trl_check(cudaFuncSetAttribute(alphasame_trunk_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    if (rc) return rc;
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int n_units = ((max_images + kImgs - 1) / kImgs + n_lanes - 1) / n_lanes;
    const int grid = sms < n_units ? sms : n_units;
    int* counter = next_counter();   // zero on entry: the previous launch on this slot reset it
    if (!counter) return TRL_E_NOMEM;
    g_last_counter[dev] = counter;
    g_last_grid[dev] = grid;
    // Highest launch priority: inside a self-play step the leaf enumeration becomes ready at about the same
    // time on a forked stream, and its blocks must queue BEHIND the trunk's CTAs.  Programmatic dependent
    // launch: the CTAs move in and set themselves up while the search kernel before them drains.
    return trl_launch_ex(alphasame_trunk_rows_kernel, dim3(grid), dim3(kThreads), (size_t)smem, (cudaStream_t)stream, true, true,
                         (const __nv_bfloat16*)images_bf16, max_images, n_blocks, n_lanes, (const uint4*)w_packed,
                         host_consts(consts, n_blocks), (const uint4*)stem_w, (__nv_bfloat16*)out_bf16, counter, n_images_dev,
                         out_row, g_trace);
}
