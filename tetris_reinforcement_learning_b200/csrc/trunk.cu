// trunk.cu — fused convolutional trunk of AlphaSame (filters = 16, kernels = 1) on the
// 5th-generation tensor cores: tcgen05.mma with TMEM accumulators, activations resident in
// shared memory across all 2*blocks convolutions of an image.
//
// Replaces AlphaSame.process_grid (reference architectures.py:120-126): conv1 5x5 (1->16) ->
// blocks x [BN-ReLU-Conv3x3, BN-ReLU-Conv3x3, +skip] -> BN-ReLU -> Conv1x1 (16->1) -> BN-ReLU ->
// flatten(400), eval mode (BatchNorm folded to per-channel scale/bias on the host).
//
// Mapping (one CTA = 8 warps = one image at a time, persistent over images, 4 CTAs per SM):
//   * An image is kept as a zero-haloed 42 x 12 grid of "pixels"; pixel p = (y+1)*12 + (x+1).
//     An activation buffer holds two planes [pixel][8 channels] bf16 (16 B per pixel per plane):
//     this IS the canonical K-major no-swizzle UMMA operand layout (8 consecutive pixels x 16 B =
//     one 128 B core matrix), so the im2col view of tap (dy,dx) is just the same buffer with the
//     descriptor start address moved by (12*dy + dx) pixels.  No im2col copy exists.
//   * A 3x3 convolution of one image = 4 M-tiles (128 pixels each, p in [13, 525)) x 9 taps of
//     tcgen05.mma M=128 N=16 K=16 (bf16 x bf16 -> fp32 in TMEM), issued by one thread;
//     accumulators: 4 tiles x 16 TMEM columns.
//   * The residual stream X lives in TMEM in fp32 for the whole network: the second convolution
//     of a block accumulates straight onto it (accumulate flag on from the first tap), so the
//     skip connection costs nothing.  The first convolution writes separate TMEM columns.
//   * Epilogue: warp w owns accumulator rows 32*(w&3).. of tiles 2*(w>>2), +1; a thread reads the
//     16 channels of its pixel (tcgen05.ld 32x32b.x16), applies bias / BN / ReLU and rewrites the
//     operand buffer IN PLACE (all MMAs of the layer have completed) in the same layout.
//   * The binary 5x5 stem is a table lookup: per kernel row, the 5 input bits select a
//     precomputed 16-channel partial sum (5 x 32 x 16 floats).
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "trl_common.cuh"

namespace {

constexpr int kThreads = 256;                 // 8 warps: warp w owns TMEM lanes 32*(w&3).. and tiles 2*(w>>2), +1
constexpr int kCtasPerSm = 4;                 // TMEM: 4 x 128 columns; registers: 4 x 256 x 64
constexpr int kPadW = 12;                     // 10 columns + 1 halo each side
constexpr int kFirstPixel = 13;               // (y=0, x=0)
constexpr int kBufPixels = 544;               // >= 4*128 + 2*12 + 2 + 1, multiple of 8
constexpr int kPlaneBytes = kBufPixels * 16;  // 8704
constexpr int kActBytes = 2 * kPlaneBytes;    // 17408: two 8-channel planes
constexpr int kWLayerBytes = 9 * 512;         // 9 taps x (16 x 16 bf16)
constexpr int kLutFloats = 5 * 32 * 16;
constexpr int kTmemCols = 128;                // X: 4 tiles x 16 fp32 columns, D1: 4 x 16
constexpr int kColX = 0, kColD = 64;
constexpr int kMaxBlocks = 20;

// shared memory carve-up (bytes)
constexpr int kOffAct = 0;                            // ONE operand buffer, rewritten in place
constexpr int kOffW = kOffAct + kActBytes;            // double buffered
constexpr int kOffLut = kOffW + 2 * kWLayerBytes;
constexpr int kOffConst = kOffLut + kLutFloats * 4;   // per block 48 floats + 50 final
constexpr int kOffRows = kOffConst + (kMaxBlocks * 48 + 64) * 4;
constexpr int kOffBar = kOffRows + 48 * 4;
constexpr int kSmemBytes = kOffBar + 16;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// K-major, SWIZZLE_NONE shared-memory matrix descriptor (cute::UMMA::SmemDescriptor):
// start>>4 [0,14) | LBO>>4 [16,30) (stride between the two 8-element K chunks) |
// SBO>>4 [32,46) (stride between 8-row core matrices) | version=1 [46,48) | layout NONE [61,64)
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}

// cute::UMMA::InstrDescriptor for kind::f16: D=f32, A=B=bf16, K-major both, N=16, M=128
constexpr uint32_t kIdesc = (1u << 4) | (1u << 7) | (1u << 10) | ((16u >> 3) << 17) | ((128u >> 4) << 24);

__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a, uint64_t b, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}\n"
        :: "r"(d_tmem), "l"(a), "l"(b), "r"(kIdesc), "r"(accumulate), "r"(0u) : "memory");
}

__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(bar) : "memory");
}

__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred q;\n\tWAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 q, [%0], %1;\n\t"
        "@q bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}\n" :: "r"(bar), "r"(parity) : "memory");
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
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};\n\t"
        "tcgen05.wait::st.sync.aligned;\n"
        :: "r"(taddr), "r"(__float_as_uint(d[0])), "r"(__float_as_uint(d[1])), "r"(__float_as_uint(d[2])),
           "r"(__float_as_uint(d[3])), "r"(__float_as_uint(d[4])), "r"(__float_as_uint(d[5])), "r"(__float_as_uint(d[6])),
           "r"(__float_as_uint(d[7])), "r"(__float_as_uint(d[8])), "r"(__float_as_uint(d[9])), "r"(__float_as_uint(d[10])),
           "r"(__float_as_uint(d[11])), "r"(__float_as_uint(d[12])), "r"(__float_as_uint(d[13])), "r"(__float_as_uint(d[14])),
           "r"(__float_as_uint(d[15])) : "memory");
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}

// write the 16 channels of pixel p into the operand buffer (two 16-byte stores, one per plane)
__device__ __forceinline__ void store_pixel(uint8_t* buf, int p, const float (&v)[16]) {
    uint4 a, b;
    a.x = pack_bf16x2(v[0], v[1]);   a.y = pack_bf16x2(v[2], v[3]);
    a.z = pack_bf16x2(v[4], v[5]);   a.w = pack_bf16x2(v[6], v[7]);
    b.x = pack_bf16x2(v[8], v[9]);   b.y = pack_bf16x2(v[10], v[11]);
    b.z = pack_bf16x2(v[12], v[13]); b.w = pack_bf16x2(v[14], v[15]);
    *reinterpret_cast<uint4*>(buf + (size_t)p * 16) = a;
    *reinterpret_cast<uint4*>(buf + kPlaneBytes + (size_t)p * 16) = b;
}

// 36 MMAs of one 3x3 convolution over the 4 M-tiles of an image.
//   first conv of a block : D1[tile]  = sum_taps A(tap, tile) * W(tap)     (overwrite)
//   second conv           : X[tile]  += sum_taps A(tap, tile) * W(tap)     (the residual add is free)
__device__ __forceinline__ void issue_conv(uint32_t act_saddr, uint32_t w_saddr, uint32_t tmem_dst, bool onto_x,
                                           uint32_t bar) {
#pragma unroll
    for (int m = 0; m < 4; ++m) {
#pragma unroll
        for (int tap = 0; tap < 9; ++tap) {
            const int dy = tap / 3, dx = tap % 3;
            const uint64_t a = umma_desc(act_saddr + (uint32_t)(128 * m + kPadW * dy + dx) * 16u, kPlaneBytes, 128u);
            const uint64_t b = umma_desc(w_saddr + (uint32_t)tap * 512u, 256u, 128u);
            umma_bf16(tmem_dst + (uint32_t)(m * 16), a, b, (tap > 0 || onto_x) ? 1u : 0u);
        }
    }
    umma_commit(bar);
}

__global__ void __launch_bounds__(kThreads, kCtasPerSm)
alphasame_trunk_kernel(const __nv_bfloat16* __restrict__ grids, int n_images, int n_blocks,
                       const uint4* __restrict__ w_packed,   // [2*n_blocks][9*512 B]
                       const float* __restrict__ consts,     // [n_blocks*48 + 50]
                       const float* __restrict__ stem_lut,   // [5][32][16]
                       __nv_bfloat16* __restrict__ out,      // [n_images][400]
                       int* __restrict__ next_image) {       // work counter (zeroed before launch)
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint32_t s_tmem_base;
    __shared__ int s_img;
    const int tid = threadIdx.x, warp = tid >> 5;
    uint8_t* act = smem + kOffAct;
    float* s_lut = reinterpret_cast<float*>(smem + kOffLut);
    float* s_const = reinterpret_cast<float*>(smem + kOffConst);
    uint32_t* s_rows = reinterpret_cast<uint32_t*>(smem + kOffRows);
    const uint32_t bar = smem_u32(smem + kOffBar);
    const int n_layers = 2 * n_blocks;

    // ---- one-time setup ----
    for (int i = tid; i < kActBytes / 16; i += kThreads) reinterpret_cast<uint4*>(act)[i] = make_uint4(0, 0, 0, 0);
    for (int i = tid; i < kLutFloats; i += kThreads) s_lut[i] = stem_lut[i];
    for (int i = tid; i < n_blocks * 48 + 50; i += kThreads) s_const[i] = consts[i];
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(bar));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(&s_tmem_base)), "r"(kTmemCols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = s_tmem_base;
    const uint32_t tmem_lane = tmem_base + ((uint32_t)((warp & 3) * 32) << 16);
    const int tile0 = (warp >> 2) * 2;   // this warp's two tiles
    const int row = tid & 127;           // accumulator row (= TMEM lane) of this thread

    uint32_t phase = 0;
    // Images are handed out dynamically: a CTA that becomes resident late (e.g. while another
    // kernel shares the GPU) simply takes fewer images instead of delaying the whole launch.
    while (true) {
        if (tid == 0) s_img = atomicAdd(next_image, 1);
        if (tid < 48) s_rows[tid] = 0;
        __syncthreads();
        const int img = s_img;
        if (img >= n_images) break;
        // ---- input: 400 bf16 {0,1} -> bit rows with a 2-cell border (for the 5x5 stem) ----
        const __nv_bfloat16* gin = grids + (size_t)img * 400;
        for (int c = tid; c < 400; c += kThreads) {
            if (__bfloat162float(gin[c]) != 0.f) atomicOr(&s_rows[c / 10 + 2], 1u << (c % 10 + 2));
        }
        for (int i = tid; i < kWLayerBytes / 16; i += kThreads)   // first layer's weights
            reinterpret_cast<uint4*>(smem + kOffW)[i] = w_packed[i];
        __syncthreads();

        // ---- stem: X = conv5x5(grid) by table lookup -> TMEM; operand = relu(bn1_0(X)) ----
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int m = tile0 + j;
            const int p = kFirstPixel + 128 * m + row;
            const int y = p / kPadW - 1, x = p % kPadW - 1;
            const bool inside = (y >= 0 && y < 40 && x >= 0 && x < 10);
            float xv[16], t[16];
#pragma unroll
            for (int c = 0; c < 16; ++c) { xv[c] = 0.f; t[c] = 0.f; }
            if (inside) {
#pragma unroll
                for (int r = 0; r < 5; ++r) {
                    const uint32_t pat = (s_rows[y + r] >> x) & 31u;
                    const float4* l = reinterpret_cast<const float4*>(s_lut + (r * 32 + pat) * 16);
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const float4 v = l[q];
                        xv[4 * q] += v.x; xv[4 * q + 1] += v.y; xv[4 * q + 2] += v.z; xv[4 * q + 3] += v.w;
                    }
                }
#pragma unroll
                for (int c = 0; c < 16; ++c) t[c] = fmaxf(fmaf(s_const[c], xv[c], s_const[16 + c]), 0.f);
            }
            tmem_st16(tmem_lane + (uint32_t)(kColX + m * 16), xv);
            store_pixel(act, p, t);
        }

        // ---- 2 * n_blocks convolutions ----
        for (int layer = 0; layer < n_layers; ++layer) {
            const bool second = layer & 1;
            const uint32_t wbuf = smem_u32(smem + kOffW + (layer & 1) * kWLayerBytes);
            // operand writes (generic proxy) -> visible to the tensor core (async proxy);
            // TMEM reads/writes of the previous phase ordered before the MMAs
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncthreads();
            if (tid == 0) {
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                issue_conv(smem_u32(act), wbuf, tmem_base + (second ? kColX : kColD), second, bar);
            }
            // prefetch the next layer's weights into the other buffer while the MMAs run
            if (layer + 1 < n_layers) {
                const uint4* wn = w_packed + (size_t)(layer + 1) * (kWLayerBytes / 16);
                uint4* wd = reinterpret_cast<uint4*>(smem + kOffW + ((layer + 1) & 1) * kWLayerBytes);
                for (int i = tid; i < kWLayerBytes / 16; i += kThreads) wd[i] = wn[i];
            }
            mbar_wait(bar, phase);
            phase ^= 1u;
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

            // all MMAs of this layer are complete: the operand buffer may be rewritten in place
            const float* cb = s_const + (layer >> 1) * 48;
            const bool last = (layer == n_layers - 1);
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int m = tile0 + j;
                const int p = kFirstPixel + 128 * m + row;
                const int y = p / kPadW - 1, x = p % kPadW - 1;
                const bool inside = (y >= 0 && y < 40 && x >= 0 && x < 10);
                float d[16], v[16];
                if (!second) {
                    // U = relu(conv1'(T) + c2)   (bn2 scale folded into the weights)
                    tmem_ld16(tmem_lane + (uint32_t)(kColD + m * 16), d);
#pragma unroll
                    for (int c = 0; c < 16; ++c) v[c] = inside ? fmaxf(d[c] + cb[32 + c], 0.f) : 0.f;
                    store_pixel(act, p, v);
                } else {
                    // X (in TMEM) already holds X + conv2(U); next operand T = relu(bn1_next(X))
                    tmem_ld16(tmem_lane + (uint32_t)(kColX + m * 16), d);
                    if (!last) {
                        const float* nb = cb + 48;
#pragma unroll
                        for (int c = 0; c < 16; ++c) v[c] = inside ? fmaxf(fmaf(nb[c], d[c], nb[16 + c]), 0.f) : 0.f;
                        store_pixel(act, p, v);
                    } else if (inside) {
                        // head of the trunk: BN-ReLU, 1x1 conv to one channel, BN-ReLU, flatten
                        const float* fc = s_const + n_blocks * 48;
                        float acc = 0.f;
#pragma unroll
                        for (int c = 0; c < 16; ++c) acc = fmaf(fc[32 + c], fmaxf(fmaf(fc[c], d[c], fc[16 + c]), 0.f), acc);
                        out[(size_t)img * 400 + y * 10 + x] = __float2bfloat16(fmaxf(fmaf(fc[48], acc, fc[49]), 0.f));
                    }
                }
            }
        }
        // the next image's stem overwrites X in TMEM: order this image's TMEM reads before it
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    }

    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"(kTmemCols));
    }
}

}  // namespace

extern "C" int trl_alphasame_trunk(const void* grids_bf16, int n_images, int n_blocks, const void* w_packed,
                                   const float* consts, const float* stem_lut, void* out_bf16, void* stream) {
    if (n_images < 0 || n_blocks < 1 || n_blocks > kMaxBlocks || !grids_bf16 || !w_packed || !consts || !stem_lut || !out_bf16)
        return TRL_E_ARG;
    if (n_images == 0) return TRL_OK;
    static bool configured[TRL_MAX_DEVICES] = {};   // the attribute is per device
    const int dev = trl_device();
    if (dev < 0) return TRL_E_CUDA;
    if (!configured[dev]) {
        int rc = trl_check(cudaFuncSetAttribute(alphasame_trunk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
        if (rc) return rc;
        configured[dev] = true;
    }
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    int grid = sms * kCtasPerSm;  // resident CTAs per SM (TMEM / register bound), persistent over images
    if (grid > n_images) grid = n_images;
    int* counter = (int*)trl_workspace(TRL_WS_TRUNK_COUNTER_TAPS, 256);
    if (!counter) return TRL_E_NOMEM;
    int rc = trl_check(cudaMemsetAsync(counter, 0, sizeof(int), (cudaStream_t)stream));
    if (rc) return rc;
    alphasame_trunk_kernel<<<grid, kThreads, kSmemBytes, (cudaStream_t)stream>>>(
        (const __nv_bfloat16*)grids_bf16, n_images, n_blocks, (const uint4*)w_packed, consts, stem_lut,
        (__nv_bfloat16*)out_bf16, counter);
    return trl_check(cudaGetLastError());
}
