// heads.cu — everything between the convolutional trunk and the policy GEMM of AlphaSame, fused.
//
// Replaces, in eval mode, the tail of AlphaSame.forward (reference architectures.py:128-142):
//   o16   = ReLU(BN1d(Linear(400 -> 16)(opponent trunk features)))            (osidedense)
//   x     = cat[own trunk features 400, own side 52, o16, opponent side 52, colour 1]   (521, padded to 528)
//   value = Sigmoid|Tanh(Linear(16 -> 1)(ReLU(BN1d(Linear(521 -> 16)(x)))))   (value_head; dropout = identity)
// The policy head Linear(521 -> 11583) stays a library GEMM on x (it is GEMM shaped: 50 GFLOP per
// 4096-leaf step).  One warp per four leaves; lanes = (k mod 8, output quad): a lane accumulates 4 outputs x
// 4 leaves over every eighth k (two LDS.128 feed 16 independent FMAs), a butterfly sums the eight k lanes.
// BatchNorm1d is folded into the linear layers on the host (trunk.py).
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "trl_common.cuh"

namespace {

constexpr int kFeat = 400, kSide = 52, kOpp = 16, kIn = 521, kPad = 528;
constexpr int kWarpsPerBlock = 8;    // x 4 leaves x 3.7 KB of staged inputs + 59 KB of weights per block
// packed weights (fp32): Wo_t[400][16], bo[16], Wv_t[528][16], bv[16], w2[16], b2
constexpr int kOffWo = 0, kOffBo = kOffWo + kFeat * 16, kOffWv = kOffBo + 16, kOffBv = kOffWv + kPad * 16,
              kOffW2 = kOffBv + 16, kOffB2 = kOffW2 + 16, kWFloats = kOffB2 + 4;

// kLeaves leaves per warp pass: the weight row of a k is loaded once and used for all of them
// (the kernel is bound by shared-memory loads: per k one weight word + one 16-byte vector of leaf inputs).
constexpr int kLeaves = 4;

__global__ void __launch_bounds__(kWarpsPerBlock * 32)
alphasame_heads_kernel(const __nv_bfloat16* __restrict__ feats,    // [2G][400]: own grids then opponent grids (or a cache)
                       const int32_t* __restrict__ own_row,        // optional: feature rows of leaf g (< 0: skip)
                       const int32_t* __restrict__ opp_row,
                       const __nv_bfloat16* __restrict__ extras,   // [G][105]
                       int G, const float* __restrict__ weights, int use_tanh,
                       __nv_bfloat16* __restrict__ x_out,          // [G][528]
                       __nv_bfloat16* __restrict__ value_out) {    // [G]
    extern __shared__ __align__(16) float sm[];
    float* w = sm;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    {   // weights -> shared memory with cp.async (no registers, all 15 16-byte copies of a thread in flight);
        // they are only waited for before the first dense layer, so the copy runs under the input gather
        constexpr int kVec = kWFloats / 4;
        static_assert(kWFloats % 4 == 0, "weights are copied in 16-byte pieces");
        const uint32_t dst = (uint32_t)__cvta_generic_to_shared(w);
        for (int i = tid; i < kVec; i += kWarpsPerBlock * 32)
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(dst + 16u * (uint32_t)i), "l"(weights + 4 * i) : "memory");
        asm volatile("cp.async.commit_group;" ::: "memory");
    }
    bool weights_ready = false;
    // per warp: xs[k][leaf] (528 x 4) and fo[k][leaf] (400 x 4), leaf-interleaved so one LDS.128 feeds 4 FMAs
    float4* xs = reinterpret_cast<float4*>(sm + kWFloats) + warp * (kPad + kFeat);
    float4* fo = xs + kPad;
    const int og = lane & 3, kk = lane >> 2;   // output quad 4og..4og+3, k = kk mod 8
    const int n_quads = (G + kLeaves - 1) / kLeaves;
    for (int q = blockIdx.x * kWarpsPerBlock + warp; q < n_quads; q += gridDim.x * kWarpsPerBlock) {
        int ra[kLeaves], rb[kLeaves];
        bool any = false;
#pragma unroll
        for (int j = 0; j < kLeaves; ++j) {
            const int g = q * kLeaves + j;
            ra[j] = (g < G) ? (own_row ? own_row[g] : g) : -1;
            rb[j] = (g < G) ? (own_row ? opp_row[g] : G + g) : -1;
            any = any || ra[j] >= 0;
        }
        // ---- stage: own features, side inputs, opponent features (zeros for skipped leaves) ----
        // all global loads of the pass are issued before the first use (the pass is latency bound otherwise)
        constexpr int kFI = (kFeat / 2 + 31) / 32;            // 7 bf16x2 words per lane and feature row
        constexpr int kEI = (2 * kSide + 1 + 31) / 32;        // 4 side inputs per lane
        uint32_t ua[kLeaves][kFI], ub[kLeaves][kFI];
        uint16_t ue[kLeaves][kEI];
#pragma unroll
        for (int j = 0; j < kLeaves; ++j) {
            const uint32_t* fa = reinterpret_cast<const uint32_t*>(feats + (size_t)(ra[j] < 0 ? 0 : ra[j]) * kFeat);
            const uint32_t* fb = reinterpret_cast<const uint32_t*>(feats + (size_t)(ra[j] < 0 ? 0 : rb[j]) * kFeat);
            const uint16_t* ex = reinterpret_cast<const uint16_t*>(extras + (size_t)(ra[j] < 0 ? 0 : q * kLeaves + j) * (2 * kSide + 1));
#pragma unroll
            for (int t = 0; t < kFI; ++t) {
                const int i = lane + 32 * t;
                const bool ok = ra[j] >= 0 && i < kFeat / 2;
                ua[j][t] = ok ? fa[i] : 0u;
                ub[j][t] = ok ? fb[i] : 0u;
            }
#pragma unroll
            for (int t = 0; t < kEI; ++t) {
                const int i = lane + 32 * t;
                ue[j][t] = (ra[j] >= 0 && i < 2 * kSide + 1) ? ex[i] : (uint16_t)0;
            }
        }
        if (!weights_ready) {
            // first pass of this warp (every thread of the block gets here exactly once, here or after the loop):
            // the gather above is in flight while the block's weights land
            asm volatile("cp.async.wait_group 0;" ::: "memory");
            __syncthreads();
            weights_ready = true;
        }
        if (!any) continue;   // warp-uniform
        // feature word i = features 2i, 2i+1 of all four leaves -> two float4 rows per tensor (STS.128)
#pragma unroll
        for (int t = 0; t < kFI; ++t) {
            const int i = lane + 32 * t;
            if (i < kFeat / 2) {
                float2 a[kLeaves], b[kLeaves];
#pragma unroll
                for (int j = 0; j < kLeaves; ++j) {
                    a[j] = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&ua[j][t]));
                    b[j] = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&ub[j][t]));
                }
                xs[2 * i] = make_float4(a[0].x, a[1].x, a[2].x, a[3].x);
                xs[2 * i + 1] = make_float4(a[0].y, a[1].y, a[2].y, a[3].y);
                fo[2 * i] = make_float4(b[0].x, b[1].x, b[2].x, b[3].x);
                fo[2 * i + 1] = make_float4(b[0].y, b[1].y, b[2].y, b[3].y);
            }
        }
#pragma unroll
        for (int t = 0; t < kEI; ++t) {
            const int i = lane + 32 * t;
            if (i < 2 * kSide + 1)
                xs[kFeat + i + (i >= kSide ? kOpp : 0)] =
                    make_float4(__bfloat162float(__ushort_as_bfloat16(ue[0][t])), __bfloat162float(__ushort_as_bfloat16(ue[1][t])),
                                __bfloat162float(__ushort_as_bfloat16(ue[2][t])), __bfloat162float(__ushort_as_bfloat16(ue[3][t])));
        }
        if (lane < kOpp) xs[kFeat + kSide + lane] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (lane < kPad - kIn) xs[kIn + lane] = make_float4(0.f, 0.f, 0.f, 0.f);
        __syncwarp();
        // ---- osidedense: 16 outputs x 400 for 4 leaves; lanes = (k mod 8, output quad) ----
        // per k one LDS.128 of weights (4 outputs) and one LDS.128 of inputs (4 leaves) feed 16 independent FMAs;
        // 50 / 66 iterations per layer instead of 200 / 264, then a 3-step butterfly over the k lanes
        float acc[4][kLeaves];
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int j = 0; j < kLeaves; ++j) acc[a][j] = 0.f;
#pragma unroll 2
        for (int k = kk; k < kFeat; k += 8) {
            const float4 wk = *reinterpret_cast<const float4*>(&w[kOffWo + k * 16 + 4 * og]);
            const float4 f = fo[k];
            const float wv4[4] = {wk.x, wk.y, wk.z, wk.w}, fv[4] = {f.x, f.y, f.z, f.w};
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int j = 0; j < kLeaves; ++j) acc[a][j] = fmaf(fv[j], wv4[a], acc[a][j]);
        }
#pragma unroll
        for (int d = 4; d <= 16; d <<= 1)
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int j = 0; j < kLeaves; ++j) acc[a][j] += __shfl_xor_sync(0xffffffffu, acc[a][j], d);
        if (kk == 0) {   // rounded like the module's bf16 output
#pragma unroll
            for (int a = 0; a < 4; ++a) {
                const float bo = w[kOffBo + 4 * og + a];
                xs[kFeat + kSide + 4 * og + a] = make_float4(__bfloat162float(__float2bfloat16(fmaxf(acc[a][0] + bo, 0.f))),
                                                             __bfloat162float(__float2bfloat16(fmaxf(acc[a][1] + bo, 0.f))),
                                                             __bfloat162float(__float2bfloat16(fmaxf(acc[a][2] + bo, 0.f))),
                                                             __bfloat162float(__float2bfloat16(fmaxf(acc[a][3] + bo, 0.f))));
            }
        }
        __syncwarp();
        // ---- x out (bf16, 528 wide) ----
        for (int i = lane; i < kPad / 2; i += 32) {
            const float4 e = xs[2 * i], o4 = xs[2 * i + 1];
            const float ev[kLeaves] = {e.x, e.y, e.z, e.w}, ov[kLeaves] = {o4.x, o4.y, o4.z, o4.w};
#pragma unroll
            for (int j = 0; j < kLeaves; ++j)
                if (ra[j] >= 0)
                    reinterpret_cast<__nv_bfloat162*>(x_out + (size_t)(q * kLeaves + j) * kPad)[i] = __floats2bfloat162_rn(ev[j], ov[j]);
        }
        // ---- value head ----
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int j = 0; j < kLeaves; ++j) acc[a][j] = 0.f;
#pragma unroll 2
        for (int k = kk; k < kPad; k += 8) {
            const float4 wk = *reinterpret_cast<const float4*>(&w[kOffWv + k * 16 + 4 * og]);
            const float4 f = xs[k];
            const float wv4[4] = {wk.x, wk.y, wk.z, wk.w}, fv[4] = {f.x, f.y, f.z, f.w};
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int j = 0; j < kLeaves; ++j) acc[a][j] = fmaf(fv[j], wv4[a], acc[a][j]);
        }
#pragma unroll
        for (int d = 4; d <= 16; d <<= 1)
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int j = 0; j < kLeaves; ++j) acc[a][j] += __shfl_xor_sync(0xffffffffu, acc[a][j], d);
        float v[kLeaves];
#pragma unroll
        for (int j = 0; j < kLeaves; ++j) {
            v[j] = 0.f;
#pragma unroll
            for (int a = 0; a < 4; ++a) v[j] = fmaf(fmaxf(acc[a][j] + w[kOffBv + 4 * og + a], 0.f), w[kOffW2 + 4 * og + a], v[j]);
            v[j] += __shfl_xor_sync(0xffffffffu, v[j], 1);
            v[j] += __shfl_xor_sync(0xffffffffu, v[j], 2);
            v[j] += w[kOffB2];
            if (lane == 0 && ra[j] >= 0)
                value_out[q * kLeaves + j] = __float2bfloat16(use_tanh ? tanhf(v[j]) : 1.f / (1.f + __expf(-v[j])));
        }
        __syncwarp();
    }
    if (!weights_ready) {   // a warp without a pass still owes the block its barrier arrival
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();
    }
}

}  // namespace

extern "C" int trl_alphasame_heads_weight_floats(void) { return kWFloats; }

static int launch_heads(const void* feats_bf16, const int32_t* own_row, const int32_t* opp_row, const void* extras_bf16,
                        int n_leaves, const float* weights, int use_tanh, void* x_out_bf16, void* value_out_bf16,
                        void* stream) {
    if (n_leaves < 0 || !feats_bf16 || !extras_bf16 || !weights || !x_out_bf16 || !value_out_bf16) return TRL_E_ARG;
    if (n_leaves == 0) return TRL_OK;
    const int smem = (kWFloats + kWarpsPerBlock * kLeaves * (kPad + kFeat)) * 4;
    static bool configured[TRL_MAX_DEVICES] = {};   // the attribute is per device
    const int dev = trl_device();
    if (dev < 0) return TRL_E_CUDA;
    if (!configured[dev]) {
        int rc = trl_check(cudaFuncSetAttribute(alphasame_heads_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        if (rc) return rc;
        configured[dev] = true;
    }
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    int blocks = ((n_leaves + kLeaves - 1) / kLeaves + kWarpsPerBlock - 1) / kWarpsPerBlock;
    if (blocks > sms) blocks = sms;
    return trl_launch_ex(alphasame_heads_kernel, dim3(blocks), dim3(kWarpsPerBlock * 32), (size_t)smem, (cudaStream_t)stream, false, false,
                         (const __nv_bfloat16*)feats_bf16, own_row, opp_row, (const __nv_bfloat16*)extras_bf16, n_leaves, weights,
                         use_tanh, (__nv_bfloat16*)x_out_bf16, (__nv_bfloat16*)value_out_bf16);
}

extern "C" int trl_alphasame_heads(const void* feats_bf16, const void* extras_bf16, int n_leaves, const float* weights,
                                   int use_tanh, void* x_out_bf16, void* value_out_bf16, void* stream) {
    return launch_heads(feats_bf16, nullptr, nullptr, extras_bf16, n_leaves, weights, use_tanh, x_out_bf16, value_out_bf16, stream);
}

extern "C" int trl_alphasame_heads_indexed(const void* cache_bf16, const int32_t* own_row, const int32_t* opp_row,
                                           const void* extras_bf16, int n_leaves, const float* weights, int use_tanh,
                                           void* x_out_bf16, void* value_out_bf16, void* stream) {
    if (!own_row || !opp_row) return TRL_E_ARG;
    return launch_heads(cache_bf16, own_row, opp_row, extras_bf16, n_leaves, weights, use_tanh, x_out_bf16, value_out_bf16, stream);
}
