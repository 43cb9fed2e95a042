// movegen_codes.cu — host movegen over shared boards with byte-coded move lists (trl_movegen_host_boards).
//
// The caller uploads each distinct board once and names the board of every call by index.  Per chunk of calls the
// sweep runs unchanged (trl_launch_movegen_warp, compact move-list mode) on boards gathered from that upload, and three
// small kernels turn its lists into the byte-coded lists of include/trl.h:
//     codes_count_kernel   one warp per call: escapes of the call; per tile of 256 calls an exclusive scan of
//                          (placements, escapes, flagged)
//     codes_scan_kernel    one block: exclusive scan of the tile totals, and the chunk totals
//     codes_write_kernel   one warp per call: codes and escapes at their call-ordered offsets, flagged calls
// Every call's bytes land at a place fixed by the counts of the calls before it, so the output does not depend on
// scheduling or on the chunking.  The encoder can also read the sweep's bit-packed masks instead (mask mode, a debug
// switch); on one B200 (1000 W) config 2 end to end took 45.0 ms per 7 M calls that way and 40.5 ms from the lists
// (DESIGN §5).
#include <cuda_runtime.h>
#include <stdint.h>

#include "trl_common.cuh"

int trl_launch_movegen_warp(const uint16_t* boards, const uint8_t* cur, const uint8_t* alt, const TrlGame* games,
                            const int32_t* index, int n, uint32_t* mask_bits, uint16_t* moves, int moves_cap,
                            uint16_t* n_moves, uint32_t* status, cudaStream_t stream, uint16_t* compact = nullptr,
                            unsigned long long compact_cap = 0, unsigned long long* compact_total = nullptr,
                            unsigned long long* offsets = nullptr);

namespace {

constexpr int kTile = 256;            // calls per scan tile = threads per block of the encoder kernels
constexpr int kTileWarps = kTile / 32;
constexpr int kCodesPerCall = 512;    // code staging per chunk: this many placements per call on average
constexpr int kMaxEscapes = TRL_POLICY_SIZE / 256;   // an escape spans >= 256 indices of the 11583: at most 45 per call
constexpr int kListPerCall = 160;     // move-list staging of the list-mode encoder (as trl_movegen_host_compact)

// chunk totals, copied back through pinned memory.  error: bit 0 a board index past the upload (gather), bit 1 a
// staging area too small for the chunk (scan)
struct CodeTotals { uint32_t codes, escapes, flagged, error; };

// Board of each call from the shared upload; an index past the upload is flagged and reads nothing.
__global__ void __launch_bounds__(256)
gather_boards_kernel(const uint4* __restrict__ all_boards, int n_boards, const uint32_t* __restrict__ board_index, int m,
                     uint4* __restrict__ boards, CodeTotals* __restrict__ tot) {
    static_assert(TRL_ROWS * 2 == 5 * sizeof(uint4), "a board is five 16-byte words");
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const uint32_t b = board_index[i];
    uint4 w[5] = {};
    if (b < (uint32_t)n_boards) {
#pragma unroll
        for (int k = 0; k < 5; ++k) w[k] = all_boards[(size_t)b * 5 + k];
    } else {
        tot->error = 1u;
    }
#pragma unroll
    for (int k = 0; k < 5; ++k) boards[(size_t)i * 5 + k] = w[k];
}

__device__ __forceinline__ int warp_max_incl(int v, int lane) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, v, d);
        if (lane >= d) v = max(v, t);
    }
    return v;
}

__device__ __forceinline__ int warp_sum_incl(int v, int lane) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, v, d);
        if (lane >= d) v += t;
    }
    return v;
}

// Mask mode: lane l owns the call's mask words 12l .. 12l+11, so its moves follow those of the lanes before it.  Within a
// lane the words are walked in registers; the move before a lane's first one is the highest set bit of the lanes
// before it, one warp max-scan per call.
constexpr int kWordsPerLane = 12;
static_assert(32 * kWordsPerLane >= TRL_MASK_WORDS, "a warp covers the mask");

struct LaneWords {
    uint32_t w[kWordsPerLane];
    int pos0;   // move index of bit 0 of w[0]
    int prev;   // the call's move before this lane's first one, -1 if none
};

__device__ __forceinline__ void load_lane_words(const uint32_t* __restrict__ mask, int lane, LaneWords& L) {
    const int w0 = lane * kWordsPerLane;
    int hi = -1;
#pragma unroll
    for (int k = 0; k < kWordsPerLane; ++k) L.w[k] = w0 + k < TRL_MASK_WORDS ? mask[w0 + k] : 0u;
#pragma unroll
    for (int k = 0; k < kWordsPerLane; ++k)
        if (L.w[k]) hi = (w0 + k) * 32 + 31 - __clz(L.w[k]);
    const int incl = warp_max_incl(hi, lane);
    const int before = __shfl_up_sync(0xffffffffu, incl, 1);
    L.pos0 = w0 * 32;
    L.prev = lane ? before : -1;
}

// Escapes of a lane's words: only the lowest move of a word can have a gap above 255.
__device__ __forceinline__ int lane_escapes(const LaneWords& L) {
    int esc = 0, p = L.prev;
#pragma unroll
    for (int k = 0; k < kWordsPerLane; ++k) {
        const uint32_t b = L.w[k];
        if (b) {
            esc += L.pos0 + k * 32 + __ffs(b) - 1 - p > 255;
            p = L.pos0 + k * 32 + 31 - __clz(b);
        }
    }
    return esc;
}

// List mode: the call's list in steps of 32 entries, lane l holding entry 32k + l with its previous move.
template <typename Emit>
__device__ __forceinline__ void walk_list(const uint16_t* __restrict__ list, int nm, int lane, Emit emit) {
    int carry = -1;   // last move of the steps before
#pragma unroll 1
    for (int base = 0; base < nm; base += 32) {
        const int j = base + lane;
        const int v = j < nm ? (int)list[j] : -1;
        int prev = __shfl_up_sync(0xffffffffu, v, 1);
        if (lane == 0) prev = carry;
        carry = __shfl_sync(0xffffffffu, v, 31);
        emit(v, prev);   // v < 0: no entry
    }
}

// Escapes of one call, summed over the warp.
template <bool FROM_LISTS>
__device__ __forceinline__ int call_escapes(const uint32_t* __restrict__ mask, const uint16_t* __restrict__ list, int nm,
                                            int lane) {
    int esc = 0;
    if (FROM_LISTS) {
        walk_list(list, nm, lane, [&](int v, int prev) { esc += v >= 0 && v - prev > 255; });
    } else {
        LaneWords L;
        load_lane_words(mask, lane, L);
        esc = lane_escapes(L);
    }
    return (int)__reduce_add_sync(0xffffffffu, (unsigned)esc);
}

constexpr int kCountWarps = 32;   // warps per block of codes_count_kernel: 8 calls of the tile each

template <bool FROM_LISTS>
__global__ void __launch_bounds__(kCountWarps * 32)
codes_count_kernel(const uint32_t* __restrict__ masks, const uint16_t* __restrict__ lists,
                   const unsigned long long* __restrict__ list_offs, const uint16_t* __restrict__ n_moves,
                   const uint32_t* __restrict__ status, int m, unsigned long long* __restrict__ local,
                   unsigned long long* __restrict__ tile_total) {
    __shared__ uint16_t s_esc[kTile];
    __shared__ unsigned long long s_warp[kTileWarps];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int tile0 = blockIdx.x * kTile;
    for (int j = warp; j < kTile; j += kCountWarps) {
        const int i = tile0 + j;
        int esc = 0;
        if (i < m) {
            const int nm = n_moves[i];
            if (nm && !(FROM_LISTS && (status[i] & TRL_ST_MOVES_TRUNC)))
                esc = call_escapes<FROM_LISTS>(masks + (size_t)i * TRL_MASK_WORDS, FROM_LISTS ? lists + list_offs[i] : nullptr,
                                               nm, lane);
        }
        if (lane == 0) s_esc[j] = (uint16_t)esc;
    }
    __syncthreads();
    // the tile's exclusive scan of (placements, escapes, flagged), packed 32 / 16 / 16 bits: a tile sums to < 2^24,
    // 256 * 45 and 256
    const int t = threadIdx.x, i = tile0 + t;
    unsigned long long v = 0, incl = 0;
    if (t < kTile) {
        if (i < m) v = (unsigned long long)n_moves[i] | ((unsigned long long)s_esc[t] << 32) |
                       ((unsigned long long)(status[i] != 0u) << 48);
        incl = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned long long u = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += u;
        }
        if (lane == 31) s_warp[warp] = incl;
    }
    __syncthreads();
    if (t < kTile) {
        unsigned long long before = 0;
        for (int k = 0; k < warp; ++k) before += s_warp[k];
        if (i < m) local[i] = before + incl - v;
        if (t == kTile - 1) tile_total[blockIdx.x] = before + incl;
    }
}

// One block: tile bases (codes, escapes, flagged) and the chunk totals.
__global__ void __launch_bounds__(1024)
codes_scan_kernel(const unsigned long long* __restrict__ tile_total, int n_tiles, uint4* __restrict__ tile_base,
                  CodeTotals* __restrict__ tot, uint32_t codes_cap, const unsigned long long* __restrict__ list_total,
                  unsigned long long list_cap) {
    __shared__ uint32_t s_warp[3][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t carry[3] = {0u, 0u, 0u};
    for (int lo = 0; lo < n_tiles; lo += 1024) {
        const int t = lo + threadIdx.x;
        const unsigned long long p = t < n_tiles ? tile_total[t] : 0ull;
        const uint32_t v[3] = {(uint32_t)p, (uint32_t)(p >> 32) & 0xffffu, (uint32_t)(p >> 48)};
        uint32_t incl[3];
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            incl[q] = (uint32_t)warp_sum_incl((int)v[q], lane);
            if (lane == 31) s_warp[q][warp] = incl[q];
        }
        __syncthreads();
        uint32_t out[3];
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            uint32_t before = carry[q];
            for (int k = 0; k < warp; ++k) before += s_warp[q][k];
            out[q] = before + incl[q] - v[q];
            for (int k = 0; k < 32; ++k) carry[q] += s_warp[q][k];
        }
        if (t < n_tiles) tile_base[t] = make_uint4(out[0], out[1], out[2], 0u);
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        tot->codes = carry[0];
        tot->escapes = carry[1];
        tot->flagged = carry[2];
        if (carry[0] > codes_cap || (list_total && *list_total > list_cap)) tot->error |= 2u;
    }
}

// Appends the gap d of one move: a byte, or byte 0 and an escape.
__device__ __forceinline__ void put_gap(int d, uint8_t*& out, uint16_t*& esc) {
    if (d > 255) {
        *esc++ = (uint16_t)d;
        *out++ = 0;
    } else {
        *out++ = (uint8_t)d;
    }
}

template <bool FROM_LISTS>
__global__ void __launch_bounds__(kTile)
codes_write_kernel(const uint32_t* __restrict__ masks, const uint16_t* __restrict__ lists,
                   const unsigned long long* __restrict__ list_offs, const uint16_t* __restrict__ n_moves,
                   const uint32_t* __restrict__ status, int m, int call_base, const unsigned long long* __restrict__ local,
                   const uint4* __restrict__ tile_base, const CodeTotals* __restrict__ tot, uint8_t* __restrict__ codes,
                   uint16_t* __restrict__ escapes, uint32_t* __restrict__ flag_index, uint32_t* __restrict__ flag_status) {
    const int lane = threadIdx.x & 31;
    const int i = blockIdx.x * kTileWarps + (threadIdx.x >> 5);
    if (i >= m) return;
    const uint4 tb = tile_base[i / kTile];
    const unsigned long long lp = local[i];
    const uint32_t flag_off = tb.z + (uint32_t)(lp >> 48);
    if (lane == 0 && status[i] != 0u) {
        flag_index[flag_off] = (uint32_t)(call_base + i);
        flag_status[flag_off] = status[i];
    }
    const int nm = n_moves[i];
    if (nm == 0 || tot->error) return;   // the host reports the error
    if (FROM_LISTS && (status[i] & TRL_ST_MOVES_TRUNC)) return;   // the list did not fit the staging: no list to read
    const uint32_t code_off = tb.x + (uint32_t)lp;
    const uint32_t esc_off = tb.y + ((uint32_t)(lp >> 32) & 0xffffu);
    if (FROM_LISTS) {
        uint8_t* out = codes + code_off + lane;
        uint16_t* esc = escapes + esc_off;
        walk_list(lists + list_offs[i], nm, lane, [&](int v, int prev) {
            const bool e = v >= 0 && v - prev > 255;
            const uint32_t eb = __ballot_sync(0xffffffffu, e);
            if (v >= 0) {
                *out = e ? 0 : (uint8_t)(v - prev);
                if (e) esc[__popc(eb & ((1u << lane) - 1u))] = (uint16_t)(v - prev);
            }
            out += 32;
            esc += __popc(eb);
        });
    } else {
        LaneWords L;
        load_lane_words(masks + (size_t)i * TRL_MASK_WORDS, lane, L);
        int cnt = 0;
#pragma unroll
        for (int k = 0; k < kWordsPerLane; ++k) cnt += __popc(L.w[k]);
        const int e = lane_escapes(L);
        uint8_t* out = codes + code_off + (warp_sum_incl(cnt, lane) - cnt);
        uint16_t* esc = escapes + esc_off + (warp_sum_incl(e, lane) - e);
        int p = L.prev;
#pragma unroll
        for (int k = 0; k < kWordsPerLane; ++k) {
            uint32_t b = L.w[k];
            while (b) {
                const int pos = L.pos0 + k * 32 + __ffs(b) - 1;
                b &= b - 1;
                put_gap(pos - p, out, esc);
                p = pos;
            }
        }
    }
}

}  // namespace

#ifndef TRL_HOST_CHUNK_LOG2
#define TRL_HOST_CHUNK_LOG2 17   // calls per staging chunk of the *_host entry points
#endif

// Encoder source of trl_movegen_host_boards: 0 = the sweep's compact move lists (default), 1 = its bit-packed masks.
// Both give the same bytes; tools/movegen_boards_bench.py times the two.
static int g_codes_source = 0;
extern "C" void trl_debug_movegen_codes_source(int source) { g_codes_source = source == 1 ? 1 : 0; }

extern "C" int trl_movegen_host_boards(const uint16_t* boards, int n_boards, const uint32_t* board_index,
                                       const uint8_t* cur, const uint8_t* alt, int n, uint8_t* codes, uint64_t codes_cap,
                                       uint16_t* escapes, uint64_t esc_cap, uint16_t* n_moves, uint32_t* flag_index,
                                       uint32_t* flag_status, uint64_t flag_cap, uint64_t* codes_total,
                                       uint64_t* esc_total, uint64_t* n_flagged) {
    if (n < 0 || !boards || !board_index || !cur || !alt || !codes || !escapes || !n_moves || !flag_index ||
        !flag_status || !codes_total || !esc_total || !n_flagged || (n > 0 && n_boards <= 0))
        return TRL_E_ARG;
    *codes_total = *esc_total = *n_flagged = 0;
    if (n == 0) return TRL_OK;
    const bool from_lists = g_codes_source == 0;
    const int chunk = 1 << TRL_HOST_CHUNK_LOG2;
    const int cmax = n < chunk ? n : chunk;
    const int tiles_max = (cmax + kTile - 1) / kTile;
    const size_t list_cap = (size_t)cmax * kListPerCall;
    const size_t stage_codes = (size_t)cmax * kCodesPerCall;
    // staging of one chunk, every region 256-byte aligned
    auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t part = al(sizeof(CodeTotals)) + al(8) +
                        (from_lists ? al(list_cap * 2) + al((size_t)cmax * 8) : al((size_t)cmax * TRL_MASK_WORDS * 4)) +
                        al((size_t)cmax * TRL_ROWS * 2) + al((size_t)cmax * 4) * 4 + al((size_t)cmax * 2) +
                        al(cmax) * 2 + al((size_t)cmax * 8) + al((size_t)tiles_max * 8) + al((size_t)tiles_max * 16) +
                        al(stage_codes) + al((size_t)cmax * kMaxEscapes * 2);
    char* ws = (char*)trl_workspace(TRL_WS_HOST_STAGE, TRL_HOST_STREAMS * part);
    if (!ws) return TRL_E_NOMEM;
    uint4* d_all = (uint4*)trl_workspace(TRL_WS_HOST_BOARDS, (size_t)n_boards * TRL_ROWS * 2);
    if (!d_all) return TRL_E_NOMEM;
    cudaStream_t st[TRL_HOST_STREAMS];
    for (int k = 0; k < TRL_HOST_STREAMS; ++k) if (!(st[k] = trl_host_stream(k))) return TRL_E_CUDA;
    // per device: pinned chunk totals and the event the chunk streams wait on for the board upload
    static CodeTotals* h_tot_of[TRL_MAX_DEVICES] = {};
    static cudaEvent_t uploaded_of[TRL_MAX_DEVICES] = {};
    const int dev = trl_device();
    if (dev < 0) return TRL_E_CUDA;
    CodeTotals*& h_tot = h_tot_of[dev];
    if (!h_tot && trl_check(cudaMallocHost(&h_tot, TRL_HOST_STREAMS * sizeof(CodeTotals))) != TRL_OK) return TRL_E_CUDA;
    cudaEvent_t& uploaded = uploaded_of[dev];
    if (!uploaded && trl_check(cudaEventCreateWithFlags(&uploaded, cudaEventDisableTiming)) != TRL_OK) return TRL_E_CUDA;

    int rc = trl_check(cudaMemcpyAsync(d_all, boards, (size_t)n_boards * TRL_ROWS * 2, cudaMemcpyHostToDevice, st[0]));
    if (!rc) rc = trl_check(cudaEventRecord(uploaded, st[0]));
    for (int k = 1; k < TRL_HOST_STREAMS && !rc; ++k) rc = trl_check(cudaStreamWaitEvent(st[k], uploaded, 0));
    if (rc) return rc;

    struct Pending { int m; uint8_t* d_codes; uint16_t* d_esc; uint32_t* d_fidx; uint32_t* d_fst; bool live; } pend[TRL_HOST_STREAMS] = {};
    uint64_t code_base = 0, esc_base = 0, flag_base = 0;
    // A ring of TRL_HOST_STREAMS chunks in flight, as in trl_movegen_host_compact: a chunk's codes, escapes and flagged
    // calls are fetched when its part is needed again, at the call-ordered place the totals of the chunks before give.
    auto drain = [&](int h) -> int {
        Pending& p = pend[h];
        if (!p.live) return TRL_OK;
        p.live = false;
        int r = trl_check(cudaStreamSynchronize(st[h]));
        if (r) return r;
        const CodeTotals t = h_tot[h];
        if (t.error) return TRL_E_ARG;   // a board index past n_boards, or more than kCodesPerCall placements per call
        if (code_base + t.codes > codes_cap || esc_base + t.escapes > esc_cap || flag_base + t.flagged > flag_cap)
            return TRL_E_ARG;                                  // caller buffer too small
        r = trl_check(cudaMemcpyAsync(codes + code_base, p.d_codes, t.codes, cudaMemcpyDeviceToHost, st[h]));
        if (!r) r = trl_check(cudaMemcpyAsync(escapes + esc_base, p.d_esc, (size_t)t.escapes * 2, cudaMemcpyDeviceToHost, st[h]));
        if (!r) r = trl_check(cudaMemcpyAsync(flag_index + flag_base, p.d_fidx, (size_t)t.flagged * 4, cudaMemcpyDeviceToHost, st[h]));
        if (!r) r = trl_check(cudaMemcpyAsync(flag_status + flag_base, p.d_fst, (size_t)t.flagged * 4, cudaMemcpyDeviceToHost, st[h]));
        code_base += t.codes;
        esc_base += t.escapes;
        flag_base += t.flagged;
        return r;
    };
    int c = 0;
    for (int off = 0; off < n && !rc; off += chunk, ++c) {
        const int h = c % TRL_HOST_STREAMS;
        rc = drain(h);
        if (rc) break;
        const int m = (n - off < chunk) ? n - off : chunk;
        const int tiles = (m + kTile - 1) / kTile;
        char* p = ws + (size_t)h * part;
        auto take = [&](size_t b) { char* q = p; p += al(b); return q; };
        CodeTotals* d_tot = (CodeTotals*)take(sizeof(CodeTotals));
        unsigned long long* d_list_total = (unsigned long long*)take(8);
        uint32_t* d_mask = nullptr;
        uint16_t* d_list = nullptr;
        unsigned long long* d_list_offs = nullptr;
        if (from_lists) {
            d_list = (uint16_t*)take(list_cap * 2);
            d_list_offs = (unsigned long long*)take((size_t)cmax * 8);
        } else {
            d_mask = (uint32_t*)take((size_t)cmax * TRL_MASK_WORDS * 4);
        }
        uint16_t* d_boards = (uint16_t*)take((size_t)cmax * TRL_ROWS * 2);
        uint32_t* d_bidx = (uint32_t*)take((size_t)cmax * 4);
        uint32_t* d_status = (uint32_t*)take((size_t)cmax * 4);
        uint32_t* d_fidx = (uint32_t*)take((size_t)cmax * 4);
        uint32_t* d_fst = (uint32_t*)take((size_t)cmax * 4);
        uint16_t* d_nm = (uint16_t*)take((size_t)cmax * 2);
        uint8_t* d_cur = (uint8_t*)take(cmax);
        uint8_t* d_alt = (uint8_t*)take(cmax);
        unsigned long long* d_local = (unsigned long long*)take((size_t)cmax * 8);
        unsigned long long* d_tile_total = (unsigned long long*)take((size_t)tiles_max * 8);
        uint4* d_tile_base = (uint4*)take((size_t)tiles_max * 16);
        uint8_t* d_codes = (uint8_t*)take(stage_codes);
        uint16_t* d_esc = (uint16_t*)take((size_t)cmax * kMaxEscapes * 2);
        cudaStream_t s = st[h];
        rc = trl_check(cudaMemsetAsync(d_tot, 0, sizeof(CodeTotals), s));
        if (!rc && from_lists) rc = trl_check(cudaMemsetAsync(d_list_total, 0, 8, s));
        if (!rc) rc = trl_check(cudaMemcpyAsync(d_bidx, board_index + off, (size_t)m * 4, cudaMemcpyHostToDevice, s));
        if (!rc) rc = trl_check(cudaMemcpyAsync(d_cur, cur + off, m, cudaMemcpyHostToDevice, s));
        if (!rc) rc = trl_check(cudaMemcpyAsync(d_alt, alt + off, m, cudaMemcpyHostToDevice, s));
        if (!rc) {
            gather_boards_kernel<<<(m + 255) / 256, 256, 0, s>>>(d_all, n_boards, d_bidx, m, (uint4*)d_boards, d_tot);
            rc = trl_check(cudaGetLastError());
        }
        if (!rc) rc = trl_launch_movegen_warp(d_boards, d_cur, d_alt, nullptr, nullptr, m, d_mask, nullptr, 0, d_nm, d_status, s,
                                              d_list, from_lists ? list_cap : 0, from_lists ? d_list_total : nullptr, d_list_offs);
        if (!rc) {
            (from_lists ? codes_count_kernel<true> : codes_count_kernel<false>)<<<tiles, kCountWarps * 32, 0, s>>>(
                d_mask, d_list, d_list_offs, d_nm, d_status, m, d_local, d_tile_total);
            codes_scan_kernel<<<1, 1024, 0, s>>>(d_tile_total, tiles, d_tile_base, d_tot, (uint32_t)stage_codes,
                                                 from_lists ? d_list_total : nullptr, list_cap);
            (from_lists ? codes_write_kernel<true> : codes_write_kernel<false>)<<<(m + kTileWarps - 1) / kTileWarps, kTile, 0, s>>>(
                d_mask, d_list, d_list_offs, d_nm, d_status, m, off, d_local, d_tile_base, d_tot, d_codes, d_esc, d_fidx, d_fst);
            rc = trl_check(cudaGetLastError());
        }
        if (!rc) rc = trl_check(cudaMemcpyAsync(&h_tot[h], d_tot, sizeof(CodeTotals), cudaMemcpyDeviceToHost, s));
        if (!rc) rc = trl_check(cudaMemcpyAsync(n_moves + off, d_nm, (size_t)m * 2, cudaMemcpyDeviceToHost, s));
        if (!rc) pend[h] = {m, d_codes, d_esc, d_fidx, d_fst, true};
    }
    for (int k = 0; k < TRL_HOST_STREAMS && !rc; ++k) rc = drain((c + k) % TRL_HOST_STREAMS);
    for (int k = 0; k < TRL_HOST_STREAMS; ++k) {
        const int r = trl_check(cudaStreamSynchronize(st[k]));
        if (!rc) rc = r;
    }
    *codes_total = code_base;
    *esc_total = esc_base;
    *n_flagged = flag_base;
    return rc;
}
