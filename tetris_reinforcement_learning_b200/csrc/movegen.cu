// movegen.cu — legal-placement enumeration for sm_100a.
//
// Replaces move_generation.get_move_matrix(player, algo='convolutional')
// (reference move_generation.py:752-789, 77-149, 325-528, 650-749) bit-exactly, including the
// FIFO-order dependent choice between the two T-spin plane groups (SURVEY 0.6 / A.2).
//
// Design (not a port): the reference keeps an emission list and de-duplicates it through a
// dict ("last flagged emission wins, else the first").  Here the emission list does not
// exist.  Per rotation and validity row we keep four 14-bit planes:
//     valid    piece fits at (mx-2, my-2)
//     visited  reached by the search
//     flagged  some rotation-flagged emission happened at this cell
//     ulk      the LAST flagged emission at this cell carried "used last kick"
// and the final answer is  placed = visited & ~valid[my+1]  (every emitted cell ends up
// visited, every visited stuck cell is emitted), split for T by flagged / ulk.
#include <cuda_runtime.h>
#include <stdio.h>
#include <time.h>
#include <stdint.h>

#include "trl_common.cuh"
#include "trl_tables.cuh"

namespace {

constexpr int kFifoCap = 1024;  // live entries; adversarial cave boards peak < 500 (SURVEY A.2-7)

// FIFO entry: mx[0:4) my[4:10) rot[10:12) roc[12] ulk[13]
__device__ __forceinline__ uint16_t fifo_pack(int mx, int my, int rot, int roc, int ulk) {
    return (uint16_t)(mx | (my << 4) | (rot << 10) | (roc << 12) | (ulk << 13));
}

struct PieceSearch {
    uint16_t valid[4][TRL_MAP_H + 1];  // [..][44] stays 0: "below the map" is never valid
    uint16_t visited[4][TRL_MAP_H + 1];
    uint16_t flagged[4][TRL_MAP_H + 1];
    uint16_t ulk[4][TRL_MAP_H + 1];
    uint16_t fifo[kFifoCap];
};

// OR an 11-bit policy row chunk into the bit-packed mask (thread-private memory).
__device__ __forceinline__ void or_chunk(uint32_t* mask, int plane, int row, uint32_t bits11) {
    int bit = (plane * TRL_POLICY_ROWS + row) * TRL_POLICY_COLS;
    int w = bit >> 5, s = bit & 31;
    mask[w] |= bits11 << s;
    if (s > 21) mask[w + 1] |= bits11 >> (32 - s);
}

// One piece type of one call.  Scalar (one thread), state in local memory.
__device__ void search_piece(PieceSearch& S, const uint16_t* rows, int type, bool via_hold,
                             uint32_t* mask, uint32_t& status) {
    uint32_t minos[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) minos[r] = c_minos[type][r];
    const int sx = trl_spawn_x(type);
    // Player.hold_piece -> create_piece spawn test (player.py:37-44, move_generation.py:112-121)
    if (via_hold && !trl_fits(rows, minos[0], sx, TRL_SPAWN_Y)) return;

    // _build_validity_maps (move_generation.py:490-528)
    for (int r = 0; r < 4; ++r) {
        for (int my = 0; my < TRL_MAP_H; ++my) {
            S.valid[r][my] = (uint16_t)trl_valid_row(rows, minos[r], my);
            S.visited[r][my] = 0;
            S.flagged[r][my] = 0;
            S.ulk[r][my] = 0;
        }
        S.valid[r][TRL_MAP_H] = 0;
        S.visited[r][TRL_MAP_H] = 0;
    }
    // _set_starting_position (move_generation.py:164-180)
    int highest = TRL_ROWS;
    for (int i = TRL_ROWS - 1; i >= 0; --i)
        if (rows[i] & TRL_FULL_ROW) highest = i;
    int sy = max(highest - (int)c_matrix_size[type], TRL_SPAWN_Y);
    if (!((S.valid[0][sy + 2] >> (sx + 2)) & 1u)) return;  // :351-352

    const bool is_T = (type == P_T);
    const bool rotates = (type != P_O);
    const int tab = (type == P_I) ? 1 : 0;

    uint32_t head = 0, tail = 0;
    S.fifo[tail++ & (kFifoCap - 1)] = fifo_pack(sx + 2, sy + 2, 0, 0, 0);

    while (head != tail) {
        uint32_t e = S.fifo[head++ & (kFifoCap - 1)];
        int mx = e & 15, my = (e >> 4) & 63, rot = (e >> 10) & 3;
        uint32_t bit = 1u << mx;
        if ((e >> 12) & 1u) {  // arrived by a kick: flagged emission if stuck (:384-394)
            if (!(S.valid[rot][my + 1] & bit)) {
                S.flagged[rot][my] |= (uint16_t)bit;
                S.ulk[rot][my] = (uint16_t)((S.ulk[rot][my] & ~bit) | (((e >> 13) & 1u) ? bit : 0u));
            }
        }
        if (S.visited[rot][my] & bit) continue;   // :397-398
        if (!(S.valid[rot][my] & bit)) continue;  // :406-407

        uint32_t reach = bit;
        for (int fy = my; fy < TRL_MAP_H && reach; ++fy) {
            uint32_t vr = S.valid[rot][fy];
            uint32_t open = vr & ~(uint32_t)S.visited[rot][fy];
            uint32_t r = reach;
            for (;;) {  // horizontal flood within the open cells (:419-423)
                uint32_t nr = r | ((r << 1) & open) | ((r >> 1) & open);
                if (nr == r) break;
                r = nr;
            }
            S.visited[rot][fy] |= (uint16_t)r;  // :425
            uint32_t next_vr = S.valid[rot][fy + 1];
            uint32_t blocked = r & ~next_vr;
            uint32_t edges = blocked | (r & ~(vr << 1)) | (r & ~(vr >> 1));  // :427-429
            if (rotates) {
                while (edges) {  // LSB -> MSB (:433-483)
                    int ex = __ffs(edges) - 1;
                    edges &= edges - 1;
#pragma unroll 1
                    for (int kd = 0; kd < 3; ++kd) {
                        int nrot = (rot + kd + 1) & 3;
                        const TrlKicks& K = c_kicks[tab][rot][kd];
                        for (int ki = 0; ki < K.n; ++ki) {
                            int nmx = ex + K.k[ki][0];
                            int nmy = fy - K.k[ki][1];
                            if ((unsigned)nmx >= (unsigned)TRL_MAP_W || (unsigned)nmy >= (unsigned)TRL_MAP_H) continue;
                            uint32_t nbit = 1u << nmx;
                            if (!(S.valid[nrot][nmy] & nbit)) continue;
                            if (nmy < 2) break;  // origin y < 0: abandon this direction (:463-464)
                            int nulk = (is_T && kd != 1 && ki == K.n - 1) ? 1 : 0;
                            if (!(S.visited[nrot][nmy] & nbit)) {
                                if (tail - head >= (uint32_t)kFifoCap) status |= TRL_ST_QUEUE_OVERFLOW;
                                else S.fifo[tail++ & (kFifoCap - 1)] = fifo_pack(nmx, nmy, nrot, 1, nulk);
                            } else if (!(S.valid[nrot][nmy + 1] & nbit)) {
                                S.flagged[nrot][nmy] |= (uint16_t)nbit;
                                S.ulk[nrot][nmy] = (uint16_t)((S.ulk[nrot][nmy] & ~nbit) | (nulk ? nbit : 0u));
                            }
                            break;  // first successful kick wins (:481)
                        }
                    }
                }
            }
            reach = r & next_vr & ~(uint32_t)S.visited[rot][fy + 1];  // :485-488
        }
    }

    // _convert_placements_to_policy (move_generation.py:650-749)
    const int base = c_plane_base[type];
    const int nrot_planes = c_plane_nrot[type];
    const bool zsi = (type == P_Z || type == P_S || type == P_I);
    for (int rot = 0; rot < 4; ++rot) {
        if (type == P_O && rot > 0) break;
        for (int my = 2; my < TRL_MAP_H - 1; ++my) {
            uint32_t placed = S.visited[rot][my] & ~(uint32_t)S.valid[rot][my + 1];
            if (!placed) continue;
            int row = my - 2;
            uint32_t bits = placed;  // bit mx == policy column x + 2
            if (zsi) {               // rot 2 -> (rot 0, row + 1); rot 3 -> (rot 1, col - 1)
                if (rot == 2) row += 1;
                else if (rot == 3) bits >>= 1;
            }
            bits &= 0x7FFu;
            int prot = rot % nrot_planes;
            if (!is_T) {
                or_chunk(mask, base + prot, row, bits);
            } else {
                uint32_t f = S.flagged[rot][my] & placed, u = S.ulk[rot][my];
                uint32_t b0 = placed & ~f, b1 = f & ~u, b2 = f & u;
                if (b0) or_chunk(mask, base + rot, row, b0 & 0x7FFu);
                if (b1) or_chunk(mask, base + 4 + rot, row, b1 & 0x7FFu);
                if (b2) or_chunk(mask, base + 8 + rot, row, b2 & 0x7FFu);
            }
        }
    }
}

// v0: one thread per call.  Bootstrap kernel: exact by construction, used to bring the
// boundary, the tests and the bench up; superseded by the warp-cooperative kernel.
__global__ void __launch_bounds__(128)
movegen_thread_kernel(const uint16_t* __restrict__ boards, const uint8_t* __restrict__ cur,
                      const uint8_t* __restrict__ alt, const TrlGame* __restrict__ games,
                      const int32_t* __restrict__ index, int n,
                      uint32_t* __restrict__ mask_bits, uint32_t* __restrict__ scratch_masks,
                      uint16_t* __restrict__ moves, int moves_cap, uint16_t* __restrict__ n_moves,
                      uint32_t* __restrict__ status) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint16_t rows[TRL_ROWS];
    int c, a;
    if (games) {
        const int gi = index ? index[i] : i;
        if (gi < 0) {  // nothing to enumerate for this item
            if (n_moves) n_moves[i] = 0;
            if (status) status[i] = 0;
            return;
        }
        const TrlPlayer& p = games[gi].players[games[gi].turn & 1];
        for (int r = 0; r < TRL_ROWS; ++r) rows[r] = p.rows[r];
        c = p.piece;
        a = (p.held != TRL_NONE) ? p.held : (p.qlen > 0 ? p.queue[0] : TRL_NONE);
    } else {
        for (int r = 0; r < TRL_ROWS; ++r) rows[r] = boards[(size_t)i * TRL_ROWS + r];
        c = cur[i];
        a = alt[i];
    }
    uint32_t* mask = (mask_bits ? mask_bits : scratch_masks) + (size_t)i * TRL_MASK_WORDS;
    for (int w = 0; w < TRL_MASK_WORDS; ++w) mask[w] = 0;
    uint32_t st = 0;
    if (c > 6 && c != TRL_NONE) c = TRL_NONE;
    if (a > 6 && a != TRL_NONE) a = TRL_NONE;
    if (c == TRL_NONE && a == TRL_NONE) st |= TRL_ST_NO_PIECE;
    PieceSearch S;
    if (c != TRL_NONE) search_piece(S, rows, c, false, mask, st);
    if (a != TRL_NONE && a != c) search_piece(S, rows, a, true, mask, st);

    int count = 0;
    uint16_t* mv = moves ? moves + (size_t)i * moves_cap : nullptr;
    for (int w = 0; w < TRL_MASK_WORDS; ++w) {
        uint32_t m = mask[w];
        while (m) {
            int b = __ffs(m) - 1;
            m &= m - 1;
            if (mv) {
                if (count < moves_cap) mv[count] = (uint16_t)(w * 32 + b);
                else st |= TRL_ST_MOVES_TRUNC;
            }
            ++count;
        }
    }
    if (n_moves) n_moves[i] = (uint16_t)count;
    if (status) status[i] = st;
}

}  // namespace

// ---------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------

// movegen_warp.cu
int trl_launch_movegen_warp(const uint16_t* boards, const uint8_t* cur, const uint8_t* alt, const TrlGame* games,
                            const int32_t* index, int n, uint32_t* mask_bits, uint16_t* moves, int moves_cap,
                            uint16_t* n_moves, uint32_t* status, cudaStream_t stream, uint16_t* compact = nullptr,
                            unsigned long long compact_cap = 0, unsigned long long* compact_total = nullptr,
                            unsigned long long* offsets = nullptr);


// Which kernel enumerates: 0 = one thread per call (movegen_thread_kernel), 1 = one warp per piece
// search (movegen_warp_kernel), -1 = automatic.  Both are bit-exact; they differ in latency/throughput.
static int g_movegen_kernel = -1;
extern "C" void trl_movegen_select_kernel(int kernel) { g_movegen_kernel = kernel; }

static int launch_movegen(const uint16_t* boards, const uint8_t* cur, const uint8_t* alt,
                          const TrlGame* games, const int32_t* index, int n, uint32_t* mask_bits, uint16_t* moves,
                          int moves_cap, uint16_t* n_moves, uint32_t* status, cudaStream_t stream, int n_total = 0) {
    if (n < 0 || (!games && (!boards || !cur || !alt)) || (moves && moves_cap <= 0)) return TRL_E_ARG;
    if (n == 0) return TRL_OK;
    // automatic = the warp kernel: ~12x lower latency on the few-thousand-call batches of a self-play
    // step and on par (slightly ahead) on multi-million-call sweeps; the thread kernel stays as an
    // independent implementation for cross-checks (tests run both).
    (void)n_total;
    if (g_movegen_kernel != 0)
        return trl_launch_movegen_warp(boards, cur, alt, games, index, n, mask_bits, moves, moves_cap, n_moves, status, stream);
    uint32_t* scratch = nullptr;
    if (!mask_bits) {
        // the v0 kernel builds the mask in global memory; without a caller buffer use the workspace
        scratch = (uint32_t*)trl_workspace(TRL_WS_MOVEGEN_MASK, (size_t)n * TRL_MASK_WORDS * sizeof(uint32_t));
        if (!scratch) return TRL_E_NOMEM;
    }
    const int block = 128;
    movegen_thread_kernel<<<(n + block - 1) / block, block, 0, stream>>>(
        boards, cur, alt, games, index, n, mask_bits, scratch, moves, moves_cap, n_moves, status);
    return trl_check(cudaGetLastError());
}

extern "C" int trl_movegen(const uint16_t* boards, const uint8_t* cur, const uint8_t* alt, int n,
                           uint32_t* mask_bits, uint16_t* moves, int moves_cap, uint16_t* n_moves,
                           uint32_t* status, void* stream) {
    return launch_movegen(boards, cur, alt, nullptr, nullptr, n, mask_bits, moves, moves_cap, n_moves, status,
                          (cudaStream_t)stream);
}

extern "C" int trl_movegen_games(const TrlGame* games, int n, uint32_t* mask_bits, uint16_t* moves,
                                 int moves_cap, uint16_t* n_moves, uint32_t* status, void* stream) {
    if (!games) return TRL_E_ARG;
    return launch_movegen(nullptr, nullptr, nullptr, games, nullptr, n, mask_bits, moves, moves_cap, n_moves,
                          status, (cudaStream_t)stream);
}

// Search-internal form: item i enumerates games[index[i]] (index[i] < 0: no moves).
int trl_movegen_indexed(const TrlGame* games, const int32_t* index, int n, uint16_t* moves, int moves_cap,
                        uint16_t* n_moves, uint32_t* status, cudaStream_t stream) {
    return launch_movegen(nullptr, nullptr, nullptr, games, index, n, nullptr, moves, moves_cap, n_moves, status, stream);
}

#ifndef TRL_HOST_CHUNK_LOG2
#define TRL_HOST_CHUNK_LOG2 17   // calls per staging chunk of the *_host entry points
#endif

extern "C" int trl_movegen_host(const uint16_t* boards, const uint8_t* cur, const uint8_t* alt, int n,
                                uint32_t* mask_bits, uint16_t* moves, int moves_cap, uint16_t* n_moves,
                                uint32_t* status) {
    if (n < 0 || !boards || !cur || !alt || (moves && moves_cap <= 0)) return TRL_E_ARG;
    if (n == 0) return TRL_OK;
    // Chunked over a ring of TRL_HOST_STREAMS streams: with pinned host buffers the H2D / D2H copies of one chunk
    // overlap the kernels of the others; the staging workspace stays bounded for multi-million-call sweeps.
    const int chunk = 1 << TRL_HOST_CHUNK_LOG2;
    const size_t per = TRL_ROWS * 2 + 2 + TRL_MASK_WORDS * 4 + (moves ? (size_t)moves_cap * 2 : 0) + 2 + 4;
    const int cmax = n < chunk ? n : chunk;
    const size_t part = (per * (size_t)cmax + 255) & ~(size_t)255;
    char* ws = (char*)trl_workspace(TRL_WS_HOST_STAGE, TRL_HOST_STREAMS * part);
    if (!ws) return TRL_E_NOMEM;
    cudaStream_t st[TRL_HOST_STREAMS];
    for (int k = 0; k < TRL_HOST_STREAMS; ++k) if (!(st[k] = trl_host_stream(k))) return TRL_E_CUDA;
    int rc = TRL_OK;
    int c = 0;
    for (int off = 0; off < n && !rc; off += chunk, ++c) {
        const int m = (n - off < chunk) ? n - off : chunk;
        const int h = c % TRL_HOST_STREAMS;
        cudaStream_t s = st[h];
        rc = trl_check(cudaStreamSynchronize(s));  // this part's previous chunk has fully drained
        if (rc) break;
        char* p = ws + (size_t)h * part;
        uint32_t* d_mask = (uint32_t*)p;  p += (size_t)m * TRL_MASK_WORDS * 4;
        uint32_t* d_status = (uint32_t*)p; p += (size_t)m * 4;
        uint16_t* d_boards = (uint16_t*)p; p += (size_t)m * TRL_ROWS * 2;
        uint16_t* d_moves = nullptr;
        if (moves) { d_moves = (uint16_t*)p; p += (size_t)m * moves_cap * 2; }
        uint16_t* d_nm = (uint16_t*)p; p += (size_t)m * 2;
        uint8_t* d_cur = (uint8_t*)p; p += m;
        uint8_t* d_alt = (uint8_t*)p; p += m;
        rc = trl_check(cudaMemcpyAsync(d_boards, boards + (size_t)off * TRL_ROWS, (size_t)m * TRL_ROWS * 2, cudaMemcpyHostToDevice, s));
        if (!rc) rc = trl_check(cudaMemcpyAsync(d_cur, cur + off, m, cudaMemcpyHostToDevice, s));
        if (!rc) rc = trl_check(cudaMemcpyAsync(d_alt, alt + off, m, cudaMemcpyHostToDevice, s));
        if (!rc) rc = launch_movegen(d_boards, d_cur, d_alt, nullptr, nullptr, m, d_mask, d_moves, moves_cap, d_nm, d_status, s, n);
        if (!rc && mask_bits) rc = trl_check(cudaMemcpyAsync(mask_bits + (size_t)off * TRL_MASK_WORDS, d_mask, (size_t)m * TRL_MASK_WORDS * 4, cudaMemcpyDeviceToHost, s));
        if (!rc && moves) rc = trl_check(cudaMemcpyAsync(moves + (size_t)off * moves_cap, d_moves, (size_t)m * moves_cap * 2, cudaMemcpyDeviceToHost, s));
        if (!rc && n_moves) rc = trl_check(cudaMemcpyAsync(n_moves + off, d_nm, (size_t)m * 2, cudaMemcpyDeviceToHost, s));
        if (!rc && status) rc = trl_check(cudaMemcpyAsync(status + off, d_status, (size_t)m * 4, cudaMemcpyDeviceToHost, s));
    }
    for (int k = 0; k < TRL_HOST_STREAMS; ++k) {
        const int r = trl_check(cudaStreamSynchronize(st[k]));
        if (!rc) rc = r;
    }
    return rc;
}

// Host entry point with COMPACT output: the ascending move lists of all calls packed back to back
// (no padding), which is what crosses PCIe.  Call i owns moves_compact[offsets[i] .. offsets[i] +
// n_moves[i]); segments are handed out by an atomic bump allocator per chunk, so their order inside a
// chunk is arbitrary.  D2H traffic: 2 B per placement + 14 B per call instead of 1448 B of mask.
extern "C" int trl_movegen_host_compact(const uint16_t* boards, const uint8_t* cur, const uint8_t* alt, int n,
                                        uint16_t* moves_compact, uint64_t capacity, uint64_t* offsets,
                                        uint16_t* n_moves, uint32_t* status, uint64_t* total_out) {
    if (n < 0 || !boards || !cur || !alt || !moves_compact || !offsets || !n_moves || !total_out) return TRL_E_ARG;
    *total_out = 0;
    if (n == 0) return TRL_OK;
    const int chunk = 1 << TRL_HOST_CHUNK_LOG2;
    const size_t list_cap = (size_t)chunk * 160;   // per-chunk staging: 160 placements per call on average (x 2 B)
    const size_t per = TRL_ROWS * 2 + 2 + 8 + 2 + 4;
    const int cmax = n < chunk ? n : chunk;
    const size_t part = ((per * (size_t)cmax + list_cap * 2 + 64) + 255) & ~(size_t)255;
    char* ws = (char*)trl_workspace(TRL_WS_HOST_STAGE, TRL_HOST_STREAMS * part);
    if (!ws) return TRL_E_NOMEM;
    cudaStream_t st[TRL_HOST_STREAMS];
    for (int k = 0; k < TRL_HOST_STREAMS; ++k) if (!(st[k] = trl_host_stream(k))) return TRL_E_CUDA;
    static unsigned long long* h_total_of[TRL_MAX_DEVICES] = {};   // pinned: the per-chunk totals come back through it
    const int dev = trl_device();
    if (dev < 0) return TRL_E_CUDA;
    unsigned long long*& h_total = h_total_of[dev];
    if (!h_total && trl_check(cudaMallocHost(&h_total, TRL_HOST_STREAMS * sizeof(unsigned long long))) != TRL_OK) return TRL_E_CUDA;
    struct Pending { int off, m; uint16_t* d_list; bool live; } pend[TRL_HOST_STREAMS] = {};
    uint64_t base = 0;
    int rc = TRL_OK;
    // A ring of TRL_HOST_STREAMS chunks in flight: the H2D copies, the two kernels and the small D2H copies (offsets,
    // counts, status, total) of a chunk are queued at once; its move list is fetched when the part is needed again
    // (three chunks later), with exactly `total` entries, at its place in the caller's buffer.
#ifdef TRL_E2E_TRACE
    auto now_ms = []() { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6; };
    const double t_begin = now_ms();
    double t_wait1 = 0, t_fix = 0, t_submit = 0;
#endif
    auto drain = [&](int h) -> int {
        Pending& p = pend[h];
        if (!p.live) return TRL_OK;
        p.live = false;
#ifdef TRL_E2E_TRACE
        const double ta = now_ms();
#endif
        int r = trl_check(cudaStreamSynchronize(st[h]));
#ifdef TRL_E2E_TRACE
        t_wait1 += now_ms() - ta;
#endif
        if (r) return r;
        const unsigned long long total = h_total[h];
        if (total > list_cap || base + total > capacity) return TRL_E_ARG;   // staging / caller buffer too small
        r = trl_check(cudaMemcpyAsync(moves_compact + base, p.d_list, (size_t)total * 2, cudaMemcpyDeviceToHost, st[h]));
        if (r) return r;
#ifdef TRL_E2E_TRACE
        const double tb = now_ms();
#endif
        for (int k = 0; k < p.m; ++k) offsets[p.off + k] += base;   // chunk-local -> global (under the copy)
        base += total;
#ifdef TRL_E2E_TRACE
        t_fix += now_ms() - tb;
#endif
        // no wait for the list copy: the next chunk of this part is queued behind it on the same stream, and the
        // call ends with a synchronisation of every stream.  (Host timeline of a 7 M-call sweep, -DTRL_E2E_TRACE: 56.5 ms =
        // 53 ms waiting for kernels + 3.5 ms of submission and offset fix-up — the copies are hidden; the kernels take
        // 52.5 ms when they write move lists instead of masks, 42 ms of it the searches.)
        return TRL_OK;
    };
    int c = 0;
    for (int off = 0; off < n && !rc; off += chunk, ++c) {
        const int h = c % TRL_HOST_STREAMS;
        rc = drain(h);   // this part's previous chunk (chunks are drained in submission order, so `base` grows in chunk order)
        if (rc) break;
#ifdef TRL_E2E_TRACE
        const double ts0 = now_ms();
#endif
        const int m = (n - off < chunk) ? n - off : chunk;
        char* p = ws + (size_t)h * part;
        unsigned long long* d_total = (unsigned long long*)p; p += 64;
        unsigned long long* d_offs = (unsigned long long*)p; p += (size_t)m * 8;
        uint32_t* d_status = (uint32_t*)p; p += (size_t)m * 4;
        uint16_t* d_boards = (uint16_t*)p; p += (size_t)m * TRL_ROWS * 2;
        uint16_t* d_nm = (uint16_t*)p; p += (size_t)m * 2;
        uint16_t* d_list = (uint16_t*)p; p += list_cap * 2;
        uint8_t* d_cur = (uint8_t*)p; p += m;
        uint8_t* d_alt = (uint8_t*)p; p += m;
        cudaStream_t s = st[h];
        rc = trl_check(cudaMemsetAsync(d_total, 0, 8, s));
        if (!rc) rc = trl_check(cudaMemcpyAsync(d_boards, boards + (size_t)off * TRL_ROWS, (size_t)m * TRL_ROWS * 2, cudaMemcpyHostToDevice, s));
        if (!rc) rc = trl_check(cudaMemcpyAsync(d_cur, cur + off, m, cudaMemcpyHostToDevice, s));
        if (!rc) rc = trl_check(cudaMemcpyAsync(d_alt, alt + off, m, cudaMemcpyHostToDevice, s));
        if (!rc) rc = trl_launch_movegen_warp(d_boards, d_cur, d_alt, nullptr, nullptr, m, nullptr, nullptr, 0, d_nm, d_status, s,
                                              d_list, list_cap, d_total, d_offs);
        if (!rc) rc = trl_check(cudaMemcpyAsync(&h_total[h], d_total, 8, cudaMemcpyDeviceToHost, s));
        if (!rc) rc = trl_check(cudaMemcpyAsync(offsets + off, d_offs, (size_t)m * 8, cudaMemcpyDeviceToHost, s));
        if (!rc) rc = trl_check(cudaMemcpyAsync(n_moves + off, d_nm, (size_t)m * 2, cudaMemcpyDeviceToHost, s));
        if (!rc && status) rc = trl_check(cudaMemcpyAsync(status + off, d_status, (size_t)m * 4, cudaMemcpyDeviceToHost, s));
        if (!rc) pend[h] = {off, m, d_list, true};
#ifdef TRL_E2E_TRACE
        t_submit += now_ms() - ts0;
#endif
    }
    // the chunks still in flight, oldest first; then every list copy has to land before the call returns
    for (int k = 0; k < TRL_HOST_STREAMS && !rc; ++k) rc = drain((c + k) % TRL_HOST_STREAMS);
    for (int k = 0; k < TRL_HOST_STREAMS; ++k) {
        const int r = trl_check(cudaStreamSynchronize(st[k]));
        if (!rc) rc = r;
    }
#ifdef TRL_E2E_TRACE
    fprintf(stderr, "[trl e2e] %d calls in %d chunks: total %.2f ms; host: submit %.2f, wait for kernels %.2f, offsets fix-up %.2f\n",
            n, c, now_ms() - t_begin, t_submit, t_wait1, t_fix);
#endif
    *total_out = base;
    return rc;
}
