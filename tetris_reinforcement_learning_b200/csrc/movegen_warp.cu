// movegen_warp.cu — warp-cooperative legal-placement enumeration.
//
// Same operator and the same bit-exact contract as movegen.cu (reference
// move_generation.get_move_matrix(player, 'convolutional'), move_generation.py:77-149, 325-528,
// 650-749, including the FIFO-order dependent choice between the two T-spin plane groups, SURVEY
// 0.6 / A.2).  Two search forms and three ways to launch them (DESIGN.md §3.1):
//
//   search_piece_rows   the row-parallel CLOSURE search (the common case): what the reference's queue
//                       computes is a closure that does not depend on the queue order, so it is run as a
//                       fix point on register-resident bit planes, lane = validity row, all four rotations
//                       at once; t_order_decide settles the one order-dependent output (the used-last-kick
//                       flag of T cells that received both flag values) from the structure of the queue where
//                       it can, and says "undecided" where it cannot;
//   search_piece_fifo   the exact FIFO search (round 1's kernel body, the specification of the T flags):
//       vv[rot][row]  low 16 bits = validity row, high 16 bits = visited row     (4 x 46 words)
//       fu[rot][row]  T: low 16 bits = flagged, high 16 bits = used-last-kick; other pieces: low 16
//                     bits = "already queued" (de-duplicates queue entries; order is irrelevant for them)
//       fifo[768]     the exploration queue (ring), entries (mx, my, rot, roc, ulk) as in movegen.cu
//     * the queue is consumed 32 entries at a time: every lane tests one entry (stuck? visited?),
//       a ballot finds the first entry that starts a flood fill, the entries before it only
//       produce their "arrived by a kick and stuck" emission (move_generation.py:384-394);
//     * the flood fill of one rotation is a serial scan over rows whose horizontal expansion is an
//       O(1) carry-propagation trick (open + seed), not a fix-point loop;
//     * kicks are evaluated for ALL edge cells of ALL rows of the fill at once: lane = row, bit =
//       column, one AND/shift per (kick direction, kick index) against the target rotation's
//       validity row ("first valid kick wins" = a running `remaining` mask, :443-481);
//     * new queue entries are appended in the reference's order (row, column LSB->MSB, direction)
//       with a warp prefix sum over per-row counts, so FIFO order — and with it the T-spin plane —
//       is reproduced exactly.  "Last flagged emission wins" (:671-677) is order dependent only when
//       emissions with different used-last-kick flags hit the same cell: the common case (all equal)
//       is applied with shared-memory atomics, the mixed case serially in reference order.
//
//   movegen_warp_kernel   two warps per call, one per piece type (latency form: self-play batches);
//   movegen_solo_kernel   one warp per call; also the legacy route of the pass form;
//   movegen_rows_kernel   the closure search alone, deferred T searches and undecided calls appended to lists, then
//                         movegen_t_order_kernel and movegen_t_exact_kernel for the deferred T searches (the pass
//                         form, for throughput: the multi-million-call sweep); movegen_list_kernel is the enumeration
//                         inside a self-play step.
// In every form the answer placed = visited & ~valid[row+1] is OR-ed into a per-call bit mask in shared
// memory, written out coalesced, and turned into the ascending move list (= np.argwhere order).
#include <cuda_runtime.h>
#include <stdint.h>

#include <mutex>

#include "trl_common.cuh"
#include "trl_tables.cuh"

namespace {

constexpr int kFifoCap = 768;             // live entries; adversarial cave boards peak < 500 (SURVEY A.2-7).
__constant__ int c_fifo_limit = kFifoCap;   // <= kFifoCap; lowered only by trl_debug_movegen_fifo_limit (tests force the overflow bit)
                                          // 768 keeps a block at 30 KB of shared memory: 7 blocks = 56 warps per SM
constexpr int kCallsPerBlock = 8;   // 16 warps, 60 KB of shared memory, 62 registers: 2 blocks per SM (measured best of 1/2/4/8;
                                    // __launch_bounds__(512, 3) = 40 registers with spills: 125 ms vs 119 ms on the sweep)
constexpr int kWarps = 2 * kCallsPerBlock;
constexpr int kVRows = TRL_MAP_H + 2;     // rows 44, 45 stay 0: "below the map" is never valid

struct PieceState {
    uint32_t vv[4][kVRows];
    uint32_t fu[4][kVRows];
    union {
        uint16_t fifo[kFifoCap];                 // exact FIFO form
        struct {                                  // closure form, T only (see t_order_decide)
            uint32_t tsnap[4][32];                // arrivals of the first two kick rounds per (rotation, lane): N | U << 16
            uint32_t tp[4][2][36];                // class planes of up to four kick passes: [pass][N_hi | U << 16, N_lo][row + 2]
        };
    };
};

struct CallState {
    alignas(16) uint32_t mask[TRL_MASK_WORDS + 2];   // 364 words = 91 x 16 B
    uint16_t woff[TRL_MASK_WORDS + 2];               // set bits before word w inside its lane's 12-word run (write_call_outputs)
    uint16_t lbase[32];                              // list position of the first set bit of lane l's run
    uint16_t rows[TRL_ROWS];
    int cur, alt, skip;
    uint32_t status;
};

__device__ __forceinline__ uint32_t fifo_pack(int mx, int my, int rot, int roc, int ulk) {
    return (uint32_t)(mx | (my << 4) | (rot << 10) | (roc << 12) | (ulk << 13));
}

// All cells reachable from `seed` by horizontal moves through `open` (seed must be a subset of
// open): the carry of open + seed runs through every run of ones above a seed.
__device__ __forceinline__ uint32_t hflood(uint32_t seed, uint32_t open) {
    const uint32_t up = ((open + seed) ^ open) & open;
    const uint32_t ro = __brev(open), rs = __brev(seed);
    const uint32_t dn = __brev(((ro + rs) ^ ro) & ro);
    return up | dn | seed;
}

// OR an 11-bit policy row chunk into the bit-packed mask in shared memory.
__device__ __forceinline__ void or_chunk(uint32_t* mask, int plane, int row, uint32_t bits11) {
    if (!bits11) return;
    const int bit = (plane * TRL_POLICY_ROWS + row) * TRL_POLICY_COLS;
    const int w = bit >> 5, s = bit & 31;
    atomicOr(&mask[w], bits11 << s);
    if (s > 21) atomicOr(&mask[w + 1], bits11 >> (32 - s));
}

// set / clear one used-last-kick bit and raise the flagged bit of a stuck cell
__device__ __forceinline__ void flag_cell(uint32_t* fu_row, uint32_t bit, bool ulk) {
    if (ulk) atomicOr(fu_row, bit | (bit << 16));
    else { atomicOr(fu_row, bit); atomicAnd(fu_row, ~(bit << 16)); }
}

// ---------------------------------------------------------------------------------------
// Row-parallel closure search (the common case; search_piece_warp below is the exact general form).
//
// Everything the reference's FIFO exploration computes is a closure that does not depend on queue order
// (SURVEY A.2-6) — except which used-last-kick flag the LAST rotation-flagged emission of a T cell
// carried.  So the search is run as a fix point on register-resident bit planes, lane = validity row
// (rows 12..43; the spawn row is >= 19 and nothing above it can be entered without kicks):
//
//   * two rotations share a register (16 bits each, validity rows are 14 bits wide, the two spare bits
//     stop the carries of hflood): VA/VB validity, RA/RB reached; A holds rotations 0 | 2 << 16, B 1 | 3 << 16,
//     so that each pair of kick passes with equal kick lists runs in one word (kick_pass_pair);
//   * fill = alternate "expand along rows" (hflood, O(1)) and "fall straight down" (a segmented
//     Hillis-Steele OR-scan over lanes, 5 shuffles, propagate masks precomputed) until nothing changes —
//     all four rotations at once, instead of one serial row scan per queue entry;
//   * kicks are evaluated only for edge cells reached since the previous round (move_generation.py:
//     427-483: first valid kick wins, lane = row, bit = column, one shift/AND per kick); targets are
//     OR-ed into per-rotation arrival planes in shared memory (for T split by the used-last-kick flag)
//     and become the seeds of the next round's fill;
//   * placed = reached & stuck; T: flagged = arrived & placed (every kick arrival at a stuck cell is a
//     flagged emission, either at its pop, :384-394, or at once, :471-479).
//
// Returns false — and the caller runs the exact FIFO search instead — in the two cases this form cannot
// decide: (i) a stuck T cell received arrivals with BOTH flag values (then the order of emissions matters,
// :671-677; a level-by-level ordering argument — rounds of this search are levels of the reference's queue —
// was tried and decides under 14 % of these cases: the two flags nearly always meet inside one level),
// (ii) something reached the two top rows of the window (a climb of more than five rows by kicks; rows
// above the window are not represented).  Counted in g_fast_stats: 24 % of the T searches, 0 of the others,
// on the BASELINE config-2 boards.
// ---------------------------------------------------------------------------------------
#ifndef TRL_ROWS_SPECIAL_I
#define TRL_ROWS_SPECIAL_I 0   // closure kernel: compile-time kick tables for the I piece too: measured SLOWER (4.63 vs 4.12 ms per 700 k calls: the code outgrows the instruction cache)
#endif
#ifndef TRL_ROWS_SPECIAL_V
#define TRL_ROWS_SPECIAL_V 1   // closure kernel: validity rows with compile-time cell offsets (A/B switch)
#endif
constexpr int kWin0 = 12;   // validity row of lane 0
constexpr int kWinRows = 36;                      // lane + 2, two zero rows either side
__constant__ int c_fast_path = 1;                 // trl_debug_movegen_fast_path(0) forces the FIFO form (tests run both)
__device__ unsigned long long g_fast_stats[16];    // [0] searches answered by the closure form, [1] handed to the FIFO form;
                                                  // with -DTRL_MOVEGEN_STATS also [2] rounds, [3] fill iterations, [4] (rotation, direction) passes, [5] kick tests
#ifdef TRL_T_TRACE
// research build: per T search, the arrival planes of every (round, target rotation, direction) pass
// (tools/t_order_study.py): [search][8 rounds][4 target rotations][3 directions][32 lanes] then [4][32] placed planes
__device__ uint32_t* g_t_trace = nullptr;
__device__ unsigned int g_t_trace_n = 0, g_t_trace_cap = 0;
constexpr int kTTraceWords = 8 * 4 * 3 * 32 + 4 * 32 + 32;   // ... then the board (rows l | rows l+32 << 16)
#endif
#ifdef TRL_MOVEGEN_STATS
#define TRL_STAT(i) (++stat_##i)
#define TRL_REASON(i) do { if ((threadIdx.x & 31) == 0) atomicAdd(&g_fast_stats[i], 1ull); } while (0)
#else
#define TRL_STAT(i) ((void)0)
#define TRL_REASON(i) ((void)0)
#endif

// R closed under "move one row down while the target is valid": P1..P16 are the propagate masks of
// window lengths 1, 2, 4, 8, 16 ending at this lane's row (zero where the window leaves the lane range,
// which also cancels the value a lane < d gets back from its own shuffle).
__device__ __forceinline__ uint32_t fall_scan(uint32_t R, uint32_t P1, uint32_t P2, uint32_t P4, uint32_t P8, uint32_t P16) {
    R |= __shfl_up_sync(0xffffffffu, R, 1) & P1;
    R |= __shfl_up_sync(0xffffffffu, R, 2) & P2;
    R |= __shfl_up_sync(0xffffffffu, R, 4) & P4;
    R |= __shfl_up_sync(0xffffffffu, R, 8) & P8;
    R |= __shfl_up_sync(0xffffffffu, R, 16) & P16;
    return R;
}

// hflood with the bit-reversed `open` precomputed (it is loop invariant in the closure search)
__device__ __forceinline__ uint32_t hflood_r(uint32_t seed, uint32_t open, uint32_t ropen) {
    const uint32_t up = ((open + seed) ^ open) & open;
    const uint32_t dn = __brev(((ropen + __brev(seed)) ^ ropen) & ropen);
    return up | dn | seed;
}

// first board row with a block (40 when the board is empty); rows in shared memory, executed by a whole warp
__device__ __forceinline__ int first_block_row(const uint16_t* rows, int lane) {
    const uint32_t b0 = __ballot_sync(0xffffffffu, (rows[lane] & TRL_FULL_ROW) != 0);
    const uint32_t b1 = __ballot_sync(0xffffffffu, lane < TRL_ROWS - 32 && (rows[(lane & 7) + 32] & TRL_FULL_ROW) != 0);
    return b0 ? (__ffs(b0) - 1) : (b1 ? 31 + __ffs(b1) : TRL_ROWS);
}

// Compile-time copy of the wall-kick table of the six non-I pieces (c_kicks[0], const.py:191-212) for the
// specialised kick passes: with the kick offsets as immediates a kick test is LDS + SHF + 2 LOP3 + vote.
struct KickList { int n; int k[6][2]; };
constexpr KickList kWallKicks[4][3] = {
    {{5, {{0, 0}, {-1, 0}, {-1, 1}, {0, -2}, {-1, -2}, {0, 0}}}, {6, {{0, 0}, {0, 1}, {1, 1}, {-1, 1}, {1, 0}, {-1, 0}}}, {5, {{0, 0}, {1, 0}, {1, 1}, {0, -2}, {1, -2}, {0, 0}}}},
    {{5, {{0, 0}, {1, 0}, {1, -1}, {0, 2}, {1, 2}, {0, 0}}}, {6, {{0, 0}, {1, 0}, {1, 2}, {1, 1}, {0, 2}, {0, 1}}}, {5, {{0, 0}, {1, 0}, {1, -1}, {0, 2}, {1, 2}, {0, 0}}}},
    {{5, {{0, 0}, {1, 0}, {1, 1}, {0, -2}, {1, -2}, {0, 0}}}, {6, {{0, 0}, {0, -1}, {-1, -1}, {1, -1}, {-1, 0}, {1, 0}}}, {5, {{0, 0}, {-1, 0}, {-1, 1}, {0, -2}, {-1, -2}, {0, 0}}}},
    {{5, {{0, 0}, {-1, 0}, {-1, -1}, {0, 2}, {-1, 2}, {0, 0}}}, {6, {{0, 0}, {-1, 0}, {-1, 2}, {-1, 1}, {0, 2}, {0, 1}}}, {5, {{0, 0}, {-1, 0}, {-1, -1}, {0, 2}, {-1, 2}, {0, 0}}}},
};

// ... and of the I piece (c_kicks[1], const.py:214-235)
constexpr KickList kIKicks[4][3] = {
    {{5, {{0, 0}, {-2, 0}, {1, 0}, {-2, -1}, {1, 2}, {0, 0}}}, {2, {{0, 0}, {0, 1}, {0, 0}, {0, 0}, {0, 0}, {0, 0}}}, {5, {{0, 0}, {-1, 0}, {2, 0}, {-1, 2}, {2, -1}, {0, 0}}}},
    {{5, {{0, 0}, {-1, 0}, {2, 0}, {-1, 2}, {2, -1}, {0, 0}}}, {2, {{0, 0}, {1, 0}, {0, 0}, {0, 0}, {0, 0}, {0, 0}}}, {5, {{0, 0}, {2, 0}, {-1, 0}, {2, 1}, {-1, -2}, {0, 0}}}},
    {{5, {{0, 0}, {2, 0}, {-1, 0}, {2, 1}, {-1, -2}, {0, 0}}}, {2, {{0, 0}, {0, -1}, {0, 0}, {0, 0}, {0, 0}, {0, 0}}}, {5, {{0, 0}, {1, 0}, {-2, 0}, {1, -2}, {-2, 1}, {0, 0}}}},
    {{5, {{0, 0}, {1, 0}, {-2, 0}, {1, -2}, {-2, 1}, {0, 0}}}, {2, {{0, 0}, {-1, 0}, {0, 0}, {0, 0}, {0, 0}, {0, 0}}}, {5, {{0, 0}, {-2, 0}, {1, 0}, {-2, -1}, {1, 2}, {0, 0}}}},
};

constexpr bool same_kicks(const KickList& a, const KickList& b) {
    if (a.n != b.n) return false;
    for (int ki = 0; ki < a.n; ++ki)
        if (a.k[ki][0] != b.k[ki][0] || a.k[ki][1] != b.k[ki][1]) return false;
    return true;
}
// The four twin pairs kick_pass_pair runs in one 32-bit word (lists equal offset for offset, const.py:191-212)
static_assert(same_kicks(kWallKicks[0][0], kWallKicks[2][2]), "twin pair (0, 0) / (2, 2)");
static_assert(same_kicks(kWallKicks[0][2], kWallKicks[2][0]), "twin pair (0, 2) / (2, 0)");
static_assert(same_kicks(kWallKicks[1][0], kWallKicks[1][2]), "twin pair (1, 0) / (1, 2)");
static_assert(same_kicks(kWallKicks[3][0], kWallKicks[3][2]), "twin pair (3, 0) / (3, 2)");

#ifdef TRL_MOVEGEN_STATS
#define TRL_COUNT(x) (++(x))
#else
#define TRL_COUNT(x) ((void)0)
#endif

// Rotation r's validity row (<< 2) in the packed planes vv[r & 1], shifted right by `sh`: source bit ex of a kick test
// <-> target bit ex + kx for sh = kx + 2.  The other rotation of the plane starts at bit 18, above anything a 14-bit edge
// row reaches with kx <= 2.
#define TRL_VV(S, r, row, sh) ((S).vv[(r) & 1][row] >> ((sh) + 16 * ((r) >> 1)))

// One (source rotation R, direction KD) pass over the new edge cells `ne` of this lane's row; TAB 0 = the six pieces
// with the common wall-kick table, 1 = the I piece.
template <int TAB, int R, int KD, class St>
__device__ __forceinline__ void kick_pass_wall(St& S, int lane, uint32_t ne, uint32_t VA, uint32_t VB, uint32_t& a0A, uint32_t& a0B, bool is_T,
                                               unsigned& n_pass, unsigned& n_test) {
    constexpr int nrot = (R + KD + 1) & 3;
    constexpr KickList K = TAB ? kIKicks[R][KD] : kWallKicks[R][KD];
#ifdef TRL_MOVEGEN_STATS
    if (__any_sync(0xffffffffu, ne)) TRL_COUNT(n_pass);
#endif
    // kick 0 is (0, 0) in every list (const.py:191-235): target = same cell of the new rotation
    const uint32_t Vn = ((nrot & 1) ? VB : VA) >> (16 * (nrot >> 1));
    const uint32_t c0 = ne & Vn;
    if (nrot & 1) a0B |= c0 << (16 * (nrot >> 1)); else a0A |= c0 << (16 * (nrot >> 1));
    uint32_t rem = ne & ~c0;
    if (!__any_sync(0xffffffffu, rem)) return;
#pragma unroll
    for (int ki = 1; ki < K.n; ++ki) {
        TRL_COUNT(n_test);
        const int kx = K.k[ki][0], ky = K.k[ki][1];
        const uint32_t cand = rem & TRL_VV(S, nrot, lane + 2 - ky, kx + 2);   // source bit ex <-> target bit ex + kx
        rem &= ~cand;
        if (cand) {
            uint32_t arr = kx >= 0 ? (cand << kx) : (cand >> -kx);
            if (KD != 1 && ki == K.n - 1 && is_T) arr <<= 16;                  // nulk (:469)
            atomicOr(&S.fu[nrot][lane + 2 - ky], arr);
        }
        if (ki + 1 < K.n && !__any_sync(0xffffffffu, rem)) return;              // every edge cell has found its kick
    }
}

template <int TAB, int R, class St>
__device__ __forceinline__ void kick_passes_wall(St& S, int lane, uint32_t ne, uint32_t VA, uint32_t VB, uint32_t& a0A, uint32_t& a0B, bool is_T,
                                                 unsigned& n_pass, unsigned& n_test) {
    kick_pass_wall<TAB, R, 0>(S, lane, ne, VA, VB, a0A, a0B, is_T, n_pass, n_test);
    kick_pass_wall<TAB, R, 1>(S, lane, ne, VA, VB, a0A, a0B, is_T, n_pass, n_test);
    kick_pass_wall<TAB, R, 2>(S, lane, ne, VA, VB, a0A, a0B, is_T, n_pass, n_test);
}

// Two (source rotation, direction) passes of the common wall-kick table with equal kick lists, one per 16-bit half:
//   R even (pair (R, KD) / (R ^ 2, KD ^ 2)): src = the packed rot0 | rot2 edge cells, both halves target the odd
//     rotation nrot, whose validity row is duplicated into both halves;
//   R odd (pair (R, KD) / (R, KD ^ 2)): src = rotation R's edge cells in both halves, the low half targets rotation 0,
//     the high half rotation 2: the packed validity plane vv[0] as it is.
// "First valid kick wins" runs per bit, so each half computes exactly its own pass.  No bit crosses between the halves: the
// edge bits of a half sit in 0..13, a kick test reads target bits ex + kx + 2 <= 16 (bit 16 of the word, and of the
// duplicated word, is always 0), and an arrival cannot leave its half downwards since `cand` implies ex + kx >= 0.  Both
// directions of every pair are != 1 (KD ^ 2 = 2 - KD), so the used-last-kick rule is the same for the two halves.
template <int R, int KD, class St>
__device__ __forceinline__ void kick_pass_pair(St& S, int lane, uint32_t src, uint32_t VA, uint32_t VB, uint32_t& a0A, uint32_t& a0B, bool is_T,
                                               unsigned& n_pass, unsigned& n_test) {
    static_assert(KD != 1, "the 180-degree passes have no twin");
    constexpr KickList K = kWallKicks[R][KD];
    constexpr int nrot = (R + KD + 1) & 3;
    static_assert((R & 1) ? nrot == 0 : (nrot & 1) != 0, "low half of an odd source targets rotation 0, an even source an odd rotation");
    constexpr uint32_t dup = nrot == 1 ? 0x1010u : 0x3232u;   // PRMT: the low / high half of the odd plane in both halves
#ifdef TRL_MOVEGEN_STATS
    if (__any_sync(0xffffffffu, src)) TRL_COUNT(n_pass);
#endif
    uint32_t rem;
    if constexpr ((R & 1) == 0) {
        const uint32_t c0 = src & __byte_perm(VB, 0u, dup);
        a0B |= nrot == 1 ? ((c0 | (c0 >> 16)) & 0xFFFFu) : ((c0 | (c0 << 16)) & 0xFFFF0000u);
        rem = src & ~c0;
    } else {
        const uint32_t c0 = src & VA;
        a0A |= c0;
        rem = src & ~c0;
    }
    if (!__any_sync(0xffffffffu, rem)) return;
#pragma unroll
    for (int ki = 1; ki < K.n; ++ki) {
        TRL_COUNT(n_test);
        const int kx = K.k[ki][0], ky = K.k[ki][1];
        const int row = lane + 2 - ky;
        uint32_t tw;
        if constexpr ((R & 1) == 0) tw = __byte_perm(S.vv[1][row], 0u, dup);
        else tw = S.vv[0][row];
        const uint32_t cand = rem & (tw >> (kx + 2));
        rem &= ~cand;
        if (cand) {
            const uint32_t arr = kx >= 0 ? (cand << kx) : (cand >> -kx);
            const bool ulk = ki == K.n - 1 && is_T;                           // nulk (:469)
            if constexpr ((R & 1) == 0) {
                const uint32_t a = (arr | (arr >> 16)) & 0xFFFFu;
                atomicOr(&S.fu[nrot][row], ulk ? a << 16 : a);
            } else {
                const uint32_t lo = ulk ? arr << 16 : arr & 0xFFFFu, hi = ulk ? arr & 0xFFFF0000u : arr >> 16;
                if (lo) atomicOr(&S.fu[0][row], lo);
                if (hi) atomicOr(&S.fu[2][row], hi);
            }
        }
        if (ki + 1 < K.n && !__any_sync(0xffffffffu, rem)) return;
    }
}

// (rot0 | rot2 << 16, rot1 | rot3 << 16) <-> (rot0 | rot1 << 16, rot2 | rot3 << 16): exchange the high half of A with the
// low half of B (its own inverse)
__device__ __forceinline__ void swap_mid_halves(uint32_t& A, uint32_t& B) {
    const uint32_t a = __byte_perm(A, B, 0x5410), b = __byte_perm(A, B, 0x7632);
    A = a;
    B = b;
}

// St: anything with uint32_t vv[>= 2][>= kWinRows], fu[4][>= kWinRows] in shared memory.  The loops are kept
// rolled on purpose: the kernels that call this are bound by instruction fetch, not by loop overhead.
// ---------------------------------------------------------------------------------------
// T: which flag did the LAST rotation-flagged emission of a cell carry, when it received both?
//
// Called (out of line, by the 3 % of the searches that need it) after the closure search found a stuck cell with
// arrivals of both flag values.  It replays the first two kick rounds with the arrivals separated by source and
// decides from the structure of the reference's queue (move_generation.py:337-488, SURVEY A.2):
//   * level 0 is the start fill F0 (rotation 0).  Its edge cells push their kick targets in (row, column,
//     direction) order, so the queue of level 1 starts with the targets e1, e2, e3 of the FIRST edge cell s* for
//     rotations 1, 2, 3 (condition C1: all three exist);
//   * level 1 therefore starts with the three fills B1, B2, B3 grown from e1, e2, e3, in that order.  If they cover
//     everything level 1 reaches (C2: the closure of ei equals the rotation's whole reach after the second fill),
//     no other fill happens in level 1 and the rest of its queue only emits;
//   * a stuck cell c of rotation R that is reached only later is unvisited during the whole of level 1: everything B1, B2,
//     B3 send there is pushed and popped in level 2 in push order (s ascending), group (c) below;
//   * for a stuck cell c of rotation R that was reached by then (c in F0 or B_R; not one of e1..e3), in time order:
//       (a) arrivals from B_s found while c is already visited (R = 0, or s > R) are emitted at once, s ascending;
//       (b) the arrivals pushed by F0 are popped afterwards;
//       (c) arrivals from B_s with s < R were pushed and are popped in level 2, s ascending — interleaved, in an order
//           this function does not know, with whatever later rounds emit at c;
//     inside one (source fill, direction) the emissions follow the source cells' (row, column) order, i.e. a fixed
//     priority of the kick indices: the used-last-kick arrival is the last one unless an arrival through a kick
//     whose source lies later in the scan ("hi") exists.
// Decided: no later-round arrival -> the last non-empty group of (c), (b), (a) in its known order; later-round
// arrivals of ONE flag value and no other value in group (c) -> that value.  Everything else (also a failed C1 / C2,
// the cells e1..e3) stays undecided and goes to the exact FIFO form.  Every search of the
// BASELINE sweep and of the adversarial test boards is compared with the oracle, decided or not.
// ---------------------------------------------------------------------------------------
template <class St>
__device__ __noinline__ bool t_order_decide(St& S, int lane, uint32_t VA, uint32_t VB, int slane, int sbit_index,
                                            uint32_t placedA, uint32_t placedB, uint32_t a0A, uint32_t a0B, bool snapped,
                                            uint32_t mixed_rots, uint32_t& ulkA, uint32_t& ulkB) {
    constexpr unsigned kAll = 0xffffffffu;
    // The closure search packs rotations (0 | 2, 1 | 3); this cold function works on (0 | 1, 2 | 3) pairs.
    swap_mid_halves(VA, VB);
    swap_mid_halves(placedA, placedB);
    swap_mid_halves(a0A, a0B);
    uint32_t oulkA = ulkA, oulkB = ulkB;
    swap_mid_halves(oulkA, oulkB);
    const uint32_t PA1 = lane >= 1 ? VA : 0u, PB1 = lane >= 1 ? VB : 0u;
    const uint32_t PA2 = PA1 & __shfl_up_sync(kAll, PA1, 1), PB2 = PB1 & __shfl_up_sync(kAll, PB1, 1);
    const uint32_t PA4 = PA2 & __shfl_up_sync(kAll, PA2, 2), PB4 = PB2 & __shfl_up_sync(kAll, PB2, 2);
    const uint32_t PA8 = PA4 & __shfl_up_sync(kAll, PA4, 4), PB8 = PB4 & __shfl_up_sync(kAll, PB4, 4);
    const uint32_t PA16 = PA8 & __shfl_up_sync(kAll, PA8, 8), PB16 = PB8 & __shfl_up_sync(kAll, PB8, 8);
    const uint32_t rVA = __brev(VA), rVB = __brev(VB);
    uint32_t dA = __shfl_down_sync(kAll, VA, 1), dB = __shfl_down_sync(kAll, VB, 1);
    if (lane == 31) { dA = 0u; dB = 0u; }
    const uint32_t innerA = dA & (VA << 1) & (VA >> 1), innerB = dB & (VB << 1) & (VB >> 1);
    auto fill = [&](uint32_t& A, uint32_t& B) {
        while (true) {
            const uint32_t a = hflood_r(A, VA, rVA), b = hflood_r(B, VB, rVB);
            A = fall_scan(a, PA1, PA2, PA4, PA8, PA16);
            B = fall_scan(b, PB1, PB2, PB4, PB8, PB16);
            if (!__any_sync(kAll, (A ^ a) | (B ^ b))) break;
        }
    };
    // one (source rotation s, direction kd) pass over the edge cells `ne`; arrivals by class into p0 = [N_hi | U << 16],
    // p1 = [N_lo] (rows indexed lane + 2); optionally the target of the single source cell (seed_lane, seed_bit)
    auto pass = [&](int s, int kd, uint32_t ne, uint32_t* p0, uint32_t* p1, int seed_lane, uint32_t seed_bit, int& hit_lane, uint32_t& hit_bit) {
        const int nrot = (s + kd + 1) & 3;
        const TrlKicks& K = c_kicks[0][s][kd];
        const int kn = K.n;
        const int lkx = K.k[kn - 1][0], lky = K.k[kn - 1][1];
        uint32_t rem = ne;
#pragma unroll 1
        for (int ki = 0; ki < kn; ++ki) {
            const int kx = K.k[ki][0], ky = K.k[ki][1];
            const uint32_t cand = rem & TRL_VV(S, nrot, lane + 2 - ky, kx + 2);
            rem &= ~cand;
            const bool is_u = kd != 1 && ki == kn - 1;
            const bool hi = kd != 1 && !is_u && (ky > lky || (ky == lky && kx < lkx));   // source later in the scan than the last kick's
            if (cand) {
                const uint32_t arr = kx >= 0 ? (cand << kx) : (cand >> -kx);
                if (is_u) atomicOr(&p0[lane + 2 - ky], arr << 16);
                else if (hi) atomicOr(&p0[lane + 2 - ky], arr);
                else atomicOr(&p1[lane + 2 - ky], arr);
            }
            if (seed_bit) {
                const bool hit = lane == seed_lane && (cand & seed_bit);
                if (__any_sync(kAll, hit)) { hit_lane = seed_lane - ky; hit_bit = kx >= 0 ? (seed_bit << kx) : (seed_bit >> -kx); }
            }
            if (!__any_sync(kAll, rem)) break;
        }
    };
    auto zero_planes = [&]() {
        __syncwarp();
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            S.tp[q][0][lane + 2] = 0u; S.tp[q][1][lane + 2] = 0u;
            if (lane < 4) { const int pad = lane < 2 ? lane : lane + 32; S.tp[q][0][pad] = 0u; S.tp[q][1][pad] = 0u; }
        }
        __syncwarp();
    };

    // later-round arrivals (rounds >= 2) per rotation of this lane's row: N | U << 16
    uint32_t late[4];
#pragma unroll
    for (int r = 0; r < 4; ++r)
        late[r] = snapped ? (S.fu[r][lane + 2] | ((((r & 2) ? a0B : a0A) >> (16 * (r & 1))) & 0xFFFFu)) : 0u;

    // ---- level 0: F0, its edge cells, the first of them ----
    uint32_t A0 = (lane == slane) ? (1u << sbit_index) : 0u, B0 = 0u;
    fill(A0, B0);
    const uint32_t F0 = A0 & 0xFFFFu;
    const uint32_t e0 = F0 & ~innerA;
    const uint32_t rows_with_edges = __ballot_sync(kAll, e0 != 0u);
    if (!rows_with_edges) { TRL_REASON(8); return false; }
    const int lstar = __ffs(rows_with_edges) - 1;
    const uint32_t e0star = __shfl_sync(kAll, e0, lstar);
    const uint32_t bstar = e0star & (0u - e0star);
    // ---- round 0: the kicks of F0 (target rotation kd + 1), classes kept for group (b), targets of s* ----
    zero_planes();
    int seed_lane[3] = {-1, -1, -1};
    uint32_t seed_bit[3] = {0u, 0u, 0u};
#pragma unroll
    for (int kd = 0; kd < 3; ++kd) pass(0, kd, e0, S.tp[kd + 1][0], S.tp[kd + 1][1], lstar, bstar, seed_lane[kd], seed_bit[kd]);
    __syncwarp();
    if (!seed_bit[0] || !seed_bit[1] || !seed_bit[2]) { TRL_REASON(9); return false; }   // C1
    uint32_t e0w0[4] = {0u, 0u, 0u, 0u}, e0w1[4] = {0u, 0u, 0u, 0u};
#pragma unroll
    for (int r = 1; r < 4; ++r) { e0w0[r] = S.tp[r][0][lane + 2]; e0w1[r] = S.tp[r][1][lane + 2]; }
    auto total = [](uint32_t w0, uint32_t w1) { return (w0 | (w0 >> 16) | w1) & 0xFFFFu; };
    // ---- level 1: the second fill, and the fills grown from e1, e2, e3 alone ----
    uint32_t A1 = A0 | (total(e0w0[1], e0w1[1]) << 16), B1 = total(e0w0[2], e0w1[2]) | (total(e0w0[3], e0w1[3]) << 16);
    fill(A1, B1);
    uint32_t SA = (lane == seed_lane[0]) ? (seed_bit[0] << 16) : 0u;
    uint32_t SB = ((lane == seed_lane[1]) ? seed_bit[1] : 0u) | ((lane == seed_lane[2]) ? (seed_bit[2] << 16) : 0u);
    fill(SA, SB);
    if (__any_sync(kAll, ((SA ^ A1) & 0xFFFF0000u) | (SB ^ B1))) { TRL_REASON(10); return false; }   // C2
    const uint32_t n1A = (A1 & ~innerA) & 0xFFFF0000u, n1B = B1 & ~innerB;              // edge cells of B1 | B2, B3
    // ---- per target rotation: the kicks of B1..B3 into it, by source, and the decision ----
    bool undecided = false;
    uint32_t ulk[4];
#pragma unroll 1
    for (int R = 0; R < 4; ++R) {
        if (!((mixed_rots >> R) & 1u)) {   // no cell of this rotation needs a decision: its flags are the union of the arrivals
            ulk[R] = (((R & 2) ? oulkB : oulkA) >> (16 * (R & 1))) & 0xFFFFu;
            continue;
        }
        zero_planes();
#pragma unroll 1
        for (int s = 1; s < 4; ++s) {
            if (s == R) continue;
            const int kd = (R - s - 1) & 3;
            const uint32_t ne = (((s & 2) ? n1B : n1A) >> (16 * (s & 1))) & 0xFFFFu;
            int hl = 0; uint32_t hb = 0u;
            if (__any_sync(kAll, ne)) pass(s, kd, ne, S.tp[s][0], S.tp[s][1], 0, 0u, hl, hb);
        }
        __syncwarp();
        const uint32_t placed = (((R & 2) ? placedB : placedA) >> (16 * (R & 1))) & 0xFFFFu;
        const uint32_t early = R == 0 ? F0 : ((((R & 2) ? SB : SA) >> (16 * (R & 1))) & 0xFFFFu);
        const uint32_t seed_cell = (R >= 1 && lane == seed_lane[R - 1]) ? seed_bit[R - 1] : 0u;
        uint32_t q_any = 0u, q_n = 0u, q_u = 0u, q_win = 0u;      // group (c): pushed by B_s, s < R
        uint32_t i_any = 0u, i_win = 0u;                          // group (a): emitted at once, s > R (all s for R = 0)
        uint32_t a_n = 0u, a_u = 0u, a_win = 0u;                  // cells reached later: every B_s pushes, s ascending
        uint32_t all_n = late[R] & 0xFFFFu, all_u = late[R] >> 16;
#pragma unroll
        for (int s = 1; s < 4; ++s) {
            const uint32_t w0 = S.tp[s][0][lane + 2], w1 = S.tp[s][1][lane + 2];
            const uint32_t nhi = w0 & 0xFFFFu, u = w0 >> 16, nlo = w1 & 0xFFFFu;
            const uint32_t any = nhi | u | nlo, win_u = u & ~nhi;
            all_n |= nhi | nlo; all_u |= u;
            a_n |= nhi | nlo; a_u |= u; a_win = (a_win & ~any) | win_u;
            if (R != 0 && s < R) { q_any |= any; q_n |= nhi | nlo; q_u |= u; q_win = (q_win & ~any) | win_u; }
            else { i_any |= any; i_win = (i_win & ~any) | win_u; }
        }
        const uint32_t b_nhi = e0w0[R] & 0xFFFFu, b_u = e0w0[R] >> 16, b_nlo = e0w1[R] & 0xFFFFu;   // group (b)
        const uint32_t b_any = b_nhi | b_u | b_nlo, b_win = b_u & ~b_nhi;
        all_n |= b_nhi | b_nlo; all_u |= b_u;
        const uint32_t l_n = late[R] & 0xFFFFu, l_u = late[R] >> 16, has_late = l_n | l_u;
        // a cell reached only after level 1 (not in F0 / B_R; it cannot have an arrival from F0 then) is unvisited during the
        // whole of level 1: everything B1..B3 send there is pushed and popped in level 2 in push order
        const uint32_t early_win = (q_any & q_win) | (~q_any & ((b_any & b_win) | (~b_any & i_win)));
        const uint32_t win = (early & early_win) | (~early & a_win);
        const uint32_t qn = (early & q_n) | (~early & a_n), qu = (early & q_u) | (~early & a_u);
        const uint32_t dec_u = (has_late & l_u & ~l_n & ~qn) | (~has_late & win);
        const uint32_t decided = (has_late & ((l_u & ~l_n & ~qn) | (l_n & ~l_u & ~qu))) | ~has_late;
        const uint32_t mixed = all_n & all_u & placed;
        const uint32_t suspect = seed_cell | (b_any & ~early);
        if (mixed & ~(decided & ~suspect)) undecided = true;
#ifdef TRL_MOVEGEN_STATS
        if (__any_sync(kAll, mixed & ~early)) TRL_REASON(11);
        if (__any_sync(kAll, mixed & suspect)) TRL_REASON(12);
        if (__any_sync(kAll, mixed & ~suspect & ~decided)) TRL_REASON(13);
#endif
        ulk[R] = ((all_u & ~mixed) | (dec_u & mixed)) & 0xFFFFu;
    }
    if (__any_sync(kAll, undecided)) { TRL_REASON(14); return false; }
    TRL_REASON(15);
    ulkA = ulk[0] | (ulk[2] << 16);
    ulkB = ulk[1] | (ulk[3] << 16);
    return true;
}

// Compile-time copy of c_minos (const.py:238-281) for the specialised validity rows: with the cell offsets as
// immediates a validity row is 4 x (SHF + LOP3) instead of 50 instructions of nibble extraction and selects.
constexpr uint32_t kMinos[7][4] = {
    {TRL_PK(0, 0, 1, 0, 1, 1, 2, 1), TRL_PK(1, 1, 1, 2, 2, 0, 2, 1), TRL_PK(0, 1, 1, 1, 1, 2, 2, 2), TRL_PK(0, 1, 0, 2, 1, 0, 1, 1)},
    {TRL_PK(0, 1, 1, 1, 2, 0, 2, 1), TRL_PK(1, 0, 1, 1, 1, 2, 2, 2), TRL_PK(0, 1, 0, 2, 1, 1, 2, 1), TRL_PK(0, 0, 1, 0, 1, 1, 1, 2)},
    {TRL_PK(0, 0, 0, 1, 1, 0, 1, 1), TRL_PK(0, 0, 0, 1, 1, 0, 1, 1), TRL_PK(0, 0, 0, 1, 1, 0, 1, 1), TRL_PK(0, 0, 0, 1, 1, 0, 1, 1)},
    {TRL_PK(0, 1, 1, 0, 1, 1, 2, 0), TRL_PK(1, 0, 1, 1, 2, 1, 2, 2), TRL_PK(0, 2, 1, 1, 1, 2, 2, 1), TRL_PK(0, 0, 0, 1, 1, 1, 1, 2)},
    {TRL_PK(0, 1, 1, 1, 2, 1, 3, 1), TRL_PK(2, 0, 2, 1, 2, 2, 2, 3), TRL_PK(0, 2, 1, 2, 2, 2, 3, 2), TRL_PK(1, 0, 1, 1, 1, 2, 1, 3)},
    {TRL_PK(0, 0, 0, 1, 1, 1, 2, 1), TRL_PK(1, 0, 1, 1, 1, 2, 2, 0), TRL_PK(0, 1, 1, 1, 2, 1, 2, 2), TRL_PK(0, 2, 1, 0, 1, 1, 1, 2)},
    {TRL_PK(0, 1, 1, 0, 1, 1, 2, 1), TRL_PK(1, 0, 1, 1, 1, 2, 2, 1), TRL_PK(0, 1, 1, 1, 1, 2, 2, 1), TRL_PK(0, 1, 1, 0, 1, 1, 1, 2)},
};

template <int TYPE, int R>
__device__ __forceinline__ uint32_t validity_row(const uint32_t (&e)[4]) {
    constexpr uint32_t mm = kMinos[TYPE][R];
    constexpr int c0 = mm & 15, r0 = (mm >> 4) & 15, c1 = (mm >> 8) & 15, r1 = (mm >> 12) & 15;
    constexpr int c2 = (mm >> 16) & 15, r2 = (mm >> 20) & 15, c3 = (mm >> 24) & 15, r3 = (mm >> 28) & 15;
    return 0x3FFFu & (e[r0] >> c0) & (e[r1] >> c1) & (e[r2] >> c2) & (e[r3] >> c3);
}

template <int TYPE>
__device__ __forceinline__ void validity_rows(const uint32_t (&e)[4], uint32_t (&v)[4]) {
    v[0] = validity_row<TYPE, 0>(e);
    v[1] = validity_row<TYPE, 1>(e);
    v[2] = validity_row<TYPE, 2>(e);
    v[3] = validity_row<TYPE, 3>(e);
}

// SPECIAL: kick passes of the non-I pieces with compile-time tables, twin passes packed (the closure kernels).
// T_ORDER: a T search with mixed flags goes through t_order_decide (St needs tsnap and tp).  Without it the search
// keeps no snapshot of the first two kick rounds and returns false ("deferred") for every T search with mixed flags:
// the sweep's first pass, which leaves the order analysis to a kernel of its own.
template <bool SPECIAL, bool T_ORDER, class St>
__device__ __forceinline__ bool search_piece_rows(St& S, const uint16_t* rows, int hi, int type, bool via_hold, uint32_t* mask) {
    const int lane = threadIdx.x & 31;
    const int sx = trl_spawn_x(type);
    const bool is_T = (type == P_T);
    // validity rows of the four rotations for this lane's row (move_generation.py:490-528)
    const int my = lane + kWin0;
    uint32_t e[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) e[k] = trl_empty_row(rows, my - 2 + k) << 2;
    uint32_t VA = 0u, VB = 0u;
    if (SPECIAL && TRL_ROWS_SPECIAL_V) {
        uint32_t v[4];
        switch (type) {
            case 0: validity_rows<0>(e, v); break;
            case 1: validity_rows<1>(e, v); break;
            case 2: validity_rows<2>(e, v); break;
            case 3: validity_rows<3>(e, v); break;
            case 4: validity_rows<4>(e, v); break;
            case 5: validity_rows<5>(e, v); break;
            default: validity_rows<6>(e, v); break;
        }
        VA = v[0] | (v[2] << 16);
        VB = v[1] | (v[3] << 16);
    } else {
#pragma unroll 1
    for (int r = 0; r < 4; ++r) {
        const uint32_t m4 = c_minos[type][r];
        uint32_t acc = 0x3FFFu;
#pragma unroll
        for (int m = 0; m < 4; ++m) {
            const uint32_t co = (m4 >> (8 * m)) & 15u, ro = (m4 >> (8 * m + 4)) & 15u;
            const uint32_t ek = ro == 0 ? e[0] : (ro == 1 ? e[1] : (ro == 2 ? e[2] : e[3]));
            acc &= ek >> co;
        }
        const uint32_t sh = acc << (16 * (r >> 1));
        if (r & 1) VB |= sh; else VA |= sh;
    }
    }
    // shared planes, row index lane + 2: validity << 2 for the kick tests, packed like VA / VB (TRL_VV); arrivals per
    // rotation (T: low half = flag clear, high half = used-last-kick)
    {
        const int pad = lane < 2 ? lane : lane + 32;
        S.vv[0][lane + 2] = VA << 2;
        S.vv[1][lane + 2] = VB << 2;
        if (lane < 4) { S.vv[0][pad] = 0u; S.vv[1][pad] = 0u; }
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            S.fu[r][lane + 2] = 0u;
            if (lane < 4) S.fu[r][pad] = 0u;
        }
    }
    // Player.hold_piece -> create_piece spawn test (player.py:37-44, move_generation.py:112-121): the spawn
    // cell (sx, 17) is validity row 19 = lane 7 of rotation 0
    const uint32_t v_spawn = __shfl_sync(0xffffffffu, VA, TRL_SPAWN_Y + 2 - kWin0);
    if (via_hold && !((v_spawn >> (sx + 2)) & 1u)) return true;
    // _set_starting_position (move_generation.py:164-180)
    const int slane = max(hi - (int)c_matrix_size[type], TRL_SPAWN_Y) + 2 - kWin0;   // 7..28
    const uint32_t vs = __shfl_sync(0xffffffffu, VA, slane);
    if (!((vs >> (sx + 2)) & 1u)) return true;                                   // :351-352

    // propagate masks of the fall scan
    const uint32_t PA1 = lane >= 1 ? VA : 0u, PB1 = lane >= 1 ? VB : 0u;
    const uint32_t PA2 = PA1 & __shfl_up_sync(0xffffffffu, PA1, 1), PB2 = PB1 & __shfl_up_sync(0xffffffffu, PB1, 1);
    const uint32_t PA4 = PA2 & __shfl_up_sync(0xffffffffu, PA2, 2), PB4 = PB2 & __shfl_up_sync(0xffffffffu, PB2, 2);
    const uint32_t PA8 = PA4 & __shfl_up_sync(0xffffffffu, PA4, 4), PB8 = PB4 & __shfl_up_sync(0xffffffffu, PB4, 4);
    const uint32_t PA16 = PA8 & __shfl_up_sync(0xffffffffu, PA8, 8), PB16 = PB8 & __shfl_up_sync(0xffffffffu, PB8, 8);
    const uint32_t rVA = __brev(VA), rVB = __brev(VB);
    // cells whose three neighbours (below, left, right) are all valid are no edge cells (:427-429)
    uint32_t dA = __shfl_down_sync(0xffffffffu, VA, 1), dB = __shfl_down_sync(0xffffffffu, VB, 1);
    if (lane == 31) { dA = 0u; dB = 0u; }
    const uint32_t innerA = dA & (VA << 1) & (VA >> 1), innerB = dB & (VB << 1) & (VB >> 1);
    __syncwarp();

#ifdef TRL_T_TRACE
    uint32_t* ttrace = nullptr;
    int tround = 0;
    if (is_T && g_t_trace) {
        unsigned slot_i = 0;
        if (lane == 0) slot_i = atomicAdd(&g_t_trace_n, 1u);
        slot_i = __shfl_sync(0xffffffffu, slot_i, 0);
        if (slot_i < g_t_trace_cap) {
            ttrace = g_t_trace + (size_t)slot_i * kTTraceWords;
            for (int k = lane; k < kTTraceWords; k += 32) ttrace[k] = 0u;
        }
    }
#endif
    const int tab = (type == P_I) ? 1 : 0;
    uint32_t RA = (lane == slane) ? (1u << (sx + 2)) : 0u, RB = 0u;
    uint32_t doneA = 0u, doneB = 0u;
    uint32_t a0A = 0u, a0B = 0u;   // arrivals by the in-place kick (0, 0): same lane, never the last kick
    int kick_rounds = 0;           // T: the arrivals of the first two kick rounds are set aside (t_order_decide)
    bool snapped = false;
    unsigned stat_4 = 0, stat_5 = 0;   // counted with -DTRL_MOVEGEN_STATS only
#ifdef TRL_MOVEGEN_STATS
    unsigned stat_2 = 0, stat_3 = 0, stat_6 = 0;
#endif
    while (true) {
        TRL_STAT(2);
        // ---- fill to the fix point (:409-425, :485-488), all rotations at once ----
        while (true) {
            TRL_STAT(3);
            // a set closed along rows to which the fall scan adds nothing is closed under both
            const uint32_t a0 = hflood_r(RA, VA, rVA), b0 = hflood_r(RB, VB, rVB);
            RA = fall_scan(a0, PA1, PA2, PA4, PA8, PA16);
            RB = fall_scan(b0, PB1, PB2, PB4, PB8, PB16);
            if (!__any_sync(0xffffffffu, (RA ^ a0) | (RB ^ b0))) break;
        }
        if (type == P_O) break;
        // ---- kicks of the edge cells reached since the last round (:427-483) ----
        const uint32_t EA = RA & ~innerA, EB = RB & ~innerB;
        const uint32_t nA = EA & ~doneA, nB = EB & ~doneB;
        doneA = EA; doneB = EB;
        if (!__any_sync(0xffffffffu, nA | nB)) break;
        if (SPECIAL && tab == 0) {
            // the eight passes with a twin as four packed passes, then the four 180-degree passes
            if (__any_sync(0xffffffffu, nA)) {
                kick_pass_pair<0, 0>(S, lane, nA, VA, VB, a0A, a0B, is_T, stat_4, stat_5);   // + (2, 2): target 1
                kick_pass_pair<0, 2>(S, lane, nA, VA, VB, a0A, a0B, is_T, stat_4, stat_5);   // + (2, 0): target 3
                kick_pass_wall<0, 0, 1>(S, lane, nA & 0xFFFFu, VA, VB, a0A, a0B, is_T, stat_4, stat_5);
                kick_pass_wall<0, 2, 1>(S, lane, nA >> 16, VA, VB, a0A, a0B, is_T, stat_4, stat_5);
            }
            const uint32_t n1 = nB & 0xFFFFu, n3 = nB >> 16;
            if (__any_sync(0xffffffffu, n1)) {
                kick_pass_pair<1, 2>(S, lane, n1 | (n1 << 16), VA, VB, a0A, a0B, is_T, stat_4, stat_5);   // + (1, 0): targets 0 | 2
                kick_pass_wall<0, 1, 1>(S, lane, n1, VA, VB, a0A, a0B, is_T, stat_4, stat_5);
            }
            if (__any_sync(0xffffffffu, n3)) {
                kick_pass_pair<3, 0>(S, lane, n3 | (n3 << 16), VA, VB, a0A, a0B, is_T, stat_4, stat_5);   // + (3, 2): targets 0 | 2
                kick_pass_wall<0, 3, 1>(S, lane, n3, VA, VB, a0A, a0B, is_T, stat_4, stat_5);
            }
        } else {
#pragma unroll 1
        for (int r = 0; r < 4; ++r) {
            const uint32_t X = (r & 1) ? nB : nA;
            const uint32_t ne = (r & 2) ? (X >> 16) : (X & 0xFFFFu);
            if (!__any_sync(0xffffffffu, ne)) continue;
            if (SPECIAL && TRL_ROWS_SPECIAL_I) {
                switch (r) {
                    case 0: kick_passes_wall<1, 0>(S, lane, ne, VA, VB, a0A, a0B, false, stat_4, stat_5); break;
                    case 1: kick_passes_wall<1, 1>(S, lane, ne, VA, VB, a0A, a0B, false, stat_4, stat_5); break;
                    case 2: kick_passes_wall<1, 2>(S, lane, ne, VA, VB, a0A, a0B, false, stat_4, stat_5); break;
                    default: kick_passes_wall<1, 3>(S, lane, ne, VA, VB, a0A, a0B, false, stat_4, stat_5); break;
                }
                continue;
            }
#pragma unroll 1
            for (int kd = 0; kd < 3; ++kd) {
                TRL_STAT(4);
                const int nrot = (r + kd + 1) & 3;
#ifdef TRL_T_TRACE
                uint32_t t_saved = 0u, t_a0A = a0A, t_a0B = a0B;
                if (ttrace) { t_saved = S.fu[nrot][lane + 2]; S.fu[nrot][lane + 2] = 0u; a0A = 0u; a0B = 0u; __syncwarp(); }
                struct TraceEnd {   // runs at every exit of this pass (continue / fall through)
                    St& S; uint32_t* tt; int nrot, kd, lane, round; uint32_t saved, sA, sB; uint32_t &a0A, &a0B;
                    __device__ ~TraceEnd() {
                        if (!tt) return;
                        __syncwarp();
                        const uint32_t d = S.fu[nrot][lane + 2];
                        const uint32_t k0 = (((nrot & 1) ? a0B : a0A) >> (16 * (nrot >> 1))) & 0xFFFFu;
                        if (round < 8) tt[((round * 4 + nrot) * 3 + kd) * 32 + lane] |= d | k0;
                        S.fu[nrot][lane + 2] = saved | d;
                        a0A |= sA; a0B |= sB;
                        __syncwarp();
                    }
                } trace_end{S, ttrace, nrot, kd, lane, tround, t_saved, t_a0A, t_a0B, a0A, a0B};
#endif
                // kick 0 is (0, 0) in every list (const.py:191-235): target = same cell of the new rotation
                const uint32_t Vn = ((nrot & 1) ? VB : VA) >> (16 * (nrot >> 1));
                const uint32_t c0 = ne & Vn;
                const uint32_t c0s = c0 << (16 * (nrot >> 1));
                if (nrot & 1) a0B |= c0s; else a0A |= c0s;
                uint32_t rem = ne & ~c0;
                if (!__any_sync(0xffffffffu, rem)) continue;
                const TrlKicks& K = c_kicks[tab][r][kd];
                const int kn = K.n;
                const uint32_t* vt = &S.vv[nrot & 1][lane + 2];
                const int vsh = 2 + 16 * (nrot >> 1);
                uint32_t* at = &S.fu[nrot][lane + 2];
#pragma unroll 1
                for (int ki = 1; ki < kn; ++ki) {
                    TRL_STAT(5);
                    const int kx = K.k[ki][0], ky = K.k[ki][1];
                    const uint32_t cand = rem & (vt[-ky] >> (kx + vsh));   // source bit ex <-> target bit ex + kx (TRL_VV)
                    rem &= ~cand;
                    if (cand) {
                        uint32_t arr = (cand << 4) >> (4 - kx);
                        if (is_T && kd != 1 && ki == kn - 1) arr <<= 16;   // nulk (:469)
                        atomicOr(&at[-ky], arr);
                    }
                    if (!__any_sync(0xffffffffu, rem)) break;            // every edge cell has found its kick
                }
            }
        }
        }
#ifdef TRL_T_TRACE
        ++tround;
#endif
        __syncwarp();
        // arrivals seed the next fill (a target is always a valid cell; T: low half = flag clear, high = set)
        {
            const uint32_t f0 = S.fu[0][lane + 2], f1 = S.fu[1][lane + 2], f2 = S.fu[2][lane + 2], f3 = S.fu[3][lane + 2];
#ifdef TRL_MOVEGEN_STATS
            if (is_T && stat_2 == 1) {   // mixed flags on a stuck cell after the first round of kicks?
                const uint32_t stA = VA & ~dA, stB = VB & ~dB;
                const uint32_t mA = (((f0 | a0A) & (f0 >> 16)) & 0xFFFFu) | ((((f2 << 16) | a0A) & f2) & 0xFFFF0000u);
                const uint32_t mB = (((f1 | a0B) & (f1 >> 16)) & 0xFFFFu) | ((((f3 << 16) | a0B) & f3) & 0xFFFF0000u);
                if (__any_sync(0xffffffffu, (mA & stA) | (mB & stB))) stat_6 = 1;
            }
#endif
            RA |= a0A | ((f0 | (f0 >> 16)) & 0xFFFFu) | ((f2 | (f2 >> 16)) << 16);
            RB |= a0B | ((f1 | (f1 >> 16)) & 0xFFFFu) | ((f3 | (f3 >> 16)) << 16);
            if constexpr (T_ORDER) {
                if (is_T && ++kick_rounds == 2) {   // later rounds accumulate from zero
                    S.tsnap[0][lane] = f0 | (a0A & 0xFFFFu); S.tsnap[1][lane] = f1 | (a0B & 0xFFFFu);
                    S.tsnap[2][lane] = f2 | (a0A >> 16); S.tsnap[3][lane] = f3 | (a0B >> 16);
                    S.fu[0][lane + 2] = 0u; S.fu[1][lane + 2] = 0u; S.fu[2][lane + 2] = 0u; S.fu[3][lane + 2] = 0u;
                    a0A = 0u; a0B = 0u;
                    snapped = true;
                    __syncwarp();
                }
            }
        }
    }
#ifdef TRL_MOVEGEN_STATS
    if (lane == 0) {
        atomicAdd(&g_fast_stats[2], (unsigned long long)stat_2); atomicAdd(&g_fast_stats[3], (unsigned long long)stat_3);
        atomicAdd(&g_fast_stats[4], (unsigned long long)stat_4); atomicAdd(&g_fast_stats[5], (unsigned long long)stat_5);
        atomicAdd(&g_fast_stats[6], (unsigned long long)stat_6);
    }
#endif
    // rows above the window would be needed: hand over to the exact form
    if (__any_sync(0xffffffffu, lane < 2 && (RA | RB))) return false;
    const uint32_t placedA = RA & ~dA, placedB = RB & ~dB;
#ifdef TRL_T_TRACE
    if (ttrace) {
        ttrace[8 * 4 * 3 * 32 + 0 * 32 + lane] = placedA & 0xFFFFu; ttrace[8 * 4 * 3 * 32 + 1 * 32 + lane] = placedB & 0xFFFFu;
        ttrace[8 * 4 * 3 * 32 + 2 * 32 + lane] = placedA >> 16; ttrace[8 * 4 * 3 * 32 + 3 * 32 + lane] = placedB >> 16;
        ttrace[8 * 4 * 3 * 32 + 4 * 32 + lane] = (uint32_t)rows[lane] | (lane < TRL_ROWS - 32 ? (uint32_t)rows[lane + 32] << 16 : 0u);
    }
#endif
    uint32_t flagA = 0u, flagB = 0u, ulkA = 0u, ulkB = 0u;   // T: some flagged emission / the last one used the last kick
    if (is_T) {
        uint32_t nA = a0A, nB = a0B, uA = 0u, uB = 0u;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            uint32_t fw = S.fu[r][lane + 2];
            if constexpr (T_ORDER) fw |= snapped ? S.tsnap[r][lane] : 0u;
            const uint32_t n = (fw & 0xFFFFu) << (16 * (r >> 1)), u = (fw >> 16) << (16 * (r >> 1));
            if (r & 1) { nB |= n; uB |= u; } else { nA |= n; uA |= u; }
        }
        flagA = nA | uA; flagB = nB | uB;
        ulkA = uA; ulkB = uB;
        const uint32_t mxA = nA & uA & placedA, mxB = nB & uB & placedB;
        const uint32_t mixed_rots = (__any_sync(0xffffffffu, mxA & 0xFFFFu) ? 1u : 0u) | (__any_sync(0xffffffffu, mxB & 0xFFFFu) ? 2u : 0u) |
                                    (__any_sync(0xffffffffu, mxA >> 16) ? 4u : 0u) | (__any_sync(0xffffffffu, mxB >> 16) ? 8u : 0u);
        if (mixed_rots) {
            // cells with both flag values: the order of emissions decides (:671-677)
            if constexpr (!T_ORDER) return false;
            else if (!t_order_decide(S, lane, VA, VB, slane, sx + 2, placedA, placedB, a0A, a0B, snapped, mixed_rots, ulkA, ulkB)) return false;
        }
    }
    // ---- _convert_placements_to_policy (move_generation.py:650-749): lane = row ----
    const int pbase = c_plane_base[type];
    const int nrot_planes = c_plane_nrot[type];
    const bool zsi = (type == P_Z || type == P_S || type == P_I);
    if (my < TRL_MAP_H - 1) {
        const int n_rot = (type == P_O) ? 1 : 4;
#pragma unroll 1
        for (int rot = 0; rot < n_rot; ++rot) {
            const uint32_t placed = (((rot & 1) ? placedB : placedA) >> (16 * (rot >> 1))) & 0xFFFFu;
            if (!placed) continue;
            int row = my - 2;
            uint32_t bits = placed;   // bit mx == policy column x + 2
            if (zsi) {                // rot 2 -> (rot 0, row + 1); rot 3 -> (rot 1, col - 1)
                if (rot == 2) row += 1;
                else if (rot == 3) bits >>= 1;
            }
            if (!is_T) {
                or_chunk(mask, pbase + rot % nrot_planes, row, bits & 0x7FFu);
            } else {
                const uint32_t f = (((rot & 1) ? flagB : flagA) >> (16 * (rot >> 1))) & placed;
                const uint32_t u = (((rot & 1) ? ulkB : ulkA) >> (16 * (rot >> 1))) & 0xFFFFu;
                or_chunk(mask, pbase + rot, row, (placed & ~f) & 0x7FFu);
                or_chunk(mask, pbase + 4 + rot, row, (f & ~u) & 0x7FFu);
                or_chunk(mask, pbase + 8 + rot, row, (f & u) & 0x7FFu);
            }
        }
    }
    return true;
}

// out-of-line copy for the kernels that also carry the FIFO form
__device__ __noinline__ bool search_piece_rows_call(PieceState& S, const uint16_t* rows, int type, bool via_hold, uint32_t* mask) {
    return search_piece_rows<false, true>(S, rows, first_block_row(rows, threadIdx.x & 31), type, via_hold, mask);
}

// One piece type of one call, executed by one converged warp.  Inlined with a constant `type` by the exact T kernel.
__device__ __forceinline__ void search_piece_fifo_body(PieceState& S, const uint16_t* rows, int type, bool via_hold, uint32_t* mask,
                                                       uint32_t& status, const uint32_t (*kpack)[4][3][2]) {
    const int lane = threadIdx.x & 31;
    uint32_t minos[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) minos[r] = c_minos[type][r];
    const int sx = trl_spawn_x(type);
    // Player.hold_piece -> create_piece spawn test (player.py:37-44, move_generation.py:112-121)
    if (via_hold && !trl_fits(rows, minos[0], sx, TRL_SPAWN_Y)) return;

    // _build_validity_maps (move_generation.py:490-528): lane = row
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        for (int my = lane; my < kVRows; my += 32) {
            S.vv[r][my] = (my < TRL_MAP_H) ? trl_valid_row(rows, minos[r], my) : 0u;
            S.fu[r][my] = 0u;
        }
    }
    // _set_starting_position (move_generation.py:164-180)
    int hi = TRL_ROWS;
    for (int i = lane; i < TRL_ROWS; i += 32)
        if (rows[i] & TRL_FULL_ROW) hi = min(hi, i);
    hi = __reduce_min_sync(0xffffffffu, hi);
    const int sy = max(hi - (int)c_matrix_size[type], TRL_SPAWN_Y);
    __syncwarp();
    if (!((S.vv[0][sy + 2] >> (sx + 2)) & 1u)) return;  // :351-352

    const bool is_T = (type == P_T);
    const bool rotates = (type != P_O);
    const int tab = (type == P_I) ? 1 : 0;

    uint32_t head = 0, tail = 1;
    if (lane == 0) S.fifo[0] = (uint16_t)fifo_pack(sx + 2, sy + 2, 0, 0, 0);
    __syncwarp();

    while (head != tail) {
        // ---- consume up to 32 queue entries: (A) emissions, find the first entry that fills ----
        const int n = min(32u, tail - head);
        const uint32_t e = (lane < n) ? S.fifo[(head + lane) % kFifoCap] : 0u;
        const int mx = e & 15, my = (e >> 4) & 63, rot = (e >> 10) & 3;
        const uint32_t bit = 1u << mx;
        const uint32_t w = S.vv[rot][my];
        const bool stuck = !(S.vv[rot][my + 1] & bit);
        const bool need = (lane < n) && !((w >> 16) & bit) && (w & bit);   // :397-398, :406-407
        const uint32_t m_need = __ballot_sync(0xffffffffu, need);
        const int first = m_need ? (__ffs(m_need) - 1) : 32;
        if (is_T) {
            // arrived by a kick and stuck: flagged emission BEFORE the visited test (:384-394)
            const bool emit = (lane < n) && (lane <= first) && ((e >> 12) & 1u) && stuck;
            const uint32_t m_emit = __ballot_sync(0xffffffffu, emit);
            if (m_emit) {
                const bool u = (e >> 13) & 1u;
                const uint32_t m_true = __ballot_sync(0xffffffffu, emit && u);
                if (m_true == 0u || m_true == m_emit) {
                    if (emit) flag_cell(&S.fu[rot][my], bit, u);
                } else if (emit) {   // mixed flags: the LAST emission of a cell wins (lane order = pop order)
                    const uint32_t grp = __match_any_sync(m_emit, e & 0xFFFu);
                    if ((31 - __clz(grp)) == lane) flag_cell(&S.fu[rot][my], bit, u);
                    else atomicOr(&S.fu[rot][my], bit);
                }
            }
        }
        head += (first < n) ? (uint32_t)(first + 1) : (uint32_t)n;
        __syncwarp();
        if (first >= n) continue;

        // ---- flood fill of rotation frot from (fmx, fmy), rows downward (:409-425, :485-488) ----
        const int frot = __shfl_sync(0xffffffffu, rot, first);
        const int fmy = __shfl_sync(0xffffffffu, my, first);
        uint32_t reach = __shfl_sync(0xffffffffu, bit, first);
        int fy = fmy;
        while (reach) {
            // one batch of at most 32 rows; lane l keeps the filled cells of row base + l
            const int base = fy;
            uint32_t myr = 0;
            uint32_t cur = S.vv[frot][fy];
            while (reach && fy < base + 32) {
                const uint32_t open = cur & ~(cur >> 16) & 0xFFFFu;
                const uint32_t r = hflood(reach, open);
                if (lane == fy - base) { myr = r; S.vv[frot][fy] = cur | (r << 16); }   // :425
                const uint32_t nxt = S.vv[frot][fy + 1];
                reach = r & nxt & ~(nxt >> 16);
                cur = nxt;
                ++fy;
            }
            const int nrows = fy - base;
            __syncwarp();
            if (!rotates) continue;

            // ---- kicks of every edge cell of the batch: lane = row, bit = column (:427-483) ----
            const int ky_row = base + lane;
            uint32_t edges = 0;
            if (lane < nrows) {
                const uint32_t vr = S.vv[frot][ky_row] & 0xFFFFu, nx = S.vv[frot][ky_row + 1] & 0xFFFFu;
                edges = (myr & ~nx) | (myr & ~(vr << 1)) | (myr & ~(vr >> 1));
            }
            // ---- small fills (the common case: caves reached by a kick): lane = (edge cell, direction) ----
            // The bit-parallel pass below costs ~500 instructions whatever the fill size; with at most 10
            // edge cells every (cell, direction) pair gets its own lane and walks its kick list serially.
            {
                const int ecnt = __popc(edges);
                int eincl = ecnt;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const int t = __shfl_up_sync(0xffffffffu, eincl, d);
                    if (lane >= d) eincl += t;
                }
                const int etotal = __shfl_sync(0xffffffffu, eincl, 31);
                if (etotal == 0) continue;
                if (etotal <= 10 && nrows <= 8) {
                    const int eoff = eincl - ecnt;
                    const int q = lane / 3, kd = lane - 3 * q;
                    int erow = 0, eq = 0;
                    uint32_t emask = 0;
                    for (int r = 0; r < nrows; ++r) {
                        const int o = __shfl_sync(0xffffffffu, eoff, r), c = __shfl_sync(0xffffffffu, ecnt, r);
                        const uint32_t ed = __shfl_sync(0xffffffffu, edges, r);
                        if (q >= o && q < o + c) { erow = r; emask = ed; eq = q - o; }
                    }
                    const bool ev = (q < etotal) && (kd < 3) && (lane < 30);
                    for (int t = 0; t < eq; ++t) emask &= emask - 1;
                    const int ex = __ffs(emask) - 1, fy0 = base + erow;
                    const int nrot = (frot + kd + 1) & 3;
                    int res = 0, tx = 0, ty = 0, nulk = 0;   // res: 1 = queue the target, 2 = flagged emission at once
                    if (ev) {
                        const uint32_t px = (*kpack)[frot][kd][0], py = (*kpack)[frot][kd][1];
                        const int kn = c_kicks[tab][frot][kd].n;
                        for (int ki = 0; ki < kn; ++ki) {
                            tx = ex + (int)((px >> (4 * ki)) & 15u) - 2;
                            ty = fy0 - ((int)((py >> (4 * ki)) & 15u) - 2);
                            if ((unsigned)tx >= (unsigned)TRL_MAP_W || (unsigned)ty >= (unsigned)TRL_MAP_H) continue;
                            const uint32_t tw = S.vv[nrot][ty];
                            if (!((tw >> tx) & 1u)) continue;
                            if (ty < 2) break;                                   // origin y < 0: direction abandoned
                            if (!((tw >> (16 + tx)) & 1u)) res = 1;
                            else if (!((S.vv[nrot][ty + 1] >> tx) & 1u)) res = 2;
                            nulk = (is_T && kd != 1 && ki == kn - 1) ? 1 : 0;
                            break;                                               // first successful kick wins
                        }
                        if (res == 1 && !is_T) {   // already queued? (order / multiplicity only matter for T)
                            if (atomicOr(&S.fu[nrot][ty], 1u << tx) & (1u << tx)) res = 0;
                        }
                    }
                    const uint32_t pm = __ballot_sync(0xffffffffu, res == 1);
                    const int total = __popc(pm);
                    if ((tail - head) + (uint32_t)total > (uint32_t)c_fifo_limit) status |= TRL_ST_QUEUE_OVERFLOW;
                    else {
                        if (res == 1)   // lane order = (row, column, direction) = the reference's queue order
                            S.fifo[(tail + (uint32_t)__popc(pm & ((1u << lane) - 1u))) % kFifoCap] = (uint16_t)fifo_pack(tx, ty, nrot, 1, nulk);
                        tail += (uint32_t)total;
                    }
                    if (is_T) {
                        const uint32_t im = __ballot_sync(0xffffffffu, res == 2);
                        if (im) {
                            const uint32_t mt = __ballot_sync(0xffffffffu, res == 2 && nulk);
                            if (mt == 0u || mt == im) {
                                if (res == 2) flag_cell(&S.fu[nrot][ty], 1u << tx, nulk != 0);
                            } else if (res == 2) {   // mixed flags: the last emission of a cell wins
                                const uint32_t grp = __match_any_sync(im, (uint32_t)(tx | (ty << 4) | (nrot << 10)));
                                if ((31 - __clz(grp)) == lane) flag_cell(&S.fu[nrot][ty], 1u << tx, nulk != 0);
                                else atomicOr(&S.fu[nrot][ty], 1u << tx);
                            }
                        }
                    }
                    __syncwarp();
                    continue;
                }
            }
            uint32_t Pu[3] = {0, 0, 0}, Im[3] = {0, 0, 0};      // sources whose kick pushes / emits at once
            uint32_t k0[3] = {0, 0, 0}, k1[3] = {0, 0, 0}, k2[3] = {0, 0, 0};   // bit planes of the winning kick index
#pragma unroll
            for (int kd = 0; kd < 3; ++kd) {
                const int nrot = (frot + kd + 1) & 3;
                const TrlKicks& K = c_kicks[tab][frot][kd];
                const int kn = K.n;
                uint32_t rem = edges;
#pragma unroll
                for (int ki = 0; ki < 6; ++ki) {
                    if (ki >= kn) break;
                    const int kx = K.k[ki][0], ty = ky_row - K.k[ki][1];
                    const bool in = (unsigned)ty < (unsigned)TRL_MAP_H;
                    const uint32_t tw = in ? S.vv[nrot][ty] : 0u;
                    const uint32_t tn = in ? S.vv[nrot][ty + 1] : 0u;
                    // source bit ex <-> target bit ex + kx
                    const uint32_t tv = kx >= 0 ? ((tw & 0xFFFFu) >> kx) : ((tw & 0xFFFFu) << -kx);
                    const uint32_t cand = rem & tv & 0x3FFFu;       // first valid kick of these sources
                    rem &= ~cand;
                    if (!__any_sync(0xffffffffu, rem | cand)) break; // every edge cell of the batch has found its kick
                    if (ty < 2 || !cand) continue;                   // origin y < 0: direction abandoned (:463-464)
                    const uint32_t tvis = kx >= 0 ? ((tw >> 16) >> kx) : ((tw >> 16) << -kx);
                    const uint32_t tfree = kx >= 0 ? ((tn & 0xFFFFu) >> kx) : ((tn & 0xFFFFu) << -kx);
                    uint32_t pu = cand & ~tvis;
                    const uint32_t im = cand & tvis & ~tfree;
                    if (!is_T) {
                        // Only T depends on the order and multiplicity of queue entries (its flagged
                        // emissions).  For the other pieces a target that is already queued need not be
                        // queued again: fu's low half doubles as the "pending" plane.
                        const uint32_t pend = in ? S.fu[nrot][ty] : 0u;
                        pu &= ~(kx >= 0 ? ((pend & 0xFFFFu) >> kx) : ((pend & 0xFFFFu) << -kx));
                        if (pu) atomicOr(&S.fu[nrot][ty], kx >= 0 ? (pu << kx) : (pu >> -kx));
                    }
                    Pu[kd] |= pu;
                    Im[kd] |= im;
                    const uint32_t s = pu | im;
                    if (ki & 1) k0[kd] |= s;
                    if (ki & 2) k1[kd] |= s;
                    if (ki & 4) k2[kd] |= s;
                }
            }
            // ---- append the pushes in reference order: row, column LSB->MSB, direction ----
            const int cnt = __popc(Pu[0]) + __popc(Pu[1]) + __popc(Pu[2]);
            int incl = cnt;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, incl, d);
                if (lane >= d) incl += t;
            }
            const int total = __shfl_sync(0xffffffffu, incl, 31);
            const bool room = (tail - head) + (uint32_t)total <= (uint32_t)c_fifo_limit;
            if (!room) status |= TRL_ST_QUEUE_OVERFLOW;
            const uint32_t any_im = is_T ? __ballot_sync(0xffffffffu, (Im[0] | Im[1] | Im[2]) != 0u) : 0u;
            if ((total && room) || any_im) {
                // per-lane pass over this row's events in (column, direction) order
                uint32_t off = tail + (uint32_t)(incl - cnt);
                uint32_t ev = Pu[0] | Pu[1] | Pu[2] | (is_T ? (Im[0] | Im[1] | Im[2]) : 0u);
                bool has_t = false, has_f = false;
                // first pass: pushes (and the flag mix of the immediate emissions)
                while (ev) {
                    const int ex = __ffs(ev) - 1;
                    ev &= ev - 1;
#pragma unroll
                    for (int kd = 0; kd < 3; ++kd) {
                        const bool p = (Pu[kd] >> ex) & 1u, i = (Im[kd] >> ex) & 1u;
                        if (!(p || i)) continue;
                        const int ki = ((k0[kd] >> ex) & 1u) | (((k1[kd] >> ex) & 1u) << 1) | (((k2[kd] >> ex) & 1u) << 2);
                        const int kn = c_kicks[tab][frot][kd].n;
                        const int nulk = (is_T && kd != 1 && ki == kn - 1) ? 1 : 0;
                        if (p) {
                            if (room) {
                                const int kx = (int)(((*kpack)[frot][kd][0] >> (4 * ki)) & 15u) - 2;
                                const int ky = (int)(((*kpack)[frot][kd][1] >> (4 * ki)) & 15u) - 2;
                                S.fifo[off % kFifoCap] = (uint16_t)fifo_pack(ex + kx, ky_row - ky, (frot + kd + 1) & 3, 1, nulk);
                                ++off;
                            }
                        } else if (nulk) has_t = true;
                        else has_f = true;
                    }
                }
                if (room) tail += (uint32_t)total;
                if (any_im) {
                    // immediate flagged emissions: target already visited and stuck (:471-479)
                    const bool mixed = __any_sync(0xffffffffu, has_t) && __any_sync(0xffffffffu, has_f);
                    const int l_end = mixed ? nrows : 1;
                    for (int l = 0; l < l_end; ++l) {           // mixed flags: rows strictly in order
                        if (mixed && lane != l) { __syncwarp(); continue; }
                        uint32_t iv = Im[0] | Im[1] | Im[2];
                        while (iv) {
                            const int ex = __ffs(iv) - 1;
                            iv &= iv - 1;
#pragma unroll
                            for (int kd = 0; kd < 3; ++kd) {
                                if (!((Im[kd] >> ex) & 1u)) continue;
                                const int ki = ((k0[kd] >> ex) & 1u) | (((k1[kd] >> ex) & 1u) << 1) | (((k2[kd] >> ex) & 1u) << 2);
                                const int kn = c_kicks[tab][frot][kd].n;
                                const bool nulk = (kd != 1 && ki == kn - 1);
                                const int kx = (int)(((*kpack)[frot][kd][0] >> (4 * ki)) & 15u) - 2;
                                const int ky = (int)(((*kpack)[frot][kd][1] >> (4 * ki)) & 15u) - 2;
                                flag_cell(&S.fu[(frot + kd + 1) & 3][ky_row - ky], 1u << (ex + kx), nulk);
                            }
                        }
                        __syncwarp();
                    }
                }
            }
            __syncwarp();
        }
    }
    __syncwarp();

    // ---- _convert_placements_to_policy (move_generation.py:650-749): lane = row ----
    const int pbase = c_plane_base[type];
    const int nrot_planes = c_plane_nrot[type];
    const bool zsi = (type == P_Z || type == P_S || type == P_I);
    for (int rot = 0; rot < 4; ++rot) {
        if (type == P_O && rot > 0) break;
        for (int my = 2 + lane; my < TRL_MAP_H - 1; my += 32) {
            const uint32_t wv = S.vv[rot][my];
            const uint32_t placed = (wv >> 16) & ~S.vv[rot][my + 1] & 0xFFFFu;
            if (!placed) continue;
            int row = my - 2;
            uint32_t bits = placed;  // bit mx == policy column x + 2
            if (zsi) {               // rot 2 -> (rot 0, row + 1); rot 3 -> (rot 1, col - 1)
                if (rot == 2) row += 1;
                else if (rot == 3) bits >>= 1;
            }
            if (!is_T) {
                or_chunk(mask, pbase + rot % nrot_planes, row, bits & 0x7FFu);
            } else {
                const uint32_t fw = S.fu[rot][my];
                const uint32_t f = fw & placed, u = fw >> 16;
                or_chunk(mask, pbase + rot, row, (placed & ~f) & 0x7FFu);
                or_chunk(mask, pbase + 4 + rot, row, (f & ~u) & 0x7FFu);
                or_chunk(mask, pbase + 8 + rot, row, (f & u) & 0x7FFu);
            }
        }
    }
}

__device__ __noinline__ void search_piece_fifo(PieceState& S, const uint16_t* rows, int type, bool via_hold, uint32_t* mask,
                                              uint32_t& status, const uint32_t (*kpack)[4][3][2]) {
    search_piece_fifo_body(S, rows, type, via_hold, mask, status, kpack);
}

// One piece type of one call: the row-parallel closure form, or the exact FIFO form where that one cannot decide.
__device__ __forceinline__ void search_piece_warp(PieceState& S, const uint16_t* rows, int type, bool via_hold, uint32_t* mask,
                                                  uint32_t& status, const uint32_t (*kpack)[4][3][2], bool exact_only = false) {
    if (!exact_only && c_fast_path && c_fifo_limit == kFifoCap) {
        const bool done = search_piece_rows_call(S, rows, type, via_hold, mask);
        if ((threadIdx.x & 31) == 0) atomicAdd(&g_fast_stats[done ? 0 : 1], 1ull);
        if (done) return;
        __syncwarp();
    }
    search_piece_fifo(S, rows, type, via_hold, mask, status, kpack);
}

// Ascending move list (= np.argwhere order, ai.py:1016-1024) of the call's shared-memory mask; the list position of a
// word's first set bit is lbase[w / 12] + woff[w].  Lane l takes the words l, l + 32, ... (the set bits of a call sit in
// a few runs of consecutive words — a policy plane is 13.4 words — so consecutive words per lane serialise on one or two
// lanes: measured 1.3 active lanes), and visits only its non-empty ones.  Kept out of line.
__device__ __noinline__ void write_move_list(const CallState& C, int lane, uint16_t* mv, int cap) {
    uint32_t nz = 0u;
#pragma unroll
    for (int j = 0; j < 12; ++j) {
        const int w = lane + 32 * j;
        if (w < TRL_MASK_WORDS && C.mask[w]) nz |= 1u << j;
    }
    while (nz) {
        const int j = __ffs(nz) - 1;
        nz &= nz - 1;
        const int w = lane + 32 * j;
        uint32_t m = C.mask[w];
        int pos = (int)C.lbase[(w * 683) >> 13] + (int)C.woff[w];   // (w * 683) >> 13 == w / 12 for w < 2040
        while (m) {
            const int b = __ffs(m) - 1;
            m &= m - 1;
            if (pos < cap) mv[pos] = (uint16_t)(w * 32 + b);
            ++pos;
        }
    }
}

// Outputs of one call, written by ONE warp from the call's shared-memory mask: the coalesced bit-packed
// mask, the ascending move list, the count and the status word.
template <int MODE = 0>   // 0: decided at run time; 1: no move list (code of the list writer dropped); 2: move list wanted
__device__ __forceinline__ void write_call_outputs(CallState& C, int i, int lane, uint32_t* __restrict__ mask_bits,
                                                   uint16_t* __restrict__ moves, int moves_cap,
                                                   uint16_t* __restrict__ n_moves, uint32_t* __restrict__ status,
                                                   uint16_t* __restrict__ compact, unsigned long long compact_cap,
                                                   unsigned long long* __restrict__ compact_total,
                                                   unsigned long long* __restrict__ offsets) {
    if (C.skip) {
        if (lane == 0) {
            if (n_moves) n_moves[i] = 0;
            if (status) status[i] = 0;
            if (compact) offsets[i] = 0;
        }
        return;
    }
    // lane owns 12 consecutive words (the last lanes fewer): counts -> prefix -> ordered writes
    const int w0 = lane * 12;
    const bool want_list = MODE == 0 ? (compact != nullptr || moves != nullptr) : (MODE == 2);
    int cnt = 0;
    uint32_t* gm = mask_bits ? mask_bits + (size_t)i * TRL_MASK_WORDS : nullptr;
#pragma unroll 1
    for (int k = 0; k < 12; ++k) {
        const int w2 = w0 + k;
        if (w2 < TRL_MASK_WORDS) {
            if (want_list) C.woff[w2] = (uint16_t)cnt;
            cnt += __popc(C.mask[w2]);
        }
        const int w3 = k * 32 + lane;                       // coalesced copy of the mask
        if (gm && w3 < TRL_MASK_WORDS) gm[w3] = C.mask[w3];
    }
    int incl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += t;
    }
    const int total = __shfl_sync(0xffffffffu, incl, 31);
    uint32_t st = C.status;
    if (want_list) {
        C.lbase[lane] = (uint16_t)(incl - cnt);
        __syncwarp();
    }
    if (want_list && compact) {
        unsigned long long off = 0;
        if (lane == 0) off = atomicAdd(compact_total, (unsigned long long)total);
        off = __shfl_sync(0xffffffffu, off, 0);
        if (off + (unsigned long long)total > compact_cap) st |= TRL_ST_MOVES_TRUNC;
        else write_move_list(C, lane, compact + off, 0x7fffffff);
        if (lane == 0) offsets[i] = off;
    }
    if (want_list && moves) {
        write_move_list(C, lane, moves + (size_t)i * moves_cap, moves_cap);
        if (total > moves_cap) st |= TRL_ST_MOVES_TRUNC;
    }
    if (lane == 0) {
        if (n_moves) n_moves[i] = (uint16_t)total;
        if (status) status[i] = st;
    }
}

// Zero the call's mask with one warp: 91 128-bit stores.
__device__ __forceinline__ void zero_mask(CallState& C, int lane) {
    static_assert((TRL_MASK_WORDS + 2) % 4 == 0, "mask is a whole number of 16-byte words");
    uint4* m4 = reinterpret_cast<uint4*>(C.mask);
#pragma unroll
    for (int k = lane; k < (TRL_MASK_WORDS + 2) / 4; k += 32) m4[k] = make_uint4(0u, 0u, 0u, 0u);
}

// Stage one call into the warp's CallState: zeroed mask, board rows, piece types (c, a) and the skip flag.
__device__ __forceinline__ void stage_call(CallState& C, int i, int lane, const uint16_t* __restrict__ boards,
                                           const uint8_t* __restrict__ cur, const uint8_t* __restrict__ alt,
                                           const TrlGame* __restrict__ games, const int32_t* __restrict__ index,
                                           int& c, int& a, int& skip) {
    c = TRL_NONE; a = TRL_NONE; skip = 0;
    if (games) {
        const int gi = index ? index[i] : i;
        if (gi < 0) skip = 1;
        else {
            const TrlPlayer& p = games[gi].players[games[gi].turn & 1];
            for (int r = lane; r < TRL_ROWS; r += 32) C.rows[r] = p.rows[r];
            c = p.piece;
            a = (p.held != TRL_NONE) ? p.held : (p.qlen > 0 ? p.queue[0] : TRL_NONE);
        }
    } else {
        for (int r = lane; r < TRL_ROWS; r += 32) C.rows[r] = boards[(size_t)i * TRL_ROWS + r];
        c = cur[i];
        a = alt[i];
    }
    if (c > 6 && c != TRL_NONE) c = TRL_NONE;
    if (a > 6 && a != TRL_NONE) a = TRL_NONE;
    if (lane == 0) {
        C.cur = c; C.alt = a; C.skip = skip;
        C.status = (!skip && c == TRL_NONE && a == TRL_NONE) ? TRL_ST_NO_PIECE : 0u;
    }
}

__global__ void __launch_bounds__(kWarps * 32)
movegen_warp_kernel(const uint16_t* __restrict__ boards, const uint8_t* __restrict__ cur,
                    const uint8_t* __restrict__ alt, const TrlGame* __restrict__ games,
                    const int32_t* __restrict__ index, int n, uint32_t* __restrict__ mask_bits,
                    uint16_t* __restrict__ moves, int moves_cap, uint16_t* __restrict__ n_moves,
                    uint32_t* __restrict__ status,
                    // compact output (optional): the lists of all calls packed without padding; call i owns
                    // compact[offsets[i] .. offsets[i] + n_moves[i]) (segments are handed out with an atomic
                    // bump allocator, so their order in the buffer is arbitrary; each list is ascending)
                    uint16_t* __restrict__ compact, unsigned long long compact_cap,
                    unsigned long long* __restrict__ compact_total, unsigned long long* __restrict__ offsets,
                    // clean-up mode (second pass of the throughput form): only the calls call_list[0 .. *call_count),
                    // every search through the exact FIFO form, a fixed grid striding over the list
                    const int32_t* __restrict__ call_list, const uint32_t* __restrict__ call_count) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    PieceState* ps = reinterpret_cast<PieceState*>(smem_raw);
    CallState* cs = reinterpret_cast<CallState*>(smem_raw + sizeof(PieceState) * kWarps);
    __shared__ uint32_t s_kpack[2][4][3][2];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int slot = warp >> 1, which = warp & 1;
    CallState& C = cs[slot];

    if (tid < 24) {   // kick offsets packed 4 bits each (+2) so a lane can index them by kick number
        const int t = tid / 12, r = (tid / 3) % 4, kd = tid % 3;
        const TrlKicks& K = c_kicks[t][r][kd];
        uint32_t px = 0, py = 0;
        for (int ki = 0; ki < K.n; ++ki) {
            px |= (uint32_t)(K.k[ki][0] + 2) << (4 * ki);
            py |= (uint32_t)(K.k[ki][1] + 2) << (4 * ki);
        }
        s_kpack[t][r][kd][0] = px;
        s_kpack[t][r][kd][1] = py;
    }
    const int n_items = call_list ? (int)call_count[0] : n;
    for (int base = blockIdx.x * kCallsPerBlock; base < n_items; base += gridDim.x * kCallsPerBlock) {
        const int j = base + slot;
        const bool live = j < n_items;
        const int i = live ? (call_list ? call_list[j] : j) : 0;
        // ---- stage the call: board rows, piece types, zeroed mask (both warps of the call) ----
        if (live) {
            for (int w2 = which * 32 + lane; w2 < TRL_MASK_WORDS + 2; w2 += 64) C.mask[w2] = 0u;
            if (which == 0) {
                int c, a, skip;
                stage_call(C, i, lane, boards, cur, alt, games, index, c, a, skip);
            }
        }
        __syncthreads();

        if (live && !C.skip) {
            const int c = C.cur, a = C.alt;
            uint32_t st = 0;
            // warp 0 of the call: the current piece; warp 1: the hold-or-next piece (de-duplicated, :103-105)
            const int type = which ? a : c;
            if (type != TRL_NONE && !(which && a == c))
                search_piece_warp(ps[warp], C.rows, type, which != 0, C.mask, st, &s_kpack[type == P_I ? 1 : 0], call_list != nullptr);
            st = __reduce_or_sync(0xffffffffu, st);
            if (st && lane == 0) atomicOr(&C.status, st);
        }
        __syncthreads();

        // ---- outputs: coalesced mask, ascending move list (= argwhere order), count, status ----
        if (live && which == 0)
            write_call_outputs(C, i, lane, mask_bits, moves, moves_cap, n_moves, status, compact, compact_cap, compact_total, offsets);
        __syncthreads();   // the slot is staged again by the next trip
    }
}

// ---------------------------------------------------------------------------------------
// Throughput form: ONE warp per call, both piece searches back to back on the same warp.
//
// In movegen_warp_kernel the two warps of a call search different piece types (an O search is a
// fraction of a T search) and then meet at a barrier: ncu counted 4.2 of the 8 warps of a scheduler
// parked at that barrier per issued instruction, i.e. half of the resident warps hid no latency.  For
// multi-million-call sweeps latency of a single call is irrelevant, so here a warp owns the whole call
// (4.5 KB of shared memory: one PieceState re-used by the two searches + the CallState), nothing in the
// kernel waits for another warp after the kick tables are staged, and a finished warp's slot is refilled by
// the next block instead of idling until the slowest search of a 16-warp block ends.
// ---------------------------------------------------------------------------------------
constexpr int kSoloWarps = 4;

struct SoloState {
    PieceState P;
    CallState C;
};

__global__ void __launch_bounds__(kSoloWarps * 32, 8)
movegen_solo_kernel(const uint16_t* __restrict__ boards, const uint8_t* __restrict__ cur,
                    const uint8_t* __restrict__ alt, const TrlGame* __restrict__ games,
                    const int32_t* __restrict__ index, int n, uint32_t* __restrict__ mask_bits,
                    uint16_t* __restrict__ moves, int moves_cap, uint16_t* __restrict__ n_moves,
                    uint32_t* __restrict__ status, uint16_t* __restrict__ compact, unsigned long long compact_cap,
                    unsigned long long* __restrict__ compact_total, unsigned long long* __restrict__ offsets,
                    // clean-up mode (the legacy route of the pass form): only the calls call_list[0 .. *call_count),
                    // T searches straight through the exact FIFO form, a fixed grid striding over the list
                    const int32_t* __restrict__ call_list, const uint32_t* __restrict__ call_count) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    __shared__ uint32_t s_kpack[2][4][3][2];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    SoloState& S = reinterpret_cast<SoloState*>(smem_raw)[warp];
    CallState& C = S.C;
    if (tid < 24) {
        const int t = tid / 12, r = (tid / 3) % 4, kd = tid % 3;
        const TrlKicks& K = c_kicks[t][r][kd];
        uint32_t px = 0, py = 0;
        for (int ki = 0; ki < K.n; ++ki) {
            px |= (uint32_t)(K.k[ki][0] + 2) << (4 * ki);
            py |= (uint32_t)(K.k[ki][1] + 2) << (4 * ki);
        }
        s_kpack[t][r][kd][0] = px;
        s_kpack[t][r][kd][1] = py;
    }
    __syncthreads();   // kick tables staged; the only block-wide barrier
    const int n_items = call_list ? (int)call_count[0] : n;
#pragma unroll 1
    for (int j = blockIdx.x * kSoloWarps + warp; j < n_items; j += gridDim.x * kSoloWarps) {
        const int i = call_list ? call_list[j] : j;
        int c, a, skip;
        zero_mask(C, lane);
        stage_call(C, i, lane, boards, cur, alt, games, index, c, a, skip);
        __syncwarp();
        if (!skip) {
            uint32_t st = 0;
            // the current piece, then the hold-or-next piece (de-duplicated, move_generation.py:103-105)
#pragma unroll 1
            for (int which = 0; which < 2; ++which) {
                const int type = which ? a : c;
                if (type == TRL_NONE || (which && a == c)) continue;
                search_piece_warp(S.P, C.rows, type, which != 0, C.mask, st, &s_kpack[type == P_I ? 1 : 0],
                                  call_list != nullptr && type == P_T);
                __syncwarp();
            }
            st = __reduce_or_sync(0xffffffffu, st);
            if (st && lane == 0) C.status |= st;
            __syncwarp();
        }
        write_call_outputs(C, i, lane, mask_bits, moves, moves_cap, n_moves, status, compact, compact_cap, compact_total, offsets);
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------
// Throughput form, in passes: the row-parallel closure search alone in a small kernel, then the T order analysis
// and the exact T search for the few calls whose T search it deferred.
//
//   pass 1  movegen_rows_kernel: both piece searches through the closure form without the T order analysis
//           (T_ORDER = false): 48 registers, no FIFO code, no cold analysis code, a loop nest small enough to stay
//           in the instruction caches (the one-kernel forms lose a quarter of their issue slots to instruction
//           fetch).  A T search with mixed flags, or one that climbed out of the row window, is DEFERRED: the other
//           piece is still searched, the call's partial mask (the other piece's bits only) is stored and the call
//           appended to the deferred list;
//   pass 2  movegen_t_order_kernel: the T search alone, closure form with the order analysis (t_order_decide).
//           Decided: merged into the partial mask, outputs written.  Undecided: appended to the exact list;
//   pass 3  movegen_t_exact_kernel: the exact FIFO search specialised for T (piece and kick table fixed at compile
//           time; no closure form, no other piece), merged into the partial mask, outputs written;
//   legacy  movegen_solo_kernel in clean-up mode: calls whose NON-T search is undecided (a climb out of the row
//           window) or whose partial mask found no room redo the whole call as before (T straight through the FIFO
//           form).  It is launched every sweep and exits at once when its list is empty.
// Only the pass that finishes a call writes n_moves, status and the move list.  The partial mask lives in the call's
// own mask_bits row when there is a mask output, otherwise in a bounded scratch (PassLists.partial).
// Passes 2 and 3 hand out their work through ticket counters (the counts exist only on the device).
// ---------------------------------------------------------------------------------------
#ifndef TRL_ROWS_SPECIAL
#define TRL_ROWS_SPECIAL 1
#endif
#ifndef TRL_ROWS_WARPS
#define TRL_ROWS_WARPS 4
#endif
#ifndef TRL_ROWS_MIN_BLOCKS
#define TRL_ROWS_MIN_BLOCKS 10
#endif
constexpr int kRowsWarps = TRL_ROWS_WARPS;
constexpr int kTWarps = 4;   // warps per block of passes 2 and 3

// pass bookkeeping in the per-stream scratch: counters, then the lists
enum : int { kCntLegacy = 0, kCntDeferred = 1, kCntExact = 2, kTicketOrder = 3, kTicketExact = 4, kCounters = 16 };
struct PassLists {
    uint32_t* counts;     // [kCounters], zeroed before pass 1
    int32_t* legacy;      // call indices for movegen_solo_kernel in clean-up mode
    int32_t* deferred;    // call indices whose T search pass 1 deferred; position j = partial-mask slot j
    int32_t* exact;       // positions j of the deferred list that pass 2 left undecided
    uint32_t* partial;    // nullptr: partial masks in mask_bits; else [deferred_cap][TRL_MASK_WORDS]
    unsigned deferred_cap;
};

struct RowsState {
    uint32_t vv[2][kWinRows];   // packed validity planes (0 | 2, 1 | 3), TRL_VV
    uint32_t fu[4][kWinRows];
};

struct RowsWarp {
    RowsState P;
    CallState C;
};

// The call's mask row to / from global memory, coalesced (words TRL_MASK_WORDS.. stay zero).
__device__ __forceinline__ void store_mask(const CallState& C, uint32_t* __restrict__ g, int lane) {
#pragma unroll 1
    for (int w = lane; w < TRL_MASK_WORDS; w += 32) g[w] = C.mask[w];
}

__device__ __forceinline__ void load_mask(CallState& C, const uint32_t* __restrict__ g, int lane) {
#pragma unroll 1
    for (int w = lane; w < TRL_MASK_WORDS + 2; w += 32) C.mask[w] = w < TRL_MASK_WORDS ? g[w] : 0u;
}

__device__ __forceinline__ uint32_t* partial_mask(const PassLists& pl, uint32_t* mask_bits, int i, unsigned j) {
    return pl.partial ? pl.partial + (size_t)j * TRL_MASK_WORDS : mask_bits + (size_t)i * TRL_MASK_WORDS;
}

// the next item of a pass-2 / pass-3 list for this warp: a ticket (a warp that drew short searches takes more)
__device__ __forceinline__ unsigned next_item(uint32_t* ticket, int lane) {
    unsigned j = 0;
    if (lane == 0) j = atomicAdd(ticket, 1u);
    return __shfl_sync(0xffffffffu, j, 0);
}

template <bool WANT_LIST>   // two instantiations: every instruction less in this kernel is instruction-cache room
__global__ void __launch_bounds__(kRowsWarps * 32, TRL_ROWS_MIN_BLOCKS)
movegen_rows_kernel(const uint16_t* __restrict__ boards, const uint8_t* __restrict__ cur,
                    const uint8_t* __restrict__ alt, const TrlGame* __restrict__ games,
                    const int32_t* __restrict__ index, int n, uint32_t* __restrict__ mask_bits,
                    uint16_t* __restrict__ moves, int moves_cap, uint16_t* __restrict__ n_moves,
                    uint32_t* __restrict__ status, uint16_t* __restrict__ compact, unsigned long long compact_cap,
                    unsigned long long* __restrict__ compact_total, unsigned long long* __restrict__ offsets,
                    const PassLists pl) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    RowsWarp& S = reinterpret_cast<RowsWarp*>(smem_raw)[warp];
    CallState& C = S.C;
    const int i = blockIdx.x * kRowsWarps + warp;
    if (i >= n) return;
    int c, a, skip;
    zero_mask(C, lane);
    stage_call(C, i, lane, boards, cur, alt, games, index, c, a, skip);
    __syncwarp();
    if (!skip) {
        const int hi = first_block_row(C.rows, lane);
        bool legacy = false, t_deferred = false;
        // the current piece, then the hold-or-next piece (de-duplicated, move_generation.py:103-105)
#pragma unroll 1
        for (int which = 0; which < 2 && !legacy; ++which) {
            const int type = which ? a : c;
            if (type == TRL_NONE || (which && a == c)) continue;
            const bool ok = search_piece_rows<TRL_ROWS_SPECIAL != 0, false>(S.P, C.rows, hi, type, which != 0, C.mask);
            if (ok) TRL_REASON(0); else TRL_REASON(1);   // instrumented builds
            __syncwarp();
            if (!ok) {
                if (type == P_T) t_deferred = true;
                else legacy = true;
            }
        }
        if (t_deferred && !legacy) {
            unsigned j = 0;
            if (lane == 0) j = atomicAdd(&pl.counts[kCntDeferred], 1u);
            j = __shfl_sync(0xffffffffu, j, 0);
            if (j < pl.deferred_cap) {
                store_mask(C, partial_mask(pl, mask_bits, i, j), lane);
                if (lane == 0) pl.deferred[j] = i;
                return;
            }
            legacy = true;   // no room for the partial mask
        }
        if (legacy) {
            if (lane == 0) pl.legacy[atomicAdd(&pl.counts[kCntLegacy], 1u)] = i;
            return;
        }
    }
    write_call_outputs<WANT_LIST ? 2 : 1>(C, i, lane, mask_bits, moves, moves_cap, n_moves, status, compact, compact_cap, compact_total, offsets);
}

// kick offsets of the common wall-kick table packed 4 bits each (+2), for the FIFO form of the T search
__device__ __forceinline__ void stage_wall_kpack(uint32_t (&kp)[4][3][2], int tid) {
    if (tid < 12) {
        const int r = tid / 3, kd = tid % 3;
        const TrlKicks& K = c_kicks[0][r][kd];
        uint32_t px = 0, py = 0;
        for (int ki = 0; ki < K.n; ++ki) {
            px |= (uint32_t)(K.k[ki][0] + 2) << (4 * ki);
            py |= (uint32_t)(K.k[ki][1] + 2) << (4 * ki);
        }
        kp[r][kd][0] = px;
        kp[r][kd][1] = py;
    }
}

// Stage deferred call j of the list for a T search: board rows, pieces, the partial mask of pass 1.  Returns via_hold
// of the T search (T is the hold-or-next piece unless it is the current one).
__device__ __forceinline__ bool stage_deferred(CallState& C, const PassLists& pl, unsigned j, int lane, const uint16_t* __restrict__ boards,
                                               const uint8_t* __restrict__ cur, const uint8_t* __restrict__ alt,
                                               const TrlGame* __restrict__ games, const int32_t* __restrict__ index,
                                               uint32_t* mask_bits, int& i) {
    i = pl.deferred[j];
    int c, a, skip;
    stage_call(C, i, lane, boards, cur, alt, games, index, c, a, skip);
    load_mask(C, partial_mask(pl, mask_bits, i, j), lane);
    __syncwarp();
    return c != P_T;
}

// Pass 2: the T search of every deferred call, closure form with the order analysis.
template <bool WANT_LIST>
__global__ void __launch_bounds__(kTWarps * 32, 8)
movegen_t_order_kernel(const uint16_t* __restrict__ boards, const uint8_t* __restrict__ cur,
                       const uint8_t* __restrict__ alt, const TrlGame* __restrict__ games,
                       const int32_t* __restrict__ index, uint32_t* __restrict__ mask_bits,
                       uint16_t* __restrict__ moves, int moves_cap, uint16_t* __restrict__ n_moves,
                       uint32_t* __restrict__ status, uint16_t* __restrict__ compact, unsigned long long compact_cap,
                       unsigned long long* __restrict__ compact_total, unsigned long long* __restrict__ offsets,
                       const PassLists pl) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    SoloState& S = reinterpret_cast<SoloState*>(smem_raw)[warp];
    CallState& C = S.C;
    const unsigned count = min(pl.counts[kCntDeferred], pl.deferred_cap);
#pragma unroll 1
    while (true) {
        const unsigned j = next_item(&pl.counts[kTicketOrder], lane);
        if (j >= count) break;
        int i;
        const bool via_hold = stage_deferred(C, pl, j, lane, boards, cur, alt, games, index, mask_bits, i);
        const bool ok = search_piece_rows<true, true>(S.P, C.rows, first_block_row(C.rows, lane), P_T, via_hold, C.mask);
        __syncwarp();
        if (!ok) {   // nothing was merged into the mask
            if (lane == 0) pl.exact[atomicAdd(&pl.counts[kCntExact], 1u)] = (int32_t)j;
            continue;
        }
        write_call_outputs<WANT_LIST ? 2 : 1>(C, i, lane, mask_bits, moves, moves_cap, n_moves, status, compact, compact_cap, compact_total, offsets);
        __syncwarp();
    }
}

// Pass 3: the exact FIFO search of the T piece for the calls pass 2 left undecided.
template <bool WANT_LIST>
__global__ void __launch_bounds__(kTWarps * 32, 8)
movegen_t_exact_kernel(const uint16_t* __restrict__ boards, const uint8_t* __restrict__ cur,
                       const uint8_t* __restrict__ alt, const TrlGame* __restrict__ games,
                       const int32_t* __restrict__ index, uint32_t* __restrict__ mask_bits,
                       uint16_t* __restrict__ moves, int moves_cap, uint16_t* __restrict__ n_moves,
                       uint32_t* __restrict__ status, uint16_t* __restrict__ compact, unsigned long long compact_cap,
                       unsigned long long* __restrict__ compact_total, unsigned long long* __restrict__ offsets,
                       const PassLists pl) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    __shared__ uint32_t s_kpack[4][3][2];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    SoloState& S = reinterpret_cast<SoloState*>(smem_raw)[warp];
    CallState& C = S.C;
    stage_wall_kpack(s_kpack, tid);
    __syncthreads();   // kick table staged; the only block-wide barrier
    const unsigned count = pl.counts[kCntExact];
#pragma unroll 1
    while (true) {
        const unsigned e = next_item(&pl.counts[kTicketExact], lane);
        if (e >= count) break;
        int i;
        const bool via_hold = stage_deferred(C, pl, (unsigned)pl.exact[e], lane, boards, cur, alt, games, index, mask_bits, i);
        uint32_t st = 0;
        search_piece_fifo_body(S.P, C.rows, P_T, via_hold, C.mask, st, &s_kpack);
        st = __reduce_or_sync(0xffffffffu, st);
        if (st && lane == 0) C.status |= st;
        __syncwarp();
        write_call_outputs<WANT_LIST ? 2 : 1>(C, i, lane, mask_bits, moves, moves_cap, n_moves, status, compact, compact_cap, compact_total, offsets);
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------
// Search-internal form over a COMPACTED work list (TrlSearchBuffers.movegen_list).
//
// Inside a self-play step the enumeration runs on a forked stream beside the network, and only for
// the leaves whose parent has no cached list (about a quarter of the games).  The network's trunk kernel
// owns a whole SM per CTA (216 KB of shared memory), so every SM that holds an enumeration block
// delays a trunk CTA.  This kernel therefore packs the work onto as FEW SMs as possible: one block =
// 16 call slots = 32 warps with 120 KB of shared memory (one block per SM), `ceil(count / 16)` blocks
// work and the others exit at once; a call slot (two warps) synchronises with its own named barrier
// and pulls the next call from a global ticket counter, so the working SMs finish together.  With
// `rounds` > 1 only ceil(count / (16 * rounds)) SMs work, each slot serving about `rounds` calls: the
// enumeration then takes longer (it has the whole network evaluation to hide behind) on fewer SMs,
// and a slot that drew a short search takes another instead of idling until the block's longest ends.
// ---------------------------------------------------------------------------------------
constexpr int kListSlots = 16;

__device__ __forceinline__ void slot_barrier(int slot) {
    asm volatile("bar.sync %0, 64;" ::"r"(slot) : "memory");
}

__global__ void __launch_bounds__(kListSlots * 64)
movegen_list_kernel(const TrlGame* __restrict__ games, const int32_t* __restrict__ index,
                    const int32_t* __restrict__ list, uint32_t* __restrict__ count_done,
                    uint16_t* __restrict__ moves, int moves_cap, uint16_t* __restrict__ n_moves, int rounds,
                    TrlSearchCtl* __restrict__ ctl) {   // optional: per-game control blocks that collect the TRL_ST_* bits
    extern __shared__ __align__(16) uint8_t smem_raw[];
    PieceState* ps = reinterpret_cast<PieceState*>(smem_raw);
    CallState* cs = reinterpret_cast<CallState*>(smem_raw + sizeof(PieceState) * kListSlots * 2);
    __shared__ int s_ticket[kListSlots];
    __shared__ uint32_t s_kpack[2][4][3][2];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int slot = warp >> 1, which = warp & 1;
    __shared__ int s_count;
    __shared__ unsigned s_warps_done;
    if (tid == 32) { s_count = (int)count_done[0]; s_warps_done = 0u; }
    {
        if (tid < 24) {
            const int t = tid / 12, r = (tid / 3) % 4, kd = tid % 3;
            const TrlKicks& K = c_kicks[t][r][kd];
            uint32_t px = 0, py = 0;
            for (int ki = 0; ki < K.n; ++ki) {
                px |= (uint32_t)(K.k[ki][0] + 2) << (4 * ki);
                py |= (uint32_t)(K.k[ki][1] + 2) << (4 * ki);
            }
            s_kpack[t][r][kd][0] = px;
            s_kpack[t][r][kd][1] = py;
        }
    }
    __syncthreads();   // the only block-wide barrier; afterwards barrier ids 0..15 belong to the call slots
    const int count = s_count;
    const int n_work = min((int)gridDim.x, (count + kListSlots * rounds - 1) / (kListSlots * rounds));
    if ((int)blockIdx.x < n_work) {
        CallState& C = cs[slot];
        while (true) {
            if (which == 0 && lane == 0) s_ticket[slot] = (int)atomicAdd(&count_done[2], 1u);
            slot_barrier(slot);
            const int j = s_ticket[slot];
            if (j >= count) break;
            const int g = list[j];
            const int gi = index[g];
            for (int w2 = which * 32 + lane; w2 < TRL_MASK_WORDS + 2; w2 += 64) C.mask[w2] = 0u;
            if (which == 0) {
                const TrlPlayer& p = games[gi].players[games[gi].turn & 1];
                for (int r = lane; r < TRL_ROWS; r += 32) C.rows[r] = p.rows[r];
                int c = p.piece;
                int a = (p.held != TRL_NONE) ? p.held : (p.qlen > 0 ? p.queue[0] : TRL_NONE);
                if (c > 6 && c != TRL_NONE) c = TRL_NONE;
                if (a > 6 && a != TRL_NONE) a = TRL_NONE;
                if (lane == 0) { C.cur = c; C.alt = a; C.skip = 0; C.status = 0u; }
            }
            slot_barrier(slot);
            {
                const int c = C.cur, a = C.alt;
                uint32_t st = 0;
                const int type = which ? a : c;
                if (type != TRL_NONE && !(which && a == c))
                    search_piece_warp(ps[warp], C.rows, type, which != 0, C.mask, st, &s_kpack[type == P_I ? 1 : 0]);
                if (st && lane == 0) atomicOr(&C.status, st);   // FIFO overflow of either piece search
            }
            slot_barrier(slot);
            if (which == 0) {
                // ascending move list (= argwhere order): lane owns 12 consecutive mask words
                const int w0 = lane * 12;
                int cnt = 0;
#pragma unroll
                for (int k = 0; k < 12; ++k) {
                    const int w2 = w0 + k;
                    if (w2 < TRL_MASK_WORDS) cnt += __popc(C.mask[w2]);
                }
                int incl = cnt;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const int t = __shfl_up_sync(0xffffffffu, incl, d);
                    if (lane >= d) incl += t;
                }
                const int total = __shfl_sync(0xffffffffu, incl, 31);
                uint16_t* mv = moves + (size_t)g * moves_cap;
                int pos = incl - cnt;
                for (int k = 0; k < 12; ++k) {
                    const int w2 = w0 + k;
                    if (w2 >= TRL_MASK_WORDS) break;
                    uint32_t m = C.mask[w2];
                    while (m) {
                        const int b = __ffs(m) - 1;
                        m &= m - 1;
                        if (pos < moves_cap) mv[pos] = (uint16_t)(w2 * 32 + b);
                        ++pos;
                    }
                }
                if (lane == 0) {
                    n_moves[g] = (uint16_t)total;
                    const uint32_t st = C.status | (total > moves_cap ? TRL_ST_MOVES_TRUNC : 0u);
                    if (st && ctl) atomicOr(&ctl[g].status, st);   // sticky: the host reads it with the other bits
                }
            }
            slot_barrier(slot);   // the mask is re-zeroed and the ticket redrawn for the next call
        }
    }
    // every block has read the count before its last warp arrives here: the last block leaves both
    // counters at zero for the next step (no memset node per step)
    __syncwarp();
    if (lane == 0 && atomicAdd(&s_warps_done, 1u) == (unsigned)(kListSlots * 2 - 1)) {
        if (atomicAdd(&count_done[1], 1u) == gridDim.x - 1) {
            count_done[0] = 0u;
            count_done[1] = 0u;
            count_done[2] = 0u;
        }
    }
}

}  // namespace

// calls per slot the compacted enumeration aims at (1 = one call per slot on ceil(count / 16) SMs)
static int g_list_rounds = 1;
extern "C" void trl_search_movegen_rounds(int rounds) { g_list_rounds = rounds < 1 ? 1 : (rounds > 16 ? 16 : rounds); }

// host-side shadows of the two debug switches (the launcher must not read device symbols: that would be a
// synchronous copy on the legacy stream at every launch)
static int g_fast_path_host = 1, g_fifo_limit_host = kFifoCap;

extern "C" int trl_debug_movegen_fast_path(int on) {
    const int v = on ? 1 : 0;
    g_fast_path_host = v;
    return trl_check(cudaMemcpyToSymbol(c_fast_path, &v, sizeof(int)));
}

// answered[0] = piece searches answered by the row-parallel closure form, answered[1] = handed to the FIFO
// form, since the last call (the counters are reset)
extern "C" int trl_debug_movegen_fast_stats(uint64_t* answered) {
    if (!answered) return TRL_E_ARG;
    unsigned long long h[16] = {0}, z[16] = {0};
    int rc = trl_check(cudaMemcpyFromSymbol(h, g_fast_stats, sizeof(h)));
    if (!rc) rc = trl_check(cudaMemcpyToSymbol(g_fast_stats, z, sizeof(z)));
    answered[0] = h[0]; answered[1] = h[1];
#ifdef TRL_MOVEGEN_STATS
    for (int k = 2; k < 16; ++k) answered[k] = h[k];   // instrumented builds: the caller passes 16 words
#endif
    return rc;
}

// research build (-DTRL_T_TRACE): device buffer of `cap` records of kTTraceWords words; returns the record size
extern "C" int trl_debug_movegen_t_trace(uint32_t* device_buffer, unsigned cap) {
#ifdef TRL_T_TRACE
    unsigned zero = 0;
    int rc = trl_check(cudaMemcpyToSymbol(g_t_trace, &device_buffer, sizeof(device_buffer)));
    if (!rc) rc = trl_check(cudaMemcpyToSymbol(g_t_trace_cap, &cap, sizeof(cap)));
    if (!rc) rc = trl_check(cudaMemcpyToSymbol(g_t_trace_n, &zero, sizeof(zero)));
    return rc ? rc : kTTraceWords;
#else
    (void)device_buffer; (void)cap;
    return TRL_E_ARG;
#endif
}

extern "C" int trl_debug_movegen_fifo_limit(int limit) {
    if (limit < 1 || limit > kFifoCap) limit = kFifoCap;
    g_fifo_limit_host = limit;
    return trl_check(cudaMemcpyToSymbol(c_fifo_limit, &limit, sizeof(int)));
}

int trl_launch_movegen_listed(const TrlGame* games, const int32_t* index, const int32_t* list, uint32_t* count_done,
                              uint16_t* moves, int moves_cap, uint16_t* n_moves, TrlSearchCtl* ctl, cudaStream_t stream) {
    if (!games || !index || !list || !count_done || !moves || !n_moves || moves_cap <= 0) return TRL_E_ARG;
    const size_t smem = sizeof(PieceState) * kListSlots * 2 + sizeof(CallState) * kListSlots;
    static int n_sm = 0;
    if (!n_sm) {
        int dev = 0, sms = 0;
        int rc = trl_check(cudaGetDevice(&dev));
        if (!rc) rc = trl_check(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        if (!rc) rc = trl_check(cudaFuncSetAttribute(movegen_list_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        if (rc) return rc;
        n_sm = sms;
    }
    movegen_list_kernel<<<n_sm, kListSlots * 64, smem, stream>>>(games, index, list, count_done, moves, moves_cap, n_moves,
                                                                g_list_rounds, ctl);
    return trl_check(cudaGetLastError());
}

// Which form of the warp-cooperative enumeration runs: -1 automatic (by batch size), 0 = two warps per call
// (latency form), 1 = one warp per call, 2 = the pass form (closure-search kernel + T passes + legacy route; the
// throughput form).  Tests force all of them.
static int g_form = -1;
extern "C" void trl_movegen_warp_form(int form) { g_form = form; }

// per-stream scratch of the pass form (PassLists): kCounters counters, the legacy, deferred and exact lists of n entries
// each, then (only without a mask output) the partial masks
struct TwoPassScratch { cudaStream_t stream; uint32_t* buf; size_t cap; bool used; };
static TwoPassScratch g_scratch[8];

static std::mutex g_scratch_mutex;   // device entry points are re-entrant per stream: the table is shared

static uint32_t* two_pass_scratch(cudaStream_t stream, size_t need) {
    std::lock_guard<std::mutex> lock(g_scratch_mutex);
    TwoPassScratch* slot = nullptr;
    for (auto& e : g_scratch) if (e.used && e.stream == stream) { slot = &e; break; }
    if (!slot) for (auto& e : g_scratch) if (!e.used) { slot = &e; e.used = true; e.stream = stream; e.buf = nullptr; e.cap = 0; break; }
    if (!slot) return nullptr;
    if (slot->cap < need) {
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(stream, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) return nullptr;
        if (slot->buf) { cudaStreamSynchronize(stream); cudaFree(slot->buf); slot->buf = nullptr; slot->cap = 0; }
        if (cudaMalloc(&slot->buf, need * sizeof(uint32_t)) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        slot->cap = need;
    }
    return slot->buf;
}

// partial masks without a mask output: max(64 Ki, n / 8) entries of 1448 B (the config-2 boards defer 6 % of the calls);
// trl_debug_movegen_partial_cap lowers the capacity so that tests reach the legacy route of a full scratch
static unsigned g_partial_cap_debug = 0;
extern "C" int trl_debug_movegen_partial_cap(int cap) {
    g_partial_cap_debug = cap > 0 ? (unsigned)cap : 0u;
    return 0;
}

// counters of the last launch of the pass form (trl_debug_movegen_pass_counts)
static uint32_t* g_last_counts = nullptr;
static unsigned g_last_deferred_cap = 0;

// counts[0] = calls whose T search pass 1 deferred (and found room), [1] = of those, calls pass 2 left to the exact T
// search, [2] = calls on the legacy route; of the last launch of the pass form.  Synchronises the device.
extern "C" int trl_debug_movegen_pass_counts(uint32_t* counts) {
    if (!counts || !g_last_counts) return TRL_E_ARG;
    uint32_t h[kCounters];
    int rc = trl_check(cudaDeviceSynchronize());
    if (!rc) rc = trl_check(cudaMemcpy(h, g_last_counts, sizeof(h), cudaMemcpyDeviceToHost));
    if (rc) return rc;
    counts[0] = h[kCntDeferred] < g_last_deferred_cap ? h[kCntDeferred] : g_last_deferred_cap;
    counts[1] = h[kCntExact];
    counts[2] = h[kCntLegacy];
    return 0;
}

// Launch the warp-cooperative enumeration (same argument contract as movegen.cu's launch_movegen).
int trl_launch_movegen_warp(const uint16_t* boards, const uint8_t* cur, const uint8_t* alt, const TrlGame* games,
                            const int32_t* index, int n, uint32_t* mask_bits, uint16_t* moves, int moves_cap,
                            uint16_t* n_moves, uint32_t* status, cudaStream_t stream, uint16_t* compact,
                            unsigned long long compact_cap, unsigned long long* compact_total,
                            unsigned long long* offsets) {
    static int n_sm = 0, t_order_blocks = 0, t_exact_blocks = 0;   // resident blocks of passes 2 and 3 per SM
    static bool configured = false;
    const size_t smem_warp = sizeof(PieceState) * kWarps + sizeof(CallState) * kCallsPerBlock;
    const size_t smem_solo = sizeof(SoloState) * kSoloWarps;
    const size_t smem_rows = sizeof(RowsWarp) * kRowsWarps;
    const size_t smem_t = sizeof(SoloState) * kTWarps;
    if (!configured) {
        int dev = 0;
        int rc = trl_check(cudaGetDevice(&dev));
        if (!rc) rc = trl_check(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
        if (!rc) rc = trl_check(cudaFuncSetAttribute(movegen_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_warp));
        if (!rc) rc = trl_check(cudaFuncSetAttribute(movegen_solo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_solo));
        if (!rc) rc = trl_check(cudaFuncSetAttribute(movegen_solo_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
        if (!rc) rc = trl_check(cudaFuncSetAttribute(movegen_rows_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_rows));
        if (!rc) rc = trl_check(cudaFuncSetAttribute(movegen_rows_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
        if (!rc) rc = trl_check(cudaFuncSetAttribute(movegen_rows_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_rows));
        if (!rc) rc = trl_check(cudaFuncSetAttribute(movegen_rows_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
        for (const void* f : {(const void*)movegen_t_order_kernel<false>, (const void*)movegen_t_order_kernel<true>,
                              (const void*)movegen_t_exact_kernel<false>, (const void*)movegen_t_exact_kernel<true>}) {
            if (!rc) rc = trl_check(cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_t));
            if (!rc) rc = trl_check(cudaFuncSetAttribute(f, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
        }
        // the two instantiations of a pass differ only in the list writer: the mask-mode one sizes the grid
        if (!rc) rc = trl_check(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&t_order_blocks, movegen_t_order_kernel<false>, kTWarps * 32, smem_t));
        if (!rc) rc = trl_check(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&t_exact_blocks, movegen_t_exact_kernel<false>, kTWarps * 32, smem_t));
        if (rc) return rc;
        configured = true;
    }
    // the throughput forms once every SM is full of warps anyway (148 SMs x 32 resident warps = 4736 calls
    // in flight): below that the two-warp form halves the latency of a batch
    int form = g_form < 0 ? (n >= 3 * 4736 ? 2 : 0) : g_form;
    // the debug switches (FIFO form only / lowered FIFO capacity) are served by the one-kernel forms
    if (form == 2 && (!g_fast_path_host || g_fifo_limit_host != kFifoCap)) form = 1;
    // pass form: counters, three lists of n entries, and without a mask output the partial masks
    unsigned deferred_cap = (unsigned)n;
    if (!mask_bits) deferred_cap = (unsigned)min(n, max(64 * 1024, n / 8));
    if (g_partial_cap_debug) deferred_cap = min(deferred_cap, g_partial_cap_debug);
    const size_t lists = kCounters + 3 * (size_t)n;
    uint32_t* scratch = form == 2 ? two_pass_scratch(stream, lists + (mask_bits ? 0 : (size_t)deferred_cap * TRL_MASK_WORDS)) : nullptr;
    if (form == 2 && !scratch) form = 1;
    if (form == 2) {
        const PassLists pl{scratch, (int32_t*)scratch + kCounters, (int32_t*)scratch + kCounters + n,
                           (int32_t*)scratch + kCounters + 2 * (size_t)n, mask_bits ? nullptr : scratch + lists, deferred_cap};
        g_last_counts = scratch;
        g_last_deferred_cap = deferred_cap;
        int rc = trl_check(cudaMemsetAsync(scratch, 0, kCounters * sizeof(uint32_t), stream));
        if (rc) return rc;
        const bool want_list = moves || compact;
        const int rows_blocks = (n + kRowsWarps - 1) / kRowsWarps;
        (want_list ? movegen_rows_kernel<true> : movegen_rows_kernel<false>)<<<rows_blocks, kRowsWarps * 32, smem_rows, stream>>>(
            boards, cur, alt, games, index, n, mask_bits, moves, moves_cap, n_moves, status, compact, compact_cap,
            compact_total, offsets, pl);
        rc = trl_check(cudaGetLastError());
        if (rc) return rc;
        (want_list ? movegen_t_order_kernel<true> : movegen_t_order_kernel<false>)<<<t_order_blocks * n_sm, kTWarps * 32, smem_t, stream>>>(
            boards, cur, alt, games, index, mask_bits, moves, moves_cap, n_moves, status, compact, compact_cap,
            compact_total, offsets, pl);
        rc = trl_check(cudaGetLastError());
        if (rc) return rc;
        (want_list ? movegen_t_exact_kernel<true> : movegen_t_exact_kernel<false>)<<<t_exact_blocks * n_sm, kTWarps * 32, smem_t, stream>>>(
            boards, cur, alt, games, index, mask_bits, moves, moves_cap, n_moves, status, compact, compact_cap,
            compact_total, offsets, pl);
        rc = trl_check(cudaGetLastError());
        if (rc) return rc;
        const int blocks = min(8 * n_sm, (n + kSoloWarps - 1) / kSoloWarps);
        movegen_solo_kernel<<<blocks, kSoloWarps * 32, smem_solo, stream>>>(
            boards, cur, alt, games, index, n, mask_bits, moves, moves_cap, n_moves, status, compact, compact_cap,
            compact_total, offsets, pl.legacy, pl.counts + kCntLegacy);
        return trl_check(cudaGetLastError());
    }
    if (form == 1) {
        const int blocks = (n + kSoloWarps - 1) / kSoloWarps;
        movegen_solo_kernel<<<blocks, kSoloWarps * 32, smem_solo, stream>>>(boards, cur, alt, games, index, n, mask_bits, moves,
                                                                           moves_cap, n_moves, status, compact, compact_cap,
                                                                           compact_total, offsets, nullptr, nullptr);
        int rc = trl_check(cudaGetLastError());
        return rc;
    }
    const int blocks = (n + kCallsPerBlock - 1) / kCallsPerBlock;
    movegen_warp_kernel<<<blocks, kWarps * 32, smem_warp, stream>>>(boards, cur, alt, games, index, n, mask_bits, moves,
                                                                   moves_cap, n_moves, status, compact, compact_cap,
                                                                   compact_total, offsets, nullptr, nullptr);
    return trl_check(cudaGetLastError());
}
