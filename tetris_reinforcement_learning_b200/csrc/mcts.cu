// mcts.cu — batched MCTS / PUCT self-play search for sm_100a: one warp per game, the tree in
// HBM as struct-of-arrays (children of a node are one contiguous run), one leaf per game per
// step so that the network sees a device-resident batch of n_games leaves.
//
// Replaces ai.MCTS / amcts (reference ai.py:299-659, 766-996) and the per-move part of
// play_game (ai.py:1610-1668).  Semantics follow SURVEY A.3 exactly, including the quirks:
// ">=" (last maximum wins) in selection, un-normalised Gamma root noise, FPU refresh of the
// played-out node's siblings only when their parent is not the root, move choice on pre-prune
// visits, pruning with N_root in the denominator.  Scores are computed in double like the
// reference's Python floats; the only approximations left are libm differences and the
// summation order of warp reductions (tolerance: DESIGN.md §Parity).
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "env_step.cuh"
#include "features_dev.cuh"
#include "trl_common.cuh"

namespace {

constexpr int kWarps = 4;
constexpr int kGameWords = sizeof(TrlGame) / 4;
constexpr unsigned kFull = 0xFFFFFFFFu;
constexpr int TRL_PATH_INTS = 64;        // per game: [0] depth, [1..31] nodes, [32..63] state slots along the selected path
constexpr int TRL_PATH_MAX_DEPTH = 30;

static_assert(sizeof(TrlSearchCtl) == 80, "TrlSearchCtl layout");
static_assert(sizeof(TrlSearchParams) == 168, "TrlSearchParams layout");
static_assert(sizeof(TrlSearchBuffers) == 280, "TrlSearchBuffers layout");
static_assert(sizeof(TrlGameEnd) == 32, "TrlGameEnd layout");
static_assert(sizeof(TrlSample) == 20 + 400 + 3 * 2 * TRL_SAMPLE_MOVES, "TrlSample layout");
static_assert(sizeof(TrlRootStats) == 112 + 2 * 4 * TRL_SAMPLE_MOVES, "TrlRootStats layout");

// Phase trace of the per-step kernel (builds with -DTRL_SEARCH_TRACE only; tools/search_trace.py): lane 0 of every
// game's warp stamps clock64() into g_search_trace[game][phase].
#ifdef TRL_SEARCH_TRACE
__device__ long long* g_search_trace = nullptr;
#define TRL_TRACE(g, lane, phase) do { if ((lane) == 0 && g_search_trace) g_search_trace[(size_t)(g) * 16 + (phase)] = clock64(); } while (0)
#else
#define TRL_TRACE(g, lane, phase) ((void)0)
#endif

__device__ __forceinline__ double negate_value(double v, bool tanh_mode) { return tanh_mode ? -v : 1.0 - v; }

// Uniform double in [0,1): purpose 3 = playout-cap coin, 4 = move choice (SURVEY A.7).
__device__ __forceinline__ double trl_uniform(uint64_t seed, uint32_t game_id, uint32_t search_no,
                                              uint32_t purpose, uint32_t idx) {
    uint32_t o[4];
    trl_philox(seed, idx, game_id, purpose, search_no, o);
    return ((double)(o[0] >> 5) * 67108864.0 + (double)(o[1] >> 6)) / 9007199254740992.0;
}

// Gamma(alpha, 1): Marsaglia-Tsang with Box-Muller normals, U^(1/alpha) boost for alpha < 1
// (replaces np.random.gamma, ai.py:489).
__device__ double trl_gamma(uint64_t seed, uint32_t game_id, uint32_t search_no, uint32_t child, double alpha) {
    const double a = alpha < 1.0 ? alpha + 1.0 : alpha;
    const double d = a - 1.0 / 3.0, c = 1.0 / sqrt(9.0 * d);
    for (uint32_t k = 0; k < 64; ++k) {
        uint32_t o[4];
        trl_philox(seed, child, game_id, 5u | (k << 8), search_no, o);
        const double u1 = ((double)o[0] + 1.0) / 4294967296.0, u2 = (double)o[1] / 4294967296.0;
        const double x = sqrt(-2.0 * log(u1)) * cos(6.283185307179586 * u2);
        double v = 1.0 + c * x;
        if (v <= 0.0) continue;
        v = v * v * v;
        const double u = ((double)o[2] + 0.5) / 4294967296.0;
        if (log(u) < 0.5 * x * x + d - d * v + d * log(v)) {
            double g = d * v;
            if (alpha < 1.0) g *= pow(((double)o[3] + 0.5) / 4294967296.0, 1.0 / alpha);
            return g;
        }
    }
    return alpha;  // unreachable in practice (acceptance > 95 % per round)
}

// warp arg-max of (score, index) with the reference's ">=" rule: among equal scores the
// LARGEST index wins (ai.py:383).
__device__ __forceinline__ void warp_argmax_last(double& score, int& idx) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const double s2 = __shfl_xor_sync(kFull, score, off);
        const int i2 = __shfl_xor_sync(kFull, idx, off);
        if (i2 >= 0 && (idx < 0 || s2 > score || (s2 == score && i2 > idx))) { score = s2; idx = i2; }
    }
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(kFull, v, off);
    return v;
}

__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v = fmax(v, __shfl_xor_sync(kFull, v, off));
    return v;
}

__device__ __forceinline__ void copy_game(uint32_t* dst, const uint32_t* src, int lane) {
    for (int w = lane; w < kGameWords; w += 32) dst[w] = src[w];
}

__device__ __forceinline__ bool game_terminal(const TrlGame* g) {
    return g->players[0].game_over || g->players[1].game_over;
}

// ---------------------------------------------------------------------------------------
// step part 1: select + materialise
// ---------------------------------------------------------------------------------------

// leaf_si / leaf_pi (all lanes): state index of the position to evaluate and of the state it was reached
// from, as written to leaf_state[g] / leaf_parent[g]; on return *sgame holds the leaf state.
__device__ void select_body(const TrlSearchBuffers& B, const TrlSearchParams& P, int g, int lane, TrlGame* sgame,
                            int& leaf_si, int& leaf_pi, const int32_t* __restrict__ row_of = nullptr, int2* parent_rows = nullptr) {
    TrlSearchCtl* ctl = &B.ctl[g];
    leaf_si = -1; leaf_pi = -1;
    if (!ctl->active) {
        if (lane == 0) {
            B.leaf_state[g] = -1; ctl->leaf_kind = 3;
            if (B.leaf_parent) B.leaf_parent[g] = -1;
            if (B.movegen_index) B.movegen_index[g] = -1;
        }
        return;
    }
    const size_t nb = (size_t)g * B.node_cap, sb = (size_t)g * B.state_cap;
    const bool tanh_mode = P.use_tanh != 0;
    uint32_t* sg = reinterpret_cast<uint32_t*>(sgame);

    if (ctl->iter == 0) {
        // new search: root = copy of the real game with queues cut to 5 previews (ai.py:304-309)
        copy_game(sg, reinterpret_cast<const uint32_t*>(&B.games[g]), lane);
        __syncwarp();
        if (lane == 0) {
            for (int pl = 0; pl < 2; ++pl)
                if (sgame->players[pl].qlen > TRL_PREVIEWS) sgame->players[pl].qlen = TRL_PREVIEWS;
            B.parent[nb] = -1; B.slot[nb] = 0; B.visits[nb] = 0; B.value_sum[nb] = 0.0; B.prior[nb] = 0.0;
            B.move[nb] = 0xFFFF;
            B.first_child[sb] = -1; B.n_children[sb] = 0; B.fpu[sb] = 0.0;
            if (B.legal_cache_n) B.legal_cache_n[sb] = -1;
            ctl->n_nodes = 1; ctl->n_states = 1; ctl->garbage_ctr = 0; ctl->max_depth = 0;
            int iters = P.max_iter;
            uint32_t fast = 0;
            if (ctl->search_no == 0) {
                // play_game's random opening (ai.py:1588-1596): ceil(Exp(0.04 * DIRICHLET_S)) plies sampled from
                // the raw policy; purpose 6 = the exponential draw (replaces np.random.exponential)
                int k = 0;
                if (P.use_random_start) {
                    const double u = trl_uniform(P.seed, B.games[g].game_id, 0u, 6u, 0u);
                    const double n = -P.random_start_scale * log(1.0 - u);
                    k = n > 0.0 ? (int)ceil(n) : 0;
                }
                ctl->random_left = k;
            }
            if (ctl->random_left > 0) {   // fast_config (ai.py:1597-1601): one iteration, no coin, no noise, not saved
                iters = 1;
                fast = 1;
            } else if (P.training && P.use_playout_cap) {  // ai.py:323-330
                const double coin = trl_uniform(P.seed, B.games[g].game_id, ctl->search_no, 3u, 0u);
                if (coin < P.playout_cap_chance) iters = P.iters_long;
                else { iters = P.iters_short; fast = 1; }
            }
            ctl->max_iter = iters; ctl->fast = fast;
        }
        __syncwarp();
        copy_game(reinterpret_cast<uint32_t*>(&B.states[sb]), sg, lane);
        __syncwarp();
    }

    // ---- select (ai.py:346-393) ----
    int node = 0, depth = 0;
    const bool forced_on = P.use_forced && P.training && !(P.use_playout_cap && ctl->fast);
    int* path = B.path ? B.path + (size_t)g * TRL_PATH_INTS : nullptr;
    int parent_s = -1, s_leaf = -1;   // state slots of the last two levels (no reload after the loop)
    while (true) {
        const int s = B.slot[nb + node];
        if (path && lane == 0 && depth <= TRL_PATH_MAX_DEPTH) { path[1 + depth] = node; path[32 + depth] = s; }
        s_leaf = s;
        if (s < 0) break;
        const int C = B.n_children[sb + s];
        if (C <= 0) break;
        const int base = B.first_child[sb + s];
        const int pv = B.visits[nb + node];
        const double sqrt_parent = sqrt((double)pv);
        const double unvisited_scale = P.cpuct * sqrt_parent / P.dpuct;
        const double fpu_q = B.fpu[sb + s];
        const bool check_forced = forced_on && node == 0;
        double best = -1.0;  // max_child_score starts at -1 (ai.py:348)
        int best_i = -1;
        for (int c0 = lane; c0 < C; c0 += 64) {
            // two children per lane with all six loads in flight (a typical node has ~50 children)
            int vcs[2]; double prs[2], vss[2];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int c = c0 + 32 * h;
                const bool in = c < C;
                vcs[h] = in ? B.visits[nb + base + c] : 0;
                prs[h] = in ? B.prior[nb + base + c] : 0.0;
                vss[h] = in ? B.value_sum[nb + base + c] : 0.0;
            }
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int c = c0 + 32 * h;
                if (c >= C) break;
                const int vc = vcs[h];
                const double pr = prs[h];
                double q, u;
                if (vc == 0) { q = fpu_q; u = unvisited_scale * pr; }
                else { q = vss[h] / (double)vc; u = P.cpuct * pr * sqrt_parent / (P.dpuct + (double)vc); }
                double score = q + u;
                if (check_forced && vc >= 1 && (double)vc < sqrt(P.c_forced * pr * (double)pv)) score = INFINITY;
                if (score >= best) { best = score; best_i = c; }
            }
        }
        warp_argmax_last(best, best_i);
        if (best_i < 0) best_i = C - 1;  // every score < -1 (tanh only): the reference would raise
        parent_s = s;
        node = base + best_i;
        ++depth;
    }

    if (path && lane == 0) path[0] = depth <= TRL_PATH_MAX_DEPTH ? depth : -1;
    TRL_TRACE(g, lane, 9);   // selection walk

    // ---- materialise the leaf (ai.py:398-403) ----
    int s = s_leaf;
    int parent_state = -1;
    int parent_cached = -1;   // number of legal moves already listed under the parent (loaded early: used after the env step)
    if (node != 0) {
        const int ps = parent_s;
        parent_state = (int)(sb + ps);
        if (B.legal_cache_n) parent_cached = B.legal_cache_n[parent_state];
        if (row_of) *parent_rows = *reinterpret_cast<const int2*>(row_of + 2 * (size_t)parent_state);   // for the encoder, in flight under the env step
        if (s < 0) s = ctl->n_states;  // first visit: new state slot (uniform across lanes)
        if (path && lane == 0 && depth <= TRL_PATH_MAX_DEPTH) path[32 + depth] = s;
        copy_game(sg, reinterpret_cast<const uint32_t*>(&B.states[sb + ps]), lane);
        __syncwarp();
        TRL_TRACE(g, lane, 10);   // parent state in shared memory
        if (lane == 0) {
            trl_env_step_scalar(sgame, (int)B.move[nb + node], false, P.seed, 1u + ctl->search_no, &ctl->garbage_ctr);
            if (B.slot[nb + node] < 0) {
                B.slot[nb + node] = s;
                B.first_child[sb + s] = -1; B.n_children[sb + s] = 0; B.fpu[sb + s] = 0.0;
                if (B.legal_cache_n) B.legal_cache_n[sb + s] = -1;   // no child of this state has been enumerated yet
                ctl->n_states = s + 1;
            }
        }
        __syncwarp();
        TRL_TRACE(g, lane, 11);   // env step
        copy_game(reinterpret_cast<uint32_t*>(&B.states[sb + s]), sg, lane);
    } else {
        copy_game(sg, reinterpret_cast<const uint32_t*>(&B.states[sb]), lane);
    }
    __syncwarp();
    if (lane == 0) {
        const TrlGame* lg = sgame;
        int kind = 0;
        double lv = 0.0;
        if (game_terminal(lg)) {  // ai.py:472-479
            kind = 2;
            const int w = lg->players[0].game_over ? 1 : 0;  // Game.winner (game.py:217-225)
            const double vmin = tanh_mode ? -1.0 : 0.0;
            lv = (w == lg->turn) ? 1.0 : vmin;
        } else {
            const TrlPlayer* p = &lg->players[lg->turn & 1];
            if (p->piece == TRL_NONE && p->held == TRL_NONE) kind = 1;  // Game.no_move
        }
        ctl->leaf = node; ctl->leaf_kind = kind; ctl->leaf_value = lv;
        if (depth > ctl->max_depth) ctl->max_depth = depth;
        leaf_si = (kind == 2) ? -1 : (int)(sb + s);
        leaf_pi = (kind == 2) ? -1 : parent_state;
        B.leaf_state[g] = leaf_si;
        if (B.leaf_parent) B.leaf_parent[g] = leaf_pi;
        if (B.movegen_index) {
            // all children of a state share the side to move's board and pieces: enumerate once per parent
            const bool hit = parent_cached >= 0;
            const bool need = !(kind == 2 || hit);
            B.movegen_index[g] = need ? (int)(sb + s) : -1;
            if (need && B.movegen_list) B.movegen_list[atomicAdd(B.movegen_count, 1u)] = g;
        }
    }
    leaf_si = __shfl_sync(kFull, leaf_si, 0);
    leaf_pi = __shfl_sync(kFull, leaf_pi, 0);
    TRL_TRACE(g, lane, 12);   // leaf classified, work list entry
}

// Gating battles (ai.py:1975-2114): two networks with their own search settings; the one that owns the side to
// move at the root runs the search.  Colours alternate by game id (ai.py:2087-2091): network 1 plays player
// (game_id & 1).  B.params2 = device array of the two parameter sets; the BATTLE kernels pick per game.
__device__ __forceinline__ int battle_owner(const TrlSearchBuffers& B, int g) {
    return (int)((B.games[g].game_id ^ (uint32_t)B.games[g].turn) & 1u);
}

template <bool BATTLE>
__global__ void __launch_bounds__(kWarps * 32)
search_select_kernel(TrlSearchBuffers B, TrlSearchParams P) {
    __shared__ __align__(16) TrlGame s_game[kWarps];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int g = blockIdx.x * kWarps + wib;
    if (g >= B.n_games) return;
    int si, pi;
    if (BATTLE) select_body(B, B.params2[battle_owner(B, g)], g, lane, &s_game[wib], si, pi);
    else select_body(B, P, g, lane, &s_game[wib], si, pi);
}

// ---------------------------------------------------------------------------------------
// step part 2: expand + backup (+ finish the search and play the move)
// ---------------------------------------------------------------------------------------

__device__ __forceinline__ float load_out(const void* p, size_t i, int dtype) {
    return dtype == 1 ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p)[i])
                      : reinterpret_cast<const float*>(p)[i];
}

// logit of the c-th legal move: dense rows are indexed by the move, gathered rows (dtype 2, written by
// policy_legal_kernel) by the position in the legal list
__device__ __forceinline__ float load_logit(const void* p, size_t row_base, const uint16_t* mv, int c, int dtype) {
    return load_out(p, row_base + (dtype == 2 ? (size_t)c : (size_t)mv[c]), dtype);
}

// Root statistics of a finished search (include/trl.h, TrlRootStats), read before policy-target pruning.  The
// children are written lane-parallel like the sample's moves; the principal variation walks down from the root,
// one warp arg-max per ply with the move choice's rule (most visits, last maximum), while the best child has visits.
__device__ void write_root_stats(const TrlSearchBuffers& B, TrlRootStats* rs, int g, int lane, size_t nb, size_t sb) {
    const int C = B.n_children[sb], base = B.first_child[sb];
    const double fpu_q = B.fpu[sb];   // the root's children keep their initial FPU (the refresh skips the root)
    for (int c = lane; c < C && c < TRL_SAMPLE_MOVES; c += 32) {
        const int id = base + c;
        const int n = B.visits[nb + id];
        rs->prior[c] = (float)B.prior[nb + id];
        rs->q[c] = (float)(n > 0 ? B.value_sum[nb + id] / (double)n : fpu_q);
    }
    int node = 0, ply = 0;
    for (; ply < TRL_PV_MAX; ++ply) {
        const int s = B.slot[nb + node];
        if (s < 0) break;
        const int Cn = B.n_children[sb + s], fb = B.first_child[sb + s];
        if (Cn <= 0) break;
        double bestn = -1.0; int bi = -1;
        for (int c = lane; c < Cn; c += 32) {
            const double n = (double)B.visits[nb + fb + c];
            if (n >= bestn) { bestn = n; bi = c; }
        }
        warp_argmax_last(bestn, bi);
        if (!(bestn > 0.0)) break;
        node = fb + bi;
        if (lane == 0) { rs->pv[ply] = B.move[nb + node]; rs->pv_visits[ply] = (uint32_t)bestn; }
    }
    if (lane == 0) {
        const int rv = B.visits[nb];
        rs->root_value = (float)(rv > 0 ? B.value_sum[nb] / (double)rv : 0.0);
        rs->root_visits = (uint32_t)rv;
        rs->slot = g;
        rs->n_children = (uint16_t)C;
        rs->pv_len = (uint16_t)ply;
        for (int k = ply; k < TRL_PV_MAX; ++k) { rs->pv[k] = 0xFFFF; rs->pv_visits[k] = 0; }
    }
}

// End of a search (ai.py:571-648) + the per-move bookkeeping of play_game (ai.py:1611-1668).  Analysis mode
// (P.stop_after_search): the record only; the real game stays as it is and the slot is parked.
__device__ void finish_search(const TrlSearchBuffers& B, const TrlSearchParams& P, int g, int lane, TrlGame* sgame) {
    TrlSearchCtl* ctl = &B.ctl[g];
    const size_t nb = (size_t)g * B.node_cap, sb = (size_t)g * B.state_cap;
    const int C = B.n_children[sb];
    const int base = B.first_child[sb];
    const int root_visits = B.visits[nb];
    uint32_t* sg = reinterpret_cast<uint32_t*>(sgame);

    int chosen = -1;
    TrlSample* rec = nullptr;
    // random opening ply (ai.py:1597-1608): one iteration, move sampled from the priors, never stored.  Read by
    // lane 0 and broadcast: lane 0 decrements the counter below.
    int random_ply = 0;
    if (lane == 0) random_ply = ctl->random_left > 0;
    random_ply = __shfl_sync(kFull, random_ply, 0);
    if (C > 0) {
        // most visited root child, LAST maximum (ai.py:579-587)
        double bestn = -1.0; int max_i = -1;
        for (int c = lane; c < C; c += 32) {
            const double n = (double)B.visits[nb + base + c];
            if (n >= bestn) { bestn = n; max_i = c; }
        }
        warp_argmax_last(bestn, max_i);

        // temperature move choice on pre-prune visits (ai.py:591-612); sequential like
        // random.choices' accumulate + bisect
        const double temp = P.training ? P.temperature : 0.0;
        if (lane == 0) {
            if (random_ply) {
                // pick_random_move_by_policy (ai.py:999-1014): random.choices(moves, priors); purpose 7
                double total = 0.0;
                for (int c = 0; c < C; ++c) total += B.prior[nb + base + c];
                const double x = trl_uniform(P.seed, B.games[g].game_id, ctl->search_no, 7u, 0u) * total;
                double cum = 0.0;
                chosen = C - 1;
                for (int c = 0; c < C - 1; ++c) {
                    cum += B.prior[nb + base + c];
                    if (cum > x) { chosen = c; break; }
                }
                ctl->random_left -= 1;
            } else if (temp == 0.0) {  // np.argmax: FIRST maximum
                int bi = 0, bn = -1;
                for (int c = 0; c < C; ++c) { const int n = B.visits[nb + base + c]; if (n > bn) { bn = n; bi = c; } }
                chosen = bi;
            } else {
                const double inv_t = 1.0 / temp;
                double wsum = 0.0;
                for (int c = 0; c < C; ++c) wsum += pow((double)B.visits[nb + base + c], inv_t);
                double total = 0.0;
                for (int c = 0; c < C; ++c) total += pow((double)B.visits[nb + base + c], inv_t) / wsum;
                const double x = trl_uniform(P.seed, B.games[g].game_id, ctl->search_no, 4u, 0u) * total;
                double cum = 0.0;
                chosen = C - 1;  // bisect(cum, x, 0, C-1): first index with cum > x, capped at C-1
                for (int c = 0; c < C - 1; ++c) {
                    cum += pow((double)B.visits[nb + base + c], inv_t) / wsum;
                    if (cum > x) { chosen = c; break; }
                }
            }
        }
        chosen = __shfl_sync(kFull, chosen, 0);

        const bool save = !ctl->fast;
        const bool want_rec = (save || P.save_all || P.stop_after_search) && !random_ply;
        uint32_t slot_i = 0;
        if (want_rec) {
            if (lane == 0) slot_i = atomicAdd(B.sample_count, 1u);
            slot_i = __shfl_sync(kFull, slot_i, 0);
            if (slot_i < (uint32_t)B.sample_cap) rec = &B.samples[slot_i];
            else if (lane == 0) ctl->status |= TRL_ST_SAMPLE_OVERFLOW;   // the record of this search is lost
        }
        if (rec)
            for (int c = lane; c < C && c < TRL_SAMPLE_MOVES; c += 32) {
                rec->moves[c] = B.move[nb + base + c];
                rec->visits_pre[c] = (uint16_t)B.visits[nb + base + c];
            }
        if (rec && B.root_stats) write_root_stats(B, &B.root_stats[slot_i], g, lane, nb, sb);

        // policy-target pruning (ai.py:619-648): mutates root-children visit counts
        if (P.use_forced && P.training && !ctl->fast) {
            const int b = base + max_i;
            const double sqrt_root = sqrt((double)root_visits);
            const double ref = B.value_sum[nb + b] / (double)B.visits[nb + b] +
                               P.cpuct * B.prior[nb + b] * sqrt_root / (P.dpuct + (double)B.visits[nb + b]);
            const double root_fpu = B.fpu[sb];
            for (int c = lane; c < C; c += 32) {
                const int id = base + c;
                int n = B.visits[nb + id];
                if (id == b || n <= 0) continue;
                const double pr = B.prior[nb + id];
                const double q = B.value_sum[nb + id] / (double)n;  // value_avg does not change while pruning
                (void)root_fpu;
                const double n_forced = sqrt(P.c_forced * pr * (double)root_visits);
                const double sc = q + P.cpuct * pr * sqrt_root / (P.dpuct + (double)root_visits);
                int count = 0;
                while (true) {
                    if (n == 1) { n = 0; break; }
                    if ((double)count < n_forced && sc < ref) { ++count; --n; }
                    else break;
                }
                B.visits[nb + id] = n;
            }
            __syncwarp();
        }
        if (rec) {
            uint32_t tot = 0;
            for (int c = lane; c < C; c += 32) {
                const int n = B.visits[nb + base + c];
                if (c < TRL_SAMPLE_MOVES) rec->visits[c] = (uint16_t)n;
                tot += (uint32_t)n;
            }
            for (int off = 16; off > 0; off >>= 1) tot += __shfl_xor_sync(kFull, tot, off);
            copy_game(reinterpret_cast<uint32_t*>(&rec->state), reinterpret_cast<const uint32_t*>(&B.states[sb]), lane);
            if (lane == 0) {
                rec->game_id = B.games[g].game_id; rec->search_no = (uint16_t)ctl->search_no;
                rec->turn = B.games[g].turn; rec->saved = save ? 1 : 0;
                rec->n_children = (uint16_t)C; rec->chosen_move = B.move[nb + base + chosen];
                rec->total_visits = tot; rec->iterations = ctl->max_iter;
            }
        }
    }

    if (P.stop_after_search) {
        if (lane == 0) {
            if (C <= 0) ctl->status |= TRL_ST_NO_PIECE;   // terminal root or no legal move: no record
            ctl->iter = 0;
            ctl->active = 0;
        }
        __syncwarp();
        return;
    }

    // ---- play the move on the real game (ai.py:1668: game.make_move(move)) ----
    copy_game(sg, reinterpret_cast<const uint32_t*>(&B.games[g]), lane);
    __syncwarp();
    if (lane == 0) {
        TrlGame* rg = sgame;
        bool over = false;
        if (C > 0) {
            const int mover = rg->turn & 1;
            TrlStepOut o = trl_env_step_scalar(rg, (int)B.move[nb + base + chosen], true, P.seed, 0u, &rg->rng_ctr);
            if (mover == 0) { ctl->lines_sent0 += o.attack; ctl->lines_cleared0 += o.rows_cleared; }
            ctl->status |= o.status;
        } else {
            ctl->status |= TRL_ST_NO_PIECE;  // root without a legal move: the reference would raise
            over = true;
        }
        ctl->search_no += 1;
        ctl->iter = 0;
        over = over || game_terminal(rg) || (int)rg->rounds >= P.max_rounds;  // ai.py:1610
        if (over) {
            const uint32_t e = atomicAdd(B.end_count, 1u);
            if (e < (uint32_t)B.end_cap) {
                TrlGameEnd ge;
                ge.game_id = rg->game_id;
                ge.winner = rg->players[0].game_over ? 1 : (rg->players[1].game_over ? 0 : -1);
                ge.plies = ctl->search_no; ge.rounds = rg->rounds;
                ge.pieces0 = rg->players[0].pieces; ge.lines_sent0 = ctl->lines_sent0;
                ge.lines_cleared0 = ctl->lines_cleared0; ge.pad_ = 0;
                B.ends[e] = ge;
            } else {
                ctl->status |= TRL_ST_END_OVERFLOW;
            }
            ctl->games_finished += 1;
            ctl->search_no = 0; ctl->lines_sent0 = 0; ctl->lines_cleared0 = 0;
            if (P.restart_finished) {
                const uint32_t id = atomicAdd(B.next_game_id, P.game_id_stride);
                trl_game_setup_scalar(rg, id, P.seed, rg->ruleset);   // the restarted game keeps its ruleset
            } else {
                ctl->active = 0;
            }
        }
    }
    __syncwarp();
    copy_game(reinterpret_cast<uint32_t*>(&B.games[g]), sg, lane);
}

__device__ void expand_body(const TrlSearchBuffers& B, const TrlSearchParams& P, int g, int lane, TrlGame* sgame,
                            const void* __restrict__ values, const void* __restrict__ logits, int logits_stride, int dtype) {
    TrlSearchCtl* ctl = &B.ctl[g];
    if (!ctl->active || ctl->leaf_kind == 3) return;
    const size_t nb = (size_t)g * B.node_cap, sb = (size_t)g * B.state_cap;
    const bool tanh_mode = P.use_tanh != 0;
    const double vmin = tanh_mode ? -1.0 : 0.0;
    const int leaf = ctl->leaf;
    const int kind = ctl->leaf_kind;
    // the selection recorded nodes and state slots along the path: no pointer chasing below when it is valid
    const int* path = B.path ? B.path + (size_t)g * TRL_PATH_INTS : nullptr;
    int pdepth = path ? path[0] : -1;
    if (pdepth >= 0 && path[1 + pdepth] != leaf) pdepth = -1;
    const int ls = pdepth >= 0 ? path[32 + pdepth] : B.slot[nb + leaf];

    TRL_TRACE(g, lane, 1);   // control block and path loaded
    double value;
    if (kind == 2) {
        value = ctl->leaf_value;
    } else {
        value = (double)load_out(values, (size_t)g, dtype == 0 ? 0 : 1);   // gathered logits (dtype 2) come with bf16 values
        // legal placements: enumerated this step, or the list stored under the parent state by a sibling
        const uint16_t* mv = B.legal + (size_t)g * B.moves_cap;
        int C = (kind == 0) ? (int)B.n_legal[g] : 0;
        if (B.movegen_status && !B.movegen_list && lane == 0 && (!B.movegen_index || B.movegen_index[g] >= 0)) {
            const uint32_t st = B.movegen_status[g] & (TRL_ST_QUEUE_OVERFLOW | TRL_ST_MOVES_TRUNC);
            if (st) ctl->status |= st;
        }
        if (B.legal_cache_n && B.movegen_index && leaf != 0) {
            // the selection left the parent's state index in leaf_parent (two dependent loads less)
            const size_t pstate = B.leaf_parent ? (size_t)B.leaf_parent[g] : sb + (size_t)B.slot[nb + B.parent[nb + leaf]];
            const int cached = B.legal_cache_n[pstate];
            uint16_t* slot_mv = B.legal_cache + pstate * (size_t)B.moves_cap;
            if (cached >= 0) {
                mv = slot_mv;
                C = (kind == 0) ? cached : 0;
            } else {
                const int n_store = min((int)B.n_legal[g], B.moves_cap);
                for (int c = lane; c < n_store; c += 32) slot_mv[c] = mv[c];
                __syncwarp();
                if (lane == 0) B.legal_cache_n[pstate] = n_store;
            }
        }
        if (C > B.moves_cap) C = B.moves_cap;
        if (C > 0 && ctl->n_nodes + C > B.node_cap) {  // arena full: the leaf stays childless
            C = 0;
            if (lane == 0) ctl->status |= TRL_ST_ARENA_FULL;
        }
        TRL_TRACE(g, lane, 2);   // legal list located (cache lookup / store)
        if (C > 0) {
            // priors over the legal moves (ai.py:411-443).  softmax over all 11583 logits followed
            // by renormalisation over the legal ones == softmax over the legal logits.
            const size_t lb = (size_t)g * (size_t)logits_stride;
            double mx = -INFINITY;
            // the first 128 legal logits stay in registers between the two passes (one dependent gather chain less)
            float lreg[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int c = lane + 32 * k;
                if (c < C) { lreg[k] = load_logit(logits, lb, mv, c, dtype); mx = fmax(mx, (double)lreg[k]); }
            }
            for (int c = lane + 128; c < C; c += 32) mx = fmax(mx, (double)load_logit(logits, lb, mv, c, dtype));
            mx = warp_max(mx);
            TRL_TRACE(g, lane, 3);   // logits gathered
            const bool root_temp = (leaf == 0) && P.use_root_softmax;
            const double inv_temp = root_temp ? 1.0 / P.root_softmax_temp : 1.0;
            const int base = ctl->n_nodes;
            double sum = 0.0;
            for (int c = lane; c < C; c += 32) {
                const int k = c >> 5;
                const double l = (k < 4) ? (double)(k == 0 ? lreg[0] : k == 1 ? lreg[1] : k == 2 ? lreg[2] : lreg[3])
                                         : (double)load_logit(logits, lb, mv, c, dtype);
                double e = exp((l - mx) * inv_temp);
                if (!(e > 0.0)) e = 1e-25;  // the reference's clamp of underflowed probabilities (ai.py:411)
                B.prior[nb + base + c] = e;
                sum += e;
            }
            sum = warp_sum(sum);
            TRL_TRACE(g, lane, 4);   // exp + first prior store
            const bool noisy = P.training && !ctl->fast && P.use_noise && leaf == 0;  // ai.py:482-499
            double alpha = P.dirichlet_alpha;
            if (noisy && P.use_dirichlet_s) alpha *= P.dirichlet_s / (double)C;
            const uint32_t gid = B.games[g].game_id;
            for (int c = lane; c < C; c += 32) {
                const int id = base + c;
                double pr = B.prior[nb + id] / sum;
                if (noisy) {
                    const double nz = B.noise_override ? B.noise_override[(size_t)g * B.moves_cap + c]
                                                       : trl_gamma(P.seed, gid, ctl->search_no, (uint32_t)c, alpha);
                    pr = pr * (1.0 - P.dirichlet_eps) + nz * P.dirichlet_eps;
                }
                B.prior[nb + id] = pr;
                B.visits[nb + id] = 0; B.value_sum[nb + id] = 0.0;
                B.parent[nb + id] = leaf; B.slot[nb + id] = -1; B.move[nb + id] = mv[c];
            }
            if (lane == 0) {
                B.first_child[sb + ls] = base; B.n_children[sb + ls] = C;
                // FPU of the fresh children (ai.py:449-456)
                B.fpu[sb + ls] = P.fpu_reduction ? fmax(vmin, negate_value(value, tanh_mode)) : fmax(vmin, P.fpu_value);
                ctl->n_nodes = base + C;
            }
        }
    }
    __syncwarp();
    TRL_TRACE(g, lane, 5);   // children created

    // ---- backup (ai.py:511-533) ----
    if (pdepth >= 0) {
        // the selection recorded the path: lane i updates the ancestor at depth i (every node gets exactly one
        // addition, as in the serial walk below)
        const double pos = negate_value(value, tanh_mode);
        const double neg = negate_value(pos, tanh_mode);
        const int leaf_turn = B.states[sb + ls].turn;
        if (lane <= pdepth) {
            const int n = path[1 + lane];
            const int ns = path[32 + lane];
            B.visits[nb + n] += 1;
            B.value_sum[nb + n] += (B.states[sb + ns].turn == leaf_turn) ? pos : neg;
        }
        if (lane == 0) { ctl->iter += 1; ctl->sims += 1; }
    } else if (lane == 0) {
        const double pos = negate_value(value, tanh_mode);
        const double neg = negate_value(pos, tanh_mode);
        const int leaf_turn = B.states[sb + ls].turn;
        int n = leaf;
        while (true) {
            const int ns = B.slot[nb + n];
            B.visits[nb + n] += 1;
            B.value_sum[nb + n] += (B.states[sb + ns].turn == leaf_turn) ? pos : neg;
            if (n == 0) break;
            n = B.parent[nb + n];
        }
        ctl->iter += 1;
        ctl->sims += 1;
    }
    __syncwarp();
    TRL_TRACE(g, lane, 6);   // backup

    // ---- FPU refresh of the played-out node's unvisited siblings (ai.py:542-565) ----
    if (leaf != 0 && P.fpu_reduction) {
        const int par = pdepth >= 1 ? path[pdepth] : B.parent[nb + leaf];
        if (par != 0) {
            const int ps = pdepth >= 1 ? path[32 + pdepth - 1] : B.slot[nb + par];
            const int C = B.n_children[sb + ps], base = B.first_child[sb + ps];
            double explored = 0.0;
            for (int c = lane; c < C; c += 32)
                if (B.visits[nb + base + c] > 0) explored += B.prior[nb + base + c];
            explored = warp_sum(explored);
            if (lane == 0) {
                const double qpar = B.value_sum[nb + par] / (double)B.visits[nb + par];
                B.fpu[sb + ps] = fmax(vmin, negate_value(qpar, tanh_mode) - P.fpu_value * sqrt(explored));
            }
        }
    }
    __syncwarp();
    TRL_TRACE(g, lane, 7);   // FPU refresh

    if (ctl->iter >= ctl->max_iter) finish_search(B, P, g, lane, sgame);
    TRL_TRACE(g, lane, 8);   // (end of search: move choice, record, real move)
}

template <bool BATTLE>
__global__ void __launch_bounds__(kWarps * 32)
search_expand_kernel(TrlSearchBuffers B, TrlSearchParams P, const void* __restrict__ values,
                     const void* __restrict__ logits, int logits_stride, int dtype) {
    __shared__ __align__(16) TrlGame s_game[kWarps];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int g = blockIdx.x * kWarps + wib;
    if (g >= B.n_games) return;
    if (BATTLE) expand_body(B, B.params2[battle_owner(B, g)], g, lane, &s_game[wib], values, logits, logits_stride, dtype);
    else expand_body(B, P, g, lane, &s_game[wib], values, logits, logits_stride, dtype);
}

// expand(t) + select(t+1): the same warp owns game g in both kernels, so running them back to back in
// one launch is exact (a warp only reads what it wrote itself; __syncwarp orders its lanes).
template <bool BATTLE>
__global__ void __launch_bounds__(kWarps * 32, 7)   // 7 blocks per SM: 4096 games are resident in one wave
search_expand_select_kernel(TrlSearchBuffers B, TrlSearchParams P, const void* __restrict__ values,
                            const void* __restrict__ logits, int logits_stride, int dtype) {
    __shared__ __align__(16) TrlGame s_game[kWarps];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int g = blockIdx.x * kWarps + wib;
    trl_grid_dep_wait();
    trl_grid_dep_launch();   // the next kernel (feature encoder / trunk) may move in as our blocks retire
    if (g >= B.n_games) return;
    int si, pi;
    if (BATTLE) {
        // the move that ends a search flips the side to move: the next search may belong to the other network
        expand_body(B, B.params2[battle_owner(B, g)], g, lane, &s_game[wib], values, logits, logits_stride, dtype);
        __syncwarp();
        select_body(B, B.params2[battle_owner(B, g)], g, lane, &s_game[wib], si, pi);
    } else {
        expand_body(B, P, g, lane, &s_game[wib], values, logits, logits_stride, dtype);
        __syncwarp();
        select_body(B, P, g, lane, &s_game[wib], si, pi);
    }
}

// ... + the feature encoding of the selected leaf (features_dev.cuh), straight from the leaf state that
// select left in shared memory: one kernel boundary and one read of the state less per simulation.
template <bool BATTLE>
__global__ void __launch_bounds__(kWarps * 32, 7)
search_expand_select_encode_kernel(TrlSearchBuffers B, TrlSearchParams P, const void* __restrict__ values,
                                   const void* __restrict__ logits, int logits_stride, int dtype, TrlEncodeArgs E) {
    __shared__ __align__(16) TrlGame s_game[kWarps];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int g = blockIdx.x * kWarps + wib;
    trl_grid_dep_wait();
    trl_grid_dep_launch();   // the next kernel (feature encoder / trunk) may move in as our blocks retire
    if (g >= B.n_games) return;
    TRL_TRACE(g, lane, 0);
    int si, pi;
    int2 prow = make_int2(-1, -1);
    if (BATTLE) {
        expand_body(B, B.params2[battle_owner(B, g)], g, lane, &s_game[wib], values, logits, logits_stride, dtype);
        __syncwarp();
        select_body(B, B.params2[battle_owner(B, g)], g, lane, &s_game[wib], si, pi, E.row_of, &prow);
    } else {
        expand_body(B, P, g, lane, &s_game[wib], values, logits, logits_stride, dtype);
        __syncwarp();
        select_body(B, P, g, lane, &s_game[wib], si, pi, E.row_of, &prow);
    }
    __syncwarp();
    if (si < 0) {
        if (lane == 0) { E.own_row[g] = -1; E.opp_row[g] = -1; }
        return;
    }
    int pos = 0;
    if (lane == 0) pos = atomicAdd(E.n_images, (pi < 0) ? 2 : 1);
    pos = __shfl_sync(kFull, pos, 0);
    const int inherit = (pi >= 0) ? ((s_game[wib].turn & 1) ? prow.y : prow.x) : -1;   // parent's cache row of the side to move
    trl_encode_cached_leaf(s_game[wib], g, si, pi, pos, lane, E, inherit);
    TRL_TRACE(g, lane, 13);   // features encoded
}

// ---------------------------------------------------------------------------------------
// policy head on the legal moves only
// ---------------------------------------------------------------------------------------
// The reference evaluates Linear(head_in -> 11583) + softmax for every leaf (architectures.py:141, ai.py:1315-1318)
// and then reads the ~50 entries of the legal moves (ai.py:411-443).  Here one warp per leaf computes exactly those
// entries: logit[c] = bias[m_c] + x . W[m_c] for the leaf's legal list (this step's enumeration or the list cached
// under the parent state, the same lookup as expand_body), fp32 accumulation, fp32 out [G][moves_cap].  The weight
// matrix (12-38 MB) stays L2 resident; no [G, 11584] tensor exists.
__device__ __forceinline__ void mma_bf16_16x8x16(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3]) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// 256-bit read-only global load (sm_100a: LDG.E.ENL2.256).
__device__ __forceinline__ void ldg256(uint32_t (&r)[8], const void* p) {
    asm volatile("ld.global.nc.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) : "l"(p));
}

// Four warps per leaf, each taking every fourth tile of 16 legal moves.  The gathered weight rows are the A operand
// of warp-level MMAs (16 legal moves x 16 inputs per instruction), x is broadcast into all eight B columns, so column
// 0 of D holds the logits; a dot product does not care about the order of its terms, so the K slots of a fragment are
// mapped to memory such that every lane reads 32 contiguous bytes of its two rows per four MMAs.  (A CUDA-core
// version spent 85 instructions per move on unpacking bf16 pairs; this one spends 6.)
//
// What binds is the L1 wavefront queue of the gather (the weight matrix is L2 resident, 216 MB of rows per 4096-leaf
// step): measured 36 us for 4096 leaves with one or four warps per leaf, with 128-bit or 256-bit loads, with x staged
// in shared memory or read through L1 — about 22 B/clk/SM.  Staging the rows in shared memory with cp.async (32 lanes
// along one row per instruction, double buffered) was slower (71 us: LDGSTS costs 8 cycles per instruction and leaves
// 12 warps per SM).  Left: TMA bulk copies of whole rows, which bypass L1 (bound by L2 at about 18 us).
constexpr int kPolicyWarpsPerLeaf = 4;

__global__ void __launch_bounds__(256)
policy_legal_kernel(TrlSearchBuffers B, const __nv_bfloat16* __restrict__ x, int k_pad, const __nv_bfloat16* __restrict__ w,
                    const __nv_bfloat16* __restrict__ bias, float* __restrict__ out) {
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int g = blockIdx.x * (8 / kPolicyWarpsPerLeaf) + wib / kPolicyWarpsPerLeaf, sub = wib % kPolicyWarpsPerLeaf;
    trl_grid_dep_wait();
    if (g >= B.n_games) return;
    const TrlSearchCtl* ctl = &B.ctl[g];
    if (!ctl->active || ctl->leaf_kind != 0) return;
    const uint16_t* mv = B.legal + (size_t)g * B.moves_cap;
    int C = (int)B.n_legal[g];
    if (B.legal_cache_n && B.movegen_index && ctl->leaf != 0) {
        const size_t pstate = B.leaf_parent ? (size_t)B.leaf_parent[g]
                                            : (size_t)g * B.state_cap + (size_t)B.slot[(size_t)g * B.node_cap + B.parent[(size_t)g * B.node_cap + ctl->leaf]];
        const int cached = B.legal_cache_n[pstate];
        if (cached >= 0) { mv = B.legal_cache + pstate * (size_t)B.moves_cap; C = cached; }
    }
    if (C > B.moves_cap) C = B.moves_cap;
    const int chunks = k_pad >> 3;                        // 16-byte pieces of a row
    const uint4* xr = reinterpret_cast<const uint4*>(x + (size_t)g * k_pad);
    float* o = out + (size_t)g * B.moves_cap;
    const int grp = lane >> 2, tig = lane & 3;
    for (int t0 = 16 * sub; t0 < C; t0 += 16 * kPolicyWarpsPerLeaf) {
        const int r0 = min(t0 + grp, C - 1), r1 = min(t0 + grp + 8, C - 1);      // rows past the list repeat the last move
        const int m0 = mv[r0], m1 = mv[r1];
        const uint4* w0 = reinterpret_cast<const uint4*>(w + (size_t)m0 * k_pad);
        const uint4* w1 = reinterpret_cast<const uint4*>(w + (size_t)m1 * k_pad);
        float d[4] = {0.f, 0.f, 0.f, 0.f};
        int kc = 0;                                       // in 16-byte chunks
#pragma unroll 2
        for (; kc + 8 <= chunks; kc += 8) {               // 64 inputs: four MMAs from one 32-byte load per row
            uint32_t u[8], v[8], xv[8];
            ldg256(u, w0 + kc + 2 * tig);
            ldg256(v, w1 + kc + 2 * tig);
            ldg256(xv, xr + kc + 2 * tig);
#pragma unroll
            for (int j = 0; j < 4; ++j) mma_bf16_16x8x16(d, u[2 * j], v[2 * j], u[2 * j + 1], v[2 * j + 1], xv[2 * j], xv[2 * j + 1]);
        }
        for (; kc + 4 <= chunks; kc += 4) {               // 32 inputs: two MMAs from one 16-byte load per row
            const uint4 u = __ldg(w0 + kc + tig), v = __ldg(w1 + kc + tig), xv = __ldg(xr + kc + tig);
            mma_bf16_16x8x16(d, u.x, v.x, u.y, v.y, xv.x, xv.y);
            mma_bf16_16x8x16(d, u.z, v.z, u.w, v.w, xv.z, xv.w);
        }
        if (kc + 2 <= chunks) {                           // 16 more inputs: 8 bytes per lane
            const uint2 u = __ldg(reinterpret_cast<const uint2*>(w0 + kc) + tig), v = __ldg(reinterpret_cast<const uint2*>(w1 + kc) + tig);
            const uint2 xv = __ldg(reinterpret_cast<const uint2*>(xr + kc) + tig);
            mma_bf16_16x8x16(d, u.x, v.x, u.y, v.y, xv.x, xv.y);
        }
        if (tig == 0) {                                   // column 0 of D: rows grp and grp + 8
            if (t0 + grp < C) o[t0 + grp] = d[0] + __bfloat162float(bias[m0]);
            if (t0 + grp + 8 < C) o[t0 + grp + 8] = d[2] + __bfloat162float(bias[m1]);
        }
    }
}

}  // namespace

extern "C" int trl_search_policy_legal(const TrlSearchBuffers* buf, const void* x_bf16, int k_pad, const void* w_bf16,
                                       const void* bias_bf16, float* logits_legal, void* stream) {
    if (!buf || buf->n_games < 0 || !buf->ctl || !buf->legal || !buf->n_legal || !x_bf16 || !w_bf16 || !bias_bf16 || !logits_legal ||
        k_pad <= 0 || (k_pad & 15))
        return TRL_E_ARG;
    if (buf->n_games == 0) return TRL_OK;
    const int leaves_per_block = 8 / kPolicyWarpsPerLeaf;
    return trl_launch_ex(policy_legal_kernel, dim3((buf->n_games + leaves_per_block - 1) / leaves_per_block), dim3(256), 0,
                         (cudaStream_t)stream, true, false, *buf, (const __nv_bfloat16*)x_bf16, k_pad, (const __nv_bfloat16*)w_bf16,
                         (const __nv_bfloat16*)bias_bf16, logits_legal);
}

// instrumented builds (-DTRL_SEARCH_TRACE): [n_games][16] clock64 stamps of the per-step kernel, or NULL to stop
extern "C" int trl_debug_search_trace(long long* device_buffer) {
#ifdef TRL_SEARCH_TRACE
    return trl_check(cudaMemcpyToSymbol(g_search_trace, &device_buffer, sizeof(device_buffer)));
#else
    (void)device_buffer;
    return TRL_E_ARG;
#endif
}

extern "C" int trl_sizeof_search_ctl(void) { return (int)sizeof(TrlSearchCtl); }
extern "C" int trl_sizeof_sample(void) { return (int)sizeof(TrlSample); }
extern "C" int trl_sizeof_root_stats(void) { return (int)sizeof(TrlRootStats); }

// analysis mode stops every game after its first search: random opening plies would never be followed by one
static bool params_ok(const TrlSearchParams* p) { return p && !(p->stop_after_search && p->use_random_start); }

static bool buffers_ok(const TrlSearchBuffers* b) {
    return b && b->n_games >= 0 && b->node_cap > 1 && b->state_cap > 1 && b->moves_cap > 0 && b->prior && b->value_sum &&
           b->visits && b->parent && b->slot && b->move && b->states && b->first_child && b->n_children && b->fpu &&
           b->ctl && b->games && b->leaf_state && b->legal && b->n_legal && b->samples && b->sample_count && b->ends &&
           b->end_count && b->next_game_id;
}

// dtype 0 / 1: dense fp32 / bf16 rows of >= 11583 logits; dtype 2: fp32 rows of moves_cap logits of the legal moves
// (trl_search_policy_legal); the values then are bf16 as with dtype 1
static bool logits_ok(const TrlSearchBuffers* b, int stride, int dtype) {
    if (dtype == 2) return stride >= b->moves_cap;
    return (dtype == 0 || dtype == 1) && stride >= TRL_POLICY_SIZE;
}

extern "C" int trl_search_select(const TrlSearchBuffers* buf, const TrlSearchParams* prm, void* stream) {
    if (!buffers_ok(buf) || !params_ok(prm)) return TRL_E_ARG;
    if (buf->n_games == 0) return TRL_OK;
    const dim3 grid((buf->n_games + kWarps - 1) / kWarps);
    if (buf->params2) search_select_kernel<true><<<grid, kWarps * 32, 0, (cudaStream_t)stream>>>(*buf, *prm);
    else search_select_kernel<false><<<grid, kWarps * 32, 0, (cudaStream_t)stream>>>(*buf, *prm);
    return trl_check(cudaGetLastError());
}

int trl_movegen_indexed(const TrlGame* games, const int32_t* index, int n, uint16_t* moves, int moves_cap,
                        uint16_t* n_moves, uint32_t* status, cudaStream_t stream);  // movegen.cu
int trl_launch_movegen_listed(const TrlGame* games, const int32_t* index, const int32_t* list, uint32_t* count,
                              uint16_t* moves, int moves_cap, uint16_t* n_moves, TrlSearchCtl* ctl, cudaStream_t stream);  // movegen_warp.cu

extern "C" int trl_search_movegen(const TrlSearchBuffers* buf, void* stream) {
    if (!buffers_ok(buf)) return TRL_E_ARG;
    if (buf->n_games == 0) return TRL_OK;
    if (buf->movegen_list && buf->movegen_count && buf->movegen_index)
        return trl_launch_movegen_listed(buf->states, buf->movegen_index, buf->movegen_list, buf->movegen_count,
                                         buf->legal, buf->moves_cap, buf->n_legal, buf->ctl, (cudaStream_t)stream);
    return trl_movegen_indexed(buf->states, buf->movegen_index ? buf->movegen_index : buf->leaf_state, buf->n_games,
                               buf->legal, buf->moves_cap, buf->n_legal, buf->movegen_status, (cudaStream_t)stream);
}

extern "C" int trl_search_expand(const TrlSearchBuffers* buf, const TrlSearchParams* prm, const void* values,
                                 const void* logits, int logits_stride, int dtype, void* stream) {
    if (!buffers_ok(buf) || !params_ok(prm) || !values || !logits || !logits_ok(buf, logits_stride, dtype))
        return TRL_E_ARG;
    if (buf->n_games == 0) return TRL_OK;
    const dim3 grid((buf->n_games + kWarps - 1) / kWarps);
    if (buf->params2) search_expand_kernel<true><<<grid, kWarps * 32, 0, (cudaStream_t)stream>>>(*buf, *prm, values, logits, logits_stride, dtype);
    else search_expand_kernel<false><<<grid, kWarps * 32, 0, (cudaStream_t)stream>>>(*buf, *prm, values, logits, logits_stride, dtype);
    return trl_check(cudaGetLastError());
}

extern "C" int trl_search_expand_select(const TrlSearchBuffers* buf, const TrlSearchParams* prm, const void* values,
                                        const void* logits, int logits_stride, int dtype, void* stream) {
    if (!buffers_ok(buf) || !params_ok(prm) || !values || !logits || !logits_ok(buf, logits_stride, dtype))
        return TRL_E_ARG;
    if (buf->n_games == 0) return TRL_OK;
    return trl_launch_ex(buf->params2 ? search_expand_select_kernel<true> : search_expand_select_kernel<false>,
                         dim3((buf->n_games + kWarps - 1) / kWarps), dim3(kWarps * 32), 0,
                         (cudaStream_t)stream, true, false, *buf, *prm, values, logits, logits_stride, dtype);
}

extern "C" int trl_search_expand_select_encode(const TrlSearchBuffers* buf, const TrlSearchParams* prm, const void* values,
                                               const void* logits, int logits_stride, int dtype, void* cache_bf16,
                                               void* images_bf16, int32_t* image_dest, int32_t* n_images,
                                               void* extras_bf16, int32_t* own_row, int32_t* opp_row, int32_t* row_of,
                                               void* stream) {
    if (!buffers_ok(buf) || !params_ok(prm) || !values || !logits || !logits_ok(buf, logits_stride, dtype) ||
        !buf->leaf_parent || !cache_bf16 || !images_bf16 || !image_dest || !n_images || !extras_bf16 || !own_row || !opp_row ||
        !row_of)
        return TRL_E_ARG;
    if (buf->n_games == 0) return TRL_OK;
    TrlEncodeArgs E;
    E.cache = (__nv_bfloat16*)cache_bf16; E.images = (__nv_bfloat16*)images_bf16; E.image_dest = image_dest;
    E.n_images = n_images; E.extras = (__nv_bfloat16*)extras_bf16; E.own_row = own_row; E.opp_row = opp_row;
    E.row_of = row_of;
    return trl_launch_ex(buf->params2 ? search_expand_select_encode_kernel<true> : search_expand_select_encode_kernel<false>,
                         dim3((buf->n_games + kWarps - 1) / kWarps), dim3(kWarps * 32), 0,
                         (cudaStream_t)stream, true, false, *buf, *prm, values, logits, logits_stride, dtype, E);
}
