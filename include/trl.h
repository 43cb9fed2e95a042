/*
 * trl.h — C ABI of the B200-native self-play hot path (libtrl_b200.so).
 *
 * Drop-in boundary for the data-generation path of mat-lee/tetris-reinforcement-learning.
 * Every entry point names the reference interface it replaces (file:line into the
 * reference checkout).  The reference is pure Python, so the binding a maintainer adds
 * is a ctypes stub (see INTEGRATION.md).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no torch / C++ types in any signature.
 *   - `*_dev` style entry points (the default, no suffix) take caller-allocated DEVICE
 *     pointers and a `cudaStream_t` passed as `void*` (NULL = legacy default stream).
 *     They never allocate, never synchronise, are stream-ordered and CUDA-graph capturable.
 *   - `*_host` entry points take HOST pointers, stage through an internal device
 *     workspace and synchronise before returning (this is what a reference-side caller
 *     such as get_move_matrix(player) binds to).
 *   - devices: a call runs on the CUDA device current in the calling thread, and every
 *     device pointer and stream it receives must belong to that device.  What the library
 *     keeps between calls (workspace, host streams, kernel attributes, debug switches) is
 *     kept per device, so one process may drive several devices (device index < 64).
 *   - return value: 0 = TRL_OK, negative = error (see TRL_E_*); never throws.
 *   - per-item anomalies (queue overflow, no legal move, ...) are reported in a per-item
 *     `status` word (TRL_ST_* bits), not in the return value.
 *
 * Encodings (reference: const.py:6-9, 68, 82-123, 238-281)
 *   - piece id = index into MINOS = "ZLOSIJT": Z0 L1 O2 S3 I4 J5 T6; 255 = none.
 *   - board = 40 rows x uint16; row 0 = top, row 39 = floor; bit c = column c occupied
 *     (reference keeps an object grid; only `!= 0` matters to the rules, board.py:23-30).
 *   - policy tensor (27, 39, 11): flat index = (plane*39 + row)*11 + (x+2), 11583 bits,
 *     bit-packed little-endian into 362 uint32 words (bit i -> word i>>5, bit i&31).
 *   - move = flat policy index (uint16) <-> reference tuple (plane, col=x, row) (ai.py:1022).
 */
#ifndef TRL_H_
#define TRL_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TRL_ROWS 40
#define TRL_COLS 10
#define TRL_SPAWN_Y 17           /* ROWS - SPAWN_ROW, const.py:6-7, piece.py:17-21 */
#define TRL_PREVIEWS 5           /* const.py PREVIEWS */
#define TRL_PLANES 27
#define TRL_POLICY_ROWS 39
#define TRL_POLICY_COLS 11
#define TRL_POLICY_SIZE 11583    /* 27*39*11, const.py:122-123 */
#define TRL_MASK_WORDS 362       /* ceil(11583/32) */
#define TRL_NONE 255
#define TRL_RULESET_S2 0
#define TRL_RULESET_S1 1
#define TRL_QUEUE_CAP 16
#define TRL_RECV_CAP 80

/* return codes */
#define TRL_OK 0
#define TRL_E_ARG (-1)           /* bad argument (NULL pointer, negative size, ...) */
#define TRL_E_CUDA (-2)          /* a CUDA runtime call failed; see trl_last_error() */
#define TRL_E_NOMEM (-3)

/* per-item status bits */
#define TRL_ST_QUEUE_OVERFLOW 0x1u   /* movegen exploration FIFO exceeded its capacity  */
#define TRL_ST_MOVES_TRUNC    0x2u   /* compact move list truncated at moves_cap        */
#define TRL_ST_NO_PIECE       0x4u   /* cur == none and alt == none (Game.no_move)      */
#define TRL_ST_RECV_OVERFLOW  0x8u   /* pending-garbage list exceeded TRL_RECV_CAP      */
#define TRL_ST_BAD_MOVE       0x10u  /* env step: move index out of range / undecodable */
#define TRL_ST_SAMPLE_OVERFLOW 0x20u /* search: the TrlSample ring was full, a record was dropped */
#define TRL_ST_ARENA_FULL     0x40u  /* search: node arena full, a leaf stayed childless */
#define TRL_ST_END_OVERFLOW   0x80u  /* search: the TrlGameEnd ring was full, a record was dropped */

/*
 * One player.  Mirrors the fields Player.copy() carries (player.py:217-233):
 * board, queue, stats.{pieces,b2b,b2b_level,combo}, game_over, piece, held_piece,
 * garbage_to_receive.  The active piece is stored as a type only: between moves it always
 * sits at its spawn location (piece.py:17-21), Game.move_piece overwrites x/y/rot
 * (game.py:56-64).  192 bytes.
 */
typedef struct TrlPlayer {
    uint16_t rows[TRL_ROWS];         /* 0   board bitrows                                 */
    int32_t  pieces;                 /* 80  stats.pieces                                  */
    int16_t  b2b;                    /* 84  stats.b2b (starts at -1)                      */
    int16_t  combo;                  /* 86  stats.combo                                   */
    uint8_t  qlen;                   /* 88  len(queue.pieces)                             */
    uint8_t  piece;                  /* 89  active piece type or TRL_NONE                 */
    uint8_t  held;                   /* 90  held piece type or TRL_NONE                   */
    uint8_t  game_over;              /* 91                                               */
    uint8_t  b2b_level;              /* 92  stats.b2b_level                               */
    uint8_t  n_recv;                 /* 93  len(garbage_to_receive)                       */
    uint8_t  pad_[2];                /* 94                                               */
    uint8_t  queue[TRL_QUEUE_CAP];   /* 96  queue.pieces, index 0 = next                  */
    uint8_t  recv[TRL_RECV_CAP];     /* 112 garbage_to_receive hole columns, 0 = first    */
} TrlPlayer;

/* Two-player game (game.py:6-32).  400 bytes. */
typedef struct TrlGame {
    TrlPlayer players[2];            /* 0                                                 */
    uint8_t  turn;                   /* 384 index of the side to move                     */
    uint8_t  ruleset;                /* 385 0 = TETR.IO season 2 ('s2', default), 1 = season 1 ('s1'):
                                            attack table (stats.py:49-86 / 88-129) and the s2-only
                                            all-spin rule (player.py:145-151)                     */
    uint16_t bag_ctr;                /* 386 number of 7-bag refills dealt so far          */
    uint32_t rounds;                 /* 388 len(history.states) (game.py:86-87)           */
    uint32_t rng_ctr;                /* 392 counter for the next garbage-column draw      */
    uint32_t game_id;                /* 396 Philox stream id (global game index)          */
} TrlGame;

/* Per-step outputs of the env step (what Player.place_piece computes, player.py:109-188). */
typedef struct TrlStepOut {
    uint8_t rows_cleared;            /* 0..4                                              */
    uint8_t attack;                  /* lines sent by Stats.get_attack (stats.py:88-129)  */
    uint8_t flags;                   /* bit0 tspin, bit1 mini, bit2 all_clear, bit3 held, */
                                     /* bit4 mover topped out, bit5 garbage received      */
    uint8_t garbage_col;             /* hole column drawn (valid iff attack > 0)          */
    uint32_t status;                 /* TRL_ST_* bits                                     */
} TrlStepOut;

/* ------------------------------------------------------------------------------------ */
/* library                                                                               */
/* ------------------------------------------------------------------------------------ */

/* ABI version of this header; bumped on any incompatible change. */
int trl_abi_version(void);

/* Programmatic dependent launch between the kernels of a self-play step (default on): the trunk kernel
 * becomes resident and loads its weights while the search kernel before it drains.  0 switches it off
 * (for A/B timing; results are identical either way). */
void trl_set_pdl(int enabled);

/* Profiling aid: a one-thread kernel writes the GPU's %globaltimer (ns) to *slot in stream order. */
int trl_stamp_globaltimer(unsigned long long* slot, void* stream);
/* Text of the last CUDA error seen by this thread's calls ("" if none). */
const char* trl_last_error(void);
/* sizeof checks for bindings: returns sizeof(TrlPlayer) / sizeof(TrlGame). */
int trl_sizeof_player(void);
int trl_sizeof_game(void);

/* ------------------------------------------------------------------------------------ */
/* legal-placement enumeration                                                           */
/* replaces move_generation.get_move_matrix(player, algo='convolutional')                */
/*   (move_generation.py:752-789 -> MoveGenerator.generate_moves :77-105,                */
/*    _generate_moves_for_piece :107-149, _convolutional_algorithm :325-488,             */
/*    _build_validity_maps :490-528, _convert_placements_to_policy :650-749)             */
/* and ai.get_move_list's argwhere ordering (ai.py:1016-1024).                           */
/* ------------------------------------------------------------------------------------ */

/*
 * boards   [n][40] uint16   board of the player to move
 * cur      [n]     uint8    active piece type (TRL_NONE if player.piece is None)
 * alt      [n]     uint8    held piece if any, else queue[0] if any, else TRL_NONE
 *                           (move_generation.py:91-105); the alt piece is only legal if it
 *                           can spawn (Player.hold_piece -> create_piece, player.py:37-44)
 * mask_bits[n][362] uint32  OUT bit-packed (27,39,11) legal mask; may be NULL
 * moves    [n][moves_cap] uint16 OUT ascending flat policy indices (= np.argwhere order);
 *                           may be NULL
 * n_moves  [n]     uint16   OUT number of legal placements (always the full count); may be NULL
 * status   [n]     uint32   OUT TRL_ST_* bits; may be NULL
 */
int trl_movegen(const uint16_t* boards, const uint8_t* cur, const uint8_t* alt, int n,
                uint32_t* mask_bits, uint16_t* moves, int moves_cap, uint16_t* n_moves,
                uint32_t* status, void* stream);

/* Same, on the side-to-move player of packed games (cur/alt derived on device). */
int trl_movegen_games(const TrlGame* games, int n, uint32_t* mask_bits, uint16_t* moves,
                      int moves_cap, uint16_t* n_moves, uint32_t* status, void* stream);

/* HOST-buffer variant of trl_movegen: copies in, runs, copies out, synchronises. */
int trl_movegen_host(const uint16_t* boards, const uint8_t* cur, const uint8_t* alt, int n,
                     uint32_t* mask_bits, uint16_t* moves, int moves_cap, uint16_t* n_moves,
                     uint32_t* status);

/*
 * trl_movegen_host with COMPACT output: the ascending move lists (np.argwhere order, what
 * get_move_list consumes, ai.py:1016-1024) of all calls packed back to back without padding.  Call i
 * owns moves_compact[offsets[i] .. offsets[i] + n_moves[i]).  Only 2 B per placement + 14 B per call
 * cross PCIe (the bit-packed mask is 1448 B per call).  capacity = length of moves_compact in
 * elements (TRL_E_ARG if too small); *total_out = number of placements written.
 */
int trl_movegen_host_compact(const uint16_t* boards, const uint8_t* cur, const uint8_t* alt, int n,
                             uint16_t* moves_compact, uint64_t capacity, uint64_t* offsets,
                             uint16_t* n_moves, uint32_t* status, uint64_t* total_out);

/*
 * Host movegen over SHARED boards with byte-coded move lists.  Each distinct board crosses PCIe once:
 * call i enumerates boards[board_index[i]] with cur[i] / alt[i] (so "every piece on each board" needs
 * no copies of the board), and its ascending move list (np.argwhere order) comes back as about 1 B
 * per placement.
 *
 * boards      [n_boards][40] uint16   the distinct boards
 * board_index [n]  uint32             board of call i; an index >= n_boards reads nothing and the call
 *                                     returns TRL_E_ARG once the run has finished (checked on the device)
 * cur, alt    [n]  uint8              as in trl_movegen
 * codes       [codes_cap] uint8       OUT, *codes_total bytes written
 * escapes     [esc_cap]  uint16       OUT, *esc_total entries written
 * n_moves     [n]  uint16             OUT number of placements of each call
 * flag_index, flag_status [flag_cap] uint32  OUT, *n_flagged entries: the calls whose TRL_ST_* word is
 *                                     not zero, as (call index, status) in ascending call index; every
 *                                     other call has status 0
 *
 * Format.  Calls are encoded in call order into the two shared streams.  For each move m of call i let
 * prev be the call's previous move (-1 before its first) and d = m - prev, 1 <= d <= 11583:
 *     d <= 255:  byte d is appended to codes
 *     d >  255:  byte 0 is appended to codes and d (uint16) to escapes
 * A call has at most 45 escapes.  Decoding needs no per-call loop (numpy):
 *     d = codes.astype(int64); d[codes == 0] = escapes
 *     cs = cumsum(d); start = cumsum(n_moves) - n_moves
 *     moves = cs - repeat(where(start > 0, cs[start - 1], 0), n_moves) - 1
 * (move_generation.decode_move_codes).  The bytes depend on the input alone, not on the run.
 *
 * TRL_E_ARG: a NULL pointer, n < 0, n > 0 with n_boards <= 0, a board index out of range, an output
 * buffer too small, or a chunk of 131072 calls averaging more than 512 placements per call (the
 * device staging).  Runs on the current device and returns when every output has landed.
 */
int trl_movegen_host_boards(const uint16_t* boards, int n_boards, const uint32_t* board_index,
                            const uint8_t* cur, const uint8_t* alt, int n, uint8_t* codes,
                            uint64_t codes_cap, uint16_t* escapes, uint64_t esc_cap, uint16_t* n_moves,
                            uint32_t* flag_index, uint32_t* flag_status, uint64_t flag_cap,
                            uint64_t* codes_total, uint64_t* esc_total, uint64_t* n_flagged);

/* Kernel used by every trl_movegen* entry point: 0 = one thread per call (csrc/movegen.cu),
 * 1 = one warp per piece search (csrc/movegen_warp.cu), -1 = automatic (default).  Both produce
 * bit-identical outputs; the choice only trades latency against throughput. */
void trl_movegen_select_kernel(int kernel);

/* Form of the warp-cooperative enumeration (csrc/movegen_warp.cu): 0 = two warps per call, one per piece
 * type (lowest latency: the few-thousand-call batches of a self-play step), 1 = one warp per call,
 * both piece searches back to back, 2 = passes: a small kernel with the row-parallel closure search
 * alone, then the T order analysis and the exact T search for the T searches it deferred, and one warp per call
 * for the few calls it could not handle (highest throughput: the multi-million-call sweeps of
 * move_generation.py:752-789), -1 = by batch size (default).
 * Bit-identical outputs. */
void trl_movegen_warp_form(int form);

/* ------------------------------------------------------------------------------------ */
/* env step                                                                              */
/* replaces Game.make_move(move, add_bag, add_history=False)                             */
/*   (game.py:40-118: move_piece, place, check_garbage; player.py:29-44, 109-205;        */
/*    board.py:12-21; stats.py:30-43, 88-129 [ruleset s2]; piece_queue.py:17-20)          */
/* ------------------------------------------------------------------------------------ */

/*
 * games  [n] TrlGame  IN/OUT, stepped in place
 * moves  [n] uint16   flat policy index of the move of the side to move; 0xFFFF = skip item
 * out    [n] TrlStepOut OUT; may be NULL
 * add_bag  != 0: refill both queues with a fresh 7-bag when the mover's queue drops below 5
 *          (game.py:82-83); bags come from Philox(seed, game_id, bag stream)
 * seed     Philox key; the garbage hole column (player.py:184-186) is
 *          draw(seed, game_id, games[i].rng_ctr++) — one draw per placement with attack > 0
 */
int trl_env_step(TrlGame* games, const uint16_t* moves, int n, TrlStepOut* out, int add_bag,
                 uint64_t seed, void* stream);
int trl_env_step_host(TrlGame* games, const uint16_t* moves, int n, TrlStepOut* out,
                      int add_bag, uint64_t seed);

/*
 * Game() + Game.setup() (game.py:8-38): empty boards, one 7-bag each (player 0 first),
 * first piece spawned, turn = 0, rounds = 1.  game_id[i] = first_game_id + i * id_stride
 * (id_stride = number of ranks when games are sharded over GPUs).
 */
int trl_game_setup(TrlGame* games, int n, uint32_t first_game_id, uint32_t id_stride, uint64_t seed,
                   void* stream);
int trl_game_setup_host(TrlGame* games, int n, uint32_t first_game_id, uint32_t id_stride, uint64_t seed);

/* ------------------------------------------------------------------------------------ */
/* network input encoding                                                                */
/* replaces ai.game_to_X + get_grids/get_pieces/get_stat/get_garbage/simplify_grid        */
/*   (ai.py:1364-1413) and the tensor stacking of BatchedEvaluator._dispatch (ai.py:724-731) */
/* ------------------------------------------------------------------------------------ */

/*
 * games  [*] TrlGame; item i encodes games[index ? index[i] : i]
 * grids  [2n][400]  OUT rows 0..n-1: grid of the side to move, rows n..2n-1: opponent (0/1)
 * extras [n][105]   OUT a_pieces(49) a_b2b a_combo a_garbage o_pieces(49) o_b2b o_combo
 *                       o_garbage color  — the non-grid inputs in torch.cat order
 *                       (architectures.py:128-140)
 * dtype  0 = float32, 1 = bfloat16
 */
int trl_encode_features(const TrlGame* games, const int32_t* index, int n, void* grids,
                        void* extras, int dtype, void* stream);

/* ------------------------------------------------------------------------------------ */
/* search (MCTS / PUCT) and the self-play episode                                         */
/* replaces ai.MCTS / amcts (ai.py:299-659, 766-996), MCTSNode/MCTSTree/NodeState         */
/*   (ai.py:237-297), get_move_list (ai.py:1016-1024), the policy clamp + root softmax +   */
/*   normalisation (ai.py:411-443), search_statistics' visit counts (ai.py:1330-1361) and  */
/*   the per-move part of play_game (ai.py:1610-1668: search -> record -> make_move).      */
/* The tree lives in HBM as struct-of-arrays; one warp per game; one leaf per game per     */
/* step (exactly the reference's BatchedEvaluator shape, ai.py:670-742).                   */
/* ------------------------------------------------------------------------------------ */

#define TRL_SAMPLE_MOVES 512

/* Config's search fields (ai.py:97-137), doubles where the reference computes in float64. */
typedef struct TrlSearchParams {
    uint64_t seed;
    double cpuct, dpuct;               /* CPUCT, DPUCT                                     */
    double fpu_value;                  /* FpuValue                                         */
    double root_softmax_temp;          /* RootSoftmaxTemp                                  */
    double temperature;                /* temperature (used only when training)            */
    double playout_cap_chance;         /* playout_cap_chance                               */
    double dirichlet_alpha, dirichlet_s, dirichlet_eps; /* DIRICHLET_ALPHA / _S / _EXPLORATION */
    double c_forced;                   /* CForcedPlayout                                   */
    int32_t max_iter;                  /* MAX_ITER                                         */
    int32_t iters_long, iters_short;   /* playout-cap iteration counts (ai.py:323-330)     */
    int32_t fpu_reduction;             /* FpuStrategy == 'reduction' (else 'absolute')     */
    int32_t use_root_softmax;
    int32_t training;
    int32_t use_playout_cap;           /* use_playout_cap_randomization                    */
    int32_t use_noise;                 /* use_dirichlet_noise                              */
    int32_t use_dirichlet_s;
    int32_t use_forced;                /* use_forced_playouts_and_policy_target_pruning    */
    int32_t use_tanh;
    int32_t save_all;
    int32_t max_rounds;                /* MAX_MOVES = 1000 (const.py:12)                   */
    int32_t restart_finished;          /* != 0: a finished game is replaced by a fresh one */
    uint32_t game_id_stride;           /* new game id = previous id + stride (ranks interleave) */
    int32_t use_random_start;          /* use_random_starting_moves (ai.py:1588-1608)      */
    double random_start_scale;         /* 0.04 * DIRICHLET_S: mean of the exponential number of opening plies */
    int32_t stop_after_search;         /* != 0: analysis mode.  A finished search always emits its TrlSample (saved
                                          still reports the playout-cap coin), plays no move, emits no TrlGameEnd,
                                          leaves games[g] untouched and parks the slot (ctl.active = 0, ctl.iter = 0),
                                          so every game stops after its own search.  Incompatible with
                                          use_random_start (TRL_E_ARG). */
    int32_t pad_;
} TrlSearchParams;

/* Per-game search control block. */
typedef struct TrlSearchCtl {
    int32_t iter;                      /* iterations done in the running search (0 = not started) */
    int32_t max_iter;                  /* iteration budget of the running search           */
    int32_t n_nodes, n_states;
    int32_t leaf;                      /* node selected in this step                       */
    int32_t leaf_kind;                 /* 0 expand, 1 evaluate only (no_move), 2 terminal, 3 idle */
    uint32_t search_no;                /* searches finished in this game (= plies played)  */
    uint32_t garbage_ctr;              /* sequential garbage draws inside the running search */
    uint32_t status;                   /* sticky TRL_ST_* bits                             */
    uint32_t fast;                     /* playout-cap short search: no noise, not saved    */
    uint32_t active;                   /* 0 = slot parked (game over and no restart)       */
    uint32_t games_finished;
    uint64_t sims;                     /* simulations run in this slot                     */
    int32_t lines_sent0, lines_cleared0; /* player 0 totals of the running game (ai.py:1518-1529) */
    double leaf_value;                 /* value of a terminal leaf                         */
    int32_t max_depth;
    int32_t random_left;               /* random opening plies still to play in this game (ai.py:1604-1610) */
} TrlSearchCtl;

/* One finished search = one training position before augmentation (ai.py:1611-1666). */
typedef struct TrlSample {
    uint32_t game_id;
    uint16_t search_no;
    uint8_t turn;                      /* side to move = owner of the sample                */
    uint8_t saved;                     /* reference `save` flag (False for fast searches)   */
    uint16_t n_children;
    uint16_t chosen_move;
    uint32_t total_visits;             /* sum of post-prune visits                          */
    int32_t iterations;
    TrlGame state;                     /* position searched (queues cut to 5 previews)      */
    uint16_t moves[TRL_SAMPLE_MOVES];  /* root children in creation (argwhere) order        */
    uint16_t visits[TRL_SAMPLE_MOVES]; /* post-prune visit counts                           */
    uint16_t visits_pre[TRL_SAMPLE_MOVES]; /* pre-prune visit counts                        */
} TrlSample;

/* One finished game (ai.py:1675-1699). */
typedef struct TrlGameEnd {
    uint32_t game_id;
    int32_t winner;                    /* 0 / 1, -1 = draw (MAX_MOVES reached)              */
    uint32_t plies;
    uint32_t rounds;
    int32_t pieces0, lines_sent0, lines_cleared0, pad_;
} TrlGameEnd;

#define TRL_PV_MAX 16

/* Root statistics of one finished search (the reference's MCTSTree root, ai.py:237-297), written to the slot of
 * the search's TrlSample: root_stats[i] belongs to samples[i].  Every value is read before policy-target
 * pruning, which changes visit counts only. */
typedef struct TrlRootStats {
    float root_value;                  /* root value_sum / visits (root.value_avg)                 */
    uint32_t root_visits;
    int32_t slot;                      /* game index g of the search in the batch                  */
    uint16_t n_children;               /* = the sample's n_children                                */
    uint16_t pv_len;                   /* plies in pv (0..TRL_PV_MAX)                               */
    uint32_t pv_visits[TRL_PV_MAX];    /* visit count of each ply's node                            */
    uint16_t pv[TRL_PV_MAX];           /* principal variation as policy indices: from the root, the most visited
                                          child (last maximum, as the move choice), while it has visits   */
    float prior[TRL_SAMPLE_MOVES];     /* per root child, sample order: the prior the PUCT used (after the root
                                          softmax temperature and the Gamma noise mix)              */
    float q[TRL_SAMPLE_MOVES];         /* value_sum / visits; for an unvisited child the FPU value the
                                          selection used                                            */
} TrlRootStats;

/* All device buffers of a search batch; caller-allocated (sizes in elements). */
typedef struct TrlSearchBuffers {
    int32_t n_games, node_cap, state_cap, moves_cap, sample_cap, end_cap, pad0_, pad1_;
    /* tree, per node [n_games * node_cap] */
    double* prior; double* value_sum; int32_t* visits; int32_t* parent; int32_t* slot; uint16_t* move;
    /* per materialised state [n_games * state_cap] */
    TrlGame* states; int32_t* first_child; int32_t* n_children; double* fpu;
    /* per game [n_games] */
    TrlSearchCtl* ctl; TrlGame* games; int32_t* leaf_state;
    uint16_t* legal; uint16_t* n_legal;      /* [n_games * moves_cap], [n_games]            */
    /* outputs */
    TrlSample* samples; uint32_t* sample_count; TrlGameEnd* ends; uint32_t* end_count;
    uint32_t* next_game_id;                  /* [1] id given to the next restarted game     */
    const double* noise_override;            /* [n_games * moves_cap] or NULL (tests)       */
    int32_t* leaf_parent;                    /* [n_games] state index of the leaf's parent, -1 = the leaf is
                                                the root / nothing to evaluate (may be NULL)            */
    /* Exact reuse of legal-placement lists between siblings (all three NULL = off).  A move changes
     * neither the OTHER player's board nor its pieces (player.py:109-188, game.py:66-118), so every
     * child of a state has the same side-to-move board / piece / hold and hence the same
     * get_move_matrix: the list is enumerated for the first child that becomes a leaf and stored
     * under the parent state. */
    uint16_t* legal_cache;                   /* [n_games * state_cap * moves_cap]                        */
    int32_t* legal_cache_n;                  /* [n_games * state_cap] number of cached moves, -1 = none  */
    int32_t* movegen_index;                  /* [n_games] state to enumerate this step or -1 (cache hit)  */
    /* Compacted work list of the leaf enumeration (both NULL = off: trl_search_movegen then walks
     * movegen_index with one call slot per game).  trl_search_select appends every game whose leaf needs
     * an enumeration; trl_search_movegen consumes the list with as few, fully occupied thread blocks as
     * the count needs (one 16-call block per SM), so the SMs it does not use are free for the network
     * kernels that run beside it, and leaves both counters at zero for the next step. */
    int32_t* path;                           /* [n_games * 64] or NULL: [0] depth of the selected leaf (-1: deeper
                                                than 30), [1 + i] node and [32 + i] state slot at depth i; lets
                                                expand / backup work without walking parent and slot links     */
    int32_t* movegen_list;                   /* [n_games] game indices, arbitrary order                   */
    uint32_t* movegen_count;                 /* [4] entries in movegen_list; finished blocks; next ticket; pad.
                                                Zero between steps (the enumeration kernel resets them)    */
    uint32_t* movegen_status;                /* [n_games] or NULL: TRL_ST_* bits of the uncompacted enumeration
                                                (movegen_list == NULL); trl_search_expand folds them into
                                                ctl.status.  The compacted enumeration writes ctl.status itself */
    const struct TrlSearchParams* params2;   /* NULL, or a DEVICE array of two parameter sets = gating battle
                                                (ai.py:1975-2114): the search of game g runs with
                                                params2[(game_id ^ side to move at the root) & 1], i.e. network 1
                                                plays player (game_id & 1) (colours alternate, ai.py:2087-2091);
                                                the `prm` argument of the calls is then ignored             */
    TrlRootStats* root_stats;                /* [sample_cap] or NULL (off): a search that writes samples[i] also
                                                writes root_stats[i]                                         */
} TrlSearchBuffers;

int trl_sizeof_search_ctl(void);
int trl_sizeof_sample(void);
int trl_sizeof_root_stats(void);

/* Step part 1: (start a search if needed,) select a leaf per game and materialise its state;
 * writes leaf_state[g] = index into `states` of the position the net must evaluate, or -1, and
 * (if leaf_parent != NULL) leaf_parent[g] = index of the state it was reached from, or -1. */
int trl_search_select(const TrlSearchBuffers* buf, const TrlSearchParams* prm, void* stream);

/* Legal placements for the selected leaves: trl_movegen_games on states[leaf_state[g]] (with the
 * sibling cache: only on states[movegen_index[g]], the leaves whose parent has no list yet). */
int trl_search_movegen(const TrlSearchBuffers* buf, void* stream);

/* Tuning knob of the compacted enumeration: calls served per call slot (default 1; 1..6 measured equal within noise on B200).  With r rounds
 * ceil(count / (16 r)) SMs work on the list, for about r search latencies. */
void trl_search_movegen_rounds(int rounds);

/* Step part 2: expand the leaf with the network outputs (values [n_games], logits
 * [n_games][logits_stride >= 11583]; dtype 0 = float32, 1 = bfloat16), root noise, backup, FPU refresh; when a
 * search has used its iteration budget: choose the move, prune, emit the sample, play the move
 * on the real game, emit the game end and restart. */
int trl_search_expand(const TrlSearchBuffers* buf, const TrlSearchParams* prm, const void* values,
                      const void* logits, int logits_stride, int dtype, void* stream);

/* trl_search_expand immediately followed by the NEXT step's trl_search_select in one kernel (the same
 * warp owns a game in both, so the fusion is exact): saves a kernel boundary per simulation.  The
 * caller runs trl_search_select once before the first step and then only movegen -> network ->
 * trl_search_expand_select per step. */
int trl_search_expand_select(const TrlSearchBuffers* buf, const TrlSearchParams* prm, const void* values,
                             const void* logits, int logits_stride, int dtype, void* stream);

/* ... and additionally trl_encode_features_cached for the selected leaves (arguments as there), from the
 * leaf state the selection left in shared memory.  *n_images must be zero on entry (the trunk kernel of
 * the step that produced `logits` has reset it).  The caller runs trl_search_select +
 * trl_encode_features_cached once before the first step. */
int trl_search_expand_select_encode(const TrlSearchBuffers* buf, const TrlSearchParams* prm, const void* values,
                                    const void* logits, int logits_stride, int dtype, void* cache_bf16,
                                    void* images_bf16, int32_t* image_dest, int32_t* n_images, void* extras_bf16,
                                    int32_t* own_row, int32_t* opp_row, int32_t* row_of, void* stream);

/*
 * Policy head on the legal moves only.  The reference computes Linear(head_in -> 11583) for every leaf
 * (architectures.py:141) and then reads the entries of the legal moves (ai.py:411-443); this call computes exactly
 * those: logits_legal[g][c] = bias[m] + x[g] . w[m] for the c-th legal move m of game g's selected leaf (this
 * step's enumeration, or the list cached under the parent state), fp32.  Run it after trl_search_movegen and before
 * trl_search_expand*, and pass logits_legal to expand with dtype = 2 and logits_stride = moves_cap (values bf16).
 * x [n_games][k_pad] bf16 (k_pad % 16 == 0), w [>= 11583][k_pad] bf16 row-major, bias [>= 11583] bf16,
 * logits_legal [n_games][moves_cap] f32.
 */
int trl_search_policy_legal(const TrlSearchBuffers* buf, const void* x_bf16, int k_pad, const void* w_bf16,
                            const void* bias_bf16, float* logits_legal, void* stream);

/* ------------------------------------------------------------------------------------ */
/* fused convolutional trunk of the policy/value net (tcgen05 tensor cores)               */
/* replaces AlphaSame.process_grid (architectures.py:120-126, blocks :27-57) in eval mode  */
/* for filters = 16, kernels = 1: conv5x5 stem -> n_blocks pre-activation residual blocks  */
/* -> BN-ReLU -> conv1x1 -> BN-ReLU -> flatten.                                            */
/* ------------------------------------------------------------------------------------ */

/*
 * grids    [n_images][400] bf16 0/1 board cells (row-major 40 x 10)
 * w_packed [2*n_blocks][9][2][2][8][8] bf16: per 3x3 tap the 16x16 weight matrix in the UMMA
 *          K-major core-matrix order [k chunk][n group][n][k] (bn2 scale folded into conv 1)
 * consts   [n_blocks*48 + 50] f32: per block bn1 scale[16], bn1 bias[16], bn2 bias[16]; then
 *          final bn scale[16], bias[16], 1x1 weights[16], last bn scale, bias
 * stem_lut [5][32][16] f32: partial sums of the 5x5 stem per kernel row and 5-bit input pattern
 * out      [n_images][400] bf16 trunk features
 */
int trl_alphasame_trunk(const void* grids_bf16, int n_images, int n_blocks, const void* w_packed,
                        const float* consts, const float* stem_lut, void* out_bf16, void* stream);

/*
 * Same operator, row-Toeplitz formulation (csrc/trunk_rows.cu): one MMA row per board row, the
 * horizontal taps folded into N (M=128 N=48 K=16 per input column and vertical tap), all weights
 * resident in shared memory, column-wavefront overlap of tensor pipe and epilogue.
 * w_packed [2*n_blocks][3 dy][2][6][8][8] bf16: per vertical tap the 48 x 16 matrix
 *          B[(j, oc), ic] = w[oc][ic][dy][2 - j] in K-major core-matrix order [k chunk][n group][n][k].
 * stem_w   [5 dy][2][20][8][8] bf16: the 5x5 stem as 5 MMAs (M=128 N=160 K=16): per kernel row the
 *          160 x 16 matrix B[(x_out, oc), k] = w[oc][dy][k - x_out] (k = input column + 2, else 0).
 * consts   as above but a HOST pointer: the folded BatchNorm constants are passed to the kernel by
 *          value (constant bank), so they cost no shared-memory bandwidth.
 * Other arguments as above.  n_blocks <= trl_alphasame_trunk_rows_max_blocks().
 */
int trl_alphasame_trunk_rows(const void* grids_bf16, int n_images, int n_blocks, const void* w_packed,
                             const float* consts, const void* stem_w, void* out_bf16, void* stream);
int trl_alphasame_trunk_rows_max_blocks(void);

/*
 * Trunk-feature reuse inside a search (exact, not an approximation).  A move only changes the
 * MOVER's board (player.py:154-176; garbage rises on the mover's own board, game.py:100-117, the
 * opponent only gets entries appended to its pending list), and AlphaSame runs the SAME trunk on
 * both boards (architectures.py:120-133).  So for a leaf reached from `parent`, the features of
 * the side to move's board are those already computed for `parent`; only the mover's new board
 * needs the trunk.  `cache` holds [n_states][2 players][400] bf16 trunk outputs.
 *
 * trl_encode_features_cached: per leaf g (leaf_state[g] >= 0) writes extras[g] (as
 * trl_encode_features), lets the leaf inherit the parent's cache row of the side to move
 * (row_of[leaf][side to move] = row_of[parent][side to move]; row_of is [n_states * 2]: the cache row
 * holding the features of (state, player); for a root leaf that board is queued too), appends the 0/1
 * cells of every board that needs the trunk to
 * `images` ([<= 2n][400] bf16, compact, *n_images = count) with image_dest[k] = cache row
 * (state*2 + player) the trunk must write, and sets own_row[g] / opp_row[g] = cache rows the heads
 * read (or -1).  *n_images must be zero on entry.
 */
int trl_encode_features_cached(const TrlGame* states, const int32_t* leaf_state, const int32_t* leaf_parent, int n,
                               void* cache_bf16, void* images_bf16, int32_t* image_dest, int32_t* n_images,
                               void* extras_bf16, int32_t* own_row, int32_t* opp_row, int32_t* row_of, void* stream);

/* trl_alphasame_trunk_rows with a device-side image count and scattered output rows:
 * out_bf16[out_row[k]][400] = trunk(images[k]) for k < *n_images_dev (capacity max_images).
 * The kernel resets *n_images_dev to 0 when it has consumed it (no memset per step). */
int trl_alphasame_trunk_rows_indexed(const void* images_bf16, int32_t* n_images_dev, int max_images,
                                     const int32_t* out_row, int n_blocks, const void* w_packed, const float* consts,
                                     const void* stem_w, void* out_bf16, void* stream);

/* Gate for a forked stream: work submitted to `stream` after this call starts only once every CTA of the
 * most recent trl_alphasame_trunk_rows_indexed launch is resident (or after 100 us).  The self-play step
 * uses it to queue the leaf enumeration BEHIND the trunk: its blocks then take over SMs as trunk CTAs
 * run out of work instead of delaying trunk CTAs at the start. */
int trl_alphasame_trunk_rows_gate(void* stream);

/* trl_alphasame_heads reading its two feature rows through indices into a cache
 * ([rows][400] bf16; own_row[g] < 0: leaf skipped). */
int trl_alphasame_heads_indexed(const void* cache_bf16, const int32_t* own_row, const int32_t* opp_row,
                                const void* extras_bf16, int n_leaves, const float* weights, int use_tanh,
                                void* x_out_bf16, void* value_out_bf16, void* stream);

/*
 * Tail of AlphaSame.forward between the trunk and the policy GEMM (architectures.py:128-142), fused:
 * osidedense (Linear 400->16, BN1d, ReLU) on the opponent features, the 521-wide concatenation
 * (written 528 wide, zero padded, bf16) and the value head (Linear 521->16, BN1d, ReLU, Linear 16->1,
 * Sigmoid|Tanh).  feats [2n][400] bf16 (own grids, then opponent grids), extras [n][105] bf16,
 * weights fp32 [trl_alphasame_heads_weight_floats()]: Wo_t[400][16], bo[16], Wv_t[528][16], bv[16],
 * w2[16], b2 (BatchNorm folded).  x_out [n][528] bf16, value_out [n] bf16.
 */
int trl_alphasame_heads(const void* feats_bf16, const void* extras_bf16, int n_leaves, const float* weights,
                        int use_tanh, void* x_out_bf16, void* value_out_bf16, void* stream);
int trl_alphasame_heads_weight_floats(void);

/* ------------------------------------------------------------------------------------ */
/* wide fused trunk (csrc/trunk_wide.cu): 32 or 64 filters, both block styles              */
/* replaces, in eval mode with BatchNorm folded,                                           */
/*   post_act = 0: AlphaSame.process_grid (architectures.py:120-126; pre-activation blocks */
/*                 :27-57; 5x5 stem) -> out [rows][400]                                    */
/*   post_act = 1: BaseResNet._process_grid (architectures.py:231-233; post-activation     */
/*                 blocks :159-171; 3x3 stem + BN + ReLU) followed by the two 1x1 collapses */
/*                 (:191-196, :210-214) -> out [rows][5][400]: channels 0-3 = bn scale *    */
/*                 own_collapse conv (its bias joins the FiLM-add term in the heads, :254), */
/*                 channel 4 = ReLU(BN(opp_collapse conv)).                                 */
/* ------------------------------------------------------------------------------------ */

/*
 * grids     [n_images][400] bf16 0/1 board cells
 * n_images_dev / out_row: optional device-side image count (<= n_images, reset to 0 when consumed) and the
 *           output row of image k (both or neither), as trl_alphasame_trunk_rows_indexed
 * w_packed  [2*n_blocks][3 dy][F/8][3F/8][8][8] bf16: per layer and vertical tap the 3F x F matrix
 *           B[(j, oc), ic] = w[oc][ic][dy][2 - j] in K-major UMMA core-matrix order
 * consts    [(2*n_blocks + 1)][3][F] f32 device: per stage (stem, then every conv) bias added to the
 *           accumulator, and for pre-activation second convs the next BatchNorm's scale and bias; then the
 *           head: W[n_out][F], scale[n_out], bias[n_out] (n_out = 1 or 5)
 * stem_lut  [taps][2^taps][F] f32 device: partial sums of one stem kernel row per input bit pattern
 * scratch   device, >= trl_trunk_wide_scratch_bytes(filters) bytes, ZERO-initialised once by the caller and
 *           then owned by launches of this operator on one stream at a time (activations stream through it)
 * status    [8] int32 device, zero-initialised: status[0] != 0 after a launch means a pipeline wait timed
 *           out (the kernel bounds every wait instead of hanging) and the outputs are invalid
 * pdl       launch as a programmatic dependent of the previous kernel in `stream`
 */
int trl_trunk_wide(const void* grids_bf16, int n_images, int32_t* n_images_dev, const int32_t* out_row,
                   int filters, int n_blocks, int post_act, int stem_taps, const void* w_packed,
                   const float* consts, const float* stem_lut, void* out_bf16, void* scratch,
                   long long scratch_bytes, int32_t* status, int pdl, void* stream);
long long trl_trunk_wide_scratch_bytes(int filters);

#ifdef __cplusplus
}
#endif
#endif /* TRL_H_ */
