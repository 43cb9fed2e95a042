"""Packed game state (include/trl.h TrlPlayer / TrlGame) as numpy structured dtypes, and
converters from/to reference-style objects.

The converters are duck-typed: they accept the reference's own `Player` / `Game`
instances (player.py:10-27, game.py:6-26) or anything exposing the same attributes, so a
reference user can hand their live objects to this package unchanged.
"""
import numpy as np

from .const import COLS, MINOS, NONE, ROWS

QUEUE_CAP = 16
RECV_CAP = 80

PLAYER_DTYPE = np.dtype({
    "names": ["rows", "pieces", "b2b", "combo", "qlen", "piece", "held", "game_over",
              "b2b_level", "n_recv", "pad_", "queue", "recv"],
    "formats": [("<u2", (ROWS,)), "<i4", "<i2", "<i2", "u1", "u1", "u1", "u1",
                "u1", "u1", ("u1", (2,)), ("u1", (QUEUE_CAP,)), ("u1", (RECV_CAP,))],
    "offsets": [0, 80, 84, 86, 88, 89, 90, 91, 92, 93, 94, 96, 112],
    "itemsize": 192,
})

GAME_DTYPE = np.dtype({
    "names": ["players", "turn", "ruleset", "bag_ctr", "rounds", "rng_ctr", "game_id"],
    "formats": [(PLAYER_DTYPE, (2,)), "u1", "u1", "<u2", "<u4", "<u4", "<u4"],
    "offsets": [0, 384, 385, 386, 388, 392, 396],
    "itemsize": 400,
})

STEPOUT_DTYPE = np.dtype({
    "names": ["rows_cleared", "attack", "flags", "garbage_col", "status"],
    "formats": ["u1", "u1", "u1", "u1", "<u4"],
    "offsets": [0, 1, 2, 3, 4],
    "itemsize": 8,
})

_PIECE_ID = {m: i for i, m in enumerate(MINOS)}


RULESETS = {"s2": 0, "s1": 1}   # TRL_RULESET_S2 / TRL_RULESET_S1 (include/trl.h)


def ruleset_id(ruleset):
    """'s2' / 's1' (Config.ruleset, ai.py:72) -> the byte stored in TrlGame.ruleset."""
    if ruleset not in RULESETS:
        raise ValueError(f"unknown ruleset {ruleset!r} (expected 's1' or 's2')")
    return RULESETS[ruleset]


def piece_id(piece_type):
    """'Z'.. 'T' or None -> 0..6 or NONE."""
    return NONE if piece_type is None else _PIECE_ID[piece_type]


def piece_name(pid):
    return None if int(pid) == NONE else MINOS[int(pid)]


def grid_to_rows(grid):
    """Board.grid (40x10, anything truthy = occupied; board.py:7) -> uint16[40] bitrows."""
    occ = np.asarray(grid) != 0
    if occ.shape != (ROWS, COLS):
        raise ValueError(f"expected a ({ROWS},{COLS}) grid, got {occ.shape}")
    weights = (1 << np.arange(COLS)).astype(np.uint16)
    return (occ.astype(np.uint16) * weights).sum(axis=1).astype(np.uint16)


def rows_to_grid(rows):
    """uint16[40] bitrows -> int8 (40,10) 0/1 grid (what simplify_grid sees, ai.py:1364-1366)."""
    rows = np.asarray(rows, dtype=np.uint16)
    return ((rows[:, None] >> np.arange(COLS)[None, :]) & 1).astype(np.int8)


def movegen_args_from_player(player):
    """(rows, cur, alt) for trl_movegen from a reference-style Player.

    alt follows MoveGenerator._get_piece_types_to_check (move_generation.py:91-105):
    the held piece if there is one, else the head of the queue, else none.
    """
    rows = grid_to_rows(player.board.grid)
    cur = piece_id(player.piece.type) if player.piece is not None else NONE
    if player.held_piece is not None:
        alt = piece_id(player.held_piece)
    elif player.queue.pieces:
        alt = piece_id(player.queue.pieces[0])
    else:
        alt = NONE
    return rows, cur, alt


def pack_player(player, out=None):
    """Reference-style Player -> PLAYER_DTYPE scalar (fields of Player.copy, player.py:217-233)."""
    rec = np.zeros((), dtype=PLAYER_DTYPE) if out is None else out
    rec["rows"] = grid_to_rows(player.board.grid)
    rec["pieces"] = player.stats.pieces
    rec["b2b"] = player.stats.b2b
    rec["combo"] = player.stats.combo
    rec["b2b_level"] = player.stats.b2b_level
    q = [piece_id(p) for p in player.queue.pieces]
    if len(q) > QUEUE_CAP:
        raise ValueError(f"queue longer than {QUEUE_CAP}")
    rec["qlen"] = len(q)
    rec["queue"] = 0
    rec["queue"][:len(q)] = q
    rec["piece"] = piece_id(player.piece.type) if player.piece is not None else NONE
    rec["held"] = piece_id(player.held_piece)
    rec["game_over"] = 1 if player.game_over else 0
    g = list(player.garbage_to_receive)
    if len(g) > RECV_CAP:
        raise ValueError(f"garbage_to_receive longer than {RECV_CAP}")
    rec["n_recv"] = len(g)
    rec["recv"] = 0
    rec["recv"][:len(g)] = g
    return rec


def pack_game(game, game_id=0, rng_ctr=0, bag_ctr=0, out=None):
    """Reference-style Game -> GAME_DTYPE scalar."""
    rec = np.zeros((), dtype=GAME_DTYPE) if out is None else out
    for i in range(2):
        pack_player(game.players[i], out=rec["players"][i])
    rec["turn"] = game.turn
    rec["ruleset"] = ruleset_id(getattr(game, "ruleset", "s2"))
    hist = getattr(game, "history", None)
    rec["rounds"] = len(hist.states) if hist is not None and hasattr(hist, "states") else 0
    rec["rng_ctr"] = rng_ctr
    rec["bag_ctr"] = bag_ctr
    rec["game_id"] = game_id
    return rec


def unpack_game(rec):
    """GAME_DTYPE scalar -> a duck-typed reference Game (game.py:6-26, player.py:10-27) carrying exactly the fields
    pack_game reads, e.g. to hand stored positions to MCTS().  pack_game(unpack_game(r)) == r except for the history
    length and the RNG counters, which a Game does not carry."""
    from types import SimpleNamespace as NS
    players = []
    for pr in rec["players"]:
        players.append(NS(board=NS(grid=rows_to_grid(pr["rows"])),
                          queue=NS(pieces=[MINOS[int(v)] for v in pr["queue"][:int(pr["qlen"])]]),
                          piece=None if int(pr["piece"]) == NONE else NS(type=MINOS[int(pr["piece"])]),
                          held_piece=piece_name(pr["held"]), game_over=bool(pr["game_over"]),
                          garbage_to_receive=[int(v) for v in pr["recv"][:int(pr["n_recv"])]],
                          stats=NS(pieces=int(pr["pieces"]), b2b=int(pr["b2b"]), combo=int(pr["combo"]),
                                   b2b_level=int(pr["b2b_level"]))))
    ruleset = {v: k for k, v in RULESETS.items()}[int(rec["ruleset"])]
    return NS(players=players, turn=int(rec["turn"]), ruleset=ruleset)


def player_state_dict(rec):
    """PLAYER_DTYPE scalar -> plain dict in the reference's vocabulary (for diffs / debugging)."""
    return {
        "rows": [int(v) for v in rec["rows"]],
        "queue": [MINOS[int(v)] for v in rec["queue"][:int(rec["qlen"])]],
        "piece": piece_name(rec["piece"]),
        "held_piece": piece_name(rec["held"]),
        "game_over": bool(rec["game_over"]),
        "garbage_to_receive": [int(v) for v in rec["recv"][:int(rec["n_recv"])]],
        "pieces": int(rec["pieces"]),
        "b2b": int(rec["b2b"]),
        "b2b_level": int(rec["b2b_level"]),
        "combo": int(rec["combo"]),
    }


def game_state_dict(rec):
    return {"turn": int(rec["turn"]),
            "players": [player_state_dict(rec["players"][i]) for i in range(2)]}


def reference_player_state_dict(player):
    """The same dict straight from a reference-style Player (no packing in between)."""
    return {
        "rows": [int(v) for v in grid_to_rows(player.board.grid)],
        "queue": list(player.queue.pieces),
        "piece": player.piece.type if player.piece is not None else None,
        "held_piece": player.held_piece,
        "game_over": bool(player.game_over),
        "garbage_to_receive": [int(v) for v in player.garbage_to_receive],
        "pieces": int(player.stats.pieces),
        "b2b": int(player.stats.b2b),
        "b2b_level": int(player.stats.b2b_level),
        "combo": int(player.stats.combo),
    }


def reference_game_state_dict(game):
    return {"turn": int(game.turn),
            "players": [reference_player_state_dict(p) for p in game.players]}


def unpack_mask(mask_bits):
    """uint32[..., 362] bit-packed masks -> bool[..., 27, 39, 11]."""
    from .const import POLICY_SHAPE, POLICY_SIZE
    words = np.ascontiguousarray(mask_bits, dtype="<u4")
    bits = np.unpackbits(words.view(np.uint8), axis=-1, bitorder="little")
    bits = bits[..., :POLICY_SIZE]
    return bits.reshape(words.shape[:-1] + POLICY_SHAPE).astype(bool)


def pack_mask(mask):
    """bool[..., 27, 39, 11] -> uint32[..., 362] (inverse of unpack_mask)."""
    from .const import MASK_WORDS, POLICY_SIZE
    m = np.asarray(mask).astype(np.uint8)
    flat = m.reshape(m.shape[:-3] + (POLICY_SIZE,))
    pad = MASK_WORDS * 32 - POLICY_SIZE
    flat = np.concatenate([flat, np.zeros(flat.shape[:-1] + (pad,), np.uint8)], axis=-1)
    return np.packbits(flat, axis=-1, bitorder="little").view("<u4")


def canonical_games(games):
    """Copy of a GAME_DTYPE array with don't-care bytes (queue slots >= qlen, recv slots >=
    n_recv, padding) zeroed, so that two states can be compared byte-wise."""
    g = np.array(games, dtype=GAME_DTYPE, copy=True)
    p = g["players"]
    qi = np.arange(QUEUE_CAP)
    ri = np.arange(RECV_CAP)
    p["queue"][qi[None, None, :] >= p["qlen"][..., None]] = 0
    p["recv"][ri[None, None, :] >= p["n_recv"][..., None]] = 0
    p["pad_"] = 0
    return g


def games_equal(a, b):
    """Per-game semantic equality of two GAME_DTYPE arrays -> bool[n]."""
    ca = canonical_games(a).view(np.uint8).reshape(len(a), -1)
    cb = canonical_games(b).view(np.uint8).reshape(len(b), -1)
    return (ca == cb).all(axis=1)
