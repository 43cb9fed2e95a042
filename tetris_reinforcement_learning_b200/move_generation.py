"""Legal-placement enumeration — host-side mirror of reference move_generation.py.

`get_move_matrix(player, algo)` keeps the reference's name, argument meaning and return type
(move_generation.py:752-789) and runs on the GPU through the C ABI (`trl_movegen_host`).
`movegen_host` / `movegen_device` are the batched forms (numpy host buffers / torch CUDA
tensors).  There is no CPU implementation here: without libtrl_b200.so these raise.
"""
import numpy as np

from . import _native
from .const import MASK_WORDS, POLICY_SHAPE, ROWS
from .state import movegen_args_from_player, unpack_mask

_ALGOS_REFERENCE = ("brute-force", "faster-but-loss", "harddrop", "convolutional")
DEFAULT_MOVES_CAP = 512  # SURVEY §7.2b: <= 314 placements seen on adversarial boards


def _ptr(a):
    return a.ctypes.data if a is not None else None


def movegen_host(boards, cur, alt, want_mask=True, want_moves=False, moves_cap=DEFAULT_MOVES_CAP):
    """Batched movegen on HOST numpy buffers (copies in, runs the kernel, copies out).

    boards uint16[n,40]; cur, alt uint8[n] (255 = none)
    -> dict(mask_bits uint32[n,362] | None, moves uint16[n,cap] | None, n_moves uint16[n], status uint32[n])
    """
    boards = np.ascontiguousarray(boards, dtype=np.uint16)
    cur = np.ascontiguousarray(cur, dtype=np.uint8)
    alt = np.ascontiguousarray(alt, dtype=np.uint8)
    n = boards.shape[0]
    if boards.shape != (n, ROWS) or cur.shape != (n,) or alt.shape != (n,):
        raise ValueError("expected boards[n,40], cur[n], alt[n]")
    mask = np.empty((n, MASK_WORDS), dtype=np.uint32) if want_mask else None
    moves = np.empty((n, moves_cap), dtype=np.uint16) if want_moves else None
    n_moves = np.empty(n, dtype=np.uint16)
    status = np.empty(n, dtype=np.uint32)
    rc = _native.lib().trl_movegen_host(_ptr(boards), _ptr(cur), _ptr(alt), n, _ptr(mask), _ptr(moves),
                                        moves_cap, _ptr(n_moves), _ptr(status))
    _native.check(rc, "trl_movegen_host")
    return {"mask_bits": mask, "moves": moves, "n_moves": n_moves, "status": status}


def movegen_host_compact(boards, cur, alt, capacity=None, out=None):
    """Batched movegen on HOST buffers with compact output (trl_movegen_host_compact): the ascending
    move lists of all calls packed back to back.

    -> dict(moves uint16[total], offsets uint64[n], n_moves uint16[n], status uint32[n], total int);
    call i owns moves[offsets[i] : offsets[i] + n_moves[i]].  `out` may carry preallocated (pinned)
    numpy arrays under the same keys (moves sized `capacity`)."""
    import ctypes
    boards = np.ascontiguousarray(boards, dtype=np.uint16)
    cur = np.ascontiguousarray(cur, dtype=np.uint8)
    alt = np.ascontiguousarray(alt, dtype=np.uint8)
    n = boards.shape[0]
    if boards.shape != (n, ROWS) or cur.shape != (n,) or alt.shape != (n,):
        raise ValueError("expected boards[n,40], cur[n], alt[n]")
    out = out or {}
    capacity = int(capacity if capacity is not None else (out["moves"].size if "moves" in out else max(1024, 160 * n)))
    moves = out.get("moves", None)
    if moves is None:
        moves = np.empty(capacity, dtype=np.uint16)
    offsets = out.get("offsets", None)
    if offsets is None:
        offsets = np.empty(n, dtype=np.uint64)
    n_moves = out.get("n_moves", None)
    if n_moves is None:
        n_moves = np.empty(n, dtype=np.uint16)
    status = out.get("status", None)
    if status is None:
        status = np.empty(n, dtype=np.uint32)
    total = ctypes.c_uint64(0)
    rc = _native.lib().trl_movegen_host_compact(_ptr(boards), _ptr(cur), _ptr(alt), n, _ptr(moves), capacity,
                                                _ptr(offsets), _ptr(n_moves), _ptr(status), ctypes.addressof(total))
    _native.check(rc, "trl_movegen_host_compact")
    return {"moves": moves, "offsets": offsets, "n_moves": n_moves, "status": status, "total": int(total.value)}


def decode_move_codes(codes, escapes, n_moves):
    """Byte-coded move lists of trl_movegen_host_boards (format in include/trl.h) -> (moves uint16[total],
    offsets uint64[n]): call i's ascending list is moves[offsets[i] : offsets[i] + n_moves[i]].  No per-call loop."""
    codes = np.asarray(codes, dtype=np.uint8)
    n_moves = np.asarray(n_moves)
    counts = n_moves.astype(np.int64)
    start = np.cumsum(counts) - counts
    if codes.size != counts.sum():
        raise ValueError(f"{codes.size} codes for {int(counts.sum())} moves")
    d = codes.astype(np.int64)
    zero = codes == 0
    if int(zero.sum()) != np.asarray(escapes).size:
        raise ValueError(f"{int(zero.sum())} escape codes for {np.asarray(escapes).size} escapes")
    d[zero] = escapes
    cs = np.cumsum(d)
    if cs.size == 0:
        return np.empty(0, dtype=np.uint16), start.astype(np.uint64)
    moves = cs - np.repeat(np.where(start > 0, cs[start - 1], 0), counts) - 1
    return moves.astype(np.uint16), start.astype(np.uint64)


def movegen_host_boards(boards, board_index, cur, alt, decode=True, out=None):
    """Batched movegen on HOST buffers over shared boards (trl_movegen_host_boards): call i enumerates
    boards[board_index[i]] with cur[i] / alt[i], and each board crosses PCIe once.

    boards uint16[n_boards,40]; board_index uint32[n] (< n_boards); cur, alt uint8[n] (255 = none).
    decode=True -> the keys of movegen_host_compact: moves uint16[total], offsets uint64[n], n_moves
    uint16[n], status uint32[n] (dense) and total.
    decode=False -> the raw streams: codes uint8, escapes uint16, n_moves uint16[n], and the flagged calls
    flag_index / flag_status uint32 (calls with a non-zero TRL_ST_* word, ascending).
    `out` may carry preallocated (pinned) numpy arrays under the keys codes, escapes, n_moves, flag_index
    and flag_status; their sizes are the capacities."""
    import ctypes
    boards = np.ascontiguousarray(boards, dtype=np.uint16)
    board_index = np.asarray(board_index)
    if board_index.dtype.kind not in "iu":
        raise ValueError("board_index must be an integer array")
    if board_index.dtype.itemsize > 4 and board_index.size and \
            (board_index.min() < 0 or board_index.max() > np.iinfo(np.uint32).max):
        raise ValueError("board_index out of range")   # would wrap into a valid index as uint32
    # (a negative int32 index becomes >= 2^31 > n_boards, which the device rejects)
    board_index = np.ascontiguousarray(board_index, dtype=np.uint32)
    cur = np.ascontiguousarray(cur, dtype=np.uint8)
    alt = np.ascontiguousarray(alt, dtype=np.uint8)
    n_boards, n = boards.shape[0], board_index.shape[0]
    if boards.shape != (n_boards, ROWS) or board_index.shape != (n,) or cur.shape != (n,) or alt.shape != (n,):
        raise ValueError("expected boards[n_boards,40], board_index[n], cur[n], alt[n]")
    out = out or {}

    def buf(key, size, dtype):
        a = out.get(key, None)
        if a is None:
            return np.empty(size, dtype=dtype)
        if a.dtype != dtype or a.ndim != 1 or not a.flags.c_contiguous:
            raise ValueError(f"out[{key!r}] must be a contiguous 1-D {np.dtype(dtype).name} array")
        return a

    # default capacities: the device staging's 512 codes per call, and the exact bounds of 45 escapes per call
    # (each spans >= 256 of the 11583 indices) and one flag per call
    codes = buf("codes", max(1024, 512 * n), np.uint8)
    escapes = buf("escapes", max(64, 45 * n), np.uint16)
    n_moves = buf("n_moves", n, np.uint16)
    flag_index = buf("flag_index", n, np.uint32)
    flag_status = buf("flag_status", flag_index.size, np.uint32)
    if n_moves.size != n:
        raise ValueError("out['n_moves'] must have n entries")
    totals = (ctypes.c_uint64 * 3)()
    addr = ctypes.addressof(totals)
    rc = _native.lib().trl_movegen_host_boards(
        _ptr(boards), n_boards, _ptr(board_index), _ptr(cur), _ptr(alt), n, _ptr(codes), codes.size, _ptr(escapes),
        escapes.size, _ptr(n_moves), _ptr(flag_index), _ptr(flag_status), min(flag_index.size, flag_status.size),
        addr, addr + 8, addr + 16)
    _native.check(rc, "trl_movegen_host_boards")
    n_codes, n_esc, n_flag = (int(v) for v in totals)
    raw = {"codes": codes[:n_codes], "escapes": escapes[:n_esc], "n_moves": n_moves,
           "flag_index": flag_index[:n_flag], "flag_status": flag_status[:n_flag]}
    if not decode:
        return raw
    moves, offsets = decode_move_codes(raw["codes"], raw["escapes"], n_moves)
    status = np.zeros(n, dtype=np.uint32)
    status[raw["flag_index"]] = raw["flag_status"]
    return {"moves": moves, "offsets": offsets, "n_moves": n_moves, "status": status, "total": int(moves.size)}


def movegen_device(boards, cur, alt, mask_bits=None, moves=None, n_moves=None, status=None):
    """Batched movegen on torch CUDA tensors of one device, stream-ordered on the current stream of that device.

    boards: uint16/int16 [n,40]; cur, alt: uint8 [n]; outputs are caller-allocated tensors
    (mask_bits int32/uint32 [n,362], moves int16/uint16 [n,cap], n_moves int16/uint16 [n],
    status int32/uint32 [n]); any output may be None.
    """
    import torch
    n = boards.shape[0]
    for t in (boards, cur, alt, mask_bits, moves, n_moves, status):
        if t is not None and (not t.is_cuda or not t.is_contiguous()):
            raise ValueError("movegen_device needs contiguous CUDA tensors")
    cap = moves.shape[1] if moves is not None else 0
    dp = lambda t: t.data_ptr() if t is not None else None  # noqa: E731
    with torch.cuda.device(boards.device):
        rc = _native.lib().trl_movegen(dp(boards), dp(cur), dp(alt), n, dp(mask_bits), dp(moves), cap,
                                       dp(n_moves), dp(status), torch.cuda.current_stream().cuda_stream)
    _native.check(rc, "trl_movegen")


def movegen_games_device(games, mask_bits=None, moves=None, n_moves=None, status=None):
    """Same, for the side to move of packed games (uint8 [n,400] CUDA tensor)."""
    import torch
    n = games.shape[0]
    cap = moves.shape[1] if moves is not None else 0
    dp = lambda t: t.data_ptr() if t is not None else None  # noqa: E731
    with torch.cuda.device(games.device):
        rc = _native.lib().trl_movegen_games(dp(games), n, dp(mask_bits), dp(moves), cap, dp(n_moves),
                                             dp(status), torch.cuda.current_stream().cuda_stream)
    _native.check(rc, "trl_movegen_games")


def get_move_matrix(player, algo="convolutional"):
    """Drop-in for move_generation.get_move_matrix: bool ndarray (27, 39, 11).

    Only the reference's default algorithm, 'convolutional' (ai.py:84), is provided — it is
    the bit-exact parity target, including its FIFO-order dependent T-spin planes.  The other
    reference algorithms find the same cells ('brute-force') or fewer ('faster-but-loss',
    'harddrop') and are not part of the data-generation path; asking for them raises
    NotImplementedError, an unknown name raises ValueError like the reference
    (move_generation.py:147-148).  `player` is not mutated.
    """
    if algo not in _ALGOS_REFERENCE:
        raise ValueError(f"Unknown algorithm: {algo}")
    if algo != "convolutional":
        raise NotImplementedError(f"algo={algo!r}: only 'convolutional' runs on the B200 path")
    rows, cur, alt = movegen_args_from_player(player)
    if cur == 255 and player.held_piece is None:
        # the reference raises AttributeError here (hold with nothing to hold, player.py:191-192);
        # Game.no_move guards every call site (ai.py:413)
        raise AttributeError("'NoneType' object has no attribute 'type'")
    res = movegen_host(rows[None, :], np.array([cur], np.uint8), np.array([alt], np.uint8))
    return unpack_mask(res["mask_bits"][0]).reshape(POLICY_SHAPE)
