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
