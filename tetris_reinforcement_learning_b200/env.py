"""Batched env step — host-side mirror of Game.make_move / Game.setup (reference game.py:28-118).

`games` are packed TrlGame records (state.GAME_DTYPE on the host, uint8[n,400] CUDA tensors on
the device).  No CPU implementation: without libtrl_b200.so these raise.
"""
import numpy as np

from . import _native
from .state import GAME_DTYPE, STEPOUT_DTYPE, ruleset_id

_RULESET_BYTE = GAME_DTYPE.fields["ruleset"][1]   # offset of TrlGame.ruleset (385)


def game_setup_host(n, first_game_id=0, seed=0, id_stride=1, ruleset="s2"):
    """n fresh games after Game(ruleset).setup() (game.py:8-32) -> GAME_DTYPE[n]."""
    games = np.zeros(n, dtype=GAME_DTYPE)
    rc = _native.lib().trl_game_setup_host(games.ctypes.data, n, int(first_game_id), int(id_stride), int(seed))
    _native.check(rc, "trl_game_setup_host")
    games["ruleset"] = ruleset_id(ruleset)
    return games


def env_step_host(games, moves, add_bag=True, seed=0):
    """Game.make_move(move, add_bag, add_history=add_bag) on every game, in place.

    games GAME_DTYPE[n] (C-contiguous), moves uint16[n] flat policy indices (0xFFFF = skip)
    -> STEPOUT_DTYPE[n] (rows_cleared, attack, flags, garbage_col, status)."""
    if games.dtype != GAME_DTYPE or not games.flags["C_CONTIGUOUS"]:
        raise ValueError("games must be a C-contiguous GAME_DTYPE array")
    moves = np.ascontiguousarray(moves, dtype=np.uint16)
    n = games.shape[0]
    if moves.shape != (n,):
        raise ValueError("moves must be uint16[n]")
    out = np.zeros(n, dtype=STEPOUT_DTYPE)
    rc = _native.lib().trl_env_step_host(games.ctypes.data, moves.ctypes.data, n, out.ctypes.data,
                                         int(bool(add_bag)), int(seed))
    _native.check(rc, "trl_env_step_host")
    return out


def game_setup_device(games, first_game_id=0, seed=0, id_stride=1, ruleset="s2"):
    """games: uint8[n,400] CUDA tensor, filled in place on the current stream of its device."""
    import torch
    with torch.cuda.device(games.device):
        rc = _native.lib().trl_game_setup(games.data_ptr(), games.shape[0], int(first_game_id), int(id_stride), int(seed),
                                          torch.cuda.current_stream().cuda_stream)
    _native.check(rc, "trl_game_setup")
    games.view(games.shape[0], GAME_DTYPE.itemsize)[:, _RULESET_BYTE] = ruleset_id(ruleset)


def env_step_device(games, moves, out=None, add_bag=True, seed=0):
    """games uint8[n,400], moves int16/uint16[n], out uint8[n,8] | None — CUDA tensors of one device, stepped on the
    current stream of that device."""
    import torch
    with torch.cuda.device(games.device):
        rc = _native.lib().trl_env_step(games.data_ptr(), moves.data_ptr(), games.shape[0],
                                        out.data_ptr() if out is not None else None, int(bool(add_bag)),
                                        int(seed), torch.cuda.current_stream().cuda_stream)
    _native.check(rc, "trl_env_step")
