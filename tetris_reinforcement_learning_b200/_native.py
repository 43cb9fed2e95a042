"""ctypes binding of libtrl_b200.so (include/trl.h).

There is NO CPU fallback: if the CUDA library is missing or fails to load, importing this
module's `lib()` raises.  Build it with `python -m tetris_reinforcement_learning_b200.build`.
"""
import ctypes
import os

from .state import GAME_DTYPE, PLAYER_DTYPE

_SO = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libtrl_b200.so")
_lib = None

ABI_VERSION = 10

c_void_p, c_int, c_u64, c_u32 = ctypes.c_void_p, ctypes.c_int, ctypes.c_uint64, ctypes.c_uint32

# name -> (restype, argtypes); pointers are passed as integers (device or host addresses)
SIGNATURES = {
    "trl_abi_version": (c_int, []),
    "trl_stamp_globaltimer": (c_int, [c_void_p, c_void_p]),
    "trl_set_pdl": (None, [c_int]),
    "trl_last_error": (ctypes.c_char_p, []),
    "trl_sizeof_player": (c_int, []),
    "trl_sizeof_game": (c_int, []),
    "trl_movegen": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int,
                            c_void_p, c_void_p, c_void_p]),
    "trl_movegen_games": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "trl_movegen_host": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int,
                                 c_void_p, c_void_p]),
    "trl_movegen_host_compact": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_u64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "trl_movegen_select_kernel": (None, [c_int]),
    "trl_movegen_warp_form": (None, [c_int]),
    "trl_search_movegen_rounds": (None, [c_int]),
    "trl_env_step": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_u64, c_void_p]),
    "trl_env_step_host": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_u64]),
    "trl_game_setup": (c_int, [c_void_p, c_int, c_u32, c_u32, c_u64, c_void_p]),
    "trl_game_setup_host": (c_int, [c_void_p, c_int, c_u32, c_u32, c_u64]),
    "trl_sizeof_search_ctl": (c_int, []),
    "trl_sizeof_sample": (c_int, []),
    "trl_sizeof_root_stats": (c_int, []),
    "trl_search_select": (c_int, [c_void_p, c_void_p, c_void_p]),
    "trl_search_movegen": (c_int, [c_void_p, c_void_p]),
    "trl_search_policy_legal": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "trl_search_expand": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "trl_search_expand_select": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "trl_search_expand_select_encode": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p,
                                                c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "trl_alphasame_trunk": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "trl_alphasame_trunk_rows": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "trl_alphasame_trunk_rows_max_blocks": (c_int, []),
    "trl_alphasame_heads": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "trl_alphasame_heads_weight_floats": (c_int, []),
    "trl_encode_features_cached": (c_int, [c_void_p] * 3 + [c_int] + [c_void_p] * 9),
    "trl_alphasame_trunk_rows_indexed": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "trl_alphasame_trunk_rows_gate": (c_int, [c_void_p]),
    "trl_alphasame_heads_indexed": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "trl_trunk_wide_scratch_bytes": (ctypes.c_longlong, [c_int]),
    "trl_trunk_wide": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                               c_void_p, c_void_p, ctypes.c_longlong, c_void_p, c_int, c_void_p]),
    "trl_encode_features": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p]),
}


class NativeLibraryError(RuntimeError):
    pass


def lib():
    """Load libtrl_b200.so once; raise loudly if it is absent or ABI-incompatible."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_SO):
        raise NativeLibraryError(
            f"{_SO} not found: the CUDA extension is not built. Run "
            "`python -m tetris_reinforcement_learning_b200.build` (needs nvcc). There is no CPU fallback.")
    L = ctypes.CDLL(_SO)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(L, name)  # AttributeError if the symbol is missing
        fn.restype, fn.argtypes = res, args
    if L.trl_abi_version() != ABI_VERSION:
        raise NativeLibraryError(f"ABI mismatch: library {L.trl_abi_version()} != binding {ABI_VERSION}")
    if L.trl_sizeof_player() != PLAYER_DTYPE.itemsize or L.trl_sizeof_game() != GAME_DTYPE.itemsize:
        raise NativeLibraryError("struct layout mismatch between include/trl.h and state.py")
    _lib = L
    return L


def check(rc, what):
    if rc != 0:
        msg = lib().trl_last_error().decode() if rc == -2 else {-1: "bad argument", -3: "out of memory"}.get(rc, "?")
        raise RuntimeError(f"{what} failed with code {rc}: {msg}")


# ---- ctypes mirrors of the search structs (include/trl.h) ----

class SearchParams(ctypes.Structure):
    _fields_ = [("seed", ctypes.c_uint64),
                ("cpuct", ctypes.c_double), ("dpuct", ctypes.c_double), ("fpu_value", ctypes.c_double),
                ("root_softmax_temp", ctypes.c_double), ("temperature", ctypes.c_double),
                ("playout_cap_chance", ctypes.c_double),
                ("dirichlet_alpha", ctypes.c_double), ("dirichlet_s", ctypes.c_double), ("dirichlet_eps", ctypes.c_double),
                ("c_forced", ctypes.c_double),
                ("max_iter", ctypes.c_int32), ("iters_long", ctypes.c_int32), ("iters_short", ctypes.c_int32),
                ("fpu_reduction", ctypes.c_int32), ("use_root_softmax", ctypes.c_int32), ("training", ctypes.c_int32),
                ("use_playout_cap", ctypes.c_int32), ("use_noise", ctypes.c_int32), ("use_dirichlet_s", ctypes.c_int32),
                ("use_forced", ctypes.c_int32), ("use_tanh", ctypes.c_int32), ("save_all", ctypes.c_int32),
                ("max_rounds", ctypes.c_int32), ("restart_finished", ctypes.c_int32),
                ("game_id_stride", ctypes.c_uint32), ("use_random_start", ctypes.c_int32),
                ("random_start_scale", ctypes.c_double), ("stop_after_search", ctypes.c_int32), ("pad_", ctypes.c_int32)]


class SearchBuffers(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in ("n_games", "node_cap", "state_cap", "moves_cap", "sample_cap",
                                              "end_cap", "pad0_", "pad1_")] + \
               [(n, ctypes.c_void_p) for n in ("prior", "value_sum", "visits", "parent", "slot", "move",
                                               "states", "first_child", "n_children", "fpu",
                                               "ctl", "games", "leaf_state", "legal", "n_legal",
                                               "samples", "sample_count", "ends", "end_count",
                                               "next_game_id", "noise_override", "leaf_parent",
                                               "legal_cache", "legal_cache_n", "movegen_index", "path",
                                               "movegen_list", "movegen_count", "movegen_status", "params2",
                                               "root_stats")]
