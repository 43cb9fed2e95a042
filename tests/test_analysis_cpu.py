"""CPU checks of the analysis interface: the ctypes mirrors and numpy dtypes of the search structs against
include/trl.h (offsets from a C compiler), the host check of analysis mode, and the public entry points'
argument order (reference ai.py:299, 1222)."""
import ctypes
import inspect
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from tetris_reinforcement_learning_b200 import _native, build
    build.build()
    return _native.lib()


def test_struct_sizes_match_the_library(lib):
    from tetris_reinforcement_learning_b200 import _native, selfplay
    assert lib.trl_sizeof_search_ctl() == selfplay.CTL_DTYPE.itemsize
    assert lib.trl_sizeof_sample() == selfplay.SAMPLE_DTYPE.itemsize
    assert lib.trl_sizeof_root_stats() == selfplay.ROOT_STATS_DTYPE.itemsize
    # the kernel's static_asserts state the sizes of the structs passed by value
    src = open(os.path.join(ROOT, "tetris_reinforcement_learning_b200", "csrc", "mcts.cu")).read()
    for name, cls in (("TrlSearchParams", _native.SearchParams), ("TrlSearchBuffers", _native.SearchBuffers)):
        size = int(re.search(r"sizeof\(%s\) == (\d+)" % name, src).group(1))
        assert ctypes.sizeof(cls) == size, name


@pytest.mark.skipif(shutil.which("gcc") is None, reason="needs a C compiler")
def test_field_offsets_match_the_header(tmp_path):
    """offsetof() of every TrlRootStats field and of the new TrlSearchParams / TrlSearchBuffers fields, as a C
    compiler lays out include/trl.h, against ROOT_STATS_DTYPE and the ctypes mirrors."""
    from tetris_reinforcement_learning_b200 import _native, selfplay
    fields = selfplay.ROOT_STATS_DTYPE.names
    lines = [f'printf("TrlRootStats.{f} %zu\\n", offsetof(TrlRootStats, {f}));' for f in fields]
    lines += ['printf("TrlRootStats %zu\\n", sizeof(TrlRootStats));',
              'printf("TrlSearchParams.stop_after_search %zu\\n", offsetof(TrlSearchParams, stop_after_search));',
              'printf("TrlSearchBuffers.root_stats %zu\\n", offsetof(TrlSearchBuffers, root_stats));']
    c = tmp_path / "offsets.c"
    c.write_text("#include <stddef.h>\n#include <stdio.h>\n#include \"trl.h\"\nint main(void) {\n" + "\n".join(lines) +
                 "\nreturn 0;\n}\n")
    exe = tmp_path / "offsets"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(c), "-o", str(exe)], check=True)
    got = dict(line.rsplit(" ", 1) for line in subprocess.run([str(exe)], check=True, capture_output=True,
                                                             text=True).stdout.splitlines())
    for f in fields:
        assert int(got[f"TrlRootStats.{f}"]) == selfplay.ROOT_STATS_DTYPE.fields[f][1], f
    assert int(got["TrlRootStats"]) == selfplay.ROOT_STATS_DTYPE.itemsize
    assert int(got["TrlSearchParams.stop_after_search"]) == _native.SearchParams.stop_after_search.offset
    assert int(got["TrlSearchBuffers.root_stats"]) == _native.SearchBuffers.root_stats.offset


def test_analysis_mode_rejects_random_openings(lib):
    """The library refuses stop_after_search together with use_random_start (checked on the host, before any
    launch: an empty batch reaches no device code), and so does the Python side."""
    from tetris_reinforcement_learning_b200 import _native
    from tetris_reinforcement_learning_b200.config import Config
    from tetris_reinforcement_learning_b200.selfplay import search_params_from_config
    b = _native.SearchBuffers()
    b.n_games, b.node_cap, b.state_cap, b.moves_cap = 0, 2, 2, 1
    for name, ctype in _native.SearchBuffers._fields_:
        if ctype is ctypes.c_void_p and name not in ("noise_override", "params2", "root_stats"):
            setattr(b, name, 64)     # never dereferenced: n_games = 0
    p = _native.SearchParams()
    p.stop_after_search, p.use_random_start = 1, 1
    assert lib.trl_search_select(ctypes.byref(b), ctypes.byref(p), None) == -1
    assert lib.trl_search_expand(ctypes.byref(b), ctypes.byref(p), 64, 64, 11583, 0, None) == -1
    p.use_random_start = 0
    assert lib.trl_search_select(ctypes.byref(b), ctypes.byref(p), None) == 0
    cfg = Config(visual=False, ruleset="s2", model="pytorch", use_random_starting_moves=True)
    assert search_params_from_config(cfg, analysis=True).stop_after_search == 1
    with pytest.raises(ValueError):
        search_params_from_config(cfg, analysis=True, random_openings=True)


def test_public_entry_points_follow_the_reference():
    from tetris_reinforcement_learning_b200 import ai
    assert list(inspect.signature(ai.MCTS).parameters)[:3] == ["config", "game", "interference_network"]
    assert list(inspect.signature(ai.evaluate).parameters) == ["config", "game", "network"]
    assert list(inspect.signature(ai.evaluate_positions).parameters) == ["config", "games", "network"]
    assert list(inspect.signature(ai.analyse).parameters) == ["config", "games", "network", "seed", "game_ids", "search_no"]


def test_search_result_carries_root_statistics():
    from tetris_reinforcement_learning_b200 import ai
    from tetris_reinforcement_learning_b200.selfplay import ROOT_STATS_DTYPE, SAMPLE_DTYPE
    s = np.zeros((), SAMPLE_DTYPE)
    s["n_children"], s["chosen_move"], s["saved"] = 3, 429, 1
    s["moves"][:3] = [5, 429, 700]
    s["visits"][:3] = s["visits_pre"][:3] = [1, 4, 2]
    r = np.zeros((), ROOT_STATS_DTYPE)
    r["n_children"], r["pv_len"], r["root_value"] = 3, 2, 0.25
    r["prior"][:3] = [0.5, 0.25, 0.25]
    r["q"][:3] = [0.1, 0.2, 0.3]
    r["pv"][:2] = [429, 17]
    r["pv_visits"][:2] = [4, 3]
    res = ai.SearchResult(s, r)
    assert res.chosen_move == 429 and res.move == ai.index_to_move(429) and res.saved
    assert res.priors.dtype == np.float32 and list(res.priors) == [0.5, 0.25, 0.25]
    assert list(res.q) == [np.float32(0.1), np.float32(0.2), np.float32(0.3)] and res.root_value == 0.25
    assert list(res.pv) == [429, 17] and list(res.pv_visits) == [4, 3]
    plain = ai.SearchResult(s)
    assert plain.priors is None and plain.pv is None and list(plain.visits) == [1, 4, 2]


def test_caches_serve_only_the_network_they_were_built_for():
    """A cache entry answers only for the object it was built from.  Deleting a network and loading the next
    checkpoint into a new one can reproduce the old key exactly (same address, same parameter versions after
    load_state_dict); the new network must still miss."""
    import gc
    import torch
    from tetris_reinforcement_learning_b200 import ai, architectures as arch
    mc = arch.AlphaSameConfig(blocks=1, filters=16)
    torch.manual_seed(0)
    checkpoints = [arch.AlphaSame(mc).state_dict() for _ in range(12)]
    cache, collisions, net = {}, 0, None
    for i, sd in enumerate(checkpoints):
        del net
        gc.collect()
        net = arch.AlphaSame(mc)
        net.load_state_dict(sd)
        key = ai._net_identity(net)
        collisions += int(key in cache)
        assert ai._cache_get(cache, key, net) is None, i
        ai._cache_put(cache, key, net, f"built for checkpoint {i}")
        assert ai._cache_get(cache, key, net) == f"built for checkpoint {i}"
        assert len(cache) <= ai._CACHE_ENTRIES
    print(f"{collisions} of {len(checkpoints)} reloaded networks reproduced a cached key")
    # objects that cannot be weakly referenced are held by their entry, so their id stays theirs
    class Slotted:
        __slots__ = ()

        def __call__(self, grids, extras):
            return grids, extras
    ev = Slotted()
    ai._cache_put(cache, ai._net_identity(ev), ev, "slotted")
    assert ai._cache_get(cache, ai._net_identity(ev), ev) == "slotted"
    assert ai._cache_get(cache, ai._net_identity(ev), Slotted()) is None


def test_engine_batch_buckets():
    from tetris_reinforcement_learning_b200 import ai
    assert [ai._engine_batch(n) for n in (1, 2, 3, 5, 64, 65, 595, 4096, 5000)] == [1, 2, 4, 8, 64, 128, 1024, 4096, 4096]


def test_unpack_game_round_trips():
    import os
    from tetris_reinforcement_learning_b200.state import GAME_DTYPE, games_equal, pack_game, unpack_game
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    games = np.load(os.path.join(root, "tests", "golden", "mcts_golden.npz"))["games"].copy().view(GAME_DTYPE).reshape(-1)
    for rec in games:
        back = pack_game(unpack_game(rec), game_id=int(rec["game_id"]), rng_ctr=int(rec["rng_ctr"]),
                         bag_ctr=int(rec["bag_ctr"]))
        back["rounds"] = rec["rounds"]          # a Game carries its history, not the count
        assert games_equal(np.array([back]), np.array([rec])).all()
