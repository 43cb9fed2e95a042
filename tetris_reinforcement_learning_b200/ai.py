"""Drop-in boundary of the data-generation path — host-side mirror of reference ai.py.

Kept verbatim from the reference (names, argument meaning, defaults, on-disk artefacts):
    Config                       ai.py:62-216     (config.py)
    instantiate_network          ai.py:1033-1085
    make_training_set            ai.py:1809-1845
    self_play_loop               ai.py:2117-2198
    MCTS                         ai.py:299-659    (one search of one reference-style Game)
    evaluate                     ai.py:1222-1319  (network value + softmax policy of one position)
    search_statistics            ai.py:1330-1361
    reflect_grid/pieces/policy   ai.py:1423-1516
    load_model, load_best_model, highest_model_number, highest_data_number   ai.py:2231-2355
Beyond the reference: analyse() searches many positions at once with root statistics, evaluate_positions()
evaluates many positions at once.
Everything that touches game rules, placements, the search or features runs on the GPU through
libtrl_b200.so; there is no CPU implementation of those in this package.
"""
import json
import math
import os
import time
import weakref
from datetime import datetime, timezone
from pathlib import Path

import numpy as np
import torch

from . import architectures
from .architectures import (AlphaSame, AlphaSameConfig, AuxBaseResNet, AuxBaseResNetConfig, BaseResNet,  # noqa: F401
                            BaseResNetConfig, build_network)   # the reference's ai.py does `from architectures import *`
from .config import Config, config_to_dict, storage_dir  # noqa: F401
from .const import MINOS, POLICY_SHAPE, PREVIEWS, index_to_move, policy_index_to_piece, policy_piece_to_index
from .state import GAME_DTYPE, pack_game, rows_to_grid

device = "cuda" if torch.cuda.is_available() else "cpu"


def logs_dir():
    p = storage_dir() / "logs"
    p.mkdir(parents=True, exist_ok=True)
    return p


# ---------------------------------------------------------------------------------------------
# networks and checkpoints
# ---------------------------------------------------------------------------------------------

def append_version_record(config, model_number):
    path = Path(config.model_dir) / "versions.jsonl"
    path.parent.mkdir(parents=True, exist_ok=True)
    entry = {"timestamp": datetime.now(timezone.utc).replace(tzinfo=None).isoformat() + "Z",
             "model_number": model_number, "backend": config.model, "config": config_to_dict(config)}
    with open(path, "a") as f:
        f.write(json.dumps(entry) + "\n")


def _require_pytorch(config):
    if config.model != "pytorch":
        raise NotImplementedError(
            f"model={config.model!r}: only the reference's model='pytorch' path exists here (Keras/TFLite are out of scope)")


def instantiate_network(config, show_summary=True, save_network=True, plot_model=False):
    """Random-init network chosen by type(config.model_config); saved as <model_dir>/0.pt with a
    versions.jsonl line; returned in TRAIN mode like the reference (only load_model calls eval())."""
    _require_pytorch(config)
    model = build_network(config.model_config, config.use_tanh).to(device)
    if show_summary:
        print(model)
    if save_network:
        os.makedirs(config.model_dir, exist_ok=True)
        torch.save(model.state_dict(), f"{config.model_dir}/0.pt")
        append_version_record(config, 0)
    return model


def _numbered(path, strip_pt):
    best = -1
    os.makedirs(path, exist_ok=True)
    for filename in os.listdir(path):
        stem = filename[:-3] if (strip_pt and filename.endswith(".pt")) else filename.split(".")[0]
        if stem.isdigit():
            best = max(best, int(stem))
    return best


def highest_model_number(config):
    _require_pytorch(config)
    return _numbered(config.model_dir, strip_pt=True)


def highest_data_number(config):
    return _numbered(config.data_dir, strip_pt=False)


def load_model(config, model_number):
    _require_pytorch(config)
    path = f"{config.model_dir}/{model_number}.pt"
    if not os.path.exists(path):
        path = f"{config.model_dir}/{model_number}"  # legacy checkpoints without an extension
    model = build_network(config.model_config, config.use_tanh)
    model.load_state_dict(torch.load(path, weights_only=True))
    model.to(device)
    model.eval()
    print(path)
    return model


def load_best_model(config):
    return load_model(config, highest_model_number(config))


def load_best_train_and_interference_models(config):
    m = load_best_model(config)
    return m, m


def get_interference_network(config, training_network):
    return training_network


# ---------------------------------------------------------------------------------------------
# training targets: visit fractions, mirror augmentation, sample layout
# ---------------------------------------------------------------------------------------------

def policy_target_from_visits(moves, visits):
    """search_statistics on a finished search: float64 (27,39,11), round(n / total, 4) at every
    root child with n != 0 (post-prune counts), zero elsewhere."""
    visits = np.asarray(visits, dtype=np.int64)
    total = int(visits.sum())
    assert total != 0
    out = np.zeros(POLICY_SHAPE, dtype=np.float64)
    flat = out.reshape(-1)
    nz = visits != 0
    flat[np.asarray(moves, dtype=np.int64)[nz]] = [round(int(n) / total, 4) for n in visits[nz]]
    return out


def search_statistics(tree):
    """Reference signature: `tree` is the SearchResult returned by MCTS()."""
    probs = policy_target_from_visits(tree.moves, tree.visits)
    return _policy_to_lists(probs)


def _policy_to_lists(p):
    """ndarray -> nested lists with int 0 where nothing was visited (like the reference's lists)."""
    lists = p.tolist()
    for plane in lists:
        for row in plane:
            for i, v in enumerate(row):
                if v == 0:
                    row[i] = 0
    return lists


def reflect_grid(grid):
    if isinstance(grid, np.ndarray):
        return np.fliplr(grid).tolist()
    return [row[::-1] for row in grid]


_PIECE_MIRROR = np.array([3, 5, 2, 0, 4, 1, 6])  # Z<->S, L<->J over "ZLOSIJT"


def reflect_pieces(piece_table):
    t = np.asarray(piece_table)
    out = np.zeros((2 + PREVIEWS, len(MINOS)), dtype=int)
    for i, row in enumerate(t):
        hit = np.flatnonzero(row == 1)
        if hit.size:
            out[i][_PIECE_MIRROR[hit[0]]] = 1
    return out


def _reflection_table():
    """plane -> (mirrored plane, piece matrix size, post-flip column adjustment)."""
    from .const import MATRIX_SIZE
    swap = {"Z": "S", "S": "Z", "L": "J", "J": "L"}
    tab = []
    for plane in range(POLICY_SHAPE[0]):
        piece, rot, tsi = policy_index_to_piece[plane]
        new_piece = swap.get(piece, piece)
        new_rot = {1: 3, 3: 1}.get(rot, rot)
        adj = 0
        if new_piece in ("Z", "S", "I") and new_rot == 3:
            adj, new_rot = -1, 1
        tab.append((policy_piece_to_index[new_piece][new_rot][tsi], MATRIX_SIZE[piece], adj))
    return tab


_REFLECT = _reflection_table()


def reflect_policy_array(p):
    """Mirror a (27,39,11) policy target: piece/rotation swap and column flip
    new_col = 10 - (col-2) - size + 2 (+ adjustment for folded Z/S/I rotations)."""
    p = np.asarray(p)
    out = np.zeros(POLICY_SHAPE, dtype=p.dtype)
    for plane, (new_plane, size, adj) in enumerate(_REFLECT):
        rows, cols = np.nonzero(p[plane] > 0)
        if rows.size:
            out[new_plane, rows, 10 - (cols - 2) - size + 2 + adj] = p[plane, rows, cols]
    return out


def reflect_policy(policy_matrix):
    return _policy_to_lists(reflect_policy_array(np.asarray(policy_matrix, dtype=np.float64)))


def features_from_state(rec):
    """game_to_X (ai.py:1399-1413) on a packed position, in the reference's python types:
    (a_grid float32 (40,10), a_pieces float32 (7,7), a_b2b, a_combo, a_garbage, o_grid, o_pieces, ...)"""
    turn = int(rec["turn"])
    out = []
    for pl in (turn, 1 - turn):
        p = rec["players"][pl]
        grid = rows_to_grid(p["rows"]).astype(np.float32)
        table = np.zeros((2 + PREVIEWS, len(MINOS)), dtype=np.float32)
        if int(p["piece"]) != 255:
            table[0, int(p["piece"])] = 1
        if int(p["held"]) != 255:
            table[1, int(p["held"])] = 1
        for j in range(min(int(p["qlen"]), PREVIEWS)):
            table[2 + j, int(p["queue"][j])] = 1
        out += [grid, table, int(p["b2b"]), int(p["combo"]), int(p["n_recv"])]
    out.append(turn)
    return tuple(out)


def samples_from_search(state_rec, moves, visits, augment=True):
    """The per-move block of play_game (ai.py:1613-1666): the (optionally x4 mirrored) samples
    of one saved search, WITHOUT the outcome value (inserted when the game ends)."""
    feats = features_from_state(state_rec)
    target = policy_target_from_visits(moves, visits)
    listify = lambda f: f.tolist() if isinstance(f, np.ndarray) else f  # noqa: E731
    if not augment:
        return [[listify(f) for f in feats] + [_policy_to_lists(target)]]
    plain, mirrored = _policy_to_lists(target), _policy_to_lists(reflect_policy_array(target))
    out = []
    for active_reflected in (0, 1):
        for other_reflected in (0, 1):
            d = [f.copy() if isinstance(f, np.ndarray) else f for f in feats]
            if active_reflected:
                d[0], d[1] = reflect_grid(d[0]), reflect_pieces(d[1])
            if other_reflected:
                d[5], d[6] = reflect_grid(d[5]), reflect_pieces(d[6])
            d = [listify(f) for f in d]
            d.append(mirrored if active_reflected else plain)
            out.append(d)
    return out


# ---------------------------------------------------------------------------------------------
# self-play
# ---------------------------------------------------------------------------------------------

def _time_seed(seed):
    return int(time.time_ns() & 0x7FFFFFFF) if seed is None else seed


def _engine_for(config, net, n_games, seed=None, device=None, **kw):
    """Engine of n_games on `device` (default: the current device).  A network is copied to that device; a callable
    evaluator is used as given and must accept inputs on it."""
    from .selfplay import SelfPlayEngine, best_evaluator
    if not torch.cuda.is_available():
        raise RuntimeError("self-play needs a CUDA device: the search, rules and placements run in libtrl_b200.so "
                           "(there is no CPU fallback)")
    seed = _time_seed(seed)
    dtype = kw.pop("dtype", torch.bfloat16)
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    with torch.cuda.device(device):
        if callable(net) and not isinstance(net, torch.nn.Module):
            evaluator = net
        else:
            import copy
            evaluator = best_evaluator(copy.deepcopy(net).to(device), dtype)  # the caller's module is left untouched
        return SelfPlayEngine(config, evaluator, n_games, seed=seed, feature_dtype=dtype, device=device, **kw)


def _shard_engines(config, net, num_games, concurrent, seed, first_game_id, game_id_stride, **kw):
    """One engine per entry of config.engine_devices, each playing its devices.shard_games share of the ids (finished
    games restart while the shard has more games than slots).  -> [(engine, shard)]."""
    from .devices import engine_devices, shard_games
    devs = engine_devices(config)
    out = []
    for sh in shard_games(num_games, concurrent, first_game_id, game_id_stride, len(devs)):
        eng = _engine_for(config, net, sh["concurrent"], seed=seed, device=devs[sh["shard"]], first_game_id=sh["first_game_id"],
                          game_id_stride=sh["game_id_stride"], restart_finished=sh["concurrent"] < sh["num_games"], **kw)
        out.append((eng, sh))
    return out


def generate_games(config, net, num_games, seed=None, concurrent=None, augment=None, dtype=torch.bfloat16,
                   first_game_id=0, game_id_stride=1, max_steps=None, compact=False):
    """Play `num_games` complete self-play games (all concurrently by default) and return
    (series_data, series_stats) like the reference's serial loop over play_game
    (ai.py:1817-1820): series_data = 13-element samples grouped per game (player 0's samples,
    then player 1's), series_stats = one APP/DSPP dict per game.  compact=True: series_data is a
    compact.CompactSet holding the same samples in the same order (sample i of the list =
    CompactSet.batch_tensors([i])), without building Python lists.

    config.engine_devices: the games are sharded by id over the listed devices (devices.shard_games), all engines
    stepped from this thread, and the records merged; the set is the one a single device plays (see Config)."""
    augment = config.augment_data if augment is None else augment
    G = int(concurrent or num_games)
    shards = _shard_engines(config, net, num_games, G, _time_seed(seed), first_game_id, game_id_stride, dtype=dtype,
                            random_openings=True)
    # steps between two drains: a game finishes at most one search per `iters_min` steps and the sample ring holds
    # 4 records per game, so at most 3 * iters_min steps may pass (random opening plies leave no record)
    iters_min = config.playout_iterations()[1] if (config.training and config.use_playout_cap_randomization) else config.MAX_ITER
    chunk = max(1, min(max(8, config.MAX_ITER // 2), 3 * max(1, iters_min)))
    per_game, finished = {}, {}
    all_samples, all_ends = [], []
    running = [(eng, sh["num_games"], set()) for eng, sh in shards]   # (engine, its share, ids it finished)
    steps = 0
    while running:
        for eng, _, _ in running:    # queue every engine's graphs before the first drain waits for its device
            eng.step(chunk)
        steps += chunk
        still = []
        for eng, quota, done in running:
            samples, ends = eng.drain()
            eng.check_status()   # overflowed FIFO / arena / rings, a root without a move: the reference asserts (ai.py:417,1347)
            if compact:       # no per-record Python: the set is assembled from the arrays at the end
                all_samples.append(samples)
                all_ends.append(ends)
            else:
                for s in samples:
                    per_game.setdefault(int(s["game_id"]), []).append(s)
            for e in ends:
                finished[int(e["game_id"])] = e
                done.add(int(e["game_id"]))
            if len(done) < quota and (max_steps is None or steps < max_steps) and eng.get_ctl()["active"].any():
                still.append((eng, quota, done))
        running = still
    data_number, model_number = highest_data_number(config) + 1, highest_model_number(config)
    series_data, series_stats = [], []
    for gid in sorted(finished)[:num_games]:
        e = finished[gid]
        winner = int(e["winner"])
        by_player = [[], []]
        for s in sorted(per_game.get(gid, []), key=lambda r: int(r["search_no"])):
            if not (s["saved"] or config.save_all):
                continue
            C = int(s["n_children"])
            by_player[int(s["turn"])].extend(samples_from_search(s["state"], s["moves"][:C], s["visits"][:C], augment))
        for pl in range(2):
            value = config.value_mid if winner == -1 else (config.value_max if winner == pl else config.value_min)
            for sample in by_player[pl]:
                sample.insert(-1, value)
        series_data.extend(by_player[0] + by_player[1])
        pieces = max(int(e["pieces0"]), 1)
        series_stats.append({"model_number": model_number, "model_version": config.model_version,
                             "data_number": data_number, "data_version": config.data_version,
                             "app": int(e["lines_sent0"]) / pieces, "dspp": int(e["lines_cleared0"]) / pieces})
    if compact:
        from .compact import CompactSet
        from .selfplay import GAME_END_DTYPE, SAMPLE_DTYPE
        series_data = CompactSet.from_records(
            np.concatenate(all_samples) if all_samples else np.zeros(0, SAMPLE_DTYPE),
            np.concatenate(all_ends) if all_ends else np.zeros(0, GAME_END_DTYPE),
            (config.value_min, config.value_mid, config.value_max), num_games=num_games, save_all=config.save_all,
            augment=augment)
    return series_data, series_stats


def make_training_set(config, interference_network, num_games, save_game=False, save_stats=True, screen=None,
                      seed=None, data_format=None):
    """Reference contract (ai.py:1809-1845): writes <data_dir>/<n>.txt (one JSON list of samples)
    when save_game, appends averaged APP/DSPP to logs/stats.jsonl when save_stats, and returns the
    sample list only when save_stats is False.  data_format="compact" (default: config.engine_data_format)
    keeps the samples as a compact.CompactSet and writes <n>.npz instead: same samples, same order,
    0.6 KB instead of 162 KB per saved search and no per-sample Python work."""
    data_format = data_format or getattr(config, "engine_data_format", None) or "json"
    if data_format not in ("json", "compact"):
        raise ValueError(f"unknown data_format {data_format!r}")
    series_data, series_stats = generate_games(config, interference_network, num_games, seed=seed,
                                               compact=(data_format == "compact"))
    if save_game:
        next_set = highest_data_number(config) + 1
        if data_format == "compact":
            series_data.save(f"{config.data_dir}/{next_set}.npz")
        else:
            with open(f"{config.data_dir}/{next_set}.txt", "w") as out_file:
                out_file.write(json.dumps(series_data))
    if save_stats:
        averaged = {
            "model_number": series_stats[0]["model_number"], "model_version": series_stats[0]["model_version"],
            "data_number": series_stats[0]["data_number"], "data_version": series_stats[0]["data_version"],
            "app": round(sum(x["app"] for x in series_stats) / len(series_stats), 3),
            "dspp": round(sum(x["dspp"] for x in series_stats) / len(series_stats), 3),
        }
        with open(logs_dir() / "stats.jsonl", "a") as out_file:
            out_file.write(json.dumps(averaged) + "\n")
    else:
        return series_data


def export_training_set_json(config, set_number, out_path=None):
    """<data_dir>/<n>.npz (compact set) -> <data_dir>/<n>.txt in the reference's format (one JSON list of 13-element
    samples, ai.py:1822-1829), for consumers that read the reference's files."""
    from .compact import CompactSet
    cset = CompactSet.load(f"{config.data_dir}/{set_number}.npz")
    out_path = out_path or f"{config.data_dir}/{set_number}.txt"
    samples = cset.to_json_samples()
    with open(out_path, "w") as f:
        f.write(json.dumps(samples))
    return out_path


class SearchResult:
    """What MCTS() and analyse() return in place of the reference's MCTSTree: the root children of the search
    (reference order), their pre- and post-prune visit counts, the chosen move and the save flag; with the root
    statistics (include/trl.h, TrlRootStats) also, per child, the prior the PUCT used (after the root softmax
    temperature and the Gamma noise mix) and the Q value (value_avg; the FPU value for an unvisited child), the
    root's value_avg and the principal variation (policy indices, most visited child first)."""

    def __init__(self, sample, stats=None):
        C = int(sample["n_children"])
        self.moves = sample["moves"][:C].astype(np.int64)
        self.visits = sample["visits"][:C].astype(np.int64)
        self.visits_pre = sample["visits_pre"][:C].astype(np.int64)
        self.iterations = int(sample["iterations"])
        self.state = sample["state"].copy()
        self.chosen_move = int(sample["chosen_move"])
        self.move = index_to_move(self.chosen_move)
        self.saved = bool(sample["saved"])
        self.priors = self.q = self.root_value = self.pv = self.pv_visits = None
        if stats is not None:
            self.priors = stats["prior"][:C].copy()
            self.q = stats["q"][:C].copy()
            self.root_value = float(stats["root_value"])
            L = int(stats["pv_len"])
            self.pv = stats["pv"][:L].astype(np.int64)
            self.pv_visits = stats["pv_visits"][:L].astype(np.int64)

    def root_children(self):
        return [(index_to_move(m), int(n)) for m, n in zip(self.moves, self.visits)]


_SEARCH_KEYS = ("MAX_ITER", "CPUCT", "DPUCT", "FpuStrategy", "FpuValue", "use_root_softmax", "RootSoftmaxTemp", "use_tanh",
                "training", "temperature", "use_playout_cap_randomization", "playout_cap_chance", "playout_cap_mult",
                "use_dirichlet_noise", "DIRICHLET_ALPHA", "DIRICHLET_S", "DIRICHLET_EXPLORATION", "use_dirichlet_s",
                "use_forced_playouts_and_policy_target_pruning", "CForcedPlayout", "ruleset", "move_algorithm")
_ANALYSE_MAX_BATCH = 4096   # positions searched concurrently by analyse(); larger inputs run in chunks of this size
_CACHE_ENTRIES = 4
# Engines and evaluators are built from a copy of the caller's network and kept between calls.  An entry is
# (weak reference to the network, value): it serves only the very object it was built for, so a network freed and
# replaced by another one at the same address (same id, same parameter versions after load_state_dict) misses.
_search_engines = {}   # (network identity + weight versions, search settings, seed, batch, device, block) -> entry
_evaluators = {}       # (network identity + weight versions, device) -> entry of evaluate() / evaluate_positions()


def _net_identity(net):
    """id plus the in-place version counters of the parameters: a trained / re-loaded network gets a new key."""
    if isinstance(net, torch.nn.Module):
        return (id(net), tuple(int(t._version) for t in list(net.parameters()) + list(net.buffers())))
    return (id(net),)


def _net_ref(net):
    try:
        return weakref.ref(net)
    except TypeError:           # not weak-referenceable: the entry keeps the object alive, so its id stays its own
        return lambda: net


def _cache_get(cache, key, net):
    entry = cache.get(key)
    return entry[1] if entry is not None and entry[0]() is net else None


def _cache_put(cache, key, net, value, device=None):
    """At most _CACHE_ENTRIES entries per device, the oldest leaving first."""
    cache.pop(key, None)
    same_device = [k for k, entry in cache.items() if entry[2] == device]
    for k in same_device[:max(0, len(same_device) - _CACHE_ENTRIES + 1)]:
        cache.pop(k)
    cache[key] = (_net_ref(net), value, device)


def release_cached_engines():
    """Drop the search engines and evaluators that MCTS(), analyse(), evaluate() and evaluate_positions() keep
    between calls (tree arenas of several GB for thousands of positions) and return their memory on every device."""
    _search_engines.clear()
    _evaluators.clear()
    if torch.cuda.is_available():
        for d in range(torch.cuda.device_count()):
            if torch.cuda.memory_reserved(d):      # empty_cache() would create a context on a device never used
                with torch.cuda.device(d):
                    torch.cuda.empty_cache()


_process_seed = []     # the time-based Philox key of every analysis engine built with seed=None in this process


def _search_engine(config, net, seed, n_games, device, block):
    """main.py-style callers search move after move with the same network (reference main.py:80,145): keep the
    analysis engine (evaluator, packed weights, tree buffers, CUDA graphs) instead of rebuilding it per call.
    `block`: the index of the caller's block of positions; every block of one call has its own engine, also when
    config.engine_devices names a device twice.  seed=None: one time-based key shared by all of them."""
    key = (_net_identity(net), tuple(repr(getattr(config, k, None)) for k in _SEARCH_KEYS), seed, int(n_games), str(device),
           int(block))
    eng = _cache_get(_search_engines, key, net)
    if eng is None:
        _search_engines.pop(key, None)      # a stale entry of a freed network frees its buffers before the new one
        if seed is None and not _process_seed:
            _process_seed.append(_time_seed(None))
        eng = _engine_for(config, net, n_games, seed=_process_seed[0] if seed is None else seed, device=device,
                          restart_finished=False, analysis=True, root_stats=True)
        _cache_put(_search_engines, key, net, eng, str(device))
    return eng


def _engine_batch(n):
    """Engine size for n positions: the next power of two, at most _ANALYSE_MAX_BATCH (extra slots stay inactive),
    so that varying input lengths share a few engines."""
    return min(_ANALYSE_MAX_BATCH, 1 << max(0, n - 1).bit_length())


def _pack_positions(games):
    """A GAME_DTYPE array (copied) or a list of reference-style Game objects -> GAME_DTYPE[n]."""
    if isinstance(games, np.ndarray) and games.dtype == GAME_DTYPE:
        return games.reshape(-1).copy()
    recs = np.zeros(len(games), dtype=GAME_DTYPE)
    for i, g in enumerate(games):
        pack_game(g, out=recs[i])
    return recs


def _per_position(x, n, name):
    a = np.broadcast_to(np.asarray(x, dtype=np.int64), (n,))
    if (a < 0).any() or (a > 0xFFFFFFFF).any():
        raise ValueError(f"{name} must hold 32-bit unsigned integers")
    return a


def _analyse_packed(config, recs, network, seed, search_no, strict):
    """One analysis-mode search per packed position, chunks of _ANALYSE_MAX_BATCH games stepped under CUDA graphs
    until every game has finished its own search.  -> [SearchResult or None] in input order.  strict: any device
    status bit raises (MCTS); otherwise a root without a legal move (NO_PIECE, also set for a terminal root) only
    yields None.  config.engine_devices: the positions are split into contiguous blocks, one per device, searched
    concurrently."""
    from .devices import contiguous_blocks, engine_devices
    from .selfplay import CTL_DTYPE, EngineStatusError
    n = len(recs)
    if n == 0:
        return []
    devs = engine_devices(config)
    # (engine, first position, end) per block with positions; no two blocks share an engine
    jobs = [(_search_engine(config, network, seed, _engine_batch(hi - lo), dev, k), lo, hi)
            for k, (dev, (lo, hi)) in enumerate(zip(devs, contiguous_blocks(n, len(devs)))) if hi > lo]
    long_iters, _ = config.playout_iterations()
    budget = long_iters if (config.training and config.use_playout_cap_randomization) else config.MAX_ITER
    out = [None] * n
    rnd = 0
    while True:     # round r: chunk r of every block (one round unless a block exceeds _ANALYSE_MAX_BATCH)
        live = []
        for eng, lo, hi in jobs:
            c0 = lo + rnd * eng.G
            if c0 >= hi:
                continue
            k = min(hi, c0 + eng.G) - c0
            games = np.zeros(eng.G, dtype=GAME_DTYPE)
            games[:k] = recs[c0:c0 + k]
            ctl = np.zeros(eng.G, dtype=CTL_DTYPE)
            ctl["active"][:k] = 1
            ctl["search_no"][:k] = search_no[c0:c0 + k]
            eng.drain()
            eng.set_games(games)
            eng.set_ctl(ctl)
            eng.step(budget)      # one simulation per game and step: every search ends within the largest budget
            live.append((eng, c0))
        if not live:
            return out
        for eng, c0 in live:
            if eng.get_ctl()["active"].any():
                raise EngineStatusError("analysis engine: a search did not finish within its iteration budget")
            samples, _ = eng.drain()
            stats = eng.drain_root_stats()
            eng.check_status(ignore=0 if strict else 0x4)
            for smp, st in zip(samples, stats):
                out[c0 + int(st["slot"])] = SearchResult(smp, st)
        rnd += 1


def analyse(config, games, network, seed=None, game_ids=None, search_no=0):
    """Search many caller-supplied positions at once on the device: one MCTS search per position with `config`'s
    settings, all positions in lock-step (the reference runs MCTS once per position, ai.py:299).

    games: a list of reference-style Game objects or a GAME_DTYPE array; they are not modified.
    game_ids, search_no: scalars or per-position arrays keying the Philox streams of each search (playout-cap coin,
    Gamma noise, temperature choice, garbage columns) exactly as MCTS()'s game_id / search_no do.  By default a
    GAME_DTYPE array keeps the game_id of its records and Game objects are numbered 0, 1, ...
    seed: the Philox key (None: a time-based one drawn once per process, shared by every block and every call).
    -> one SearchResult per position, in input order; None for a position that is already over or has no legal
    move at the root (MCTS raises there).  Any other device status raises EngineStatusError."""
    _require_pytorch(config)
    recs = _pack_positions(games)
    n = len(recs)
    if game_ids is not None:
        recs["game_id"] = _per_position(game_ids, n, "game_ids")
    elif not (isinstance(games, np.ndarray) and games.dtype == GAME_DTYPE):
        recs["game_id"] = np.arange(n)
    return _analyse_packed(config, recs, network, seed, _per_position(search_no, n, "search_no"), strict=False)


def MCTS(config, game, interference_network, seed=None, game_id=0, search_no=0):
    """One search of one reference-style `Game` (ai.py:299): returns (move=(plane, col, row),
    SearchResult, save_bool).  `game` is not mutated.  No random opening plies here, whatever
    config.use_random_starting_moves says: only play_game draws them (ai.py:1588-1608).
    The one-position case of analyse(); a root without a legal move raises EngineStatusError."""
    _require_pytorch(config)
    rec = np.zeros(1, dtype=GAME_DTYPE)
    pack_game(game, game_id=game_id, out=rec[0])
    res = _analyse_packed(config, rec, interference_network, seed, _per_position(search_no, 1, "search_no"), strict=True)[0]
    if res is None:
        raise RuntimeError("search produced no result (game already over or no legal move)")
    return res.move, res, res.saved


def _evaluator_for(network, device):
    """best_evaluator of a copy of `network` on `device` in bf16 (fused trunk + heads where supported), cached per
    network and device.  A callable evaluator is used as given."""
    from .selfplay import best_evaluator
    if callable(network) and not isinstance(network, torch.nn.Module):
        return network
    key = (_net_identity(network), str(device))
    ev = _cache_get(_evaluators, key, network)
    if ev is None:
        import copy
        _evaluators.pop(key, None)
        with torch.cuda.device(device):
            ev = best_evaluator(copy.deepcopy(network).to(device), torch.bfloat16)
        _cache_put(_evaluators, key, network, ev, str(device))
    return ev


def _evaluate_packed(network, recs, device=None):
    """Network outputs for packed positions: trl_encode_features (bf16) on `device` (default: the current one), then
    the network's best_evaluator there.  -> (values float32 [n], logits float32 [n, 11583]) on that device."""
    from . import _native
    from .const import POLICY_SIZE
    if not torch.cuda.is_available():
        raise RuntimeError("evaluate needs a CUDA device: the feature encoder and the network kernels run in "
                           "libtrl_b200.so (there is no CPU fallback)")
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    n = len(recs)
    with torch.cuda.device(dev):
        d_games = torch.from_numpy(np.ascontiguousarray(recs).view(np.uint8).reshape(-1)).to(dev)
        grids = torch.empty((2 * n, 1, 40, 10), dtype=torch.bfloat16, device=dev)
        extras = torch.empty((n, 105), dtype=torch.bfloat16, device=dev)
        rc = _native.lib().trl_encode_features(d_games.data_ptr(), None, n, grids.data_ptr(), extras.data_ptr(), 1,
                                               torch.cuda.current_stream(dev).cuda_stream)
        _native.check(rc, "trl_encode_features")
        with torch.no_grad():
            values, logits = _evaluator_for(network, dev)(grids, extras)
        return values.reshape(-1).float(), logits[:, :POLICY_SIZE].float()


def evaluate_positions(config, games, network):
    """Batched evaluate(): games = a list of reference-style Game objects or a GAME_DTYPE array.
    -> (values float32 [N], policies float32 [N, 27, 39, 11], each the softmax over all 11583 logits).
    config.engine_devices: the positions are split into contiguous blocks, one per device."""
    from .devices import contiguous_blocks, engine_devices
    _require_pytorch(config)
    recs = _pack_positions(games)
    n = len(recs)
    values = np.zeros(n, dtype=np.float32)
    policies = np.zeros((n,) + tuple(POLICY_SHAPE), dtype=np.float32)
    devs = engine_devices(config)
    blocks = [(dev, lo, hi) for dev, (lo, hi) in zip(devs, contiguous_blocks(n, len(devs))) if hi > lo]
    for start in range(0, max([hi - lo for _, lo, hi in blocks], default=0), _ANALYSE_MAX_BATCH):
        outs = []
        for dev, lo, hi in blocks:     # queue chunk `start` of every block, then copy the results back
            c0, c1 = lo + start, min(hi, lo + start + _ANALYSE_MAX_BATCH)
            if c0 < c1:
                v, logits = _evaluate_packed(network, recs[c0:c1], dev)
                with torch.cuda.device(dev):
                    outs.append((c0, c1, v, torch.softmax(logits, dim=1)))
        for c0, c1, v, p in outs:
            values[c0:c1] = v.cpu().numpy()
            policies[c0:c1] = p.cpu().numpy().reshape((c1 - c0,) + tuple(POLICY_SHAPE))
    return values, policies


def evaluate(config, game, network):
    """The reference's evaluate (ai.py:1222-1319): one position -> (value float, policy float32 ndarray (27,39,11),
    the softmax over all 11583 logits)."""
    packed = isinstance(game, (np.ndarray, np.void)) and game.dtype == GAME_DTYPE
    values, policies = evaluate_positions(config, np.array(game, dtype=GAME_DTYPE).reshape(1) if packed else [game],
                                          network)
    return float(values[0]), policies[0]


def self_play_loop(config, skip_first_set=False):
    """Reference loop (ai.py:2117-2198): self-play set -> train on the last sets -> gate the
    challenger against the best network -> promote.  Never returns."""
    from . import training
    best_train, best_infer = load_best_train_and_interference_models(config)
    training_config = config.copy()
    training_config.training = True
    it = 0
    while True:
        it += 1
        challenger, challenger_infer = load_best_train_and_interference_models(config)
        if not skip_first_set:
            print(f"Starting training loop {it} with network version {highest_model_number(config)}")
            for _ in range(config.training_loops):
                # compact sets by default: the JSON writer caps this call at 1.7e4 games/h against 2.5e6 (DESIGN.md 3.5);
                # training.load_data_and_train_model reads both, export_training_set_json() writes the reference's <n>.txt
                make_training_set(training_config, challenger_infer, num_games=config.training_games,
                                  save_game=True, save_stats=True, data_format=config.engine_data_format or "compact")
                print("Finished making training set")
        else:
            skip_first_set = False
        training.load_data_and_train_model(config, challenger, data=None)
        challenger_infer = get_interference_network(config, challenger)
        print("Finished training network")
        next_ver = highest_model_number(config) + 1
        print(f"Battling a challenger against version {next_ver - 1}")
        win_loss, win = training.battle_networks(challenger_infer, config, best_infer, config, config.gating_threshold,
                                                 config.gating_threshold_type, config.battle_games,
                                                 network_1_title="Challenger", network_2_title="Best")
        print(f"Challenger {win_loss[0]} - {win_loss[1]} Best")
        with open(logs_dir() / "gating_log.jsonl", "a") as f:
            f.write(json.dumps({"model_version": config.model_version, "challenger_number": next_ver,
                                "challenger_wins": int(win_loss[0]), "best_wins": int(win_loss[1]),
                                "total_games": config.battle_games,
                                "win_rate": float(win_loss[0]) / config.battle_games, "accepted": bool(win)}) + "\n")
        if win:
            print(f"Challenger version {next_ver} won and is now the best network")
            torch.save(challenger.state_dict(), f"{config.model_dir}/{next_ver}.pt")
            append_version_record(config, next_ver)
            best_infer = challenger_infer
