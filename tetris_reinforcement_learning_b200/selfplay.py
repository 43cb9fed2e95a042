"""Device-resident batched self-play engine.

Replaces the body of make_training_set / _make_training_set_async / aplay_game / amcts /
BatchedEvaluator (reference ai.py:670-996, 1702-1869): G games per GPU advance in lock-step,
one MCTS simulation per game per step:

    select+materialise (mcts.cu) -> legal placements of the leaves (movegen_warp.cu)
    -> feature encode (features.cu) -> policy/value net on the G-leaf batch
    -> expand+backup(+finish search, play the move, restart finished games) (mcts.cu)

With the fused AlphaSame evaluator (trunk.CachedTrunkEvaluator) a step is launched as
    forked stream:  gate -> enumeration of the leaves without a cached sibling list (compacted work list)
    main stream  :  trunk -> heads -> policy GEMM -> [expand(t) + select(t+1) + encode(t+1)] (one kernel)
(DESIGN.md section 3.4).  Steps are captured into CUDA graphs (steps_per_graph per launch); there are no
host round-trips inside a step.  Finished searches leave `TrlSample` records (position, root children,
post-prune visit counts) and finished games `TrlGameEnd` records in HBM ring buffers that the host
drains between graph replays (drain(): pinned, double-buffered).
"""
import ctypes
import functools

import numpy as np
import torch

from . import _native
from .const import POLICY_SIZE
from .state import GAME_DTYPE

SAMPLE_MOVES = 512

CTL_DTYPE = np.dtype({
    "names": ["iter", "max_iter", "n_nodes", "n_states", "leaf", "leaf_kind", "search_no", "garbage_ctr", "status",
              "fast", "active", "games_finished", "sims", "lines_sent0", "lines_cleared0", "leaf_value",
              "max_depth", "random_left"],
    "formats": ["<i4", "<i4", "<i4", "<i4", "<i4", "<i4", "<u4", "<u4", "<u4", "<u4", "<u4", "<u4", "<u8",
                "<i4", "<i4", "<f8", "<i4", "<i4"],
    "offsets": [0, 4, 8, 12, 16, 20, 24, 28, 32, 36, 40, 44, 48, 56, 60, 64, 72, 76],
    "itemsize": 80,
})

SAMPLE_DTYPE = np.dtype({
    "names": ["game_id", "search_no", "turn", "saved", "n_children", "chosen_move", "total_visits", "iterations",
              "state", "moves", "visits", "visits_pre"],
    "formats": ["<u4", "<u2", "u1", "u1", "<u2", "<u2", "<u4", "<i4", GAME_DTYPE,
                ("<u2", (SAMPLE_MOVES,)), ("<u2", (SAMPLE_MOVES,)), ("<u2", (SAMPLE_MOVES,))],
    "offsets": [0, 4, 6, 7, 8, 10, 12, 16, 20, 420, 420 + 2 * SAMPLE_MOVES, 420 + 4 * SAMPLE_MOVES],
    "itemsize": 420 + 6 * SAMPLE_MOVES,
})

PV_MAX = 16

# TrlRootStats (include/trl.h): root statistics of one search, at the slot index of its TrlSample
ROOT_STATS_DTYPE = np.dtype({
    "names": ["root_value", "root_visits", "slot", "n_children", "pv_len", "pv_visits", "pv", "prior", "q"],
    "formats": ["<f4", "<u4", "<i4", "<u2", "<u2", ("<u4", (PV_MAX,)), ("<u2", (PV_MAX,)),
                ("<f4", (SAMPLE_MOVES,)), ("<f4", (SAMPLE_MOVES,))],
    "offsets": [0, 4, 8, 12, 14, 16, 80, 112, 112 + 4 * SAMPLE_MOVES],
    "itemsize": 112 + 8 * SAMPLE_MOVES,
})

GAME_END_DTYPE = np.dtype({
    "names": ["game_id", "winner", "plies", "rounds", "pieces0", "lines_sent0", "lines_cleared0", "pad_"],
    "formats": ["<u4", "<i4", "<u4", "<u4", "<i4", "<i4", "<i4", "<i4"],
    "offsets": [0, 4, 8, 12, 16, 20, 24, 28],
    "itemsize": 32,
})


STATUS_BITS = {0x1: "QUEUE_OVERFLOW (movegen FIFO)", 0x2: "MOVES_TRUNC (move list longer than moves_cap)",
               0x4: "NO_PIECE (root without a legal move)", 0x8: "RECV_OVERFLOW (pending-garbage list)",
               0x10: "BAD_MOVE", 0x20: "SAMPLE_OVERFLOW (sample ring full: records dropped)",
               0x40: "ARENA_FULL (node arena full: a leaf stayed childless)",
               0x80: "END_OVERFLOW (game-end ring full: records dropped)"}


class EngineStatusError(RuntimeError):
    """A device-side TRL_ST_* bit is set: the data of this run is not what the reference would have produced
    (the reference asserts / raises in these situations, ai.py:417,1347)."""


def search_params_from_config(config, seed=0, restart_finished=True, game_id_stride=1, save_all=None, max_rounds=None,
                              random_openings=False, analysis=False):
    """Config (ai.py:97-137) -> TrlSearchParams.  random_openings: only play_game draws random opening plies
    (ai.py:1588-1608); MCTS() and battle_networks never do, whatever config.use_random_starting_moves says.
    analysis: every game stops after its own search (TrlSearchParams.stop_after_search)."""
    from .const import MAX_MOVES
    p = _native.SearchParams()
    p.seed = int(seed)
    p.cpuct, p.dpuct, p.fpu_value = float(config.CPUCT), float(config.DPUCT), float(config.FpuValue)
    p.root_softmax_temp = float(config.RootSoftmaxTemp)
    p.temperature = float(config.temperature)
    p.playout_cap_chance = float(config.playout_cap_chance)
    p.dirichlet_alpha, p.dirichlet_s = float(config.DIRICHLET_ALPHA), float(config.DIRICHLET_S)
    p.dirichlet_eps = float(config.DIRICHLET_EXPLORATION)
    p.c_forced = float(config.CForcedPlayout)
    p.max_iter = int(config.MAX_ITER)
    p.iters_long, p.iters_short = config.playout_iterations()
    if config.FpuStrategy not in ("reduction", "absolute"):
        raise ValueError(f"unknown FpuStrategy {config.FpuStrategy!r}")
    p.fpu_reduction = int(config.FpuStrategy == "reduction")
    p.use_root_softmax = int(bool(config.use_root_softmax))
    p.training = int(bool(config.training))
    p.use_playout_cap = int(bool(config.use_playout_cap_randomization))
    p.use_noise = int(bool(config.use_dirichlet_noise))
    p.use_dirichlet_s = int(bool(config.use_dirichlet_s))
    p.use_forced = int(bool(config.use_forced_playouts_and_policy_target_pruning))
    p.use_tanh = int(bool(config.use_tanh))
    p.save_all = int(bool(config.save_all if save_all is None else save_all))
    p.max_rounds = int(MAX_MOVES if max_rounds is None else max_rounds)
    p.restart_finished = int(bool(restart_finished))
    p.game_id_stride = int(game_id_stride)
    # random opening plies sampled from the raw policy (ai.py:1588-1608); scale = 0.04 * DIRICHLET_S
    p.use_random_start = int(bool(random_openings) and bool(getattr(config, "use_random_starting_moves", False)))
    p.random_start_scale = 0.04 * float(config.DIRICHLET_S)
    p.stop_after_search = int(bool(analysis))
    if p.stop_after_search and p.use_random_start:
        raise ValueError("analysis mode searches the given positions only: random opening plies cannot run in it")
    return p


def _on_device(method):
    """Run an engine method with the engine's device current: the library launches on, and allocates for, the current
    device, and graph capture takes its stream from it.  An engine on cuda:1 then works while cuda:0 is current."""
    @functools.wraps(method)
    def run(self, *args, **kwargs):
        with torch.cuda.device(self.device):
            return method(self, *args, **kwargs)
    return run


class SelfPlayEngine:
    """G concurrent self-play games on one GPU (`device`; every method runs with it current).

    evaluator(grids [2G,1,40,10], extras [G,105]) -> (values [G] or [G,1], logits [G,11583]);
    tensors of `feature_dtype` in, float32 or bfloat16 out.  Normally a network's
    `forward_packed` (see make_net_evaluator); tests inject a deterministic function.

    analysis=True: analysis mode (include/trl.h, TrlSearchParams.stop_after_search): each game runs one search
    of the position it holds, emits its sample and goes inactive; the games are left as they were.
    root_stats=True: every sample also gets a TrlRootStats record (priors, Q values, root value, principal
    variation), read with drain_root_stats() after drain().
    """

    def __init__(self, config, evaluator, n_games, device="cuda:0", seed=0, first_game_id=0, game_id_stride=1,
                 feature_dtype=torch.float32, node_cap=None, sample_cap=None, restart_finished=True, save_all=None,
                 max_rounds=None, use_cuda_graph=True, overlap_movegen=True, reuse_trunk_features=True,
                 reuse_sibling_placements=True, compact_movegen=True, fuse_expand_select=True, fuse_encode=True,
                 steps_per_graph=4, parallel_backup=True, random_openings=False, gather_policy=True, analysis=False,
                 root_stats=False):
        from .state import ruleset_id
        self.ruleset = ruleset_id(config.ruleset)   # 's2' (default) or 's1': attack table + all-spin rule
        if config.move_algorithm != "convolutional":
            raise NotImplementedError("only move_algorithm='convolutional' is implemented on the device path")
        self.lib = _native.lib()
        self.config, self.evaluator = config, evaluator
        self.G = int(n_games)
        self.device = torch.device(device)
        self.params = search_params_from_config(config, seed, restart_finished, game_id_stride, save_all, max_rounds,
                                                random_openings, analysis)
        self.analysis = bool(analysis)
        self.seed = int(seed)
        self.feature_dtype = feature_dtype
        self.use_cuda_graph = use_cuda_graph
        self.overlap_movegen = overlap_movegen
        # exact trunk-feature reuse (trunk.CachedTrunkEvaluator) when the evaluator offers it
        self.cached_eval = getattr(evaluator, "cached", None) if (reuse_trunk_features and feature_dtype == torch.bfloat16) else None
        iters_max = max(self.params.max_iter, self.params.iters_long if (config.training and config.use_playout_cap_randomization) else 0)
        self.state_cap = iters_max + 2
        # node arena per game: a search of n iterations creates sum(children) nodes; 49 per expansion on average,
        # but open boards with two rotatable pieces sustain > 96 (14 of 7e5 searches overflowed an arena of 96 n)
        self.node_cap = int(node_cap) if node_cap else max(1024, iters_max * 256)
        self.moves_cap = SAMPLE_MOVES
        self.sample_cap = int(sample_cap) if sample_cap else max(4 * self.G, 1024)
        self.end_cap = max(2 * self.G, 1024)
        G, dev = self.G, self.device
        nn_, ns = G * self.node_cap, G * self.state_cap
        z = lambda n, dt: torch.zeros(n, dtype=dt, device=dev)  # noqa: E731
        self.t = {
            "prior": z(nn_, torch.float64), "value_sum": z(nn_, torch.float64), "visits": z(nn_, torch.int32),
            "parent": z(nn_, torch.int32), "slot": z(nn_, torch.int32), "move": z(nn_, torch.int16),
            "states": z(ns * 400, torch.uint8), "first_child": z(ns, torch.int32), "n_children": z(ns, torch.int32),
            "fpu": z(ns, torch.float64),
            "ctl": z(G * CTL_DTYPE.itemsize, torch.uint8), "games": z(G * 400, torch.uint8),
            "leaf_state": z(G, torch.int32), "legal": z(G * self.moves_cap, torch.int16), "n_legal": z(G, torch.int16),
            "samples": z(self.sample_cap * SAMPLE_DTYPE.itemsize, torch.uint8), "sample_count": z(1, torch.int32),
            "ends": z(self.end_cap * GAME_END_DTYPE.itemsize, torch.uint8), "end_count": z(1, torch.int32),
            "next_game_id": z(1, torch.int32), "leaf_parent": z(G, torch.int32), "path": z(G * 64, torch.int32),
            "movegen_status": z(G, torch.int32),
        }
        self.root_stats = bool(root_stats)
        if self.root_stats:
            self.t["root_stats"] = z(self.sample_cap * ROOT_STATS_DTYPE.itemsize, torch.uint8)
        self._last_root_stats = np.zeros(0, ROOT_STATS_DTYPE)
        # exact reuse of legal-placement lists between siblings (include/trl.h, TrlSearchBuffers.legal_cache)
        self.reuse_sibling_placements = bool(reuse_sibling_placements)
        if self.reuse_sibling_placements:
            self.t["legal_cache"] = z(ns * self.moves_cap, torch.int16)
            self.t["legal_cache_n"] = torch.full((ns,), -1, dtype=torch.int32, device=dev)
            self.t["movegen_index"] = z(G, torch.int32)
            if compact_movegen:
                # compacted work list of the leaf enumeration: it then occupies ceil(count / 16) SMs instead
                # of all of them next to the trunk kernel (include/trl.h, TrlSearchBuffers.movegen_list)
                self.t["movegen_list"] = z(G, torch.int32)
                self.t["movegen_count"] = z(4, torch.int32)
        # expand(t) and select(t+1) as one kernel; `_selected` = the next step's leaves are already chosen
        self.fuse_expand_select = bool(fuse_expand_select)
        # ... and the feature encoding of the selected leaves in the same kernel (cached evaluator only)
        self.fuse_encode = bool(fuse_encode) and self.fuse_expand_select and self.cached_eval is not None
        self._selected = False
        self._encoded = False
        fdt = feature_dtype
        self.grids = torch.zeros((2 * G, 1, 40, 10), dtype=fdt, device=dev)
        self.extras = torch.zeros((G, 105), dtype=fdt, device=dev)
        self.noise_override = None
        b = _native.SearchBuffers()
        b.n_games, b.node_cap, b.state_cap, b.moves_cap = G, self.node_cap, self.state_cap, self.moves_cap
        b.sample_cap, b.end_cap = self.sample_cap, self.end_cap
        for name, ten in self.t.items():
            setattr(b, name, ten.data_ptr())
        b.noise_override = None
        b.leaf_parent = self.t["leaf_parent"].data_ptr()
        if not parallel_backup:
            b.path = None        # the backup then walks the parent links serially
        self.buf = b
        # policy head evaluated on the legal moves only (needs the cached evaluator, which owns the head input x)
        self.gather_policy = bool(gather_policy) and self.cached_eval is not None and getattr(self.cached_eval, "gather_policy", False)
        self._cache_bufs = self.cached_eval.make_buffers(ns, G, dev, self.moves_cap) if self.cached_eval is not None else None
        assert self.lib.trl_sizeof_search_ctl() == CTL_DTYPE.itemsize and self.lib.trl_sizeof_sample() == SAMPLE_DTYPE.itemsize
        assert self.lib.trl_sizeof_root_stats() == ROOT_STATS_DTYPE.itemsize
        self._pinned, self._pinned_i = None, 0      # host staging of drain()
        self._graph = None
        self._graph_k = None                        # steps_per_graph consecutive steps as ONE graph launch
        self.steps_per_graph = max(1, int(steps_per_graph))
        self._stamps = None
        self._graph_has_select = True
        self._side = None
        self._values = self._logits = None
        self.steps_done = 0
        self.new_games(first_game_id, game_id_stride)

    # ---- state access -----------------------------------------------------------------
    @_on_device
    def new_games(self, first_game_id=0, stride=1):
        """Fresh Game.setup() in every slot; ids first, first+stride, ..."""
        games = self.t["games"].view(self.G, 400)
        rc = self.lib.trl_game_setup(games.data_ptr(), self.G, int(first_game_id), int(stride), self.seed,
                                     torch.cuda.current_stream(self.device).cuda_stream)
        _native.check(rc, "trl_game_setup")
        games[:, GAME_DTYPE.fields["ruleset"][1]] = self.ruleset   # restarted games inherit it (mcts.cu)
        self.t["next_game_id"].fill_(int(first_game_id + self.G * stride))
        ctl = np.zeros(self.G, dtype=CTL_DTYPE)
        ctl["active"] = 1
        self.set_ctl(ctl)
        self._invalidate_selection()

    def _invalidate_selection(self):
        """The host changed games / controls: a selection made by the fused expand+select kernel is
        stale, and so is the work list it left for the enumeration.  (Re-selecting an unchanged game
        reaches the same leaf but advances its in-search garbage-column counter, so change controls
        before the first step or between searches if runs must be reproducible step by step.)"""
        self._selected = False
        self._encoded = False
        if "movegen_count" in self.t:
            self.t["movegen_count"].zero_()
        if getattr(self, "_cache_bufs", None) is not None:
            self._cache_bufs["count"].zero_()    # images queued by a fused encode of the stale selection

    @_on_device
    def set_games(self, games_np):
        assert games_np.dtype == GAME_DTYPE and games_np.shape == (self.G,)
        self.t["games"].copy_(torch.from_numpy(np.ascontiguousarray(games_np).view(np.uint8).reshape(-1)).to(self.device))
        self._invalidate_selection()

    @_on_device
    def get_games(self):
        return self.t["games"].cpu().numpy().view(GAME_DTYPE).reshape(-1)

    @_on_device
    def set_ctl(self, ctl_np):
        assert ctl_np.dtype == CTL_DTYPE and ctl_np.shape == (self.G,)
        self.t["ctl"].copy_(torch.from_numpy(np.ascontiguousarray(ctl_np).view(np.uint8).reshape(-1)).to(self.device))
        self._invalidate_selection()

    @_on_device
    def get_ctl(self):
        return self.t["ctl"].cpu().numpy().view(CTL_DTYPE).reshape(-1)

    @_on_device
    def set_noise_override(self, noise):
        """noise: float64 [G, moves_cap] Gamma draws used instead of the in-kernel sampler (tests)."""
        self.noise_override = torch.as_tensor(noise, dtype=torch.float64, device=self.device).contiguous()
        self.buf.noise_override = self.noise_override.data_ptr()
        self._graph = self._graph_k = None

    # ---- one simulation per game ---------------------------------------------------------
    def _step_eager(self):
        main = torch.cuda.current_stream(self.device)
        lib, st = self.lib, main.cuda_stream
        bp, pp = ctypes.byref(self.buf), ctypes.byref(self.params)
        stamp = self._stamp
        stamp(0, st)
        if not self._selected:
            _native.check(lib.trl_search_select(bp, pp, st), "trl_search_select")
        stamp(1, st)
        # the leaves' legal placements only feed `expand`: enumerate them on a forked stream, concurrently
        # with the network (joined before expand).  overlap_movegen = "trunk": next to feature encoding and
        # the trunk; "heads": next to the heads kernel and the policy GEMM (the trunk is bound by shared-
        # memory bandwidth, which the enumeration also lives on); False: serially before the network.
        def fork_movegen():
            if self._side is None:
                self._side = torch.cuda.Stream(self.device)
            self._side.wait_stream(main)
            stamp(8, self._side.cuda_stream)
            _native.check(lib.trl_search_movegen(bp, self._side.cuda_stream), "trl_search_movegen")
            stamp(9, self._side.cuda_stream)

        mode = self.overlap_movegen
        if mode is True:
            mode = getattr(self.cached_eval, "overlap_mode", "tail") if self.cached_eval is not None else "trunk"
        if mode in ("heads", "tail") and self.cached_eval is None:
            mode = "trunk"
        # "tail": the enumeration depends on the feature encoder (an event) but is submitted AFTER the trunk
        # kernel, so the trunk's CTAs take every SM first and the enumeration's blocks move in as trunk CTAs
        # run out of work (the last, partial wave of the trunk leaves a third of the SMs idle)
        enc_done = None

        def mark_encoded():
            nonlocal enc_done
            enc_done = torch.cuda.Event()
            enc_done.record(main)

        def fork_movegen_tail():
            if self._side is None:
                self._side = torch.cuda.Stream(self.device)
            self._side.wait_event(enc_done)
            _native.check(lib.trl_alphasame_trunk_rows_gate(self._side.cuda_stream), "trl_alphasame_trunk_rows_gate")
            stamp(8, self._side.cuda_stream)
            _native.check(lib.trl_search_movegen(bp, self._side.cuda_stream), "trl_search_movegen")
            stamp(9, self._side.cuda_stream)
        if not mode:
            stamp(8, st)
            _native.check(lib.trl_search_movegen(bp, st), "trl_search_movegen")
            stamp(9, st)
        elif mode == "trunk":
            fork_movegen()
        def join_movegen():
            if self.overlap_movegen and self._side is not None:
                main.wait_stream(self._side)

        if self.cached_eval is not None:
            with torch.no_grad():
                values, logits = self.cached_eval(self._cache_bufs, self.t["states"], self.t["leaf_state"], self.t["leaf_parent"], self.extras,
                                                  after_trunk=fork_movegen if mode == "heads" else (fork_movegen_tail if mode == "tail" else None),
                                                  before_trunk=mark_encoded if mode == "tail" else None, encoded=self._encoded,
                                                  search_buffers=bp if self.gather_policy else None, join_movegen=join_movegen)
        else:
            dt = 0 if self.feature_dtype == torch.float32 else 1
            _native.check(lib.trl_encode_features(self.t["states"].data_ptr(), self.t["leaf_state"].data_ptr(), self.G,
                                                  self.grids.data_ptr(), self.extras.data_ptr(), dt, st), "trl_encode_features")
            with torch.no_grad():
                values, logits = self.evaluator(self.grids, self.extras)
        values = values.reshape(-1)
        if values.dtype != logits.dtype and not (logits.dtype == torch.float32 and logits.shape[1] == self.moves_cap
                                                  and values.dtype == torch.bfloat16 and self.cached_eval is not None):
            values = values.to(logits.dtype)
        gathered = logits.dim() == 2 and logits.shape[1] == self.moves_cap and logits.dtype == torch.float32 and \
            self.cached_eval is not None and self.gather_policy     # logits of the legal moves only (trl_search_policy_legal)
        if not (values.is_contiguous() and logits.dim() == 2 and logits.shape[0] == self.G and
                (gathered or logits.shape[1] >= POLICY_SIZE) and logits.stride(1) == 1):
            raise ValueError("evaluator must return contiguous values [G] and row-major logits [G, >=11583]")
        if logits.dtype not in (torch.float32, torch.bfloat16):
            raise ValueError("evaluator outputs must be float32 or bfloat16")
        if gathered and values.dtype != torch.bfloat16:
            raise ValueError("gathered logits come with bfloat16 values")
        self._values, self._logits = values, logits  # keep alive (graph-owned memory when captured)
        stamp(5, st)
        if self.overlap_movegen:
            main.wait_stream(self._side)
        ldt = 2 if gathered else (0 if logits.dtype == torch.float32 else 1)
        if self.fuse_encode:
            cb = self._cache_bufs
            _native.check(lib.trl_search_expand_select_encode(
                bp, pp, values.data_ptr(), logits.data_ptr(), logits.stride(0), ldt, cb["cache"].data_ptr(),
                cb["images"].data_ptr(), cb["dest"].data_ptr(), cb["count"].data_ptr(), self.extras.data_ptr(),
                cb["own"].data_ptr(), cb["opp"].data_ptr(), cb["rowof"].data_ptr(), st), "trl_search_expand_select_encode")
        else:
            fn, name = ((lib.trl_search_expand_select, "trl_search_expand_select") if self.fuse_expand_select
                        else (lib.trl_search_expand, "trl_search_expand"))
            _native.check(fn(bp, pp, values.data_ptr(), logits.data_ptr(), logits.stride(0), ldt, st), name)
        self._selected = self.fuse_expand_select
        self._encoded = self.fuse_encode
        stamp(6, st)

    @_on_device
    def enable_timeline(self):
        """Profiling: %globaltimer stamps between the kernels of a step (slots: 0 start, 1 after select,
        2 after encode, 3 after trunk, 4 after heads, 5 after policy GEMM, 6 after expand(+select), 8/9 around
        the forked enumeration).  Perturbs the step by one tiny kernel per stamp; re-captures the graph."""
        self._stamps = torch.zeros(16, dtype=torch.int64, device=self.device)
        self._graph = self._graph_k = None
        self.steps_per_graph = 1
        if self.cached_eval is not None:
            self.cached_eval.stamp = self._stamp

    def _stamp(self, k, stream):
        if self._stamps is not None:
            _native.check(self.lib.trl_stamp_globaltimer(self._stamps.data_ptr() + 8 * k, stream), "trl_stamp_globaltimer")

    @_on_device
    def step(self, n=1):
        """Advance every game by n simulations."""
        if not self.use_cuda_graph:
            for _ in range(n):
                self._step_eager()
            self.steps_done += n
            return
        if self._graph is None:
            side = torch.cuda.Stream(self.device)
            side.wait_stream(torch.cuda.current_stream(self.device))
            with torch.cuda.stream(side):
                for _ in range(2):  # warm-up: allocator, cuDNN/cuBLAS plans, library workspaces
                    self._step_eager()
            torch.cuda.current_stream(self.device).wait_stream(side)
            self.steps_done += 2
            n -= 2
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._step_eager()
            self._graph = g
            self._graph_has_select = not self.fuse_expand_select
        if n > 0 and not self._graph_has_select and not self._selected:
            # the host touched games / controls after the capture: choose (and encode) the leaves once outside the graph
            _native.check(self.lib.trl_search_select(ctypes.byref(self.buf), ctypes.byref(self.params),
                                                     torch.cuda.current_stream(self.device).cuda_stream), "trl_search_select")
            self._selected = True
            if self.fuse_encode:
                self.cached_eval.encode(self._cache_bufs, self.t["states"], self.t["leaf_state"], self.t["leaf_parent"], self.extras)
                self._encoded = True
        n = max(n, 0)
        self.steps_done += n
        K = self.steps_per_graph
        if K > 1 and n >= K:
            if self._graph_k is None:
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    for _ in range(K):
                        self._step_eager()
                self._graph_k = g
            for _ in range(n // K):
                self._graph_k.replay()
            n %= K
        for _ in range(n):
            self._graph.replay()

    # ---- outputs ----------------------------------------------------------------------------
    @_on_device
    def drain(self, copy=True):
        """-> (samples SAMPLE_DTYPE[k], game_ends GAME_END_DTYPE[m]) accumulated since the last drain.

        The records cross PCIe into one of two pinned staging buffers (used alternately).  copy=False returns
        views into that buffer, valid until the next-but-one drain (no second host copy of ~3.5 KB per record)."""
        if self._pinned is None:
            mk = lambda n: torch.empty(n, dtype=torch.uint8, pin_memory=True)  # noqa: E731
            self._pinned = [(mk(self.sample_cap * SAMPLE_DTYPE.itemsize), mk(self.end_cap * GAME_END_DTYPE.itemsize), mk(8))
                            for _ in range(2)]
        hs, he, hc = self._pinned[self._pinned_i]
        self._pinned_i ^= 1
        hc[:4].copy_(self.t["sample_count"].view(torch.uint8), non_blocking=True)
        hc[4:].copy_(self.t["end_count"].view(torch.uint8), non_blocking=True)
        torch.cuda.synchronize(self.device)
        cnt = hc.numpy().view(np.uint32)
        if int(cnt[0]) > self.sample_cap or int(cnt[1]) > self.end_cap:
            # the kernels also set TRL_ST_SAMPLE_OVERFLOW / TRL_ST_END_OVERFLOW in the games that lost a record
            raise EngineStatusError(f"record rings overflowed between two drains: {int(cnt[0])} samples (capacity "
                                    f"{self.sample_cap}), {int(cnt[1])} game ends (capacity {self.end_cap}); drain more "
                                    "often or pass a larger sample_cap")
        ns, ne = int(cnt[0]), int(cnt[1])
        nsb, neb = ns * SAMPLE_DTYPE.itemsize, ne * GAME_END_DTYPE.itemsize
        hs[:nsb].copy_(self.t["samples"][:nsb], non_blocking=True)
        he[:neb].copy_(self.t["ends"][:neb], non_blocking=True)
        if self.root_stats:
            self._last_root_stats = self.t["root_stats"][:ns * ROOT_STATS_DTYPE.itemsize].cpu().numpy().view(ROOT_STATS_DTYPE).copy()
        self.t["sample_count"].zero_()
        self.t["end_count"].zero_()
        torch.cuda.synchronize(self.device)
        samples = hs[:nsb].numpy().view(SAMPLE_DTYPE)
        ends = he[:neb].numpy().view(GAME_END_DTYPE)
        return (samples.copy(), ends.copy()) if copy else (samples, ends)

    def drain_root_stats(self):
        """-> ROOT_STATS_DTYPE[k]: the root statistics of the k samples the last drain() returned, in the same order
        (record i belongs to sample i).  Empty unless the engine was built with root_stats=True."""
        return self._last_root_stats

    def status_bits(self):
        """OR of the sticky TRL_ST_* bits of all games (0 = clean)."""
        return int(np.bitwise_or.reduce(self.get_ctl()["status"])) if self.G else 0

    @_on_device
    def check_status(self, ignore=0):
        """Raise EngineStatusError if any game carries a status bit outside `ignore`."""
        st = self.get_ctl()["status"]
        bad = st & ~np.uint32(ignore)
        if bad.any():
            bits = int(np.bitwise_or.reduce(bad))
            names = [n for b, n in STATUS_BITS.items() if bits & b]
            raise EngineStatusError(f"{int((bad != 0).sum())} of {self.G} games report device status 0x{bits:x}: " + "; ".join(names))

    def total_sims(self):
        return int(self.get_ctl()["sims"].sum())


def best_evaluator(net, dtype=torch.bfloat16):
    """The fastest evaluator for `net`: a fused tcgen05 trunk where the architecture allows it (AlphaSame with
    16 filters: csrc/trunk_rows.cu; AlphaSame / BaseResNet / AuxBaseResNet with 32 or 64 filters:
    csrc/trunk_wide.cu), else the plain PyTorch path."""
    from . import trunk, trunk_wide
    if dtype == torch.bfloat16 and trunk.supports(net):
        return trunk.make_fused_evaluator(net, dtype)
    if dtype == torch.bfloat16 and trunk_wide.supports(net):
        return trunk_wide.make_wide_evaluator(net, dtype)
    return make_net_evaluator(net, dtype)


def make_net_evaluator(net, dtype=torch.bfloat16, channels_last=None):
    """Wrap a network (architectures.*) as an engine evaluator: eval mode, `dtype` weights,
    packed inputs (no host tensors).  channels_last=None picks the faster cuDNN layout for the 40x10
    boards, measured on B200 at 4096 leaves per step: NCHW for 32 filters (BaseResNet / AuxBaseResNet(8,32):
    17.1 vs 20.1 ms), channels-last from 64 filters (AlphaSame(20,64): 51.5 vs 61.4 ms)."""
    if channels_last is None:
        widths = [m.out_channels for m in net.modules() if isinstance(m, torch.nn.Conv2d)]
        channels_last = bool(widths) and max(widths) >= 64
    net = net.eval().to(dtype)
    if channels_last:
        net = net.to(memory_format=torch.channels_last)

    def evaluate(grids, extras):
        if channels_last:
            grids = grids.contiguous(memory_format=torch.channels_last)
        out = net.forward_packed(grids, extras)
        return out[0], out[1]

    return evaluate


def shard_for_rank(rank, world, games_per_gpu):
    """Self-play shards independently: rank r owns game ids r, r + world, r + 2*world, ... so the
    set of games played (and each game's Philox streams) is the same for any GPU count; there
    is no collective on the data path.  -> dict(first_game_id, game_id_stride, n_games)."""
    if not (0 <= rank < world):
        raise ValueError("rank out of range")
    return {"first_game_id": int(rank), "game_id_stride": int(world), "n_games": int(games_per_gpu)}
