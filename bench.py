#!/usr/bin/env python
"""bench.py — headline benchmark of the self-play hot path (contract: see DESIGN.md §Measurement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--boards B] [--dump-outputs DIR]

A "step" is one pass of legal-placement enumeration over BASELINE config 2: B = 1,000,000
random s2 boards x 7 current pieces with a second (hold) piece = 7,000,000 get_move_matrix
calls per GPU (weak scaling: every rank owns its own board shard, no collective on the data
path).  `value` = placements/s with inputs resident in HBM; `e2e` = the same metric through the
reference-facing C-ABI call with pinned HOST buffers (H2D + kernel + D2H inside the timed region).
One JSON line is printed by rank 0.  The workload is seeded, so the same arguments give the same inputs in every
run; --dump-outputs DIR writes what the last timed step returned (see dump_outputs) for comparing two builds.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

PROFILE_JSON = ("profiles/r2_movegen_rows.json",)   # tools/ncu_extract.py of the two-pass throughput form
SCALAR_PROFILE_JSON = "profiles/r2_movegen_thread.json"   # the one-thread-per-call kernel = the scalar restatement on the GPU
ALGO_BYTES_PER_CALL = 80 + 4 + 1448  # board + (cur, alt, pad) in, bit-packed (27,39,11) mask out (SURVEY §8d)
METRIC = "placements/sec (movegen)"
UNIT = "placements/s"


def load_ncu_profile():
    """Per-call ncu figures of the sweep's kernels from the tracked extraction of the .ncu-rep (tools/ncu_extract.py):
    movegen_rows_kernel (the dominant kernel: closure search) and movegen_solo_kernel in clean-up mode (the calls
    whose T-spin flags the closure search cannot decide).  None if no profile is committed."""
    for rel in PROFILE_JSON:
        path = os.path.join(ROOT, rel)
        if not os.path.exists(path):
            continue
        with open(path) as f:
            d = json.load(f)
        out = {"source": f"{rel} ({d['report']}, extracted at {d['extracted_at_commit']})", "kernels": {}}
        for l in d["launches"]:
            if not l.get("units"):
                continue
            m = {k: v["value"] for k, v in l["metrics"].items()}
            warp_inst = m.get("smsp__inst_executed.sum", 0.0)
            name = "movegen_rows_kernel" if "movegen_rows_kernel" in l["kernel"] else (
                "movegen_solo_kernel(clean-up)" if "movegen_solo_kernel" in l["kernel"] else None)
            if name is None:
                continue
            out["calls"] = l["units"]
            out["kernels"][name] = {
                "dram_bytes_per_call": l.get("dram_bytes_per_unit"),
                "issue_slots_busy_pct": m.get("smsp__issue_active.avg.pct_of_peak_sustained_active"),
                "alu_pipe_pct_of_peak": m.get("sm__inst_executed_pipe_alu.avg.pct_of_peak_sustained_active"),
                "threads_per_warp_instruction": m.get("smsp__thread_inst_executed_per_inst_executed.ratio"),
                "warp_instructions_per_call": warp_inst / l["units"] if warp_inst else None,
                "thread_instructions_per_call": l.get("thread_instructions_per_unit"),
                "registers_per_thread": m.get("launch__registers_per_thread"),
                "achieved_warps_per_sm_pct": m.get("sm__warps_active.avg.pct_of_peak_sustained_active"),
                "kernel_ms_under_ncu": m.get("gpu__time_duration.sum"),
                "no_instruction_stall_warps_per_issue": m.get("smsp__average_warps_issue_stalled_no_instruction_per_issue_active.ratio"),
                "barrier_stall_warps_per_issue": m.get("smsp__average_warps_issue_stalled_barrier_per_issue_active.ratio")}
        if "movegen_rows_kernel" in out["kernels"]:
            ks = out["kernels"]
            tot = sum(k["kernel_ms_under_ncu"] or 0.0 for k in ks.values())
            out["dominant_kernel_share_of_step"] = (ks["movegen_rows_kernel"]["kernel_ms_under_ncu"] or 0.0) / tot if tot else None
            out["dram_bytes_per_call"] = sum(k["dram_bytes_per_call"] or 0.0 for k in ks.values())
            out["thread_instructions_per_call"] = sum(k["thread_instructions_per_call"] or 0.0 for k in ks.values())
            return out
    return None


def load_scalar_profile():
    """Thread-level instruction count per call of the scalar restatement (movegen_thread_kernel: one thread runs the
    reference's algorithm for one call), the 'algorithmic int-ops' of SURVEY 8(d)."""
    path = os.path.join(ROOT, SCALAR_PROFILE_JSON)
    if not os.path.exists(path):
        return None
    with open(path) as f:
        d = json.load(f)
    for l in d["launches"]:
        if "movegen_thread_kernel" in l["kernel"] and l.get("thread_instructions_per_unit"):
            return {"source": f"{SCALAR_PROFILE_JSON} ({d['report']}, extracted at {d['extracted_at_commit']})",
                    "thread_instructions_per_call": l["thread_instructions_per_unit"], "calls": l["units"]}
    return None


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples nvidia-smi SM clocks / throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def make_workload(n_boards, rank):
    from tetris_reinforcement_learning_b200 import synth
    return synth.movegen_workload(n_boards, seed=synth.DEFAULT_SEED + 1000 * rank)


DUMP_CALLS = 8192   # sampled calls: 8192 x 1448 mask bytes x 4 B = 47.4 MB keeps a dump under 64 MB


def dump_outputs(out_dir, d_mask, d_n, d_st):
    """What the sweep returned to its caller for a fixed, seeded sample of the calls, as out_dir/<name>.npy:
    call_index (which calls), mask_bytes (the bit-packed (27,39,11) masks as their 1448 little-endian bytes),
    n_moves, and status_bits (the 32 TRL_ST_* bits of the status word, bit j in column j).  Values are small
    integers in float32, so a single flipped mask bit or status flag fails a comparison at any relative tolerance
    below 1e-3.  Two builds run with the same arguments dump the same calls and can be compared array by array."""
    import torch
    n = d_mask.shape[0]
    idx = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_CALLS), replace=False))
    sel = torch.from_numpy(idx).to(d_mask.device)
    mask = np.ascontiguousarray(d_mask[sel].cpu().numpy().astype("<u4"))
    status = np.ascontiguousarray(d_st[sel].cpu().numpy().astype("<u4"))
    arrays = {"call_index": idx.astype(np.float64),
              "mask_bytes": mask.view(np.uint8).astype(np.float32),
              "n_moves": d_n[sel].cpu().numpy().view(np.uint16).astype(np.float32),
              "status_bits": np.unpackbits(status.view(np.uint8).reshape(-1, 4), axis=1, bitorder="little").astype(np.float32)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def cpu_baseline(boards, cur, alt, target_s=12.0, device_masks=None, device_counts=None):
    """The oracle port (plain C, pthreads over all host cores) on a bounded sample of the workload.  The masks it
    computes are compared with the device's masks of the same calls (parity inside the bench run)."""
    from oracle import oracle
    cores = os.cpu_count() or 1
    probe = min(boards.shape[0], 7 * 2000)
    t0 = time.perf_counter()
    _, _, _, tot = oracle.movegen_batch(boards[:probe], cur[:probe], alt[:probe], n_threads=cores, want_masks=True)
    dt = time.perf_counter() - t0
    n = int(min(boards.shape[0], max(probe, probe * target_s / max(dt, 1e-3))))
    n -= n % 7
    t0 = time.perf_counter()
    want_masks, want_n, _, tot = oracle.movegen_batch(boards[:n], cur[:n], alt[:n], n_threads=cores, want_masks=True)
    dt = time.perf_counter() - t0
    out = {"value": tot / dt, "unit": UNIT, "cores": cores, "kind": "port",
           "sample": f"first {n // 7} boards x 7 pieces ({n} calls, {tot} placements) of the same workload, "
                     f"{dt:.1f} s, oracle/trl_oracle.c with {cores} pthreads",
           "python_reference_per_core": 3.7e4,
           "python_reference_note": "unmodified reference get_move_matrix measured in the build container (SURVEY §6); "
                                    "it cannot travel to the GPU box"}
    parity = None
    if device_masks is not None:
        mism = 0
        for lo in range(0, n, 200_000):
            hi = min(n, lo + 200_000)
            got = device_masks[lo:hi].cpu().numpy().view(np.uint32)
            mism += int((got != want_masks[lo:hi]).any(axis=1).sum())
        if device_counts is not None:
            mism += int((device_counts[:n].cpu().numpy().view(np.uint16) != want_n).sum())
        parity = {"parity_checked_calls": n, "mismatches": mism,
                  "how": "bit-packed (27,39,11) masks and counts of the device run vs oracle/trl_oracle.c on the same calls"}
    return out, parity


def cpu_selfplay_worker(seconds, index):
    """One process of the CPU self-play baseline: the oracle's restatement of ai.MCTS (oracle/mcts_oracle.py, C env
    step and placements) driving the repo's AlphaSame(10,16) on ONE CPU thread, BASELINE config 1 (MAX_ITER=160,
    playout-cap randomisation on).  Stands in for reference ai.py:1570-1699 play_game, which cannot travel to the box.
    Prints one JSON line."""
    import torch
    torch.set_num_threads(1)
    from oracle import features_oracle, mcts_oracle, oracle
    from tetris_reinforcement_learning_b200 import architectures as arch
    from tetris_reinforcement_learning_b200.config import Config
    oracle.lib()
    torch.manual_seed(0)
    mc = arch.AlphaSameConfig(blocks=10, filters=16)
    net = arch.AlphaSame(mc).eval()
    cfg = Config(visual=False, ruleset="s2", model="pytorch", model_config=mc, MAX_ITER=160, CPUCT=0.75, training=True)
    evals = [0]

    def evaluate(rec):
        grids, extras = features_oracle.encode(rec)
        with torch.no_grad():
            v, logits = net.forward_packed(torch.from_numpy(grids).reshape(2, 1, 40, 10), torch.from_numpy(extras)[None])
        evals[0] += 1
        return float(v.reshape(-1)[0]), torch.softmax(logits[0], dim=0).numpy().reshape(27, 39, 11)

    seed, gid = 20261018, 1000 + index
    games = oracle.game_setup(1, gid, seed)
    sims = plies = finished = 0
    search_no = 0
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        res = mcts_oracle.search(cfg, games, evaluate, mcts_oracle.SearchTape(seed, gid, search_no))
        sims += res["iterations"]
        plies += 1
        search_no += 1
        oracle.env_step(games, np.array([res["move"]], dtype=np.uint16), True, seed)
        if mcts_oracle.is_terminal(games[0]) or int(games[0]["rounds"]) >= 1000:
            finished += 1
            gid += 10000
            games = oracle.game_setup(1, gid, seed)
            search_no = 0
    dt = time.perf_counter() - t0
    print(json.dumps({"sims": sims, "plies": plies, "games_finished": finished, "evals": evals[0], "seconds": dt}), flush=True)


def cpu_selfplay_baseline(seconds=12.0, mean_plies=None):
    """P = host cores single-threaded worker processes of cpu_selfplay_worker; sims/s summed over the processes."""
    cores = os.cpu_count() or 1
    env = dict(os.environ, OMP_NUM_THREADS="1", MKL_NUM_THREADS="1", CUDA_VISIBLE_DEVICES="")
    t0 = time.perf_counter()
    procs = [subprocess.Popen([sys.executable, os.path.abspath(__file__), "--cpu-selfplay-worker", str(seconds), "--worker-index", str(i)],
                              stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, env=env) for i in range(cores)]
    outs = []
    for pr in procs:
        try:
            o, _ = pr.communicate(timeout=seconds * 6 + 180)
            outs.append(json.loads(o.strip().splitlines()[-1]))
        except Exception:
            pr.kill()
    wall = time.perf_counter() - t0
    if not outs:
        return {"unavailable": "no CPU self-play worker finished"}
    sims_per_s = sum(o["sims"] / o["seconds"] for o in outs)
    plies_per_s = sum(o["plies"] / o["seconds"] for o in outs)
    out = {"sims_per_sec": sims_per_s, "sims_per_sec_per_core": sims_per_s / len(outs), "cores": len(outs), "kind": "port",
           "moves_per_sec": plies_per_s, "games_finished": sum(o["games_finished"] for o in outs),
           "sample": f"{len(outs)} single-threaded processes x {seconds:.0f} s of self-play searches (oracle/mcts_oracle.py + "
                     "oracle/trl_oracle.c env step and placements + AlphaSame(10,16) fp32 on CPU, MAX_ITER=160 with playout-cap "
                     f"randomisation: 400 / 80 iterations per move); wall {wall:.0f} s incl. process start",
           "python_reference_per_core": {"sims_per_sec": 82, "games_per_hour": 29,
                                         "note": "unmodified reference play_game in the build container (BASELINE.md §2)"}}
    if mean_plies and mean_plies == mean_plies:
        out["games_per_hour"] = plies_per_s / mean_plies * 3600.0
        out["games_per_hour_note"] = (f"derived: measured moves/s / {mean_plies:.1f} plies per game (the mean game length the GPU "
                                      "engine measured in this run); a CPU game takes minutes, none completes inside the sample")
    return out


def run_selfplay(args, rank, world, local_rank):
    """BASELINE config 3 (4096 concurrent games per GPU, AlphaSame(10,16) random init bf16,
    MAX_ITER=160, Gamma root noise + FPU reduction): MCTS simulations/s and self-play games/hour.
    One engine step = one simulation in every game; the whole step is one CUDA graph."""
    import torch
    import torch.distributed as dist
    from tetris_reinforcement_learning_b200 import architectures as arch
    from tetris_reinforcement_learning_b200.config import Config
    from tetris_reinforcement_learning_b200.selfplay import SelfPlayEngine, best_evaluator, make_net_evaluator, shard_for_rank
    dev = torch.device("cuda", local_rank)
    torch.manual_seed(0)
    mc = arch.AlphaSameConfig(blocks=10, filters=16)
    net = arch.AlphaSame(mc).to(dev)
    ev = make_net_evaluator(net, torch.bfloat16) if args.net_path == "pytorch" else best_evaluator(net, torch.bfloat16)
    G = args.games
    sh = shard_for_rank(rank, world, G)

    def engine(max_iter, n_games=G, forced=None, evaluator=None, model_config=None, playout_cap=False, **kw):
        cfg = Config(visual=False, ruleset="s2", model="pytorch", model_config=model_config or mc, MAX_ITER=max_iter, CPUCT=0.75,
                     training=True, use_playout_cap_randomization=playout_cap, use_dirichlet_noise=True, FpuStrategy="reduction",
                     use_forced_playouts_and_policy_target_pruning=args.forced if forced is None else forced)
        return SelfPlayEngine(cfg, evaluator or ev, n_games, device=dev, seed=20261018, first_game_id=sh["first_game_id"],
                              game_id_stride=sh["game_id_stride"], feature_dtype=torch.bfloat16, **kw)

    def timed(eng, steps=None):
        steps = steps or args.selfplay_steps
        eng.step(12)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        eng.step(steps)
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        return e0.elapsed_time(e1)

    def extra_leg(name, steps, max_iter, forced=False, net_cfg=None, what="", playout_cap=False):
        """One more sims/s line: same games per GPU, another search setting or another network; max over ranks."""
        evaluator, flops_board, net_name = None, 37.2e6 / 2, "AlphaSame(blocks=10, filters=16)"
        if net_cfg is not None:
            torch.manual_seed(0)
            wide_net = arch.build_network(net_cfg).to(dev)
            evaluator = best_evaluator(wide_net, torch.bfloat16)
            f, b = net_cfg.filters, net_cfg.blocks
            stem = 25 if isinstance(net_cfg, arch.AlphaSameConfig) else 9
            flops_board = 2.0 * 400 * (stem * f + 2 * b * 9 * f * f)
            net_name = f"{type(wide_net).__name__}(blocks={b}, filters={f})"
        torch.cuda.reset_peak_memory_stats(dev)
        mem0 = torch.cuda.memory_allocated(dev)
        e = engine(max_iter, forced=forced, evaluator=evaluator, model_config=net_cfg, playout_cap=playout_cap)
        fused = e.cached_eval is not None
        arena = {"node_cap_per_game": e.node_cap, "state_cap_per_game": e.state_cap,
                 "tree_bytes": int(sum(e.t[k].numel() * e.t[k].element_size() for k in ("prior", "value_sum", "visits", "parent", "slot", "move")))}
        t = timed(e, steps)
        arena["hbm_peak_bytes_engine"] = int(torch.cuda.max_memory_allocated(dev) - mem0)
        st = e.get_ctl()["status"]
        if evaluator is not None and hasattr(evaluator, "trunk"):
            evaluator.trunk.check()
        del e
        torch.cuda.empty_cache()
        tt = torch.tensor([t], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t = float(tt[0])
        v = G * world * steps / (t * 1e-3)
        return {"what": what, "value": v, "unit": "sims/s", "games_per_gpu": G, "n_gpus": world, "steps": steps, "max_iter": max_iter,
                "ms_per_step": t / steps, "net": net_name + " bf16, random init", "fused_trunk": fused,
                "forced_playouts_and_pruning": bool(forced), "playout_cap_randomization": bool(playout_cap),
                "status_nonzero_rank0": int((st != 0).sum()), "memory": arena,
                "roofline": {"bound": "tensor", "unit": "TFLOP/s", "peak": load_tensor_peak(),
                             "achieved": v / world * flops_board / 1e12, "frac": v / world * flops_board / 1e12 / load_tensor_peak(),
                             "flops_counted": "trunk convolutions of ONE board per simulation (trunk-feature reuse); heads and policy "
                                              "GEMM not counted"}}

    eng = engine(160)
    eng_flags = eng
    reuse = eng.cached_eval is not None
    ms = timed(eng)
    samples, _ = eng.drain()
    ctl = eng.get_ctl()
    # own kernels per step (the cuBLAS policy GEMM is not counted): with the cached evaluator gate, enumeration,
    # trunk, heads, expand+select+encode; else select, enumeration, encode, expand (+ the PyTorch net)
    launches_per_step = 5 if reuse else 4
    ms_both = None
    if reuse and not args.no_game_length:
        # the same step with BOTH boards of every leaf through the trunk (the reference's amount of work)
        del eng
        torch.cuda.empty_cache()
        eng2 = engine(160, reuse_trunk_features=False, reuse_sibling_placements=False)
        ms_both = timed(eng2)
        del eng2
        torch.cuda.empty_cache()
    # self-play games/hour, MEASURED: the same engine keeps playing complete games at MAX_ITER=160 (finished
    # games restart in place); after one mean game length of warm-up, count the games that END inside a timed
    # window of about two mean game lengths.  (The mean game length itself comes from the ends seen.)
    games_done, game_ms, mean_plies, plies = 0, 0.0, float("nan"), []
    n_samples_drained, d2h_bytes, game_status_nonzero, game_status_or = 0, 0, 0, 0
    if not args.no_game_length:
        # End to end: the sample and game-end records are drained to the host every `chunk` steps INSIDE the timed
        # window (device sync + D2H of the ring buffers, as make_training_set does), so no record is dropped.
        eng = engine(160)
        chunk = 448                       # at most 3 searches per game in 448 steps: 12 288 records < the 16 384-record ring
        warm_steps = int(args.game_warm_steps)
        for _ in range(max(1, warm_steps // chunk)):
            eng.step(chunk)
            eng.drain()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ends_all, n_samples_drained, d2h_bytes = [], 0, 0
        n_chunks = max(1, int(args.game_steps) // chunk)
        for _ in range(n_chunks):
            eng.step(chunk)
            smp, ends = eng.drain(copy=False)     # views into pinned staging; a consumer would serialise them here
            ends_all.append(ends.copy())
            n_samples_drained += len(smp)
            d2h_bytes += smp.nbytes + ends.nbytes
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        game_ms = e0.elapsed_time(e1)
        args.game_steps = n_chunks * chunk
        ends = np.concatenate(ends_all) if ends_all else np.zeros(0)
        games_done = len(ends)
        st_all = eng.get_ctl()["status"]
        game_status_nonzero = int((st_all != 0).sum())
        game_status_or = int(np.bitwise_or.reduce(st_all)) if len(st_all) else 0
        plies = [int(e["plies"]) for e in ends]
        mean_plies = float(np.mean(plies)) if plies else float("nan")
        del eng
        torch.cuda.empty_cache()
    extra = {}
    if not args.no_config4:
        extra["config4_forced_playouts"] = extra_leg(
            "config4", args.selfplay_steps, 160, forced=True,
            what="BASELINE config 4: the config-3 engine with forced playouts + policy-target pruning, same games per GPU, every GPU "
                 "count the driver runs (weak scaling)")
    if not args.no_wide:
        extra["config5_net"] = extra_leg(
            "config5", 48, 800, net_cfg=arch.AlphaSameConfig(blocks=20, filters=64), playout_cap=True,
            what="BASELINE config 5's network and search budget in the self-play engine: AlphaSame(20, 64), MAX_ITER=800 with playout-cap "
                 "randomisation (searches of 2000 / 400 iterations: the node arena is sized for 2000), through csrc/trunk_wide.cu "
                 "(through PyTorch / cuDNN the same step took 51 ms in round 1)")
        extra["config_default_net"] = extra_leg(
            "default", 96, 400, net_cfg=arch.AuxBaseResNetConfig(),
            what="the reference's Config default (ai.py:83): AuxBaseResNet(8, 32), MAX_ITER=400, through csrc/trunk_wide.cu "
                 "(PyTorch / cuDNN: 17 ms per step in round 1)")
    stats = torch.tensor([ms, float(G * args.selfplay_steps), float(len(samples)), ms_both or 0.0, game_ms, float(games_done)],
                         dtype=torch.float64, device=dev)
    if world > 1:
        mx = stats.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = stats.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        ms, sims, nsamples, ms_both = float(mx[0]), float(sm[1]), float(sm[2]), (float(mx[3]) or None)
        game_ms, games_done = float(mx[4]), float(sm[5])
    else:
        sims, nsamples = float(stats[1]), float(stats[2])
    sims_per_s = sims / (ms * 1e-3)
    flops_per_eval = 86.5e6  # AlphaSame(10,16), both grids (SURVEY §8d)
    flops_done = (86.5e6 - 37.2e6) if reuse else 86.5e6   # with reuse one board per leaf goes through the trunk
    return {
        "_launches": launches_per_step * args.selfplay_steps,
        **extra,
        "mcts_sims_per_sec": {
            "value": sims_per_s, "unit": "sims/s", "games_per_gpu": G, "n_gpus": world, "steps": args.selfplay_steps,
            "ms_per_step": ms / args.selfplay_steps, "max_iter": 160, "net": "AlphaSame(blocks=10, filters=16) bf16, " + ("PyTorch/cuDNN" if args.net_path == "pytorch" else
                                                               "row-Toeplitz tcgen05 trunk + fused heads kernel + cuBLAS policy GEMM") + ", CUDA graph (4 steps per launch)",
            "step": "enumeration of the leaves without a cached sibling list (compacted, queued behind the trunk on a forked stream) || "
                    "trunk -> heads -> policy GEMM -> expand + select + feature encoding of the next leaves (one kernel)",
            "trunk_feature_reuse": reuse, "sibling_placement_reuse": bool(getattr(eng_flags, "reuse_sibling_placements", False)),
            "trunk_feature_reuse_note": "exact: a move changes only the mover's board, so per simulation one board goes through the "
                                        "trunk and the other board's features are the parent state's (bit-identical searches, "
                                        "tests/test_gpu_trunk.py::test_trunk_feature_reuse_is_exact)",
            "value_without_reuse": (sims / (ms_both * 1e-3)) if ms_both else None,
            "ms_per_step_without_reuse": (ms_both / args.selfplay_steps) if ms_both else None,
            "without_reuse_note": "both boards of every leaf through the trunk and legal placements enumerated for every leaf "
                                  "(the amount of work the reference does per simulation)",
            "searches_finished": nsamples, "status_nonzero": int((ctl["status"] != 0).sum()),
            "roofline": {"bound": "tensor", "achieved": sims_per_s / world * flops_done / 1e12,
                         "peak": load_tensor_peak(), "unit": "TFLOP/s",
                         "frac": sims_per_s / world * flops_done / 1e12 / load_tensor_peak(),
                         "flops_per_simulation_executed": flops_done, "flops_per_simulation_reference": flops_per_eval,
                         "note": "executed FLOPs (with reuse: one trunk pass + heads per simulation); the trunk is bound by the "
                                 "128 B/clk shared-memory operand fetch of N=48 MMAs, not by tensor math (DESIGN.md)"},
        },
        "selfplay_games_per_hour": {
            "value": (games_done / (game_ms * 1e-3) * 3600.0) if game_ms > 0 else None,
            "unit": "games/h", "measured": True, "games_finished_in_window": games_done,
            "window_ms": game_ms, "window_steps": int(args.game_steps), "warmup_steps": int(args.game_warm_steps),
            "mean_plies_per_game": mean_plies,
            "how": "complete self-play games (MAX_ITER=160 simulations per move, Gamma root noise, temperature move choice, "
                   "finished games restart in place) that ended inside the timed window, all GPUs; the sample and game-end "
                   "records are drained to the host every 448 steps inside the window (rank 0's counts below)",
            "samples_drained_rank0": n_samples_drained, "d2h_bytes_rank0": d2h_bytes, "status_nonzero_rank0": game_status_nonzero,
            "status_bits_rank0": game_status_or,   # TRL_ST_* (include/trl.h) OR-ed over the games
        },
    }


def load_tensor_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["bf16_tflops_sustained"])
    return 1400.0


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path = the oracle port
    (the reference is pure Python and cannot travel to the GPU box), all host threads."""
    if rank != 0:
        return
    from oracle import oracle
    oracle.build()
    cores = os.cpu_count() or 1
    n_boards = args.boards
    sample_boards = max(1000, min(n_boards, args.ref_sample_boards))
    boards, cur, alt = make_workload(sample_boards, 0)
    times, tot = [], 0
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        _, _, _, tot = oracle.movegen_batch(boards, cur, alt, n_threads=cores, want_masks=True)
        if it >= args.warmup:
            times.append(time.perf_counter() - t0)
    dt = float(np.mean(times))
    value = tot / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u16", "data": "synthetic",
        "config": {"workload": f"BASELINE config 2 movegen sweep: {n_boards} random s2 boards x 7 pieces with hold "
                               f"(each CPU step = a bounded sample of {sample_boards} boards x 7)",
                   "boards": n_boards, "calls_per_step": int(boards.shape[0])},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{sample_boards} boards x 7 pieces per step, oracle/trl_oracle.c, {cores} pthreads"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from tetris_reinforcement_learning_b200 import _native, move_generation
    from tetris_reinforcement_learning_b200.const import MASK_WORDS

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    L = _native.lib()

    boards, cur, alt = make_workload(args.boards, rank)
    n = boards.shape[0]
    d_boards = torch.from_numpy(boards.view(np.int16)).to(dev)
    d_cur, d_alt = torch.from_numpy(cur).to(dev), torch.from_numpy(alt).to(dev)
    d_mask = torch.empty((n, MASK_WORDS), dtype=torch.int32, device=dev)
    d_n = torch.empty(n, dtype=torch.int16, device=dev)
    d_st = torch.empty(n, dtype=torch.int32, device=dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        move_generation.movegen_device(d_boards, d_cur, d_alt, d_mask, None, d_n, d_st)

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    placements = int(d_n.to(torch.int64).sum().item())
    bad_status = int((d_st != 0).sum().item())

    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    ev[0].record()
    for k in range(args.steps):
        step()
        ev[k + 1].record()
    barrier()
    clocks = sampler.stop()
    kernel_ms = [ev[k].elapsed_time(ev[k + 1]) for k in range(args.steps)]
    total_ms = ev[0].elapsed_time(ev[args.steps])
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, d_mask, d_n, d_st)

    # ---- e2e: the reference-facing host call with pinned host buffers ----
    h_boards = torch.from_numpy(boards.view(np.int16)).pin_memory()
    h_cur, h_alt = torch.from_numpy(cur).pin_memory(), torch.from_numpy(alt).pin_memory()
    h_n = torch.empty(n, dtype=torch.int16).pin_memory()
    h_st = torch.empty(n, dtype=torch.int32).pin_memory()
    # secondary leg: the dense encoding (bit-packed (27,39,11) masks).  It is bound by PCIe / host memory, not by
    # the GPU, so it runs on a bounded prefix of the workload (<= 1.4 M calls = 2 GB of pinned masks per rank).
    n_mask = min(n, 1_400_000)
    h_mask = torch.empty((n_mask, MASK_WORDS), dtype=torch.int32).pin_memory()

    def e2e_step():
        rc = L.trl_movegen_host(h_boards.data_ptr(), h_cur.data_ptr(), h_alt.data_ptr(), n_mask, h_mask.data_ptr(),
                                None, 0, h_n.data_ptr(), h_st.data_ptr())
        _native.check(rc, "trl_movegen_host")

    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    d_n_host = d_n.cpu().numpy()
    e2e_ok = bool(np.array_equal(h_n.numpy()[:n_mask], d_n_host[:n_mask]))
    placements_mask = int(d_n_host[:n_mask].astype(np.int64).sum())
    h2d = n * (80 + 2)
    d2h = n_mask * (MASK_WORDS * 4 + 2 + 4)

    # the same enumeration returned as COMPACT ascending move lists (np.argwhere order, what get_move_list
    # consumes, ai.py:1016-1024): 2 B per placement + 14 B per call cross PCIe instead of 1448 B of mask
    del h_mask
    cap = int(placements * 1.02) + 4096
    h_moves = torch.empty(cap, dtype=torch.int16).pin_memory()
    h_off = torch.empty(n, dtype=torch.int64).pin_memory()
    h_n2 = torch.empty(n, dtype=torch.int16).pin_memory()
    import ctypes
    tot = ctypes.c_uint64(0)

    def e2e_list_step():
        rc = L.trl_movegen_host_compact(h_boards.data_ptr(), h_cur.data_ptr(), h_alt.data_ptr(), n, h_moves.data_ptr(), cap,
                                        h_off.data_ptr(), h_n2.data_ptr(), h_st.data_ptr(), ctypes.addressof(tot))
        _native.check(rc, "trl_movegen_host_compact")

    e2e_list_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_list_step()
    torch.cuda.synchronize()
    e2e_list_s = (time.perf_counter() - t0) / e2e_steps
    e2e_list_ok = bool(np.array_equal(h_n2.numpy(), d_n_host)) and int(tot.value) == placements \
        and not bool((h_st.numpy() != 0).any())
    d2h_list = placements * 2 + n * (8 + 2 + 4)
    del h_moves

    cpu_line, parity = None, None
    if world == 1 and not args.no_cpu_baseline:
        from oracle import oracle
        oracle.build()
        step()                      # the device masks of the timed configuration, compared call by call below
        torch.cuda.synchronize()
        cpu_line, parity = cpu_baseline(boards, cur, alt, device_masks=d_mask, device_counts=d_n)
    # free the sweep's buffers before the self-play leg
    del d_mask
    torch.cuda.empty_cache()
    also = None
    if not args.no_selfplay:
        also = run_selfplay(args, rank, world, local_rank)

    # ---- reduce over ranks: max time, summed work ----
    stats = torch.tensor([total_ms, e2e_s, float(placements), float(np.mean(kernel_ms)), e2e_list_s, float(placements_mask)],
                         dtype=torch.float64, device=dev)
    if world > 1:
        mx = stats.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = stats.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        total_ms, e2e_s, kern_ms, e2e_list_s = float(mx[0]), float(mx[1]), float(mx[3]), float(mx[4])
        placements_all, placements_mask_all = float(sm[2]), float(sm[5])
    else:
        kern_ms, placements_all, placements_mask_all = float(np.mean(kernel_ms)), float(placements), float(placements_mask)

    if rank != 0:
        return
    peak, peak_src = load_peaks()
    achieved = ALGO_BYTES_PER_CALL * n / (kern_ms * 1e-3) / 1e9
    value = placements_all * args.steps / (total_ms * 1e-3)
    prof, scalar = load_ncu_profile(), load_scalar_profile()
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": int(prof["dram_bytes_per_call"] * n) if prof and prof.get("dram_bytes_per_call") else None,
                "traffic_unit": "bytes per launch",
                "traffic_source": (f"ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per call of a {int(prof['calls'])}-call "
                                   f"launch, scaled to this launch's call count; {prof['source']}") if prof else None,
                "peak_source": peak_src, "kernel": "movegen_rows_kernel",
                "algorithmic_bytes_per_call": ALGO_BYTES_PER_CALL, "kernel_ms": kern_ms,
                "kernel_ms_how": "CUDA events around one sweep = movegen_rows_kernel + movegen_solo_kernel in clean-up mode (two launches "
                                 "inside the library call); `achieved` divides by this whole time, the dominant kernel's share is ncu.dominant_kernel_share_of_step",
                "note": "integer-issue bound, not HBM bound (SURVEY §8d): the DRAM traffic is at the algorithmic minimum; "
                        "what binds is the issue rate (85 % of the issue slots busy in the dominant kernel), see int_ops",
                "ncu": prof}
    # SURVEY 8(d): roofline on integer issue.  per_call = thread-level instructions of the SCALAR restatement of the
    # algorithm (one thread per call, ncu); achieved = per_call x calls/s; peak = 148 SMs x 4 schedulers x 32 lanes x f_SM
    f_sm = (clocks.get("sm_mhz") or clocks.get("sm_max_mhz") or 1965.0) * 1e6
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    peak_ops = sms * 4 * 32 * f_sm
    calls_per_s = n / (kern_ms * 1e-3)
    if scalar:
        roofline["int_ops"] = {
            "per_call": scalar["thread_instructions_per_call"], "achieved": scalar["thread_instructions_per_call"] * calls_per_s,
            "peak": peak_ops, "unit": "thread instructions/s", "frac": scalar["thread_instructions_per_call"] * calls_per_s / peak_ops,
            "peak_how": f"{sms} SMs x 4 issue slots x 32 lanes x {f_sm / 1e6:.0f} MHz (SM clock sampled during the timed region)",
            "per_call_source": scalar["source"],
            "executed_per_call": prof.get("thread_instructions_per_call") if prof else None,
            "executed_frac": (prof["thread_instructions_per_call"] * calls_per_s / peak_ops) if prof and prof.get("thread_instructions_per_call") else None,
            "note": "per_call = what the one-thread-per-call kernel (the reference's algorithm, scalar) executes; executed_per_call = "
                    "what the two kernels of the sweep execute (row-parallel bit planes do redundant lane work); frac is useful work / peak"}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u16", "data": "synthetic",
        "config": {"workload": f"BASELINE config 2 movegen sweep: {args.boards} random s2 boards x 7 pieces with hold per GPU "
                               "(3 board families, seed 20261018), ruleset s2, algo convolutional",
                   "boards_per_gpu": args.boards, "calls_per_step_per_gpu": n,
                   "placements_per_step_per_gpu": placements, "l2": "inputs+outputs (>10 GB/step) exceed the 126 MB L2",
                   "status_nonzero": bad_status},
        "roofline": roofline,
        "e2e": {"value": placements_all / e2e_list_s, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h_list,
                "steps": e2e_steps, "matches_device_run": e2e_list_ok,
                "api": "trl_movegen_host_compact: pinned host buffers in, ascending uint16 move lists (np.argwhere order, "
                       "ai.py:1016-1024) packed back to back + offsets/counts/status out; H2D + kernel + D2H inside the timed region",
                "as_bit_packed_masks": {"value": placements_mask_all / e2e_s, "unit": UNIT, "calls_per_step_per_gpu": n_mask,
                                        "h2d_bytes_per_step": n_mask * (80 + 2), "d2h_bytes_per_step": d2h, "matches_device_run": e2e_ok,
                                        "api": "trl_movegen_host: the same enumeration returned as bit-packed (27,39,11) masks "
                                               "(1448 B per call): bound by PCIe / host memory, does not scale with the GPU count"}},
        "gpu_launches": 2 * args.steps,   # movegen_rows_kernel + movegen_solo_kernel (clean-up) per sweep
        "clocks": clocks,
    }
    if cpu_line is not None:
        line["cpu_baseline"] = cpu_line
        line["config"].update(parity or {})
        if also is not None and not args.no_cpu_selfplay:
            mp = also["selfplay_games_per_hour"].get("mean_plies_per_game")
            line["cpu_baseline"]["selfplay"] = cpu_selfplay_baseline(args.cpu_selfplay_seconds, mp)
    if also is not None:
        line["also"] = also
        line["gpu_launches"] += also.pop("_launches", 0)
    emit(line)


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line of the contract, on the process's real stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    # Libraries chat on stdout (e.g. "NCCL version ..." when the box exports NCCL_DEBUG=VERSION): keep fd 1 for
    # the JSON line only and send everything else to stderr.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--boards", type=int, default=1_000_000, help="boards per GPU (x7 pieces = calls per step)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--ref-sample-boards", type=int, default=40_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-selfplay", action="store_true", help="skip the sims/s + games/h leg")
    ap.add_argument("--games", type=int, default=4096, help="concurrent self-play games per GPU")
    ap.add_argument("--selfplay-steps", type=int, default=320)
    ap.add_argument("--no-game-length", action="store_true", help="skip the games/h run and the no-reuse run (profiling)")
    ap.add_argument("--game-warm-steps", type=int, default=9000, help="steps before the games/h window (about one game length)")
    ap.add_argument("--game-steps", type=int, default=18000, help="steps of the games/h window (about two game lengths)")
    ap.add_argument("--net-path", default="fused", choices=["fused", "pytorch"])
    ap.add_argument("--forced", action="store_true", help="forced playouts + policy-target pruning in the main self-play leg")
    ap.add_argument("--no-config4", action="store_true", help="skip the config-4 leg (forced playouts + pruning)")
    ap.add_argument("--no-wide", action="store_true", help="skip the wide-net legs (config 5 net, Config-default net)")
    ap.add_argument("--no-cpu-selfplay", action="store_true")
    ap.add_argument("--cpu-selfplay-seconds", type=float, default=12.0)
    ap.add_argument("--cpu-selfplay-worker", type=float, default=0.0, help=argparse.SUPPRESS)
    ap.add_argument("--worker-index", type=int, default=0, help=argparse.SUPPRESS)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write a seeded sample of the last sweep's outputs (rank 0's shard) "
                         "as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.cpu_selfplay_worker > 0:
        os.dup2(_REAL_STDOUT, 1)
        cpu_selfplay_worker(args.cpu_selfplay_worker, args.worker_index)
        return
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
