"""Per-kernel time of the config-2 movegen sweep and the work that reaches each pass.

    python tools/movegen_passes.py [--boards 1000000] [--sweeps 10] [--out DIR] [--per-piece]

Runs the sweep bench.py times (mask output, device-resident inputs) under torch.profiler with CUDA activities and
prints every kernel's time per sweep, then the pass counts of one sweep outside the profiler: calls whose T search
pass 1 deferred, calls the T order analysis left undecided (they take the exact T search), and calls on the legacy
route (movegen_solo_kernel in clean-up mode).  A library without the pass-count getter prints only the kernel times.

--per-piece instead times the sweep's boards once per piece type t with cur = alt = t, so that every call is one search
of that piece, with CUDA events around `--sweeps` sweeps after three warm-up sweeps, and prints ms per sweep per piece.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tetris_reinforcement_learning_b200 import _native, move_generation, synth  # noqa: E402
from tetris_reinforcement_learning_b200.const import MASK_WORDS  # noqa: E402


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,driver_version", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:   # the timings are still worth printing
        return f"unknown ({e})"


def pass_counts(L):
    """(deferred, undecided, legacy) of the last launch of the pass form, or None for a library without the getter."""
    try:
        fn = L.trl_debug_movegen_pass_counts
    except AttributeError:
        return None
    c = (ctypes.c_uint32 * 3)()
    _native.check(fn(c), "trl_debug_movegen_pass_counts")
    return tuple(int(v) for v in c)


def per_piece(args, d_b, d_mask, d_n, d_st):
    from tetris_reinforcement_learning_b200.const import MINOS
    n = d_b.shape[0]
    res = {"card": card(), "calls": n, "sweeps": args.sweeps, "ms_per_sweep": {}}
    print(f"card: {res['card']}")
    print(f"config-2 boards, {n} calls with cur = alt = t (one search per call), {args.sweeps} sweeps, CUDA events")
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for t in range(7):
        d_t = torch.full((n,), t, dtype=torch.uint8, device=d_b.device)
        for _ in range(3):
            move_generation.movegen_device(d_b, d_t, d_t, d_mask, None, d_n, d_st)
        start.record()
        for _ in range(args.sweeps):
            move_generation.movegen_device(d_b, d_t, d_t, d_mask, None, d_n, d_st)
        stop.record()
        stop.synchronize()
        ms = start.elapsed_time(stop) / args.sweeps
        res["ms_per_sweep"][MINOS[t]] = ms
        print(f"  {MINOS[t]}  {ms:9.3f} ms/sweep  {1e6 * ms / n:7.3f} ns/search")
    print(f"  sum of the seven: {sum(res['ms_per_sweep'].values()):.3f} ms")
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "movegen_per_piece.json"), "w") as f:
            json.dump(res, f, indent=1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--boards", type=int, default=1_000_000)
    ap.add_argument("--sweeps", type=int, default=10)
    ap.add_argument("--out", default=None, help="also write the result as JSON into this directory")
    ap.add_argument("--per-piece", action="store_true", help="time one search per call, per piece type (cur = alt = t)")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "movegen_passes.py needs a CUDA device"
    L = _native.lib()
    dev = torch.device("cuda:0")
    boards, cur, alt = synth.movegen_workload(args.boards)
    n = boards.shape[0]
    d_b = torch.from_numpy(boards.view(np.int16)).to(dev)
    d_c, d_a = torch.from_numpy(cur).to(dev), torch.from_numpy(alt).to(dev)
    d_mask = torch.empty((n, MASK_WORDS), dtype=torch.int32, device=dev)
    d_n = torch.empty(n, dtype=torch.int16, device=dev)
    d_st = torch.empty(n, dtype=torch.int32, device=dev)

    def sweep():
        move_generation.movegen_device(d_b, d_c, d_a, d_mask, None, d_n, d_st)

    if args.per_piece:
        per_piece(args, d_b, d_mask, d_n, d_st)
        return

    for _ in range(3):
        sweep()
    torch.cuda.synchronize()
    counts = pass_counts(L)

    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.sweeps):
            sweep()
        torch.cuda.synchronize()
    per_kernel = {}
    for e in prof.events():
        if e.device_type.name != "CUDA":
            continue
        k = per_kernel.setdefault(e.name, [0.0, 0])
        k[0] += e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
        k[1] += 1
    total = sum(v[0] for v in per_kernel.values())
    res = {"card": card(), "calls": n, "sweeps": args.sweeps, "kernels": {}, "pass_counts": None}
    print(f"card: {res['card']}")
    print(f"config-2 sweep, {n} calls, {args.sweeps} sweeps under torch.profiler (CUDA activities)")
    for name, (us, cnt) in sorted(per_kernel.items(), key=lambda kv: -kv[1][0]):
        short = name.replace("(anonymous namespace)::", "").removeprefix("void ").split("(")[0]
        res["kernels"][short] = {"ms_per_sweep": us / args.sweeps / 1e3, "launches_per_sweep": cnt / args.sweeps}
        print(f"  {us / args.sweeps / 1e3:9.3f} ms/sweep  {100.0 * us / max(total, 1e-9):5.1f} %  "
              f"{cnt / args.sweeps:4.1f} launches/sweep  {short}")
    print(f"  {total / args.sweeps / 1e3:9.3f} ms/sweep in all")
    if counts is None:
        print("pass counts: not available in this library")
    else:
        d, u, g = counts
        res["pass_counts"] = {"deferred": d, "undecided": u, "legacy": g}
        print(f"pass counts: deferred {d} ({100.0 * d / n:.3f} % of the calls), undecided {u} ({100.0 * u / n:.3f} %), "
              f"legacy {g}")
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "movegen_passes.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
