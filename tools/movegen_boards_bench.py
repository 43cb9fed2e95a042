"""End-to-end A/B of the two compact host movegen entry points on BASELINE config 2 (every board x 7 pieces):

    compact        trl_movegen_host_compact: every call uploads its board; 2 B per placement + 14 B per call come back
    boards         trl_movegen_host_boards: each board is uploaded once; byte codes (about 1 B per placement) come back;
                   the encoder reads the sweep's compact move lists (the default)
    boards_masks   the same entry point with the encoder reading the sweep's bit-packed masks instead

All host buffers are pinned.  The legs alternate in one process, --rounds x --steps timed steps each after warm-up.
Reports placements/s end to end, H2D / D2H bytes per step (from the counts), escapes per call, the host decode time of
the byte codes (decode_move_codes, measured apart from the transfer) and the card name and power limit.

    python tools/movegen_boards_bench.py [--boards 1000000] [--rounds 3] [--steps 3] [--out results.json]
    torchrun --nproc_per_node 8 tools/movegen_boards_bench.py      # one process per GPU: the scaling of both paths
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tetris_reinforcement_learning_b200 import _native, synth  # noqa: E402
from tetris_reinforcement_learning_b200.move_generation import decode_move_codes  # noqa: E402

CHUNK = 1 << 17   # calls per chunk of the host entry points (TRL_HOST_CHUNK_LOG2)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out
    except Exception as e:  # noqa: BLE001
        return [f"nvidia-smi unavailable: {e}"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--boards", type=int, default=1_000_000)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=synth.DEFAULT_SEED)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("gloo")
    L = _native.lib()
    L.trl_debug_movegen_codes_source.argtypes = [ctypes.c_int]
    L.trl_debug_movegen_codes_source.restype = None

    # ---- workload: config 2, each rank its own boards ----
    nb = args.boards
    boards = synth.random_boards(nb, seed=args.seed + rank)
    i = np.repeat(np.arange(nb), 7)
    k = np.tile(np.arange(7), nb)
    cur = k.astype(np.uint8)
    alt = ((k + 1 + i % 6) % 7).astype(np.uint8)
    n = cur.size

    def pinned(shape, dtype):
        tdt = {np.uint8: torch.uint8, np.uint16: torch.int16, np.uint32: torch.int32, np.uint64: torch.int64}[dtype]
        return torch.empty(shape, dtype=tdt).pin_memory().numpy().view(dtype)

    h_boards = pinned((nb, 40), np.uint16); h_boards[:] = boards
    h_exp = pinned((n, 40), np.uint16); h_exp[:] = np.repeat(boards, 7, axis=0)
    h_idx = pinned(n, np.uint32); h_idx[:] = i
    h_cur = pinned(n, np.uint8); h_cur[:] = cur
    h_alt = pinned(n, np.uint8); h_alt[:] = alt
    # compact outputs
    cap = 160 * n
    c_moves = pinned(cap, np.uint16)
    c_off = pinned(n, np.uint64)
    c_n = pinned(n, np.uint16)
    c_st = pinned(n, np.uint32)
    c_tot = ctypes.c_uint64(0)
    # byte-code outputs
    b_codes = pinned(160 * n, np.uint8)
    b_esc = pinned(45 * n, np.uint16)
    b_n = pinned(n, np.uint16)
    b_fi = pinned(n, np.uint32)
    b_fs = pinned(n, np.uint32)
    b_tot = (ctypes.c_uint64 * 3)()
    ta = ctypes.addressof(b_tot)
    p = lambda a: a.ctypes.data  # noqa: E731

    def compact():
        rc = L.trl_movegen_host_compact(p(h_exp), p(h_cur), p(h_alt), n, p(c_moves), cap, p(c_off), p(c_n), p(c_st),
                                        ctypes.addressof(c_tot))
        _native.check(rc, "trl_movegen_host_compact")

    def codes(source):
        def step():
            L.trl_debug_movegen_codes_source(source)
            rc = L.trl_movegen_host_boards(p(h_boards), nb, p(h_idx), p(h_cur), p(h_alt), n, p(b_codes), b_codes.size,
                                           p(b_esc), b_esc.size, p(b_n), p(b_fi), p(b_fs), n, ta, ta + 8, ta + 16)
            L.trl_debug_movegen_codes_source(0)
            _native.check(rc, "trl_movegen_host_boards")
        return step

    legs = {"compact": compact, "boards": codes(0), "boards_masks": codes(1)}
    for f in legs.values():   # warm-up: workspace, streams, pinned totals, kernel attributes
        f(); f()
    times = {name: [] for name in legs}
    for _ in range(args.rounds):
        for name, f in legs.items():
            for _ in range(args.steps):
                if dist:
                    dist.barrier()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                f()
                dt = time.perf_counter() - t0
                if dist:
                    t = torch.tensor([dt], dtype=torch.float64)
                    dist.all_reduce(t, op=dist.ReduceOp.MAX)
                    dt = float(t[0])
                times[name].append(dt)

    # ---- outputs of the last steps: agreement and counts ----
    compact()
    codes(0)()
    n_codes, n_esc, n_flag = (int(v) for v in b_tot)
    placements = int(c_tot.value)
    t0 = time.perf_counter()
    moves, offsets = decode_move_codes(b_codes[:n_codes], b_esc[:n_esc], b_n)
    decode_s = time.perf_counter() - t0
    nm = c_n.astype(np.int64)
    pos = np.repeat(c_off.astype(np.int64) - offsets.astype(np.int64), nm) + np.arange(placements)
    agree = bool(np.array_equal(b_n, c_n) and n_codes == placements and np.array_equal(c_moves[pos], moves)
                 and np.array_equal(b_fi[:n_flag], np.flatnonzero(c_st)))
    n_chunks = (n + CHUNK - 1) // CHUNK
    bytes_ = {
        # boards, cur, alt in; lists, offsets, counts, status and one total per chunk out
        "compact": {"h2d": n * (80 + 2), "d2h": 2 * placements + n * (8 + 2 + 4) + 8 * n_chunks},
        # each board once, then board index, cur, alt; codes, escapes, counts, flagged pairs and 16 B of totals per chunk
        "boards": {"h2d": nb * 80 + n * (4 + 2),
                   "d2h": n_codes + 2 * n_esc + 2 * n + 8 * n_flag + 16 * n_chunks},
    }
    bytes_["boards_masks"] = bytes_["boards"]

    if world > 1:
        t = torch.tensor([placements, n_esc, n, decode_s, float(agree)], dtype=torch.float64)
        s = t.clone(); dist.all_reduce(s)
        mn = t.clone(); dist.all_reduce(mn, op=dist.ReduceOp.MIN)
        placements_all, esc_all, n_all = float(s[0]), float(s[1]), float(s[2])
        agree = bool(mn[4] > 0)
    else:
        placements_all, esc_all, n_all = float(placements), float(n_esc), float(n)
    if rank != 0:
        dist.destroy_process_group()
        return
    res = {
        "card": card(), "world": world, "boards_per_rank": nb, "calls_per_rank": n, "placements_per_rank": placements,
        "rounds": args.rounds, "steps": args.steps,
        "escapes_per_call": esc_all / n_all, "flagged_per_rank": n_flag,
        "host_decode_ms_per_rank": decode_s * 1e3, "outputs_agree": agree, "legs": {},
    }
    for name, ts in times.items():
        per_round = [float(np.mean(ts[r * args.steps:(r + 1) * args.steps])) for r in range(args.rounds)]
        res["legs"][name] = {
            "ms_per_step_by_round": [t * 1e3 for t in per_round],
            "placements_per_s": placements_all / float(np.mean(ts)),
            "placements_per_s_by_round": [placements_all / t for t in per_round],
            "h2d_bytes_per_step_per_rank": bytes_[name]["h2d"], "d2h_bytes_per_step_per_rank": bytes_[name]["d2h"],
        }
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    if dist:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
