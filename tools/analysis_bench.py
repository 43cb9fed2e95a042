"""Throughput of the analysis path: ai.analyse on a batch of positions against sequential ai.MCTS calls on the
same positions, and, as the yardstick, the self-play step rate of the same network at the same batch size.

    python tools/analysis_bench.py [--positions 4096] [--iters 160] [--mcts-calls 64] [--out results.json]

Positions are mid-game states from the oracle's random play (seeded).  Every timed window ends with a device
synchronise; each measurement is preceded by an untimed call of the same shape (engine allocation, CUDA-graph
capture).  Prints the card's name and power limit with the numbers; needs a CUDA device.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        power = q.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def timed(fn):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--positions", type=int, default=4096)
    ap.add_argument("--iters", type=int, default=160)
    ap.add_argument("--mcts-calls", type=int, default=64)
    ap.add_argument("--selfplay-steps", type=int, default=160)
    ap.add_argument("--out", default=None, help="write the results as JSON here as well")
    args = ap.parse_args()

    import numpy as np
    import torch
    if not torch.cuda.is_available():
        sys.exit("analysis_bench needs a CUDA device")
    from oracle import oracle
    from oracle.pin_against_reference import random_midgame
    from tetris_reinforcement_learning_b200 import ai, architectures as arch
    from tetris_reinforcement_learning_b200.config import Config
    from tetris_reinforcement_learning_b200.selfplay import SelfPlayEngine, best_evaluator
    from tetris_reinforcement_learning_b200.state import unpack_game
    oracle.build()

    name, power = card()
    print(f"device: {name}, power limit {power}")
    recs = random_midgame(np.random.default_rng(1), args.positions, 6)
    results = {"device": name, "power_limit": power, "positions": args.positions, "iters": args.iters, "nets": []}
    torch.manual_seed(0)
    nets = [("AlphaSame(10,16)", arch.AlphaSameConfig(blocks=10, filters=16)),
            ("Config default " + type(Config(visual=False).model_config).__name__, Config(visual=False).model_config)]
    for label, mc in nets:
        net = arch.build_network(mc, False).to("cuda:0").eval()
        cfg = Config(visual=False, ruleset="s2", model="pytorch", model_config=mc, MAX_ITER=args.iters, training=False)

        ai.analyse(cfg, recs, net, seed=1)                                   # engine + graph capture
        t_an, res = timed(lambda: ai.analyse(cfg, recs, net, seed=1))
        n_ok = sum(r is not None for r in res)

        sub = [recs[i] for i in range(len(recs)) if res[i] is not None][:args.mcts_calls]   # MCTS raises on the others
        games = [unpack_game(r) for r in sub]
        ai.MCTS(cfg, games[0], net, seed=1)                                   # one-game engine + graph capture
        t_mc, _ = timed(lambda: [ai.MCTS(cfg, g, net, seed=1) for g in games])

        eng = SelfPlayEngine(cfg, best_evaluator(net), args.positions, seed=1, feature_dtype=torch.bfloat16,
                             sample_cap=4 * args.positions)
        eng.step(8)
        eng.drain()
        t_sp, _ = timed(lambda: eng.step(args.selfplay_steps))
        eng.drain()
        del eng

        row = {"net": label,
               "analyse_s": t_an, "analyse_positions_per_s": args.positions / t_an, "analyse_searched": n_ok,
               "mcts_s": t_mc, "mcts_positions_per_s": len(games) / t_mc,
               "speedup": (args.positions / t_an) / (len(games) / t_mc),
               "analyse_sims_per_s": args.positions * args.iters / t_an,
               "selfplay_sims_per_s": args.positions * args.selfplay_steps / t_sp}
        results["nets"].append(row)
        print(f"{label}: analyse {args.positions} positions x {args.iters} iterations in {t_an:.3f} s = "
              f"{row['analyse_positions_per_s']:.0f} positions/s ({n_ok} searched); {len(games)} sequential MCTS calls "
              f"in {t_mc:.3f} s = {row['mcts_positions_per_s']:.1f} positions/s; speed-up {row['speedup']:.0f}x; "
              f"simulations/s: analyse {row['analyse_sims_per_s']:.3g}, self-play step {row['selfplay_sims_per_s']:.3g}")
        ai.release_cached_engines()
    print(json.dumps(results))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
