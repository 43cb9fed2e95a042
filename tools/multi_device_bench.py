"""Self-play and gating throughput of one process driving 1, 2, 4 and 8 devices (Config.engine_devices).

    python tools/multi_device_bench.py [--games-per-device 4096] [--max-iter 160] [--battle-games 512] [--out FILE]

For each device count D (up to the visible devices): generate_games(compact=True) of D x games-per-device games with
BASELINE config-3 settings (AlphaSame(10,16) random init bf16, MAX_ITER 160, Gamma root noise, FPU reduction, training
searches), all concurrent, and battle_networks of D x battle-games battles; games/h of the whole call (engine
construction and graph capture included, after one warm-up call that loads the modules).  The host thread's time in
SelfPlayEngine.step (graph launches), in drain (which waits for the device) and in the status reads is reported
against the wall time: a host-bound thread shows up as little wait and much launch / bookkeeping time.  Prints the
GPU name and power limit of the same run, and the torchrun figure of DESIGN.md section 5 for comparison.  One JSON
line per measurement.
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

TORCHRUN_GAMES_PER_H_8GPU = 3.95e7     # DESIGN.md section 5: config 3 under torchrun, one process per GPU, 8 x B200


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError):
        q = []
    return q


class HostClock:
    """Wraps SelfPlayEngine.step / drain / get_ctl and sums the host thread's time in each."""

    def __init__(self):
        from tetris_reinforcement_learning_b200 import selfplay
        self.cls = selfplay.SelfPlayEngine
        self.t = {"step": 0.0, "drain": 0.0, "get_ctl": 0.0}
        self.orig = {k: getattr(self.cls, k) for k in self.t}
        for k, fn in self.orig.items():
            setattr(self.cls, k, self._timed(k, fn))

    def _timed(self, name, fn):
        def run(eng, *a, **kw):
            t0 = time.perf_counter()
            try:
                return fn(eng, *a, **kw)
            finally:
                self.t[name] += time.perf_counter() - t0
        return run

    def reset(self):
        for k in self.t:
            self.t[k] = 0.0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games-per-device", type=int, default=4096)
    ap.add_argument("--max-iter", type=int, default=160)
    ap.add_argument("--battle-games", type=int, default=512, help="battles per device")
    ap.add_argument("--counts", default="1,2,4,8")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import os
    import tempfile
    # generate_games numbers its set after <Storage>/data: a scratch Storage unless the caller names one
    os.environ.setdefault("TRL_STORAGE", tempfile.mkdtemp(prefix="trl_mdb_"))
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("multi_device_bench needs CUDA devices")
    from tetris_reinforcement_learning_b200 import ai, architectures as arch, training
    from tetris_reinforcement_learning_b200.config import Config
    n_vis = torch.cuda.device_count()
    info = gpu_info()
    lines = [{"gpus_visible": n_vis, "gpu": info, "torchrun_games_per_h_8gpu": TORCHRUN_GAMES_PER_H_8GPU}]
    print(json.dumps(lines[0]), flush=True)
    torch.manual_seed(0)
    net = arch.AlphaSame(arch.AlphaSameConfig(blocks=10, filters=16)).cuda().eval()

    def cfg(devs, max_iter):
        c = Config(visual=False, ruleset="s2", model="pytorch", model_config=arch.AlphaSameConfig(blocks=10, filters=16),
                   MAX_ITER=max_iter, CPUCT=0.75, training=True, use_playout_cap_randomization=False,
                   use_dirichlet_noise=True, FpuStrategy="reduction")
        c.engine_devices = devs
        return c

    clock = HostClock()
    counts = [d for d in (int(x) for x in args.counts.split(",")) if d <= n_vis]
    ai.generate_games(cfg(list(range(max(counts))), 8), net, 8 * max(counts), seed=1, compact=True)   # warm-up
    base = None
    for d in counts:
        devs = list(range(d))
        n = args.games_per_device * d
        torch.cuda.synchronize()
        clock.reset()
        t0 = time.perf_counter()
        cs, stats = ai.generate_games(cfg(devs, args.max_iter), net, n, seed=20261018, compact=True)
        wall = time.perf_counter() - t0
        gph = len(stats) / wall * 3600
        base = base or gph
        rec = {"what": "generate_games", "devices": d, "games": len(stats), "searches": len(cs), "wall_s": round(wall, 3),
               "games_per_h": gph, "scaling_vs_1": gph / base, "host_step_s": round(clock.t["step"], 3),
               "host_drain_s": round(clock.t["drain"], 3), "host_status_s": round(clock.t["get_ctl"], 3),
               "host_other_s": round(wall - sum(clock.t.values()), 3)}
        if d == 8:
            rec["vs_torchrun_8gpu"] = gph / TORCHRUN_GAMES_PER_H_8GPU
        print(json.dumps(rec), flush=True)
        lines.append(rec)
        nb = args.battle_games * d
        c = cfg(devs, args.max_iter)
        c.training = False
        clock.reset()
        t0 = time.perf_counter()
        wins, _ = training.battle_networks(net, c, net, c, None, "more", nb, seed=3)
        wall = time.perf_counter() - t0
        rec = {"what": "battle_networks", "devices": d, "games": int(wins.sum()), "wall_s": round(wall, 3),
               "games_per_h": wins.sum() / wall * 3600, "host_step_s": round(clock.t["step"], 3),
               "host_drain_s": round(clock.t["drain"], 3), "host_status_s": round(clock.t["get_ctl"], 3)}
        print(json.dumps(rec), flush=True)
        lines.append(rec)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
