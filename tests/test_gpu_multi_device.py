"""GPU tests of Config.engine_devices (-m gpu): self-play sets, gating battles and analysis sharded over devices from
one process give what one device gives.

On one GPU the sharding is exercised with engine_devices=[0, 0] (two engines on one device); with two or more GPUs
the same checks run with [0, 1] and "all", and every entry point family is called on device 1 after device 0 in one
process (per-device library state: workspace, host streams, kernel attributes, pass-form scratch, debug switches)."""
import copy

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _storage(tmp_path, monkeypatch):
    """generate_games numbers its set after the Storage directory's data sets: keep it out of the tree."""
    monkeypatch.setenv("TRL_STORAGE", str(tmp_path / "Storage"))


def _n_gpus():
    import torch
    return torch.cuda.device_count()


def _device_lists():
    out = [[0, 0]]
    if _n_gpus() >= 2:
        out += [[0, 1], "all"]
    return out


def _net(kind):
    import torch
    from tetris_reinforcement_learning_b200 import architectures as arch
    torch.manual_seed(0)
    if kind == "alphasame10x16":    # rows trunk (csrc/trunk_rows.cu)
        return arch.AlphaSame(arch.AlphaSameConfig(blocks=10, filters=16)).cuda().eval()
    return arch.AuxBaseResNet(arch.AuxBaseResNetConfig(blocks=1, filters=32)).cuda().eval()   # wide trunk


def _cfg(devices=None, **kw):
    from tetris_reinforcement_learning_b200.config import Config
    base = dict(visual=False, ruleset="s2", model="pytorch", MAX_ITER=8, training=True, use_random_starting_moves=True,
                use_playout_cap_randomization=True)
    base.update(kw)
    c = Config(**base)
    c.engine_devices = devices
    return c


def _assert_sets_equal(a, b):
    assert len(a) == len(b) > 0
    assert np.array_equal(a.state.view(np.uint8), b.state.view(np.uint8))
    for name in ("value", "offsets", "moves", "frac"):
        assert np.array_equal(getattr(a, name), getattr(b, name)), name


@pytest.mark.parametrize("devices", _device_lists(), ids=str)
@pytest.mark.parametrize("kind", ["alphasame10x16", "aux1x32"])
def test_generate_games_sharded_equals_one_device(kind, devices):
    from tetris_reinforcement_learning_b200 import ai
    net = _net(kind)
    one, stats_one = ai.generate_games(_cfg(None), net, 10, seed=7, compact=True)
    many, stats_many = ai.generate_games(_cfg(devices), net, 10, seed=7, compact=True)
    _assert_sets_equal(one, many)
    assert stats_one == stats_many


def _per_game(cs):
    """CompactSet -> {game id: [(position bytes, value, moves, fractions) of its saved searches, in set order]}."""
    out = {}
    for i in range(cs.n_searches):
        lo, hi = cs.offsets[i], cs.offsets[i + 1]
        out.setdefault(int(cs.state[i]["game_id"]), []).append(
            (cs.state[i:i + 1].view(np.uint8).tobytes(), float(cs.value[i]), cs.moves[lo:hi].tobytes(), cs.frac[lo:hi].tobytes()))
    return out


@pytest.mark.parametrize("devices", _device_lists(), ids=str)
def test_generate_games_json_sharded_equals_one_device(devices):
    """The reference's sample lists (make_training_set's default format): merged per game in id order like one device's."""
    from tetris_reinforcement_learning_b200 import ai
    net = _net("alphasame10x16")
    one, stats_one = ai.generate_games(_cfg(None), net, 6, seed=9)
    many, stats_many = ai.generate_games(_cfg(devices), net, 6, seed=9)
    assert len(one) > 0 and one == many
    assert stats_one == stats_many


@pytest.mark.parametrize("devices", _device_lists(), ids=str)
def test_generate_games_with_restarts_keeps_every_common_game(devices):
    """concurrent < num_games: finished slots restart with new ids.  Which games make the set may differ between the
    runs; every game present in both has the same samples."""
    from tetris_reinforcement_learning_b200 import ai
    net = _net("alphasame10x16")
    one = _per_game(ai.generate_games(_cfg(None), net, 8, seed=3, concurrent=5, compact=True)[0])
    many = _per_game(ai.generate_games(_cfg(devices), net, 8, seed=3, concurrent=5, compact=True)[0])
    common = set(one) & set(many)
    assert len(common) >= 4
    for gid in common:
        assert one[gid] == many[gid], gid


@pytest.mark.parametrize("devices", _device_lists(), ids=str)
def test_battle_networks_sharded_tally(devices):
    from tetris_reinforcement_learning_b200 import training
    a = _net("alphasame10x16")
    b = copy.deepcopy(a)
    with __import__("torch").no_grad():
        for p in b.parameters():
            p.mul_(0.9)
    c1 = _cfg(None, MAX_ITER=6, training=False, use_random_starting_moves=False)
    want = training.battle_networks(a, c1, b, c1, 0.5, "more", 12, seed=4)
    cN = _cfg(devices, MAX_ITER=6, training=False, use_random_starting_moves=False)
    got = training.battle_networks(a, cN, b, cN, 0.5, "more", 12, seed=4)
    assert np.array_equal(want[0], got[0]) and want[1] == got[1] and want[0].sum() == 12


def _positions(n, seed=11):
    from tetris_reinforcement_learning_b200 import env, move_generation
    games = env.game_setup_host(n, 0, seed)
    for _ in range(6):
        pl = games["players"][np.arange(n), games["turn"]]
        res = move_generation.movegen_host(np.ascontiguousarray(pl["rows"]), pl["piece"].copy(),
                                           np.where(pl["held"] != 255, pl["held"], pl["queue"][:, 0]).astype(np.uint8),
                                           want_mask=False, want_moves=True, moves_cap=128)
        env.env_step_host(games, res["moves"][:, 0].astype(np.uint16), True, seed)
    return games


@pytest.mark.parametrize("devices", _device_lists(), ids=str)
@pytest.mark.parametrize("kind,n", [("alphasame10x16", 8), ("alphasame10x16", 9), ("aux1x32", 8), ("aux1x32", 9)])
def test_analyse_and_evaluate_positions_sharded(kind, n, devices):
    """n = 8 on [0, 0]: two blocks of the same size on one device (each needs its own engine); n = 9: blocks of 5 and 4."""
    import torch
    from tetris_reinforcement_learning_b200 import ai
    from tetris_reinforcement_learning_b200.devices import contiguous_blocks, engine_devices
    net = _net(kind)
    recs = _positions(n)
    c1 = _cfg(None, use_random_starting_moves=False)
    cN = _cfg(devices, use_random_starting_moves=False)
    want = ai.analyse(c1, recs, net, seed=2, search_no=1)
    got = ai.analyse(cN, recs, net, seed=2, search_no=1)
    assert len(want) == len(got) == n
    for w, g in zip(want, got):
        assert (w is None) == (g is None)
        if w is None:
            continue
        for name in ("moves", "visits", "visits_pre", "priors", "q", "pv", "pv_visits"):
            assert np.array_equal(getattr(w, name), getattr(g, name)), name
        assert (w.chosen_move, w.iterations, w.saved, w.root_value) == (g.chosen_move, g.iterations, g.saved, g.root_value)
    # evaluate_positions: trunk, heads and values are the project's kernels and bit-identical at any batch size
    v1, p1 = ai.evaluate_positions(c1, recs, net)
    vN, pN = ai.evaluate_positions(cN, recs, net)
    assert np.array_equal(v1.view(np.uint32), vN.view(np.uint32))
    # the dense policy GEMM (cuBLAS) may pick another algorithm for another batch size: a block's logits are within one
    # bf16 rounding of the one-device batch rows (the bound of tests/test_gpu_analysis.py), each nearest to its own row,
    # and the block's policies are exactly the softmax of its logits
    _, l_all = ai._evaluate_packed(net, recs)
    devs = engine_devices(cN)
    for dev, (lo, hi) in zip(devs, contiguous_blocks(n, len(devs))):
        if hi == lo:
            continue
        _, lb = ai._evaluate_packed(net, recs[lo:hi], dev)
        assert np.array_equal(pN[lo:hi].reshape(hi - lo, -1), torch.softmax(lb, 1).cpu().numpy())
        lb = lb.to(l_all.device)
        assert ((lb - l_all[lo:hi]).abs() <= 2 ** -7 * l_all[lo:hi].abs() + 1e-4).all()
        for i in range(lo, hi):
            assert int((l_all - lb[i - lo]).abs().amax(1).argmin()) == i
    ai.release_cached_engines()


def _entry_points_on(dev):
    """Every entry point family on `dev`, called while cuda:0 is the current device -> dict of host arrays."""
    import torch
    from tetris_reinforcement_learning_b200 import _native, ai, env, move_generation, synth, trunk, trunk_wide
    from tetris_reinforcement_learning_b200 import architectures as arch
    L = _native.lib()
    out = {}
    boards, cur, alt = synth.movegen_workload(300, seed=5, caves=True)
    d_boards = torch.from_numpy(boards.view(np.int16)).to(dev)
    d_cur, d_alt = torch.from_numpy(cur).to(dev), torch.from_numpy(alt).to(dev)
    n = boards.shape[0]
    # every launch form of the enumeration, and the one-thread kernel
    for name, form, kernel in (("warp2", 0, -1), ("warp1", 1, -1), ("pass", 2, -1), ("thread", -1, 0)):
        L.trl_movegen_warp_form(form)
        L.trl_movegen_select_kernel(kernel)
        try:
            mask = torch.zeros((n, 362), dtype=torch.int32, device=dev)
            moves = torch.zeros((n, 256), dtype=torch.int16, device=dev)
            nm = torch.zeros(n, dtype=torch.int16, device=dev)
            move_generation.movegen_device(d_boards, d_cur, d_alt, mask, moves, nm, None)
            out["mg_" + name] = (mask.cpu().numpy(), moves.cpu().numpy(), nm.cpu().numpy())
        finally:
            L.trl_movegen_warp_form(-1)
            L.trl_movegen_select_kernel(-1)
    with torch.cuda.device(dev):      # host entry points follow the current device
        r = move_generation.movegen_host(boards, cur, alt, want_mask=True, want_moves=True, moves_cap=256)
        out["mg_host"] = (r["mask_bits"], r["moves"], r["n_moves"])
        c = move_generation.movegen_host_compact(boards, cur, alt)
        out["mg_host_compact"] = (c["n_moves"], np.sort(c["moves"]), c["total"])
        g = env.game_setup_host(64, 0, 9)
        env.env_step_host(g, out["mg_host"][1][:64, 0].astype(np.uint16), True, 9)
        out["env_host"] = g.view(np.uint8).copy()
    d_games = torch.zeros((64, 400), dtype=torch.uint8, device=dev)
    env.game_setup_device(d_games, 0, 9)
    env.env_step_device(d_games, torch.from_numpy(out["mg_host"][1][:64, 0].copy()).to(dev), None, True, 9)
    out["env_dev"] = d_games.cpu().numpy()
    # features + fused trunk + heads (rows trunk), taps trunk, wide trunk
    torch.manual_seed(0)
    a16 = arch.AlphaSame(arch.AlphaSameConfig(blocks=4, filters=16)).to(dev).eval()
    recs = g
    v, logits = ai._evaluate_packed(a16, recs, dev)
    out["eval_rows"] = (v.cpu().numpy(), logits.cpu().numpy())
    grids = (torch.rand((40, 1, 40, 10), generator=torch.Generator().manual_seed(1)) < 0.3).to(dev, torch.bfloat16)
    out["taps"] = trunk.trunk_forward(trunk.pack_alphasame_trunk(a16, layout="taps"), grids).float().cpu().numpy()
    torch.manual_seed(0)
    w32 = arch.AuxBaseResNet(arch.AuxBaseResNetConfig(blocks=1, filters=32)).to(dev).eval()
    wt = trunk_wide.WideTrunk(trunk_wide.pack_wide_trunk(w32), dev)
    out["wide"] = trunk_wide.wide_trunk_forward(wt, grids).float().cpu().numpy()
    # a captured search step (graph replays) of an engine on `dev`
    cfg = _cfg(None, MAX_ITER=6)
    eng = ai._engine_for(cfg, a16, 32, seed=3, device=dev, random_openings=True)
    eng.step(12)
    samples, ends = eng.drain()
    eng.check_status()
    out["engine"] = (samples.view(np.uint8).copy(), eng.get_games().view(np.uint8).copy())
    return out


@pytest.mark.skipif("_n_gpus() < 2", reason="needs two GPUs: device 1 after device 0 in one process")
def test_every_entry_point_on_device_1_after_device_0():
    import torch
    torch.cuda.set_device(0)
    want = _entry_points_on(torch.device("cuda:0"))
    got = _entry_points_on(torch.device("cuda:1"))
    assert torch.cuda.current_device() == 0
    assert want.keys() == got.keys()
    for k in want:
        w, g = want[k], got[k]
        w, g = (w if isinstance(w, tuple) else (w,)), (g if isinstance(g, tuple) else (g,))
        for a, b in zip(w, g):
            assert np.array_equal(np.asarray(a), np.asarray(b)), k
    for name in ("mg_warp2", "mg_warp1", "mg_pass", "mg_thread"):
        assert np.array_equal(want[name][0], want["mg_host"][0].view(np.int32)), name


@pytest.mark.skipif("_n_gpus() < 2", reason="needs two GPUs: a debug switch set on device 0 and used on device 1")
def test_debug_switch_reaches_device_1_and_is_refused_inside_a_capture():
    """trl_debug_movegen_fifo_limit set while device 0 is current: device 1's next launch gets the lowered FIFO (its
    calls overflow like device 0's).  After the switch is reset on device 0, device 1 still holds the lowered limit; a
    launch inside a capture cannot copy the switch over and fails, the next launch outside a capture does."""
    import torch
    from tetris_reinforcement_learning_b200 import _native, move_generation, synth
    L = _native.lib()
    torch.cuda.set_device(0)
    boards, cur, alt = synth.movegen_workload(300, seed=5, caves=True)

    def args(dev):
        n = boards.shape[0]
        return (torch.from_numpy(boards.view(np.int16)).to(dev), torch.from_numpy(cur).to(dev), torch.from_numpy(alt).to(dev),
                None, torch.zeros((n, 256), dtype=torch.int16, device=dev), torch.zeros(n, dtype=torch.int16, device=dev),
                torch.zeros(n, dtype=torch.int32, device=dev))

    def status(dev):
        a = args(dev)
        move_generation.movegen_device(*a)
        return a[6].cpu().numpy()

    d0, d1 = torch.device("cuda:0"), torch.device("cuda:1")
    clean = status(d1)
    assert not (clean & 1).any()
    assert L.trl_debug_movegen_fifo_limit(2) == 0
    try:
        s0, s1 = status(d0), status(d1)
    finally:
        assert L.trl_debug_movegen_fifo_limit(0) == 0
    assert (s0 & 1).any() and np.array_equal(s0, s1)
    a = args(d1)
    with torch.cuda.device(d1):
        g = torch.cuda.CUDAGraph()
        with pytest.raises(RuntimeError):
            with torch.cuda.graph(g):
                move_generation.movegen_device(*a)
    assert np.array_equal(status(d1), clean)
    assert torch.cuda.current_device() == 0
