"""GPU tests of the analysis path (-m gpu): analysis-mode search (TrlSearchParams.stop_after_search), the root
statistics record (TrlRootStats), ai.analyse / ai.MCTS on it, and ai.evaluate / ai.evaluate_positions.

Searches run with the oracle's integer-hash evaluator (oracle/features_oracle.py), whose float32 outputs are
bit-identical on both sides, on the reference vectors of tests/golden/mcts_golden*.npz."""
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from tetris_reinforcement_learning_b200.config import Config  # noqa: E402
from tetris_reinforcement_learning_b200.state import GAME_DTYPE, unpack_game  # noqa: E402

NO_PIECE = 0x4


def config_families(iters):
    """The four search settings the golden vectors were produced with."""
    base = dict(visual=False, ruleset="s2", model="pytorch", MAX_ITER=iters, CPUCT=0.75)
    return [
        Config(training=False, **base),
        Config(training=True, **base),
        Config(training=True, use_forced_playouts_and_policy_target_pruning=True,
               use_playout_cap_randomization=False, **base),
        Config(training=True, FpuStrategy="absolute", use_tanh=True, use_root_softmax=False, **base),
    ]


def fake_evaluator_torch(device, tanh=False):
    """oracle/features_oracle.fake_outputs in torch (bit-identical float32 values / logits)."""
    import torch
    from oracle import features_oracle as fo
    wg = torch.from_numpy(fo.W_GRID).to(device)
    we = torch.from_numpy(fo.W_EXTRA).to(device)
    j = torch.arange(11583, dtype=torch.int64, device=device)

    def ev(grids, extras):
        G = extras.shape[0]
        g = grids.reshape(2, G, 400).permute(1, 0, 2).reshape(G, 800).to(torch.int64)
        e = extras.to(torch.int64) + 2
        h = ((g * wg).sum(1) + (e * we).sum(1)) & 0x7FFFFFFF
        value = ((h % 997) + 1).to(torch.float32) / 1000.0
        if tanh:
            value = 2 * value - 1
        logits = ((((h >> 3)[:, None] * (2 * j + 1)[None, :]) + 7 * j * j) % 4096).to(torch.float32) / fo.LOGIT_DIV
        return value.contiguous(), logits.contiguous()
    return ev


_EVALUATORS = {}


def evaluator(tanh):
    """One evaluator object per value mode, so that ai's engine cache is reused across calls."""
    import torch
    if tanh not in _EVALUATORS:
        _EVALUATORS[tanh] = fake_evaluator_torch(torch.device("cuda:0"), tanh)
    return _EVALUATORS[tanh]


def load(golden_dir, name):
    g = np.load(os.path.join(golden_dir, name))
    return g, g["games"].copy().view(GAME_DTYPE).reshape(-1)


@pytest.mark.parametrize("vectors", ["mcts_golden.npz", "mcts_golden_160.npz"])
def test_analyse_matches_reference_vectors(golden_dir, vectors):
    """analyse() on the golden positions: root children and their order, save flags bit-exact; visit counts under
    the criteria of test_gpu_search.test_search_vs_reference_vectors (total-variation distance <= 0.02 per
    search, at least 95 % of searches identical, the chosen move exact where the visits are)."""
    from tetris_reinforcement_learning_b200 import ai
    golden, games = load(golden_dir, vectors)
    exact = total = 0
    worst_tv = 0.0
    for fam, cfg in enumerate(config_families(int(golden["iters"]))):
        sel = np.flatnonzero(golden["family"] == fam)
        res = ai.analyse(cfg, games[sel], evaluator(cfg.use_tanh), seed=int(golden["seed"]),
                         game_ids=games[sel]["game_id"], search_no=sel)
        assert len(res) == len(sel)
        for r, k in zip(res, sel):
            C = int(golden["n_children"][k])
            assert r is not None and len(r.moves) == C
            assert np.array_equal(r.moves, golden["child_moves"][k][:C])
            assert r.saved == bool(golden["save"][k])
            want = golden["child_visits"][k][:C].astype(np.float64)
            got = r.visits.astype(np.float64)
            worst_tv = max(worst_tv, 0.5 * np.abs(want / max(want.sum(), 1) - got / max(got.sum(), 1)).sum())
            total += 1
            if np.array_equal(want, got):
                exact += 1
                assert r.chosen_move == int(golden["move"][k])
    print(f"analyse vs the reference: {exact}/{total} searches identical, worst total-variation distance {worst_tv:.4f}")
    assert worst_tv <= 0.02 and exact >= 0.95 * total


@pytest.mark.parametrize("vectors", ["mcts_golden.npz", "mcts_golden_160.npz"])
def test_analyse_equals_mcts(golden_dir, vectors):
    """analyse(batch)[k] is MCTS(position k) bit for bit, Game objects in both."""
    from tetris_reinforcement_learning_b200 import ai
    golden, games = load(golden_dir, vectors)
    seed = int(golden["seed"])
    for fam, cfg in enumerate(config_families(int(golden["iters"]))):
        sel = np.flatnonzero(golden["family"] == fam)
        objs = [unpack_game(games[k]) for k in sel]
        ids = games[sel]["game_id"]
        batch = ai.analyse(cfg, objs, evaluator(cfg.use_tanh), seed=seed, game_ids=ids, search_no=sel)
        for i, k in enumerate(sel):
            move, one, saved = ai.MCTS(cfg, objs[i], evaluator(cfg.use_tanh), seed=seed, game_id=int(ids[i]),
                                       search_no=int(k))
            b = batch[i]
            assert move == b.move and saved == b.saved and one.chosen_move == b.chosen_move
            for name in ("moves", "visits", "visits_pre", "priors", "q", "pv", "pv_visits"):
                assert np.array_equal(getattr(one, name), getattr(b, name)), (fam, int(k), name)
            assert one.root_value == b.root_value and one.state.tobytes() == b.state.tobytes()


ORACLE_TREE = ("first_child", "n_children", "visits", "value_avg", "move_of")


def oracle_search_with_tree(cfg, rec, seed, game_id, search_no, noise):
    """mcts_oracle.search plus its tree as it stands when the search returns: the struct-of-arrays lists named in
    ORACLE_TREE, read from the function's frame by a profile hook, so the pinned oracle runs unchanged.  A profiler
    installed before (coverage, ...) keeps receiving its events; a renamed or missing list fails here, not later.
    noise: the Gamma draws to use, or None."""
    from oracle import features_oracle as fo, mcts_oracle
    tape = mcts_oracle.SearchTape(seed, game_id, search_no)
    if noise is not None:
        tape.gamma = lambda alpha, n: np.asarray(noise[:n], dtype=np.float64)
    tree = {}
    previous = sys.getprofile()

    def hook(frame, event, arg):
        if event == "return" and frame.f_code is mcts_oracle.search.__code__:
            tree.update({k: frame.f_locals[k] for k in ORACLE_TREE if k in frame.f_locals})
        if previous is not None:
            previous(frame, event, arg)
    sys.setprofile(hook)
    try:
        res = mcts_oracle.search(cfg, np.array(rec, dtype=GAME_DTYPE).reshape(1), fo.fake_evaluate, tape)
    finally:
        sys.setprofile(previous)
    missing = [k for k in ORACLE_TREE if k not in tree]
    assert not missing, f"mcts_oracle.search no longer keeps its tree in {missing}: update ORACLE_TREE"
    assert len(tree["visits"]) == res["n_nodes"]
    return res, tree


def device_priors(cfg, rec, noisy, noise_row):
    """The kernel's root priors restated in fp64 (mcts.cu, expand_body): softmax of the legal logits in double,
    temperature 1 / RootSoftmaxTemp at the root, the 1e-25 clamp, then the noise mix."""
    from oracle import features_oracle as fo, mcts_oracle
    root = mcts_oracle.truncate_previews(rec)[0]
    _, logits = fo.fake_outputs(fo.fake_hash(*fo.encode(root)))
    moves = mcts_oracle.legal_moves(root)
    lg = logits[moves].astype(np.float64)
    inv = 1.0 / cfg.RootSoftmaxTemp if cfg.use_root_softmax else 1.0
    e = np.exp((lg - lg.max()) * inv)
    e[~(e > 0)] = 1e-25
    pr = e / e.sum()
    if noisy:
        pr = pr * (1.0 - cfg.DIRICHLET_EXPLORATION) + noise_row[:len(pr)] * cfg.DIRICHLET_EXPLORATION
    return pr


def _ulps_f32(a, b):
    ia = np.asarray(a, np.float32).view(np.int32).astype(np.int64)
    ib = np.asarray(b, np.float32).view(np.int32).astype(np.int64)
    return np.abs(ia - ib)


@pytest.mark.parametrize("noise", [False, True])
def test_root_stats_against_the_oracle(golden_dir, oracle, noise):
    """Priors, Q values, root value and the first two plies of the principal variation against the fp64 oracle
    search, noise off (families without it) and on (the same Gamma draws on both sides: the oracle's tape on the
    device through set_noise_override).  Priors: bit-equal to the fp64 restatement of the kernel's formula as
    float32, and within 8 float32 ulps of the oracle's (the oracle keeps the reference's float32 softmax and
    division, the kernel computes in double: emulated on a CPU, 2 ulps at most with the root softmax, 5
    without).  Q and root value within 1e-6."""
    import torch
    from oracle import mcts_oracle
    from tetris_reinforcement_learning_b200.selfplay import SelfPlayEngine
    golden, games = load(golden_dir, "mcts_golden.npz")
    seed = int(golden["seed"])
    fams = config_families(int(golden["iters"]))
    cases = [(0, fams[0]), (3, Config(visual=False, ruleset="s2", model="pytorch", MAX_ITER=int(golden["iters"]),
                                      CPUCT=0.75, training=True, use_dirichlet_noise=False, use_root_softmax=False))]
    if noise:
        cases = [(1, fams[1]), (2, fams[2])]
    n_prior = n_prior_equal = worst_ulps = 0
    for fam, cfg in cases:
        sel = np.flatnonzero(golden["family"] == fam)
        G = len(sel)
        eng = SelfPlayEngine(cfg, evaluator(cfg.use_tanh), G, seed=seed, restart_finished=False, analysis=True,
                             root_stats=True)
        draws = np.zeros((G, eng.moves_cap))
        for i, k in enumerate(sel):
            tape = mcts_oracle.SearchTape(seed, int(games[k]["game_id"]), int(k))
            C = len(mcts_oracle.legal_moves(mcts_oracle.truncate_previews(games[k])[0]))
            alpha = cfg.DIRICHLET_ALPHA * (cfg.DIRICHLET_S / C if cfg.use_dirichlet_s else 1.0)
            draws[i, :C] = tape.gamma(alpha, C)
        if noise:
            eng.set_noise_override(draws)
        eng.set_games(games[sel])
        ctl = eng.get_ctl()
        ctl["search_no"] = sel
        eng.set_ctl(ctl)
        long_iters, _ = cfg.playout_iterations()
        eng.step(long_iters if (cfg.training and cfg.use_playout_cap_randomization) else cfg.MAX_ITER)
        samples, _ = eng.drain()
        stats = eng.drain_root_stats()
        assert len(samples) == len(stats) == G
        eng.check_status()
        for s, st in zip(samples, stats):
            i = int(st["slot"])
            k = int(sel[i])
            res, tree = oracle_search_with_tree(cfg, games[k], seed, int(games[k]["game_id"]), k,
                                                draws[i] if noise else None)
            C = int(s["n_children"])
            assert int(st["n_children"]) == C == len(res["moves"])
            assert list(s["visits_pre"][:C]) == res["visits_pre"], k   # same tree shape on both sides
            noisy = bool(cfg.training and cfg.use_dirichlet_noise and s["saved"])
            assert np.array_equal(st["prior"][:C], device_priors(cfg, games[k], noisy, draws[i]).astype(np.float32)), k
            ulps = _ulps_f32(st["prior"][:C], np.asarray(res["priors"], np.float64).astype(np.float32))
            assert ulps.max() <= 8, (k, int(ulps.max()))
            worst_ulps = max(worst_ulps, int(ulps.max()))
            n_prior += C
            n_prior_equal += int((ulps == 0).sum())
            kids = range(tree["first_child"][0], tree["first_child"][0] + tree["n_children"][0])
            want_q = np.array([tree["value_avg"][c] for c in kids], np.float64)
            assert np.abs(st["q"][:C].astype(np.float64) - want_q).max() <= 1e-6, k
            assert abs(float(st["root_value"]) - res["root_value_avg"]) <= 1e-6
            # principal variation: most visited child (last maximum) of the root, then of that child
            pre = res["visits_pre"]
            i0 = max(range(C), key=lambda c: (pre[c], c))
            assert int(st["pv_len"]) >= 1 and int(st["pv"][0]) == res["moves"][i0] and int(st["pv_visits"][0]) == pre[i0]
            node = tree["first_child"][0] + i0
            n1 = tree["n_children"][node]
            grand = [tree["visits"][c] for c in range(tree["first_child"][node], tree["first_child"][node] + n1)] if n1 > 0 else []
            if grand and max(grand) > 0:
                j = max(range(n1), key=lambda c: (grand[c], c))
                assert int(st["pv_len"]) >= 2 and int(st["pv"][1]) == tree["move_of"][tree["first_child"][node] + j], k
                assert int(st["pv_visits"][1]) == grand[j]
            else:
                assert int(st["pv_len"]) == 1
    print(f"root priors vs the oracle: {n_prior_equal}/{n_prior} bit-equal as float32, at most {worst_ulps} ulps apart")


def mixed_positions(golden, games, n):
    """n positions cycling through the golden ones with varied search numbers (so that both playout-cap budgets
    occur), every 7th already over and every 11th without a piece to play."""
    recs = np.zeros(n, dtype=GAME_DTYPE)
    sno = np.zeros(n, dtype=np.int64)
    kind = np.zeros(n, dtype=np.int64)
    for i in range(n):
        k = i % len(games)
        recs[i] = games[k]
        recs[i]["game_id"] = 1000 + i
        sno[i] = 3 * i + 1
        if i % 7 == 5:
            recs[i]["players"][1 - int(recs[i]["turn"])]["game_over"] = 1
            kind[i] = 1
        elif i % 11 == 8:
            p = recs[i]["players"][int(recs[i]["turn"])]
            p["piece"], p["held"] = 255, 255
            kind[i] = 2
    return recs, sno, kind


def test_analysis_mode_invariants(golden_dir, oracle):
    """Analysis mode on a mixed batch: the games are left as they were, no game end is written, every game ends
    inactive after exactly its own budget of simulations, an unsearchable root writes no sample and raises
    NO_PIECE only; analyse() returns None for it.  Batches of 1, 5 and 4 x SMs + 3 positions give identical
    results (CUDA-graph chunks of 4 steps and budgets that are no multiple of it)."""
    import torch
    from oracle import mcts_oracle
    from tetris_reinforcement_learning_b200 import ai
    from tetris_reinforcement_learning_b200.selfplay import SelfPlayEngine
    golden, games = load(golden_dir, "mcts_golden.npz")
    cfg = config_families(22)[1]     # playout cap: long and short budgets (55 and 11) in one batch
    long_iters, short_iters = cfg.playout_iterations()
    assert long_iters % 4 and short_iters % 4
    seed = 9
    n_big = 4 * torch.cuda.get_device_properties(0).multi_processor_count + 3
    recs, sno, kind = mixed_positions(golden, games, n_big)

    G = 64
    eng = SelfPlayEngine(cfg, evaluator(False), G, seed=seed, restart_finished=False, analysis=True, root_stats=True)
    eng.set_games(recs[:G])
    ctl = eng.get_ctl()
    ctl["search_no"] = sno[:G]
    eng.set_ctl(ctl)
    eng.step(long_iters + 5)        # steps after the last search finished change nothing
    samples, ends = eng.drain()
    stats = eng.drain_root_stats()
    ctl = eng.get_ctl()
    assert eng.get_games().tobytes() == recs[:G].tobytes()
    assert len(ends) == 0 and (ctl["active"] == 0).all() and (ctl["iter"] == 0).all()
    assert (ctl["search_no"] == sno[:G]).all() and (ctl["games_finished"] == 0).all()
    budgets = np.array([long_iters if mcts_oracle.SearchTape(seed, int(recs[i]["game_id"]), int(sno[i])).coin()
                        < cfg.playout_cap_chance else short_iters for i in range(G)])
    assert (budgets == long_iters).any() and (budgets == short_iters).any()
    assert np.array_equal(ctl["sims"], budgets)
    assert np.array_equal(ctl["status"], np.where(kind[:G] > 0, NO_PIECE, 0))
    searched = sorted(int(st["slot"]) for st in stats)
    assert searched == [i for i in range(G) if kind[i] == 0] and len(samples) == len(stats)
    for s, st in zip(samples, stats):
        i = int(st["slot"])
        assert int(s["iterations"]) == budgets[i] and int(s["game_id"]) == int(recs[i]["game_id"])
        assert bool(s["saved"]) == (budgets[i] == long_iters)     # saved still reports the coin
        assert int(s["visits_pre"][:int(s["n_children"])].sum()) == budgets[i] - 1
    with pytest.raises(Exception, match="NO_PIECE"):
        eng.check_status()

    ev = evaluator(False)
    big = ai.analyse(cfg, recs, ev, seed=seed, search_no=sno)
    assert [r is None for r in big] == list(kind > 0)
    fives = [r for lo in range(0, 40, 5) for r in ai.analyse(cfg, recs[lo:lo + 5], ev, seed=seed, search_no=sno[lo:lo + 5])]
    ones = [ai.analyse(cfg, recs[i:i + 1], ev, seed=seed, search_no=sno[i:i + 1])[0] for i in range(12)]
    for other in (fives, ones):
        for a, b in zip(big, other):
            assert (a is None) == (b is None)
            if a is None:
                continue
            for name in ("moves", "visits", "visits_pre", "priors", "q", "pv", "pv_visits"):
                assert np.array_equal(getattr(a, name), getattr(b, name)), name
            assert (a.chosen_move, a.saved, a.root_value, a.iterations) == (b.chosen_move, b.saved, b.root_value, b.iterations)
    with pytest.raises(Exception, match="NO_PIECE"):
        ai.MCTS(cfg, unpack_game(recs[5]), ev, seed=seed)


@pytest.mark.parametrize("net", ["fake", "alphasame"])
def test_root_stats_do_not_perturb_self_play(net):
    """An ordinary self-play engine with the root-statistics ring on produces bit-identical samples, game ends and
    games to the same seeded run without it; one record per drained sample, with the sample's child count."""
    import torch
    from tetris_reinforcement_learning_b200 import architectures as arch
    from tetris_reinforcement_learning_b200.selfplay import SelfPlayEngine, best_evaluator
    cfg = Config(visual=False, ruleset="s2", model="pytorch", MAX_ITER=8, training=True,
                 use_forced_playouts_and_policy_target_pruning=True)
    if net == "fake":
        ev, kw = evaluator(False), dict(use_cuda_graph=False)
    else:
        torch.manual_seed(0)
        ev, kw = best_evaluator(arch.AlphaSame(arch.AlphaSameConfig(blocks=2, filters=16)).to("cuda:0")), \
            dict(feature_dtype=torch.bfloat16)
    out = []
    for rs in (False, True):
        eng = SelfPlayEngine(cfg, ev, 48, seed=7, save_all=True, restart_finished=False, max_rounds=6, sample_cap=4096,
                             root_stats=rs, **kw)
        eng.step(150)
        samples, ends = eng.drain()
        out.append((samples, ends, eng.get_games(), eng.get_ctl(), eng.drain_root_stats()))
    (s0, e0, g0, c0, r0), (s1, e1, g1, c1, r1) = out
    assert len(s0) > 100 and len(e0) > 0
    assert len(r0) == 0 and len(r1) == len(s1)
    assert all(int(st["slot"]) >= 0 and int(st["n_children"]) == int(s["n_children"]) for s, st in zip(s1, r1))
    # the rings fill in the order warps finish their searches: compare in (game id, search number) order, the
    # root-statistics records following their samples
    o0, o1 = np.lexsort((s0["search_no"], s0["game_id"])), np.lexsort((s1["search_no"], s1["game_id"]))
    s0, s1, r1 = s0[o0], s1[o1], r1[o1]
    e0, e1 = np.sort(e0, order=["game_id"]), np.sort(e1, order=["game_id"])
    assert s0.tobytes() == s1.tobytes() and e0.tobytes() == e1.tobytes() and g0.tobytes() == g1.tobytes()
    assert c0.tobytes() == c1.tobytes()
    assert np.array_equal(r1["n_children"], s1["n_children"])
    for s, st in zip(s1, r1):
        C = int(s["n_children"])
        pre = s["visits_pre"][:C]
        if pre.max() == 0:          # a one-iteration search expands the root only
            assert int(st["pv_len"]) == 0
        else:
            assert int(st["pv"][0]) == int(s["moves"][:C][np.flatnonzero(pre == pre.max())[-1]])
            assert int(st["pv_visits"][0]) == int(pre.max())


def _nets():
    import torch
    from tetris_reinforcement_learning_b200 import architectures as arch
    torch.manual_seed(4)
    return {"alphasame_10_16": arch.AlphaSame(arch.AlphaSameConfig(blocks=10, filters=16)),
            "alphasame_20_64": arch.AlphaSame(arch.AlphaSameConfig(blocks=20, filters=64)),
            "aux_8_32": arch.AuxBaseResNet(arch.AuxBaseResNetConfig(blocks=8, filters=32))}


@pytest.mark.parametrize("name", ["alphasame_10_16", "alphasame_20_64", "aux_8_32"])
def test_evaluate(name):
    """evaluate_positions rows vs evaluate one position at a time, policies summing to 1, and the fused
    evaluator's values / logits against the fp32 module on the oracle's encoding of the same positions, with the
    tolerances of tests/test_gpu_trunk*.py for the fused evaluators (value within 0.03, logits within
    5 % of max |logit| + 0.05)."""
    import torch
    from oracle import features_oracle as fo
    from oracle.pin_against_reference import random_midgame
    from tetris_reinforcement_learning_b200 import ai
    from tetris_reinforcement_learning_b200.const import POLICY_SIZE
    net = _nets()[name].to("cuda:0").eval()
    cfg = Config(visual=False, ruleset="s2", model="pytorch")
    recs = random_midgame(np.random.default_rng(5), 40, 6)
    values, policies = ai.evaluate_positions(cfg, recs, net)
    assert values.shape == (40,) and policies.shape == (40, 27, 39, 11)
    assert np.abs(policies.reshape(40, -1).astype(np.float64).sum(1) - 1.0).max() <= 1e-5
    # one position at a time.  The policy GEMM may pick another algorithm for a single row: its bf16 logits may then
    # differ by one rounding (2^-7 relative; 1e-4 absolute where a sum cancels), the value by one bf16 ulp.  Each
    # single result must also be nearest to its own row of the batch (a mis-indexed position fails there).
    _, l_all = ai._evaluate_packed(net, recs)
    exact_rows = 0
    for i in range(0, 40, 3):
        v, p = ai.evaluate(cfg, recs[i], net)
        assert isinstance(v, float) and p.shape == (27, 39, 11)
        v1, l1 = ai._evaluate_packed(net, recs[i:i + 1])
        assert v == float(v1[0]) and np.array_equal(p, torch.softmax(l1, 1).cpu().numpy().reshape(27, 39, 11))
        assert abs(v - float(values[i])) <= 2 ** -8, (i, v, float(values[i]))
        assert ((l1[0] - l_all[i]).abs() <= 2 ** -7 * l_all[i].abs() + 1e-4).all(), i
        dist = (l_all - l1).abs().amax(1)
        others = torch.arange(40, device=dist.device) != i
        assert (dist[others] > dist[i]).all(), i
        exact_rows += int(v == float(values[i]) and torch.equal(l1[0], l_all[i]))
    print(f"{name}: {exact_rows}/14 single-position evaluations bit-equal to their batch row")
    # fp32 module on the oracle's encoding
    enc = [fo.encode(r) for r in recs]
    grids = torch.from_numpy(np.concatenate([np.stack([e[0][0] for e in enc]), np.stack([e[0][1] for e in enc])])
                             .astype(np.float32)).reshape(80, 1, 40, 10).cuda()
    extras = torch.from_numpy(np.stack([e[1] for e in enc]).astype(np.float32)).cuda()
    with torch.no_grad():
        out = net.forward_packed(grids, extras)
    v_ref, l_ref = out[0].reshape(-1), out[1][:, :POLICY_SIZE]
    v_got, l_got = ai._evaluate_packed(net, recs)
    assert (v_got - v_ref).abs().max().item() < 0.03
    assert (l_got - l_ref).abs().max().item() < 0.05 * l_ref.abs().max().item() + 0.05
    assert np.allclose(torch.softmax(l_got, 1).cpu().numpy().reshape(40, 27, 39, 11), policies, rtol=0, atol=0)


def test_caches_follow_a_reloaded_network():
    """Checkpoint after checkpoint through the same variable, the old network freed each time (a new one may then
    sit at the same address with the same parameter versions): evaluate_positions() and analyse() must answer with
    the network they are given, i.e. equal what a freshly built evaluator / engine returns."""
    import gc
    import torch
    from oracle.pin_against_reference import random_midgame
    from tetris_reinforcement_learning_b200 import ai, architectures as arch
    mc = arch.AlphaSameConfig(blocks=2, filters=16)
    cfg = Config(visual=False, ruleset="s2", model="pytorch", model_config=mc, MAX_ITER=6, training=False)
    torch.manual_seed(3)
    checkpoints = [arch.AlphaSame(mc).state_dict() for _ in range(6)]
    recs = random_midgame(np.random.default_rng(2), 8, 4)
    ai.release_cached_engines()
    seen_ids, reused, values = set(), 0, []
    net = None
    for sd in checkpoints:
        del net
        gc.collect()
        net = arch.AlphaSame(mc)
        net.load_state_dict(sd)
        net = net.to("cuda:0").eval()
        reused += int(id(net) in seen_ids)
        seen_ids.add(id(net))
        v, p = ai.evaluate_positions(cfg, recs, net)
        res = ai.analyse(cfg, recs, net, seed=1)
        ai.release_cached_engines()
        v_new, p_new = ai.evaluate_positions(cfg, recs, net)
        res_new = ai.analyse(cfg, recs, net, seed=1)
        assert np.array_equal(v, v_new) and np.array_equal(p, p_new)
        for a, b in zip(res, res_new):
            assert (a is None) == (b is None)
            if a is not None:
                assert np.array_equal(a.priors, b.priors) and np.array_equal(a.visits, b.visits)
                assert a.root_value == b.root_value
        values.append(v)
    assert all(not np.array_equal(values[i], values[j]) for i in range(len(values)) for j in range(i))
    print(f"{reused} of {len(checkpoints)} networks reused an earlier network's address")
