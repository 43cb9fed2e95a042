"""GPU tests of the status plumbing of the self-play path: every overflow the device can hit is forced and
must come back as its own TRL_ST_* bit in ctl.status and as an exception from the public calls (the reference
asserts in these situations, ai.py:417,1347)."""
import numpy as np
import pytest

from test_gpu_search import fake_evaluator_torch

pytestmark = pytest.mark.gpu

ST_QUEUE_OVERFLOW, ST_MOVES_TRUNC, ST_SAMPLE_OVERFLOW, ST_ARENA_FULL = 0x1, 0x2, 0x20, 0x40


def _cfg(**kw):
    from tetris_reinforcement_learning_b200.config import Config
    base = dict(visual=False, ruleset="s2", model="pytorch", MAX_ITER=6, training=True, use_playout_cap_randomization=False)
    base.update(kw)
    return Config(**base)


@pytest.mark.parametrize("compact", [True, False])
def test_fifo_overflow_inside_a_search_reaches_ctl_status(compact):
    """The exploration FIFO of the leaf enumeration (movegen_list_kernel / movegen_warp_kernel) lowered to 2 entries:
    every search overflows it and the bit must arrive in ctl.status through both enumeration paths."""
    import torch
    from tetris_reinforcement_learning_b200 import _native
    from tetris_reinforcement_learning_b200.selfplay import EngineStatusError, SelfPlayEngine
    lib = _native.lib()
    eng = SelfPlayEngine(_cfg(), fake_evaluator_torch(torch.device("cuda:0")), 32, seed=1, use_cuda_graph=False,
                         compact_movegen=compact, max_rounds=2)
    assert lib.trl_debug_movegen_fifo_limit(2) == 0
    try:
        eng.step(4)
        torch.cuda.synchronize()
    finally:
        assert lib.trl_debug_movegen_fifo_limit(0) == 0     # back to the full capacity
    st = eng.get_ctl()["status"]
    assert (st & ST_QUEUE_OVERFLOW).all()
    with pytest.raises(EngineStatusError, match="QUEUE_OVERFLOW"):
        eng.check_status()
    # and a clean engine afterwards stays clean
    eng2 = SelfPlayEngine(_cfg(), fake_evaluator_torch(torch.device("cuda:0")), 32, seed=1, use_cuda_graph=False, max_rounds=2)
    eng2.step(20)
    assert eng2.status_bits() == 0


def test_sample_ring_overflow_has_its_own_bit():
    import torch
    from tetris_reinforcement_learning_b200.selfplay import EngineStatusError, SelfPlayEngine
    eng = SelfPlayEngine(_cfg(), fake_evaluator_torch(torch.device("cuda:0")), 16, seed=2, use_cuda_graph=False,
                         sample_cap=1, max_rounds=3)
    eng.step(6)                                   # 16 searches finish, one record fits
    st = eng.get_ctl()["status"]
    assert int((st & ST_SAMPLE_OVERFLOW != 0).sum()) == 15 and not (st & ST_MOVES_TRUNC).any()
    with pytest.raises(EngineStatusError, match="overflowed"):
        eng.drain()


def test_node_arena_overflow_has_its_own_bit():
    import torch
    from tetris_reinforcement_learning_b200.selfplay import SelfPlayEngine
    eng = SelfPlayEngine(_cfg(), fake_evaluator_torch(torch.device("cuda:0")), 16, seed=3, use_cuda_graph=False,
                         node_cap=40, max_rounds=3)
    eng.step(6)
    st = eng.get_ctl()["status"]
    assert (st & ST_ARENA_FULL).any() and not (st & ST_QUEUE_OVERFLOW).any()


def test_generate_games_raises_on_device_status():
    import torch
    from tetris_reinforcement_learning_b200 import _native, ai
    from tetris_reinforcement_learning_b200.selfplay import EngineStatusError
    lib = _native.lib()
    assert lib.trl_debug_movegen_fifo_limit(2) == 0
    try:
        with pytest.raises(EngineStatusError):
            ai.generate_games(_cfg(), fake_evaluator_torch(torch.device("cuda:0")), 8, seed=4, dtype=torch.float32, max_steps=64)
    finally:
        assert lib.trl_debug_movegen_fifo_limit(0) == 0


def test_save_all_with_random_openings_generates_a_set(tmp_path, monkeypatch):
    """ADVICE r1: save_all + use_random_starting_moves used to store records of one-iteration opening searches with
    zero visits, which crashed the target construction (assert total != 0)."""
    import torch
    from tetris_reinforcement_learning_b200 import ai
    monkeypatch.setenv("TRL_STORAGE", str(tmp_path / "Storage"))   # generate_games numbers the set from <data_dir>
    cfg = _cfg(use_random_starting_moves=True, save_all=True, use_playout_cap_randomization=True, MAX_ITER=8)
    for compact in (False, True):
        data, stats = ai.generate_games(cfg, fake_evaluator_torch(torch.device("cuda:0")), 12, seed=5, dtype=torch.float32,
                                        compact=compact)
        assert len(stats) == 12 and len(data) > 0
