"""CPU tests of Config.engine_devices: parsing and validation, the game-id shard arithmetic of generate_games /
battle_networks, the contiguous blocks of analyse / evaluate_positions, and Config.copy() carrying the knob."""
import pytest

from tetris_reinforcement_learning_b200 import devices
from tetris_reinforcement_learning_b200.config import Config


def test_parse_engine_devices():
    assert devices.parse_engine_devices(None, 8, 3) == [3]
    assert devices.parse_engine_devices("all", 4, 0) == [0, 1, 2, 3]
    assert devices.parse_engine_devices([0, 0], 1, 0) == [0, 0]
    assert devices.parse_engine_devices((1, 0, 1), 2, 0) == [1, 0, 1]
    for bad in ("ALL", "cuda:0", [], [0, 2], [-1], [True], [0.0], 0, {0: 1}, [None]):
        with pytest.raises(ValueError):
            devices.parse_engine_devices(bad, 2, 0)
    with pytest.raises(ValueError):
        devices.parse_engine_devices("all", 0, 0)


def test_split_evenly():
    assert devices.split_evenly(10, 3) == [4, 3, 3]
    assert devices.split_evenly(2, 4) == [1, 1, 0, 0]
    assert devices.split_evenly(0, 2) == [0, 0]
    with pytest.raises(ValueError):
        devices.split_evenly(3, 0)


def _ids(shard):
    return [shard["first_game_id"] + j * shard["game_id_stride"] for j in range(shard["num_games"])]


@pytest.mark.parametrize("n,concurrent,first,stride,d", [(10, 10, 0, 1, 2), (13, 5, 0, 1, 4), (7, 7, 3, 8, 3),
                                                          (1, 1, 0, 1, 8), (100, 64, 2, 4, 8), (5, 1, 0, 1, 2)])
def test_shard_games_union_is_one_device(n, concurrent, first, stride, d):
    shards = devices.shard_games(n, concurrent, first, stride, d)
    one = _ids(devices.shard_games(n, concurrent, first, stride, 1)[0])
    assert one == [first + i * stride for i in range(n)]
    ids = [i for sh in shards for i in _ids(sh)]
    assert len(ids) == len(set(ids)) and sorted(ids) == one      # disjoint, union = one device's ids
    assert sum(sh["num_games"] for sh in shards) == n
    for sh in shards:
        assert sh["game_id_stride"] == stride * d and 1 <= sh["concurrent"] <= sh["num_games"]
    assert sum(sh["concurrent"] for sh in shards) >= min(concurrent, n)


def test_shard_games_composes_with_ranks():
    """Rank r of W (first_game_id=r, game_id_stride=W) sharded over D devices: the ranks' shards together are the
    ids 0 .. W*n-1 of one device, each exactly once."""
    W, D, n = 4, 3, 11
    ids = [i for r in range(W) for sh in devices.shard_games(n, n, r, W, D) for i in _ids(sh)]
    assert sorted(ids) == list(range(W * n))


def test_contiguous_blocks():
    assert devices.contiguous_blocks(10, 3) == [(0, 4), (4, 7), (7, 10)]
    assert devices.contiguous_blocks(1, 2) == [(0, 1), (1, 1)]
    assert devices.contiguous_blocks(0, 2) == [(0, 0), (0, 0)]


def test_config_knob_default_and_copy():
    c = Config()
    assert c.engine_devices is None and Config.engine_devices is None
    c.engine_devices = [0, 0]
    assert c.copy().engine_devices == [0, 0]
    c.engine_devices = "all"
    d = c.copy()
    assert d.engine_devices == "all" and Config().engine_devices is None
