"""CPU suite for the byte-coded move lists of trl_movegen_host_boards (format in include/trl.h): a plain Python
encoder, the vectorised decoder move_generation.decode_move_codes, and the argument checks of the entry point, which
return before any CUDA call."""
import numpy as np
import pytest

from tetris_reinforcement_learning_b200.const import POLICY_SIZE
from tetris_reinforcement_learning_b200.move_generation import decode_move_codes


def encode_reference(lists):
    """One call after the other, one move after the other: gap d to the previous move (-1 first); d <= 255 is a
    byte, a larger d is byte 0 plus d in the escape stream."""
    codes, escapes = [], []
    for moves in lists:
        prev = -1
        for m in moves:
            d = int(m) - prev
            assert 1 <= d <= POLICY_SIZE
            if d <= 255:
                codes.append(d)
            else:
                codes.append(0)
                escapes.append(d)
            prev = int(m)
    n_moves = np.array([len(m) for m in lists], dtype=np.uint16)
    return np.array(codes, dtype=np.uint8), np.array(escapes, dtype=np.uint16), n_moves


def _roundtrip(lists):
    codes, escapes, n_moves = encode_reference(lists)
    moves, offsets = decode_move_codes(codes, escapes, n_moves)
    assert moves.dtype == np.uint16 and offsets.dtype == np.uint64
    assert moves.size == sum(len(m) for m in lists)
    for i, want in enumerate(lists):
        o = int(offsets[i])
        assert np.array_equal(moves[o:o + len(want)], np.asarray(want, dtype=np.uint16)), i
    return codes, escapes


def test_edge_gaps_and_first_moves():
    lists = [
        [254, 509],                 # d = 255 (byte), then 255
        [255, 511],                 # d = 256 (escape), then 256
        [0, 1, 2],                  # first move 0: d = 1
        [11582],                    # first move 11582: d = 11583, the largest gap
        [],                         # empty call in the middle
        [0, 11582],                 # d = 11582 after a first move of 0
        [],
    ]
    codes, escapes = _roundtrip(lists)
    assert list(codes[:4]) == [255, 255, 0, 0]
    assert list(escapes[:3]) == [256, 256, 11583]


def test_all_empty_and_no_calls():
    moves, offsets = decode_move_codes(np.empty(0, np.uint8), np.empty(0, np.uint16), np.zeros(5, np.uint16))
    assert moves.size == 0 and list(offsets) == [0] * 5
    moves, offsets = decode_move_codes(np.empty(0, np.uint8), np.empty(0, np.uint16), np.zeros(0, np.uint16))
    assert moves.size == 0 and offsets.size == 0


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_random_ascending_lists(seed):
    rng = np.random.default_rng(seed)
    lists = []
    for _ in range(400):
        k = int(rng.choice([0, 1, 2, 5, 40, 300, 1200]))
        hi = int(rng.integers(k, 1300)) if rng.random() < 0.5 else POLICY_SIZE   # dense lists, or sparse ones
        lists.append(np.sort(rng.choice(hi, size=k, replace=False)).tolist())
    codes, escapes = _roundtrip(lists)
    assert (codes == 0).sum() == escapes.size and escapes.size > 0


def test_decoder_rejects_inconsistent_streams():
    codes, escapes, n_moves = encode_reference([[300, 301]])
    with pytest.raises(ValueError):
        decode_move_codes(codes, escapes[:0], n_moves)
    with pytest.raises(ValueError):
        decode_move_codes(codes, escapes, np.array([3], np.uint16))


@pytest.fixture(scope="module")
def lib():
    from tetris_reinforcement_learning_b200 import _native, build
    build.build()
    return _native.lib()


def test_bad_arguments_are_rejected_without_a_gpu(lib):
    import ctypes
    b = np.zeros((2, 40), np.uint16)
    idx = np.zeros(4, np.uint32)
    cur = np.zeros(4, np.uint8)
    codes = np.zeros(64, np.uint8)
    esc = np.zeros(64, np.uint16)
    nm = np.zeros(4, np.uint16)
    fi = np.zeros(4, np.uint32)
    fs = np.zeros(4, np.uint32)
    tot = (ctypes.c_uint64 * 3)()
    t = ctypes.addressof(tot)
    p = lambda a: a.ctypes.data  # noqa: E731
    good = [p(b), 2, p(idx), p(cur), p(cur), 4, p(codes), 64, p(esc), 64, p(nm), p(fi), p(fs), 4, t, t + 8, t + 16]
    for k in (0, 2, 3, 4, 6, 8, 10, 11, 12, 14, 15, 16):   # every pointer, NULL in turn
        args = list(good)
        args[k] = None
        assert lib.trl_movegen_host_boards(*args) == -1, k
    args = list(good); args[5] = -1                          # n < 0
    assert lib.trl_movegen_host_boards(*args) == -1
    for nb in (0, -3):                                       # n > 0 without boards
        args = list(good); args[1] = nb
        assert lib.trl_movegen_host_boards(*args) == -1


def test_wrapper_validates_shapes_and_dtypes():
    from tetris_reinforcement_learning_b200.move_generation import movegen_host_boards
    b = np.zeros((3, 40), np.uint16)
    c = np.zeros(4, np.uint8)
    with pytest.raises(ValueError):
        movegen_host_boards(b, np.zeros(4, np.float32), c, c)
    with pytest.raises(ValueError):
        movegen_host_boards(b, np.zeros(3, np.uint32), c, c)
    with pytest.raises(ValueError):
        movegen_host_boards(np.zeros((3, 39), np.uint16), np.zeros(4, np.uint32), c, c)
    with pytest.raises(ValueError):
        movegen_host_boards(b, np.array([0, 1, 2, 1 << 32], np.int64), c, c)
    with pytest.raises(ValueError):
        movegen_host_boards(b, np.array([0, -1, 2, 1], np.int64), c, c)
    with pytest.raises(ValueError):
        movegen_host_boards(b, np.zeros(4, np.uint32), c, c, out={"codes": np.zeros(16, np.uint16)})
