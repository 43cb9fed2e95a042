"""trl_movegen_host_boards (csrc/movegen_codes.cu): movegen over shared boards with byte-coded move lists.

700 000 calls (100 000 boards x 7 pieces) are 5.3 chunks of 131072 calls, so the ring of four host streams wraps and
the last chunk is partial.  The decoded lists are compared with the masks of trl_movegen_host on the expanded boards,
with trl_movegen_host_compact and, on a subset, with the C oracle; the raw bytes with a Python encoder."""
import ctypes
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from tetris_reinforcement_learning_b200 import move_generation as mg, synth  # noqa: E402

N_BOARDS = 100_000
NONE = 255


def _pieces(n_boards):
    i = np.repeat(np.arange(n_boards), 7)
    k = np.tile(np.arange(7), n_boards)
    return k.astype(np.uint8), ((k + 1 + i % 6) % 7).astype(np.uint8)


def _workload(pattern):
    caves = pattern == "caves"
    boards = synth.random_boards(N_BOARDS, seed=7, caves=caves)
    cur, alt = _pieces(N_BOARDS)
    if pattern == "random":   # repeated and unused boards
        idx = np.random.default_rng(5).integers(0, N_BOARDS, size=7 * N_BOARDS).astype(np.uint32)
    else:
        idx = np.repeat(np.arange(N_BOARDS, dtype=np.uint32), 7)
    return boards, idx, cur, alt


def encode_expected(moves, n_moves):
    """Vectorised form of the format in include/trl.h, from call-ordered lists."""
    m = moves.astype(np.int64)
    start = np.cumsum(n_moves.astype(np.int64)) - n_moves
    prev = np.empty_like(m)
    prev[1:] = m[:-1]
    first = start[n_moves > 0]
    prev[first] = -1
    d = m - prev
    return np.where(d <= 255, d, 0).astype(np.uint8), d[d > 255].astype(np.uint16)


def encode_reference(lists):
    """Plain Python encoder: one move after the other."""
    codes, escapes = [], []
    for moves in lists:
        prev = -1
        for mv in moves:
            d = int(mv) - prev
            codes.append(d if d <= 255 else 0)
            if d > 255:
                escapes.append(d)
            prev = int(mv)
    return np.array(codes, np.uint8), np.array(escapes, np.uint16)


def _mask_lists_equal(masks, moves, offsets, n_moves, lo, hi):
    """Calls lo..hi-1: the decoded lists are the set bits of their masks, ascending."""
    bits = np.unpackbits(masks[lo:hi].view(np.uint8), axis=1, bitorder="little")
    _, col = np.nonzero(bits)
    a = int(offsets[lo])
    b = int(offsets[hi - 1]) + int(n_moves[hi - 1])
    return np.array_equal(col.astype(np.uint16), moves[a:b])


@pytest.fixture(scope="module", params=["repeat", "random", "caves"])
def run(request):
    boards, idx, cur, alt = _workload(request.param)
    raw = mg.movegen_host_boards(boards, idx, cur, alt, decode=False)
    raw = {k: v.copy() for k, v in raw.items()}
    res = mg.movegen_host_boards(boards, idx, cur, alt)
    return request.param, boards, idx, cur, alt, raw, res


def test_against_masks_and_compact(run):
    _, boards, idx, cur, alt, raw, res = run
    exp = boards[idx]
    ref = mg.movegen_host(exp, cur, alt, want_mask=True)
    assert np.array_equal(res["n_moves"], ref["n_moves"])
    assert np.array_equal(res["status"], ref["status"])
    assert res["total"] == int(ref["n_moves"].sum())
    n = cur.size
    for lo in range(0, n, 25_000):
        assert _mask_lists_equal(ref["mask_bits"], res["moves"], res["offsets"], res["n_moves"], lo, min(n, lo + 25_000)), lo
    del ref
    comp = mg.movegen_host_compact(exp, cur, alt)
    assert np.array_equal(comp["n_moves"], res["n_moves"]) and comp["total"] == res["total"]
    nm = res["n_moves"].astype(np.int64)
    pos = np.repeat(comp["offsets"].astype(np.int64) - res["offsets"].astype(np.int64), nm) + np.arange(res["total"])
    assert np.array_equal(comp["moves"][pos], res["moves"])


def test_bytes_match_the_encoders(run):
    pattern, boards, idx, cur, alt, raw, res = run
    codes, escapes = encode_expected(res["moves"], res["n_moves"])
    assert np.array_equal(raw["codes"], codes)
    assert np.array_equal(raw["escapes"], escapes)
    if pattern == "caves":
        assert escapes.size > 0
    # the plain encoder on a slice of calls spanning a chunk boundary: its bytes sit at the slice's offsets
    lo, hi = 131_072 - 2_500, 131_072 + 2_500
    lists = [res["moves"][int(res["offsets"][i]):int(res["offsets"][i]) + int(res["n_moves"][i])] for i in range(lo, hi)]
    c_ref, e_ref = encode_reference(lists)
    c0 = int(res["offsets"][lo])
    e0 = int((raw["codes"][:c0] == 0).sum())
    assert np.array_equal(raw["codes"][c0:c0 + c_ref.size], c_ref)
    assert np.array_equal(raw["escapes"][e0:e0 + e_ref.size], e_ref)
    # a second run gives the same bytes
    again = mg.movegen_host_boards(boards, idx, cur, alt, decode=False)
    for k in raw:
        assert np.array_equal(again[k], raw[k]), k


def test_oracle_subset(run, oracle):
    _, boards, idx, cur, alt, raw, res = run
    sel = np.arange(0, cur.size, cur.size // 5000)[:5000]
    want_masks, want_n, want_st, _ = oracle.movegen_batch(boards[idx[sel]], cur[sel], alt[sel],
                                                          n_threads=os.cpu_count() or 1)
    assert np.array_equal(res["n_moves"][sel], want_n)
    assert np.array_equal(res["status"][sel], want_st)
    for j, i in enumerate(sel):
        ref = np.flatnonzero(np.unpackbits(want_masks[j].view(np.uint8), bitorder="little"))
        o = int(res["offsets"][i])
        assert np.array_equal(res["moves"][o:o + int(res["n_moves"][i])], ref), i


def test_mask_mode_encoder_gives_the_same_bytes():
    """The A/B variant (encoder reading the sweep's masks) against the default (reading its move lists)."""
    from tetris_reinforcement_learning_b200 import _native
    L = _native.lib()
    L.trl_debug_movegen_codes_source.argtypes = [ctypes.c_int]
    L.trl_debug_movegen_codes_source.restype = None
    boards, idx, cur, alt = _workload("caves")
    idx, cur, alt = idx[:300_000], cur[:300_000], alt[:300_000]
    want = {k: v.copy() for k, v in mg.movegen_host_boards(boards, idx, cur, alt, decode=False).items()}
    L.trl_debug_movegen_codes_source(1)
    try:
        got = mg.movegen_host_boards(boards, idx, cur, alt, decode=False)
    finally:
        L.trl_debug_movegen_codes_source(0)
    for k in want:
        assert np.array_equal(got[k], want[k]), k


def test_flagged_calls():
    boards = synth.random_boards(2_000, seed=3)
    blocked = boards[:40].copy()
    blocked[:, 8:] = 0x3FE                      # every row from the spawn area down full but for column 0
    boards = np.concatenate([boards, blocked])
    cur, alt = _pieces(boards.shape[0])
    idx = np.repeat(np.arange(boards.shape[0], dtype=np.uint32), 7)
    k = np.arange(cur.size)
    cur[k % 11 == 3] = NONE
    alt[k % 11 == 3] = NONE
    cur[k % 17 == 4] = NONE                     # alt only
    ref = mg.movegen_host(boards[idx], cur, alt, want_mask=False)
    raw = mg.movegen_host_boards(boards, idx, cur, alt, decode=False)
    want = np.flatnonzero(ref["status"])
    assert np.array_equal(raw["flag_index"], want)
    assert np.array_equal(raw["flag_status"], ref["status"][want])
    none = (cur == NONE) & (alt == NONE)
    assert np.all(raw["flag_status"][np.isin(want, np.flatnonzero(none))] & 0x4)   # TRL_ST_NO_PIECE
    assert np.isin(np.flatnonzero(none), want).all()
    assert np.all(raw["n_moves"][none] == 0)
    assert np.all(raw["n_moves"][-7 * 40:] == 0)   # nothing spawns on the blocked boards
    assert np.array_equal(raw["n_moves"], ref["n_moves"])


def test_errors_and_recovery():
    boards = synth.random_boards(3_000, seed=4)
    cur, alt = _pieces(3_000)
    idx = np.repeat(np.arange(3_000, dtype=np.uint32), 7)
    good = {k: v.copy() for k, v in mg.movegen_host_boards(boards, idx, cur, alt, decode=False).items()}
    bad = idx.copy()
    bad[12_345] = 3_000
    with pytest.raises(RuntimeError, match="code -1"):
        mg.movegen_host_boards(boards, bad, cur, alt, decode=False)
    bad[12_345] = 0xFFFFFFFF
    with pytest.raises(RuntimeError, match="code -1"):
        mg.movegen_host_boards(boards, bad, cur, alt, decode=False)
    again = mg.movegen_host_boards(boards, idx, cur, alt, decode=False)   # the next valid call is right
    for k in good:
        assert np.array_equal(again[k], good[k]), k
    nc, ne = good["codes"].size, good["escapes"].size
    assert ne > 0
    with pytest.raises(RuntimeError, match="code -1"):
        mg.movegen_host_boards(boards, idx, cur, alt, out={"codes": np.empty(nc - 1, np.uint8)})
    with pytest.raises(RuntimeError, match="code -1"):
        mg.movegen_host_boards(boards, idx, cur, alt, out={"escapes": np.empty(ne - 1, np.uint16)})
    exact = mg.movegen_host_boards(boards, idx, cur, alt, decode=False,
                                   out={"codes": np.empty(nc, np.uint8), "escapes": np.empty(ne, np.uint16)})
    assert np.array_equal(exact["codes"], good["codes"]) and np.array_equal(exact["escapes"], good["escapes"])
    empty = mg.movegen_host_boards(boards, idx[:0], cur[:0], alt[:0])
    assert empty["total"] == 0 and empty["moves"].size == 0 and empty["offsets"].size == 0


def test_second_device_gives_the_same_bytes():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible GPUs")
    boards, idx, cur, alt = _workload("random")
    with torch.cuda.device(0):
        want = {k: v.copy() for k, v in mg.movegen_host_boards(boards, idx, cur, alt, decode=False).items()}
    with torch.cuda.device(1):
        got = mg.movegen_host_boards(boards, idx, cur, alt, decode=False)
    for k in want:
        assert np.array_equal(got[k], want[k]), k
