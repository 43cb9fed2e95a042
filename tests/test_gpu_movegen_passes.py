"""The pass form of the movegen sweep (csrc/movegen_warp.cu, DESIGN §3.1): pass 1 defers T searches with mixed flags,
pass 2 runs the T order analysis, pass 3 the exact T search, and the legacy route redoes whole calls.  Every output is
compared bit for bit with the one-kernel form and with the C oracle."""
import ctypes
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from tetris_reinforcement_learning_b200 import synth  # noqa: E402
from tetris_reinforcement_learning_b200.const import MASK_WORDS  # noqa: E402

T, NONE = 6, 255


def _lib():
    from tetris_reinforcement_learning_b200 import _native
    return _native.lib()


def _pass_counts():
    c = (ctypes.c_uint32 * 3)()
    assert _lib().trl_debug_movegen_pass_counts(c) == 0
    return {"deferred": c[0], "undecided": c[1], "legacy": c[2]}


def _fifo_fallbacks():
    st = (ctypes.c_uint64 * 16)()
    assert _lib().trl_debug_movegen_fast_stats(st) == 0
    return int(st[1])


@pytest.fixture
def form():
    """Select a launch form of the warp kernels for the duration of a test."""
    L = _lib()
    L.trl_movegen_select_kernel(1)
    yield L.trl_movegen_warp_form
    L.trl_movegen_select_kernel(-1)
    L.trl_movegen_warp_form(-1)
    assert L.trl_debug_movegen_partial_cap(0) == 0


def _t_heavy_calls():
    """The adversarial cave boards with every 5th hold piece a T, then T as the current piece, as the hold piece, as
    both, next to a missing piece, and calls with no piece at all."""
    boards, cur, alt = synth.movegen_workload(20_000, seed=77, caves=True)
    cur = cur.copy(); alt = alt.copy()
    alt[::5] = T
    k = np.arange(cur.size)
    cur[k % 23 == 1] = T
    alt[k % 23 == 2] = T; cur[k % 23 == 2] = np.where(cur[k % 23 == 2] == T, 0, cur[k % 23 == 2])
    cur[k % 23 == 3] = T; alt[k % 23 == 3] = T
    cur[k % 23 == 4] = NONE; alt[k % 23 == 4] = T
    cur[k % 23 == 5] = T; alt[k % 23 == 5] = NONE
    cur[k % 23 == 6] = NONE; alt[k % 23 == 6] = NONE
    return np.ascontiguousarray(boards), cur, alt


def _moves_from_mask(mask_row):
    return np.flatnonzero(np.unpackbits(mask_row.view(np.uint8), bitorder="little"))


@pytest.fixture(scope="module")
def t_heavy(oracle):
    boards, cur, alt = _t_heavy_calls()
    want = oracle.movegen_batch(boards, cur, alt, n_threads=os.cpu_count() or 1)
    return boards, cur, alt, want


def _device_run(boards, cur, alt, want_mask, moves_cap=0):
    import torch
    from tetris_reinforcement_learning_b200 import move_generation
    dev = torch.device("cuda:0")
    n = cur.size
    d_b = torch.from_numpy(boards.view(np.int16)).to(dev)
    d_c, d_a = torch.from_numpy(cur).to(dev), torch.from_numpy(alt).to(dev)
    mask = torch.full((n, MASK_WORDS), -1, dtype=torch.int32, device=dev) if want_mask else None
    moves = torch.full((n, moves_cap), -1, dtype=torch.int16, device=dev) if moves_cap else None
    d_n = torch.full((n,), -1, dtype=torch.int16, device=dev)
    d_st = torch.full((n,), -1, dtype=torch.int32, device=dev)
    move_generation.movegen_device(d_b, d_c, d_a, mask, moves, d_n, d_st)
    torch.cuda.synchronize()
    out = {"n": d_n.cpu().numpy().view(np.uint16), "status": d_st.cpu().numpy().view(np.uint32)}
    if want_mask:
        out["mask"] = mask.cpu().numpy().view(np.uint32)
    if moves_cap:
        out["moves"] = moves.cpu().numpy().view(np.uint16)
    return out


def _check_against_oracle(out, want, moves_cap=0):
    want_masks, want_n, want_st, _ = want
    trunc = np.uint32(2)   # TRL_ST_MOVES_TRUNC: the list of a call with more moves than moves_cap is cut, n is the full count
    assert np.array_equal(out["status"] & ~trunc, want_st)
    assert np.array_equal((out["status"] & trunc) != 0, want_n > moves_cap if moves_cap else np.zeros(want_n.size, bool))
    assert np.array_equal(out["n"], want_n)
    if "mask" in out:
        bad = np.flatnonzero((out["mask"] != want_masks).any(axis=1))
        assert bad.size == 0, f"{bad.size} masks differ, first calls {bad[:5]}"
    if moves_cap:
        for j in range(0, want_n.size, 7):
            ref = _moves_from_mask(want_masks[j])[:moves_cap]
            assert np.array_equal(out["moves"][j, :ref.size], ref), j


def test_passes_mask_mode_match_form1_and_oracle(form, t_heavy):
    boards, cur, alt, want = t_heavy
    form(1)
    one = _device_run(boards, cur, alt, want_mask=True)
    form(2)
    two = _device_run(boards, cur, alt, want_mask=True)
    counts = _pass_counts()
    for k in one:
        assert np.array_equal(one[k], two[k]), k
    _check_against_oracle(two, want)
    assert counts["deferred"] > 100 and counts["undecided"] > 0, counts   # every pass had work


def test_passes_moves_mode_match_form1_and_oracle(form, t_heavy):
    """No mask output: the partial masks of the deferred calls live in the bounded scratch."""
    boards, cur, alt, want = t_heavy
    form(1)
    one = _device_run(boards, cur, alt, want_mask=False, moves_cap=256)
    form(2)
    two = _device_run(boards, cur, alt, want_mask=False, moves_cap=256)
    assert _pass_counts()["deferred"] > 100
    for k in one:
        assert np.array_equal(one[k], two[k]), k
    _check_against_oracle(two, want, moves_cap=256)


def test_passes_host_compact_match_oracle(form, t_heavy):
    from tetris_reinforcement_learning_b200 import move_generation
    boards, cur, alt, want = t_heavy
    want_masks, want_n, want_st, _ = want
    form(2)
    res = move_generation.movegen_host_compact(boards, cur, alt)
    assert np.array_equal(res["n_moves"], want_n) and np.array_equal(res["status"], want_st)
    for i in range(0, cur.size, 3):
        seg = res["moves"][int(res["offsets"][i]): int(res["offsets"][i]) + int(res["n_moves"][i])]
        assert np.array_equal(seg, _moves_from_mask(want_masks[i])), i


def test_pass_counts_on_config2_boards(form):
    """Pass 2 sees every deferred call and leaves a subset to pass 3; what reaches the FIFO form (pass 3 plus the
    legacy route) is what the one-kernel form sends there; the config-2 boards need no legacy route."""
    boards, cur, alt = synth.movegen_workload(20_000)
    form(1)
    _fifo_fallbacks()                       # reset
    one = _device_run(boards, cur, alt, want_mask=True)
    fallbacks = _fifo_fallbacks()
    form(2)
    two = _device_run(boards, cur, alt, want_mask=True)
    counts = _pass_counts()
    for k in one:
        assert np.array_equal(one[k], two[k]), k
    assert counts["legacy"] == 0, counts
    assert counts["deferred"] >= counts["undecided"] > 0, counts
    assert counts["undecided"] + counts["legacy"] == fallbacks, (counts, fallbacks)


@pytest.mark.parametrize("want_mask", [True, False])
def test_partial_mask_overflow_takes_legacy_route(form, t_heavy, want_mask):
    """With room for only 100 partial masks every further deferred call is redone by the legacy route: same outputs."""
    boards, cur, alt, want = t_heavy
    L = _lib()
    form(2)
    full = _device_run(boards, cur, alt, want_mask=want_mask, moves_cap=0 if want_mask else 256)
    n_deferred = _pass_counts()["deferred"]
    assert L.trl_debug_movegen_partial_cap(100) == 0
    low = _device_run(boards, cur, alt, want_mask=want_mask, moves_cap=0 if want_mask else 256)
    counts = _pass_counts()
    assert counts["deferred"] == 100 and counts["legacy"] >= n_deferred - 100, (counts, n_deferred)
    for k in full:
        assert np.array_equal(full[k], low[k]), k
    _check_against_oracle(low, want, moves_cap=0 if want_mask else 256)


# Boards on which the current piece, which is not a T, climbs from its spawn pocket by wall kicks to origin rows
# <= 11: above the row window of the closure search, so the call takes the legacy route.
CLIMB_I = [0x000] * 11 + [0x066, 0x104, 0x166, 0x111, 0x001, 0x087, 0x205, 0x280, 0x100, 0x368, 0x00A, 0x0CE, 0x28C,
                          0x140, 0x388, 0x3C8, 0x03F, 0x2CA, 0x0B0, 0x0B0, 0x1AC, 0x312, 0x204, 0x120, 0x3A0, 0x3E5,
                          0x046, 0x32C, 0x128]
CLIMB_L = [0x000] * 7 + [0x193, 0x0A4, 0x041, 0x044, 0x023, 0x229, 0x08B, 0x016, 0x283, 0x105, 0x001, 0x300, 0x085,
                         0x077, 0x051, 0x150, 0x0D0, 0x12D, 0x021, 0x220, 0x001, 0x191, 0x383, 0x01D, 0x208, 0x160,
                         0x154, 0x0F8, 0x0D2, 0x0B0, 0x220, 0x050, 0x068]


def test_window_climb_of_a_non_t_piece_takes_legacy_route(form, oracle):
    rows = np.array([CLIMB_I, CLIMB_L, CLIMB_I, CLIMB_L], np.uint16)
    cur = np.array([4, 1, 4, 1], np.uint8)
    alt = np.array([4, 1, T, T], np.uint8)
    want = oracle.movegen_batch(rows, cur, alt)
    placed_rows = np.unpackbits(want[0].view(np.uint8), axis=1, bitorder="little")[:, :27 * 39 * 11]
    assert placed_rows.reshape(4, 27, 39, 11)[:, :, :12].any(axis=(1, 2, 3)).all()   # placements at origin rows <= 11
    form(2)
    out = _device_run(rows, cur, alt, want_mask=True)
    assert _pass_counts()["legacy"] == 4
    _check_against_oracle(out, want)
