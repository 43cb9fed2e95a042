"""The I piece's packed kick passes in the closure search of the movegen sweep (csrc/movegen_warp.cu, kick_pass_pair_i):
I-heavy calls on cave boards and on the config-2 boards, in the pass form, compared bit for bit with the one-kernel form
(the generic kick loop over the constant-memory table) and with the C oracle.  Cave boards make the I piece kick a lot,
so the |kx| = 2 kicks of every packed pass, whose tests read the target plane up to the bit below its other half, are
reached."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from tetris_reinforcement_learning_b200 import synth  # noqa: E402
from tetris_reinforcement_learning_b200.const import MASK_WORDS, MINOS  # noqa: E402

I, T, NONE = MINOS.index("I"), MINOS.index("T"), 255


def _lib():
    from tetris_reinforcement_learning_b200 import _native
    return _native.lib()


@pytest.fixture
def form():
    """Select a launch form of the warp kernels for the duration of a test."""
    L = _lib()
    L.trl_movegen_select_kernel(1)
    yield L.trl_movegen_warp_form
    L.trl_movegen_select_kernel(-1)
    L.trl_movegen_warp_form(-1)


def _i_heavy_calls(caves):
    """I as the current piece, as the hold piece, as both, next to a T, next to a missing piece, on every board."""
    boards, cur, alt = synth.movegen_workload(12_000, seed=91, caves=caves)
    cur = cur.copy(); alt = alt.copy()
    k = np.arange(cur.size)
    alt[k % 3 == 0] = I
    cur[k % 3 == 1] = I
    cur[k % 13 == 2] = I; alt[k % 13 == 2] = I
    cur[k % 13 == 5] = I; alt[k % 13 == 5] = T
    cur[k % 13 == 6] = T; alt[k % 13 == 6] = I
    cur[k % 13 == 7] = NONE; alt[k % 13 == 7] = I
    cur[k % 13 == 8] = I; alt[k % 13 == 8] = NONE
    return np.ascontiguousarray(boards), cur, alt


@pytest.fixture(scope="module", params=[True, False], ids=["caves", "config2"])
def i_heavy(request, oracle):
    boards, cur, alt = _i_heavy_calls(request.param)
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


@pytest.mark.parametrize("want_mask", [True, False], ids=["mask", "moves"])
def test_i_heavy_passes_match_form1_and_oracle(form, i_heavy, want_mask):
    boards, cur, alt, want = i_heavy
    want_masks, want_n, want_st, _ = want
    cap = 0 if want_mask else 256
    form(1)
    one = _device_run(boards, cur, alt, want_mask, cap)
    form(2)
    two = _device_run(boards, cur, alt, want_mask, cap)
    for k in one:
        assert np.array_equal(one[k], two[k]), k
    trunc = np.uint32(2)   # TRL_ST_MOVES_TRUNC
    assert np.array_equal(two["status"] & ~trunc, want_st)
    assert np.array_equal(two["n"], want_n)
    if want_mask:
        bad = np.flatnonzero((two["mask"] != want_masks).any(axis=1))
        assert bad.size == 0, f"{bad.size} masks differ, first calls {bad[:5]}"
    else:
        for j in range(0, want_n.size, 5):
            ref = np.flatnonzero(np.unpackbits(want_masks[j].view(np.uint8), bitorder="little"))[:cap]
            assert np.array_equal(two["moves"][j, :ref.size], ref), j
