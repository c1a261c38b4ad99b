"""Game rules: oracle restatement vs the reference's known-answer tests, the compiled
reference and the committed golden vectors; product SWAR header (host build) vs oracle."""
import ctypes as C
import os

import numpy as np
import pytest

from util import step_rnd

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = np.load(os.path.join(ROOT, "tests", "golden", "rules.npz"))


# ---- known-answer tests restated from tests/cpp/move_test.cpp:10-56 ---------------------------
def test_move_codec_known_answers(oracle):
    d0 = oracle.move_decode(0)    # id 0 = a4 -> b4 (move right from (0,0))
    assert list(d0) == [0, -1, 0, 0, 0, 1]
    d48 = oracle.move_decode(48)  # id 48 = base at a4
    assert d48[0] == 1 and d48[1] == 0 and (d48[4], d48[5]) == (0, 0)
    assert oracle.encode_place(2, 3, 1) == 75
    assert oracle.encode_place(3, 1, 2) == 93
    assert oracle.encode_move(1, 2, 2, 2) == 18
    for mid in range(96):
        d = oracle.move_decode(mid)
        back = oracle.encode_place(d[4], d[5], d[1]) if d[0] else oracle.encode_move(*d[2:6])
        assert back == mid


# ---- tests/cpp/game_test.cpp:6-26, 66-123 -----------------------------------------------------
def test_start_position(oracle):
    st = oracle.start()
    mask, lines = oracle.legal(st)
    assert not lines
    assert mask[0] == 0 and mask[1] == 0xFFFF0000 and mask[2] == 0xFFFFFFFF  # exactly the 48 places
    enc = oracle.encode(st)
    assert (enc[:64] == 0).all() and (enc[64:] == 1.0).all()


def test_first_move_encoding_and_frozen_square(oracle):
    for mid in range(48, 96):
        st = oracle.do_move(oracle.start(), mid)
        piece, sq = (mid - 48) // 16, (mid - 48) % 16
        enc = oracle.encode(st)
        assert enc[:64].sum() == 2 and enc[4 * sq + piece] == 1 and enc[4 * sq + 3] == 1
        # the mover is now player 2 (4,4,4); player 1's used type shows 0.75 in slots 3..5
        assert list(enc[64:67]) == [1, 1, 1]
        assert enc[67 + piece] == 0.75 and enc[67:].sum() == 2.75
        mask, lines = oracle.legal(st)
        assert not lines
        for p in range(3):  # frozen square blocks every placement on it
            assert not (mask[(48 + 16 * p + sq) >> 5] >> ((48 + 16 * p + sq) & 31)) & 1


# ---- tests/cpp/game_test.cpp:51-63 and node_test.cpp:29-46 ------------------------------------
def _state(board_bits, to_play, pieces):
    w0 = 0
    for b in board_bits:
        w0 |= 1 << b
    w1 = sum(p << (8 * i) for i, p in enumerate(pieces)) | (to_play << 48)
    return np.array([w0, w1], np.uint64)


def test_terminal_position_with_line(oracle):
    st = _state([2 * 4 + 2, 5 * 4 + 2, 8 * 4 + 2, 8 * 4 + 3], 1, [4, 4, 2, 4, 4, 3])
    mask, lines = oracle.legal(st)
    assert lines and not mask.any()


def test_four_capitals_in_a_row_is_terminal(oracle):
    st = _state([0 * 4 + 2, 1 * 4 + 2, 2 * 4 + 2, 3 * 4 + 2, 3 * 4 + 3], 0, [4, 4, 2, 4, 4, 2])
    mask, lines = oracle.legal(st)
    assert lines and not mask.any()


def test_two_crossing_lines_leave_no_move(oracle):
    """game_test.cpp:508-527: a plus-shaped pair of lines (row + column) has no legal reply."""
    for row in (1, 2):
        for col in (1, 2):
            for piece in range(3):
                st = oracle.start()
                for r, c in ((row - 1, col), (row + 1, col), (row, col - 1), (row, col + 1), (row, col)):
                    st = oracle.do_move(st, oracle.encode_place(r, c, piece))
                mask, lines = oracle.legal(st)
                assert lines and not mask.any()


# ---- golden vectors generated from the compiled reference -------------------------------------
def test_oracle_matches_golden_rules(oracle):
    states, seed = GOLD["states"], int(GOLD["seed"])
    rnd = step_rnd(seed, len(states))
    masks, flags, nxt, enc = oracle.step_batch(states, rnd)
    assert (masks == GOLD["masks"]).all()
    assert (flags == GOLD["flags"]).all()
    assert (nxt == GOLD["next"]).all()
    assert (enc == GOLD["enc"].astype(np.float32)).all()
    fl = GOLD["flags"]
    assert ((fl & 3) == 1).sum() > 100 and ((fl >> 2) & 1).sum() > 1000  # losses and lines covered


def test_oracle_state_generator_reproduces_the_golden_states(oracle):
    """The golden states are the reference harness's play-outs for seed 777 (make_golden.py); the
    oracle's generator, which the larger tests draw their positions from, replays them exactly."""
    states = GOLD["states"]
    assert oracle.gen_states(777, len(states)).tobytes() == states.tobytes()


def test_oracle_matches_compiled_reference_rules(oracle, ref):
    states = ref.gen_states(31337, 300000)
    rnd = step_rnd(5, len(states))
    a = ref.step_batch(states, rnd)
    b = oracle.step_batch(states, rnd)
    for x, y in zip(a, b):
        assert x.tobytes() == y.tobytes()


# ---- the product's SWAR rules header, compiled for the host -----------------------------------
def _shim():
    path = os.path.join(ROOT, "tests", "host_shim", "librules_host.so")
    if not os.path.exists(path):
        pytest.skip("host shim not built")
    return C.CDLL(path)


def test_swar_rules_header_matches_golden():
    from corintho_ai_b200 import planes_from_reference_order, reference_order_from_planes
    lib = _shim()
    states, seed = GOLD["states"], int(GOLD["seed"])
    pl = planes_from_reference_order(states)
    assert (reference_order_from_planes(pl) == states).all()
    n = len(states)
    mf = np.zeros((n, 4), np.uint32)
    nx = np.zeros((n, 2), np.uint64)
    enc = np.zeros((n, 70), np.float32)
    vp = C.c_void_p
    lib.shim_step_batch(C.c_int64(n), pl.ctypes.data_as(vp), C.c_uint64(seed), mf.ctypes.data_as(vp),
                        nx.ctypes.data_as(vp), enc.ctypes.data_as(vp))
    assert (mf[:, :3] == GOLD["masks"]).all()
    assert (mf[:, 3] == GOLD["flags"]).all()
    assert (reference_order_from_planes(nx) == GOLD["next"]).all()
    assert (enc == GOLD["enc"].astype(np.float32)).all()
    lib.shim_step_rnd.restype = C.c_uint32
    r = step_rnd(seed, 64)
    assert [lib.shim_step_rnd(C.c_uint64(seed), C.c_uint64(i)) for i in range(64)] == list(r)


def test_basic_moves_is_the_legal_mask_when_no_line_exists(oracle):
    """The paired game-logic kernel (game_step.cuh) finishes positions without a line from the
    basic-rule mask alone (basic_moves_pair, the paired form of basic_moves()) and queues the
    others: basic_moves()'s line flag must equal legal_moves_t's and, when no line exists, its mask
    must be the legal mask. 300 k reachable positions + the golden set."""
    from corintho_ai_b200 import planes_from_reference_order
    lib = _shim()
    lib.shim_basic_moves_check.restype = C.c_int64
    for states in (GOLD["states"], oracle.gen_states(4242, 300000)):
        pl = planes_from_reference_order(states)
        bad = lib.shim_basic_moves_check(C.c_int64(len(pl)), pl.ctypes.data_as(C.c_void_p))
        assert bad == 0


def test_paired_fast_path_forms_equal_the_plain_ones(oracle):
    """k_game_step_pairw (game_step.cuh) runs basic_moves_pair / nth_move_lut / do_move_lut; on the
    host they must agree with basic_moves / nth_move / do_move for every position, every legal move
    and every rank. 300 k reachable positions + the golden set, paired first-with-last."""
    from corintho_ai_b200 import planes_from_reference_order
    lib = _shim()
    lib.shim_fast_path_check.restype = C.c_int64
    for states in (GOLD["states"], oracle.gen_states(777, 300000)):
        pl = planes_from_reference_order(states)
        bad = lib.shim_fast_path_check(C.c_int64(len(pl)), pl.ctypes.data_as(C.c_void_p))
        assert bad == 0


def test_capital_fixups_are_exercised(oracle):
    """Q2: short capital row/column lines occur in the golden set (top==capital, short line)."""
    states = GOLD["states"]
    w0 = states[:, 0]
    caps = np.zeros((len(states), 16), bool)
    for s in range(16):
        caps[:, s] = ((w0 >> np.uint64(4 * s + 2)) & np.uint64(1)).astype(bool)
    rows = caps.reshape(-1, 4, 4)
    short = (rows[:, :, :3].all(2) ^ rows[:, :, 1:].all(2)).any(1)
    cols = (rows[:, :3, :].all(1) ^ rows[:, 1:, :].all(1)).any(1)
    assert short.sum() > 20 and cols.sum() > 20
