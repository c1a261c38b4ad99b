"""K1 game-logic kernel through the C ABI vs golden vectors (from the compiled reference), vs
the oracle at 1M states, and size-independent properties at the BASELINE configs[1] size.
The large tests take their positions from the oracle's generator, the same code they compare
with; the golden vectors (test_game_step_matches_golden, and the generator pinned to the
reference's play-outs in test_oracle_rules.py) keep both tied to the reference."""
import os

import numpy as np
import pytest

import corintho_ai_b200 as cb
from util import step_rnd

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = np.load(os.path.join(ROOT, "tests", "golden", "rules.npz"))


def test_game_step_matches_golden():
    states, seed = GOLD["states"], int(GOLD["seed"])
    mf, nx, enc = cb.game_step(cb.planes_from_reference_order(states), seed, want_encoding=True)
    assert (mf[:, :3] == GOLD["masks"]).all()
    assert (mf[:, 3] == GOLD["flags"]).all()
    assert (cb.reference_order_from_planes(nx) == GOLD["next"]).all()
    assert (enc == GOLD["enc"].astype(np.float32)).all()


@pytest.mark.parametrize("n", [0, 1, 31, 33, 257, 4097])
def test_game_step_ragged_sizes(oracle, n):
    states = GOLD["states"][:n]
    mf, nx, enc = cb.game_step(cb.planes_from_reference_order(states), 9, want_encoding=True)
    if n == 0:
        assert mf.shape[0] == 0
        return
    masks, flags, nxt, e2 = oracle.step_batch(states, step_rnd(9, n))
    assert (mf[:, :3] == masks).all() and (mf[:, 3] == flags).all()
    assert (cb.reference_order_from_planes(nx) == nxt).all()
    assert enc.tobytes() == e2.tobytes()


@pytest.mark.parametrize("n", [1, 2, 255, 256, 257, 511, 512, 513, 767, 1025, 4097, 20000])
def test_game_step_ragged_sizes_without_encoding(oracle, n):
    """The paired kernel (two positions per thread, 512 per trip): every tail shape -- a lone
    position, a thread whose second position is past the end, a partly filled last trip."""
    states = GOLD["states"][:n]
    mf, nx, _ = cb.game_step(cb.planes_from_reference_order(states), 11)
    masks, flags, nxt, _ = oracle.step_batch(states, step_rnd(11, n), want_enc=False)
    assert (mf[:, :3] == masks).all() and (mf[:, 3] == flags).all()
    assert (cb.reference_order_from_planes(nx) == nxt).all()


def test_game_step_many_trips_per_cta_vs_oracle(oracle):
    """The paired kernel with several trips per CTA against the oracle on 2^24 positions (2^22
    reachable positions tiled 4x, a different random word for every index). The grid is at most
    8 waves of resident CTAs: 148 SMs x 4 CTAs (64 registers, 256 threads) x 8 = 4 736 CTAs of
    512 positions per trip = 2.42 M positions per sweep, so every CTA makes about 7 trips. A warp
    queues about 10 of its 64 positions per trip (the ones with a line), about 66 over its trips,
    so every warp flushes 32 queued positions inside the loop, the prefetch of the next trip is
    used, and the drain finishes what is left."""
    states = np.tile(oracle.gen_states(4711, 1 << 22), (4, 1))
    n = len(states)
    mf, nx, _ = cb.game_step(cb.planes_from_reference_order(states), 5)
    masks, flags, nxt, _ = oracle.step_batch(states, step_rnd(5, n), want_enc=False, threads=8)
    assert (mf[:, :3] == masks).all() and (mf[:, 3] == flags).all()
    assert (cb.reference_order_from_planes(nx) == nxt).all()


def test_game_step_1m_states_vs_oracle(oracle):
    """BASELINE.json configs[1] size: 1M reachable states, bit-exact against the oracle."""
    n = 1 << 20
    states = oracle.gen_states(20261018, n)
    mf, nx, _ = cb.game_step(cb.planes_from_reference_order(states), 77)
    masks, flags, nxt, _ = oracle.step_batch(states, step_rnd(77, n), want_enc=False, threads=8)
    assert (mf[:, :3] == masks).all() and (mf[:, 3] == flags).all()
    assert (cb.reference_order_from_planes(nx) == nxt).all()


def test_game_step_properties_at_full_size():
    """Size-independent properties on 4M states derived on the device itself (next states fed
    back in): mask popcount == n_legal, chosen move is legal, exactly one frozen square after a
    move, piece counts never increase, terminal states map to themselves."""
    n = 1 << 22
    st = np.tile(cb.planes_from_reference_order(GOLD["states"]), (n // len(GOLD["states"]) + 1, 1))[:n]
    for rnd in range(3):
        mf, nx, _ = cb.game_step(st, 1000 + rnd)
        pop = np.zeros(n, np.int64)
        for w in range(3):
            pop += np.array([bin(x).count("1") for x in range(65536)], np.int64)[mf[:, w] & 0xFFFF]
            pop += np.array([bin(x).count("1") for x in range(65536)], np.int64)[mf[:, w] >> 16]
        nl = (mf[:, 3] >> 8) & 0xFF
        assert (pop == nl).all()
        chosen = (mf[:, 3] >> 16) & 0xFF
        live = nl > 0
        c = chosen[live].astype(np.int64)
        assert ((mf[live][np.arange(c.size), c >> 5] >> (c & 31).astype(np.uint32)) & 1).all()
        assert (chosen[~live] == 0x7F).all() and (nx[~live] == st[~live]).all()
        frozen = (nx[live, 0] >> np.uint64(48)).astype(np.int64)
        assert ((frozen & (frozen - 1)) == 0).all() and (frozen != 0).all()
        res = mf[:, 3] & 3
        assert ((res != 0) == ~live).all()
        st = nx
