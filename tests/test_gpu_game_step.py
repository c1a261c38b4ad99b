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


@pytest.mark.parametrize("env", [{}, {"CB200_K1_WAVES": "1"}, {"CB200_K1_PAIR": "0"}, {"CB200_K1_PAIR": "1"},
                                 {"CB200_K1_PAIR": "2"}, {"CB200_K1_PAIR": "3"}, {"CB200_K1_PAIR": "4"},
                                 {"CB200_K1_PAIR": "5"}, {"CB200_K1_SPLIT": "1"}, {"CB200_K1_SELECT_ONLY": "1"}],
                         ids=["paired", "paired-one-wave", "paired-branchy-finish", "paired-branchy-finish-prefetch",
                              "paired-cta-queue", "paired-7-ctas", "paired-prefetch-6-ctas", "paired-joint-finish-no-prefetch",
                              "split", "select-only"])
def test_game_step_kernel_forms_vs_oracle(oracle, monkeypatch, env):
    """Every form of the game-logic kernel (paired with a queue per warp, prefetch and the joint
    branch-free finish = default; without either; with a queue per CTA; register-capped builds;
    split; select-only) and the default with a single
    wave of CTAs (many trips per CTA: the queues wrap through several flushes) against the oracle
    on 256 k reachable positions."""
    for k in ("CB200_K1_WAVES", "CB200_K1_PAIR", "CB200_K1_SPLIT", "CB200_K1_SELECT_ONLY"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    n = 1 << 18
    states = oracle.gen_states(4711, n)
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
