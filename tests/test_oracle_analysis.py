"""The analysis restatement on the oracle (tests/analysis_oracle.cpp, the batched DockerMC) pinned to
the oracle's testing-mode Trainer, and the structural state check the engine applies to positions it
is given. CPU only."""
import ctypes

import numpy as np
import pytest

import corintho_ai_b200 as cb
from analysis_oracle import AnalysisOracle, play_analysis
from oracle.pyoracle import synth_eval


@pytest.fixture(scope="module")
def oracle():
    """The oracle with the analysis object added (its Trainer is the oracle's own)."""
    return AnalysisOracle()


def trainer_first_move(oracle, seed, game, ms, spe, c_puct, eps):
    """Play the first move of game `game` of a testing-mode oracle Trainer with seed `seed` (a
    one-game shard: the same generator seed as game `game` of the whole run) and return
    (chosen move, root child visits [96], root child evaluations [96], counters)."""
    kw = {"first_game": game} if game else {}
    t = oracle.trainer(1, "", seed, ms, spe, c_puct, eps, testing=True, **kw)
    to_play = game % 2  # selects the game while its first player (to_play_ 0) moves
    ev = np.zeros(spe, np.float32)
    pr = np.zeros((spe, 96), np.float32)
    while oracle.counters(t)["moves"] == 0:
        t.do_iteration(ev, pr, to_play)
        n = t.num_requests(to_play)
        if n:
            e, p = synth_eval(t.write_requests(to_play))
            ev[:n], pr[:n] = e, p
    # Re-rooting copies the chosen subtree out of the mover's arena and leaves the arena as it
    # was, and the opponent's first tree has an arena of its own: right after the first move the
    # spare arena holds the mover's tree as it stood when the move was chosen (root at word 0).
    _, arenas = oracle.dump_arena(t, 0, 0)
    words, _ = oracle.dump_arena(t, 0, int(arenas[2]))
    visits = np.zeros(96, np.int32)
    evals = np.zeros(96, np.float32)
    for e in range(int(words[4] & 0xff)):
        s = words[8 + 4 * e: 12 + 4 * e]
        if (s[3] >> 20) & 1:
            visits[s[3] & 0x7f] = s[1]
            evals[s[3] & 0x7f] = s[0:1].view(np.float32)[0]
    # the move: tree 0's new root is the position it leads to
    out = np.zeros(8, np.int64)
    root = np.zeros(4, np.uint32)
    f = oracle.lib.orc_trainer_dump_tree
    f.restype = ctypes.c_int
    f(ctypes.c_void_p(t.h), 0, 0, out.ctypes.data_as(ctypes.c_void_p), root.ctypes.data_as(ctypes.c_void_p), 4)
    after = root.view(np.uint64)
    start = oracle.start()
    moves = [m for m in range(96) if (oracle.do_move(start, m) == after).all()]
    assert len(moves) == 1
    return moves[0], visits, evals, oracle.counters(t)


@pytest.mark.parametrize("seed,ms,spe,c_puct,eps", [
    (1, 64, 16, 1.0, 0.25), (7, 400, 8, 2.0, 0.0), (3, 1, 1, 1.0, 0.25), (11, 50, 1, 0.5, 0.25),
    (2024, 96, 16, 1.0, 0.0)])
def test_analysis_of_the_start_reproduces_the_trainers_first_move(oracle, seed, ms, spe, c_puct, eps):
    """Position i of an analysis is seeded like game i of a Trainer (the i-th output of
    mt19937(seed)). SelfPlayer draws nothing from its generator before the first search (the first
    doIteration queues the root, the first draws are the Dirichlet noise of its evaluation), so
    both streams line up without an offset: move, root child visits / evaluations and the work
    counters must equal those of the Trainer's first move."""
    k = 4
    a = oracle.analysis(np.stack([oracle.start()] * k), seed, ms, spe, c_puct, eps)
    play_analysis(a)
    r = a.results()
    sims = evals = 0
    for i in range(k):
        move, visits, child_evals, c = trainer_first_move(oracle, seed, i, ms, spe, c_puct, eps)
        assert r["moves"][i] == move
        assert r["results"][i] == 0
        if visits.sum() == 0:  # no child visited (max_searches 1): the tree was rebuilt in place
            assert r["visits"][i].sum() == 0
        else:
            assert (r["visits"][i] == visits).all()
            assert (r["evals"][i].view(np.uint32) == child_evals.view(np.uint32)).all()
        sims += c["simulations"]
        evals += c["leaf_evals"]
    assert a.counters() == {"simulations": sims, "leaf_evals": evals}


def test_outputs_depend_on_the_position_index_only(oracle):
    st = oracle.gen_states(9, 96)
    full = oracle.analysis(st, 5, 48, 8, 1.0, 0.25)
    play_analysis(full)
    head = oracle.analysis(st[:40], 5, 48, 8, 1.0, 0.25)
    play_analysis(head)
    a, b = full.results(), head.results()
    for k in a:
        assert (a[k][:40] == b[k]).all(), k


def test_terminal_positions_are_not_searched(oracle):
    st = oracle.gen_states(17, 3000)
    term = np.array([not oracle.legal(s)[0].any() for s in st])
    assert term.sum() >= 20
    a = oracle.analysis(st, 1, 32, 16, 1.0, 0.25)
    rec = []
    play_analysis(a, record=rec)
    r = a.results()
    assert (r["moves"][term] == -1).all() and (r["moves"][~term] >= 0).all()
    lines = np.array([oracle.legal(s)[1] for s in st[term]])
    assert (r["results"][term] == np.where(lines, 1, 2)).all()
    assert (r["visits"][term] == 0).all() and (r["values"][term] == 0).all()
    # no request row is ever a terminal input
    assert a.counters()["leaf_evals"] == sum(len(x) for x in rec)


def test_state_invariants_hold_on_a_million_reachable_positions(oracle):
    """The candidate invariants of the check (frozen squares occupied; per kind, pieces on the
    board = 8 - both hands) accept every position of 1 000 000 random play-outs, start and terminal
    positions included -- in the oracle and in the engine's host-side check."""
    st = oracle.gen_states(0, 1_000_000)
    assert (st[0] == oracle.start()).all()
    cst = cb.planes_from_reference_order(st)
    ok = cb.check_states(cst)
    assert ok.all(), np.flatnonzero(~ok)[:10]
    for s in st[::997]:
        assert oracle.state_valid(s)


def crafted(oracle):
    """(name, reference-order state) pairs that the check must reject, made from a mid-game state."""
    st = oracle.gen_states(3, 40)[25]
    w0, w1 = int(st[0]), int(st[1])
    out = []
    out.append(("side to move 2", [w0, (w1 & ~(0xff << 48)) | (2 << 48)]))
    out.append(("byte 7 set", [w0, w1 | (1 << 56)]))
    # the start position with five and three bases in the hands: only the hand limit is broken
    s0, s1 = (int(x) for x in oracle.start())
    out.append(("five bases in a hand", [s0, (s1 & ~0xff & ~(0xff << 24)) | 5 | (3 << 24)]))
    # frozen plane on an empty square
    occ = 0
    for sq in range(16):
        if (w0 >> (4 * sq)) & 0x7:
            occ |= 1 << sq
    empty = next(sq for sq in range(16) if not (occ >> sq) & 1)
    out.append(("frozen empty square", [w0 | (1 << (4 * empty + 3)), w1]))
    # a base on the board that is also still counted in a hand
    out.append(("piece counted twice", [w0 | (1 << (4 * empty)), w1]))
    return [(n, np.array(s, np.uint64)) for n, s in out]


def test_crafted_malformed_states_are_rejected(oracle):
    good = oracle.gen_states(3, 40)[25]
    assert oracle.state_valid(good) and cb.check_states(cb.planes_from_reference_order(good[None]))[0]
    bad = crafted(oracle)
    for name, s in bad:
        assert not oracle.state_valid(s), name
        assert not cb.check_states(cb.planes_from_reference_order(s[None]))[0], name
        with pytest.raises(ValueError):
            oracle.analysis(np.stack([good, s]), 0, 8, 4)
    assert cb.lib().cb200_check_states(-1, None, None) < 0
