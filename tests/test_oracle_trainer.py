"""Tree search / self-play: oracle restatement vs the golden transcripts generated from the
compiled reference, vs the compiled reference itself, plus the reference's own property
checks (tests/cpp/trainer_test.cpp:22-175, selfplayer_test.cpp:94-143) run on the oracle."""
import os

import numpy as np
import pytest

from oracle.pyoracle import ADVERSARIAL_EVALUATORS, synth_eval
from util import TRAINER_GRID, grid_key, run_trainer

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = np.load(os.path.join(ROOT, "tests", "golden", "trainer.npz"))


def make(L, cfg):
    g, s, ms, spe, cp, eps, testing = cfg
    return L.trainer(num_games=g, seed=s, max_searches=ms, searches_per_eval=spe, c_puct=cp,
                     epsilon=eps, testing=testing)


def check_against_golden(r, cfg):
    k = grid_key(cfg)
    assert r["rounds"] == int(GOLD[k + "/rounds"])
    assert (r["counts"] == GOLD[k + "/counts"]).all()
    assert (r["to_play"] == GOLD[k + "/to_play"]).all()
    assert r["req_hash"].encode() == bytes(GOLD[k + "/req_hash"])
    assert r["num_samples"] == int(GOLD[k + "/num_samples"])
    assert r["score"].tobytes() == GOLD[k + "/score"].tobytes()
    assert r["mate"].tobytes() == GOLD[k + "/mate"].tobytes()
    if not cfg[6]:
        assert r["samples_hash"].encode() == bytes(GOLD[k + "/samples_hash"])
        if k + "/gs" in GOLD:
            gs, ev, pr = r["samples"]
            assert gs.tobytes() == GOLD[k + "/gs"].tobytes()
            assert ev.tobytes() == GOLD[k + "/ev"].tobytes()  # incl. the +0.0/-0.0 draw labels (Q10)
            assert pr.tobytes() == GOLD[k + "/pr"].tobytes()


@pytest.mark.parametrize("cfg", TRAINER_GRID, ids=grid_key)
def test_oracle_matches_golden_transcripts(oracle, cfg):
    r = run_trainer(make(oracle, cfg), synth_eval, cfg[6])
    check_against_golden(r, cfg)


@pytest.mark.parametrize("cfg", [(5, 4242, 48, 16, 1.0, 0.25, False), (4, 9, 160, 7, 2.0, 0.1, False),
                                 (6, 3, 32, 4, 1.0, 0.25, True)], ids=grid_key)
def test_oracle_matches_compiled_reference(oracle, ref, cfg):
    a = run_trainer(make(ref, cfg), synth_eval, cfg[6])
    b = run_trainer(make(oracle, cfg), synth_eval, cfg[6])
    assert a["rounds"] == b["rounds"] and (a["counts"] == b["counts"]).all()
    assert a["req_hash"] == b["req_hash"]
    assert a["score"].tobytes() == b["score"].tobytes() and a["mate"].tobytes() == b["mate"].tobytes()
    if not cfg[6]:
        assert a["samples_hash"] == b["samples_hash"]


@pytest.mark.parametrize("evaluator", sorted(ADVERSARIAL_EVALUATORS))
@pytest.mark.parametrize("cfg", [(5, 4242, 48, 16, 1.0, 0.25, False), (6, 3, 32, 4, 1.0, 0.0, True)],
                         ids=grid_key)
def test_oracle_matches_compiled_reference_with_degenerate_evaluators(oracle, ref, cfg, evaluator):
    """The same comparison under tie storms, all-zero and subnormal probabilities: the
    reference's NaN max and x86 lround decide the priors there."""
    f = ADVERSARIAL_EVALUATORS[evaluator]
    a = run_trainer(make(ref, cfg), f, cfg[6])
    b = run_trainer(make(oracle, cfg), f, cfg[6])
    assert a["rounds"] == b["rounds"] and (a["counts"] == b["counts"]).all()
    assert a["req_hash"] == b["req_hash"]
    assert a["score"].tobytes() == b["score"].tobytes() and a["mate"].tobytes() == b["mate"].tobytes()
    assert cfg[6] or a["samples_hash"] == b["samples_hash"]


def test_max_searches_1_quirk(oracle):
    """SURVEY.md Q3: with max_searches=1 every game goes 95,94,93,92 and ends in 4 plies."""
    t = oracle.trainer(num_games=2, seed=1, max_searches=1, searches_per_eval=1)
    r = run_trainer(t, synth_eval)
    assert r["num_samples"] == 8
    gs, ev, pr = r["samples"]
    ident = pr[::8]
    assert [int(np.argmax(row)) for row in ident[:4]] == [95, 94, 93, 92]


@pytest.mark.parametrize("games,ms,spe", [(1, 16, 16), (3, 96, 16), (3, 2, 1)])
def test_reference_property_checks_on_oracle(oracle, games, ms, spe):
    """trainer_test.cpp:22-136 property sweep (subset), random evaluator like the reference."""
    rng = np.random.default_rng(12345)

    def rand_eval(req):
        n = req.shape[0]
        assert 0 < n <= games * spe
        assert ((req >= 0) & (req <= 1)).all()
        return rng.uniform(-1, 1, n).astype(np.float32), rng.uniform(0, 1, (n, 96)).astype(np.float32)

    t = oracle.trainer(num_games=games, seed=12345, max_searches=ms, searches_per_eval=spe)
    r = run_trainer(t, rand_eval)
    ns = r["num_samples"]
    assert 0 < ns <= 40 * games
    gs, ev, pr = r["samples"]
    assert ((gs >= 0) & (gs <= 1)).all() and ((ev >= -1) & (ev <= 1)).all()
    assert ((pr >= 0) & (pr <= 1)).all()
    assert np.allclose(pr.sum(1), 1.0, atol=0.01)
    gs8, pr8 = gs.reshape(ns, 8, 70), pr.reshape(ns, 8, 96)
    for k in range(1, 8):  # every symmetry is a permutation of the identity sample
        assert (np.sort(gs8[:, k], 1) == np.sort(gs8[:, 0], 1)).all()
        assert (np.sort(pr8[:, k], 1) == np.sort(pr8[:, 0], 1)).all()


def test_testing_mode_writes_no_samples(oracle):
    t = oracle.trainer(num_games=4, seed=3, max_searches=16, searches_per_eval=4, testing=True)
    r = run_trainer(t, synth_eval, testing=True)
    assert r["num_samples"] == 0 and 0.0 <= float(r["score"]) <= 1.0
