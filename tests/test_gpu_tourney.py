"""Match / Tourney on the GPU (csrc/match.cuh) through the C ABI: golden transcripts generated
from the compiled reference, the oracle side by side, and the reference's own property checks
(tests/cpp/tourney_test.cpp, match_test.cpp: games finish, scores are 0 / 0.5 / 1)."""
import os

import numpy as np
import pytest

import corintho_ai_b200 as cb
from util import TOURNEY_CASES, make_tourney, run_tourney

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = np.load(os.path.join(ROOT, "tests", "golden", "tourney.npz"))


class _Engine:
    """Adapter so that util.make_tourney can build the engine's Tourney like the oracle's."""
    def tourney(self, num_threads, log_folder):
        return cb.Tourney(num_threads, log_folder)


@pytest.mark.parametrize("name", list(TOURNEY_CASES))
def test_engine_tourney_matches_golden_transcripts(name):
    r = run_tourney(make_tourney(_Engine(), name))
    assert r["rounds"] == int(GOLD[name + "/rounds"])
    assert (r["models"] == GOLD[name + "/models"]).all()
    assert (r["counts"] == GOLD[name + "/counts"]).all()
    assert r["req_hash"].encode() == bytes(GOLD[name + "/req_hash"])  # every request row, bit exact
    assert (r["scores"] == GOLD[name + "/scores"]).all()


def test_engine_tourney_matches_oracle_on_a_larger_field(oracle):
    """40 matches between four searching players (two models) and a random player."""
    def build(L):
        t = L.tourney(2, "")
        t.add_player(0, 0, 96, 16, 1.0, 0.25)
        t.add_player(1, 0, 40, 8, 3.0, 0.0)
        t.add_player(2, 1, 64, 5, 1.0, 0.5)
        t.add_player(3, 1, 24, 24, 0.5, 0.25)
        t.add_player(4, -1, 1, 1, 1.0, 0.25, True)
        for i in range(40):
            t.add_match(i % 5, (i * 3 + 1) % 5)
        return t
    a = run_tourney(build(oracle))
    eng = build(_Engine())
    b = run_tourney(eng)
    assert a["rounds"] == b["rounds"] and (a["counts"] == b["counts"]).all()
    assert a["req_hash"] == b["req_hash"]
    assert (a["scores"] == b["scores"]).all()
    c = eng.counters()
    assert c["simulations"] > 0 and c["moves"] > 0 and c["leaf_evals"] == int(a["counts"].sum())


def test_tourney_protocol_and_errors(tmp_path):
    t = cb.Tourney(1, "")
    with pytest.raises(cb.Corintho200Error):
        t.addMatch(0, 1)  # unknown players
    t.addPlayer(0, 0, 32, 8, 1.0, 0.25)
    t.addPlayer(1, -1, 1, 1, 1.0, 0.25, True)
    with pytest.raises(cb.Corintho200Error):
        t.addPlayer(2, 0, 0, 8, 1.0, 0.25)  # invalid budget
    for _ in range(4):
        t.addMatch(0, 1)
        t.addMatch(1, 0)
    assert not t.all_done() and t.num_requests(-1) == 0
    with pytest.raises(cb.Corintho200Error):
        t.addMatch(0, 1)  # the device state exists now
    r = run_tourney(t)
    assert t.all_done() and len(r["scores"]) == 8
    assert set(r["scores"][:, 2]) <= {0.0, 0.5, 1.0}
    f = tmp_path / "scores.txt"
    t.writeScores(str(f))
    rows = f.read_text().split("\n")
    assert rows[0].split()[:2] == ["0", "1"] and rows[1].split()[:2] == ["1", "0"]


@pytest.mark.parametrize("precision", ["fp32", "bf16", "fp16", "bf16x3"])
@pytest.mark.parametrize("name", ["two_models", "with_random", "deeper"])
def test_fused_tourney_equals_oracle_driven_by_the_same_networks(oracle, name, precision):
    """Fused tourney (cb200_tourney_set_weights / cb200_tourney_run): every model id has a
    device-resident network and the whole loop of rating/tourney.pyx:112-173 runs on the GPU.
    The oracle's Tourney, driven through that loop with the same networks (the engine's own
    kernels as evaluators, so the numbers are bit-identical), must end with the same scores."""
    players, matches = TOURNEY_CASES[name]
    model_ids = sorted({p[1] for p in players if p[1] >= 0})
    weights = {m: cb.fold_batchnorm(cb.random_weights(100 + m)) for m in model_ids}
    eng = make_tourney(_Engine(), name)
    for m in model_ids:
        eng.set_weights(m, weights[m], precision)
    assert eng.run(0)
    assert eng.all_done()
    helpers = {}
    for m in model_ids:
        h = cb.Trainer(64, "", 1, 64, 16)
        h.set_weights(weights[m], 0, precision)
        helpers[m] = h
    ref = run_tourney(make_tourney(oracle, name), {m: (lambda req, h=helpers[m]: h.evaluate(req)) for m in model_ids})
    got = np.array(eng.scores(), np.float64).reshape(-1, 3)
    assert (got == ref["scores"]).all()
    c = eng.counters()
    assert c["leaf_evals"] == int(ref["counts"].sum()) and c["simulations"] > 0


def test_fused_tourney_bounded_rounds_and_errors():
    players, matches = TOURNEY_CASES["two_models"]
    t = make_tourney(_Engine(), "two_models")
    with pytest.raises(cb.Corintho200Error):
        t.run(0)  # no weights yet
    for m in (0, 1):
        t.set_weights(m, cb.fold_batchnorm(cb.random_weights(7 + m)), "bf16")
    done, calls = False, 0
    while not done:
        done = t.run(5)
        calls += 1
        assert calls < 1000
    assert calls > 1 and len(t.scores()) == len(matches)
