"""Analysis on the GPU (csrc/analysis.cuh, cb200_analysis_*): bit-exact against the oracle's
analysis driven with the engine's own network kernels, batch independence, errors, counters."""
import numpy as np
import pytest

import corintho_ai_b200 as cb
from analysis_oracle import AnalysisOracle, play_analysis

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def oracle():
    """The oracle with the analysis restatement of tests/analysis_oracle.cpp added."""
    return AnalysisOracle()

N = 4096
PARAMS = [  # (max_searches, searches_per_eval, c_puct, epsilon)
    (1, 1, 1.0, 0.25),
    (64, 16, 1.0, 0.0),
    (400, 16, 2.0, 0.25),
    (64, 1, 0.5, 0.25),
]


def network_evaluator(weights, precision):
    """f(request rows) -> (eval, probs) through the engine's own network kernels (a helper Trainer's
    resident network, in slices of its capacity), so the oracle sees bit-identical answers."""
    helper = cb.Trainer(64, "", 1, 64, 16)
    helper.set_weights(weights, 0, precision)
    cap = 64 * 16

    def f(req):
        ev = np.zeros(len(req), np.float32)
        pr = np.zeros((len(req), 96), np.float32)
        for i in range(0, len(req), cap):
            ev[i:i + cap], pr[i:i + cap] = helper.evaluate(req[i:i + cap])
        return ev, pr
    return f


@pytest.fixture(scope="module")
def positions(oracle):
    st = oracle.gen_states(5, N)  # reference bit order; terminal positions included
    assert sum(1 for s in st if not oracle.legal(s)[0].any()) > 50
    return st


@pytest.mark.parametrize("precision", ["fp32", "bf16", "fp16", "bf16x3"])
@pytest.mark.parametrize("ms,spe,c_puct,eps", PARAMS)
def test_analysis_equals_oracle_driven_by_the_same_network(oracle, positions, precision, ms, spe, c_puct,
                                                           eps):
    weights = cb.fold_batchnorm(cb.random_weights(31))
    seed = 1000 + ms
    a = cb.Analysis(N, ms, spe, c_puct, eps)
    a.set_weights(weights, precision)
    got = a.run(cb.planes_from_reference_order(positions), seed)
    o = oracle.analysis(positions, seed, ms, spe, c_puct, eps)
    rec = []
    play_analysis(o, network_evaluator(weights, precision), record=rec)
    ref = o.results()
    assert (got["moves"] == ref["moves"]).all()
    assert (got["results"] == ref["results"]).all()
    assert (got["values"].view(np.uint32) == ref["values"].view(np.uint32)).all()
    assert (got["visits"] == ref["visits"]).all()
    assert (got["evals"].view(np.uint32) == ref["evals"].view(np.uint32)).all()
    c = a.counters()
    assert c == o.counters()
    assert c["leaf_evals"] == sum(len(r) for r in rec)  # the requests the oracle had served


def test_batch_independence_and_reuse(oracle, positions):
    st = cb.planes_from_reference_order(positions[:2048])
    weights = cb.fold_batchnorm(cb.random_weights(5))
    a = cb.Analysis(2048, 48, 8, 1.0, 0.25)
    a.set_weights(weights, "bf16")
    full = a.run(st, 77)
    half = a.run(st[:1024], 77)
    for k in full:
        assert (full[k][:1024] == half[k]).all(), k
    again = a.run(st, 77)
    for k in full:
        assert (full[k] == again[k]).all(), k
    # reused with a smaller n and another seed = a fresh object
    small = a.run(st[100:400], 3)
    fresh = cb.Analysis(300, 48, 8, 1.0, 0.25)
    fresh.set_weights(weights, "bf16")
    ref = fresh.run(st[100:400], 3)
    for k in ref:
        assert (small[k] == ref[k]).all(), k
    # without evals the other outputs are unchanged
    no_ev = a.run(st[100:400], 3, evals=False)
    assert "evals" not in no_ev and all((no_ev[k] == ref[k]).all() for k in no_ev)


def test_errors_leave_the_object_usable(oracle, positions):
    L = cb.lib()
    st = cb.planes_from_reference_order(positions[:64])
    a = cb.Analysis(64, 16, 4, 1.0, 0.25)
    with pytest.raises(cb.Corintho200Error):
        a.run(st)  # no weights yet
    a.set_weights(cb.fold_batchnorm(cb.random_weights(2)), "fp32")
    ok = a.run(st, 9)
    h = a._h
    buf = {k: np.zeros_like(v) for k, v in ok.items()}

    def raw(n, states, moves=True):
        return L.cb200_analysis_run(h, n, cb._ptr(states), 9, cb._ptr(buf["moves"]) if moves else None,
                                    cb._ptr(buf["results"]), cb._ptr(buf["values"]), cb._ptr(buf["visits"]),
                                    cb._ptr(buf["evals"]))
    big = np.concatenate([st, st])
    assert raw(65, big) == -1  # n > max_positions
    assert raw(0, st) == -1
    assert raw(64, st, moves=False) == -1  # null output
    bad = st.copy()
    bad[7, 1] |= np.uint64(1) << np.uint64(56)  # byte 7 set
    assert raw(64, bad) == -1
    assert b"not a valid cstate" in L.cb200_last_error()
    assert L.cb200_analysis_set_weights(h, None, cb.WEIGHT_FLOATS, 0) == -1
    for args in [(0, 16, 4, 1.0, 0.25), (8, 0, 4, 1.0, 0.25), (8, 16, 65, 1.0, 0.25), (8, 16, 4, 0.0, 0.25),
                 (8, 16, 4, 1.0, 1.5)]:
        with pytest.raises(cb.Corintho200Error):
            cb.Analysis(*args)
    again = a.run(st, 9)
    for k in ok:
        assert (ok[k] == again[k]).all(), k
