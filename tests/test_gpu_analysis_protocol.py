"""The analysis' external-evaluator protocol on the GPU (cb200_analysis_begin .. _results): round by
round equal to the oracle's analysis (orc_analysis_*) driven by the same evaluator, equal to the
fused run, device forms equal to host forms, and the protocol's errors."""
import numpy as np
import pytest

import corintho_ai_b200 as cb
from analysis_oracle import AnalysisOracle
from oracle.pyoracle import tie_storm_eval
from test_gpu_analysis import N, PARAMS, network_evaluator
from torch_net import torch_network

pytestmark = pytest.mark.gpu

ERR_ARG, ERR_OVERFLOW, ERR_STATE = -1, -3, -4


@pytest.fixture(scope="module")
def oracle():
    return AnalysisOracle()


@pytest.fixture(scope="module")
def positions(oracle):
    st = oracle.gen_states(5, N)  # the positions of test_gpu_analysis.py, terminal ones included
    assert sum(1 for s in st if not oracle.legal(s)[0].any()) > 50
    return st


def synthetic_evaluator(seed):
    """Answers no network of the engine can produce: a seeded hash of each row's bits gives 97
    uniforms; the value is tanh(4u - 2), in (-1, 1), and the probabilities a softmax of 8u."""
    mult, mix = np.uint64(0x100000001B3), np.uint64(0xD6E8FEB86659FD93)
    h0 = np.uint64((0x9E3779B97F4A7C15 * (seed + 1)) % (1 << 64))

    def f(rows):
        q = np.ascontiguousarray(rows, np.float32).reshape(-1, 70).view(np.uint32).astype(np.uint64)
        h = np.full(q.shape[0], h0, np.uint64)
        with np.errstate(over="ignore"):
            for j in range(70):
                h = (h ^ q[:, j]) * mult
                h ^= h >> np.uint64(29)
            m = h[:, None] + np.arange(97, dtype=np.uint64)[None, :] * mix
            m ^= m >> np.uint64(32)
            m *= mix
            m ^= m >> np.uint64(32)
        u = (m >> np.uint64(40)).astype(np.float64) / float(1 << 24)
        z = 8.0 * u[:, 1:]
        e = np.exp(z - z.max(1, keepdims=True))
        return np.tanh(4.0 * u[:, 0] - 2.0).astype(np.float32), (e / e.sum(1, keepdims=True)).astype(np.float32)
    return f


def finish(a, evaluator, answers=(None, None)):
    """Drive an open session to its end; returns the outputs."""
    while not a.do_iteration(*answers):
        answers = evaluator(a.write_requests())
    return a.results()


def assert_same_outputs(got, ref):
    assert set(got) == set(ref)
    for k in ref:
        if ref[k].dtype == np.float32:  # values and evals compared as bits
            assert (got[k].view(np.uint32) == ref[k].view(np.uint32)).all(), k
        else:
            assert (got[k] == ref[k]).all(), k


@pytest.mark.parametrize("evaluator", ["fp32", "bf16", "synthetic", "tie_storm"])
@pytest.mark.parametrize("ms,spe,c_puct,eps", PARAMS)
def test_protocol_equals_oracle_round_by_round(oracle, positions, evaluator, ms, spe, c_puct, eps):
    if evaluator == "synthetic":
        f = synthetic_evaluator(ms)
    elif evaluator == "tie_storm":
        f = tie_storm_eval
    else:
        f = network_evaluator(cb.fold_batchnorm(cb.random_weights(31)), evaluator)
    seed = 2000 + ms
    a = cb.Analysis(N, ms, spe, c_puct, eps)
    a.begin(cb.planes_from_reference_order(positions), seed)
    o = oracle.analysis(positions, seed, ms, spe, c_puct, eps)
    assert a.num_requests() == o.num_requests() == 0
    answers, rounds, rows_served = (None, None), 0, 0
    while True:
        done = a.do_iteration(*answers)
        assert done == o.do_iteration(*answers), rounds
        if done:
            break
        n = a.num_requests()
        assert n == o.num_requests(), rounds
        rows = a.write_requests()
        assert rows.shape == (n, 70)
        assert (rows.view(np.uint32) == o.write_requests().view(np.uint32)).all(), rounds
        answers = f(rows)
        rounds, rows_served = rounds + 1, rows_served + n
    assert a.num_requests() == 0
    assert_same_outputs(a.results(), o.results())
    c = a.counters()
    assert c == o.counters()
    assert c["leaf_evals"] == rows_served


@pytest.mark.parametrize("precision", ["fp32", "bf16", "fp16", "bf16x3"])
@pytest.mark.parametrize("ms,spe,c_puct,eps", PARAMS)
def test_protocol_with_the_network_equals_the_fused_run(positions, precision, ms, spe, c_puct, eps):
    weights = cb.fold_batchnorm(cb.random_weights(31))
    st = cb.planes_from_reference_order(positions)
    a = cb.Analysis(N, ms, spe, c_puct, eps)
    got = a.search(st, 3000 + ms, network_evaluator(weights, precision))
    counters = a.counters()
    a.set_weights(weights, precision)
    ref = a.run(st, 3000 + ms)
    assert_same_outputs(got, ref)
    assert counters == a.counters()
    no_evals = a.search(st[:512], 3000 + ms, network_evaluator(weights, precision), evals=False)
    assert "evals" not in no_evals and all((no_evals[k] == ref[k][:512]).all() for k in no_evals)


def test_device_forms_equal_host_forms_on_a_side_stream(positions):
    import torch
    dev = torch.device("cuda", 0)
    net = torch_network(cb.fold_batchnorm(cb.random_weights(7)), dev)
    st = cb.planes_from_reference_order(positions)
    ms, spe = 96, 16
    on_host, on_dev = cb.Analysis(N, ms, spe, 1.0, 0.25), cb.Analysis(N, ms, spe, 1.0, 0.25)
    rows_d = torch.full((N * spe, 70), float("nan"), device=dev)
    torch.cuda.synchronize(dev)  # the fill ran on the default stream
    stream = torch.cuda.Stream(device=dev)
    L = cb.lib()
    try:
        with torch.cuda.stream(stream):
            assert L.cb200_set_stream(stream.cuda_stream) == 0
            on_host.begin(st, 5)
            on_dev.begin(st, 5)
            empty = torch.empty(0, device=dev)
            ans_d, ans_h, rounds = (empty, empty), (None, None), 0
            while True:
                done = on_dev.do_iteration_device(*ans_d)
                assert done == on_host.do_iteration(*ans_h), rounds
                if done:
                    break
                n = on_dev.num_requests()
                assert n == on_host.num_requests() > 0
                on_dev.write_requests_device(rows_d)
                ans_d = net(rows_d[:n])  # queued on the side stream behind the packing kernel
                rows_h = on_host.write_requests()
                assert np.array_equal(rows_d[:n].cpu().numpy().view(np.uint32), rows_h.view(np.uint32)), rounds
                ans_h = tuple(t.cpu().numpy() for t in ans_d)
                rounds += 1
    finally:
        L.cb200_set_stream(None)
    assert rounds > 2
    assert_same_outputs(on_dev.results(), on_host.results())
    assert on_dev.counters() == on_host.counters()
    # a host buffer handed to a device form is refused, and the session stays as it was
    on_dev.begin(st[:64], 5)
    assert not on_dev.do_iteration_device(empty, empty)
    n = on_dev.num_requests()
    host_rows = np.zeros((n, 70), np.float32)
    assert L.cb200_analysis_write_requests_device(on_dev._h, cb._ptr(host_rows)) == ERR_ARG
    assert b"not device memory" in L.cb200_last_error()
    assert on_dev.num_requests() == n


def test_protocol_errors_leave_the_object_usable(positions):
    L = cb.lib()
    st = cb.planes_from_reference_order(positions[:64])
    syn = synthetic_evaluator(3)
    a = cb.Analysis(64, 16, 4, 1.0, 0.25)
    h = a._h
    out = cb._analysis_outputs(64, True)

    def raw_results():
        return L.cb200_analysis_results(h, *(cb._ptr(out[k]) for k in ("moves", "results", "values", "visits",
                                                                       "evals")))
    buf = np.zeros((64 * 4, 96), np.float32)
    # out of order: nothing but begin before the first session
    assert L.cb200_analysis_num_requests(h) == ERR_STATE
    assert L.cb200_analysis_write_requests(h, cb._ptr(buf)) == ERR_STATE
    assert L.cb200_analysis_do_iteration(h, None, None, 0) == ERR_STATE
    assert raw_results() == ERR_STATE
    with pytest.raises(cb.Corintho200Error, match="no open session"):
        a.num_requests()
    ref = a.search(st, 9, syn)
    # too few answer rows, null answers and early results are refused; the session goes on
    a.begin(st, 9)
    assert not a.do_iteration()
    n = a.num_requests()
    assert n > 0
    ev, pr = syn(a.write_requests())
    assert L.cb200_analysis_do_iteration(h, cb._ptr(ev), cb._ptr(pr), n - 1) == ERR_ARG
    assert L.cb200_analysis_do_iteration(h, None, None, n) == ERR_ARG
    assert raw_results() == ERR_STATE
    assert b"not done" in L.cb200_last_error()
    assert_same_outputs(finish(a, syn, (ev, pr)), ref)
    # after completion do_iteration returns 1 and does no work; results may be read again
    c = a.counters()
    assert a.do_iteration() and a.num_requests() == 0 and a.counters() == c
    assert_same_outputs(a.results(), ref)
    # a rejected state in begin: no session is left open
    bad = st.copy()
    bad[7, 1] |= np.uint64(1) << np.uint64(56)
    with pytest.raises(cb.Corintho200Error, match="not a valid cstate"):
        a.begin(bad, 9)
    assert L.cb200_analysis_num_requests(h) == ERR_STATE
    # begin during an open session restarts it
    a.begin(st[:10], 1)
    assert not a.do_iteration()
    a.begin(st, 9)
    assert_same_outputs(finish(a, syn), ref)
    # run in the middle of a session discards it; then a new begin
    weights = cb.fold_batchnorm(cb.random_weights(2))
    a.set_weights(weights, "fp32")
    a.begin(st, 9)
    assert not a.do_iteration()
    fused = a.run(st, 9)
    assert L.cb200_analysis_num_requests(h) == ERR_STATE
    assert_same_outputs(a.search(st, 9, network_evaluator(weights, "fp32")), fused)
    assert_same_outputs(a.search(st, 9, syn), ref)


def test_batch_independence(positions):
    st = cb.planes_from_reference_order(positions[:2048])
    syn = synthetic_evaluator(11)
    a = cb.Analysis(2048, 48, 8, 1.0, 0.25)
    full = a.search(st, 77, syn)
    half = a.search(st[:1024], 77, syn)
    for k in full:
        assert (full[k][:1024] == half[k]).all(), k
    part = a.search(st[100:400], 3, syn)
    alone = cb.Analysis(300, 48, 8, 1.0, 0.25).search(st[100:400], 3, syn)
    assert_same_outputs(part, alone)


def test_overflow_ends_the_session_and_the_object_stays_usable(oracle, positions, monkeypatch):
    monkeypatch.setenv("CB200_ARENA_NODES", "24")
    a = cb.Analysis(64, 64, 16, 1.0, 0.25)
    monkeypatch.delenv("CB200_ARENA_NODES")
    st = cb.planes_from_reference_order(positions[:64])
    with pytest.raises(cb.Corintho200Error, match=f"error {ERR_OVERFLOW}") as e:
        a.search(st, 1, synthetic_evaluator(1))
    assert "arena" in str(e.value)
    assert cb.lib().cb200_analysis_num_requests(a._h) == ERR_STATE
    terminal = [i for i, s in enumerate(positions) if not oracle.legal(s)[0].any()][:16]
    got = a.search(cb.planes_from_reference_order(positions[terminal]), 1, synthetic_evaluator(1))
    assert (got["moves"] == -1).all() and np.isin(got["results"], [1, 2]).all()
