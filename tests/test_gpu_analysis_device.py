"""Analysis with positions and outputs in device memory (cb200_analysis_run_device, one persistent
kernel): bit for bit equal to cb200_analysis_run -- itself pinned to the oracle by
test_gpu_analysis.py -- over batch shapes that cross the CTA dealing and the device MT19937 block
boundaries, per-position errors, stream order without host synchronisation, graph capture, and the
errors of the call itself."""
import ctypes as C

import numpy as np
import pytest
import torch

import corintho_ai_b200 as cb
from analysis_oracle import AnalysisOracle

pytestmark = pytest.mark.gpu

ERR_ARG, ERR_OVERFLOW, ERR_STATE = -1, -3, -4
N = 4096
PARAMS = [  # (max_searches, searches_per_eval, c_puct, epsilon)
    (1, 1, 1.0, 0.25),
    (64, 16, 1.0, 0.0),
    (400, 16, 2.0, 0.25),
    (64, 1, 0.5, 0.25),
    (128, 64, 1.0, 0.25),
]
KEYS = ("moves", "results", "values", "visits", "evals")
GAMES_PER_CTA = {"bf16": 16, "fp16": 16, "bf16x3": 8}


@pytest.fixture(scope="module")
def oracle():
    return AnalysisOracle()


@pytest.fixture(scope="module")
def positions(oracle):
    """Reachable positions (engine plane order) and which of them have no legal move."""
    st = oracle.gen_states(5, 8192)
    terminal = np.array([not oracle.legal(s)[0].any() for s in st])
    assert terminal[:N].sum() > 50
    return cb.planes_from_reference_order(st), terminal


@pytest.fixture(scope="module")
def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def weights(seed=31):
    return cb.fold_batchnorm(cb.random_weights(seed))


def dev(states):
    return torch.from_numpy(np.ascontiguousarray(states).view(np.int64)).cuda()


def host(out):
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32) if a.dtype.itemsize == 4 else a


def assert_same(got, ref, keys=KEYS, rows=slice(None)):
    for k in keys:
        if k in ref:
            assert np.array_equal(bits(got[k])[rows], bits(ref[k])[rows]), k


@pytest.mark.parametrize("precision", ["bf16", "fp16", "bf16x3"])
@pytest.mark.parametrize("ms,spe,c_puct,eps", PARAMS)
def test_run_device_equals_run(positions, precision, ms, spe, c_puct, eps):
    st = positions[0][:N]
    seed = 2000 + ms
    a = cb.Analysis(N, ms, spe, c_puct, eps)
    a.set_weights(weights(), precision)
    ref = a.run(st, seed)
    ref_counters = a.counters()
    got = host(a.run_device(dev(st), seed))
    assert_same(got, ref)
    assert got["status"].tolist() == [0, 0]
    assert a.counters() == ref_counters
    no_ev = host(a.run_device(dev(st), seed, evals=False))
    assert "evals" not in no_ev
    assert_same(no_ev, ref, KEYS[:4])
    assert a.counters() == ref_counters


@pytest.mark.parametrize("precision", ["bf16", "bf16x3"])
def test_batch_shapes_equal_the_prefix_of_run(positions, sms, precision):
    k = GAMES_PER_CTA[precision] * sms
    sizes = [1, 2, 623, 624, 625, k - 1, k, k + 1, 3 * k + 5]
    big = max(sizes)
    st, terminal = positions[0][:big], positions[1][:big]
    a = cb.Analysis(big, 64, 16, 1.0, 0.25)
    a.set_weights(weights(7), precision)
    ref = a.run(st, 11)
    st_d = dev(st)
    for n in sizes:
        got = host(a.run_device(st_d[:n], 11))
        assert_same(got, {key: v[:n] for key, v in ref.items()})
        assert got["status"].tolist() == [0, 0], n
    # the device seed stream matters: another seed changes most searched positions
    other = host(a.run_device(st_d, 12))
    searched = ~terminal
    differ = (other["visits"] != ref["visits"]).any(1)
    assert differ[searched].mean() > 0.5
    assert not differ[terminal].any()


def malformed(st, i, kind):
    w0, w1 = int(st[i, 0]), int(st[i, 1])
    if kind == "byte7":
        w1 |= 1 << 56
    elif kind == "side2":
        w1 = (w1 & ~(0xFF << 48)) | (2 << 48)
    elif kind == "frozen":
        occupied = (w0 | (w0 >> 16) | (w0 >> 32)) & 0xFFFF
        sq = next(s for s in range(16) if not (occupied >> s) & 1)
        w0 |= 1 << (48 + sq)
    elif kind == "count":
        h = w1 & 0xFF  # one more base piece in the first hand than the board leaves
        w1 = (w1 & ~0xFF) | (h + 1 if h < 4 else h - 1)
    return np.array([w0, w1], np.uint64)


def test_rejected_states_are_reported_per_position(positions):
    st = positions[0][:512]
    a = cb.Analysis(1024, 48, 8, 1.0, 0.25)
    a.set_weights(weights(3), "bf16")
    # random 128-bit words mixed in: the kernel rejects what cb200_check_states rejects
    rng = np.random.default_rng(4)
    mixed = np.empty((1024, 2), np.uint64)
    mixed[0::2] = st
    mixed[1::2] = rng.integers(0, np.iinfo(np.uint64).max, size=(512, 2), dtype=np.uint64, endpoint=True)
    got = host(a.run_device(dev(mixed), 5))
    invalid = ~cb.check_states(mixed)
    assert invalid.sum() >= 500
    assert np.array_equal(got["results"] == ERR_ARG, invalid)
    assert got["status"].tolist() == [int(invalid.sum()), ERR_ARG]
    # malformed states at chosen indices: move -1, result -1, zeros; every other index as in run
    ref = a.run(st, 6)
    bad = st.copy()
    chosen = {3: "byte7", 50: "side2", 100: "frozen", 200: "count", 511: "count"}
    for i, kind in chosen.items():
        bad[i] = malformed(st, i, kind)
    assert not cb.check_states(bad[list(chosen)]).any()
    got = host(a.run_device(dev(bad), 6))
    idx = np.array(sorted(chosen))
    assert (got["moves"][idx] == -1).all() and (got["results"][idx] == ERR_ARG).all()
    assert (bits(got["values"][idx]) == 0).all()
    assert (got["visits"][idx] == 0).all() and (bits(got["evals"][idx]) == 0).all()
    keep = np.ones(len(st), bool)
    keep[idx] = False
    assert_same(got, ref, rows=keep)
    assert got["status"].tolist() == [len(chosen), ERR_ARG]


def test_overflow_is_reported_per_position(positions, monkeypatch):
    monkeypatch.setenv("CB200_ARENA_NODES", "24")
    a = cb.Analysis(64, 64, 16, 1.0, 0.25)
    monkeypatch.delenv("CB200_ARENA_NODES")
    a.set_weights(weights(2), "bf16")
    st_all, term_all = positions
    terminal = np.flatnonzero(term_all)[:16]
    searched = np.flatnonzero(~term_all)[:48]
    st = np.concatenate([st_all[searched], st_all[terminal]])
    got = host(a.run_device(dev(st), 1))
    over = got["results"] == ERR_OVERFLOW
    assert over.sum() > 0 and not over[48:].any()
    assert (got["moves"][over] == -1).all() and (got["visits"][over] == 0).all()
    assert (bits(got["values"][over]) == 0).all() and (bits(got["evals"][over]) == 0).all()
    assert np.isin(got["results"][48:], [1, 2]).all() and (got["moves"][48:] == -1).all()
    assert got["status"].tolist() == [int(over.sum()), ERR_OVERFLOW]
    again = host(a.run_device(dev(st), 1))
    assert_same(again, got, KEYS + ("status",))
    with pytest.raises(cb.Corintho200Error, match=f"error {ERR_OVERFLOW}"):
        a.run(st, 1)


def test_stream_order_without_host_synchronisation(positions):
    L = cb.lib()
    st_all, term_all = positions
    src = st_all[np.flatnonzero(~term_all)[:2000]]
    n = len(src)
    a = cb.Analysis(n, 64, 16, 1.0, 0.25)
    a.set_weights(weights(9), "bf16")
    a.run_device(dev(src[:16]), 1)  # warm-up: weights and buffers
    torch.cuda.synchronize()
    stream = torch.cuda.Stream()
    try:
        with torch.cuda.stream(stream):
            assert L.cb200_set_stream(stream.cuda_stream) == 0
            x = dev(src)
            mf = torch.empty((n, 4), dtype=torch.int32, device="cuda")
            nxt = torch.empty((n, 2), dtype=torch.int64, device="cuda")
            # the game step writes the states the analysis reads, with nothing between them
            assert L.cb200_game_step_device(n, C.c_void_p(x.data_ptr()), 99, C.c_void_p(mf.data_ptr()),
                                            C.c_void_p(nxt.data_ptr()), None) == 0
            out = a.run_device(nxt, 21)
            copies = {k: v.clone() for k, v in out.items()}  # a torch op on the same stream
            # the call returns while the stream is still busy in front of it
            torch.cuda._sleep(1 << 30)
            a.run_device(nxt, 21, out=out)
            assert not stream.query()
        stream.synchronize()
    finally:
        L.cb200_set_stream(None)
    got = {k: v.cpu().numpy() for k, v in copies.items()}
    states = nxt.cpu().numpy().view(np.uint64)
    assert cb.check_states(states).all()
    ref = a.run(states, 21)
    assert_same(got, ref)
    assert_same(host(out), ref)


def test_graph_capture_and_replay(positions):
    L = cb.lib()
    st = positions[0]
    n = 1000
    a = cb.Analysis(n, 64, 16, 1.0, 0.25)
    a.set_weights(weights(12), "bf16x3")
    static = dev(st[:n])
    out = a.run_device(static, 8)  # warm-up: the first call uploads and allocates
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    stream = torch.cuda.Stream()
    try:
        with torch.cuda.graph(graph, stream=stream):
            assert L.cb200_set_stream(stream.cuda_stream) == 0
            a.run_device(static, 8, out=out)
    finally:
        L.cb200_set_stream(None)
    for lo in (2000, 5000):
        batch = st[lo:lo + n]
        static.copy_(dev(batch))
        graph.replay()
        got = host(out)
        ref = a.run(batch, 8)
        assert_same(got, ref)
        assert got["status"].tolist() == [0, 0]


def test_call_errors_leave_the_object_usable(positions):
    L = cb.lib()
    st = positions[0][:64]
    a = cb.Analysis(64, 16, 4, 1.0, 0.25)
    h = a._h
    st_d = dev(st)
    out = {"moves": torch.zeros(64, dtype=torch.int32, device="cuda"),
           "results": torch.zeros(64, dtype=torch.int32, device="cuda"),
           "values": torch.zeros(64, dtype=torch.float32, device="cuda"),
           "visits": torch.zeros((64, 96), dtype=torch.int32, device="cuda"),
           "evals": torch.zeros((64, 96), dtype=torch.float32, device="cuda"),
           "status": torch.zeros(2, dtype=torch.int32, device="cuda")}
    ptr = {k: C.c_void_p(v.data_ptr()) for k, v in out.items()}

    def raw(n=64, states=None, **over):
        p = dict(ptr, **over)
        states = C.c_void_p(st_d.data_ptr()) if states is None else states
        return L.cb200_analysis_run_device(h, n, states, 4, p["moves"], p["results"], p["values"], p["visits"],
                                           p["evals"], p["status"])
    assert raw() == ERR_STATE  # no weights
    a.set_weights(weights(2), "fp32")
    assert raw() == ERR_STATE
    assert b"fp32" in L.cb200_last_error()
    a.set_weights(weights(2), "bf16")
    assert raw() == 0
    first = host(out)
    assert first["status"].tolist() == [0, 0]
    host_buf = np.zeros(64, np.int32)
    misaligned = torch.zeros(64 * 2 + 2, dtype=torch.int64, device="cuda")
    misaligned[1:129].copy_(st_d.view(-1))
    for rc in (raw(n=0), raw(n=65), raw(moves=None), raw(results=C.c_void_p(host_buf.ctypes.data)),
               raw(states=C.c_void_p(misaligned.data_ptr() + 8))):
        assert rc == ERR_ARG
    # a device run discards an open protocol session
    a.begin(st, 4)
    assert raw() == 0
    assert L.cb200_analysis_num_requests(h) == ERR_STATE
    for v in out.values():
        v.zero_()
    assert raw() == 0
    again = host(out)
    assert_same(again, first, KEYS + ("status",))
    assert_same(again, a.run(st, 4))
