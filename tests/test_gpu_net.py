"""Network kernels and the fused (device-resident) self-play loop."""
import numpy as np
import pytest

import corintho_ai_b200 as cb
from netref import forward_folded
from oracle.pyoracle import synth_eval
from util import run_trainer

pytestmark = pytest.mark.gpu


def sample_positions(oracle, n, seed=1):
    rng = np.random.default_rng(seed)
    rows = []
    while len(rows) < n:
        st = oracle.start()
        for _ in range(40):
            rows.append(oracle.encode(st))
            mask, _ = oracle.legal(st)
            ids = [m for m in range(96) if (mask[m >> 5] >> (m & 31)) & 1]
            if not ids:
                break
            st = oracle.do_move(st, int(rng.choice(ids)))
    return np.stack(rows[:n])


def test_fp32_network_matches_numpy(oracle):
    """Stated tolerance (BASELINE.json north_star): 1e-5 relative in fp32."""
    x = sample_positions(oracle, 1000)
    flat = cb.fold_batchnorm(cb.random_weights(11))
    t = cb.Trainer(64, "", 1, 32, 16)
    t.set_weights(flat, 0, "fp32")
    ev, pr = t.evaluate(x)
    v64, p64 = forward_folded(flat, x, np.float64)
    assert np.max(np.abs(ev - v64) / np.maximum(np.abs(v64), 1e-3)) < 1e-5
    assert np.max(np.abs(pr - p64) / p64) < 1e-5
    assert np.allclose(pr.sum(1), 1.0, atol=1e-5)


def test_fp32_network_ragged_batches(oracle):
    x = sample_positions(oracle, 300, seed=3)
    flat = cb.fold_batchnorm(cb.random_weights(12))
    t = cb.Trainer(32, "", 1, 32, 16)
    t.set_weights(flat, 0, "fp32")
    full_e, full_p = t.evaluate(x)
    for n in (1, 127, 128, 129, 255):
        e, p = t.evaluate(x[:n])
        assert e.tobytes() == full_e[:n].tobytes() and p.tobytes() == full_p[:n].tobytes()


def test_fused_selfplay_equals_oracle_driven_by_the_same_network(oracle):
    """Fused mode keeps everything on the device. Driving the ORACLE with the engine's own
    network outputs (same kernel, so bit-identical evaluations) must reproduce the fused run:
    samples, results and exact simulation counters."""
    flat = cb.fold_batchnorm(cb.random_weights(21))
    cfg = dict(num_games=24, seed=9, max_searches=64, searches_per_eval=16, c_puct=1.0, epsilon=0.25)
    fused = cb.Trainer(cfg["num_games"], "", cfg["seed"], cfg["max_searches"], cfg["searches_per_eval"],
                       cfg["c_puct"], cfg["epsilon"])
    fused.set_weights(flat, 0, "fp32")
    assert fused.run_selfplay(0, stagger=True)
    helper = cb.Trainer(cfg["num_games"], "", 1, 64, cfg["searches_per_eval"])
    helper.set_weights(flat, 0, "fp32")
    o = oracle.trainer(**cfg)
    r = run_trainer(o, lambda req: helper.evaluate(req))
    gs, ev, pr = fused.write_samples()
    assert fused.num_samples() == r["num_samples"]
    assert gs.tobytes() == r["samples"][0].tobytes()
    assert ev.tobytes() == r["samples"][1].tobytes()
    assert pr.tobytes() == r["samples"][2].tobytes()
    assert fused.score().tobytes() == r["score"].tobytes()
    oc, ec = oracle.counters(o), fused.counters()
    assert (oc["simulations"], oc["moves"], oc["leaf_evals"]) == (ec["simulations"], ec["moves"], ec["leaf_evals"])


def test_fused_testing_mode_two_models(oracle):
    """Two-model (gating-match) mode, fused. The device loop evaluates every pending request
    with the model that owns it before the owning side iterates (tp = 0, 1, 0, 1, ...). The
    reference's Python caller instead re-enters doIteration with STALE answer buffers right
    after it flips to_play (main.pyx:151-154) -- a caller-side quirk the external-evaluator
    API reproduces by construction (test_gpu_trainer.py); here the oracle is driven with the
    same clean alternation."""
    fa, fb = cb.fold_batchnorm(cb.random_weights(1)), cb.fold_batchnorm(cb.random_weights(2))
    G, MS, SPE = 16, 32, 8
    t = cb.Trainer(G, "", 4, MS, SPE, 1.0, 0.25, 0, 1, True)
    t.set_weights(fa, 0, "fp32")
    t.set_weights(fb, 1, "fp32")
    assert t.run_selfplay(0)
    assert t.num_samples() == 0 and 0.0 <= float(t.score()) <= 1.0
    h = [cb.Trainer(G, "", 1, 16, SPE) for _ in range(2)]
    h[0].set_weights(fa, 0, "fp32")
    h[1].set_weights(fb, 0, "fp32")
    o = oracle.trainer(num_games=G, seed=4, max_searches=MS, searches_per_eval=SPE, c_puct=1.0,
                       epsilon=0.25, testing=True)
    ev = np.zeros(G * SPE, np.float32)
    pr = np.zeros((G * SPE, 96), np.float32)
    done, tp = False, 0
    while not done:
        n = o.num_requests(tp)
        if n:  # main.pyx:74-81: the "new" model (0) answers to_play==0 requests
            e, p = h[tp].evaluate(o.write_requests(tp))
            ev[:n], pr[:n] = e, p
        done = o.do_iteration(ev, pr, tp)
        tp = 1 - tp
    assert t.score().tobytes() == o.score().tobytes()
    oc, ec = oracle.counters(o), t.counters()
    assert (oc["simulations"], oc["moves"], oc["leaf_evals"]) == (ec["simulations"], ec["moves"], ec["leaf_evals"])
    assert (t.game_results() != 0).all()


def test_fused_testing_mode_two_models_persistent(oracle, monkeypatch):
    """Same match with both networks on the tensor cores: the whole run happens in the persistent
    kernel, where every CTA keeps one row region per model. Compared with the oracle driven by
    the same two networks, and with the engine's own lock-step path."""
    fa, fb = cb.fold_batchnorm(cb.random_weights(5)), cb.fold_batchnorm(cb.random_weights(6))
    G, MS, SPE = 40, 48, 8

    def engine_run():
        t = cb.Trainer(G, "", 4, MS, SPE, 1.0, 0.0, 0, 1, True)
        t.set_weights(fa, 0, "bf16")
        t.set_weights(fb, 1, "bf16")
        t.set_profiling(True)
        assert t.run_selfplay(0)
        return t

    t = engine_run()
    assert t.kernel_times()["fused_tail"]["launches"] >= 1
    h = [cb.Trainer(G, "", 1, 16, SPE) for _ in range(2)]
    h[0].set_weights(fa, 0, "bf16")
    h[1].set_weights(fb, 0, "bf16")
    o = oracle.trainer(num_games=G, seed=4, max_searches=MS, searches_per_eval=SPE, c_puct=1.0,
                       epsilon=0.0, testing=True)
    ev = np.zeros(G * SPE, np.float32)
    pr = np.zeros((G * SPE, 96), np.float32)
    done, tp = False, 0
    while not done:
        n = o.num_requests(tp)
        if n:
            e, p = h[tp].evaluate(o.write_requests(tp))
            ev[:n], pr[:n] = e, p
        done = o.do_iteration(ev, pr, tp)
        tp = 1 - tp
    oc, ec = oracle.counters(o), t.counters()
    assert t.score().tobytes() == o.score().tobytes()
    assert (oc["simulations"], oc["moves"], oc["leaf_evals"]) == (ec["simulations"], ec["moves"], ec["leaf_evals"])
    assert (t.game_results() != 0).all()
    monkeypatch.setenv("CB200_NO_PERSISTENT", "1")
    u = engine_run()
    assert u.kernel_times()["fused_tail"]["launches"] == 0
    assert (u.game_results() == t.game_results()).all() and u.score().tobytes() == t.score().tobytes()
    uc = u.counters()
    assert (uc["simulations"], uc["moves"], uc["leaf_evals"]) == (ec["simulations"], ec["moves"], ec["leaf_evals"])


def test_bf16_tensor_core_network(oracle):
    """tcgen05 bf16 kernel. Stated tolerance (BASELINE.json north_star): 2e-2 in bf16 against
    the fp32 network; against a numpy emulation that rounds weights and activations to bf16 the
    same way (fp32 accumulation) it must be much tighter."""
    x = sample_positions(oracle, 1500, seed=7)
    flat = cb.fold_batchnorm(cb.random_weights(11))
    t = cb.Trainer(128, "", 1, 32, 16)
    t.set_weights(flat, 0, "bf16")
    ev, pr = t.evaluate(x)
    assert np.isfinite(ev).all() and np.isfinite(pr).all()
    assert np.allclose(pr.sum(1), 1.0, atol=1e-3)
    vb, pb = forward_folded(flat, x, np.float64, round_bf16=True)
    v64, p64 = forward_folded(flat, x, np.float64)
    e_emul = np.max(np.abs(pr - pb) / pb), np.max(np.abs(ev - vb))
    e_fp32 = np.max(np.abs(pr - p64) / p64), np.max(np.abs(ev - v64))
    print("bf16 kernel vs bf16 emulation: probs rel %.3e value abs %.3e; vs fp64 net: probs rel %.3e value abs %.3e"
          % (e_emul + e_fp32))
    assert e_emul[0] < 5e-3 and e_emul[1] < 5e-3
    assert e_fp32[0] < 2e-2 and e_fp32[1] < 2e-2
    # ragged batch sizes and row independence
    for n in (1, 127, 129, 255, 257, 1000):
        e2, p2 = t.evaluate(x[:n])
        assert e2.tobytes() == ev[:n].tobytes() and p2.tobytes() == pr[:n].tobytes()


@pytest.mark.parametrize("spe", [16, 20])
def test_fused_selfplay_bf16_equals_oracle_driven_by_the_same_network(oracle, spe):
    """Same as the fp32 fused test with the tensor-core evaluator: the kernel is deterministic
    per position, so the oracle fed with its outputs must reproduce the fused run exactly.
    searches_per_eval 16 ends in the persistent kernel, 20 (more than its 16 rows per game)
    stays in the lock-step loop."""
    flat = cb.fold_batchnorm(cb.random_weights(33))
    cfg = dict(num_games=40, seed=5, max_searches=48, searches_per_eval=spe, c_puct=1.0, epsilon=0.25)
    fused = cb.Trainer(cfg["num_games"], "", cfg["seed"], cfg["max_searches"], cfg["searches_per_eval"],
                       cfg["c_puct"], cfg["epsilon"])
    fused.set_weights(flat, 0, "bf16")
    assert fused.run_selfplay(0, stagger=True)
    helper = cb.Trainer(cfg["num_games"], "", 1, 64, cfg["searches_per_eval"])
    helper.set_weights(flat, 0, "bf16")
    o = oracle.trainer(**cfg)
    r = run_trainer(o, lambda req: helper.evaluate(req))
    gs, ev, pr = fused.write_samples()
    assert fused.num_samples() == r["num_samples"]
    assert gs.tobytes() == r["samples"][0].tobytes()
    assert ev.tobytes() == r["samples"][1].tobytes()
    assert pr.tobytes() == r["samples"][2].tobytes()
    oc, ec = oracle.counters(o), fused.counters()
    assert (oc["simulations"], oc["moves"], oc["leaf_evals"]) == (ec["simulations"], ec["moves"], ec["leaf_evals"])


def test_fused_selfplay_is_independent_of_parking_and_stream_groups(monkeypatch):
    """Scheduling knobs of the fused loop must not change any result: a game that parks in the
    middle of a doIteration (CB200_YIELD budget) resumes exactly where it stopped, and stream
    groups only change which games share a launch. Samples, scores and the exact counters are
    compared byte for byte against the plain lock-step run."""
    flat = cb.fold_batchnorm(cb.random_weights(8))
    G, MS, SPE = 160, 96, 16

    def run(env):
        for k in ("CB200_YIELD", "CB200_YIELD_MIN_LIVE", "CB200_GROUPS"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        t = cb.Trainer(G, "", 77, MS, SPE, 1.0, 0.25)
        t.set_weights(flat, 0, "bf16")
        assert t.run_selfplay(0, stagger=True)
        gs, ev, pr = t.write_samples()
        c = t.counters()
        return (gs.tobytes(), ev.tobytes(), pr.tobytes(), t.score().tobytes(),
                (c["simulations"], c["moves"], c["leaf_evals"])), c["iterations"]

    base, it0 = run({"CB200_YIELD": "0", "CB200_GROUPS": "1"})
    parked, it1 = run({"CB200_YIELD": "7", "CB200_YIELD_MIN_LIVE": "1", "CB200_GROUPS": "1"})
    assert parked == base
    assert it1 > it0  # the tiny budget really did cut iterations into several launches
    grouped, _ = run({"CB200_YIELD": "20", "CB200_YIELD_MIN_LIVE": "1", "CB200_GROUPS": "2"})
    assert grouped == base
    default, _ = run({})
    assert default == base


KNOB_SETS = [
    {"CB200_NO_LIVE_LIST": "1"}, {"CB200_NO_OVERLAP": "1", "CB200_GROUPS": "3"},
    {"CB200_PS_NO_REDEAL": "1"}, {"CB200_PS_REDEAL_PCT": "10", "CB200_PS_REDEAL_MIN": "4"},
    {"CB200_PS_YIELD": "24", "CB200_PS_YIELD_MIN_LIVE": "1"}, {"CB200_PS_CAPACITY": "40"},
    {"CB200_PS_CAPACITY": "2368"}, {"CB200_PS_CAPACITY": "2368", "CB200_PS_YIELD": "24", "CB200_PS_YIELD_MIN_LIVE": "1"},
    {"CB200_GROUPS": "8", "CB200_YIELD": "30", "CB200_YIELD_MIN_LIVE": "16"},
]


def test_fused_selfplay_is_independent_of_every_other_knob(monkeypatch):
    """DESIGN.md section 5's knob table: live lists, network CTA form, persistent re-deal policy,
    persistent parking, take-over threshold -- none may change a byte of the samples, the score or
    the exact counters (600 games: several stream groups, both persistent kernel widths after the
    hand-over)."""
    flat = cb.fold_batchnorm(cb.random_weights(21))
    knobs = sorted({k for ks in KNOB_SETS for k in ks})

    def run(env):
        for k in knobs:
            monkeypatch.delenv(k, raising=False)
        # lock-step loop until 100 games are left (the default would hand 600 games to the
        # persistent kernels at once and leave the lock-step knobs untested), then the persistent tail
        monkeypatch.setenv("CB200_PS_CAPACITY", "100")
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        t = cb.Trainer(600, "", 321, 64, 16, 1.0, 0.25)
        t.set_weights(flat, 0, "bf16")
        assert t.run_selfplay(0, stagger=False)
        gs, ev, pr = t.write_samples()
        c = t.counters()
        return (gs.tobytes(), ev.tobytes(), pr.tobytes(), t.score().tobytes(),
                (c["simulations"], c["moves"], c["leaf_evals"]))

    base = run({})
    t = cb.Trainer(600, "", 321, 64, 16, 1.0, 0.25)   # CB200_PS_CAPACITY=100 is still set: both loops run
    t.set_weights(flat, 0, "bf16")
    t.set_profiling(True)
    assert t.run_selfplay(0, stagger=False)
    kt = t.kernel_times()
    assert kt["game_step"]["launches"] >= 20 and kt["fused_tail"]["launches"] >= 1
    for env in KNOB_SETS:
        assert run(env) == base, env


def test_persistent_tail_equals_lock_step(monkeypatch):
    """Once the live games fit on the device at 8 per SM the run continues in one persistent
    kernel (game step + network per CTA). It must play exactly the games of the lock-step loop,
    also when the run is cut into bounded calls that stop and re-enter the persistent kernel."""
    flat = cb.fold_batchnorm(cb.random_weights(12))
    G, MS, SPE = 96, 80, 16

    def result(t):
        gs, ev, pr = t.write_samples()
        c = t.counters()
        return (gs.tobytes(), ev.tobytes(), pr.tobytes(), t.score().tobytes(),
                (c["simulations"], c["moves"], c["leaf_evals"]))

    monkeypatch.setenv("CB200_NO_PERSISTENT", "1")
    a = cb.Trainer(G, "", 31, MS, SPE, 1.0, 0.25)
    a.set_weights(flat, 0, "bf16")
    assert a.run_selfplay(0, stagger=False)
    base = result(a)
    monkeypatch.delenv("CB200_NO_PERSISTENT")
    b = cb.Trainer(G, "", 31, MS, SPE, 1.0, 0.25)
    b.set_weights(flat, 0, "bf16")
    b.set_profiling(True)
    assert b.run_selfplay(0, stagger=False)
    kt = b.kernel_times()
    assert kt["fused_tail"]["launches"] >= 1 and kt["game_step"]["launches"] >= 1
    assert result(b) == base
    # bounded calls: 40 lock-step iterations, then the persistent kernel 7 rounds at a time
    c = cb.Trainer(G, "", 31, MS, SPE, 1.0, 0.25)
    c.set_weights(flat, 0, "fp16")
    c.set_weights(flat, 0, "bf16")
    done = c.run_selfplay(40, stagger=False)
    calls = 0
    while not done:
        done = c.run_selfplay(7, stagger=False)
        calls += 1
        assert calls < 10000
    assert calls > 3
    assert result(c) == base
    # and a run after reset() starts in lock-step mode again
    c.reset(31)
    assert c.run_selfplay(0, stagger=False)
    assert result(c) == base


def _trained_like_params(seed):
    """Random weights with non-trivial biases and BatchNorm statistics, so that the folded
    biases are non-zero (random init has b = 0, beta = 0)."""
    rng = np.random.default_rng(seed)
    p = cb.random_weights(seed)
    for L in p["layers"]:
        n = L["gamma"].size
        L["gamma"] = rng.uniform(0.5, 1.5, n).astype(np.float32)
        L["beta"] = rng.uniform(-0.3, 0.3, n).astype(np.float32)
        L["mean"] = rng.uniform(-0.1, 0.3, n).astype(np.float32)
        L["var"] = rng.uniform(0.5, 2.0, n).astype(np.float32)
        L["b"] = rng.uniform(-0.2, 0.2, n).astype(np.float32)
    p["head"]["bv"] = rng.uniform(-0.2, 0.2, 1).astype(np.float32)
    p["head"]["bp"] = rng.uniform(-0.5, 0.5, 96).astype(np.float32)
    return p


def test_networks_with_nonzero_biases(oracle):
    """Bias handling: fp32 kernel adds fp32 biases; the tensor-core kernel carries them through
    the GEMM as a bf16 hi + lo pair on two constant-one activation columns."""
    x = sample_positions(oracle, 700, seed=11)
    flat = cb.fold_batchnorm(_trained_like_params(4))
    v64, p64 = forward_folded(flat, x, np.float64)
    t = cb.Trainer(64, "", 1, 32, 16)
    t.set_weights(flat, 0, "fp32")
    ev, pr = t.evaluate(x)
    assert np.max(np.abs(ev - v64) / np.maximum(np.abs(v64), 1e-3)) < 1e-5
    assert np.max(np.abs(pr - p64) / p64) < 1e-5
    t.set_weights(flat, 0, "bf16")
    ev, pr = t.evaluate(x)
    vb, pb = forward_folded(flat, x, np.float64, round_bf16=True)
    e_emul = np.max(np.abs(pr - pb) / pb), np.max(np.abs(ev - vb))
    e_fp = np.max(np.abs(pr - p64) / p64), np.max(np.abs(ev - v64))
    print("nonzero-bias bf16: vs emulation probs rel %.3e value abs %.3e; vs fp64 probs rel %.3e value abs %.3e" % (e_emul + e_fp))
    assert e_emul[0] < 5e-3 and e_emul[1] < 5e-3
    assert e_fp[0] < 2e-2 and e_fp[1] < 2e-2


def _trained_flat():
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    return np.load(os.path.join(root, "tests", "golden", "trained_net.npz"))["flat"]


def test_trained_checkpoint_on_both_kernels(oracle):
    """A shipped reference checkpoint. Its folded BatchNorm scales reach ~240, so fp32 arithmetic
    itself (numpy float32 vs float64 forward) is off by 1.3e-5 absolute on the outputs; the fp32
    kernel must stay within 5e-5 of the float64 network. bf16 operands are too coarse for this
    network (CPU emulation: max value error 0.19, argmax agreement 88 %), which is why the
    tensor-core kernel also takes fp16 operands. On these off-distribution random positions even
    10-bit operands leave a few outliers, so the fp16 bar is: mean absolute error < 5e-3, max
    < 5e-2, argmax agreement > 97 %; the fp32 kernel is the exact evaluator."""
    flat = _trained_flat()
    x = sample_positions(oracle, 600, seed=21)
    v64, p64 = forward_folded(flat, x, np.float64)
    t = cb.Trainer(64, "", 1, 32, 16)
    t.set_weights(flat, 0, "fp32")
    ev, pr = t.evaluate(x)
    assert np.max(np.abs(ev - v64)) < 5e-5 and np.max(np.abs(pr - p64)) < 5e-5
    for prec in ("bf16", "fp16"):
        t.set_weights(flat, 0, prec)
        ev, pr = t.evaluate(x)
        agree = np.mean(pr.argmax(1) == p64.argmax(1))
        print("trained net %s: value err max %.3e mean %.3e | probs err max %.3e mean %.3e | argmax agreement %.3f"
              % (prec, np.max(np.abs(ev - v64)), np.mean(np.abs(ev - v64)), np.max(np.abs(pr - p64)),
                 np.mean(np.abs(pr - p64)), agree))
    assert np.max(np.abs(ev - v64)) < 5e-2 and np.max(np.abs(pr - p64)) < 5e-2
    assert np.mean(np.abs(ev - v64)) < 5e-3 and agree > 0.97


def test_trained_network_beats_random_network():
    """Functional check of the whole engine with real weights: the reference's trained network
    (model 0, 'new') against a random-init network in the two-model gating mode."""
    t = cb.Trainer(64, "", 11, 100, 16, 1.0, 0.25, 0, 1, True)
    t.set_weights(_trained_flat(), 0, "fp16")
    t.set_weights(cb.fold_batchnorm(cb.random_weights(5)), 1, "fp16")
    assert t.run_selfplay(0)
    score = float(t.score())
    print("trained vs random-init network over 64 games: score %.3f" % score)
    assert score > 0.9


def _net_fixture():
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    z = np.load(os.path.join(root, "tests", "golden", "net_fixture.npz"))
    return z, z["positions"].astype(np.float32) / np.float32(4)


def test_kernels_against_the_hand_evaluated_reference_graph():
    """PINNED network parity: the outputs of the reference's own shipped TFLite graph, executed
    operator by operator (tests/golden/make_net_fixture.py), against every CUDA evaluator.
    Stated tolerances (BASELINE.json north_star): fp32 1e-5 relative -- here 5e-5 absolute on
    outputs in [-1, 1] because float32 execution of this graph is itself 1e-5 off its float64
    execution; tensor cores 2e-2, met by the bf16x3 operand mode (single bf16 / fp16 operands
    are reported, not asserted: they miss the bar on trained checkpoints)."""
    z, x = _net_fixture()
    v64, p64 = z["value64"], z["policy64"]
    flat = _trained_flat()
    t = cb.Trainer(64, "", 1, 32, 16)
    t.set_weights(flat, 0, "fp32")
    ev, pr = t.evaluate(x)
    assert np.abs(ev - v64).max() < 5e-5 and np.abs(pr - p64).max() < 5e-5
    assert np.abs(ev - z["value"]).max() < 5e-5 and np.abs(pr - z["policy"]).max() < 5e-5
    for prec in ("bf16", "fp16", "bf16x3"):
        t.set_weights(flat, 0, prec)
        ev, pr = t.evaluate(x)
        print("fixture %-7s value err max %.3e mean %.3e | policy err max %.3e | argmax agreement %.4f"
              % (prec, np.abs(ev - v64).max(), np.abs(ev - v64).mean(), np.abs(pr - p64).max(),
                 np.mean(pr.argmax(1) == p64.argmax(1))))
    # the loop ends on bf16x3
    assert np.abs(ev - v64).max() < 2e-2 and np.abs(pr - p64).max() < 2e-2
    assert np.abs(ev - v64).max() < 2e-3 and np.abs(pr - p64).max() < 2e-3  # what it actually achieves
    assert np.mean(pr.argmax(1) == p64.argmax(1)) > 0.995
    # ragged batches / row independence in the split mode
    for n in (1, 127, 129, 255, 257, 500):
        e2, p2 = t.evaluate(x[:n])
        assert e2.tobytes() == ev[:n].tobytes() and p2.tobytes() == pr[:n].tobytes()


def test_fused_selfplay_bf16x3_equals_oracle_driven_by_the_same_network(oracle):
    """Fused run with the trained checkpoint on the bf16x3 tensor-core path (lock-step loop: the
    split operands need the whole shared memory) == the oracle fed by the same kernel."""
    flat = _trained_flat()
    cfg = dict(num_games=40, seed=8, max_searches=48, searches_per_eval=16, c_puct=1.0, epsilon=0.25)
    fused = cb.Trainer(cfg["num_games"], "", cfg["seed"], cfg["max_searches"], cfg["searches_per_eval"],
                       cfg["c_puct"], cfg["epsilon"])
    fused.set_weights(flat, 0, "bf16x3")
    assert fused.run_selfplay(0, stagger=True)
    helper = cb.Trainer(cfg["num_games"], "", 1, 64, cfg["searches_per_eval"])
    helper.set_weights(flat, 0, "bf16x3")
    o = oracle.trainer(**cfg)
    r = run_trainer(o, lambda req: helper.evaluate(req))
    gs, ev, pr = fused.write_samples()
    assert fused.num_samples() == r["num_samples"]
    assert gs.tobytes() == r["samples"][0].tobytes()
    assert ev.tobytes() == r["samples"][1].tobytes()
    assert pr.tobytes() == r["samples"][2].tobytes()


@pytest.mark.parametrize("testing", [False, True])
def test_bf16x3_persistent_tail_equals_lock_step(monkeypatch, testing):
    """bf16x3 networks (hi + lo operand copies: 154 KB of shared memory for one tile) run the persistent
    kernel at 8 games per CTA; one- and two-model runs must equal the lock-step loop byte for byte."""
    w0, w1 = cb.fold_batchnorm(cb.random_weights(41)), cb.fold_batchnorm(cb.random_weights(42))

    def run():
        t = cb.Trainer(200, "", 17, 64, 16, 1.0, 0.0 if testing else 0.25, 0, 1, testing)
        t.set_weights(w0, 0, "bf16x3")
        if testing:
            t.set_weights(w1, 1, "bf16x3")
        t.set_profiling(True)
        assert t.run_selfplay(0, stagger=False)
        c = t.counters()
        r = (t.score().tobytes(), t.avg_mate_length().tobytes(), (c["simulations"], c["moves"], c["leaf_evals"]))
        if not testing:
            r += tuple(a.tobytes() for a in t.write_samples())
        return r, t.kernel_times()

    monkeypatch.setenv("CB200_NO_PERSISTENT", "1")
    base, kt0 = run()
    assert kt0["fused_tail"]["launches"] == 0
    monkeypatch.delenv("CB200_NO_PERSISTENT")
    got, kt1 = run()
    assert kt1["fused_tail"]["launches"] >= 1
    assert got == base
