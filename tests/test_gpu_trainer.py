"""Self-play engine (external-evaluator mode, through the C ABI) vs the golden transcripts that
were generated from the compiled reference, and vs the oracle on further configurations.
Bit-exact: every request row of every round, all samples, score and mate length."""
import os

import numpy as np
import pytest

import corintho_ai_b200 as cb
from diag import first_divergence
from oracle.pyoracle import ADVERSARIAL_EVALUATORS, play_out, synth_eval
from test_oracle_trainer import check_against_golden
from util import TRAINER_GRID, grid_key, run_trainer

pytestmark = pytest.mark.gpu


def make_engine(cfg, **kw):
    g, s, ms, spe, cp, eps, testing = cfg
    return cb.Trainer(g, "", s, ms, spe, cp, eps, 0, 1, testing, **kw)


def make_oracle(oracle, cfg):
    g, s, ms, spe, cp, eps, testing = cfg
    return oracle.trainer(num_games=g, seed=s, max_searches=ms, searches_per_eval=spe, c_puct=cp,
                          epsilon=eps, testing=testing)


def explain(oracle, cfg):
    return first_divergence(lambda: make_engine(cfg), lambda: make_oracle(oracle, cfg), oracle,
                            synth_eval, cfg[6])


@pytest.mark.parametrize("cfg", TRAINER_GRID, ids=grid_key)
def test_engine_matches_golden_transcripts(oracle, cfg):
    r = run_trainer(make_engine(cfg), synth_eval, cfg[6])
    try:
        check_against_golden(r, cfg)
    except AssertionError:
        pytest.fail("engine != reference transcript; first divergence: " + explain(oracle, cfg))


EXTRA = [
    (64, 12345, 200, 16, 1.0, 0.25, False),   # BASELINE.json configs[0] shape
    (40, 77, 8, 4, 1.0, 0.25, False),         # staggered start: 40 games / 8 searches -> div 5
    (33, 5, 50, 50, 3.0, 0.25, False),        # spe == max_searches, >32 games (ragged CTA)
    (10, 2, 1600, 16, 1.0, 0.0, True),        # evaluation-match shape: 1600 sims, no noise
]


@pytest.mark.parametrize("cfg", EXTRA, ids=grid_key)
def test_engine_matches_oracle(oracle, cfg):
    a = run_trainer(make_oracle(oracle, cfg), synth_eval, cfg[6])
    e = make_engine(cfg)
    b = run_trainer(e, synth_eval, cfg[6])
    ok = (a["rounds"] == b["rounds"] and (a["counts"] == b["counts"]).all() and a["req_hash"] == b["req_hash"]
          and a["score"].tobytes() == b["score"].tobytes() and a["mate"].tobytes() == b["mate"].tobytes()
          and (cfg[6] or a["samples_hash"] == b["samples_hash"]))
    if not ok:
        pytest.fail("engine != oracle; first divergence: " + explain(oracle, cfg))
    o = make_oracle(oracle, cfg)
    run_trainer(o, synth_eval, cfg[6])
    oc, ec = oracle.counters(o), e.counters()
    assert (oc["simulations"], oc["moves"], oc["leaf_evals"]) == (ec["simulations"], ec["moves"], ec["leaf_evals"])


@pytest.mark.parametrize("evaluator", sorted(ADVERSARIAL_EVALUATORS))
@pytest.mark.parametrize("cfg", [(24, 9, 100, 8, 1.0, 0.25, False), (8, 3, 300, 16, 1.0, 0.0, True)],
                         ids=grid_key)
def test_engine_matches_oracle_with_degenerate_evaluators(oracle, cfg, evaluator):
    """Tie storms, all-zero legal probabilities and subnormal probabilities, in training and
    testing mode: the PUCT tie-breaks, move choice and the NaN / inf prior paths."""
    f = ADVERSARIAL_EVALUATORS[evaluator]
    a = run_trainer(make_oracle(oracle, cfg), f, cfg[6])
    b = run_trainer(make_engine(cfg), f, cfg[6])
    assert a["rounds"] == b["rounds"] and (a["counts"] == b["counts"]).all()
    assert a["req_hash"] == b["req_hash"]
    assert a["score"].tobytes() == b["score"].tobytes() and a["mate"].tobytes() == b["mate"].tobytes()
    assert cfg[6] or a["samples_hash"] == b["samples_hash"]


def test_sharded_trainers_equal_single_trainer():
    """Multi-GPU partitioning rule (SURVEY.md 8e): shards of one seed stream reproduce the
    single-trainer run game by game. In the 1 300-game run the second shard starts before output
    624 of the seed stream and ends after output 1 248, so its seeds come from three MT19937
    blocks, the first of them entered part-way."""
    for (games, seed, max_searches, spe), shards in (((12, 31, 32, 8), ((0, 5), (5, 7))),
                                                     ((1300, 17, 4, 4), ((0, 600), (600, 700)))):
        whole = make_engine((games, seed, max_searches, spe, 1.0, 0.25, False))
        play_out(whole, synth_eval)
        st_w, pr_w, lb_w, go_w = whole.raw_samples()
        parts = []
        for first, cnt in shards:
            t = cb.Trainer(cnt, "", seed, max_searches, spe, 1.0, 0.25, 0, 1, False, total_games=games,
                           first_game=first)
            # shards of a staggered run start later; drive them with the same loop
            play_out(t, synth_eval, allow_empty=True)
            st, pr, lb, go = t.raw_samples()
            parts.append((st, pr, lb, go + first))
        st = np.concatenate([p[0] for p in parts])
        assert st.tobytes() == st_w.tobytes()
        assert np.concatenate([p[1] for p in parts]).tobytes() == pr_w.tobytes()
        assert np.concatenate([p[2] for p in parts]).tobytes() == lb_w.tobytes()
        assert (np.concatenate([p[3] for p in parts]) == go_w).all()


def test_write_scores_and_errors(tmp_path):
    t = make_engine((4, 3, 16, 4, 1.0, 0.25, False))
    run_trainer(t, synth_eval)
    f = tmp_path / "score_verbose.txt"
    t.writeScores(str(f))
    txt = f.read_text().splitlines()
    assert txt[0].startswith("First player wins: ") and len(txt) == 6
    with pytest.raises(cb.Corintho200Error):
        cb.Trainer(0, "", 1, 16, 4)
    with pytest.raises(cb.Corintho200Error):
        cb.Trainer(2, "", 1, 4, 16)  # max_searches < searches_per_eval (trainer.cpp:30)


def test_arena_overflow_fails_loudly(monkeypatch):
    monkeypatch.setenv("CB200_ARENA_NODES", "20")
    t = make_engine((2, 3, 200, 16, 1.0, 0.25, False))
    with pytest.raises(cb.Corintho200Error):
        run_trainer(t, synth_eval)


def test_raw_samples_device_rows_match_host_rows():
    import torch
    from corintho_ai_b200.dist import device_rows_as_tensor, pack_raw_samples
    t = make_engine((6, 3, 24, 8, 1.0, 0.25, False))
    run_trainer(t, synth_eval)
    st, pr, lb, go = t.raw_samples()
    ptr, n = t.raw_samples_device()
    rows = device_rows_as_tensor(ptr, n, 102, torch.device("cuda", 0)).cpu().numpy()
    assert n == st.shape[0]
    assert rows.tobytes() == pack_raw_samples(st, pr, lb, go, first_game=0).tobytes()


def test_streamed_samples_equal_write_samples():
    """Streaming sample output (finished games' rows copied to pinned host memory during the
    run, completion order) holds exactly Trainer::writeSamples' rows: a stable sort by game
    index restores trainer.cpp:103-113's order byte for byte. Also across reset()."""
    flat = cb.fold_batchnorm(cb.random_weights(4))
    t = cb.Trainer(300, "", 3, 48, 16, 1.0, 0.25)
    t.set_weights(flat, 0, "bf16")
    t.stream_samples()
    for seed in (3, 11):
        t.reset(seed)
        assert t.run_selfplay(0, stagger=False)
        gs, ev, pr, game_of = t.streamed_samples()
        assert game_of.shape[0] == t.num_samples()
        assert len(np.unique(game_of)) == 300
        order = np.argsort(game_of, kind="stable")
        rows = (order[:, None] * 8 + np.arange(8)[None, :]).ravel()
        g2, e2, p2 = t.write_samples()
        assert gs[rows].tobytes() == g2.tobytes()
        assert ev[rows].tobytes() == e2.tobytes()
        assert pr[rows].tobytes() == p2.tobytes()
    # a capacity that is too small is reported, and the classic path still works
    t.stream_samples(100)
    t.reset(3)
    assert t.run_selfplay(0, stagger=False)
    with pytest.raises(cb.Corintho200Error):
        t.streamed_samples()
    assert t.write_samples()[0].shape[0] == t.num_samples() * 8


def test_sample_folder_written_from_the_engine(tmp_path, oracle):
    """SURVEY 8f-2 end to end: the CUDA Trainer's samples go through save_samples into the
    reference's on-disk layout (main.pyx:189-204) and equal the oracle's for the same run."""
    from corintho_ai_b200.samples import load_samples, save_samples
    cfg = (6, 21, 64, 16, 1.0, 0.25, False)
    eng = make_engine(cfg)
    run_trainer(eng, synth_eval)
    rows = save_samples(eng, str(tmp_path / "samples" / "gen_3"))
    assert rows == eng.num_samples() * 8 and rows > 0
    for name in ("game_states", "evaluation_labels", "probability_labels"):
        z = np.load(tmp_path / "samples" / "gen_3" / (name + ".npz"))
        assert z.files == ["arr_0"] and z["arr_0"].dtype == np.float32
    gs, ev, pr = load_samples(str(tmp_path / "samples" / "gen_3"))
    o = oracle.trainer(num_games=6, seed=21, max_searches=64, searches_per_eval=16, c_puct=1.0, epsilon=0.25)
    r = run_trainer(o, synth_eval)
    assert gs.tobytes() == r["samples"][0].tobytes()
    assert ev.tobytes() == r["samples"][1].tobytes()
    assert pr.tobytes() == r["samples"][2].tobytes()


def test_raw_sample_buffer_survives_growth_of_the_augmented_buffer():
    """Regression (advisor, round 1): write_samples used to free the raw-sample device buffer
    when its own buffer grew; the next raw_samples_device then wrote into (or freed again) memory
    it no longer owned. Sequence: few samples -> both buffers sized small -> many samples -> the
    augmented buffer grows -> raw rows again."""
    import torch
    from corintho_ai_b200.dist import device_rows_as_tensor
    flat = cb.fold_batchnorm(cb.random_weights(2))
    t = cb.Trainer(96, "", 5, 48, 16, 1.0, 0.25)
    t.set_weights(flat, 0, "fp32")
    assert not t.run_selfplay(12, stagger=False)  # a few moves per game only
    few = t.num_samples()
    assert few > 0
    t.write_samples()
    ptr0, n0 = t.raw_samples_device()
    assert n0 == few
    done = t.run_selfplay(0, stagger=False)
    assert done and t.num_samples() * 8 > (few * 8) * 5 // 4 + 1024  # the cached buffer must grow
    t.write_samples()
    ptr1, n1 = t.raw_samples_device()
    st, pr, lb, go = t.raw_samples()
    assert n1 == t.num_samples()
    dev_rows = device_rows_as_tensor(ptr1, n1, 102, torch.device("cuda", 0)).cpu().numpy()
    assert np.array_equal(np.ascontiguousarray(dev_rows[:, 4:100]), pr)
    assert np.array_equal(dev_rows[:, 100], lb)
    # and once more after the buffers are warm
    ptr2, n2 = t.raw_samples_device()
    assert (ptr2, n2) == (ptr1, n1)


def test_nccl_allgather_single_rank_returns_own_rows():
    """cb200_trainer_allgather_samples with a one-rank NCCL communicator made through the C ABI
    (unique id -> comm): the result is the rank's own raw rows, in order."""
    import torch
    from corintho_ai_b200.dist import device_rows_as_tensor
    idbuf = np.zeros(128, np.uint8)
    L = cb.lib()
    assert L.cb200_nccl_unique_id(idbuf.ctypes.data) == 0
    comm = L.cb200_nccl_comm_create(0, 1, idbuf.ctypes.data)
    assert comm
    t = cb.Trainer(32, "", 9, 32, 8, 1.0, 0.25)
    t.set_weights(cb.fold_batchnorm(cb.random_weights(1)), 0, "fp32")
    assert t.run_selfplay(0)
    ptr, n, counts = t.allgather_samples(comm, 1)
    st, pr, lb, go = t.raw_samples()
    assert n == t.num_samples() and counts.tolist() == [n]
    rows = device_rows_as_tensor(ptr, n, 102, torch.device("cuda", 0)).cpu().numpy()
    assert np.array_equal(np.ascontiguousarray(rows[:, 4:100]), pr) and np.array_equal(rows[:, 100], lb)
    assert np.array_equal(np.ascontiguousarray(rows[:, 101]).view(np.int32), go)
    import ctypes
    L.cb200_nccl_comm_destroy(ctypes.c_void_p(comm))
