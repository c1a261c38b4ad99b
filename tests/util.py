"""Shared helpers for the test-suite (numpy only)."""
import hashlib
import os
import subprocess

import numpy as np

M64 = np.uint64(0xFFFFFFFFFFFFFFFF)

# A checkout of the original corintho-ai project (the directory that holds corintho_ai/), where
# oracle/Makefile builds the compiled reference from: the tests that compare with its sources or
# shipped models directly skip without one.
_ORACLE = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle")
_r = subprocess.run(["make", "-s", "--no-print-directory", "-C", _ORACLE, "print-ref"],
                    capture_output=True, text=True)
REFERENCE = _r.stdout.strip() if _r.returncode == 0 else ""
NO_REFERENCE = ("no checkout of the original project at %r (oracle/Makefile REF; set CORINTHO_AI_REFERENCE)"
                % REFERENCE)


def reference_file(rel):
    """Path of `rel` inside the original project's checkout, or None when it is not available."""
    p = os.path.join(REFERENCE, rel) if REFERENCE else ""
    return p if p and os.path.exists(p) else None


def step_rnd(seed, n):
    """numpy twin of cb200::step_rnd (corintho_ai_b200/csrc/rules.cuh): per-state random word."""
    i = np.arange(n, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = np.uint64(seed) + (i + np.uint64(1)) * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    return (z >> np.uint64(32)).astype(np.uint32)


def sha(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def run_trainer(trainer, evaluator, testing=False, allow_empty=False):
    """Drive any Trainer-like object through main.pyx:142-170's loop and digest everything the
    reference API exposes: per-round request counts + request rows, samples, score, mate length."""
    from oracle.pyoracle import play_out
    rec = []
    rounds = play_out(trainer, evaluator=evaluator, to_play=0 if testing else -1, record=rec,
                      allow_empty=allow_empty)
    counts = np.array([r.shape[0] for _, r in rec], np.int32)
    tps = np.array([tp for tp, _ in rec], np.int32)
    req_hash = sha(*[r for _, r in rec]) if rec else sha(np.zeros(0))
    out = {"rounds": rounds, "counts": counts, "to_play": tps, "req_hash": req_hash,
           "num_samples": trainer.num_samples(), "score": np.float32(trainer.score()),
           "mate": np.float32(trainer.avg_mate_length())}
    if not testing:
        gs, ev, pr = trainer.write_samples()
        out["samples"] = (gs, ev, pr)
        out["samples_hash"] = sha(gs, ev, pr)
    return out


TRAINER_GRID = [
    # (num_games, seed, max_searches, spe, c_puct, epsilon, testing)
    (1, 12345, 1, 1, 1.0, 0.25, False),
    (3, 12345, 2, 1, 1.0, 0.25, False),
    (3, 12345, 2, 2, 1.0, 0.25, False),
    (3, 12345, 16, 1, 1.0, 0.25, False),
    (3, 12345, 16, 16, 1.0, 0.25, False),
    (3, 12345, 96, 16, 1.0, 0.25, False),
    (3, 12345, 96, 96, 1.0, 0.25, False),
    (3, 12345, 400, 16, 1.0, 0.25, False),
    (1, 12345, 400, 400, 1.0, 0.25, False),
    (16, 7, 200, 16, 3.0, 0.25, False),
    (8, 99, 800, 16, 1.0, 0.0, False),
    (8, 5, 100, 8, 1.0, 0.25, True),
    (6, 21, 64, 16, 1.0, 0.0, True),
    (4, 11, 1600, 16, 3.0, 0.25, False),
]


def grid_key(cfg):
    g, seed, ms, spe, cp, eps, testing = cfg
    return f"g{g}_s{seed}_m{ms}_e{spe}_c{cp}_x{eps}_t{int(testing)}"


# ---- Tourney / Match (SURVEY 8f-1) -------------------------------------------------------------
# name -> (players [(player_id, model_id, max_searches, spe, c_puct, epsilon, random)], matches)
TOURNEY_CASES = {
    "two_models": ([(0, 0, 64, 8, 1.0, 0.25, False), (1, 1, 48, 4, 1.5, 0.1, False)],
                   [(0, 1), (1, 0), (0, 1), (1, 0), (0, 0)]),
    "with_random": ([(0, 0, 64, 8, 1.0, 0.25, False), (1, 1, 48, 4, 1.5, 0.1, False),
                     (2, -1, 1, 1, 1.0, 0.25, True), (3, 0, 32, 16, 1.0, 0.0, False)],
                    [(0, 1), (1, 0), (0, 2), (2, 1), (3, 0), (1, 3), (2, 3), (2, 2)]),
    "deeper": ([(10, 3, 200, 16, 1.0, 0.25, False), (11, 5, 120, 16, 2.0, 0.0, False),
                (12, -2, 1, 1, 1.0, 0.25, True)],
               [(10, 11), (11, 10), (12, 10), (11, 12), (10, 10)]),
}


def make_tourney(L, name, num_threads=2):
    players, matches = TOURNEY_CASES[name]
    t = L.tourney(num_threads, "")
    for pl in players:
        t.add_player(*pl)
    for a, b in matches:
        t.add_match(a, b)
    return t


def run_tourney(tourney, evaluators=None):
    """Drive a Tourney-like object through rating/tourney.pyx:112-173's loop and digest what
    the reference API exposes: per-evaluation model id + request rows, and the final scores."""
    import hashlib
    from oracle.pyoracle import play_tourney
    rec = []
    rounds = play_tourney(tourney, evaluators, record=rec)
    h = hashlib.sha256()
    for mid, req in rec:
        h.update(np.int32(mid).tobytes())
        h.update(np.ascontiguousarray(req, np.float32).tobytes())
    return {"rounds": rounds, "models": np.array([m for m, _ in rec], np.int32),
            "counts": np.array([r.shape[0] for _, r in rec], np.int32),
            "req_hash": h.hexdigest(),
            "scores": np.array(tourney.scores(), np.float64).reshape(-1, 3)}


# ---- per-game text logs (SURVEY 8f-3): name -> (Trainer kwargs, first to_play of the driver) ----
LOG_CASES = {
    "train": (dict(num_games=5, seed=7, max_searches=40, searches_per_eval=8, c_puct=1.0, epsilon=0.25,
                   num_logged=3), -1),
    "test": (dict(num_games=4, seed=11, max_searches=32, searches_per_eval=4, c_puct=1.5, epsilon=0.0,
                  num_logged=2, testing=True), 0),
}

LOGGED_MATCHES = (0, 2, 3, 7)  # indices into TOURNEY_CASES["with_random"][1] written as text logs
