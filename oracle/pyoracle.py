"""TEST INFRASTRUCTURE ONLY: ctypes loaders for the two CPU checkers.

  RefLib    -> oracle/_ref/libcorintho_ref.so   (the unmodified reference behind ref_harness.cpp)
  OracleLib -> oracle/libcorintho_oracle.so     (this repo's CPU restatement)

Both expose the same function set under the prefixes ``ref_`` / ``orc_`` so tests can run the
same driver against either. Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs import this module; the product package never does.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF_SO = os.path.join(HERE, "_ref", "libcorintho_ref.so")
ORACLE_SO = os.path.join(HERE, "libcorintho_oracle.so")

_u64p = np.ctypeslib.ndpointer(np.uint64, flags="C_CONTIGUOUS")
_u32p = np.ctypeslib.ndpointer(np.uint32, flags="C_CONTIGUOUS")
_f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
_i64p = np.ctypeslib.ndpointer(np.int64, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")


class _Lib:
    """Common surface of the reference shim and the oracle."""

    def __init__(self, path, prefix):
        if not os.path.exists(path):
            raise FileNotFoundError(f"{path} missing: run `make -C oracle` (build() does)")
        self.path = path
        self.prefix = prefix
        self.lib = C.CDLL(path)
        L, p = self.lib, prefix

        def fn(name, restype, argtypes):
            f = getattr(L, p + name)
            f.restype = restype
            f.argtypes = argtypes
            return f

        self._line_breaker = fn("line_breaker", None, [C.c_int, _u32p])
        self._gamma = fn("gamma_sample", C.c_float, [C.c_int])
        self._move_decode = fn("move_decode", None, [C.c_int, _i32p])
        self.encode_place = fn("encode_place", C.c_int, [C.c_int] * 3)
        self.encode_move = fn("encode_move", C.c_int, [C.c_int] * 4)
        self._start = fn("game_start", None, [_u64p])
        self._legal = fn("game_legal", C.c_int, [_u64p, _u32p])
        self._do_move = fn("game_do_move", None, [_u64p, C.c_int, _u64p])
        self._encode = fn("game_encode", None, [_u64p, _f32p])
        self._step_batch = fn("game_step_batch", None,
                              [C.c_int64, _u64p, _u32p, _u32p, _u32p, _u64p, C.c_void_p, C.c_int])
        self._t_create = fn("trainer_create", C.c_void_p,
                            [C.c_int, C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float,
                             C.c_int, C.c_int, C.c_int])
        self._t_destroy = fn("trainer_destroy", None, [C.c_void_p])
        self._t_iter = fn("trainer_do_iteration", C.c_int,
                          [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int])
        self._t_nreq = fn("trainer_num_requests", C.c_int, [C.c_void_p, C.c_int])
        self._t_wreq = fn("trainer_write_requests", None, [C.c_void_p, _f32p, C.c_int])
        self._t_nsamp = fn("trainer_num_samples", C.c_int, [C.c_void_p])
        self._t_wsamp = fn("trainer_write_samples", None, [C.c_void_p, _f32p, _f32p, _f32p])
        self._t_score = fn("trainer_score", C.c_float, [C.c_void_p])
        self._t_mate = fn("trainer_avg_mate_length", C.c_float, [C.c_void_p])
        self._gen = fn("gen_states", C.c_int64, [C.c_uint64, C.c_int64, _u64p])

    # ---- tables
    def line_breaker(self, idx):
        out = np.zeros(3, np.uint32)
        self._line_breaker(idx, out)
        return out

    def gamma_sample(self, i):
        return np.float32(self._gamma(i))

    def move_decode(self, mid):
        out = np.zeros(6, np.int32)
        self._move_decode(mid, out)
        return out

    # ---- rules
    def start(self):
        st = np.zeros(2, np.uint64)
        self._start(st)
        return st

    def legal(self, st):
        mask = np.zeros(3, np.uint32)
        lines = self._legal(np.ascontiguousarray(st, np.uint64), mask)
        return mask, bool(lines)

    def do_move(self, st, move):
        out = np.zeros(2, np.uint64)
        self._do_move(np.ascontiguousarray(st, np.uint64), int(move), out)
        return out

    def encode(self, st):
        out = np.zeros(70, np.float32)
        self._encode(np.ascontiguousarray(st, np.uint64), out)
        return out

    def gen_states(self, seed, n):
        """n reachable states: every position of uniformly random legal play-outs (splitmix64)."""
        out = np.zeros((n, 2), np.uint64)
        self._gen(seed, n, out)
        return out

    def step_batch(self, states, rnd, want_enc=True, threads=1):
        states = np.ascontiguousarray(states, np.uint64).reshape(-1, 2)
        n = states.shape[0]
        rnd = np.ascontiguousarray(rnd, np.uint32)
        masks = np.zeros((n, 3), np.uint32)
        flags = np.zeros(n, np.uint32)
        nxt = np.zeros((n, 2), np.uint64)
        enc = np.zeros((n, 70), np.float32) if want_enc else None
        self._step_batch(n, states, rnd, masks, flags, nxt,
                         enc.ctypes.data if enc is not None else None, threads)
        return masks, flags, nxt, enc

    def trainer(self, *a, **kw):
        return _Trainer(self, *a, **kw)

    def tourney(self, *a, **kw):
        return _Tourney(self, *a, **kw)


class _Trainer:
    """Mirror of the reference Trainer (cpp/include/trainer.h:17-53) over either library."""

    def __init__(self, L, num_games, log_folder="", seed=0, max_searches=1600,
                 searches_per_eval=16, c_puct=1.0, epsilon=0.25, num_logged=0, num_threads=1,
                 testing=False, first_game=0):
        self.L = L
        self.num_games = num_games
        self.spe = searches_per_eval
        if first_game:  # oracle only: a shard of a larger run (the engine's multi-GPU partitioning)
            f = getattr(L.lib, L.prefix + "trainer_create_shard")
            f.restype = C.c_void_p
            f.argtypes = [C.c_int, C.c_int, C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_float,
                          C.c_float, C.c_int, C.c_int, C.c_int]
            self.h = f(first_game, num_games, log_folder.encode(), seed, max_searches,
                       searches_per_eval, c_puct, epsilon, num_logged, num_threads, int(testing))
            return
        self.h = L._t_create(num_games, log_folder.encode(), seed, max_searches,
                             searches_per_eval, c_puct, epsilon, num_logged, num_threads,
                             int(testing))

    def close(self):
        if self.h:
            self.L._t_destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()

    def do_iteration(self, evals=None, probs=None, to_play=-1):
        ep = evals.ctypes.data if evals is not None else None
        pp = probs.ctypes.data if probs is not None else None
        r = self.L._t_iter(self.h, ep, pp, to_play)
        if r < 0:
            raise RuntimeError("trainer error (arena/path overflow)")
        return bool(r)

    def num_requests(self, to_play=-1):
        return self.L._t_nreq(self.h, to_play)

    def write_requests(self, to_play=-1):
        n = self.num_requests(to_play)
        out = np.zeros((max(n, 1), 70), np.float32)
        self.L._t_wreq(self.h, out, to_play)
        return out[:n]

    def num_samples(self):
        return self.L._t_nsamp(self.h)

    def write_samples(self):
        n = self.num_samples()
        gs = np.zeros((max(n, 1) * 8, 70), np.float32)
        ev = np.zeros(max(n, 1) * 8, np.float32)
        pr = np.zeros((max(n, 1) * 8, 96), np.float32)
        self.L._t_wsamp(self.h, gs, ev, pr)
        return gs[:n * 8], ev[:n * 8], pr[:n * 8]

    def score(self):
        return np.float32(self.L._t_score(self.h))

    def avg_mate_length(self):
        return np.float32(self.L._t_mate(self.h))


class _Tourney:
    """Mirror of the reference Tourney (cpp/include/tourney.h:12-46) over either library."""

    def __init__(self, L, num_threads=1, log_folder=""):
        self.L = L
        lib, p = L.lib, L.prefix

        def fn(name, restype, argtypes):
            f = getattr(lib, p + name)
            f.restype, f.argtypes = restype, argtypes
            return f

        self._destroy = fn("tourney_destroy", None, [C.c_void_p])
        self._add_player = fn("tourney_add_player", None,
                              [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int])
        self._add_match = fn("tourney_add_match", None, [C.c_void_p, C.c_int, C.c_int, C.c_int])
        self._all_done = fn("tourney_all_done", C.c_int, [C.c_void_p])
        self._nreq = fn("tourney_num_requests", C.c_int, [C.c_void_p, C.c_int])
        self._wreq = fn("tourney_write_requests", None, [C.c_void_p, _f32p, C.c_int])
        self._iter = fn("tourney_do_iteration", None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int])
        self._wscores = fn("tourney_write_scores", None, [C.c_void_p, C.c_char_p])
        self.h = fn("tourney_create", C.c_void_p, [C.c_int, C.c_char_p])(num_threads, log_folder.encode())
        self.max_rows = 0   # upper bound of one model's request rows (sum of searches_per_eval)
        self.model_ids = []
        self._spe = {}

    def close(self):
        if self.h:
            self._destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()

    def add_player(self, player_id, model_id, max_searches=1600, searches_per_eval=16, c_puct=1.0,
                   epsilon=0.25, random=False):
        self._add_player(self.h, player_id, model_id, max_searches, searches_per_eval, c_puct,
                         epsilon, int(random))
        self._spe[player_id] = searches_per_eval
        if model_id not in self.model_ids:
            self.model_ids.append(model_id)

    def add_match(self, player1, player2, logging=False):
        self._add_match(self.h, player1, player2, int(logging))
        self.max_rows += self._spe[player1] + self._spe[player2]

    def all_done(self):
        return bool(self._all_done(self.h))

    def num_requests(self, model_id):
        return self._nreq(self.h, model_id)

    def write_requests(self, model_id):
        n = self.num_requests(model_id)
        out = np.zeros((max(n, 1), 70), np.float32)
        self._wreq(self.h, out, model_id)
        return out[:n]

    def do_iteration(self, evals, probs, model_id):
        self._iter(self.h, evals.ctypes.data, probs.ctypes.data, model_id)

    def scores(self):
        """writeScores (tourney.cpp:34-42) parsed back: rows (player1, player2, score)."""
        import tempfile
        with tempfile.NamedTemporaryFile("r", suffix=".txt") as f:
            self._wscores(self.h, f.name.encode())
            rows = [ln.split() for ln in open(f.name).read().splitlines() if ln.strip()]
        return [(int(a), int(b), float(c)) for a, b, c in rows]


class RefLib(_Lib):
    def __init__(self):
        super().__init__(REF_SO, "ref_")

    def space_symmetry(self, k, j):
        return self.lib.ref_space_symmetry(k, j)

    def move_symmetry(self, k, j):
        return self.lib.ref_move_symmetry(k, j)


class OracleLib(_Lib):
    def __init__(self):
        super().__init__(ORACLE_SO, "orc_")
        f = self.lib.orc_trainer_counters
        f.restype = None
        f.argtypes = [C.c_void_p, _i64p]
        self._counters = f

    def game_results(self, trainer):
        f = self.lib.orc_trainer_game_results
        f.restype, f.argtypes = None, [C.c_void_p, _i32p]
        out = np.zeros(trainer.num_games, np.int32)
        f(trainer.h, out)
        return out

    def counters(self, trainer):
        out = np.zeros(3, np.int64)
        self._counters(trainer.h, out)
        return {"simulations": int(out[0]), "moves": int(out[1]), "leaf_evals": int(out[2])}


def have_ref():
    return os.path.exists(REF_SO)


# ---- deterministic synthetic evaluator shared by every parity test --------------------------
def synth_eval(game_states):
    """Pure function of the 70-float request rows -> (eval[n] in [-1,1), probs[n,96] in (0,1]).

    Integer hashing only, so it is bit-reproducible everywhere. Like the reference's own tests
    (tests/cpp/trainer_test.cpp:37-49) the probabilities are NOT normalised; the search
    renormalises over legal moves (trainmc.cpp:212-234).
    """
    gs = np.ascontiguousarray(game_states, np.float32).reshape(-1, 70)
    n = gs.shape[0]
    q = np.rint(gs * 4.0).astype(np.uint64)  # entries are multiples of 1/4
    h = np.full(n, 0x9E3779B97F4A7C15, np.uint64)
    with np.errstate(over="ignore"):
        for j in range(70):
            h = (h ^ q[:, j]) * np.uint64(0x100000001B3)
            h ^= h >> np.uint64(29)
        ev = ((h >> np.uint64(11)) & np.uint64(0xFFFF)).astype(np.float32) / np.float32(32768.0) \
            - np.float32(1.0)
        k = np.arange(96, dtype=np.uint64)[None, :]
        m = (h[:, None] + k * np.uint64(0xD6E8FEB86659FD93))
        m ^= m >> np.uint64(32)
        m *= np.uint64(0xD6E8FEB86659FD93)
        m ^= m >> np.uint64(32)
        pr = ((m & np.uint64(0xFFFF)).astype(np.float32) + np.float32(1.0)) / np.float32(65536.0)
    return ev.astype(np.float32), np.ascontiguousarray(pr, np.float32)


def play_out(trainer, evaluator=synth_eval, to_play=-1, record=None, max_iters=10_000_000,
             allow_empty=False):
    """Drive a Trainer-like object exactly like main.pyx:142-170 (play_games).

    ``record``: optional list receiving (n_requests, request_rows.copy()) per iteration.
    Returns the number of evaluation rounds.
    """
    G, spe = trainer.num_games, trainer.spe
    evals = np.zeros(G * spe, np.float32)
    probs = np.zeros((G * spe, 96), np.float32)
    rounds = 0
    for _ in range(max_iters):
        if trainer.do_iteration(evals, probs, to_play):
            return rounds
        n = trainer.num_requests(to_play)
        if n == 0:
            if to_play != -1:
                to_play = 1 - to_play
                continue
            if allow_empty:  # a shard whose staggered games have not started yet
                continue
            raise RuntimeError("No requests during training")
        req = trainer.write_requests(to_play)
        if record is not None:
            record.append((to_play, req.copy()))
        e, p = evaluator(req)
        evals[:n] = e
        probs[:n] = p
        rounds += 1
    raise RuntimeError("play_out did not terminate")


def play_tourney(tourney, evaluators=None, record=None, max_rounds=10_000_000):
    """Drive a Tourney-like object exactly like rating/tourney.pyx:112-173 (play_games): for every
    model id (negative ids are the random players' dummy models) fetch the requests, evaluate,
    doIteration -- the answer buffers persist between calls as in the reference loop.

    ``evaluators``: {model_id: f(rows) -> (eval, probs)}; default synth_eval for every model.
    ``record``: optional list receiving (model_id, request_rows.copy()) per evaluation.
    """
    rows = max(tourney.max_rows, 1)
    evals = np.zeros(rows, np.float32)
    probs = np.zeros((rows, 96), np.float32)
    rounds = 0
    while not tourney.all_done():
        for mid in tourney.model_ids:
            n = tourney.num_requests(mid) if mid >= 0 else 0
            if n > 0:
                req = tourney.write_requests(mid)
                if record is not None:
                    record.append((mid, req.copy()))
                f = (evaluators or {}).get(mid, synth_eval)
                e, p = f(req)
                evals[:n] = e
                probs[:n] = p
            tourney.do_iteration(evals, probs, mid)
        rounds += 1
        if rounds > max_rounds:
            raise RuntimeError("play_tourney did not terminate")
    return rounds
