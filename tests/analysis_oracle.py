"""TEST INFRASTRUCTURE ONLY: the analysis restatement (tests/analysis_oracle.cpp, the batched DockerMC
on top of the CPU oracle) built into a library of its own and bound with ctypes.

The library is compiled on first use with the oracle's flags into the temporary directory, under a
name derived from the sources, so the repository tree is never written. Besides the analysis object
it carries every oracle entry point (it includes oracle/corintho_oracle.cpp), so one ``AnalysisOracle``
serves as the oracle Trainer too -- which the white-box arena dump needs."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle.pyoracle import OracleLib, _Lib, synth_eval

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SOURCES = [os.path.join(HERE, "analysis_oracle.cpp"), os.path.join(ROOT, "oracle", "corintho_oracle.cpp"),
           os.path.join(ROOT, "oracle", "corintho_oracle.h"), os.path.join(ROOT, "oracle", "oracle_tables.inc")]
# the oracle's flags (oracle/Makefile ORFLAGS)
FLAGS = ["-O2", "-std=c++17", "-fopenmp", "-fPIC", "-Wall", "-Wextra", "-ffp-contract=off"]

_u64p = np.ctypeslib.ndpointer(np.uint64, flags="C_CONTIGUOUS")
_u32p = np.ctypeslib.ndpointer(np.uint32, flags="C_CONTIGUOUS")
_f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
_i64p = np.ctypeslib.ndpointer(np.int64, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")


def build():
    h = hashlib.sha256()
    for p in SOURCES:
        with open(p, "rb") as f:
            h.update(f.read())
    h.update(" ".join(FLAGS).encode())
    out = os.path.join(tempfile.gettempdir(), f"corintho_analysis_oracle_{os.getuid()}_{h.hexdigest()[:16]}.so")
    if not os.path.exists(out):
        tmp = f"{out}.{os.getpid()}.tmp"
        subprocess.run(["/usr/bin/g++", *FLAGS, "-shared", "-o", tmp, SOURCES[0]], check=True,
                       capture_output=True)
        os.replace(tmp, out)
    return out


class AnalysisOracle(OracleLib):
    """OracleLib over the analysis library: the oracle's surface plus analysis(), state_valid() and
    dump_arena()."""

    def __init__(self):
        _Lib.__init__(self, build(), "orc_")
        f = self.lib.orc_trainer_counters
        f.restype, f.argtypes = None, [C.c_void_p, _i64p]
        self._counters = f

    def state_valid(self, st):
        f = self.lib.orc_state_valid
        f.restype, f.argtypes = C.c_int, [_u64p]
        return bool(f(np.ascontiguousarray(st, np.uint64).reshape(2)))

    def analysis(self, *a, **kw):
        return _Analysis(self, *a, **kw)

    def dump_arena(self, trainer, game, arena, cap=1 << 22):
        """(words of one arena of a trainer game, [tree 0 arena, tree 1 arena, spare arena])."""
        f = self.lib.orc_trainer_dump_arena
        f.restype, f.argtypes = C.c_int, [C.c_void_p, C.c_int, C.c_int, _u32p, C.c_int, _i32p]
        words = np.zeros(cap, np.uint32)
        out = np.zeros(3, np.int32)
        n = f(trainer.h, game, arena, words, cap, out)
        return words[:n], out


class _Analysis:
    """The batched DockerMC of tests/analysis_oracle.cpp (orc_analysis_*): states in reference bit
    order; drive with play_analysis()."""

    def __init__(self, L, states, seed=0, max_searches=1600, searches_per_eval=16, c_puct=1.0,
                 epsilon=0.25):
        lib = L.lib

        def fn(name, restype, argtypes):
            f = getattr(lib, "orc_analysis_" + name)
            f.restype, f.argtypes = restype, argtypes
            return f

        self._destroy = fn("destroy", None, [C.c_void_p])
        self._nreq = fn("num_requests", C.c_int, [C.c_void_p])
        self._wreq = fn("write_requests", None, [C.c_void_p, _f32p])
        self._iter = fn("do_iteration", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p])
        self._results = fn("results", None, [C.c_void_p, _i32p, _i32p, _f32p, _i32p, _f32p])
        self._counters = fn("counters", None, [C.c_void_p, _i64p])
        st = np.ascontiguousarray(states, np.uint64).reshape(-1, 2)
        self.n = st.shape[0]
        self.h = fn("create", C.c_void_p, [C.c_int, _u64p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float])(
            self.n, st, seed, max_searches, searches_per_eval, c_puct, epsilon)
        if not self.h:
            raise ValueError("orc_analysis_create rejected its arguments")

    def close(self):
        if self.h:
            self._destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()

    def num_requests(self):
        return self._nreq(self.h)

    def write_requests(self):
        n = self.num_requests()
        out = np.zeros((max(n, 1), 70), np.float32)
        self._wreq(self.h, out)
        return out[:n]

    def do_iteration(self, evals=None, probs=None):
        r = self._iter(self.h, evals.ctypes.data if evals is not None else None,
                       probs.ctypes.data if probs is not None else None)
        if r < 0:
            raise RuntimeError("analysis error (arena/path overflow)")
        return bool(r)

    def results(self):
        n = self.n
        out = {"moves": np.zeros(n, np.int32), "results": np.zeros(n, np.int32),
               "values": np.zeros(n, np.float32), "visits": np.zeros((n, 96), np.int32),
               "evals": np.zeros((n, 96), np.float32)}
        self._results(self.h, out["moves"], out["results"], out["values"], out["visits"], out["evals"])
        return out

    def counters(self):
        out = np.zeros(2, np.int64)
        self._counters(self.h, out)
        return {"simulations": int(out[0]), "leaf_evals": int(out[1])}


def play_analysis(analysis, evaluator=synth_eval, record=None, max_rounds=1_000_000):
    """Drive an analysis object: do_iteration, then evaluate its requests, until every position
    has chosen its move. Returns the number of evaluation rounds."""
    evals = probs = None
    for rounds in range(max_rounds):
        if analysis.do_iteration(evals, probs):
            return rounds
        req = analysis.write_requests()
        if record is not None:
            record.append(req.copy())
        evals, probs = evaluator(req)
        evals = np.ascontiguousarray(evals, np.float32)
        probs = np.ascontiguousarray(probs, np.float32)
    raise RuntimeError("play_analysis did not terminate")
