"""corintho_ai_b200 -- host-side mirror of the reference's self-play interface over the
B200 engine (libcorintho_b200.so, C ABI in include/corintho_b200.h).

The class :class:`Trainer` has the member names, argument meaning and call protocol of the
reference's C++ ``Trainer`` (corintho_ai/cpp/include/trainer.h:17-53) as bound by its Cython
layer (corintho_ai/python/main.pyx:17-38): ``doIteration / num_requests / writeRequests /
writeSamples / num_samples / score / avg_mate_length / writeScores``. There is no CPU
fallback: importing works anywhere, but every compute call raises ``Corintho200Error`` unless
the CUDA library is built and a B200-class GPU is usable.
"""
import ctypes as C
import os

import numpy as np

__all__ = ["Trainer", "Tourney", "Analysis", "check_states", "Corintho200Error", "game_step", "lib",
           "build", "NUM_MOVES", "STATE_SIZE", "WEIGHT_FLOATS", "planes_from_reference_order", "reference_order_from_planes",
           "random_weights", "fold_batchnorm"]

NUM_MOVES = 96      # util.h:43
STATE_SIZE = 70     # util.h:41
NUM_SYMMETRIES = 8  # util.h:47
WEIGHT_FLOATS = 127997

_HERE = os.path.dirname(os.path.abspath(__file__))
# CB200_LIB selects another build of the same library (the instrumented `make prof` variant)
LIB_PATH = os.environ.get("CB200_LIB") or os.path.join(_HERE, "libcorintho_b200.so")


class Corintho200Error(RuntimeError):
    pass


_lib = None


def build(verbose=False):
    """Compile libcorintho_b200.so in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    import subprocess
    r = subprocess.run(["make", "-C", os.path.join(_HERE, "csrc")], capture_output=True, text=True)
    if verbose or r.returncode != 0:
        print(r.stdout, r.stderr)
    if r.returncode != 0:
        raise Corintho200Error("building libcorintho_b200.so failed")
    return LIB_PATH


def lib():
    """Load the CUDA library (fails loudly when it has not been built)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise Corintho200Error(
            f"{LIB_PATH} is missing: the CUDA extension is not built "
            "(run `python -c 'import __graft_entry__ as g; g.build()'`). There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, u64, f32 = C.c_void_p, C.c_int, C.c_int64, C.c_uint64, C.c_float
    sig = {
        "cb200_last_error": (C.c_char_p, []),
        "cb200_device_count": (i32, []),
        "cb200_set_device": (i32, [i32]),
        "cb200_set_stream": (i32, [vp]),
        "cb200_launch_count": (i64, []),
        "cb200_game_step": (i32, [i64, vp, u64, vp, vp, vp]),
        "cb200_game_step_device": (i32, [i64, vp, u64, vp, vp, vp]),
        "cb200_trainer_create": (vp, [i32, C.c_char_p, i32, i32, i32, f32, f32, i32, i32, i32]),
        "cb200_trainer_create_shard": (vp, [i32, i32, i32, C.c_char_p, i32, i32, i32, f32, f32,
                                            i32, i32]),
        "cb200_trainer_destroy": (None, [vp]),
        "cb200_trainer_do_iteration": (i32, [vp, vp, vp, i32]),
        "cb200_trainer_num_requests": (i32, [vp, i32]),
        "cb200_trainer_write_requests": (i32, [vp, vp, i32]),
        "cb200_trainer_num_samples": (i32, [vp]),
        "cb200_trainer_write_samples": (i32, [vp, vp, vp, vp]),
        "cb200_trainer_score": (f32, [vp]),
        "cb200_trainer_avg_mate_length": (f32, [vp]),
        "cb200_trainer_write_scores": (i32, [vp, C.c_char_p]),
        "cb200_trainer_counters": (i32, [vp, vp]),
        "cb200_trainer_write_raw_samples": (i32, [vp, vp, vp, vp, vp]),
        "cb200_trainer_game_results": (i32, [vp, vp]),
        "cb200_trainer_raw_samples_device": (i32, [vp, vp, vp]),
        "cb200_trainer_stream_samples": (i32, [vp, i64]),
        "cb200_trainer_streamed_samples": (i32, [vp, vp, vp, vp, vp, vp]),
        "cb200_nccl_unique_id": (i32, [vp]),
        "cb200_nccl_comm_create": (vp, [i32, i32, vp]),
        "cb200_nccl_comm_destroy": (None, [vp]),
        "cb200_trainer_allgather_samples": (i32, [vp, vp, vp, vp, vp]),
        "cb200_trainer_set_weights": (i32, [vp, i32, vp, C.c_size_t, i32]),
        "cb200_trainer_evaluate": (i32, [vp, i32, i32, vp, vp, vp]),
        "cb200_trainer_run_selfplay": (i32, [vp, i32, i32]),
        "cb200_trainer_dump_tree": (i32, [vp, i32, i32, vp, vp, i32]),
        "cb200_trainer_reset": (i32, [vp, i32]),
        "cb200_trainer_phase_profile": (i32, [vp, i32, vp]),
        "cb200_trainer_set_profiling": (i32, [vp, i32]),
        "cb200_trainer_kernel_times": (i32, [vp, vp, vp]),
        "cb200_trainer_phase_split": (i32, [vp, vp]),
        "cb200_trainer_phase_times": (i32, [vp, vp]),
        "cb200_tourney_create": (vp, [i32, C.c_char_p]),
        "cb200_tourney_destroy": (None, [vp]),
        "cb200_tourney_add_player": (i32, [vp, i32, i32, i32, i32, f32, f32, i32]),
        "cb200_tourney_add_match": (i32, [vp, i32, i32, i32]),
        "cb200_tourney_all_done": (i32, [vp]),
        "cb200_tourney_num_requests": (i32, [vp, i32]),
        "cb200_tourney_write_requests": (i32, [vp, vp, i32]),
        "cb200_tourney_do_iteration": (i32, [vp, vp, vp, i32, i32]),
        "cb200_tourney_write_scores": (i32, [vp, C.c_char_p]),
        "cb200_tourney_counters": (i32, [vp, vp]),
        "cb200_tourney_set_weights": (i32, [vp, i32, vp, C.c_size_t, i32]),
        "cb200_tourney_run": (i32, [vp, i32]),
        "cb200_analysis_create": (vp, [i32, i32, i32, f32, f32]),
        "cb200_analysis_destroy": (None, [vp]),
        "cb200_analysis_set_weights": (i32, [vp, vp, C.c_size_t, i32]),
        "cb200_analysis_run": (i32, [vp, i32, vp, i32, vp, vp, vp, vp, vp]),
        "cb200_analysis_counters": (i32, [vp, vp]),
        "cb200_analysis_begin": (i32, [vp, i32, vp, i32]),
        "cb200_analysis_num_requests": (i32, [vp]),
        "cb200_analysis_write_requests": (i32, [vp, vp]),
        "cb200_analysis_do_iteration": (i32, [vp, vp, vp, i32]),
        "cb200_analysis_results": (i32, [vp, vp, vp, vp, vp, vp]),
        "cb200_analysis_write_requests_device": (i32, [vp, vp]),
        "cb200_analysis_do_iteration_device": (i32, [vp, vp, vp, i32]),
        "cb200_analysis_run_device": (i32, [vp, i32, vp, i32, vp, vp, vp, vp, vp, vp]),
        "cb200_check_states": (i64, [i64, vp, vp]),
    }
    for name, (res, args) in sig.items():
        f = getattr(L, name)
        f.restype, f.argtypes = res, args
    _lib = L
    return L


def nccl_comm_from_torch(dist, rank, world, device):
    """An NCCL communicator owned by this library for the ranks of a torch.distributed job: rank 0
    draws the ncclUniqueId, torch.distributed (any backend) carries its 128 bytes to the others."""
    import torch
    idbuf = np.zeros(128, np.uint8)
    if rank == 0:
        _check(lib().cb200_nccl_unique_id(_ptr(idbuf)))
    t = torch.from_numpy(idbuf).to(device)
    dist.broadcast(t, src=0)
    idbuf = np.ascontiguousarray(t.cpu().numpy())
    comm = lib().cb200_nccl_comm_create(rank, world, _ptr(idbuf))
    if not comm:
        raise Corintho200Error("cb200_nccl_comm_create: " + lib().cb200_last_error().decode())
    return comm


def _check(rc):
    if rc < 0:
        raise Corintho200Error(f"corintho_b200 error {rc}: {lib().cb200_last_error().decode()}")
    return rc


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _in_f32(a, min_size, what):
    """Input buffer of the reference API (typed float memoryview in main.pyx:30-38): converted to
    a C-contiguous float32 array; fewer than `min_size` elements is an error, never a short read."""
    if a is None:
        if min_size > 0:
            raise Corintho200Error(f"{what}: buffer is None but {min_size} floats are needed")
        return None
    b = np.ascontiguousarray(a, np.float32)
    if b.size < min_size:
        raise Corintho200Error(f"{what}: {b.size} floats given, {min_size} needed")
    return b


def _out_f32(a, min_size, what):
    """Output buffer written through a raw pointer: must already be float32, C-contiguous,
    writable and large enough (the reference's Cython signature rejects anything else)."""
    if not isinstance(a, np.ndarray) or a.dtype != np.float32 or not a.flags.c_contiguous \
            or not a.flags.writeable:
        raise Corintho200Error(f"{what}: need a writable C-contiguous float32 numpy array")
    if a.size < min_size:
        raise Corintho200Error(f"{what}: {a.size} floats given, {min_size} needed")
    return a


# ---- packed state helpers -----------------------------------------------------------------
def planes_from_reference_order(states):
    """[n,2] u64 with board bit row*16+col*4+t (reference Game::board_ order) -> cstate planes."""
    st = np.ascontiguousarray(states, np.uint64).reshape(-1, 2)
    w0 = st[:, 0]
    out = np.zeros_like(w0)
    for s in range(16):
        for t in range(4):
            out |= ((w0 >> np.uint64(4 * s + t)) & np.uint64(1)) << np.uint64(16 * t + s)
    return np.ascontiguousarray(np.stack([out, st[:, 1]], 1))


def reference_order_from_planes(states):
    st = np.ascontiguousarray(states, np.uint64).reshape(-1, 2)
    w0 = st[:, 0]
    out = np.zeros_like(w0)
    for s in range(16):
        for t in range(4):
            out |= ((w0 >> np.uint64(16 * t + s)) & np.uint64(1)) << np.uint64(4 * s + t)
    return np.ascontiguousarray(np.stack([out, st[:, 1]], 1))


def game_step(states, seed=0, want_encoding=False):
    """Game-logic step on host arrays of cstates -> (mask_flags[n,4] u32, next[n,2] u64, enc)."""
    st = np.ascontiguousarray(states, np.uint64).reshape(-1, 2)
    n = st.shape[0]
    mf = np.zeros((n, 4), np.uint32)
    nx = np.zeros((n, 2), np.uint64)
    enc = np.zeros((n, STATE_SIZE), np.float32) if want_encoding else None
    _check(lib().cb200_game_step(n, _ptr(st), seed, _ptr(mf), _ptr(nx), _ptr(enc)))
    return mf, nx, enc


# ---- network weights ----------------------------------------------------------------------
def random_weights(seed=0):
    """Random-init network of the reference architecture (wrapper.py:256-271): Glorot-uniform
    Dense kernels, zero biases, BatchNorm at its initial state (gamma 1, beta 0, mean 0, var 1,
    eps 1e-3). Returns the *unfolded* parameter dict; see fold_batchnorm()."""
    rng = np.random.default_rng(seed)
    dims = [STATE_SIZE] + [100] * 12
    layers = []
    for i in range(12):
        fan_in, fan_out = dims[i], dims[i + 1]
        lim = np.sqrt(6.0 / (fan_in + fan_out))
        layers.append({
            "W": rng.uniform(-lim, lim, size=(fan_in, fan_out)).astype(np.float32),
            "b": np.zeros(fan_out, np.float32),
            "gamma": np.ones(fan_out, np.float32), "beta": np.zeros(fan_out, np.float32),
            "mean": np.zeros(fan_out, np.float32), "var": np.ones(fan_out, np.float32),
        })
    lim_v, lim_p = np.sqrt(6.0 / (100 + 1)), np.sqrt(6.0 / (100 + NUM_MOVES))
    head = {
        "Wv": rng.uniform(-lim_v, lim_v, size=(100, 1)).astype(np.float32),
        "bv": np.zeros(1, np.float32),
        "Wp": rng.uniform(-lim_p, lim_p, size=(100, NUM_MOVES)).astype(np.float32),
        "bp": np.zeros(NUM_MOVES, np.float32),
    }
    return {"layers": layers, "head": head}


def fold_batchnorm(params, eps=1e-3):
    """Fold each inference-time BatchNormalization (which FOLLOWS the ReLU, wrapper.py:259-266)
    into the next Dense and flatten to the C-ABI weight vector (127997 floats, fp32):
    y = relu(xW+b); z = s*y + t with s = gamma/sqrt(var+eps), t = beta - mean*s;
    next Dense: zW' + b' = y (diag(s) W') + (t W' + b')."""
    out = []
    s = np.ones(STATE_SIZE, np.float64)
    t = np.zeros(STATE_SIZE, np.float64)
    for L in params["layers"]:
        W = L["W"].astype(np.float64)
        b = L["b"].astype(np.float64)
        out.append((s[:, None] * W).astype(np.float32).ravel())
        out.append((t @ W + b).astype(np.float32))
        s = L["gamma"].astype(np.float64) / np.sqrt(L["var"].astype(np.float64) + eps)
        t = L["beta"].astype(np.float64) - L["mean"].astype(np.float64) * s
    H = params["head"]
    Wh = np.concatenate([H["Wv"], H["Wp"]], 1).astype(np.float64)
    bh = np.concatenate([H["bv"], H["bp"]]).astype(np.float64)
    out.append((s[:, None] * Wh).astype(np.float32).ravel())
    out.append((t @ Wh + bh).astype(np.float32))
    flat = np.concatenate(out).astype(np.float32)
    assert flat.size == WEIGHT_FLOATS, flat.size
    return flat


class Trainer:
    """Drop-in for the reference ``Trainer`` (trainer.h:17-53) on one GPU.

    Reference-named methods (camelCase, as in the Cython binding) and snake_case aliases are
    both provided. numpy float32 buffers are passed as raw pointers exactly like
    main.pyx:132-165 does.
    """

    def __init__(self, num_games, log_folder="", seed=0, max_searches=1600, searches_per_eval=16,
                 c_puct=1.0, epsilon=0.25, num_logged=0, num_threads=1, testing=False,
                 total_games=None, first_game=0):
        L = lib()
        self.num_games = int(num_games)
        self.spe = int(searches_per_eval)
        self.max_searches = int(max_searches)
        self.testing = bool(testing)
        if total_games is None:
            h = L.cb200_trainer_create(num_games, log_folder.encode(), seed, max_searches,
                                       searches_per_eval, c_puct, epsilon, num_logged,
                                       num_threads, int(testing))
        else:
            h = L.cb200_trainer_create_shard(total_games, first_game, num_games,
                                             log_folder.encode(), seed, max_searches,
                                             searches_per_eval, c_puct, epsilon, num_logged,
                                             int(testing))
        if not h:
            raise Corintho200Error("Trainer: " + L.cb200_last_error().decode())
        self._h = C.c_void_p(h)

    def close(self):
        if getattr(self, "_h", None):
            lib().cb200_trainer_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- reference API ------------------------------------------------------------------
    def doIteration(self, evaluations=None, probabilities=None, to_play=-1):
        # the answers of the requests that are pending for this side (none on the first call)
        n = self.num_requests(to_play)
        ev = _in_f32(evaluations, n, "doIteration: evaluations")
        pr = _in_f32(probabilities, n * NUM_MOVES, "doIteration: probabilities")
        return bool(_check(lib().cb200_trainer_do_iteration(self._h, _ptr(ev), _ptr(pr), to_play)))

    def num_requests(self, to_play=-1):
        return _check(lib().cb200_trainer_num_requests(self._h, to_play))

    def writeRequests(self, game_states, to_play=-1):
        n = self.num_requests(to_play)
        _out_f32(game_states, n * STATE_SIZE, "writeRequests: game_states")
        _check(lib().cb200_trainer_write_requests(self._h, _ptr(game_states), to_play))

    def num_samples(self):
        return _check(lib().cb200_trainer_num_samples(self._h))

    def writeSamples(self, game_states, eval_samples, prob_samples):
        rows = self.num_samples() * NUM_SYMMETRIES
        _out_f32(game_states, rows * STATE_SIZE, "writeSamples: game_states")
        _out_f32(eval_samples, rows, "writeSamples: eval_samples")
        _out_f32(prob_samples, rows * NUM_MOVES, "writeSamples: prob_samples")
        _check(lib().cb200_trainer_write_samples(self._h, _ptr(game_states), _ptr(eval_samples),
                                                 _ptr(prob_samples)))

    def score(self):
        return np.float32(lib().cb200_trainer_score(self._h))

    def avg_mate_length(self):
        return np.float32(lib().cb200_trainer_avg_mate_length(self._h))

    def writeScores(self, file):
        _check(lib().cb200_trainer_write_scores(self._h, str(file).encode()))

    # ---- snake_case conveniences returning fresh arrays (what the test drivers call) ------
    def do_iteration(self, evals=None, probs=None, to_play=-1):
        return self.doIteration(evals, probs, to_play)

    def write_requests(self, to_play=-1):
        n = self.num_requests(to_play)
        out = np.zeros((max(n, 1), STATE_SIZE), np.float32)
        if n:
            self.writeRequests(out, to_play)
        return out[:n]

    def write_samples(self):
        n = self.num_samples()
        gs = np.zeros((max(n, 1) * 8, STATE_SIZE), np.float32)
        ev = np.zeros(max(n, 1) * 8, np.float32)
        pr = np.zeros((max(n, 1) * 8, NUM_MOVES), np.float32)
        if n:
            self.writeSamples(gs, ev, pr)
        return gs[:n * 8], ev[:n * 8], pr[:n * 8]

    # ---- engine-only ------------------------------------------------------------------------
    def counters(self):
        out = np.zeros(4, np.int64)
        _check(lib().cb200_trainer_counters(self._h, _ptr(out)))
        return {"simulations": int(out[0]), "moves": int(out[1]), "leaf_evals": int(out[2]),
                "iterations": int(out[3])}

    def set_weights(self, flat_weights, model=0, precision="fp32"):
        w = np.ascontiguousarray(flat_weights, np.float32)
        prec = {"fp32": 0, "bf16": 1, "fp16": 2, "bf16x3": 3}[precision]
        _check(lib().cb200_trainer_set_weights(self._h, model, _ptr(w), w.size, prec))

    def evaluate(self, game_states, model=0):
        gs = np.ascontiguousarray(game_states, np.float32).reshape(-1, STATE_SIZE)
        n = gs.shape[0]
        ev = np.zeros(n, np.float32)
        pr = np.zeros((n, NUM_MOVES), np.float32)
        _check(lib().cb200_trainer_evaluate(self._h, model, n, _ptr(gs), _ptr(ev), _ptr(pr)))
        return ev, pr

    def run_selfplay(self, max_iterations=0, stagger=False):
        return bool(_check(lib().cb200_trainer_run_selfplay(self._h, max_iterations, int(stagger))))

    def phase_profile(self, enable=True):
        out = np.zeros(16, np.uint64)
        _check(lib().cb200_trainer_phase_profile(self._h, int(enable), _ptr(out)))
        return out

    def reset(self, seed):
        _check(lib().cb200_trainer_reset(self._h, int(seed)))

    def set_profiling(self, enable=True):
        _check(lib().cb200_trainer_set_profiling(self._h, int(enable)))

    def kernel_times(self):
        ms = np.zeros(8, np.float64)
        ln = np.zeros(8, np.int64)
        _check(lib().cb200_trainer_kernel_times(self._h, _ptr(ms), _ptr(ln)))
        names = ["scan", "pack", "network", "game_step", "fused_tail", "fused_tail_wide"]
        return {n: {"ms": float(ms[i]), "launches": int(ln[i])} for i, n in enumerate(names)}

    def phase_split(self):
        """Simulations / leaf evaluations done by lock-step launches vs in total (profiling on)."""
        out = np.zeros(4, np.int64)
        _check(lib().cb200_trainer_phase_split(self._h, _ptr(out)))
        return {"lockstep_simulations": int(out[0]), "simulations": int(out[1]),
                "lockstep_leaf_evals": int(out[2]), "leaf_evals": int(out[3])}

    def phase_times(self):
        """Host-clock ms spent in the lock-step phase / in the persistent kernels since the last
        set_profiling() call."""
        out = np.zeros(2, np.float64)
        _check(lib().cb200_trainer_phase_times(self._h, _ptr(out)))
        return {"lockstep_ms": float(out[0]), "tail_ms": float(out[1])}

    def raw_samples(self):
        n = self.num_samples()
        st = np.zeros((max(n, 1), 2), np.uint64)
        pr = np.zeros((max(n, 1), NUM_MOVES), np.float32)
        lb = np.zeros(max(n, 1), np.float32)
        go = np.zeros(max(n, 1), np.int32)
        _check(lib().cb200_trainer_write_raw_samples(self._h, _ptr(st), _ptr(pr), _ptr(lb), _ptr(go)))
        return st[:n], pr[:n], lb[:n], go[:n]

    def raw_samples_device(self):
        """(device pointer, n_rows) of the [n_rows][102] float row block (see the C header)."""
        ptr = C.c_void_p()
        n = C.c_int()
        _check(lib().cb200_trainer_raw_samples_device(self._h, C.byref(ptr), C.byref(n)))
        return ptr.value or 0, n.value

    def stream_samples(self, max_samples=-1):
        """Enable (or with 0 disable) streaming of finished games' samples to pinned host memory
        during run_selfplay (see cb200_trainer_stream_samples in the C header)."""
        _check(lib().cb200_trainer_stream_samples(self._h, int(max_samples)))

    def streamed_samples(self):
        """(game_states[n*8,70], eval_samples[n*8], prob_samples[n*8,96], game_of[n]) as numpy views
        of the trainer's pinned host buffers (valid until the next reset / run); rows in game
        completion order, 8 consecutive rows per sample."""
        gs, ev, pr, go = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_void_p()
        n = C.c_int()
        _check(lib().cb200_trainer_streamed_samples(self._h, C.byref(gs), C.byref(ev), C.byref(pr),
                                                    C.byref(go), C.byref(n)))
        n = n.value
        if n == 0:
            return (np.zeros((0, STATE_SIZE), np.float32), np.zeros(0, np.float32),
                    np.zeros((0, NUM_MOVES), np.float32), np.zeros(0, np.int32))

        def view(ptr, ctype, shape):
            count = int(np.prod(shape))
            return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(ctype)), shape=(count,)).reshape(shape)
        return (view(gs, C.c_float, (n * 8, STATE_SIZE)), view(ev, C.c_float, (n * 8,)),
                view(pr, C.c_float, (n * 8, NUM_MOVES)), view(go, C.c_int32, (n,)))

    def allgather_samples(self, nccl_comm, world):
        """NCCL all-gather of every rank's un-augmented samples (collective). Returns (device
        pointer, total rows, rows per rank); rows are [n][102] floats in global game order."""
        ptr, n = C.c_void_p(), C.c_int()
        counts = np.zeros(world, np.int32)
        _check(lib().cb200_trainer_allgather_samples(self._h, C.c_void_p(nccl_comm), C.byref(ptr),
                                                     C.byref(n), _ptr(counts)))
        return ptr.value or 0, n.value, counts

    def game_results(self):
        out = np.zeros(self.num_games, np.int32)
        _check(lib().cb200_trainer_game_results(self._h, _ptr(out)))
        return out

    def dump_tree(self, game, player, cap=1 << 22):
        out = np.zeros(8, np.int64)
        words = np.zeros(cap, np.uint32)
        used = _check(lib().cb200_trainer_dump_tree(self._h, game, player, _ptr(out), _ptr(words), cap))
        return out, words[:min(used, cap)]


class Tourney:
    """Mirror of the reference Tourney (corintho_ai/cpp/include/tourney.h:12-46) as the Cython
    binding exposes it (corintho_ai/rating/tourney.pyx:13-25): addPlayer, addMatch, all_done,
    num_requests, writeRequests, doIteration, writeScores -- same argument meaning. Matches run on
    the GPU (csrc/match.cuh); the network stays with the caller, one model id at a time."""

    def __init__(self, num_threads=1, log_folder=""):
        self._h = lib().cb200_tourney_create(int(num_threads), str(log_folder).encode())
        if not self._h:
            raise Corintho200Error(lib().cb200_last_error().decode())
        self.model_ids = []   # in first-seen order, like tourney.pyx builds its list
        self.max_rows = 0     # upper bound of one call's request rows
        self._spe = {}

    def close(self):
        if getattr(self, "_h", None):
            lib().cb200_tourney_destroy(self._h)
            self._h = None

    def __del__(self):
        self.close()

    def addPlayer(self, player_id, model_id, max_searches=1600, searches_per_eval=16, c_puct=1.0,
                  epsilon=0.25, random=False):
        _check(lib().cb200_tourney_add_player(self._h, player_id, model_id, max_searches,
                                              searches_per_eval, c_puct, epsilon, int(random)))
        self._spe[player_id] = searches_per_eval
        if model_id not in self.model_ids:
            self.model_ids.append(model_id)

    def addMatch(self, player1, player2, logging=False):
        _check(lib().cb200_tourney_add_match(self._h, player1, player2, int(logging)))
        self.max_rows += self._spe[player1] + self._spe[player2]

    def all_done(self):
        return bool(_check(lib().cb200_tourney_all_done(self._h)))

    def num_requests(self, model_id):
        return _check(lib().cb200_tourney_num_requests(self._h, int(model_id)))

    def writeRequests(self, game_states, model_id):
        _out_f32(game_states, self.num_requests(model_id) * STATE_SIZE, "writeRequests: game_states")
        _check(lib().cb200_tourney_write_requests(self._h, _ptr(game_states), int(model_id)))

    def doIteration(self, evals, probs, model_id):
        evals = np.ascontiguousarray(evals, np.float32)
        probs = np.ascontiguousarray(probs, np.float32)
        rows = min(evals.shape[0], probs.shape[0])
        _check(lib().cb200_tourney_do_iteration(self._h, _ptr(evals), _ptr(probs), rows, int(model_id)))

    def writeScores(self, filename):
        _check(lib().cb200_tourney_write_scores(self._h, str(filename).encode()))

    def counters(self):
        out = np.zeros(4, np.int64)
        _check(lib().cb200_tourney_counters(self._h, _ptr(out)))
        return {"simulations": int(out[0]), "moves": int(out[1]), "leaf_evals": int(out[2]),
                "iterations": int(out[3])}

    # ---- engine-only: fused tourney (device-resident networks per model id) -------------------
    def set_weights(self, model_id, flat_weights, precision="fp32"):
        w = np.ascontiguousarray(flat_weights, np.float32)
        prec = {"fp32": 0, "bf16": 1, "fp16": 2, "bf16x3": 3}[precision]
        _check(lib().cb200_tourney_set_weights(self._h, int(model_id), _ptr(w), w.size, prec))

    def run(self, max_rounds=0):
        """Play rounds of rating/tourney.pyx:112-173 on the device; True when every match is over."""
        return bool(_check(lib().cb200_tourney_run(self._h, int(max_rounds))))

    # snake_case conveniences shared with the test drivers
    add_player = addPlayer
    add_match = addMatch
    do_iteration = doIteration

    def write_requests(self, model_id):
        n = self.num_requests(model_id)
        out = np.zeros((max(n, 1), STATE_SIZE), np.float32)
        self.writeRequests(out, model_id)
        return out[:n]

    def scores(self):
        import tempfile
        with tempfile.NamedTemporaryFile("r", suffix=".txt") as f:
            self.writeScores(f.name)
            rows = [ln.split() for ln in open(f.name).read().splitlines() if ln.strip()]
        return [(int(a), int(b), float(c)) for a, b, c in rows]


def _out_buf(a, dtype, min_size, what):
    """Output buffer of a given dtype with the checks of _out_f32."""
    if not isinstance(a, np.ndarray) or a.dtype != dtype or not a.flags.c_contiguous \
            or not a.flags.writeable:
        raise Corintho200Error(f"{what}: need a writable C-contiguous {np.dtype(dtype).name} numpy array")
    if a.size < min_size:
        raise Corintho200Error(f"{what}: {a.size} elements given, {min_size} needed")
    return a


def _dev_buf(t, min_size, what, dtypes=("torch.float32",)):
    """Device buffer of the analysis' device forms: a contiguous CUDA tensor of one of `dtypes` with
    at least `min_size` elements. Duck-typed on torch.Tensor's dtype / device / is_contiguous /
    numel / data_ptr, so this package does not import torch. Returns the device address."""
    try:
        dtype, device = str(t.dtype), t.device
        contiguous, numel = bool(t.is_contiguous()), int(t.numel())
    except (AttributeError, TypeError):
        raise Corintho200Error(f"{what}: need a CUDA tensor, got {type(t).__name__}") from None
    if dtype not in dtypes or getattr(device, "type", None) != "cuda" or not contiguous:
        want = " or ".join(d.replace("torch.", "") for d in dtypes)
        raise Corintho200Error(f"{what}: need a contiguous {want} CUDA tensor, got {dtype} on {device}"
                               f"{'' if contiguous else ' (not contiguous)'}")
    if numel < min_size:
        raise Corintho200Error(f"{what}: {numel} elements given, {min_size} needed")
    return int(t.data_ptr())


def _dev_f32(t, min_size, what):
    return _dev_buf(t, min_size, what)


def check_states(states):
    """Structural check of cstates [n,2] u64 (see cb200_check_states): bool array, True = valid.
    Needs no GPU."""
    st = np.ascontiguousarray(states, np.uint64).reshape(-1, 2)
    ok = np.zeros(st.shape[0], np.uint8)
    _check(lib().cb200_check_states(st.shape[0], _ptr(st), _ptr(ok)))
    return ok.astype(bool)


class Analysis:
    """The engine's move and search statistics for given positions: the batched form of the
    reference's DockerMC (corintho_ai/cpp/src/dockermc.cpp) that docker/choose_move.pyx serves.
    Every position is searched by one testing-mode TrainMC with the device-resident network, which
    then chooses its move; see cb200_analysis_run in include/corintho_b200.h for the exact meaning
    of every output."""

    def __init__(self, max_positions, max_searches=1600, searches_per_eval=16, c_puct=1.0,
                 epsilon=0.25):
        L = lib()
        h = L.cb200_analysis_create(int(max_positions), int(max_searches), int(searches_per_eval),
                                    float(c_puct), float(epsilon))
        if not h:
            raise Corintho200Error("Analysis: " + L.cb200_last_error().decode())
        self._h = C.c_void_p(h)
        self.max_positions = int(max_positions)

    def close(self):
        if getattr(self, "_h", None):
            lib().cb200_analysis_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_weights(self, flat_weights, precision="fp32"):
        w = _in_f32(flat_weights, WEIGHT_FLOATS, "set_weights: weights")
        prec = {"fp32": 0, "bf16": 1, "fp16": 2, "bf16x3": 3}[precision]
        _check(lib().cb200_analysis_set_weights(self._h, _ptr(w), w.size, prec))

    setWeights = set_weights

    def run(self, states, seed=0, evals=True):
        """states: [n,2] u64 cstates. Returns {"moves" [n] i32, "results" [n] i32, "values" [n]
        f32, "visits" [n,96] i32, "evals" [n,96] f32 (only with evals=True)}."""
        st = _analysis_states(states, "run")
        out = _analysis_outputs(st.shape[0], evals)
        self.run_into(st, seed, **out)
        return out

    def run_into(self, states, seed, moves, results, values, visits, evals=None):
        """run() into caller-owned buffers (checked like the Trainer's output buffers)."""
        st = np.ascontiguousarray(states, np.uint64).reshape(-1, 2)
        n = st.shape[0]
        _out_buf(moves, np.int32, n, "run: moves")
        _out_buf(results, np.int32, n, "run: results")
        _out_f32(values, n, "run: values")
        _out_buf(visits, np.int32, n * NUM_MOVES, "run: visits")
        if evals is not None:
            _out_f32(evals, n * NUM_MOVES, "run: evals")
        _check(lib().cb200_analysis_run(self._h, n, _ptr(st), int(seed), _ptr(moves), _ptr(results),
                                        _ptr(values), _ptr(visits), _ptr(evals)))

    def counters(self):
        """{simulations, leaf_evals} of the last run or session (running totals while one is open)."""
        out = np.zeros(2, np.int64)
        _check(lib().cb200_analysis_counters(self._h, _ptr(out)))
        return {"simulations": int(out[0]), "leaf_evals": int(out[1])}

    # ---- external-evaluator protocol: the caller's network answers the requests -----------------
    # begin; until do_iteration(...) returns True: write_requests, evaluate, do_iteration; results.
    # See cb200_analysis_begin in include/corintho_b200.h for the protocol's rules.
    def begin(self, states, seed=0):
        """Open a session on [n,2] u64 cstates (no weights needed); restarts an open one."""
        st = _analysis_states(states, "begin")
        _check(lib().cb200_analysis_begin(self._h, st.shape[0], _ptr(st), int(seed)))
        self._n = st.shape[0]

    def num_requests(self):
        return _check(lib().cb200_analysis_num_requests(self._h))

    def write_requests(self, out=None):
        """The pending request rows: a fresh [num_requests, 70] float32 array, or written into `out`
        (a writable C-contiguous float32 array of at least num_requests * 70 floats), returned."""
        n = self.num_requests()
        if out is None:
            buf = np.zeros((max(n, 1), STATE_SIZE), np.float32)
            _check(lib().cb200_analysis_write_requests(self._h, _ptr(buf)))
            return buf[:n]
        _out_f32(out, n * STATE_SIZE, "write_requests: out")
        _check(lib().cb200_analysis_write_requests(self._h, _ptr(out)))
        return out

    def do_iteration(self, eval=None, probs=None):
        """One round with the answers to the last write_requests (eval [n], probs [n,96], row-major;
        None for the first call). True when every position is done."""
        n = self.num_requests()
        ev = _in_f32(eval, n, "do_iteration: eval")
        pr = _in_f32(probs, n * NUM_MOVES, "do_iteration: probs")
        rows = 0 if ev is None or pr is None else min(ev.size, pr.size // NUM_MOVES)
        return bool(_check(lib().cb200_analysis_do_iteration(self._h, _ptr(ev), _ptr(pr), rows)))

    def results(self, evals=True):
        """The outputs of run() for the finished session."""
        out = _analysis_outputs(getattr(self, "_n", 0), evals)
        _check(lib().cb200_analysis_results(self._h, _ptr(out["moves"]), _ptr(out["results"]),
                                            _ptr(out["values"]), _ptr(out["visits"]), _ptr(out.get("evals"))))
        return out

    def write_requests_device(self, rows):
        """Pack the pending request rows into a float32 CUDA tensor of at least num_requests * 70
        elements, on the library's current stream (cb200_set_stream), without waiting."""
        n = self.num_requests()
        _check(lib().cb200_analysis_write_requests_device(self._h, _dev_f32(rows, n * STATE_SIZE,
                                                                            "write_requests_device: rows")))
        return rows

    def do_iteration_device(self, eval, probs):
        """do_iteration with float32 CUDA tensors (eval [>= n], probs [>= n, 96] row-major), read in
        place on the library's current stream; the writes to them must be ordered before it."""
        n = self.num_requests()
        ev = _dev_f32(eval, n, "do_iteration_device: eval")
        pr = _dev_f32(probs, n * NUM_MOVES, "do_iteration_device: probs")
        rows = min(int(eval.numel()), int(probs.numel()) // NUM_MOVES)
        return bool(_check(lib().cb200_analysis_do_iteration_device(self._h, ev, pr, rows)))

    def run_device(self, states, seed=0, out=None, evals=True):
        """run() on positions already on the GPU, in one persistent kernel on the library's current
        stream (cb200_set_stream), returning without waiting: the outputs are complete in the order
        of that stream, and `states` must not change before then. states: a contiguous int64 or
        uint64 CUDA tensor [n, 2] of cstate words; needs bf16, fp16 or bf16x3 weights. out=None
        allocates the outputs with torch on the states' device; else `out` is a dict of the caller's
        CUDA tensors "moves" [n] int32, "results" [n] int32, "values" [n] float32, "visits" [n, 96]
        int32 and optionally "evals" [n, 96] float32 and "status" [2] int32, written in place.
        Returns the dict run() returns plus "status" = {positions with an error result, most
        negative error result or 0}: a rejected state gets result -1, an overflowed search -3, both
        with move -1. See cb200_analysis_run_device in include/corintho_b200.h."""
        shape = tuple(getattr(states, "shape", ()))
        if len(shape) != 2 or shape[1] != 2 or shape[0] < 1:
            raise Corintho200Error("run_device: states must be an [n, 2] CUDA tensor of cstate words")
        n = int(shape[0])
        st = _dev_buf(states, 2 * n, "run_device: states", ("torch.int64", "torch.uint64"))
        if out is None or "status" not in out:
            import torch
            dev = states.device
            res = {"status": torch.zeros(2, dtype=torch.int32, device=dev)}
            if out is None:
                res.update(moves=torch.empty(n, dtype=torch.int32, device=dev),
                           results=torch.empty(n, dtype=torch.int32, device=dev),
                           values=torch.empty(n, dtype=torch.float32, device=dev),
                           visits=torch.empty((n, NUM_MOVES), dtype=torch.int32, device=dev))
                if evals:
                    res["evals"] = torch.empty((n, NUM_MOVES), dtype=torch.float32, device=dev)
            else:
                res.update(out)
        else:
            res = dict(out)
        if not evals:
            res.pop("evals", None)
        i32 = ("torch.int32",)
        ptrs = [_dev_buf(res["moves"], n, "run_device: moves", i32),
                _dev_buf(res["results"], n, "run_device: results", i32),
                _dev_buf(res["values"], n, "run_device: values"),
                _dev_buf(res["visits"], n * NUM_MOVES, "run_device: visits", i32),
                _dev_buf(res["evals"], n * NUM_MOVES, "run_device: evals") if "evals" in res else None,
                _dev_buf(res["status"], 2, "run_device: status", i32)]
        _check(lib().cb200_analysis_run_device(self._h, n, st, int(seed), *ptrs))
        return res

    def search(self, states, seed, evaluator, evals=True):
        """run() with the caller's network: evaluator(rows [k,70] float32) -> (eval [k], probs [k,96])
        answers every round's requests. Returns the dict run() returns."""
        self.begin(states, seed)
        answers = (None, None)
        while not self.do_iteration(*answers):
            answers = evaluator(self.write_requests())
        return self.results(evals)


def _analysis_states(states, what):
    st = np.ascontiguousarray(states, np.uint64)
    if st.ndim != 2 or st.shape[1] != 2:
        raise Corintho200Error(f"{what}: states must be an [n, 2] array of cstate words")
    return st


def _analysis_outputs(n, evals):
    out = {"moves": np.zeros(n, np.int32), "results": np.zeros(n, np.int32),
           "values": np.zeros(n, np.float32), "visits": np.zeros((n, NUM_MOVES), np.int32)}
    if evals:
        out["evals"] = np.zeros((n, NUM_MOVES), np.float32)
    return out
