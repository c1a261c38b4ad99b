#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 Corintho self-play engine.

Metric (BASELINE.json): MCTS simulations/sec (plus self-play moves/sec) per box.
Workload at every N: BASELINE.json configs[2] per GPU -- 4096 concurrent games x 800
sims/move, searches_per_eval 16, c_puct 1.0, epsilon 0.25, random-init network of the
reference architecture -- run to completion of all games ("step" = one such self-play pass).
For N > 1 the games of one seed stream are sharded contiguously across ranks (weak scaling,
no collective on the hot path) and the finished samples are all-gathered over NCCL
(configs[3] uses the same code with --games-per-gpu 32768).

  python bench.py [--gpus N] [--steps K] [--warmup W]          engine arm
  python bench.py ... --dump-outputs DIR                       + the last timed step's samples as .npy
  python bench.py --impl reference ...                         reference CPU arm
Under torchrun (N > 1) every rank runs; rank 0 prints the single JSON line.
"""
import argparse
from ctypes import c_void_p as C_void_p
import gc
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ALGO_BYTES_PER_SIM = 1670.0      # SURVEY.md 8(d): algorithmic bytes per simulation @800 sims
FLOP_PER_EVAL = 253400.0         # SURVEY.md 8(d): unpadded dense FLOPs per leaf evaluation
# dram__bytes_read.sum + dram__bytes_write.sum of ONE k_iterate launch with all 4096 games live
# (65 536 simulations = 109.4 MB algorithmic), from the `ncu --set full` capture summarised in
# profiles/r02_ncu_k_iterate_lanes16_vs_32.txt; profiles/r01_ncu_k_iterate_k_mlp_tc_v3.txt gives
# 1.36 MB for k_mlp_tc
NCU_DRAM_BYTES_PER_DENSE_LAUNCH = {"game_step": 149.888000e6 + 59.357440e6, "network": 1.356032e6 + 0.000256e6}
NCU_SOURCE = "profiles/r02_ncu_k_iterate_6ctas.txt, k_iterate<1, 32, 6>"
DUMP_BUDGET_BYTES = 64 * 10**6


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0,
            "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "200", "-i", str(self.gpu)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(",") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1])), mx.append(float(r[2]))
                for nm, v in zip(names, r[4:8]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


def workload_desc(args, n_gpus):
    return {
        "workload": ("BASELINE.json configs[2] per GPU: batched self-play, %d concurrent games x %d sims/move, "
                     "searches_per_eval %d, c_puct %.1f, epsilon %.2f, all games to completion"
                     % (args.games_per_gpu, args.sims, args.spe, args.c_puct, args.epsilon)),
        "games_per_gpu": args.games_per_gpu, "total_games": args.games_per_gpu * n_gpus,
        "max_searches": args.sims, "searches_per_eval": args.spe,
        "network": "70 -> 12x[Dense100,ReLU,BN folded] -> {tanh 1, softmax 96}, random init (Glorot-uniform)",
        "staggered_start": False,
        "parallelism": "games sharded contiguously across %d GPU(s); no collective on the hot path; "
                       "samples all-gathered (NCCL) after the run" % n_gpus,
        "l2_policy": "inputs larger than L2: per-GPU node arenas are several GB (>> 126 MB L2); "
                     "every step starts from re-initialised game state",
    }


# ----------------------------------------------------------------------------------------------
def cpu_mlp(flat):
    """fp32 CPU evaluator with the engine's weights (stands in for the reference's Keras predict,
    main.pyx:70-83; Keras/TensorFlow are not installable here)."""
    import torch
    dims = [70] + [100] * 12 + [97]
    Ws, bs, off = [], [], 0
    for l in range(13):
        K, N = dims[l], dims[l + 1]
        Ws.append(torch.from_numpy(flat[off:off + K * N].reshape(K, N).copy()))
        off += K * N
        bs.append(torch.from_numpy(flat[off:off + N].copy()))
        off += N

    def f(rows):
        with torch.no_grad():
            h = torch.from_numpy(np.ascontiguousarray(rows, np.float32))
            for l in range(13):
                h = torch.addmm(bs[l], h, Ws[l])
                if l < 12:
                    h = torch.relu_(h)
            ev = torch.tanh(h[:, 0])
            pr = torch.softmax(h[:, 1:], 1)
        return ev.numpy(), pr.numpy()
    return f


_EXACT_SIMS = {}


def time_cpu_reference(args, flat, games, budget_s=None):
    """Time the reference's own CPU implementation of the path (oracle/_ref when it was built
    from /root/reference, else the oracle port) on `games` games of the engine's workload.
    Returns dict(value sims/s, moves/s, cores, kind, sample, seconds, play_s, predict_s)."""
    # the tree (OpenMP in the compiled reference) and the network (torch's own thread pool) take
    # turns on the same cores: idle workers of either pool must sleep, not spin
    os.environ.setdefault("OMP_WAIT_POLICY", "PASSIVE")
    os.environ.setdefault("GOMP_SPINCOUNT", "0")
    from oracle.pyoracle import OracleLib, RefLib, have_ref
    kind = "reference" if have_ref() else "port"
    L = RefLib() if kind == "reference" else OracleLib()
    cores = os.cpu_count() or 1
    import torch
    torch.set_num_threads(cores)
    ev_fn = cpu_mlp(flat)
    cfg = dict(num_games=games, seed=12345, max_searches=args.sims, searches_per_eval=args.spe,
               c_puct=args.c_puct, epsilon=args.epsilon, num_threads=cores)
    t = L.trainer(**cfg)
    evals = np.zeros(games * args.spe, np.float32)
    probs = np.zeros((games * args.spe, 96), np.float32)
    served, play_s, pred_s = 0, 0.0, 0.0
    t0 = time.perf_counter()
    complete = True
    while True:
        a = time.perf_counter()
        done = t.do_iteration(evals, probs, -1)
        play_s += time.perf_counter() - a
        if done:
            break
        n = t.num_requests(-1)
        req = t.write_requests(-1)
        a = time.perf_counter()
        e, p = ev_fn(req)
        evals[:n], probs[:n] = e, p
        pred_s += time.perf_counter() - a
        served += n
        if budget_s and time.perf_counter() - t0 > budget_s:
            complete = False
            break
    secs = time.perf_counter() - t0
    moves = t.num_samples()
    # every simulation either queues a leaf evaluation or ends in a terminal node; the exact
    # simulation count of the identical run comes from the oracle port's counter (bit-identical
    # search), measured outside the timed region when the run completed.
    sims = served
    sims_exact = False
    if complete and games <= 512:
        key = (games, args.sims, args.spe, args.c_puct, args.epsilon)
        if key not in _EXACT_SIMS:  # same seed every time: replay once, outside the timed region
            O = OracleLib()
            o = O.trainer(**cfg)
            from oracle.pyoracle import play_out
            play_out(o, evaluator=ev_fn)
            c = O.counters(o)
            _EXACT_SIMS[key] = (c["simulations"], c["leaf_evals"])
        if _EXACT_SIMS[key][1] == served:
            sims, sims_exact = _EXACT_SIMS[key][0], True
    return {"value": sims / secs, "unit": "sims/s", "moves_per_sec": moves / secs, "cores": cores,
            "kind": kind, "seconds": secs, "play_seconds": play_s, "predict_seconds": pred_s,
            "simulations": int(sims), "simulations_exact": sims_exact, "leaf_evals": int(served),
            "moves": int(moves), "complete": complete,
            "sample": "%d games x %d sims/move (spe %d) of the same workload, %s; C++/OpenMP tree with %d "
                      "threads + torch-CPU fp32 network (Keras unavailable)"
                      % (games, args.sims, args.spe, "to completion" if complete else "time-bounded", cores)}


def measure_game_logic(torch, cb, dev, n=1 << 26, reps=10):
    """BASELINE.json configs[1]: legal-move generation + terminal test + do_move on reachable
    states, device-resident (cb200_game_step_device). 64 Mi states per launch (>> L2: 1 GiB in,
    2 GiB out); the states are produced on the device by the kernel itself from the start
    position (next states fed back), so they are reachable. Returns states/s and the HBM
    roofline with the algorithmic 46 B/state of SURVEY.md 8(d) (48 B actually moved)."""
    import ctypes as C
    L = cb.lib()
    a = torch.zeros((n, 2), dtype=torch.int64, device=dev)
    a[:, 1] = 0x0000040404040404  # start position
    b = torch.empty_like(a)
    mf = torch.empty((n, 4), dtype=torch.int32, device=dev)
    for r in range(12):  # random legal play: every state gets its own random move sequence
        rc = L.cb200_game_step_device(n, C.c_void_p(a.data_ptr()), 1000 + r, C.c_void_p(mf.data_ptr()),
                                      C.c_void_p(b.data_ptr()), None)
        assert rc == 0
        a, b = b, a
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for r in range(reps):
        L.cb200_game_step_device(n, C.c_void_p(a.data_ptr()), 77 + r, C.c_void_p(mf.data_ptr()),
                                 C.c_void_p(b.data_ptr()), None)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    pk = peaks()
    gbs = 46.0 * n / (ms * 1e-3) / 1e9
    return {"states_per_sec": n / (ms * 1e-3), "states_per_launch": n, "ms_per_launch": ms,
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s",
                         "frac": gbs / pk["hbm_gbs"], "algorithmic_bytes_per_state": 46, "moved_bytes_per_state": 48,
                         "note": "paired kernel (two positions per thread finished together branch-free, a queue per warp, table-driven nth_move / do_move): "
                                 "10.7 warp instructions per position, ALU pipe 76 %, issue slots 71 %, DRAM 45 % busy in the ncu capture (of the form before the joint finish) "
                                 "profiles/r02_ncu_k_game_step_pair.txt -- no single limiter left; forms and history in "
                                 "profiles/r02_k1_paired_variants.txt"}}


# ----------------------------------------------------------------------------------------------
def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    import corintho_ai_b200 as cb
    flat = cb.fold_batchnorm(cb.random_weights(0))
    for _ in range(args.warmup):
        time_cpu_reference(args, flat, 4)
    sims = secs = moves = 0.0
    last = None
    for _ in range(args.steps):
        last = time_cpu_reference(args, flat, args.ref_games)
        sims += last["simulations"]
        secs += last["seconds"]
        moves += last["moves"]
    value = sims / secs
    line = {
        "impl": "reference", "metric": "mcts_simulations_per_sec", "value": value, "unit": "sims/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "moves_per_sec": moves / secs,
        "config": dict(workload_desc(args, args.gpus), reference_sample_games=args.ref_games),
        "cpu_baseline": {"value": value, "unit": "sims/s", "cores": last["cores"], "kind": last["kind"],
                         "sample": last["sample"], "play_seconds": last["play_seconds"],
                         "predict_seconds": last["predict_seconds"],
                         "evaluator_free_sims_per_sec": last["simulations"] / max(1e-9, last["play_seconds"])},
        "e2e": {"value": value, "unit": "sims/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def samples_digest(tr):
    """sha256 over the un-augmented samples of a finished run (game order): packed states, move
    probabilities, value labels, game indices."""
    import hashlib
    st, pr, lb, go = tr.raw_samples()
    h = hashlib.sha256()
    for a in (st, pr, lb, go):
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def dump_outputs(out_dir, tr, dist=None):
    """Write what a caller of the timed path receives after its last step: Trainer.write_samples()
    (game states [rows, 70], value labels [rows], move probabilities [rows, 96]; 8 symmetry rows per
    move) as float32, and the step's work counters (simulations, moves, leaf evaluations) as float64.
    When the rows exceed the 64 MB budget, a fixed seeded sample of them is written, in row order,
    with their indices in sample_rows.npy (float64), so that two builds can be compared row by row.
    With several GPUs each rank holds the rows of its contiguous shard of the games: rows are numbered
    in global game order (rank 0's first), the sample is drawn over all of them and rank 0 gathers and
    writes it, so the files are those of one trainer running every game. Returns None on other ranks."""
    gs, ev, pr = tr.write_samples()
    c = tr.counters()
    mine = np.array([gs.shape[0], c["simulations"], c["moves"], c["leaf_evals"]], np.int64)
    rank, world = (0, 1) if dist is None else (dist.get_rank(), dist.get_world_size())
    every = [mine]
    if dist is not None:
        every = [None] * world
        dist.all_gather_object(every, mine)
    every = np.stack(every)
    first, rows = int(every[:rank, 0].sum()), int(every[:, 0].sum())
    row_bytes = 4 * (gs.shape[1] + 1 + pr.shape[1]) + 8
    keep = min(rows, (DUMP_BUDGET_BYTES - (1 << 16)) // row_bytes)
    idx = np.arange(rows) if keep == rows else np.sort(np.random.default_rng(0).choice(rows, keep, replace=False))
    loc = idx[(idx >= first) & (idx < first + gs.shape[0])] - first
    parts = [(gs[loc], ev[loc], pr[loc])]
    if dist is not None:
        gathered = [None] * world if rank == 0 else None
        dist.gather_object(parts[0], gathered, dst=0)
        parts = gathered
    if rank != 0:
        return None
    arrays = {"game_states": np.concatenate([p[0] for p in parts]),
              "eval_samples": np.concatenate([p[1] for p in parts]),
              "prob_samples": np.concatenate([p[2] for p in parts]),
              "sample_rows": idx.astype(np.float64),
              "counters": every[:, 1:].sum(0).astype(np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return {"dir": out_dir, "rows": rows, "rows_written": int(keep), "files": sorted(arrays)}


def run_engine_arm(args, rank, world, local_rank):
    import torch
    import corintho_ai_b200 as cb
    dist = None
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # keep stdout = the one JSON line
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        # NCCL announces its version on stdout while the communicator is created: keep stdout for
        # the one JSON line by pointing fd 1 at stderr until the first collective has completed
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            warm = torch.zeros(1, device=torch.device("cuda", local_rank))
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    L = cb.lib()
    if L.cb200_set_device(local_rank) != 0:
        raise SystemExit("cb200_set_device failed: " + L.cb200_last_error().decode())
    dev = torch.device("cuda", local_rank)
    G = args.games_per_gpu
    flat = cb.fold_batchnorm(cb.random_weights(0))
    pinned_w = torch.from_numpy(flat).pin_memory()

    def make_trainer():
        t = cb.Trainer(G, "", 12345, args.sims, args.spe, args.c_puct, args.epsilon, 0, 1, False,
                       total_games=G * world, first_game=rank * G)
        t.set_weights(flat, 0, args.precision)
        return t

    tr = make_trainer()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_steps(t):
        """K steps of the workload: game state re-initialised (untimed), inputs resident in HBM,
        CUDA events around the run, barrier + synchronize on both sides."""
        ms, sims, moves, evals, iters = 0.0, 0, 0, 0, 0
        for k in range(args.steps):
            t.reset(2000 + k)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            t.run_selfplay(0, stagger=False)
            e1.record()
            barrier()
            ms += e0.elapsed_time(e1)
            c = t.counters()
            sims += c["simulations"]; moves += c["moves"]; evals += c["leaf_evals"]; iters += c["iterations"]
        return ms, sims, moves, evals, iters

    # ---- warm-up (untimed)
    for w in range(args.warmup):
        tr.reset(1000 + w)
        tr.run_selfplay(0, stagger=False)
    barrier()

    # ---- (1) device-timed steps: `value`
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = L.cb200_launch_count()
    tr.set_profiling(False)  # clears the phase clocks
    dev_ms, sims, moves, evals, iters = timed_steps(tr)
    launches = L.cb200_launch_count() - launches0
    phase_ms = tr.phase_times()  # of the timed (un-profiled) pass
    digest_timed = samples_digest(tr)
    dumped = dump_outputs(args.dump_outputs, tr, dist) if args.dump_outputs else None

    # ---- (2) the SAME steps on the SAME schedule (stream groups, parking, persistent tail) with a
    # CUDA-event pair around every kernel launch, recorded on the stream the kernel is launched on:
    # per-kernel-class durations for the roofline. Kernels of different stream groups overlap, so
    # the class times add up to more than the step (the overlap factor is reported); the event
    # records cost host time, so `value` comes from pass (1) and this pass reports
    # ms_per_step_profiled.
    tr.set_profiling(True)
    prof_ms, prof_sims, _, prof_evals, _ = timed_steps(tr)
    kt = tr.kernel_times()
    split = tr.phase_split()
    tr.set_profiling(False)
    digest_prof = samples_digest(tr)
    if digest_prof != digest_timed:
        raise SystemExit("bench.py: the profiled pass produced different samples than the timed pass")

    # ---- (3) reference execution of the same steps: ONE stream group, lock-step all the way (no
    # parking, no persistent kernel). Its kernels run alone, back to back, so its per-launch times
    # are the kernels' own; and its samples must hash equal to the timed schedule's.
    del tr
    gc.collect()
    saved = {k: os.environ.get(k) for k in ("CB200_GROUPS", "CB200_NO_PERSISTENT", "CB200_YIELD")}
    os.environ.update(CB200_GROUPS="1", CB200_NO_PERSISTENT="1", CB200_YIELD="0")
    tr = make_trainer()
    tr.set_profiling(True)
    iso_ms, iso_sims, _, iso_evals, _ = timed_steps(tr)
    kt_iso = tr.kernel_times()
    tr.set_profiling(False)
    digest_iso = samples_digest(tr)
    for k, v in saved.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = v
    if digest_iso != digest_timed:
        raise SystemExit("bench.py: the single-group lock-step pass produced different samples than the timed pass")
    del tr
    gc.collect()
    tr = make_trainer()
    clocks = sampler.stop() if rank == 0 else None
    game_logic = measure_game_logic(torch, cb, dev) if rank == 0 else None

    # ---- (4) end-to-end steps through the public API with host buffers: pinned weights -> device,
    # seeds/control blocks -> device, self-play, samples (8 symmetries) -> pinned host memory
    e2e = run_e2e(args, tr, torch, dist, dev, pinned_w, flat, G, barrier)
    digest_e2e = samples_digest(tr)
    if digest_e2e != digest_timed:
        raise SystemExit("bench.py: the end-to-end pass produced different samples than the timed pass")

    # ---- aggregate over ranks: max time, summed work
    if dist is not None:
        tt = torch.tensor([dev_ms, e2e["seconds"]], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dev_ms, e2e["seconds"] = float(tt[0]), float(tt[1])
        ww = torch.tensor([sims, moves, evals, e2e["sims"], launches], device=dev, dtype=torch.int64)
        dist.all_reduce(ww, op=dist.ReduceOp.SUM)
        sims, moves, evals, e2e["sims"], launches = (int(x) for x in ww)
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    pk = peaks()
    value = sims / (dev_ms * 1e-3)
    # work per kernel class of the profiled pass: lock-step launches vs persistent kernels
    ls_sims, ls_evals = split["lockstep_simulations"], split["lockstep_leaf_evals"]
    tail_sims, tail_evals = split["simulations"] - ls_sims, split["leaf_evals"] - ls_evals
    tail_ms = kt["fused_tail"]["ms"] + kt["fused_tail_wide"]["ms"]
    tail_launches = kt["fused_tail"]["launches"] + kt["fused_tail_wide"]["launches"]
    classes = {
        "game_step": {"kernel": "k_iterate (tree search game step, lock-step phase)", "ms": kt["game_step"]["ms"],
                      "launches": kt["game_step"]["launches"], "simulations": ls_sims},
        "network": {"kernel": "k_mlp_tc (policy/value network, lock-step phase)", "ms": kt["network"]["ms"],
                    "launches": kt["network"]["launches"], "leaf_evals": ls_evals},
        "fused_tail": {"kernel": "k_selfplay_persistent (game step + network per CTA, tail phase)", "ms": tail_ms,
                       "launches": tail_launches, "simulations": tail_sims, "leaf_evals": tail_evals},
    }
    total_class_ms = sum(c["ms"] for c in classes.values())
    dom = max(classes, key=lambda k: classes[k]["ms"])
    share = {k: classes[k]["ms"] / max(1e-9, total_class_ms) for k in classes}

    def hbm_roof(cls, traffic):
        c = classes[cls]
        per_launch_bytes = ALGO_BYTES_PER_SIM * c["simulations"] / max(1, c["launches"])
        ach = per_launch_bytes / (c["ms"] / max(1, c["launches"]) * 1e-3) / 1e9
        return {"kernel": c["kernel"], "bound": "hbm", "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s",
                "frac": ach / pk["hbm_gbs"], "traffic": traffic,
                "algorithmic_bytes_per_launch": per_launch_bytes, "avg_launch_us": 1e3 * c["ms"] / max(1, c["launches"])}

    if dom == "network":
        c = classes["network"]
        per_launch_flop = FLOP_PER_EVAL * c["leaf_evals"] / max(1, c["launches"])
        ach = per_launch_flop / (c["ms"] / max(1, c["launches"]) * 1e-3) / 1e12
        roof = {"kernel": c["kernel"], "bound": "tensor", "achieved": ach, "peak": pk["bf16_tflops_sustained"],
                "unit": "TFLOP/s", "frac": ach / pk["bf16_tflops_sustained"],
                "traffic": NCU_DRAM_BYTES_PER_DENSE_LAUNCH["network"]}
    elif dom == "fused_tail":
        roof = hbm_roof("fused_tail", None)
    else:
        roof = hbm_roof("game_step", NCU_DRAM_BYTES_PER_DENSE_LAUNCH["game_step"])
    roof["traffic_note"] = ("dram__bytes of ONE game-step launch with every game live (ncu --set full, " + NCU_SOURCE +
                            "): 209.2 MB for 109.4 MB algorithmic; `achieved` averages over all lock-step "
                            "launches of the run, most of which carry fewer games")
    roof["peak_source"] = pk["source"]
    roof["measured_on"] = ("the timed schedule itself: %d stream groups, parking, persistent tail; CUDA-event pair per "
                           "launch on the launching stream (pass 2)" % int(os.environ.get(
                               "CB200_GROUPS", 6 if G >= 2048 else (2 if G >= 512 else 1))))
    roof["kernel_time_share"] = share
    roof["kernel_ms_per_step"] = {k: classes[k]["ms"] / args.steps for k in classes}
    roof["kernel_launches_per_step"] = {k: classes[k]["launches"] / args.steps for k in classes}
    roof["stream_overlap_factor"] = total_class_ms / max(1e-9, prof_ms)
    # GPU-level rates of the two phases of the TIMED pass (host clock between the synchronisation
    # points that separate them; simulations per phase from the profiled pass of the same games):
    # what the whole device achieves while the overlapping kernels of a phase run
    roof["phases_of_the_timed_pass"] = {
        "lockstep": {"ms_per_step": phase_ms["lockstep_ms"] / args.steps, "simulations_per_step": ls_sims / args.steps,
                     "algorithmic_gbs": ALGO_BYTES_PER_SIM * ls_sims / max(1e-9, phase_ms["lockstep_ms"] * 1e-3) / 1e9,
                     "frac_of_hbm_peak": ALGO_BYTES_PER_SIM * ls_sims / max(1e-9, phase_ms["lockstep_ms"] * 1e-3) / 1e9 / pk["hbm_gbs"]},
        "persistent_tail": {"ms_per_step": phase_ms["tail_ms"] / args.steps, "simulations_per_step": tail_sims / args.steps,
                            "algorithmic_gbs": ALGO_BYTES_PER_SIM * tail_sims / max(1e-9, phase_ms["tail_ms"] * 1e-3) / 1e9,
                            "frac_of_hbm_peak": ALGO_BYTES_PER_SIM * tail_sims / max(1e-9, phase_ms["tail_ms"] * 1e-3) / 1e9 / pk["hbm_gbs"]},
    }
    roof["note"] = ("sum of kernel-class times per step = %.1f ms = %.2f x the profiled step (%.1f ms): kernels of "
                    "different stream groups overlap. Whole-step algorithmic rates of the timed pass: %.1f GB/s tree "
                    "traffic, %.2f TFLOP/s network"
                    % (total_class_ms / args.steps, total_class_ms / max(1e-9, prof_ms), prof_ms / args.steps,
                       ALGO_BYTES_PER_SIM * sims / (dev_ms * 1e-3) / 1e9, FLOP_PER_EVAL * evals / (dev_ms * 1e-3) / 1e12))
    # the other classes, same arithmetic, for the record
    roof["other"] = {}
    if classes["game_step"]["launches"] and dom != "game_step":
        roof["other"]["game_step"] = hbm_roof("game_step", NCU_DRAM_BYTES_PER_DENSE_LAUNCH["game_step"])
    if tail_launches and dom != "fused_tail":
        roof["other"]["fused_tail"] = hbm_roof("fused_tail", None)
    if classes["network"]["launches"]:
        roof["other"]["network_tflops"] = FLOP_PER_EVAL * ls_evals / (classes["network"]["ms"] * 1e-3) / 1e12
    # kernels alone (pass 3: one stream group, lock-step all the way)
    roof["isolated"] = {
        "ms_per_step": iso_ms / args.steps,
        "game_step_avg_launch_us": 1e3 * kt_iso["game_step"]["ms"] / max(1, kt_iso["game_step"]["launches"]),
        "network_avg_launch_us": 1e3 * kt_iso["network"]["ms"] / max(1, kt_iso["network"]["launches"]),
        "game_step_gbs": ALGO_BYTES_PER_SIM * iso_sims / max(1e-9, kt_iso["game_step"]["ms"] * 1e-3) / 1e9,
        "network_tflops": FLOP_PER_EVAL * iso_evals / max(1e-9, kt_iso["network"]["ms"] * 1e-3) / 1e12,
        "game_step_share": kt_iso["game_step"]["ms"] / max(1e-9, kt_iso["game_step"]["ms"] + kt_iso["network"]["ms"]),
    }

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        r = time_cpu_reference(args, flat, args.ref_games)
        cpu = {"value": r["value"], "unit": "sims/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"],
               "moves_per_sec": r["moves_per_sec"], "play_seconds": r["play_seconds"],
               "predict_seconds": r["predict_seconds"], "simulations_exact": r["simulations_exact"],
               "evaluator_free_sims_per_sec": r["simulations"] / max(1e-9, r["play_seconds"])}

    line = {
        "metric": "mcts_simulations_per_sec", "value": value, "unit": "sims/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
        "config": workload_desc(args, world),
        "moves_per_sec": moves / (dev_ms * 1e-3), "leaf_evals_per_sec": evals / (dev_ms * 1e-3),
        "simulations_per_step": sims / args.steps, "iterations_per_step": iters / args.steps,
        "ms_per_step_profiled": prof_ms / args.steps,
        "samples_sha256": digest_timed,
        "samples_check": "timed pass == profiled pass == single-group lock-step pass == end-to-end pass",
        "game_logic": game_logic,
        "e2e": {"value": e2e["sims"] / e2e["seconds"], "unit": "sims/s", "h2d_bytes_per_step": e2e["h2d"] // args.steps,
                "d2h_bytes_per_step": e2e["d2h"] // args.steps, "seconds_per_step": e2e["seconds"] / args.steps,
                "nccl_gather_seconds_per_step": e2e["gather_s"] / args.steps if world > 1 else 0.0,
                "path": e2e["path"]},
        "gpu_launches": int(launches),
        "roofline": roof,
        "cpu_baseline": cpu,
        "clocks": clocks,
    }
    if dumped is not None:
        line["dumped_outputs"] = dumped
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def run_e2e(args, tr, torch, dist, dev, pinned_w, flat, G, barrier):
    """End-to-end steps through the public API: host weights in, host samples out (all 8
    symmetries of every move, 668 B per row). The samples of finished games are streamed to
    the trainer's pinned host buffers during the run (Trainer.stream_samples), so the 370 MB
    device->host transfer overlaps the self-play instead of following it; the timed region ends
    when the last row is in host memory. Rows come in game completion order with a game index
    per sample (see include/corintho_b200.h)."""
    # staging capacity in samples: a game lasts ~19 moves on average (33 at most observed)
    tr.stream_samples(G * 32 if G <= 8192 else G * 24)
    tr.reset(2000)
    tr.run_selfplay(0, stagger=False)  # untimed warm-up of the streaming path
    tr.streamed_samples()
    comm, world = None, 1
    if dist is not None:  # the engine's own NCCL communicator (C ABI), warmed up once
        import corintho_ai_b200 as cb
        world = dist.get_world_size()
        comm = cb.nccl_comm_from_torch(dist, dist.get_rank(), world, dev)
        tr.allgather_samples(comm, world)
    out = {"seconds": 0.0, "sims": 0, "h2d": 0, "d2h": 0, "gather_s": 0.0,
           "path": "set_weights(pinned host) + reset + run_selfplay with streamed samples (8 symmetries, "
                   "completion order + game index) + streamed_samples() = all rows in pinned host memory"}
    for k in range(args.steps):
        barrier()
        t0 = time.perf_counter()
        tr.set_weights(pinned_w.numpy(), 0, args.precision)
        tr.reset(2000 + k)
        tr.run_selfplay(0, stagger=False)
        gs, ev, pr, game_of = tr.streamed_samples()
        if comm is not None:  # all-gather the finished (un-augmented) samples over NCCL (C ABI)
            g0 = time.perf_counter()
            ptr_all, n_all, per_rank = tr.allgather_samples(comm, world)
            out["gather_s"] += time.perf_counter() - g0
        torch.cuda.synchronize()
        out["seconds"] += time.perf_counter() - t0
        if comm is not None and (n_all != int(per_rank.sum()) or int(per_rank[dist.get_rank()]) != tr.num_samples()):
            raise SystemExit("bench.py: the NCCL sample gather is inconsistent")
        if game_of.shape[0] != tr.num_samples():
            raise SystemExit("bench.py: the streamed samples are incomplete")
        out["sims"] += tr.counters()["simulations"]
        out["h2d"] += flat.nbytes + G * (20 + 24 + 1) * 4  # weights + control blocks, tree headers, seeds
        out["d2h"] += gs.nbytes + ev.nbytes + pr.nbytes + game_of.nbytes
    # the streamed rows of the last step, brought into game order, must be writeSamples' rows
    order = np.argsort(game_of, kind="stable")
    rows = (order[:, None] * 8 + np.arange(8)[None, :]).ravel()
    g2, e2, p2 = tr.write_samples()
    if not (np.array_equal(gs[rows].view(np.uint32), g2.view(np.uint32)) and
            np.array_equal(ev[rows].view(np.uint32), e2.view(np.uint32)) and
            np.array_equal(pr[rows].view(np.uint32), p2.view(np.uint32))):
        raise SystemExit("bench.py: streamed samples differ from Trainer::writeSamples")
    if comm is not None:
        # the gathered rows of the last step: every rank's samples, in global game order
        from corintho_ai_b200.dist import device_rows_as_tensor
        games = device_rows_as_tensor(ptr_all, n_all, 102, dev)[:, 101].contiguous().view(torch.int32).cpu().numpy()
        if not (np.all(np.diff(games) >= 0) and games[0] == 0 and games[-1] == G * world - 1 and
                len(np.unique(games)) == G * world):
            raise SystemExit("bench.py: the gathered samples are not in global game order")
        import corintho_ai_b200 as cb
        cb.lib().cb200_nccl_comm_destroy(C_void_p(comm))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--games-per-gpu", type=int, default=4096)
    ap.add_argument("--sims", type=int, default=800)
    ap.add_argument("--spe", type=int, default=16)
    ap.add_argument("--c-puct", type=float, default=1.0)
    ap.add_argument("--epsilon", type=float, default=0.25)
    ap.add_argument("--precision", default=os.environ.get("CB200_PRECISION", "bf16"), choices=["bf16", "fp32"])
    ap.add_argument("--ref-games", type=int, default=256, help="games in one CPU-reference sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the samples of the last timed step, of all ranks, as DIR/<name>.npy "
                         "(engine arm, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "engine":
        ap.error("--dump-outputs writes the engine's outputs: it needs --impl engine")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world == 1 and args.gpus != 1:
        # launched without torchrun: run the requested shape on this one process' GPU count
        args.gpus = 1
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
    else:
        run_engine_arm(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
