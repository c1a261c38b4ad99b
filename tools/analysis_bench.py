#!/usr/bin/env python
"""Analysis throughput (cb200_analysis_run): reachable positions from random play-outs searched with
800 searches each (searches_per_eval 16, random-init network, bf16 and bf16x3), timed with device
synchronisation, next to the fused tourney's simulations/s measured in the same process as a
reference point. Prints one JSON line per measurement.
    python tools/analysis_bench.py [--out FILE] [--sizes 4096,32768] [--sims 800] [--repeats 3]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import corintho_ai_b200 as cb  # noqa: E402
from oracle.pyoracle import OracleLib  # noqa: E402


def card():
    name = torch.cuda.get_device_name(0)
    try:  # read-only query of the board's power limit
        limit = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return {"gpu": name, "power_limit": limit}


def time_analysis(states, sims, spe, precision, weights, repeats):
    a = cb.Analysis(len(states), sims, spe, 1.0, 0.25)
    a.set_weights(weights, precision)
    a.run(states[:256], seed=1)  # warm-up (network upload, first launches)
    best = None
    for r in range(repeats):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = a.run(states, seed=100 + r)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        c = a.counters()
        if best is None or dt < best[0]:
            best = (dt, c)
    dt, c = best
    searched = int((out["moves"] >= 0).sum())
    a.close()
    return {"what": "analysis", "positions": len(states), "searched": searched, "max_searches": sims,
            "searches_per_eval": spe, "precision": precision, "seconds": round(dt, 4),
            "positions_per_s": round(len(states) / dt, 1), "simulations": c["simulations"],
            "simulations_per_s": round(c["simulations"] / dt, 1), "leaf_evals": c["leaf_evals"]}


def time_tourney(sims, spe, precision, weights, matches_per_side):
    t = cb.Tourney(1, "")
    t.addPlayer(0, 0, sims, spe, 1.0, 0.25)
    t.addPlayer(1, 1, sims, spe, 1.0, 0.25)
    for _ in range(matches_per_side):
        t.addMatch(0, 1)
        t.addMatch(1, 0)
    t.set_weights(0, weights, precision)
    t.set_weights(1, weights, precision)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    assert t.run(0)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    c = t.counters()
    t.close()
    return {"what": "fused_tourney", "matches": 2 * matches_per_side, "max_searches": sims,
            "searches_per_eval": spe, "precision": precision, "seconds": round(dt, 4),
            "simulations": c["simulations"], "simulations_per_s": round(c["simulations"] / dt, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--sizes", default="4096,32768")
    ap.add_argument("--sims", type=int, default=800)
    ap.add_argument("--spe", type=int, default=16)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--tourney-matches", type=int, default=256, help="matches per seat order")
    args = ap.parse_args()
    lines = []

    def emit(d):
        s = json.dumps(d)
        print(s, flush=True)
        lines.append(s)

    emit(dict(card(), torch=torch.__version__))
    weights = cb.fold_batchnorm(cb.random_weights(0))
    sizes = [int(x) for x in args.sizes.split(",")]
    all_states = cb.planes_from_reference_order(OracleLib().gen_states(2024, max(sizes)))
    for precision in ("bf16", "bf16x3"):
        for n in sizes:
            try:  # 32 768 positions x 800 searches take ~99 GB of node arenas
                emit(time_analysis(all_states[:n], args.sims, args.spe, precision, weights, args.repeats))
            except cb.Corintho200Error as e:
                emit({"what": "analysis", "positions": n, "precision": precision, "error": str(e)})
        emit(time_tourney(args.sims, args.spe, precision, weights, args.tourney_matches))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
