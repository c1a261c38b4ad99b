#!/usr/bin/env python
"""Cost of the analysis' external-evaluator protocol (cb200_analysis_begin .. _results). On the same
reachable positions, in one process, three ways to search them: the protocol on host buffers, the
protocol on device buffers, both with a torch restatement of the network (fp32) as the caller's
evaluator, and the fused cb200_analysis_run with the resident network (fp32 and bf16). Each protocol
line splits its wall time into the evaluator's part (the torch network, and for host buffers its
host<->device copies) and the protocol's own part per round (summary read-back, request packing,
answer and row copies, game-step kernel). Prints one JSON line per measurement.
    python tools/analysis_protocol_bench.py [--out FILE] [--sizes 4096,32768] [--sims 800] [--repeats 3]"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402

import corintho_ai_b200 as cb  # noqa: E402
from analysis_bench import card  # noqa: E402
from oracle.pyoracle import OracleLib  # noqa: E402
from torch_net import torch_network  # noqa: E402


def protocol_pass(a, states, seed, net, on_device, rows_d):
    """One search of every position through the protocol; returns (outputs, seconds, evaluator
    seconds, rounds)."""
    dev = rows_d.device
    eval_s, rounds = 0.0, 0
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    a.begin(states, seed)
    if on_device:
        empty = torch.empty(0, device=dev)
        ans = (empty, empty)
        while not a.do_iteration_device(*ans):
            n = a.num_requests()
            a.write_requests_device(rows_d)
            te = time.perf_counter()
            ans = net(rows_d[:n])
            torch.cuda.synchronize()
            eval_s += time.perf_counter() - te
            rounds += 1
    else:
        ans = (None, None)
        while not a.do_iteration(*ans):
            rows = a.write_requests()
            te = time.perf_counter()
            v, p = net(torch.from_numpy(rows).to(dev))
            ans = (v.cpu().numpy(), p.cpu().numpy())
            eval_s += time.perf_counter() - te
            rounds += 1
    out = a.results()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0, eval_s, rounds


def time_protocol(states, sims, spe, net, on_device, repeats):
    n = len(states)
    a = cb.Analysis(n, sims, spe, 1.0, 0.25)
    rows_d = torch.empty((n * spe, cb.STATE_SIZE), device="cuda")
    protocol_pass(a, states[:256], 1, net, on_device, rows_d)  # warm-up
    best = None
    for _ in range(repeats):
        out, dt, eval_s, rounds = protocol_pass(a, states, 100, net, on_device, rows_d)
        if best is None or dt < best[1]:
            best = (out, dt, eval_s, rounds, a.counters())
    out, dt, eval_s, rounds, c = best
    a.close()
    line = {"what": "protocol_device" if on_device else "protocol_host", "positions": n,
            "searched": int((out["moves"] >= 0).sum()), "max_searches": sims, "searches_per_eval": spe,
            "evaluator": "torch fp32", "rounds": rounds, "seconds": round(dt, 4),
            "evaluator_seconds": round(eval_s, 4),
            "protocol_ms_per_round": round(1e3 * (dt - eval_s) / max(rounds, 1), 3),
            "positions_per_s": round(n / dt, 1), "simulations": c["simulations"],
            "simulations_per_s": round(c["simulations"] / dt, 1), "leaf_evals": c["leaf_evals"]}
    return line, out


def time_fused(states, sims, spe, precision, weights, repeats):
    a = cb.Analysis(len(states), sims, spe, 1.0, 0.25)
    a.set_weights(weights, precision)
    a.run(states[:256], seed=1)  # warm-up (network upload, first launches)
    best = None
    for r in range(repeats):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        a.run(states, seed=100 + r)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, a.counters())
    dt, c = best
    a.close()
    return {"what": "fused_run", "positions": len(states), "max_searches": sims, "searches_per_eval": spe,
            "precision": precision, "seconds": round(dt, 4), "positions_per_s": round(len(states) / dt, 1),
            "simulations": c["simulations"], "simulations_per_s": round(c["simulations"] / dt, 1),
            "leaf_evals": c["leaf_evals"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--sizes", default="4096,32768")
    ap.add_argument("--sims", type=int, default=800)
    ap.add_argument("--spe", type=int, default=16)
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    lines = []

    def emit(d):
        s = json.dumps(d)
        print(s, flush=True)
        lines.append(s)

    emit(dict(card(), torch=torch.__version__))
    weights = cb.fold_batchnorm(cb.random_weights(0))
    net = torch_network(weights, torch.device("cuda", 0))
    sizes = [int(x) for x in args.sizes.split(",")]
    all_states = cb.planes_from_reference_order(OracleLib().gen_states(2024, max(sizes)))
    for n in sizes:
        st = all_states[:n]
        try:  # 32 768 positions x 800 searches take ~99 GB of node arenas
            host, out_h = time_protocol(st, args.sims, args.spe, net, False, args.repeats)
            emit(host)
            dev, out_d = time_protocol(st, args.sims, args.spe, net, True, args.repeats)
            # the same evaluator on the same rows: the two forms should agree on every move
            dev["same_moves_as_host"] = bool((out_h["moves"] == out_d["moves"]).all())
            emit(dev)
            for precision in ("fp32", "bf16"):
                emit(time_fused(st, args.sims, args.spe, precision, weights, args.repeats))
        except cb.Corintho200Error as e:
            emit({"positions": n, "error": str(e)})
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
