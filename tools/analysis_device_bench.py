#!/usr/bin/env python
"""Analysis with positions already on the GPU: (a) cb200_analysis_run from host arrays, (b)
cb200_analysis_run_device on device-resident states (CUDA events on the stream), (c) replay of a
CUDA graph captured from (b). Reachable positions from random play-outs, 800 searches each
(searches_per_eval 16, random-init network), bf16 and bf16x3; every time is the best of --repeats
after a warm-up, and the three forms are checked to give identical outputs in the same process.
Prints one JSON line per measurement and writes them (plus a table) next to --out.
    python tools/analysis_device_bench.py [--out profiles/r05_analysis_device_bench.jsonl]
                                          [--sizes 1,16,148,2368,4096,32768] [--sims 800]"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import corintho_ai_b200 as cb  # noqa: E402
from analysis_bench import card  # noqa: E402
from oracle.pyoracle import OracleLib  # noqa: E402

KEYS = ("moves", "results", "values", "visits", "evals")


def same(x, y):
    return all(np.array_equal(np.ascontiguousarray(x[k]).view(np.uint8), np.ascontiguousarray(y[k]).view(np.uint8))
               for k in KEYS)


def to_host(out):
    return {k: v.cpu().numpy() for k, v in out.items()}


def measure(states, sims, spe, precision, weights, repeats, seed=5):
    n = len(states)
    L = cb.lib()
    a = cb.Analysis(n, sims, spe, 1.0, 0.25)
    a.set_weights(weights, precision)
    # (a) run from host arrays
    ref = a.run(states, seed)  # warm-up
    t_run = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        out_a = a.run(states, seed)
        dt = time.perf_counter() - t0
        t_run = dt if t_run is None else min(t_run, dt)
    sims_done = a.counters()["simulations"]
    # (b) run_device on the library's stream (a side stream of torch)
    stream = torch.cuda.Stream()
    st_d = torch.from_numpy(np.ascontiguousarray(states).view(np.int64)).cuda()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_dev = t_graph = None
    try:
        with torch.cuda.stream(stream):
            assert L.cb200_set_stream(stream.cuda_stream) == 0
            out = a.run_device(st_d, seed)  # warm-up: buffers, shared-memory attribute
            stream.synchronize()
            for _ in range(repeats):
                ev0.record(stream)
                a.run_device(st_d, seed, out=out)
                ev1.record(stream)
                ev1.synchronize()
                dt = ev0.elapsed_time(ev1) / 1e3
                t_dev = dt if t_dev is None else min(t_dev, dt)
            out_b = to_host(out)
            status = out["status"].tolist()
            assert a.counters()["simulations"] == sims_done
            # (c) replay of a captured graph of (b)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=stream):
                a.run_device(st_d, seed, out=out)
            for v in out.values():
                v.zero_()
            for _ in range(repeats + 1):  # the first replay is the warm-up
                ev0.record(stream)
                graph.replay()
                ev1.record(stream)
                ev1.synchronize()
                dt = ev0.elapsed_time(ev1) / 1e3
                t_graph = dt if t_graph is None else min(t_graph, dt)
            out_c = to_host(out)
            del graph
    finally:
        L.cb200_set_stream(None)
    identical = same(ref, out_a) and same(out_a, out_b) and same(out_a, out_c) and status == [0, 0]
    a.close()
    return {"what": "analysis_device", "positions": n, "searched": int((out_a["moves"] >= 0).sum()),
            "max_searches": sims, "searches_per_eval": spe, "precision": precision, "simulations": sims_done,
            "run_s": round(t_run, 6), "run_device_s": round(t_dev, 6), "graph_replay_s": round(t_graph, 6),
            "run_sims_per_s": round(sims_done / t_run, 1), "run_device_sims_per_s": round(sims_done / t_dev, 1),
            "graph_sims_per_s": round(sims_done / t_graph, 1), "outputs_identical": identical}


def table(lines, head):
    rows = [head, "",
            "| precision | positions | run (a) | run_device (b) | graph replay (c) | (a)/(b) | sims/s (b) | identical |",
            "|---|---|---|---|---|---|---|---|"]
    for d in lines:
        if d.get("what") != "analysis_device":
            continue
        rows.append(f"| {d['precision']} | {d['positions']} | {d['run_s'] * 1e3:.3f} ms | "
                    f"{d['run_device_s'] * 1e3:.3f} ms | {d['graph_replay_s'] * 1e3:.3f} ms | "
                    f"{d['run_s'] / d['run_device_s']:.2f} | {d['run_device_sims_per_s']:.3e} | "
                    f"{d['outputs_identical']} |")
    return "\n".join(rows) + "\n"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="JSON lines; a .txt table is written beside it")
    ap.add_argument("--sizes", default="1,16,148,2368,4096,32768")
    ap.add_argument("--sims", type=int, default=800)
    ap.add_argument("--spe", type=int, default=16)
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(d)

    info = dict(card(), torch=torch.__version__)
    emit(info)
    weights = cb.fold_batchnorm(cb.random_weights(0))
    sizes = [int(x) for x in args.sizes.split(",")]
    all_states = cb.planes_from_reference_order(OracleLib().gen_states(2024, max(sizes)))
    for precision in ("bf16", "bf16x3"):
        for n in sizes:
            emit(measure(all_states[:n], args.sims, args.spe, precision, weights, args.repeats))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("".join(json.dumps(d) + "\n" for d in lines))
        head = (f"Analysis, positions on the device: {info['gpu']}, power limit {info['power_limit']}; "
                f"{args.sims} searches, spe {args.spe}, best of {args.repeats} after a warm-up "
                "((a) host clock around the synchronous call, (b) and (c) CUDA events on the stream).")
        with open(os.path.splitext(args.out)[0] + ".txt", "w") as f:
            f.write(table(lines, head))


if __name__ == "__main__":
    main()
