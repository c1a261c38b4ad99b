"""Sweep parking budget / stream groups for the fused self-play run (min of N repetitions)."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import corintho_ai_b200 as cb
games = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
groups = [int(x) for x in (sys.argv[3] if len(sys.argv) > 3 else "1").split(",")]
budgets = [x for x in (sys.argv[4] if len(sys.argv) > 4 else "0,96").split(",")]
w = cb.fold_batchnorm(cb.random_weights(0))
for g in groups:
    os.environ["CB200_GROUPS"] = str(g)
    for b in budgets:
        fv = ""
        y, _, ml = b.partition(":")
        os.environ["CB200_YIELD"] = y
        if ml: os.environ["CB200_YIELD_MIN_LIVE"] = ml
        else: os.environ.pop("CB200_YIELD_MIN_LIVE", None)
        t = cb.Trainer(games, "", 12345, 800, 16, 1.0, 0.25)  # reads the schedule knobs
        t.set_weights(w, 0, "bf16")
        t.run_selfplay(0, stagger=False)  # warm-up: full run
        ts = []
        for r in range(reps):
            t.reset(12345)
            t0 = time.perf_counter()
            t.run_selfplay(0, stagger=False)
            ts.append(time.perf_counter() - t0)
        c = t.counters()
        print("groups %d yield %-8s min %.4f s med %.4f s  iterations %d  sims/s %.3e" % (g, b + ("/" + fv if fv else ""), min(ts), sorted(ts)[len(ts)//2], c["iterations"], c["simulations"] / min(ts)), flush=True)
        del t
