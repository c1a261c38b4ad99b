"""Small run of every new device path for compute-sanitizer (memcheck / racecheck):
   compute-sanitizer --tool memcheck python tools/san_small.py"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import corintho_ai_b200 as cb

flat = cb.fold_batchnorm(cb.random_weights(0))
# fused training run with stream groups, live lists, persistent tail, streamed samples
os.environ["CB200_GROUPS"] = "2"
t = cb.Trainer(160, "", 3, 48, 16, 1.0, 0.25)
t.set_weights(flat, 0, "bf16")
t.stream_samples()
assert t.run_selfplay(0, stagger=True)
gs, ev, pr, go = t.streamed_samples()
assert go.shape[0] == t.num_samples()
t.write_samples(); t.raw_samples_device()
# bf16x3 network, two-model testing mode, fused tourney, K1
v = cb.Trainer(32, "", 5, 32, 8, 1.0, 0.0, 0, 1, True)
v.set_weights(flat, 0, "bf16x3"); v.set_weights(flat, 1, "bf16x3")
assert v.run_selfplay(0)
T = cb.Tourney(1, "")
T.addPlayer(0, 0, 32, 8, 1.0, 0.25); T.addPlayer(1, 1, 24, 4, 1.5, 0.1); T.addPlayer(2, -1, 1, 1, 1.0, 0.25, True)
for a, b in ((0, 1), (1, 0), (0, 2), (2, 1)):
    T.addMatch(a, b)
T.set_weights(0, flat, "bf16"); T.set_weights(1, flat, "fp32")
assert T.run(0)
st = np.zeros((5000, 2), np.uint64); st[:, 1] = 0x0000040404040404
for r in range(6):
    mf, st, _ = cb.game_step(st, 100 + r)
print("san_small OK", t.counters(), len(T.scores()))
