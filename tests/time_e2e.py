import os, sys, time, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
from cropnerf_b200 import engine
dev = torch.device("cuda:0")
model = bench.build_model(dev, "mixed")
tr = engine.Trainer(model)
host = [bench.host_batch(4096, seed=i) for i in range(4)]
step = 0
for _ in range(5):
    rb, tg = bench.to_bundle(host[step % 4], dev); tr.train_iteration(step, rb, tg); step += 1
torch.cuda.synchronize()
T = {"h2d": 0, "call": 0, "item": 0}
for _ in range(20):
    t0 = time.perf_counter()
    rb, tg = bench.to_bundle(host[step % 4], dev)
    t1 = time.perf_counter()
    st = tr.train_iteration(step, rb, tg); step += 1
    t2 = time.perf_counter()
    v = float(st["loss"].item())
    t3 = time.perf_counter()
    T["h2d"] += t1 - t0; T["call"] += t2 - t1; T["item"] += t3 - t2
print({k: round(v / 20 * 1e3, 3) for k, v in T.items()})
import cProfile, pstats
pr = cProfile.Profile(); pr.enable()
for _ in range(20):
    rb, tg = bench.to_bundle(host[step % 4], dev)
    st = tr.train_iteration(step, rb, tg); step += 1
    v = float(st["loss"].item())
pr.disable()
pstats.Stats(pr).sort_stats("cumulative").print_stats(25)
